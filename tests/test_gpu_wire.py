"""Compact wire format on the GPU ("next" row N3): nrm_expand_compact rebuilds the reference's packed float64 tensors bit for
bit, so the scoring forward and a whole training step fed with ids equal the same calls fed with the packed tensors."""
import numpy as np
import pytest
import torch

import news_recommendation_model_b200 as nrm
from news_recommendation_model_b200 import _lib, wire
from fixtures import load_weights
from oracle.wire_port import expand_reference

pytestmark = pytest.mark.gpu


def _host_packed(table, cb):
    return expand_reference(table.rows.numpy(), cb.hist_article.numpy(), cb.hist_time.numpy(), cb.hist_click.numpy(),
                            cb.cand_article.numpy(), cb.cand_time.numpy())


@pytest.mark.parametrize('B,H,C', [(1, 1, 1), (7, 50, 5), (33, 200, 40)])
def test_expand_matches_host_restatement_bit_for_bit(B, H, C):
    table = wire.make_article_table(3000, seed=B)
    cb = wire.make_compact_batch(table, B, H, C, seed=10 + B, variable_history=True, variable_candidates=C > 5)
    cb.hist_article[0, 0] = 10 ** 6          # out of range -> pad article
    cb.cand_article[-1, -1] = -5
    xh, xt, xg = _host_packed(table, cb)
    d = wire.expand(table.to('cuda'), cb.to('cuda'))
    assert torch.equal(d.x_history.cpu(), xh) and torch.equal(d.x_target.cpu(), xt) and torch.equal(d.x_global.cpu(), xg)
    assert torch.equal(d.label.cpu(), cb.label.double())


def test_expand_refuses_cpu_tensors_and_wrong_dtypes():
    table = wire.make_article_table(10)
    cb = wire.make_compact_batch(table, 2, 3, 2)
    with pytest.raises(nrm.NrmError):
        wire.expand_into(table, cb, torch.empty(2, 3, 80, dtype=torch.float64), torch.empty(2, 2, 78, dtype=torch.float64),
                         torch.empty(2, 2, 3, dtype=torch.float64), None)
    dcb = cb.to('cuda'); dcb.hist_article = dcb.hist_article.long()
    with pytest.raises(ValueError):
        wire.expand(table.to('cuda'), dcb)


def test_scoring_forward_is_identical_for_both_wire_formats():
    table = wire.make_article_table(5000, seed=3)
    cb = wire.make_compact_batch(table, 40, 200, 30, seed=4, user_num=50, variable_history=True, variable_candidates=True)
    xh, xt, xg = _host_packed(table, cb)
    m = nrm.UserModel(50)
    m.load_state_dict(load_weights('validation'), strict=False)
    m.to('cuda').eval().set_precision('bf16x3')
    with torch.no_grad():
        ref = m(xh.cuda(), xt.cuda(), xg.cuda())
        d = wire.expand(table.to('cuda'), cb.to('cuda'))
        out = m(d.x_history, d.x_target, d.x_global)
    assert torch.equal(out, ref)


@pytest.mark.parametrize('precision', ['bf16x3', 'fp32'])
def test_compact_train_step_launches_what_the_packed_one_does_and_ends_with_its_bits(precision):
    """The compact batch is the direct input of the row kernels (nrm_forward_compact / nrm_backward_compact, no packed tensors) in
    every precision: an eager step launches as many kernels as one fed the packed tensors (no expansion kernel runs), and three
    training steps end with the same bits as feeding the reference's packed float64 tensors."""
    B, H, C = 64, 50, 5
    lib = _lib.load()
    table = wire.make_article_table(2000, seed=5)
    batches = [wire.make_compact_batch(table, B, H, C, seed=20 + i, user_num=100) for i in range(3)]
    results, launches = [], []
    for fmt in ('packed', 'compact'):
        m = nrm.UserModel(100)
        m.load_state_dict(load_weights('train'), strict=False)
        m.to('cuda').train().set_precision(precision)
        tr = nrm.FusedTrainStep(m, B, H, C, lr=1e-3, weight_decay=1e-5, articles=table.to('cuda'))
        feeds = []
        for cb in batches:
            if fmt == 'packed':
                xh, xt, xg = _host_packed(table, cb)
                feeds.append(nrm.synthetic.Batch(cb.impression_id, cb.user_id, xh, xt, xg, cb.label.double(), cb.label.double(), cb.empty_num).pin())
            else:
                feeds.append(cb.pin())
        losses = [tr.step(feed).item() for feed in feeds]
        torch.cuda.synchronize()
        results.append((losses, m.flat_parameters().buf.clone(), m.bn.running_mean.clone(), m.bn.running_var.clone()))
        tr.use_graph = False                     # one step more, eager: count the library's kernel launches
        n0 = lib.nrm_launch_count()
        tr.step(feeds[0]).item()
        launches.append(lib.nrm_launch_count() - n0)
    (l0, p0, r0, v0), (l1, p1, r1, v1) = results
    assert l0 == l1
    assert torch.equal(p0, p1) and torch.equal(r0, r1) and torch.equal(v0, v1)
    assert launches[0] == launches[1] > 0, launches


def test_slot_recaptures_its_graph_when_the_wire_format_changes():
    B, H, C = 16, 20, 5
    table = wire.make_article_table(500, seed=6)
    cb = wire.make_compact_batch(table, B, H, C, seed=1, user_num=100)
    xh, xt, xg = _host_packed(table, cb)
    packed = nrm.synthetic.Batch(cb.impression_id, cb.user_id, xh, xt, xg, cb.label.double(), cb.label.double(), cb.empty_num)
    m = nrm.UserModel(100)
    m.load_state_dict(load_weights('train'), strict=False)
    m.to('cuda').train()
    tr = nrm.FusedTrainStep(m, B, H, C, lr=0.0, weight_decay=0.0, nslots=1, articles=table.to('cuda'))
    a = tr.step(packed).item()
    b = tr.step(cb).item()
    c = tr.step(packed).item()
    assert a == b == c           # lr = 0: the same batch gives the same loss through either format (BN in batch-stat mode)


def test_records_through_the_prefetch_loader_train_like_the_packed_path_bit_for_bit():
    """The loader row N4 end to end: the reference's record list (tool/process_data.py:252 layout) -> wire.from_records ->
    wire.PrefetchLoader (background thread, fixed pinned ring, ragged last batch) -> FusedTrainStep, against the same impressions
    fed as packed float64 tensors in the same order: every loss and the final weights are bit-identical."""
    from news_recommendation_model_b200.synthetic import Batch, make_batch
    N, B, H, C, U = 40, 16, 50, 5, 60
    full = make_batch(N, H, C, seed=808, user_num=U, fp32_exact=True, variable_history=True)
    records = [[full.impression_id[i].numpy(), full.user_id[i].numpy(), full.x_history[i].numpy(), full.x_target[i].numpy(),
                full.x_global[i].numpy(), full.label[i].numpy(), full.label_id[i].numpy(), full.empty_num[i].numpy()] for i in range(N)]
    ds = wire.from_records(records, pin=True)

    def fresh():
        m = nrm.UserModel(U)
        m.load_state_dict(load_weights('train'), strict=False)
        return m.to('cuda').train()
    ma, mb = fresh(), fresh()
    ta = nrm.FusedTrainStep(ma, B, H, C, lr=1e-3, weight_decay=1e-5, articles=ds.table.to('cuda'))
    tb = nrm.FusedTrainStep(mb, B, H, C, lr=1e-3, weight_decay=1e-5)
    la = [ta.step(cb) for cb in wire.PrefetchLoader(ds, B, depth=2)]
    la = None or la
    lb = []
    for s in range(0, N, B):
        sl = Batch(*[getattr(full, f)[s:s + B] for f in full.__dataclass_fields__])
        lb.append(tb.step(sl.pin()))
    assert len(la) == len(lb) == 3
    va, vb = [h.item() for h in la], [h.item() for h in lb]
    assert va == vb, (va, vb)
    assert torch.equal(ma.flat_parameters().buf, mb.flat_parameters().buf)
    assert torch.equal(ma.bn.running_mean, mb.bn.running_mean)
