"""Pool negatives on the GPU: NegativeSampler.sample against the integer reference (tests/negatives_ref.py) id for id, the sampling
invariants and distributions at scale, and FusedTrainStep(negatives=...) against the same step fed pre-sampled batches."""
import numpy as np
import pytest
import torch
from scipy.stats import chisquare

import negatives_ref as R
import news_recommendation_model_b200 as nrm
from fixtures import load_weights
from news_recommendation_model_b200 import negatives, wire

pytestmark = pytest.mark.gpu


def _table(n):
    return wire.ArticleTable(torch.zeros(n, wire.ARTICLE_COLS, device='cuda'))


def _batch(table, B, H, C0, seed, no_positive_every=0):
    cb = wire.make_compact_batch(table, B, H, C0, seed=seed, user_num=100, variable_history=True, variable_candidates=C0 >= 5)
    if no_positive_every:
        cb.label[2::no_positive_every] = 0.0                 # impressions 2, 2 + n, ... without a positive
    return cb.to('cuda')


def _check_against_reference(s, cb, step, row_offset, weights):
    B, H, C0 = cb.shape
    got = s.sample(cb, step=step, row_offset=row_offset)
    ids, times, labels = R.sample(cb.hist_article.tolist(), cb.cand_article.tolist(), cb.cand_time.tolist(), cb.label.tolist(),
                                  s.pool_article.tolist(), weights, s.table.n, s.k, s.seed, step, row_offset)
    assert got.shape == (B, H, C0 + s.k)
    for f in ('cand_article', 'cand_time', 'label'):
        assert torch.equal(getattr(got, f)[:, :C0], getattr(cb, f))
    assert got.cand_article[:, C0:].tolist() == ids
    assert got.cand_time[:, C0:].tolist() == times
    assert got.label[:, C0:].tolist() == labels
    assert torch.equal(got.empty_num, cb.empty_num + torch.tensor([r.count(0) for r in ids], device='cuda'))
    return ids


@pytest.mark.parametrize('B, H, C0, k, n, weighted', [
    (1, 50, 5, 4, 2000, False),
    (37, 256, 7, 64, 400, True),           # H + C0 + k close to the pool: exclusions and exhausted budgets
    (8, 20, 3, 1, 5000, True),
    (1024, 200, 5, 16, 5000, False),
    (1024, 32, 5, 64, 100_000, True),
])
def test_sample_equals_the_reference(B, H, C0, k, n, weighted):
    table = _table(n)
    g = torch.Generator().manual_seed(B * k)
    weights = torch.randint(0, 5, (n - 1,), generator=g) if weighted else None
    s = negatives.NegativeSampler(table, k=k, seed=0x9E3779B97F4A7C15 + B, weights=weights)
    cb = _batch(table, B, H, C0, seed=B + H, no_positive_every=5)
    ids = _check_against_reference(s, cb, step=3 + k, row_offset=B, weights=None if weights is None else weights.tolist())
    assert any(i != 0 for r in ids for i in r)


def test_small_pool_exhausts_the_attempt_budget():
    table = _table(3000)
    pool = torch.arange(1, 11, dtype=torch.int32)
    cb = _batch(table, 64, 30, 5, seed=4)
    cb.hist_article[:, :3] = torch.arange(1, 4, dtype=torch.int32, device='cuda')       # three pool ids in every history
    for weights in (None, torch.tensor([1000] + [1] * 9)):
        s = negatives.NegativeSampler(table, k=12, seed=5, pool_article=pool, weights=weights)
        ids = _check_against_reference(s, cb, step=0, row_offset=0, weights=None if weights is None else weights.tolist())
        assert all(r.count(0) >= 5 for r in ids)            # at most 10 - 3 ids per impression


def test_invariants_and_distributions_at_scale():
    B, H, C0, k, n = 4096, 50, 5, 16, 50_001
    table = _table(n)
    cb = _batch(table, B, H, C0, seed=8)
    uni = negatives.NegativeSampler(table, k=k, seed=1)
    w = torch.arange(1, n, dtype=torch.int64) % 4                                          # weights 0, 1, 2, 3 by id
    wei = negatives.NegativeSampler(table, k=k, seed=1, weights=w)
    for s in (uni, wei):
        neg = s.sample(cb, step=7).cand_article[:, C0:]
        assert bool((neg > 0).all())                                                         # a big pool never runs out
        assert bool(((neg >= 1) & (neg < n)).all())
        assert not bool((neg[:, :, None] == cb.hist_article[:, None, :]).any())
        assert not bool((neg[:, :, None] == cb.cand_article[:, None, :]).any())
        srt = neg.sort(1).values
        assert bool((srt[:, 1:] != srt[:, :-1]).all())
        counts = torch.bincount(neg.reshape(-1).long(), minlength=n).cpu()
        if s is uni:
            binned = counts[1:].reshape(100, 500).sum(1).double().numpy()
            p = chisquare(binned).pvalue
        else:
            assert int(counts[1:][w == 0].sum()) == 0
            by_w = np.array([int(counts[1:][w == c].sum()) for c in (1, 2, 3)], dtype=np.float64)
            expect = np.array([int(w[w == c].sum()) for c in (1, 2, 3)], dtype=np.float64)
            p = chisquare(by_w, expect / expect.sum() * by_w.sum()).pvalue
        assert p > 1e-3, p


def _model(precision):
    m = nrm.UserModel(100)
    m.load_state_dict(load_weights('train'), strict=False)
    return m.to('cuda').train().set_precision(precision)


def _state(m, tr):
    return [m.flat_parameters().buf.clone(), m.bn.running_mean.clone(), m.bn.running_var.clone(), m.bn.num_batches_tracked.clone(),
            tr.exp_avg.clone(), tr.exp_avg_sq.clone()]


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


B, H, C0, K = 64, 50, 5, 4


def _setup(n_batches, ragged=None):
    table = wire.make_article_table(3000, seed=5).to('cuda')
    cbs = [wire.make_compact_batch(table, B, H, C0, seed=80 + i, user_num=100, variable_history=True).to('cuda') for i in range(n_batches)]
    if ragged:
        cbs[-1] = wire.CompactBatch(*[getattr(cbs[-1], f)[:ragged] for f in cbs[-1].__dataclass_fields__])
    return table, cbs, negatives.NegativeSampler(table, k=K, seed=12345)


@pytest.mark.parametrize('use_graph', [True, False])
@pytest.mark.parametrize('precision', ['bf16x3', 'fp32'])
def test_fused_step_samples_as_the_standalone_sampler(precision, use_graph):
    """Three steps, the last a ragged 37 impressions: with negatives= against the step without it fed sampler.sample(cb_i, step=i)."""
    table, cbs, s = _setup(3, ragged=37)
    runs = []
    for sampled in (True, False):
        m = _model(precision)
        tr = nrm.FusedTrainStep(m, B, H, C0 + K, lr=1e-3, weight_decay=1e-5, articles=table, negatives=s if sampled else None,
                                use_graph=use_graph)
        losses = [tr.step(cb if sampled else s.sample(cb, step=i)).item() for i, cb in enumerate(cbs)]
        torch.cuda.synchronize()
        runs.append((losses, _state(m, tr)))
    (l0, s0), (l1, s1) = runs
    assert l0 == l1 and _same(s0, s1)


def test_fused_step_refuses_packed_batches_and_other_widths():
    table, cbs, s = _setup(1)
    tr = nrm.FusedTrainStep(_model('bf16x3'), B, H, C0 + K, articles=table, negatives=s)
    with pytest.raises(ValueError, match='CompactBatches only'):
        tr.load(wire.expand(table, cbs[0]))
    with pytest.raises(ValueError, match='does not fit'):
        tr.load(s.sample(cbs[0]))
    with pytest.raises(ValueError, match='needs articles'):
        nrm.FusedTrainStep(_model('bf16x3'), B, H, C0 + K, negatives=s)


def test_graph_replays_draw_afresh_and_runs_repeat_bit_for_bit():
    table, cbs, s = _setup(1)
    runs = []
    for _ in range(2):
        tr = nrm.FusedTrainStep(_model('bf16x3'), B, H, C0 + K, articles=table, negatives=s, nslots=1)
        drawn = []
        for i in range(3):                               # one slot: every step replays the same graph
            tr.step(cbs[0]).item()
            drawn.append(tr.slots[0].compact.cand_article.clone())
            assert torch.equal(drawn[-1], s.sample(cbs[0], step=i).cand_article)
        assert not torch.equal(drawn[0], drawn[1]) and not torch.equal(drawn[1], drawn[2])
        runs.append(_state(tr.model, tr) + drawn)
    assert _same(runs[0], runs[1])


def test_resume_from_state_dict_draws_what_the_uninterrupted_run_draws():
    table, cbs, s = _setup(4)
    a = _model('bf16x3')
    ta = nrm.FusedTrainStep(a, B, H, C0 + K, articles=table, negatives=s)
    for cb in cbs[:2]:
        ta.step(cb)
    sd_model = {k: v.detach().clone() for k, v in a.state_dict().items()}
    sd_opt = ta.state_dict()
    la = [ta.step(cb) for cb in cbs[2:]]
    b = nrm.UserModel(100)
    b.load_state_dict(sd_model)
    b.to('cuda').train().set_precision('bf16x3')
    tb = nrm.FusedTrainStep(b, B, H, C0 + K, articles=table, negatives=s)
    tb.load_state_dict(sd_opt)
    lb = [tb.step(cb) for cb in cbs[2:]]
    assert [h.item() for h in la] == [h.item() for h in lb]
    torch.cuda.synchronize()
    assert _same(_state(a, ta), _state(b, tb))


class _OneProcessDP:
    """Single-process stand-in for `dp.DataParallel(sync_bn=True)` as rank `rank`: no peer memory, one rank's statistics."""
    sync_bn = True
    world = 1

    def __init__(self, rank):
        self.rank = rank

    class buckets:
        @staticmethod
        def reduce(grads, begin, end):
            pass

        @staticmethod
        def wait():
            pass

    def peer_context(self, *args, **kwargs):
        return None

    def all_reduce_stats(self, sums, local_rows):
        return local_rows


def test_data_parallel_rank_draws_with_its_row_offset():
    table, cbs, s = _setup(2)
    m = _model('bf16x3')
    m._dp = _OneProcessDP(rank=3)
    tr = nrm.FusedTrainStep(m, B, H, C0 + K, articles=table, negatives=s)
    for i, cb in enumerate(cbs):
        tr.step(cb).item()
        assert torch.equal(tr.slots[i].compact.cand_article, s.sample(cb, step=i, row_offset=3 * B).cand_article)
