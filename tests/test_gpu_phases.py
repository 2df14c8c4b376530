"""The whole training-step entry points against their phases.

`nrm_forward[_compact]` is `nrm_forward_encoder[_compact]` + `nrm_forward_head`, `nrm_backward[_compact]` is
`nrm_backward_head[_deferred]` + `nrm_backward_encoder[_compact]`, and an eval `nrm_forward_scores[_compact]` is an eval
`nrm_forward[_compact]` that also writes the attention scores.  Synchronised BatchNorm runs the split calls; a single-process
stand-in for `DataParallel` reaches that branch of `FusedTrainStep` on one GPU, where it must train as the whole calls do."""
import ctypes

import pytest
import torch

import news_recommendation_model_b200 as nrm
from news_recommendation_model_b200 import _lib, wire
from fixtures import load_weights

pytestmark = pytest.mark.gpu

H, C = 50, 5
MODE_TRAIN = 3                 # NRM_MODE_BN_BATCH_STATS | NRM_MODE_KEEP_FOR_BWD
CASES = [(fmt, precision, B) for fmt in ('packed', 'compact') for precision in ('fp32', 'bf16', 'bf16x3') for B in (1, 33)]


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _model(precision):
    m = nrm.UserModel(100)
    m.load_state_dict(load_weights('train'), strict=False)
    return m.to('cuda').train().set_precision(precision)


class _Case:
    """One batch in one wire format: `args` are the leading arguments of the entry points, `sfx` the suffix of their names."""

    def __init__(self, fmt, precision, B):
        self.lib, self.B = _lib.load(), B
        self.model = _model(precision)
        self.flat = self.model.flat_parameters()
        self.precision = self.model._precision_code()
        self.table = wire.make_article_table(2000, seed=5).to('cuda')
        self.cb = wire.make_compact_batch(self.table, B, H, C, seed=40 + B, user_num=100, variable_history=True).to('cuda')
        if fmt == 'packed':
            d = wire.expand(self.table, self.cb)
            self.keep = (d.x_history, d.x_target, d.x_global)
            self.args = (_p(d.x_history), _p(d.x_target), C * 78, _p(d.x_global), C * 3)
            self.sfx = ''
        else:
            cb = self.cb
            self.keep = _lib.CompactBatchStruct(self.table.rows.data_ptr(), self.table.n, cb.hist_article.data_ptr(), cb.hist_time.data_ptr(),
                                                cb.hist_click.data_ptr(), cb.cand_article.data_ptr(), cb.cand_time.data_ptr(), None, None)
            self.args = (ctypes.byref(self.keep),)
            self.sfx = '_compact'
        g = torch.Generator(device='cuda').manual_seed(B)
        self.dlogits = torch.randn(B, C, device='cuda', generator=g)

    def call(self, name, *rest):
        fn = getattr(self.lib, name)
        rc = fn(*rest)
        assert rc == 0, (name, self.lib.nrm_last_error())

    def state(self, mode):
        """Fresh BatchNorm buffers, logits and workspace."""
        bn = self.model.bn
        ws = torch.empty(int(self.lib.nrm_workspace_bytes(self.B, H, C, mode)), dtype=torch.uint8, device='cuda')
        return (bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone(),
                torch.empty(self.B, C, device='cuda'), ws)

    def forward(self, split, mode=MODE_TRAIN):
        mean, var, nbt, logits, ws = st = self.state(mode)
        B, f, prec = self.B, self.flat, self.precision
        n0 = self.lib.nrm_launch_count()
        if split:
            sums = torch.full((528,), float('nan'), dtype=torch.float64, device='cuda')
            self.call('nrm_forward_encoder' + self.sfx, *self.args, B, H, C, _p(f.buf), mode, prec, _p(sums), _p(ws), ws.numel(), None)
            self.call('nrm_forward_head', B, H, C, _p(f.buf), _p(mean), _p(var), _p(nbt), mode, prec, _p(sums), B * C, _p(logits), _p(ws),
                      ws.numel(), None)
        else:
            self.call('nrm_forward' + self.sfx, *self.args, B, H, C, _p(f.buf), _p(mean), _p(var), _p(nbt), mode, prec, _p(logits), _p(ws),
                      ws.numel(), None)
        return st, self.lib.nrm_launch_count() - n0

    def backward(self, head, ws):
        """head: None (nrm_backward[_compact]) or the head entry point of the split pair."""
        B, f, prec = self.B, self.flat, self.precision
        grads = torch.zeros(f.total, device='cuda')
        n0 = self.lib.nrm_launch_count()
        if head is None:
            self.call('nrm_backward' + self.sfx, *self.args, B, H, C, _p(f.buf), MODE_TRAIN, prec, _p(self.dlogits), _p(grads), _p(ws),
                      ws.numel(), None)
        else:
            sums = torch.full((528,), float('nan'), dtype=torch.float64, device='cuda')
            self.call(head, B, H, C, _p(f.buf), prec, _p(self.dlogits), _p(grads), _p(sums), _p(ws), ws.numel(), None)
            self.call('nrm_backward_encoder' + self.sfx, *self.args, B, H, C, _p(f.buf), MODE_TRAIN, prec, _p(sums), B * C, _p(grads), _p(ws),
                      ws.numel(), None)
        return grads, self.lib.nrm_launch_count() - n0


def _equal(a, b):
    """Bit for bit (NaN payloads and the sign of zero included)."""
    if a.dtype.is_floating_point:
        a, b = (t.view(torch.int32 if t.element_size() == 4 else torch.int64) for t in (a, b))
    return a.dtype == b.dtype and torch.equal(a, b)


@pytest.mark.parametrize('fmt,precision,B', CASES)
def test_forward_equals_encoder_then_head(fmt, precision, B):
    case = _Case(fmt, precision, B)
    whole, n_whole = case.forward(split=False)
    split, n_split = case.forward(split=True)
    torch.cuda.synchronize()
    for a, b in zip(whole[:4], split[:4]):                      # running mean, running var, num_batches_tracked, logits
        assert _equal(a, b)
    assert int(whole[2]) == int(case.model.bn.num_batches_tracked) + 1
    assert n_whole == n_split > 0


@pytest.mark.parametrize('fmt,precision,B', CASES)
def test_backward_equals_head_then_encoder(fmt, precision, B):
    case = _Case(fmt, precision, B)
    results = []
    for head in (None, 'nrm_backward_head_deferred', 'nrm_backward_head'):
        st, _ = case.forward(split=False)
        results.append(case.backward(head, st[4]))
    torch.cuda.synchronize()
    (g_whole, n_whole), (g_deferred, n_deferred), (g_head, n_head) = results
    assert g_whole.abs().sum() > 0
    assert _equal(g_whole, g_deferred) and _equal(g_whole, g_head)
    assert n_whole == n_deferred == n_head > 0


@pytest.mark.parametrize('fmt,precision,B', CASES)
def test_eval_scores_forward_has_the_eval_forward_logits(fmt, precision, B):
    case = _Case(fmt, precision, B)
    (_, _, _, logits, _), _ = case.forward(split=False, mode=0)
    mean, var, nbt, logits_s, ws = case.state(0)
    scores = torch.full((2, B, C, H), float('nan'), device='cuda')
    case.call('nrm_forward_scores' + case.sfx, *case.args, B, H, C, _p(case.flat.buf), _p(mean), _p(var), _p(nbt), 0, case.precision,
              _p(logits_s), _p(scores), _p(ws), ws.numel(), None)
    torch.cuda.synchronize()
    assert _equal(logits, logits_s)


class _OneProcessDP:
    """Single-process stand-in for `dp.DataParallel(sync_bn=True)`: no peer memory, statistics and gradients of one rank."""
    sync_bn = True
    world = 1

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


@pytest.fixture
def one_process_dp():
    return _OneProcessDP()


@pytest.mark.parametrize('precision', ['fp32', 'bf16x3'])
@pytest.mark.parametrize('fmt', ['packed', 'compact'])
def test_fused_train_step_split_branch_trains_as_the_whole_calls(fmt, precision, one_process_dp):
    B = 33
    table = wire.make_article_table(2000, seed=5).to('cuda')
    batches = [wire.make_compact_batch(table, B, H, C, seed=60 + i, user_num=100).to('cuda') for i in range(3)]
    if fmt == 'packed':
        batches = [wire.expand(table, cb) for cb in batches]
    runs = []
    for dp in (None, one_process_dp):
        m = _model(precision)
        m._dp = dp
        tr = nrm.FusedTrainStep(m, B, H, C, lr=1e-3, weight_decay=1e-5, articles=table)
        assert tr.use_graph == (dp is None)                     # the split branch runs eagerly, the whole calls in a graph
        losses = [tr.step(b).item() for b in batches]
        torch.cuda.synchronize()
        runs.append((losses, m.flat_parameters().buf.clone(), m.bn.running_mean.clone(), m.bn.running_var.clone(),
                     m.bn.num_batches_tracked.clone(), tr.exp_avg.clone(), tr.exp_avg_sq.clone()))
    (l0, *t0), (l1, *t1) = runs
    assert l0 == l1
    for a, b in zip(t0, t1):
        assert _equal(a, b)
