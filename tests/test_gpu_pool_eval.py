"""Pool evaluation (nrm_pool_rank) through news_recommendation_model_b200.recommend: rank_targets against its float64 host
restatement (tests/pool_eval_ref.py) on edge cases, its agreement with the recommender's own selection (nrm_pool_topk), evaluate
in every precision, run-to-run identity and the C entry point's argument errors."""
import ctypes

import numpy as np
import pytest
import torch

import parity as P
from fixtures import load_weights
from pool_eval_ref import edge_case, host_pool_metrics, host_rank_targets
from news_recommendation_model_b200 import NrmError, _lib, recommend, wire

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp32', 'bf16', 'bf16x3']
N_ARTICLES = 3000
COUNTS = ('rank', 'greater', 'equal')


def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() if a is not None else None for a in arrays]


def _check_exact(got, ref, ks=(1, 5, 100)):
    for name in ('position',) + COUNTS:
        assert torch.equal(getattr(got, name).cpu(), torch.from_numpy(ref[name])), name
    assert torch.equal(got.n_eligible.cpu(), torch.from_numpy(ref['n_eligible']))
    assert np.array_equal(got.score.cpu().double().numpy(), ref['score'], equal_nan=True)
    m, mref = recommend.pool_metrics(got, ks), host_pool_metrics(ref, ks)
    for name, v in m.items():
        assert v.device == got.rank.device
        assert np.allclose(v.cpu().double().numpy(), mref[name], rtol=0, atol=1e-6, equal_nan=True), name


def _check_close(got, ref):
    """M >= 2: the fp32 softmax mean differs from the float64 score in the last bits; each count may differ from the host's only
    by positions whose host score is within 1e-6 relative of the target's."""
    assert torch.equal(got.position.cpu(), torch.from_numpy(ref['position']))
    assert torch.equal(got.n_eligible.cpu(), torch.from_numpy(ref['n_eligible']))
    s = ref['scores']
    score = got.score.cpu().double().numpy()
    for b, p in zip(*np.nonzero(ref['position'] >= 0)):
        v = ref['score'][b, p]
        assert abs(score[b, p] - v) <= 1e-6 * abs(v), (b, p)
        near = int(np.sum(np.abs(s[b] - v) <= 1e-6 * abs(v))) - 1            # nan rows compare False
        for name in COUNTS:
            assert abs(int(getattr(got, name)[b, p]) - int(ref[name][b, p])) <= near, (name, b, p)


@pytest.mark.parametrize('M', [1, 2])
@pytest.mark.parametrize('exclude', [True, False])
@pytest.mark.parametrize('shape', [dict(), dict(N=8), dict(B=1), dict(N=200, P=40)], ids=str)
def test_rank_targets_against_the_host_restatement(M, exclude, shape):
    logits, pool, hist, targets, n_articles = edge_case(M, 10 + M, **shape)
    x, pa, ha, tg = _cuda(logits, pool, hist if exclude else None, targets)
    got = recommend.rank_targets(x if M > 1 else x[0], tg, pa, n_articles, hist_article=ha)
    ref = host_rank_targets(logits, targets, pool, n_articles, hist if exclude else None)
    assert got.rank.dtype == torch.int64 and got.score.dtype == torch.float32 and got.n_eligible.shape == (targets.shape[0],)
    if M == 1:
        _check_exact(got, ref)
    else:
        _check_close(got, ref)


@pytest.mark.parametrize('M', [1, 2])
@pytest.mark.parametrize('exclude', [True, False])
def test_ranks_agree_with_the_recommender(M, exclude):
    """A rankable target is in select(k) iff rank < k, and at index rank; quantised logits force ties."""
    rng = np.random.default_rng(M * 2 + exclude)
    B, N, Pn = 8, 2000, 64
    logits = (np.round(rng.normal(size=(M, B, N)) * 8) / 8).astype(np.float32)
    logits[:, 0, ::13] = 0.5
    pool = rng.permutation(np.arange(1, N_ARTICLES))[:N].astype(np.int32)
    pool[::211] = 0
    hist = rng.choice(pool, (B, 40)).astype(np.int32)
    targets = np.where(rng.random((B, Pn)) < 0.9, rng.choice(pool, (B, Pn)), rng.integers(0, N_ARTICLES, (B, Pn))).astype(np.int32)
    targets[:, :5] = hist[:, :5]
    x, pa, ha, tg = _cuda(logits, pool, hist if exclude else None, targets)
    r = recommend.rank_targets(x, tg, pa, N_ARTICLES, hist_article=ha)
    assert (r.rank >= 0).sum() > B * Pn // 2
    pos_r, rank_r = r.position.cpu().numpy(), r.rank.cpu().numpy()
    for k in (1, 10, 100, 1024):
        sel = recommend.select(x, k, pa, N_ARTICLES, hist_article=ha).position.cpu().numpy()
        for b in range(B):
            rankable = set(pos_r[b][pos_r[b] >= 0].tolist())
            in_sel = {int(n): i for i, n in enumerate(sel[b]) if n in rankable}
            assert in_sel == {int(n): int(q) for n, q in zip(pos_r[b], rank_r[b]) if 0 <= q < k}, (k, b)


def _model(precision, weights='train'):
    model, _ = P.build_models(load_weights(weights), 40)
    return model.set_precision(precision)


_TABLES = {}


def _table(n=N_ARTICLES):
    if n not in _TABLES:
        _TABLES[n] = wire.make_article_table(n - 1, seed=5).to('cuda')
    return _TABLES[n]


def _users_pool_targets(B, H, N, Pn, seed, n=N_ARTICLES):
    """Users, a pool of N distinct ids of the n-article table, and targets: pool ids, pads, an out-of-range id, clicked ids."""
    cb = wire.make_compact_batch(_table(n), B, H, 1, seed=seed, user_num=40, variable_history=True).to('cuda')
    rng = np.random.default_rng(seed)
    pool = rng.permutation(np.arange(1, n))[:N].astype(np.int32)
    pt = torch.full((N,), int(wire.pack_time(np.array([1, 6, 17, 9])).view(np.int32)), dtype=torch.int32, device='cuda')
    targets = rng.choice(np.concatenate([pool, [0, 0, n + 1]]), (B, Pn)).astype(np.int32)
    targets[:, :3] = cb.hist_article[:, :3].cpu().numpy()                  # clicked
    pa, tg = _cuda(pool, targets)
    return cb.hist_article, cb.hist_time, cb.hist_click, pt, pa, tg


@pytest.mark.parametrize('precision', PRECISIONS)
def test_evaluate_against_pool_logits_and_the_host(precision):
    model = _model(precision)
    ha, ht, hc, pt, pa, tg = _users_pool_targets(7, 50, 300, 24, seed=3)
    ks = (1, 10, 50)
    for exclude in (True, False):
        m, r = recommend.evaluate(model, _table(), ha, ht, hc, pt, tg, ks=ks, pool_article=pa, exclude_clicked=exclude, chunk=64)
        logits = recommend.pool_logits(model, _table(), ha, ht, hc, pt, pool_article=pa)
        ref = host_rank_targets(logits.cpu().numpy(), tg.cpu().numpy(), pa.cpu().numpy(), N_ARTICLES,
                                ha.cpu().numpy() if exclude else None)
        _check_exact(r, ref, ks)
        assert set(m) == set(recommend.pool_metrics(r, ks))
    # an ensemble: evaluate is rank_targets on the stacked pool logits, bit for bit
    models = [model, _model(precision, 'validation')]
    m, r = recommend.evaluate(models, _table(), ha, ht, hc, pt, tg, ks=ks, pool_article=pa)
    x = torch.stack([recommend.pool_logits(mm, _table(), ha, ht, hc, pt, pool_article=pa) for mm in models])
    r2 = recommend.rank_targets(x, tg, pa, N_ARTICLES, hist_article=ha)
    for a, b in zip(r, r2):
        assert torch.equal(a, b) or torch.equal(torch.nan_to_num(a, 7.0), torch.nan_to_num(b, 7.0))
    _check_close(r, host_rank_targets(x.cpu().numpy(), tg.cpu().numpy(), pa.cpu().numpy(), N_ARTICLES, ha.cpu().numpy()))


def test_evaluate_at_scale():
    model, n = _model('bf16x3'), 25000
    ha, ht, hc, pt, pa, tg = _users_pool_targets(64, 200, 20000, 1024, seed=4, n=n)
    m, r = recommend.evaluate(model, _table(n), ha, ht, hc, pt, tg, ks=(10, 100, 1000), pool_article=pa)
    logits = recommend.pool_logits(model, _table(n), ha, ht, hc, pt, pool_article=pa)
    ref = host_rank_targets(logits.cpu().numpy(), tg.cpu().numpy(), pa.cpu().numpy(), n, ha.cpu().numpy())
    _check_exact(r, ref, (10, 100, 1000))
    assert (r.rank >= 1024).any()                                           # ranks beyond what top_articles can return


def test_two_calls_are_bit_identical():
    logits, pool, hist, targets, n_articles = edge_case(2, 21, B=16, N=3000, P=1024, n_articles=2500)
    x, pa, ha, tg = _cuda(logits, pool, hist, targets)
    a = recommend.rank_targets(x, tg, pa, n_articles, hist_article=ha)
    b = recommend.rank_targets(x, tg, pa, n_articles, hist_article=ha)
    for u, v in zip(a, b):
        assert torch.equal(u.view(torch.int32) if u.dtype == torch.float32 else u, v.view(torch.int32) if v.dtype == torch.float32 else v)


def test_bad_arguments_return_einval():
    lib = _lib.load()
    B, N = 2, 100
    x = torch.zeros(17, B, N, device='cuda')
    pa = torch.arange(1, N + 1, dtype=torch.int32, device='cuda')
    tg = torch.ones(B, 1025, dtype=torch.int32, device='cuda')
    outs = [torch.empty(B, 1025, dtype=torch.int32, device='cuda') for _ in range(4)]
    score = torch.empty(B, 1025, device='cuda')
    ne = torch.empty(B, dtype=torch.int32, device='cuda')
    p = lambda t: ctypes.c_void_p(t.data_ptr())

    def call(M, Pn):
        return lib.nrm_pool_rank(p(x), M, B * N, B, N, p(pa), N_ARTICLES, None, 0, p(tg), Pn, *(p(o) for o in outs), p(score), p(ne), None)
    assert call(1, 0) == -1
    assert call(1, 1025) == -1 and b'1024' in lib.nrm_last_error()
    assert call(17, 4) == -1 and b'16' in lib.nrm_last_error()
    assert call(16, 1024) == 0
    torch.cuda.synchronize()
    with pytest.raises(NrmError):
        recommend.rank_targets(x[0].cpu(), tg[:, :4].cpu(), pa.cpu(), N_ARTICLES)          # valid arguments, CPU tensors
