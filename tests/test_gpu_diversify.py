"""Pool diversification (nrm_pool_diversify) through news_recommendation_model_b200.recommend: bit identity with select at lam = 1,
exact agreement with the float64 host greedy (tests/diversify_ref.py) where every value is exactly representable, a step-by-step
replay of random inputs in float64, diverse_articles in every precision, run-to-run identity, a large case and the C entry
point's argument errors."""
import ctypes

import numpy as np
import pytest
import torch

import parity as P
from diversify_ref import exact_rows, greedy, relevance, unit_vectors
from fixtures import load_weights
from news_recommendation_model_b200 import NrmError, _lib, recommend, wire

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp32', 'bf16', 'bf16x3']
N_ARTICLES = 3000
# Replay tolerance: a pick's float64 gain may fall short of the best float64 gain by the float32 rounding of rel, the unit vectors
# and the 64-term dot products (each about 1e-7 relative).  On a B200 the largest shortfall over these tests was 0: every float32
# pick was also the float64 argmax.  1e-5 allows for near-ties that float32 breaks the other way.
REPLAY_TOL = 1e-5


def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() if a is not None else None for a in arrays]


def _random_case(seed, B, N, M=1, n_articles=N_ARTICLES, n_categories=6):
    """Logits with ties and NaN, a pool with pads, out-of-range and repeated ids, histories, and a table with all-zero vectors
    and a handful of categories (so that caps bind)."""
    rng = np.random.default_rng(seed)
    logits = (np.round(rng.normal(size=(M, B, N)) * 8) / 8).astype(np.float32)
    logits[:, :, ::17] = np.nan
    pool = rng.integers(1, n_articles, N).astype(np.int32)
    pool[::31] = 0
    pool[5::37] = n_articles + 4
    hist = rng.choice(pool, (B, 30)).astype(np.int32)
    rows = rng.normal(size=(n_articles, 80)).astype(np.float32)
    rows[::11, :64] = 0.0
    rows[:, 64] = rng.integers(0, n_categories, n_articles)
    return logits, pool, hist, rows


def _table(rows):
    return wire.ArticleTable(torch.from_numpy(rows).cuda())


def _same(a, b):
    """torch.equal for int tensors, bit equality for float tensors (NaN == NaN)."""
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b)


@pytest.mark.parametrize('M', [1, 2])
@pytest.mark.parametrize('exclude', [True, False])
def test_lambda_one_without_cap_is_select(M, exclude):
    logits, pool, hist, rows = _random_case(10 + M, 6, 1500, M)
    x, pa, ha = _cuda(logits, pool, hist if exclude else None)
    xx = x if M > 1 else x[0]
    table = _table(rows)
    for k in (1, 10, 100, 512):
        sel = recommend.select(xx, k, pa, N_ARTICLES, hist_article=ha)
        d = recommend.diversify(xx, k, pa, table, lam=1.0, hist_article=ha)
        assert d.position.dtype == torch.int64 and d.gain.dtype == torch.float32 and d.gain.shape == (6, k)
        assert torch.equal(d.position, sel.position) and torch.equal(d.article, sel.article) and _same(d.score, sel.score), k
    # k = K' = 512 with fewer eligible positions than that
    small = logits[:, :, :520]
    x, pa = _cuda(small, pool[:520])
    sel = recommend.select(x, 512, pa, N_ARTICLES, hist_article=ha)
    d = recommend.diversify(x, 512, pa, table, lam=1.0, candidates=512, hist_article=ha)
    assert (sel.position < 0).any()
    assert torch.equal(d.position, sel.position) and _same(d.score, sel.score)
    assert torch.equal(torch.isnan(d.gain), d.position < 0)


def test_lambda_one_with_a_cap_is_the_host_greedy():
    logits, pool, hist, rows = _random_case(3, 8, 2000)
    x, pa, ha = _cuda(logits[0], pool, hist)
    table = _table(rows)
    cand = recommend.select(x, 256, pa, N_ARTICLES, hist_article=ha)
    for q in (1, 3, 20):
        d = recommend.diversify(x, 60, pa, table, lam=1.0, candidates=256, max_per_category=q, hist_article=ha)
        ref = greedy(cand.position.cpu().numpy(), cand.score.cpu().numpy(), pool, rows, N_ARTICLES, 60, 1.0, q)
        assert np.array_equal(d.position.cpu().numpy(), ref['position']), q
        assert np.array_equal(d.score.cpu().double().numpy(), ref['score'], equal_nan=True), q
        assert np.allclose(d.gain.cpu().double().numpy(), ref['gain'], rtol=0, atol=1e-6, equal_nan=True), q
        if q == 1:
            assert (d.position[:, 6:] == -1).all()                             # 6 categories


@pytest.mark.parametrize('scale', [1.0, 2.0 ** 127], ids=['unit', 'near_flt_max'])
def test_exactly_representable_inputs_match_the_host(scale):
    """Unit vectors of four +-0.5 entries and scores on a grid whose range is a power of two: every rel, similarity and gain is
    exact in float32, so the GPU must reproduce the float64 greedy exactly, ties included.  scale 2^127: scores +-2^127, +-2^126
    and 0, whose range overflows float32."""
    rng = np.random.default_rng(4)
    B, N, n = 8, 300, 400
    rows = exact_rows(n, 4, rng)
    pool = rng.integers(1, n, N).astype(np.int32)
    grid = rng.integers(0, 9, (1, B, N)) / 8.0 if scale == 1.0 else (rng.integers(0, 5, (1, B, N)) - 2) / 2.0
    grid[0, :, 0], grid[0, :, 1] = grid.min(), grid.max()
    logits = (grid * scale).astype(np.float32)
    logits[0, :, 7::23] = np.nan
    x, pa = _cuda(logits[0], pool)
    table = _table(rows)
    for lam in (0.0, 0.25, 0.5, 0.75, 1.0):
        for q in (0, 1, 3):
            d = recommend.diversify(x, 40, pa, table, lam=lam, max_per_category=q)
            cand = recommend.select(x, N, pa, n)
            ref = greedy(cand.position.cpu().numpy(), cand.score.cpu().numpy(), pool, rows, n, 40, lam, q)
            assert np.array_equal(d.position.cpu().numpy(), ref['position']), (lam, q)
            assert np.array_equal(d.score.cpu().double().numpy(), ref['score'], equal_nan=True), (lam, q)
            assert np.array_equal(d.gain.cpu().double().numpy(), ref['gain'], equal_nan=True), (lam, q)


def _replay(cand_pos, cand_score, pool, rows, n_articles, got_pos, got_gain, lam, q):
    """Recompute every step's gains in float64 given the GPU's earlier picks; -> the largest shortfall of a pick's gain below the
    step's best gain.  Asserts that picks are distinct candidates that respect the cap, and that the GPU stops only when nothing
    can be picked."""
    u = unit_vectors(rows)
    cats = np.trunc(rows[:, 64]).astype(np.int64)
    worst = 0.0
    for b in range(cand_pos.shape[0]):
        pos = cand_pos[b]
        ok = pos >= 0
        ids = np.where(ok, pool[np.maximum(pos, 0)], 0)
        rel = np.where(ok, relevance(np.where(ok, cand_score[b].astype(np.float64), np.nan)), 0.0)
        U, cat = u[ids], cats[ids]
        index = {int(p): i for i, p in enumerate(pos) if p >= 0}
        m, live, count = np.zeros(pos.size), ok.copy(), {}
        for t in range(got_pos.shape[1]):
            p = int(got_pos[b, t])
            if p < 0:
                assert not live.any() and (got_pos[b, t:] == -1).all(), (b, t)
                break
            i = index[p]
            assert live[i], (b, t)
            gain = lam * rel - (1.0 - lam) * m
            worst = max(worst, float(gain[live].max() - gain[i]))
            assert abs(float(got_gain[b, t]) - gain[i]) <= REPLAY_TOL, (b, t)
            live[i] = False
            sim = (U * U[i]).sum(1)
            m = sim if t == 0 else np.maximum(m, sim)
            count[cat[i]] = count.get(cat[i], 0) + 1
            if q > 0 and count[cat[i]] >= q:
                live &= cat != cat[i]
    return worst


@pytest.mark.parametrize('lam', [0.0, 0.3, 0.7, 0.9])
@pytest.mark.parametrize('q', [0, 2])
def test_random_inputs_replay_in_float64(lam, q):
    logits, pool, hist, rows = _random_case(5, 16, 4000, M=2)
    logits = np.random.default_rng(6).normal(size=logits.shape).astype(np.float32)     # no ties: a clean replay
    x, pa, ha = _cuda(logits, pool, hist)
    table = _table(rows)
    d = recommend.diversify(x, 50, pa, table, lam=lam, candidates=200, max_per_category=q, hist_article=ha)
    cand = recommend.select(x, 200, pa, N_ARTICLES, hist_article=ha)
    worst = _replay(cand.position.cpu().numpy(), cand.score.cpu().numpy(), pool, rows, N_ARTICLES, d.position.cpu().numpy(),
                    d.gain.cpu().numpy(), lam, q)
    print(f'replay lam={lam} q={q}: largest shortfall {worst:.3g}')
    assert worst <= REPLAY_TOL


def _model(precision, weights='train'):
    model, _ = P.build_models(load_weights(weights), 40)
    return model.set_precision(precision)


@pytest.mark.parametrize('precision', PRECISIONS)
def test_diverse_articles_is_diversify_of_pool_logits(precision):
    table = wire.make_article_table(N_ARTICLES - 1, seed=5).to('cuda')
    table.rows[:, 64] = torch.arange(table.n, device='cuda') % 5                  # a handful of categories: the cap binds
    cb = wire.make_compact_batch(table, 6, 50, 1, seed=3, user_num=40, variable_history=True).to('cuda')
    rng = np.random.default_rng(3)
    pa = torch.from_numpy(rng.integers(0, N_ARTICLES, 700).astype(np.int32)).cuda()
    pt = torch.full((700,), int(wire.pack_time(np.array([1, 6, 17, 9])).view(np.int32)), dtype=torch.int32, device='cuda')
    models = [_model(precision), _model(precision, 'validation')]
    for ms in (models[0], models):
        for exclude in (True, False):
            got = recommend.diverse_articles(ms, table, cb.hist_article, cb.hist_time, cb.hist_click, pt, 20, lam=0.6, candidates=300,
                                             max_per_category=3, pool_article=pa, exclude_clicked=exclude, chunk=64)
            ml = ms if isinstance(ms, list) else [ms]
            x = torch.stack([recommend.pool_logits(m, table, cb.hist_article, cb.hist_time, cb.hist_click, pt, pool_article=pa) for m in ml])
            ref = recommend.diversify(x, 20, pa, table, lam=0.6, candidates=300, max_per_category=3,
                                      hist_article=cb.hist_article if exclude else None)
            for a, b in zip(got, ref):
                assert _same(a, b)
            assert (got.position >= 0).sum(1).max() == 15                         # 5 categories x 3
    ild, ncat = recommend.list_diversity(table, got.article)
    top = recommend.top_articles(models, table, cb.hist_article, cb.hist_time, cb.hist_click, pt, 20, pool_article=pa, exclude_clicked=False)
    ild0, ncat0 = recommend.list_diversity(table, top.article)
    assert ild.device == got.article.device and ncat.dtype == torch.int64 and (ncat == 5).all() and (ncat0 <= 5).all()


def test_two_calls_are_bit_identical():
    logits, pool, hist, rows = _random_case(7, 64, 5000, M=2)
    x, pa, ha = _cuda(logits, pool, hist)
    table = _table(rows)
    a = recommend.diversify(x, 100, pa, table, lam=0.5, max_per_category=4, hist_article=ha)
    b = recommend.diversify(x, 100, pa, table, lam=0.5, max_per_category=4, hist_article=ha)
    for u, v in zip(a, b):
        assert _same(u, v)


def test_at_scale():
    B, N, n = 1024, 20000, 25000
    rng = np.random.default_rng(8)
    g = torch.Generator(device='cuda').manual_seed(8)
    x = torch.randn(B, N, device='cuda', generator=g)
    pool = rng.permutation(np.arange(1, n))[:N].astype(np.int32)
    rows = rng.normal(size=(n, 80)).astype(np.float32)
    rows[:, 64] = rng.integers(0, 8, n)
    hist = rng.choice(pool, (B, 100)).astype(np.int32)
    pa, ha = _cuda(pool, hist)
    table = _table(rows)
    sel = recommend.select(x, 100, pa, n, hist_article=ha)
    d = recommend.diversify(x, 100, pa, table, lam=1.0, candidates=512, hist_article=ha)
    assert torch.equal(d.position, sel.position) and _same(d.score, sel.score)
    d = recommend.diversify(x, 100, pa, table, lam=0.7, candidates=512, max_per_category=20, hist_article=ha)
    assert (d.position >= 0).all()
    cand = recommend.select(x, 512, pa, n, hist_article=ha)
    users = slice(0, 1024, 128)
    worst = _replay(cand.position[users].cpu().numpy(), cand.score[users].cpu().numpy(), pool, rows, n,
                    d.position[users].cpu().numpy(), d.gain[users].cpu().numpy(), 0.7, 20)
    assert worst <= REPLAY_TOL


def test_bad_arguments_return_einval():
    lib = _lib.load()
    B, N, K = 2, 600, 512
    cpos = torch.zeros(B, K, dtype=torch.int32, device='cuda')
    cval = torch.zeros(B, K, device='cuda')
    pa = torch.ones(N, dtype=torch.int32, device='cuda')
    rows = torch.zeros(10, 80, device='cuda')
    pos = torch.empty(B, K, dtype=torch.int32, device='cuda')
    val, gain = torch.empty(B, K, device='cuda'), torch.empty(B, K, device='cuda')
    p = lambda t: ctypes.c_void_p(t.data_ptr())

    def call(n_cand=K, k=10, lam=0.5, q=0, B=B, N=N, n_articles=10, null=None):
        ptrs = [p(cpos), p(cval), p(pa), p(rows), p(pos), p(val), p(gain)]
        if null is not None:
            ptrs[null] = None
        return lib.nrm_pool_diversify(ptrs[0], ptrs[1], B, n_cand, k, lam, q, ptrs[2], N, ptrs[3], n_articles, ptrs[4], ptrs[5], ptrs[6], None)
    for null in range(7):
        assert call(null=null) == -1 and b'null' in lib.nrm_last_error()
    for kw in (dict(B=0), dict(N=0), dict(n_articles=0), dict(n_cand=0), dict(n_cand=513), dict(n_cand=300, N=200), dict(k=0),
               dict(k=513), dict(k=11, n_cand=10), dict(lam=float('nan')), dict(lam=-0.01), dict(lam=1.01), dict(q=-1)):
        assert call(**kw) == -1, kw
    assert call(lam=1.0) == 0 and call(n_cand=512, k=512, lam=0.0, q=1) == 0
    torch.cuda.synchronize()
    assert (pos[:, 1:] == -1).all()                                              # one article, one category, cap 1: one pick
    with pytest.raises(NrmError):
        recommend.diversify(torch.zeros(2, 5), 2, pa[:5].cpu(), wire.ArticleTable(rows), lam=0.5)   # CPU logits
