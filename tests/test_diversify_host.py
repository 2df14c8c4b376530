"""Pool diversification (news_recommendation_model_b200.recommend.diversify / diverse_articles / list_diversity) on the host: the
float64 restatement (tests/diversify_ref.py) against a brute-force greedy written out with Python floats, its limiting cases, and
the argument checks that run before any device is touched."""
import math

import numpy as np
import pytest
import torch

from diversify_ref import exact_rows, greedy, host_diversify, relevance
from recommend_ref import host_top_articles
from news_recommendation_model_b200 import NrmError, recommend, wire

FLT_MAX = float(np.finfo(np.float32).max)


def _brute(cand_pos, cand_score, pool, rows, n_articles, k, lam, q):
    """One user at a time, every remaining candidate's gain recomputed from scratch at every step (Python floats)."""
    out = []
    for pos, sc in zip(np.asarray(cand_pos).tolist(), np.asarray(cand_score, dtype=np.float64).tolist()):
        cands = [(i, p, s) for i, (p, s) in enumerate(zip(pos, sc)) if p >= 0 and 1 <= pool[p] < n_articles]
        fin = [s for _, _, s in cands if math.isfinite(s)]
        lo, hi = (min(fin), max(fin)) if fin else (0.0, 0.0)

        def rel(s):
            if s == math.inf:
                return 1.0
            if s == -math.inf:
                return 0.0
            return 1.0 if hi == lo else (s - lo) / (hi - lo)

        def unit(p):
            v = [float(x) for x in rows[pool[p], :64]]
            n = math.sqrt(sum(x * x for x in v))
            return [x / n for x in v] if n > 0 else v

        def cat(p):
            return int(rows[pool[p], 64])
        picks = []
        while len(picks) < k:
            best = None
            for i, p, s in cands:
                if any(i == j for j, _, _ in picks):
                    continue
                if q > 0 and sum(cat(pp) == cat(p) for _, pp, _ in picks) >= q:
                    continue
                sim = max((sum(a * b for a, b in zip(unit(p), unit(pp))) for _, pp, _ in picks), default=0.0)
                g = lam * rel(s) - (1 - lam) * sim
                if best is None or g > best[0]:
                    best = (g, i, p, s)
            if best is None:
                break
            picks.append((best[1], best[2], best[0]))
        out.append([p for _, p, _ in picks] + [-1] * (k - len(picks)))
    return np.array(out, dtype=np.int64)


def _case(seed, B=4, N=60, n_articles=50, n_categories=4, exact=False, zero_every=7):
    rng = np.random.default_rng(seed)
    pool = rng.integers(0, n_articles + 3, N).astype(np.int32)             # pads, out-of-range and repeated ids
    rows = exact_rows(n_articles, n_categories, rng, zero_every) if exact else rng.normal(size=(n_articles, 80)).astype(np.float32)
    if not exact:
        rows[::zero_every] = 0.0
        rows[:, 64] = rng.integers(0, n_categories, n_articles)
    logits = rng.normal(size=(1, B, N)).astype(np.float32)
    logits[0, :, ::9] = np.nan
    hist = rng.choice(pool, (B, 6)).astype(np.int32)
    return logits, pool, rows, hist


@pytest.mark.parametrize('lam', [0.0, 0.3, 0.7, 1.0])
@pytest.mark.parametrize('q', [0, 1, 2])
@pytest.mark.parametrize('seed', [1, 2])
def test_restatement_against_brute_force(lam, q, seed):
    logits, pool, rows, hist = _case(seed)
    pos, val = host_top_articles(logits, pool, 50, 20, hist)
    got = greedy(pos, val, pool, rows, 50, 8, lam, q)
    assert np.array_equal(got['position'], _brute(pos, val, pool, rows, 50, 8, lam, q))
    picked = got['position'] >= 0
    assert np.array_equal(np.isnan(got['score']), ~picked) and np.array_equal(np.isnan(got['gain']), ~picked)


def test_lambda_one_is_the_sorted_order():
    logits, pool, rows, hist = _case(3, B=6, N=200)
    for k in (1, 10, 40):
        pos, val = host_top_articles(logits, pool, 50, k, hist)
        got = host_diversify(logits, pool, 50, rows, k, 1.0, 40, 0, hist)
        assert np.array_equal(got['position'], pos) and np.array_equal(got['score'], val, equal_nan=True)


def test_lambda_zero_picks_by_dissimilarity():
    """lam = 0: the first pick is the best candidate (every gain is 0), then always a candidate least similar to the picks."""
    logits, pool, rows, _ = _case(4, N=300, n_articles=300)
    pos, val = host_top_articles(logits, pool, 300, 30)
    got = greedy(pos, val, pool, rows, 300, 10, 0.0)
    assert np.array_equal(got['position'][:, 0], pos[:, 0]) and (got['gain'][:, 0] == 0).all()
    assert np.array_equal(got['position'], _brute(pos, val, pool, rows, 300, 10, 0.0, 0))
    assert (np.diff(got['gain'][:, 1:], axis=1) <= 0).all()                  # after the first pick m only grows


def test_caps_that_exhaust_every_category():
    logits, pool, rows, _ = _case(5, n_categories=3)
    pos, val = host_top_articles(logits, pool, 50, 30)
    got = greedy(pos, val, pool, rows, 50, 10, 0.5, q=2)
    n = (got['position'] >= 0).sum(1)
    assert (n == 6).all()                                                    # 3 categories x 2, then nothing can be picked
    assert np.isnan(got['score'][:, 6:]).all() and (got['position'][:, 6:] == -1).all()
    assert np.array_equal(got['position'], _brute(pos, val, pool, rows, 50, 10, 0.5, 2))


def test_fewer_eligible_positions_than_k():
    logits, pool, rows, hist = _case(6, N=12)
    pos, val = host_top_articles(logits, pool, 50, 12, hist)
    got = greedy(pos, val, pool, rows, 50, 12, 0.6)
    assert np.array_equal((got['position'] >= 0).sum(1), (pos >= 0).sum(1))
    assert np.array_equal(got['position'], _brute(pos, val, pool, rows, 50, 12, 0.6, 0))


def test_all_zero_vectors_have_similarity_zero():
    logits, pool, rows, _ = _case(7)
    rows[:, :64] = 0.0
    pos, val = host_top_articles(logits, pool, 50, 20)
    got = greedy(pos, val, pool, rows, 50, 10, 0.4)
    assert np.array_equal(got['position'], pos[:, :10])                      # m = 0 throughout: the relevance order
    for b in range(pos.shape[0]):
        rel = relevance(val[b][pos[b] >= 0])
        n = min(10, rel.size)
        assert np.array_equal(got['gain'][b, :n], 0.4 * rel[:n])


@pytest.mark.parametrize('scores', [
    [np.inf, 3.0, 1.0, -np.inf, 2.0, np.inf],
    [2.0, 2.0, 2.0, 2.0, 2.0, 2.0],
    [FLT_MAX, -FLT_MAX, 0.0, FLT_MAX / 2, -FLT_MAX, 1.0],
    [np.inf, -np.inf, -np.inf, np.inf, np.inf, -np.inf],
], ids=['inf', 'equal', 'flt_max', 'only_inf'])
def test_infinite_equal_and_huge_scores(scores):
    s = np.array(scores)
    rel = relevance(s)
    assert rel.min() >= 0 and rel.max() <= 1 and not np.isnan(rel).any()
    assert (rel[s == np.inf] == 1).all() and (rel[s == -np.inf] == 0).all()
    fin = np.isfinite(s)
    if fin.any() and s[fin].max() > s[fin].min():
        assert rel[fin][np.argmax(s[fin])] == 1 and rel[fin][np.argmin(s[fin])] == 0
    elif fin.any():
        assert (rel[fin] == 1).all()
    rng = np.random.default_rng(8)
    rows = exact_rows(10, 3, rng)
    pool = np.arange(1, 7, dtype=np.int32)
    logits = s.astype(np.float32)[None, None]
    pos, val = host_top_articles(logits, pool, 10, 6)
    for lam, q in ((1.0, 0), (0.5, 0), (0.5, 1), (0.0, 2)):
        got = greedy(pos, val, pool, rows, 10, 6, lam, q)
        assert np.array_equal(got['position'], _brute(pos, val, pool, rows, 10, 6, lam, q)), (lam, q)
        if (lam, q) == (1.0, 0):
            assert np.array_equal(got['position'], pos)


def test_list_diversity_against_its_definition():
    rng = np.random.default_rng(9)
    rows = rng.normal(size=(20, 80)).astype(np.float32)
    rows[3, :64] = 0.0
    rows[:, 64] = rng.integers(0, 4, 20)
    table = wire.ArticleTable(torch.from_numpy(rows))
    article = torch.tensor([[1, 2, 3, 4], [5, -1, 5, 0], [6, -1, -1, -1], [-1, -1, -1, -1], [7, 8, 25, 9]])
    ild, ncat = recommend.list_diversity(table, article)
    assert ild.dtype == torch.float32 and ncat.dtype == torch.int64
    for b, ids in enumerate(article.tolist()):
        ids = [a for a in ids if 1 <= a < 20]
        def unit(a):
            v = rows[a, :64].astype(np.float64)
            n = np.linalg.norm(v)
            return v / n if n > 0 else v
        pairs = [1 - unit(a) @ unit(c) for i, a in enumerate(ids) for c in ids[i + 1:]]
        if pairs:
            assert abs(ild[b].item() - np.mean(pairs)) <= 1e-6
        else:
            assert math.isnan(ild[b].item())
        assert ncat[b].item() == len({int(rows[a, 64]) for a in ids})


def _table(n=6):
    return wire.ArticleTable(torch.zeros(n, wire.ARTICLE_COLS))


def test_diversify_checks_its_arguments_before_the_device():
    x = torch.zeros(2, 5)
    pa = torch.arange(1, 6, dtype=torch.int32)
    table = _table()
    for kw in (dict(k=0), dict(k=4, candidates=3), dict(k=1, candidates=6), dict(k=1, candidates=0), dict(k=True), dict(k=2.0),
               dict(lam=1.5), dict(lam=-0.1), dict(lam=float('nan')), dict(lam=None), dict(lam=True), dict(max_per_category=-1),
               dict(max_per_category=1.0), dict(candidates=True)):
        args = dict(k=2, lam=0.5)
        args.update(kw)
        with pytest.raises(ValueError):
            recommend.diversify(x, args.pop('k'), pa, table, **args)
    with pytest.raises(ValueError):
        recommend.diversify(torch.zeros(600, 2, 600)[0], 1, pa, table, lam=0.5, candidates=513)
    with pytest.raises(ValueError):
        recommend.diversify(x, 2, pa, object(), lam=0.5)
    with pytest.raises(ValueError):
        recommend.diversify(x, 2, pa, wire.ArticleTable(torch.zeros(6, 79)), lam=0.5)
    with pytest.raises(ValueError):
        recommend.diversify(torch.zeros(5), 2, pa, table, lam=0.5)
    with pytest.raises(NrmError):
        recommend.diversify(x, 2, pa, table, lam=0.5, max_per_category=0)          # valid arguments, CPU tensors


def test_diverse_articles_checks_its_arguments_before_the_device():
    table = _table()
    ha = torch.ones(2, 3, dtype=torch.int32)
    ht, hc = torch.zeros(2, 3, dtype=torch.int32), torch.zeros(2, 3, 2)
    pa, pt = torch.arange(1, 6, dtype=torch.int32), torch.zeros(5, dtype=torch.int32)
    model = torch.nn.Module()                                                # never reached
    for kw in (dict(k=6), dict(k=3, candidates=2), dict(k=2, lam=2.0), dict(k=2, max_per_category=-3), dict(k=2, chunk=12)):
        args = dict(k=2, lam=0.5, pool_article=pa)
        args.update(kw)
        with pytest.raises(ValueError):
            recommend.diverse_articles(model, table, ha, ht, hc, pt, args.pop('k'), **args)
    with pytest.raises(ValueError):
        recommend.diverse_articles([model] * 17, table, ha, ht, hc, pt, 2, lam=0.5, pool_article=pa)
    with pytest.raises(ValueError):
        recommend.diverse_articles(model, table, ha, ht, hc, pt[:4], 2, lam=0.5, pool_article=pa)
    with pytest.raises(NrmError):
        recommend.diverse_articles(model, table, ha, ht, hc, pt, 2, lam=0.5, pool_article=pa)


def test_list_diversity_checks_its_arguments():
    table = _table()
    for bad in (torch.ones(4, dtype=torch.int64), torch.ones(2, 3), torch.ones(2, 3, dtype=torch.bool), [[1, 2]]):
        with pytest.raises(ValueError):
            recommend.list_diversity(table, bad)
    with pytest.raises(ValueError):
        recommend.list_diversity(object(), torch.ones(2, 3, dtype=torch.int64))
