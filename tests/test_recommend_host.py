"""Pool recommendation (news_recommendation_model_b200.recommend) on the host: the float64 reference of the selection against a
brute-force stable sort, and the argument checks that need no device."""
import math

import numpy as np
import pytest
import torch

from recommend_ref import host_top_articles
from news_recommendation_model_b200 import NrmError, recommend, wire


def _brute_force(logits, pool_article, n_articles, k, hist_article):
    """Python's sorted(..., reverse=True) over the eligible positions, one user at a time, scores from math.exp."""
    M, B, N = logits.shape
    pos = np.full((B, k), -1, dtype=np.int64)
    val = np.full((B, k), np.nan)
    for b in range(B):
        clicked = set(int(h) for h in hist_article[b] if h != 0) if hist_article is not None else set()
        elig = [n for n in range(N) if 1 <= pool_article[n] < n_articles and int(pool_article[n]) not in clicked
                and not any(math.isnan(float(logits[m, b, n])) for m in range(M))]
        if M == 1:
            score = {n: float(logits[0, b, n]) for n in elig}
        else:
            score = {n: 0.0 for n in elig}
            for m in range(M):
                mx = max(float(logits[m, b, n]) for n in elig)
                z = sum(math.exp(float(logits[m, b, n]) - mx) for n in elig)
                for n in elig:
                    score[n] += math.exp(float(logits[m, b, n]) - mx) / z / M
        order = sorted(elig, key=lambda n: score[n], reverse=True)[:k]
        for j, n in enumerate(order):
            pos[b, j] = n
            val[b, j] = score[n]
    return pos, val


@pytest.mark.parametrize('M', [1, 2, 3])
@pytest.mark.parametrize('exclude', [True, False])
def test_reference_selection_is_the_stable_descending_sort(M, exclude):
    rng = np.random.default_rng(M * 10 + exclude)
    B, N, H, n_articles = 5, 60, 12, 40
    logits = rng.integers(-4, 5, (M, B, N)).astype(np.float32) / 2          # few distinct values: many exact ties
    logits[:, 1, 7] = np.nan
    logits[0, 2, 11] = np.nan                                                # NaN in one model only: not eligible either
    logits[:, 3, 4] = -0.0
    logits[:, 3, 5] = 0.0
    pool = rng.integers(-2, n_articles + 3, N).astype(np.int32)               # 0, negative and out-of-range ids
    pool[10:14] = pool[20]                                                   # duplicate ids are independent positions
    hist = rng.integers(0, n_articles, (B, H)).astype(np.int32)
    hist[:, -3:] = 0
    hist[4] = pool[np.clip(np.arange(H), 0, N - 1)]                          # user 4 has read most of the pool
    for k in (1, 7, N):
        ha = hist if exclude else None
        pos, val = host_top_articles(logits, pool, n_articles, k, ha)
        bpos, bval = _brute_force(logits, pool, n_articles, k, ha)
        assert np.array_equal(pos, bpos), (k, pos, bpos)
        assert np.allclose(val, bval, rtol=1e-12, atol=0, equal_nan=True)
    assert (pos == -1).any()                                                 # k = N: slots past the eligible positions


def _users(B=2, H=3, N=5, device='cpu'):
    ha = torch.ones(B, H, dtype=torch.int32, device=device)
    return ha, torch.zeros(B, H, dtype=torch.int32, device=device), torch.zeros(B, H, 2, device=device), \
        torch.zeros(N, dtype=torch.int32, device=device), torch.arange(1, N + 1, dtype=torch.int32, device=device)


def test_pool_calls_check_their_arguments_before_the_device():
    table = wire.ArticleTable(torch.zeros(6, wire.ARTICLE_COLS))
    ha, ht, hc, pt, pa = _users()
    model = torch.nn.Module()                                                # never reached: the arguments are checked first
    for chunk in (0, 12, -8, 8.0, True):
        with pytest.raises(ValueError):
            recommend.pool_logits(model, table, ha, ht, hc, pt, pool_article=pa, chunk=chunk)
    for k in (0, 6, 1025, 2.0, True):
        with pytest.raises(ValueError):
            recommend.top_articles(model, table, ha, ht, hc, pt, k, pool_article=pa)
    with pytest.raises(ValueError):
        recommend.pool_logits(model, table, ha.long(), ht, hc, pt, pool_article=pa)          # dtype
    with pytest.raises(ValueError):
        recommend.pool_logits(model, table, ha, ht[:, :2], hc, pt, pool_article=pa)          # shape
    with pytest.raises(ValueError):
        recommend.pool_logits(model, table, ha, ht, hc, pt[:4], pool_article=pa)             # pool_time vs pool_article
    with pytest.raises(ValueError):
        recommend.pool_logits(model, wire.ArticleTable(torch.zeros(8, wire.ARTICLE_COLS)), ha, ht, hc, pt)   # default pool: 7 articles
    with pytest.raises(ValueError):
        recommend.pool_logits(model, wire.ArticleTable(torch.zeros(6, 79)), ha, ht, hc, pt, pool_article=pa)
    with pytest.raises(ValueError):
        recommend.top_articles([model] * 17, table, ha, ht, hc, pt, 1, pool_article=pa)
    with pytest.raises(NrmError):
        recommend.pool_logits(model, table, ha, ht, hc, pt, pool_article=pa)                 # CPU tensors: no fallback
    with pytest.raises(NrmError):
        recommend.top_articles(model, table, ha, ht, hc, pt, 2, pool_article=pa)


def test_select_checks_its_arguments_before_the_device():
    pa = torch.arange(1, 6, dtype=torch.int32)
    with pytest.raises(ValueError):
        recommend.select(torch.zeros(2, 5), 6, pa, 10)                        # k > N
    with pytest.raises(ValueError):
        recommend.select(torch.zeros(2, 5), 0, pa, 10)
    with pytest.raises(ValueError):
        recommend.select(torch.zeros(2, 2000), 1025, torch.arange(2000, dtype=torch.int32), 10)
    with pytest.raises(ValueError):
        recommend.select(torch.zeros(2, 5, dtype=torch.float64), 1, pa, 10)
    with pytest.raises(ValueError):
        recommend.select(torch.zeros(17, 2, 5), 1, pa, 10)                    # more than 16 models
    with pytest.raises(ValueError):
        recommend.select(torch.zeros(2, 5), 1, pa.long(), 10)
    with pytest.raises(ValueError):
        recommend.select(torch.zeros(2, 5), 1, pa, 10, hist_article=torch.zeros(3, 4, dtype=torch.int32))
    with pytest.raises(NrmError):
        recommend.select(torch.zeros(2, 5), 2, pa, 10)
