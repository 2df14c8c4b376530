"""Host restatement of pool diversification (news_recommendation_model_b200.recommend.diversify / nrm_pool_diversify) in float64
numpy: greedy maximal marginal relevance over `select`'s candidates (recommend_ref.host_top_articles), with a cap per category."""
import numpy as np

from recommend_ref import host_top_articles

PCA_COLS, CATEGORY_COL = 64, 64


def unit_vectors(rows):
    """[n,80] article rows -> [n,64] float64 PCA vectors scaled to unit length (all-zero rows stay zero)."""
    v = np.asarray(rows, dtype=np.float64)[:, :PCA_COLS]
    n = np.sqrt((v * v).sum(1, keepdims=True))
    return np.where(n > 0, v / np.where(n > 0, n, 1.0), 0.0)


def relevance(score):
    """Candidate scores (float64, any length) -> min-max normalised over the finite ones; +inf -> 1, -inf -> 0, all equal -> 1."""
    s = np.asarray(score, dtype=np.float64)
    rel = np.ones_like(s)
    fin = np.isfinite(s)
    if fin.any():
        lo, hi = s[fin].min(), s[fin].max()
        if hi > lo:
            rel[fin] = (s[fin] - lo) / (hi - lo)
    rel[s == -np.inf] = 0.0
    return rel


def greedy(cand_pos, cand_score, pool_article, rows, n_articles, k, lam, q=0):
    """cand_pos / cand_score [B,K'] (`select`'s position / score; -1 = no candidate) -> dict of [B,k] arrays: position (int64),
    score and gain (float64); -1 / NaN past the picks.  Each step takes the largest gain = lam * rel - (1 - lam) * max sim to the
    picks, ties to the lower candidate index; with q > 0 a category with q picks is closed."""
    cand_pos = np.asarray(cand_pos)
    B = cand_pos.shape[0]
    u = unit_vectors(rows)
    cats = np.trunc(np.asarray(rows)[:, CATEGORY_COL]).astype(np.int64)
    pa = np.asarray(pool_article)
    out = dict(position=np.full((B, k), -1, np.int64), score=np.full((B, k), np.nan), gain=np.full((B, k), np.nan))
    for b in range(B):
        pos = cand_pos[b]
        ok = pos >= 0
        ids = np.where(ok, pa[np.maximum(pos, 0)], 0)
        ok &= (ids >= 1) & (ids < n_articles)
        s = np.asarray(cand_score[b], dtype=np.float64)
        rel = np.where(ok, relevance(np.where(ok, s, np.nan)), 0.0)
        U = u[ids]
        cat = cats[ids]
        m = np.zeros(pos.size)
        live = ok.copy()
        count = {}
        for t in range(k):
            if not live.any():
                break
            gain = lam * rel - (1.0 - lam) * m
            j = int(np.argmax(np.where(live, gain, -np.inf)))          # first maximum: the lower index
            out['position'][b, t], out['score'][b, t], out['gain'][b, t] = pos[j], s[j], gain[j]
            live[j] = False
            sim = (U * U[j]).sum(1)                                      # the same sum for equal vectors (a matrix product may differ)
            m = sim if t == 0 else np.maximum(m, sim)                        # may be negative
            count[cat[j]] = count.get(cat[j], 0) + 1
            if q > 0 and count[cat[j]] >= q:
                live &= cat != cat[j]
    return out


def host_diversify(logits, pool_article, n_articles, rows, k, lam, candidates, q=0, hist_article=None):
    """The whole of `diversify`: host_top_articles(candidates), then greedy."""
    pos, val = host_top_articles(logits, pool_article, n_articles, candidates, hist_article)
    return greedy(pos, val, pool_article, rows, n_articles, k, lam, q)


def exact_rows(n_articles, n_categories, rng, zero_every=7):
    """[n_articles,80] float32 rows whose PCA vectors have four entries +-0.5 among the first 8 columns (norm exactly 1, every dot
    product a multiple of 1/4, so every similarity is exact in float32), every `zero_every`-th row all zero; categories in
    [0, n_categories)."""
    rows = np.zeros((n_articles, 80), np.float32)
    for a in range(1, n_articles):
        if a % zero_every:
            cols = rng.choice(8, 4, replace=False)
            rows[a, cols] = rng.choice([-0.5, 0.5], 4)
        rows[a, CATEGORY_COL] = rng.integers(0, n_categories)
    return rows
