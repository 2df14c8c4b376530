"""Host restatement of the pool selection (news_recommendation_model_b200.recommend.select / nrm_pool_topk) in float64 numpy."""
import numpy as np


def eligible(logits, pool_article, n_articles, hist_article=None):
    """[M,B,N] logits -> [B,N] bool: id in [1, n_articles), no NaN logit in any model, not among the user's non-pad history ids."""
    pa = np.asarray(pool_article)
    ok = ((pa >= 1) & (pa < n_articles))[None, :] & ~np.isnan(np.asarray(logits)).any(0)
    if hist_article is not None:
        ha = np.asarray(hist_article)
        for b in range(ok.shape[0]):
            ok[b] &= ~np.isin(pa, ha[b][ha[b] != 0])
    return ok


def scores(logits, ok):
    """The ranking score [B,N] in float64 (NaN where not eligible): the logit for one model, else the mean over the models of the
    softmax over each user's eligible positions."""
    x = np.asarray(logits, dtype=np.float64)
    if x.shape[0] == 1:
        return np.where(ok, x[0], np.nan)
    out = np.zeros(ok.shape)
    for xm in x:
        xm = np.where(ok, xm, -np.inf)
        mx = xm.max(1, keepdims=True)
        e = np.where(ok, np.exp(xm - np.where(np.isfinite(mx), mx, 0.0)), 0.0)
        out += e / np.maximum(e.sum(1, keepdims=True), np.finfo(np.float64).tiny)
    return np.where(ok, out / x.shape[0], np.nan)


def top_positions(score, ok, k):
    """-> [B,k] int64 positions: eligible positions by descending score, ties to the lower position; -1 past the eligible ones."""
    B, N = score.shape
    out = np.full((B, k), -1, dtype=np.int64)
    for b in range(B):
        idx = np.flatnonzero(ok[b])
        order = idx[np.lexsort((idx, -score[b, idx]))][:k]      # last key is primary: -score ascending, then position
        out[b, :order.size] = order
    return out


def host_top_articles(logits, pool_article, n_articles, k, hist_article=None):
    """[M,B,N] (or [B,N]) logits -> (positions [B,k] int64, scores [B,k] float64, NaN past the eligible positions)."""
    x = np.asarray(logits)
    if x.ndim == 2:
        x = x[None]
    ok = eligible(x, pool_article, n_articles, hist_article)
    s = scores(x, ok)
    pos = top_positions(s, ok, k)
    val = np.where(pos >= 0, np.take_along_axis(s, np.maximum(pos, 0), 1), np.nan)
    return pos, val
