"""Host restatement of pool evaluation (news_recommendation_model_b200.recommend.rank_targets / pool_metrics, nrm_pool_rank) in
float64 numpy.  Eligibility and scores come from recommend_ref; ranks from a brute-force stable sorted(..., reverse=True)."""
import math

import numpy as np

from recommend_ref import eligible, scores


def host_rank_targets(logits, targets, pool_article, n_articles, hist_article=None):
    """[M,B,N] (or [B,N]) logits, targets [B,P] -> dict of position / rank / greater / equal [B,P] int64 (-1: not rankable),
    score [B,P] float64 (NaN likewise), n_eligible [B] int64, and the float64 scores [B,N] (NaN where not eligible)."""
    x = np.asarray(logits)
    if x.ndim == 2:
        x = x[None]
    ok = eligible(x, pool_article, n_articles, hist_article)
    s = scores(x, ok)
    pa = np.asarray(pool_article)
    tg = np.asarray(targets)
    B, P = tg.shape
    out = {name: np.full((B, P), -1, dtype=np.int64) for name in ('position', 'rank', 'greater', 'equal')}
    out['score'] = np.full((B, P), np.nan)
    out['n_eligible'] = ok.sum(1).astype(np.int64)
    out['scores'] = s
    for b in range(B):
        elig = [n for n in range(pa.size) if ok[b, n]]
        order = sorted(elig, key=lambda n: s[b, n], reverse=True)       # stable: ties keep the lower position first
        rank_of = {n: r for r, n in enumerate(order)}
        neg_desc = -s[b, order]                                         # ascending
        seen = set()
        for p in range(P):
            t = int(tg[b, p])
            if t in seen:
                continue
            seen.add(t)
            if not 1 <= t < n_articles:
                continue
            held = [n for n in np.flatnonzero(pa == t) if ok[b, n]]
            if not held:
                continue
            n = min(held, key=lambda m: rank_of[m])                    # a repeated pool id: the occurrence ranked first
            v = s[b, n]
            out['position'][b, p] = n
            out['rank'][b, p] = rank_of[n]
            out['greater'][b, p] = np.searchsorted(neg_desc, -v, 'left')
            out['equal'][b, p] = np.searchsorted(neg_desc, -v, 'right') - out['greater'][b, p] - 1
            out['score'][b, p] = v
    return out


def host_pool_metrics(r, ks=(10,)):
    """Per-user metrics from host_rank_targets' output, by their definitions: float64 [B] (NaN for a user without a rankable
    target, and for auc without an eligible negative); auc is computed from the scores by pairwise comparison."""
    rank, s = r['rank'], r['scores']
    B = rank.shape[0]
    out = {f'{m}@{k}': np.full(B, np.nan) for k in ks for m in ('hit', 'recall', 'ndcg')}
    out.update(rr=np.full(B, np.nan), auc=np.full(B, np.nan), n_targets=(rank >= 0).sum(1))
    for b in range(B):
        rk = rank[b][rank[b] >= 0]
        T = rk.size
        if T == 0:
            continue
        for k in ks:
            top = rk[rk < k]
            out[f'hit@{k}'][b] = float(top.size > 0)
            out[f'recall@{k}'][b] = top.size / T
            out[f'ndcg@{k}'][b] = sum(1 / math.log2(q + 2) for q in top) / sum(1 / math.log2(i + 2) for i in range(min(T, k)))
        out['rr'][b] = 1 / (rk.min() + 1)
        pos_n = set(int(n) for n in r['position'][b] if n >= 0)
        neg = ~np.isnan(s[b])
        neg[list(pos_n)] = False
        sp, sn = s[b, list(pos_n)], s[b, neg]
        if sn.size:
            out['auc'][b] = ((sp[:, None] > sn[None, :]).sum() + 0.5 * (sp[:, None] == sn[None, :]).sum()) / (sp.size * sn.size)
    return out


def edge_case(M, seed, B=6, N=60, P=12, n_articles=40):
    """Logits [M,B,N] float32 with exact ties, NaN, +-0; a pool with distinct ids (0, negative and out-of-range ids included);
    histories; targets [B,P] (P >= 4) with pads, out-of-range ids, ids missing from the pool, clicked ids, repeats and NaN positions.
    User 5 has no rankable target."""
    rng = np.random.default_rng(seed)
    logits = (rng.integers(-4, 5, (M, B, N)) / 2).astype(np.float32)       # few distinct values: many exact ties
    for m, b, n, v in ((slice(None), 1, 7, np.nan), (0, 2, 11, np.nan),    # NaN in one model only: not eligible either
                       (slice(None), 3, 4, -0.0), (slice(None), 3, 5, 0.0)):
        if b < B and n < N:
            logits[m, b, n] = v
    ids = rng.permutation(np.arange(1, n_articles))[:n_articles - 6]       # 5 real ids are not in the pool
    pool = np.concatenate([ids, [0, -3, n_articles, n_articles + 5], np.arange(n_articles + 10, n_articles + 10 + max(N, 1))])
    pool = rng.permutation(pool[:max(N, ids.size + 4)])[:N].astype(np.int32)
    special = [n for n in (4, 5, 7, 11) if n < N]                          # real ids where the targets below need them
    spare = [n for n in range(N) if n not in special and 1 <= pool[n] < n_articles]
    for n in special:
        if not 1 <= pool[n] < n_articles and spare:
            m = spare.pop()
            pool[n], pool[m] = pool[m], pool[n]
    hist = rng.integers(0, n_articles, (B, 8)).astype(np.int32)
    hist[:, -2:] = 0
    targets = rng.integers(0, n_articles + 3, (B, P)).astype(np.int32)
    targets[:, 0] = hist[:, 0]                                              # a clicked article
    targets[:, 1] = targets[:, 2]                                           # a repeat
    targets[:, 3] = 0
    for b, p, n in ((1, 4, 7), (2, 4, 11), (3, 4, 4), (3, 5, 5)):           # NaN positions, then -0.0 and +0.0
        if b < B and p < P and n < N:
            targets[b, p] = pool[n]
    if B > 4:
        targets[4, P - 1] = -1
    if B > 5:
        targets[5] = 0
        targets[5, :min(P, 2)] = (n_articles, n_articles + 1)[:min(P, 2)]  # nothing rankable
    return logits, pool, hist, targets, n_articles
