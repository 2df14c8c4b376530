"""The pool-negative rules of include/nrm_b200.h (nrm_sample_negatives) restated on Python integers, one attempt at a time."""
import bisect

MASK32 = 0xFFFFFFFF
M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(ctr, key):
    """Philox4x32-10 of a 4-word counter and a 2-word key (Random123's philox4x32 with 10 rounds)."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & MASK32, (p0 >> 32) ^ c3 ^ k1, p0 & MASK32
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return c0, c1, c2, c3


def pool_cdf(pool_article, weights, n_articles):
    """Inclusive prefix sums of the weights (None: 1 each), ids outside [1, n_articles) at weight 0."""
    cdf, s = [], 0
    for i, a in enumerate(pool_article):
        w = 1 if weights is None else int(weights[i])
        s += w if 1 <= a < n_articles else 0
        cdf.append(s)
    return cdf


def draw(cdf, seed, step, row, attempt):
    """Pool position of one attempt."""
    x = philox4x32_10((attempt, row, step & MASK32, step >> 32), (seed & MASK32, seed >> 32))
    u = x[0] | x[1] << 32
    r = (u * cdf[-1]) >> 64
    return bisect.bisect_right(cdf, r)            # the first n with cdf[n] > r


def sample_row(hist, cand, cand_time, label, pool_article, cdf, n_articles, k, seed, step, row):
    """One impression: (ids, times, labels) of the k appended columns."""
    first = next((c for c in range(len(cand)) if label[c] > 0), None)
    if first is None or cdf[-1] == 0:
        return [0] * k, [0] * k, [0.0] * k
    excluded = {a for a in hist if a != 0} | set(cand)
    ids = []
    for attempt in range(32 * k):
        if len(ids) == k:
            break
        a = pool_article[draw(cdf, seed, step, row, attempt)]
        if 1 <= a < n_articles and a not in excluded:
            ids.append(a)
            excluded.add(a)
    t = cand_time[first]
    return ids + [0] * (k - len(ids)), [t] * len(ids) + [0] * (k - len(ids)), [0.0] * k


def sample(hist_article, cand_article, cand_time, label, pool_article, weights, n_articles, k, seed, step=0, row_offset=0):
    """Lists of rows in, the appended [B][k] ids, times and labels out."""
    cdf = pool_cdf(pool_article, weights, n_articles)
    out = [sample_row(hist_article[b], cand_article[b], cand_time[b], label[b], pool_article, cdf, n_articles, k, seed, step,
                      row_offset + b) for b in range(len(cand_article))]
    return [o[0] for o in out], [o[1] for o in out], [o[2] for o in out]
