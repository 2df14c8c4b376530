"""Recommendation from a shared article pool: every user against the same N articles, each user's k best unread ones.

The reference scores the [B,C] candidates that come with each impression (test.py, verify.py, train.py).  A recommender is also
used the other way round: take the articles that are live now (for EB-NeRD, the `wire.ArticleTable` already resident on the
device), score all of them for every active user and return each user's k best, leaving out what the user has already read.

    logits = recommend.pool_logits(model, table, hist_article, hist_time, hist_click, pool_time)      # [B, n-1]: every real article
    rec = recommend.top_articles([m1, m2], table, hist_article, hist_time, hist_click, pool_time, 10)  # rec.article [B,10], best first

`pool_logits` runs the eval forward over the pool in chunks (`nrm_forward_pool`): the row kernels read the users' ids and each chunk's
article ids as they are, the chunk shared by all users, so the memory is that of a (B, H, chunk) forward, and the logits are, bit for bit, those of
`model.eval()(x_history, x_target, x_global)` with the pool broadcast as every user's candidates.  `top_articles` selects on the
GPU (`nrm_pool_topk`): the score is the logit for one model and, for an ensemble, the mean over the models of the softmax over the
user's eligible articles (test.py:58-63); the order is Python's stable `sorted(..., reverse=True)` (test.py:124-127).  Eligible are
the pool positions whose article id is in [1, n_articles), whose logits are not NaN and, with `exclude_clicked`, whose article
is not among the user's non-pad history ids; duplicate ids in the pool are independent positions.

The same ranking measures itself (`nrm_pool_rank`): given each user's held-out clicked articles, `rank_targets` returns where every
one lands in that user's ranking of the whole pool, `pool_metrics` turns those ranks into recall@k, nDCG@k, MRR and AUC, and
`evaluate` runs the three steps from the models:

    metrics, ranks = recommend.evaluate([m1, m2], table, hist_article, hist_time, hist_click, pool_time, targets, ks=(10, 100))
    torch.nanmean(metrics['ndcg@10'])

A ranking by relevance alone tends to fill a user's list with near-copies.  `diversify` / `diverse_articles` re-rank each user's
best candidates by greedy maximal marginal relevance over the articles' PCA vectors, optionally with a cap per category
(`nrm_pool_diversify`), and `list_diversity` measures what that bought:

    rec = recommend.diverse_articles(model, table, hist_article, hist_time, hist_click, pool_time, 10, lam=0.7, max_per_category=3)
    ild, n_categories = recommend.list_diversity(table, rec.article)"""
from __future__ import annotations

import numbers
from typing import NamedTuple, Optional

import torch

from . import _lib, engine, wire
from .engine import _stream

TOPK_MAX = 1024
TARGETS_MAX = 1024
CANDIDATES_MAX = 512                  # diversify: one thread per candidate in a 512-thread CTA
MODELS_MAX = 16
CHUNK_ALIGN = 8                       # the attention's candidate group: every multiple of it gives the same logits
WORKSPACE_TARGET = 1 << 30            # chunk=None: the largest chunk whose workspace stays under 1 GiB


class Recommendations(NamedTuple):
    article: torch.Tensor     # [B,k] int64 pool article ids, best first (-1: fewer than k eligible positions)
    position: torch.Tensor    # [B,k] int64 positions in the pool (-1 likewise)
    score: torch.Tensor       # [B,k] float32 ranking scores (NaN where the position is -1)


class TargetRanks(NamedTuple):
    """Per held-out target (b, p), counted over user b's eligible pool positions; -1 / NaN where the target is not rankable."""
    position: torch.Tensor    # [B,P] int64 the target's pool position
    rank: torch.Tensor        # [B,P] int64 positions ahead of it in top_articles' order: it is among top_articles(k) iff rank < k
    greater: torch.Tensor     # [B,P] int64 positions with a strictly larger score
    equal: torch.Tensor       # [B,P] int64 other positions with an equal score
    score: torch.Tensor       # [B,P] float32 its ranking score
    n_eligible: torch.Tensor  # [B] int64 the user's eligible positions


def _check_k(k, N: int) -> None:
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= min(N, TOPK_MAX):
        raise ValueError(f'k must be an integer in [1, min(N, {TOPK_MAX})] = [1, {min(N, TOPK_MAX)}], got {k!r}')


def _check_users_and_pool(table, hist_article, hist_time, hist_click, pool_time, pool_article, k=None, targets=None):
    """-> (B, H, N, pool_article); ValueError for shapes / dtypes / layout / k / targets (with `targets`, also for a pool that
    repeats an id), NrmError for tensors that are not on a CUDA device."""
    if not isinstance(table, wire.ArticleTable):
        raise ValueError('table must be a wire.ArticleTable')
    rows = table.rows
    if rows.dtype != torch.float32 or rows.dim() != 2 or rows.shape[1] != wire.ARTICLE_COLS or not rows.is_contiguous():
        raise ValueError(f'article table must be contiguous float32 [n, {wire.ARTICLE_COLS}]')
    if hist_article.dim() != 2:
        raise ValueError(f'hist_article must be [B,H], got {tuple(hist_article.shape)}')
    B, H = hist_article.shape
    if pool_article is None:
        pool_article = torch.arange(1, table.n, dtype=torch.int32, device=rows.device)
    N = int(pool_article.shape[0]) if pool_article.dim() == 1 else -1
    for name, t, shape, dt in (('hist_article', hist_article, (B, H), torch.int32), ('hist_time', hist_time, (B, H), torch.int32),
                               ('hist_click', hist_click, (B, H, 2), torch.float32), ('pool_article', pool_article, (N,), torch.int32),
                               ('pool_time', pool_time, (N,), torch.int32)):
        if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous():
            raise ValueError(f'{name} must be contiguous {dt} {list(shape)}, got {t.dtype} {list(t.shape)}')
    if B == 0 or H == 0 or N <= 0:
        raise ValueError(f'need B, H, N >= 1 (got {B}, {H}, {N})')
    if k is not None:
        _check_k(k, N)
    if targets is not None:
        _check_targets(targets, B)
        if not targets.is_contiguous():
            raise ValueError('targets must be contiguous')
        _check_distinct_pool(pool_article, table.n)
    tensors = (rows, hist_article, hist_time, hist_click, pool_article, pool_time) + ((targets,) if targets is not None else ())
    if not all(t.is_cuda for t in tensors):
        raise _lib.NrmError('recommend runs on CUDA tensors only (no CPU fallback)')
    if any(t.device != rows.device for t in tensors):
        raise ValueError('the article table, the users and the pool must be on the same device')
    return B, H, N, pool_article


def _check_chunk(chunk) -> None:
    if chunk is not None and (isinstance(chunk, bool) or not isinstance(chunk, int) or chunk <= 0 or chunk % CHUNK_ALIGN):
        raise ValueError(f'chunk must be a positive multiple of {CHUNK_ALIGN}, got {chunk!r}')


def default_chunk(B: int, H: int, N: int) -> int:
    """The largest multiple of 8, at most N rounded up to one, whose `nrm_pool_workspace_bytes` stays under 1 GiB (8 if none)."""
    lib = _lib.load()
    lo, hi = 1, (N + CHUNK_ALIGN - 1) // CHUNK_ALIGN           # in units of CHUNK_ALIGN
    if int(lib.nrm_pool_workspace_bytes(B, H, N, hi * CHUNK_ALIGN)) <= WORKSPACE_TARGET:
        return hi * CHUNK_ALIGN
    while lo < hi:                                               # the workspace grows with the chunk
        mid = (lo + hi + 1) // 2
        if int(lib.nrm_pool_workspace_bytes(B, H, N, mid * CHUNK_ALIGN)) <= WORKSPACE_TARGET:
            lo = mid
        else:
            hi = mid - 1
    return lo * CHUNK_ALIGN


def _forward_pool(model, table, hist_article, hist_time, hist_click, pool_time, pool_article, B, H, N, chunk, out) -> None:
    lib = _lib.load()
    dev = hist_article.device
    flat = model.flat_parameters()
    if flat.device != dev:
        raise _lib.NrmError(f'model is on {flat.device} but inputs are on {dev}')
    ws = torch.empty(int(lib.nrm_pool_workspace_bytes(B, H, N, chunk)), dtype=torch.uint8, device=dev)
    users = engine.compact(table, wire.CompactBatch(None, None, hist_article, hist_time, hist_click, pool_article, pool_time, None, None))
    p = engine._ptr
    _lib.check(lib.nrm_forward_pool(*users.args, B, H, N, chunk, p(flat.buf), p(model.bn.running_mean), p(model.bn.running_var),
                                    model._precision_code(), p(out), p(ws), ws.numel(), _stream(dev)), 'nrm_forward_pool')


def pool_logits(model, table: wire.ArticleTable, hist_article, hist_time, hist_click, pool_time, *,
                pool_article: Optional[torch.Tensor] = None, chunk: Optional[int] = None) -> torch.Tensor:
    """[B,N] float32 logits of `model` (a `UserModel`) for B users (compact histories: `hist_article` / `hist_time` int32 [B,H],
    article id 0 = pad row, `hist_click` float32 [B,H,2]) against a pool of N articles (`pool_article` int32 [N], default: every
    real article of `table`, ids 1..n-1; `pool_time` int32 [N] packed time buckets, `wire.pack_time`, one time for all users).

    Bit for bit `model.eval()(x_history, x_target, x_global)` with the pool as every user's candidates, in the model's precision;
    eval semantics whatever `model.training` says (BatchNorm reads its running statistics and writes nothing), under no_grad.
    `chunk`: pool articles per forward, a positive multiple of 8 (the result does not depend on it); None: `default_chunk`."""
    _check_chunk(chunk)
    B, H, N, pa = _check_users_and_pool(table, hist_article, hist_time, hist_click, pool_time, pool_article)
    with torch.no_grad():
        logits = torch.empty(B, N, dtype=torch.float32, device=hist_article.device)
        _forward_pool(model, table, hist_article, hist_time, hist_click, pool_time, pa, B, H, N,
                      chunk if chunk is not None else default_chunk(B, H, N), logits)
    return logits


def select(logits: torch.Tensor, k: int, pool_article: torch.Tensor, n_articles: int, *,
           hist_article: Optional[torch.Tensor] = None) -> Recommendations:
    """The selection `top_articles` runs, on given logits: [B,N] (one model) or [M,B,N] (an ensemble of M <= 16 models) float32.
    `hist_article` [B,H] int32: leave out the pool positions whose article the user has clicked (None: no exclusion)."""
    if logits.dim() == 2:
        logits = logits.unsqueeze(0)
    if logits.dim() != 3 or logits.dtype != torch.float32 or not 1 <= logits.shape[0] <= MODELS_MAX:
        raise ValueError(f'logits must be float32 [B,N] or [M,B,N] with M <= {MODELS_MAX}, got {logits.dtype} {list(logits.shape)}')
    M, B, N = logits.shape
    _check_k(k, N)
    if tuple(pool_article.shape) != (N,) or pool_article.dtype != torch.int32:
        raise ValueError(f'pool_article must be int32 [{N}], got {pool_article.dtype} {list(pool_article.shape)}')
    if hist_article is not None and (hist_article.dim() != 2 or hist_article.shape[0] != B or hist_article.dtype != torch.int32):
        raise ValueError(f'hist_article must be int32 [B,H] with B = {B}, got {hist_article.dtype} {list(hist_article.shape)}')
    for t in (logits, pool_article, hist_article):
        if t is not None and not t.is_cuda:
            raise _lib.NrmError('recommend runs on CUDA tensors only (no CPU fallback)')
        if t is not None and t.device != logits.device:
            raise ValueError('logits, pool_article and hist_article must be on the same device')
    x = logits.contiguous()
    pa = pool_article.contiguous()
    ha = hist_article.contiguous() if hist_article is not None else None
    H = int(ha.shape[1]) if ha is not None else 0
    dev = x.device
    pos = torch.empty(B, k, dtype=torch.int32, device=dev)
    val = torch.empty(B, k, dtype=torch.float32, device=dev)
    p = engine._ptr
    _lib.check(_lib.load().nrm_pool_topk(p(x), M, B * N, B, N, k, p(pa), int(n_articles), p(ha), H, p(pos), p(val), _stream(dev)),
               'nrm_pool_topk')
    pos = pos.to(torch.int64)
    article = torch.where(pos >= 0, pa.to(torch.int64)[pos.clamp(min=0)], torch.full_like(pos, -1))
    return Recommendations(article, pos, val)


def _check_targets(targets, B: int) -> int:
    """-> P; ValueError unless targets is int32 [B,P] with 1 <= P <= 1024."""
    if not isinstance(targets, torch.Tensor) or targets.dim() != 2 or targets.shape[0] != B or targets.dtype != torch.int32:
        raise ValueError(f'targets must be int32 [B,P] with B = {B}, got {getattr(targets, "dtype", type(targets))} '
                         f'{list(getattr(targets, "shape", []))}')
    P = int(targets.shape[1])
    if not 1 <= P <= TARGETS_MAX:
        raise ValueError(f'targets must have 1 <= P <= {TARGETS_MAX} slots per user, got {P}')
    return P


def _check_distinct_pool(pool_article: torch.Tensor, n_articles: int) -> None:
    """ValueError if an article id in [1, n_articles) occurs twice in the pool (one device sync for a CUDA pool)."""
    ids = pool_article[(pool_article >= 1) & (pool_article < n_articles)]
    if torch.unique(ids).numel() != ids.numel():
        raise ValueError('pool_article holds a repeated article id: a target would have two ranks')


def _rank(x, targets, pa, n_articles, ha) -> TargetRanks:
    M, B, N = x.shape
    P = int(targets.shape[1])
    H = int(ha.shape[1]) if ha is not None else 0
    dev = x.device
    out = [torch.empty(B, P, dtype=torch.int32, device=dev) for _ in range(4)]
    score = torch.empty(B, P, dtype=torch.float32, device=dev)
    n_eligible = torch.empty(B, dtype=torch.int32, device=dev)
    p = engine._ptr
    _lib.check(_lib.load().nrm_pool_rank(p(x), M, B * N, B, N, p(pa), int(n_articles), p(ha), H, p(targets), P, *(p(t) for t in out),
                                         p(score), p(n_eligible), _stream(dev)), 'nrm_pool_rank')
    position, rank, greater, equal = (t.to(torch.int64) for t in out)
    return TargetRanks(position, rank, greater, equal, score, n_eligible.to(torch.int64))


def rank_targets(logits: torch.Tensor, targets: torch.Tensor, pool_article: torch.Tensor, n_articles: int, *,
                 hist_article: Optional[torch.Tensor] = None) -> TargetRanks:
    """Where each user's held-out targets land in the ranking `select` takes its first k entries of, on given logits ([B,N] or
    [M,B,N] float32, M <= 16): the same eligibility, scores and stable order over the whole pool, with no limit on the rank.

    `targets` int32 [B,P], 1 <= P <= 1024: article ids, 0 = pad slot.  A target is rankable if its id is in [1, n_articles), an
    eligible pool position holds it, and no earlier slot of the user's row holds the same id; the others get position, rank,
    greater and equal -1 and score NaN.  A rankable target is in `select(logits, k, ...)` iff its rank < k, at index rank.
    `pool_article` must not repeat an id in [1, n_articles) (ValueError): a target would have two ranks.  That check costs one
    device synchronisation per call."""
    if logits.dim() == 2:
        logits = logits.unsqueeze(0)
    if logits.dim() != 3 or logits.dtype != torch.float32 or not 1 <= logits.shape[0] <= MODELS_MAX:
        raise ValueError(f'logits must be float32 [B,N] or [M,B,N] with M <= {MODELS_MAX}, got {logits.dtype} {list(logits.shape)}')
    M, B, N = logits.shape
    _check_targets(targets, B)
    if tuple(pool_article.shape) != (N,) or pool_article.dtype != torch.int32:
        raise ValueError(f'pool_article must be int32 [{N}], got {pool_article.dtype} {list(pool_article.shape)}')
    if hist_article is not None and (hist_article.dim() != 2 or hist_article.shape[0] != B or hist_article.dtype != torch.int32):
        raise ValueError(f'hist_article must be int32 [B,H] with B = {B}, got {hist_article.dtype} {list(hist_article.shape)}')
    _check_distinct_pool(pool_article, n_articles)
    for t in (logits, targets, pool_article, hist_article):
        if t is not None and not t.is_cuda:
            raise _lib.NrmError('recommend runs on CUDA tensors only (no CPU fallback)')
        if t is not None and t.device != logits.device:
            raise ValueError('logits, targets, pool_article and hist_article must be on the same device')
    return _rank(logits.contiguous(), targets.contiguous(), pool_article.contiguous(),
                 n_articles, hist_article.contiguous() if hist_article is not None else None)


def _check_ks(ks) -> tuple:
    ks = tuple(ks)
    if not ks or any(isinstance(k, bool) or not isinstance(k, int) or k < 1 for k in ks):
        raise ValueError(f'ks must be a non-empty sequence of positive integers, got {ks!r}')
    return ks


def pool_metrics(ranks: TargetRanks, ks=(10,)) -> dict:
    """Per-user metrics of pool recommendation from `rank_targets`' output, on its device.  T = the user's rankable targets.

    For each k in `ks`, float32 [B]: `hit@k` 1 if some target has rank < k; `recall@k` #{rank < k} / T; `ndcg@k` the sum over
    targets with rank < k of 1 / log2(rank + 2) over the ideal sum_{i < min(T, k)} 1 / log2(i + 2) (binary gains, as
    `metrics.batch_metrics`).  Also `rr` 1 / (min rank + 1); `auc` the tie-averaged ROC AUC (sklearn's `roc_auc_score`) over the
    user's eligible positions with the targets as positives, float32 [B]; `n_targets` T, int64 [B].  A user with T = 0, or (auc)
    with no eligible position that is not a target, gets NaN: average with `torch.nanmean`.

    The AUC needs no scores: a target with `greater` positions above it and `equal` tied has n_eligible - 1 - greater - equal below,
    and summed over the targets the pairs of two targets contribute exactly T (T - 1) / 2, which leaves the target-negative pairs."""
    ks = _check_ks(ks)
    valid = ranks.rank >= 0
    T = valid.sum(1)
    Tf = T.to(torch.float64)
    nan = torch.full_like(Tf, float('nan'))
    rank = ranks.rank.to(torch.float64)
    out = {}
    for k in ks:
        top = valid & (ranks.rank < k)
        hits = top.sum(1).to(torch.float64)
        dcg = torch.where(top, 1.0 / torch.log2(rank + 2.0), torch.zeros_like(rank)).sum(1)
        ideal_terms = 1.0 / torch.log2(torch.arange(min(k, ranks.rank.shape[1]), dtype=torch.float64, device=rank.device) + 2.0)
        ideal = torch.cumsum(ideal_terms, 0)[(T.clamp(max=k) - 1).clamp(min=0)]
        out[f'hit@{k}'] = torch.where(T > 0, (hits > 0).to(torch.float64), nan).float()
        out[f'recall@{k}'] = torch.where(T > 0, hits / Tf.clamp(min=1), nan).float()
        out[f'ndcg@{k}'] = torch.where(T > 0, dcg / ideal, nan).float()
    best = torch.where(valid, ranks.rank, torch.full_like(ranks.rank, torch.iinfo(torch.int64).max)).min(1).values
    out['rr'] = torch.where(T > 0, 1.0 / (best.clamp(max=torch.iinfo(torch.int32).max).to(torch.float64) + 1.0), nan).float()
    ne = ranks.n_eligible.to(torch.float64)
    g, e = ranks.greater.to(torch.float64), ranks.equal.to(torch.float64)
    below = torch.where(valid, ne[:, None] - 1.0 - g - e + 0.5 * e, torch.zeros_like(g)).sum(1)
    n_neg = ne - Tf
    out['auc'] = torch.where((T > 0) & (n_neg > 0), (below - Tf * (Tf - 1.0) / 2.0) / (Tf * n_neg).clamp(min=1), nan).float()
    out['n_targets'] = T
    return out


def evaluate(models, table: wire.ArticleTable, hist_article, hist_time, hist_click, pool_time, targets, *, ks=(10,),
             pool_article: Optional[torch.Tensor] = None, exclude_clicked: bool = True, chunk: Optional[int] = None):
    """Offline evaluation of pool recommendation: `pool_logits` of every model in `models` (one `UserModel` or up to 16), then
    `rank_targets` of each user's held-out clicked articles `targets` (int32 [B,P], 0 = pad) in the ranking `top_articles` uses,
    then `pool_metrics`.  Arguments as for `top_articles`.  -> (metrics dict, TargetRanks)."""
    if isinstance(models, torch.nn.Module):
        models = [models]
    models = list(models)
    if not 1 <= len(models) <= MODELS_MAX:
        raise ValueError(f'need 1 to {MODELS_MAX} models, got {len(models)}')
    _check_chunk(chunk)
    ks = _check_ks(ks)
    B, H, N, pa = _check_users_and_pool(table, hist_article, hist_time, hist_click, pool_time, pool_article, targets=targets)
    with torch.no_grad():
        logits = torch.empty(len(models), B, N, dtype=torch.float32, device=hist_article.device)
        c = chunk if chunk is not None else default_chunk(B, H, N)
        for m, model in enumerate(models):
            _forward_pool(model, table, hist_article, hist_time, hist_click, pool_time, pa, B, H, N, c, logits[m])
        ranks = _rank(logits, targets, pa, table.n, hist_article if exclude_clicked else None)
        return pool_metrics(ranks, ks), ranks


def top_articles(models, table: wire.ArticleTable, hist_article, hist_time, hist_click, pool_time, k: int, *,
                 pool_article: Optional[torch.Tensor] = None, exclude_clicked: bool = True,
                 chunk: Optional[int] = None) -> Recommendations:
    """Each user's `k` best eligible pool articles, best first: `pool_logits` of every model in `models` (one `UserModel` or a
    sequence of them, all in eval semantics), then `select`.  One model ranks by its logit; several rank by the mean of their
    softmaxes over the user's eligible positions (test.py:58-63).  Ties go to the lower pool position (test.py:124-127).  With
    `exclude_clicked` the articles in the user's history are left out.  1 <= k <= min(N, 1024); when fewer than k positions are
    eligible the remaining slots hold article -1, position -1 and score NaN."""
    if isinstance(models, torch.nn.Module):
        models = [models]
    models = list(models)
    if not 1 <= len(models) <= MODELS_MAX:
        raise ValueError(f'need 1 to {MODELS_MAX} models, got {len(models)}')
    _check_chunk(chunk)
    B, H, N, pa = _check_users_and_pool(table, hist_article, hist_time, hist_click, pool_time, pool_article, k)
    with torch.no_grad():
        logits = torch.empty(len(models), B, N, dtype=torch.float32, device=hist_article.device)
        c = chunk if chunk is not None else default_chunk(B, H, N)
        for m, model in enumerate(models):
            _forward_pool(model, table, hist_article, hist_time, hist_click, pool_time, pa, B, H, N, c, logits[m])
        return select(logits, k, pa, table.n, hist_article=hist_article if exclude_clicked else None)


class DiverseRecommendations(NamedTuple):
    article: torch.Tensor     # [B,k] int64 pool article ids in pick order (-1: fewer than k picks)
    position: torch.Tensor    # [B,k] int64 positions in the pool (-1 likewise)
    score: torch.Tensor       # [B,k] float32 the pick's ranking score, as `select` returns it (NaN where the position is -1)
    gain: torch.Tensor        # [B,k] float32 its MMR objective when it was picked (NaN likewise)


def _check_diversify(k, N: int, lam, candidates, max_per_category) -> tuple:
    """-> (K', q); ValueError unless 1 <= k <= K' <= min(N, 512) (K' = candidates, default min(N, 512)), lam is a number in [0, 1]
    and max_per_category is None or an integer >= 0 (q = 0: no cap)."""
    kc = min(N, CANDIDATES_MAX) if candidates is None else candidates
    if isinstance(kc, bool) or not isinstance(kc, int) or not 1 <= kc <= min(N, CANDIDATES_MAX):
        raise ValueError(f'candidates must be an integer in [1, min(N, {CANDIDATES_MAX})] = [1, {min(N, CANDIDATES_MAX)}], got {kc!r}')
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= kc:
        raise ValueError(f'k must be an integer in [1, candidates] = [1, {kc}], got {k!r}')
    if isinstance(lam, bool) or not isinstance(lam, numbers.Real) or not 0.0 <= float(lam) <= 1.0:     # NaN fails the comparison
        raise ValueError(f'lam must be a number in [0, 1], got {lam!r}')
    q = 0 if max_per_category is None else max_per_category
    if isinstance(q, bool) or not isinstance(q, int) or q < 0:
        raise ValueError(f'max_per_category must be None or an integer >= 0, got {max_per_category!r}')
    return kc, q


def _check_table(table) -> None:
    if not isinstance(table, wire.ArticleTable):
        raise ValueError('table must be a wire.ArticleTable')
    rows = table.rows
    if rows.dtype != torch.float32 or rows.dim() != 2 or rows.shape[1] != wire.ARTICLE_COLS or not rows.is_contiguous():
        raise ValueError(f'article table must be contiguous float32 [n, {wire.ARTICLE_COLS}]')


def _diversify(cand: Recommendations, k: int, lam, q: int, pa, table) -> DiverseRecommendations:
    B, kc = cand.position.shape
    N = int(pa.shape[0])
    dev = pa.device
    cpos = cand.position.to(torch.int32)
    pos = torch.empty(B, k, dtype=torch.int32, device=dev)
    val = torch.empty(B, k, dtype=torch.float32, device=dev)
    gain = torch.empty(B, k, dtype=torch.float32, device=dev)
    p = engine._ptr
    _lib.check(_lib.load().nrm_pool_diversify(p(cpos), p(cand.score), B, kc, k, float(lam), q, p(pa), N, p(table.rows), table.n,
                                              p(pos), p(val), p(gain), _stream(dev)), 'nrm_pool_diversify')
    pos = pos.to(torch.int64)
    article = torch.where(pos >= 0, pa.to(torch.int64)[pos.clamp(min=0)], torch.full_like(pos, -1))
    return DiverseRecommendations(article, pos, val, gain)


def diversify(logits: torch.Tensor, k: int, pool_article: torch.Tensor, table: wire.ArticleTable, *, lam: float,
              candidates: Optional[int] = None, max_per_category: Optional[int] = None,
              hist_article: Optional[torch.Tensor] = None) -> DiverseRecommendations:
    """Each user's `k` articles re-ranked for diversity by greedy maximal marginal relevance (MMR) over the article embeddings, on
    given logits ([B,N] or [M,B,N] float32, M <= 16).

    The candidates are `select(logits, candidates, pool_article, table.n, hist_article=hist_article)` (default candidates =
    min(N, 512)): the user's best eligible positions with `select`'s scores.  Relevance is the score min-max normalised over the
    user's candidates (finite scores; +inf -> 1, -inf -> 0, all equal -> 1), similarity the cosine of the articles' PCA vectors
    (table columns 0-63; 0 for an all-zero vector).  Each step picks the candidate with the largest
    gain = lam * relevance - (1 - lam) * (max similarity to the articles already picked), ties to the better `select` slot; with
    `max_per_category` = q a category (table column 64) gets at most q picks.  It stops after k picks or when nothing can be picked;
    the remaining slots hold article -1, position -1, score and gain NaN.  lam = 1 without a cap returns `select(logits, k, ...)`'s
    positions and scores bit for bit; lam = 0 picks by dissimilarity alone.  1 <= k <= candidates <= min(N, 512), 0 <= lam <= 1."""
    _check_table(table)
    if logits.dim() not in (2, 3):
        raise ValueError(f'logits must be float32 [B,N] or [M,B,N] with M <= {MODELS_MAX}, got {logits.dtype} {list(logits.shape)}')
    kc, q = _check_diversify(k, int(logits.shape[-1]), lam, candidates, max_per_category)
    if not logits.is_cuda or not table.rows.is_cuda:
        raise _lib.NrmError('recommend runs on CUDA tensors only (no CPU fallback)')
    if table.rows.device != logits.device:
        raise ValueError('logits and the article table must be on the same device')
    cand = select(logits, kc, pool_article, table.n, hist_article=hist_article)
    return _diversify(cand, k, lam, q, pool_article.contiguous(), table)


def diverse_articles(models, table: wire.ArticleTable, hist_article, hist_time, hist_click, pool_time, k: int, *, lam: float,
                     candidates: Optional[int] = None, max_per_category: Optional[int] = None,
                     pool_article: Optional[torch.Tensor] = None, exclude_clicked: bool = True,
                     chunk: Optional[int] = None) -> DiverseRecommendations:
    """`top_articles` re-ranked for diversity: `pool_logits` of every model in `models`, then `diversify`.  Arguments as for
    `top_articles` and `diversify`."""
    if isinstance(models, torch.nn.Module):
        models = [models]
    models = list(models)
    if not 1 <= len(models) <= MODELS_MAX:
        raise ValueError(f'need 1 to {MODELS_MAX} models, got {len(models)}')
    _check_chunk(chunk)
    _check_table(table)
    N = int(pool_article.shape[0]) if pool_article is not None and pool_article.dim() == 1 else table.n - 1
    kc, q = _check_diversify(k, N, lam, candidates, max_per_category)
    B, H, N, pa = _check_users_and_pool(table, hist_article, hist_time, hist_click, pool_time, pool_article)
    with torch.no_grad():
        logits = torch.empty(len(models), B, N, dtype=torch.float32, device=hist_article.device)
        c = chunk if chunk is not None else default_chunk(B, H, N)
        for m, model in enumerate(models):
            _forward_pool(model, table, hist_article, hist_time, hist_click, pool_time, pa, B, H, N, c, logits[m])
        cand = select(logits, kc, pa, table.n, hist_article=hist_article if exclude_clicked else None)
        return _diversify(cand, k, lam, q, pa, table)


def list_diversity(table: wire.ArticleTable, article: torch.Tensor) -> tuple:
    """What a recommendation list offers besides relevance, per user: -> (ild float32 [B], n_categories int64 [B]) for `article`
    [B,k] (the `article` of `top_articles` / `diverse_articles`; ids outside [1, table.n), such as -1, are no article).
    `ild`: intra-list diversity, the mean of 1 - cos(u_i, u_j) over the pairs of the list's articles, with the cosine of the PCA
    vectors as `diversify` uses it (0 for an all-zero vector), in float64; NaN for fewer than two articles.  `n_categories`: the
    number of distinct categories ((int) of table column 64) in the list.  Plain torch on the article's device (no kernel)."""
    _check_table(table)
    if not isinstance(article, torch.Tensor) or article.dim() != 2 or article.dtype.is_floating_point or article.dtype == torch.bool:
        raise ValueError(f'article must be an integer [B,k] tensor, got {getattr(article, "dtype", type(article))}')
    if article.device != table.rows.device:
        raise ValueError('article and the article table must be on the same device')
    valid = (article >= 1) & (article < table.n)
    r = table.rows[torch.where(valid, article, torch.zeros_like(article)).long()]          # [B,k,80]
    v = r[..., :64].double()
    norm = v.norm(dim=-1, keepdim=True)
    u = torch.where(norm > 0, v / norm.clamp(min=torch.finfo(torch.float64).tiny), torch.zeros_like(v))
    sim = u @ u.transpose(1, 2)
    k = article.shape[1]
    upper = torch.ones(k, k, dtype=torch.bool, device=article.device).triu(1)
    pair = valid[:, :, None] & valid[:, None, :] & upper
    n_pairs = pair.sum((1, 2))
    ild = torch.where(n_pairs > 0, torch.where(pair, 1.0 - sim, torch.zeros_like(sim)).sum((1, 2)) / n_pairs.clamp(min=1),
                      torch.full_like(n_pairs, float('nan'), dtype=torch.float64))
    cat = torch.where(valid, r[..., 64].double().trunc(), torch.full_like(valid, float('inf'), dtype=torch.float64)).sort(1).values
    real = torch.isfinite(cat)
    n_cat = real[:, :1].sum(1) + ((cat[:, 1:] != cat[:, :-1]) & real[:, 1:]).sum(1)
    return ild.float(), n_cat.to(torch.int64)
