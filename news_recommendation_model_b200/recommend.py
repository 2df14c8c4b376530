"""Recommendation from a shared article pool: every user against the same N articles, each user's k best unread ones.

The reference scores the [B,C] candidates that come with each impression (test.py, verify.py, train.py).  A recommender is also
used the other way round: take the articles that are live now (for EB-NeRD, the `wire.ArticleTable` already resident on the
device), score all of them for every active user and return each user's k best, leaving out what the user has already read.

    logits = recommend.pool_logits(model, table, hist_article, hist_time, hist_click, pool_time)      # [B, n-1]: every real article
    rec = recommend.top_articles([m1, m2], table, hist_article, hist_time, hist_click, pool_time, 10)  # rec.article [B,10], best first

`pool_logits` runs the eval forward over the pool in chunks (`nrm_forward_pool`): the pool rows are expanded once per chunk and
shared by all users, so the memory is that of a (B, H, chunk) forward, and the logits are, bit for bit, those of
`model.eval()(x_history, x_target, x_global)` with the pool broadcast as every user's candidates.  `top_articles` selects on the
GPU (`nrm_pool_topk`): the score is the logit for one model and, for an ensemble, the mean over the models of the softmax over the
user's eligible articles (test.py:58-63); the order is Python's stable `sorted(..., reverse=True)` (test.py:124-127).  Eligible are
the pool positions whose article id is in [1, n_articles), whose logits are not NaN and, with `exclude_clicked`, whose article
is not among the user's non-pad history ids; duplicate ids in the pool are independent positions."""
from __future__ import annotations

import ctypes
from typing import NamedTuple, Optional

import torch

from . import _lib, engine, wire

TOPK_MAX = 1024
MODELS_MAX = 16
CHUNK_ALIGN = 8                       # the attention's candidate group: every multiple of it gives the same logits
WORKSPACE_TARGET = 1 << 30            # chunk=None: the largest chunk whose workspace stays under 1 GiB


class Recommendations(NamedTuple):
    article: torch.Tensor     # [B,k] int64 pool article ids, best first (-1: fewer than k eligible positions)
    position: torch.Tensor    # [B,k] int64 positions in the pool (-1 likewise)
    score: torch.Tensor       # [B,k] float32 ranking scores (NaN where the position is -1)


def _stream(dev) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _check_k(k, N: int) -> None:
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= min(N, TOPK_MAX):
        raise ValueError(f'k must be an integer in [1, min(N, {TOPK_MAX})] = [1, {min(N, TOPK_MAX)}], got {k!r}')


def _check_users_and_pool(table, hist_article, hist_time, hist_click, pool_time, pool_article, k=None):
    """-> (B, H, N, pool_article); ValueError for shapes / dtypes / layout / k, NrmError for tensors that are not on a CUDA device."""
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
    tensors = (rows, hist_article, hist_time, hist_click, pool_article, pool_time)
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
    cs = _lib.CompactBatchStruct(table.rows.data_ptr(), table.n, hist_article.data_ptr(), hist_time.data_ptr(), hist_click.data_ptr(),
                                 pool_article.data_ptr(), pool_time.data_ptr(), None, None)
    p = engine._ptr
    _lib.check(lib.nrm_forward_pool(ctypes.byref(cs), B, H, N, chunk, p(flat.buf), p(model.bn.running_mean), p(model.bn.running_var),
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
