"""Pool negatives for training: k extra candidates per impression, drawn from an article pool on the GPU.

An impression's own candidates are the few articles shown next to the click; a model trained on them alone is never asked to
push down the rest of the pool that `recommend.top_articles` ranks.  `NegativeSampler` appends k negatives drawn from the pool
(`nrm_sample_negatives`, one warp per impression).  `FusedTrainStep(..., negatives=sampler)` runs it at the start of every step,
inside the captured graph, with the step counter read on the device; `sample` is the standalone form
(`wire.expand(table, sampler.sample(cb, step))` -> `model(...)`).

Rules (include/nrm_b200.h states them for the kernel):

* Pool: `pool_article` int32 [N], default every real article 1..n-1 of the table.  Weights: non-negative integers [N], None =
  uniform; a position whose id is outside [1, n) has weight 0.  Position n is drawn with probability weight(n) / total.
* Draw: attempt a of impression b at step t takes u = the first 64 bits of Philox4x32-10(counter (a, row_offset + b, t lo, t hi),
  key (seed lo, seed hi)), r = (u * total) >> 64, and the first position whose inclusive weight prefix sum exceeds r.
* Eligibility: an id already in the impression's history, its own candidates or its accepted negatives is rejected.  Attempts
  run in order; the i-th accepted id fills column C0 + i; sampling stops after k acceptances or 32 k attempts, and what is left
  are pad columns (article 0, time 0, label 0).
* Time: a negative carries the time of the impression's first positive column, so the model cannot tell it from the click by
  age (time-matched negatives).  An impression without a positive gets k pad columns.
* Step: t counts completed optimizer steps.  A run resumed from `FusedTrainStep.state_dict()` draws what the uninterrupted run
  would have drawn.  Rows: `row_offset` is rank * B under data parallelism, so N ranks x B impressions draw what one process on
  N * B impressions draws.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from .engine import _ptr, _stream
from .wire import ArticleTable, CompactBatch

K_MAX = 64
SET_MAX = 16384           # H + C0 + k: the entries of the kernel's per-impression exclusion table
TOTAL_MAX = 1 << 62


class NegativeSampler:
    """Draws `k` pool negatives per impression (1 <= k <= 64) with a 64-bit `seed`.

    `table`: the `wire.ArticleTable` the batches index.  `pool_article`: int32 [N] article ids (default: 1..table.n-1).
    `weights`: non-negative integer [N] (default: uniform).  The int64 prefix sum `cdf` of the weights is built once, on the
    table's device, with ids outside [1, table.n) at weight 0; a total of 0 or above 2^62 raises ValueError."""

    def __init__(self, table: ArticleTable, k: int = 4, seed: int = 0, pool_article: Optional[torch.Tensor] = None,
                 weights: Optional[torch.Tensor] = None):
        if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= K_MAX:
            raise ValueError(f'k must be an integer in [1, {K_MAX}] (got {k!r})')
        if isinstance(seed, bool) or not isinstance(seed, int) or not 0 <= seed < 1 << 64:
            raise ValueError(f'seed must be an integer in [0, 2^64) (got {seed!r})')
        dev = table.rows.device
        n = table.n
        if pool_article is None:
            pool_article = torch.arange(1, n, dtype=torch.int32, device=dev)
        if pool_article.dim() != 1 or pool_article.numel() == 0 or pool_article.dtype != torch.int32:
            raise ValueError('pool_article must be a non-empty int32 [N] tensor')
        if pool_article.numel() >= 1 << 31:
            raise ValueError('the pool holds at most 2^31 - 1 positions')
        pool_article = pool_article.to(dev).contiguous()
        in_range = (pool_article >= 1) & (pool_article < n)
        if weights is None:
            w = in_range.to(torch.int64)
        else:
            if weights.dim() != 1 or weights.numel() != pool_article.numel():
                raise ValueError(f'weights must be [N] = [{pool_article.numel()}] (got {tuple(weights.shape)})')
            if weights.dtype.is_floating_point or weights.dtype.is_complex or weights.dtype == torch.bool:
                raise ValueError(f'weights must be an integer tensor (got {weights.dtype})')
            w = weights.to(device=dev, dtype=torch.int64)
            if bool((w < 0).any()):
                raise ValueError('weights must be non-negative')
            w = torch.where(in_range, w, torch.zeros_like(w))
            # the int64 prefix sum below must not wrap: bound the total in float64 first (relative error < 2^-20 for N < 2^31)
            if float(w.to(torch.float64).sum()) > TOTAL_MAX * (1 + 2.0 ** -20):
                raise ValueError('the total weight exceeds 2^62')
        cdf = torch.cumsum(w, 0)
        total = int(cdf[-1])
        if total == 0 or total > TOTAL_MAX:
            raise ValueError(f'the total weight of the pool must be in [1, 2^62] (got {total}); ids outside [1, {n}) weigh 0')
        self.table, self.k, self.seed = table, k, seed
        self.pool_article, self.cdf, self.total = pool_article, cdf, total

    @property
    def N(self) -> int:
        return int(self.pool_article.numel())

    def sample_into(self, cb: CompactBatch, C0: int, step: torch.Tensor, row_offset: int = 0, rows: Optional[int] = None) -> None:
        """Enqueue the kernel on the current stream: fill columns C0..C0+k-1 of the device batch `cb` ([B, C0 + k] candidate
        arrays) from its first C0 columns, for its first `rows` impressions (default all).  `step`: int64 device tensor whose
        first element is t."""
        B, H, C = cb.shape
        rows = B if rows is None else rows
        if C != C0 + self.k:
            raise ValueError(f'the batch has {C} candidate columns; this sampler needs C0 + k = {C0} + {self.k}')
        if not (cb.hist_article.is_cuda and self.cdf.is_cuda and step.is_cuda):
            raise _lib.NrmError('NegativeSampler runs on CUDA tensors only (no CPU fallback)')
        if cb.hist_article.device != self.cdf.device:
            raise ValueError(f'the batch is on {cb.hist_article.device}, the sampler on {self.cdf.device}')
        if step.dtype != torch.int64:
            raise ValueError('step must be an int64 device tensor')
        for t, dt in ((cb.hist_article, torch.int32), (cb.cand_article, torch.int32), (cb.cand_time, torch.int32), (cb.label, torch.float32)):
            if t.dtype != dt or not t.is_contiguous():
                raise ValueError('CompactBatch tensors must be contiguous int32 / float32 as documented')
        _lib.check(_lib.load().nrm_sample_negatives(_ptr(cb.hist_article), H, _ptr(cb.cand_article), _ptr(cb.cand_time), _ptr(cb.label),
                                                    rows, C, C0, _ptr(self.pool_article), _ptr(self.cdf), self.N, self.table.n, self.seed,
                                                    _ptr(step), row_offset, _stream(self.cdf.device)), 'nrm_sample_negatives')

    def sample(self, cb: CompactBatch, step: int = 0, row_offset: int = 0) -> CompactBatch:
        """Device CompactBatch [B,C0] -> a new device CompactBatch [B,C0+k]: columns 0..C0-1 as in `cb`, then the negatives.  The
        new batch shares `cb`'s history, user and impression tensors; `empty_num` counts the appended pad columns too."""
        if isinstance(step, bool) or not isinstance(step, int) or not 0 <= step < 1 << 63:
            raise ValueError(f'step must be an integer in [0, 2^63) (got {step!r})')
        B, H, C0 = cb.shape
        dev = cb.cand_article.device
        widen = lambda t: torch.cat((t, t.new_zeros(B, self.k)), 1)          # noqa: E731
        out = CompactBatch(cb.impression_id, cb.user_id, cb.hist_article, cb.hist_time, cb.hist_click, widen(cb.cand_article),
                           widen(cb.cand_time), widen(cb.label), cb.empty_num)
        self.sample_into(out, C0, torch.tensor([step], dtype=torch.int64, device=dev), row_offset)
        out.empty_num = cb.empty_num + (out.cand_article[:, C0:] == 0).sum(1)
        return out
