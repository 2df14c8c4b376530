"""Attention scores as an output: "which past clicks made the model rank this article high?"

The reference's model is DIN-style: for every (candidate, clicked article) pair each of its two pointwise attentions computes a
score, `s_label = label_attention(x_label_t, x_label_h)` and `s_ti = text_img_attention(pca_t, pca_h)`, both [B,C,H,1]
(`user_invariant_interest_model.py:83-87`, `PointwiseAttentionExpanded.forward`, `attention_model.py:52-97`), and pools the
history rows with them.  `attention_scores` returns those scores, computed by the same kernels as the logits in one eval-mode
forward (`nrm_forward_scores`): the [B,C,H,64] label projection of the history the scores depend on never leaves the kernels.
`top_history` turns them into the k history clicks that drove each candidate (`nrm_history_topk`, on the GPU).

    s = explain.attention_scores(model, x_history, x_target, x_global)     # logits [B,C], label / text_img [B,C,H]
    top = explain.top_history(s, 5, x_history=x_history)                   # label_idx [B,C,5] ... pad rows left out

Pad history rows get scores too, and they enter the pooled sum, because the reference does not mask them (an all-zero packed
row embeds as the id-0 rows of the embedding tables, so its label features are not zero); `top_history` leaves them out when it
is told where they are."""
from __future__ import annotations

from typing import NamedTuple, Optional, Union

import torch

from . import _lib, engine, wire
from .config import HIST_COLS
from .engine import _ptr, _stream

TOPK_MAX = 64


class AttentionScores(NamedTuple):
    logits: torch.Tensor      # [B,C] float32, bit-identical to model.eval()(...) in the model's precision
    label: torch.Tensor       # [B,C,H] float32: label_attention scores
    text_img: torch.Tensor    # [B,C,H] float32: text_img_attention scores


class HistoryTopK(NamedTuple):
    label_idx: torch.Tensor       # [B,C,k] int64 history positions, best first (-1: fewer than k real clicks)
    label_score: torch.Tensor     # [B,C,k] float32 (NaN where the index is -1)
    text_img_idx: torch.Tensor
    text_img_score: torch.Tensor


def _scores(model, inputs, B, H, C, dev) -> AttentionScores:
    """One eval-mode `nrm_forward_scores` of `inputs` (an engine binding)."""
    with torch.no_grad():
        flat = model.flat_parameters()
        if flat.device != dev:
            raise _lib.NrmError(f'model is on {flat.device} but inputs are on {dev}')
        ws = model._runtime().workspace(B, H, C, engine.MODE_EVAL, dev)
        logits = torch.empty(B, C, dtype=torch.float32, device=dev)
        scores = torch.empty(2, B, C, H, dtype=torch.float32, device=dev)
        engine.call(inputs, 'nrm_forward_scores', B, H, C, _ptr(flat.buf), _ptr(model.bn.running_mean), _ptr(model.bn.running_var),
                    _ptr(model.bn.num_batches_tracked), engine.MODE_EVAL, model._precision_code(), _ptr(logits), _ptr(scores), _ptr(ws),
                    ws.numel(), _stream(dev))
    return AttentionScores(logits, scores[0], scores[1])


def attention_scores(model, x_history, x_target, x_global) -> AttentionScores:
    """Logits and both branches' attention scores of `model` (a `UserModel`) for the reference's packed float64 inputs
    (`x_target` / `x_global` may be the column-trimmed views of test.py:53-54).

    Always eval semantics, whatever `model.training` says: BatchNorm normalises with its running statistics and they are
    neither read as batch statistics nor updated, so explaining a batch in the middle of training does not move the model.
    Runs under `torch.no_grad()` in the model's precision; the logits equal `model.eval()(x_history, x_target, x_global)`
    bit for bit."""
    with torch.no_grad():
        inputs = engine.prepare_inputs(x_history, x_target, x_global)
    return _scores(model, inputs, x_history.shape[0], x_history.shape[1], x_target.shape[1], inputs.xh.device)


def attention_scores_compact(model, table: wire.ArticleTable, cb: wire.CompactBatch) -> AttentionScores:
    """`attention_scores` for a device `wire.CompactBatch` and its `ArticleTable`: the row kernels read the compact format
    directly (`nrm_forward_scores_compact`).  Same results, bit for bit, as `attention_scores` on `wire.expand(table, cb)`."""
    if not (table.rows.is_cuda and cb.hist_article.is_cuda):
        raise _lib.NrmError('attention_scores_compact runs on CUDA tensors only (no CPU fallback)')
    if table.rows.dtype != torch.float32 or table.rows.dim() != 2 or table.rows.shape[1] != wire.ARTICLE_COLS \
            or not table.rows.is_contiguous():
        raise ValueError(f'article table must be contiguous float32 [n, {wire.ARTICLE_COLS}]')
    B, H, C = cb.shape
    for t, shape, dt in ((cb.hist_article, (B, H), torch.int32), (cb.hist_time, (B, H), torch.int32),
                         (cb.hist_click, (B, H, 2), torch.float32), (cb.cand_article, (B, C), torch.int32),
                         (cb.cand_time, (B, C), torch.int32)):
        if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous() or t.device != cb.hist_article.device:
            raise ValueError('CompactBatch tensors must be contiguous int32 / float32 [B,H] / [B,H,2] / [B,C] on one device')
    return _scores(model, engine.compact(table, cb), B, H, C, cb.hist_article.device)


def top_history(scores: Union[AttentionScores, torch.Tensor], k: int, *, x_history: Optional[torch.Tensor] = None,
                hist_article: Optional[torch.Tensor] = None) -> HistoryTopK:
    """The `k` history positions with the largest scores for every candidate, per branch, best first; ties go to the lower
    position (Python's stable `sorted(..., reverse=True)`, as test.py:124-127 ranks candidates).

    `scores`: what `attention_scores` returned, or a [2,B,C,H] float32 tensor (branch 0 = label).  Pad history rows are left
    out when one of `x_history` (packed [B,H,80]: all-zero rows are the ETL's padding) or `hist_article` (compact [B,H]: id 0)
    is given; when an impression has fewer than `k` real clicks the remaining slots hold index -1 and score NaN.
    1 <= k <= min(H, 64)."""
    if isinstance(scores, AttentionScores):
        if scores.label.dim() != 3 or scores.label.shape != scores.text_img.shape:
            raise ValueError('AttentionScores.label / text_img must both be [B,C,H]')
        s = torch.stack((scores.label, scores.text_img))
    else:
        s = scores
    if s.dim() != 4 or s.shape[0] != 2:
        raise ValueError(f'scores must be [2,B,C,H], got {tuple(s.shape)}')
    _, B, C, H = s.shape
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= min(H, TOPK_MAX):
        raise ValueError(f'k must be an integer in [1, min(H, {TOPK_MAX})] = [1, {min(H, TOPK_MAX)}], got {k!r}')
    if x_history is not None and hist_article is not None:
        raise ValueError('pass at most one of x_history / hist_article')
    if x_history is not None and (x_history.dim() != 3 or tuple(x_history.shape) != (B, H, HIST_COLS)):
        raise ValueError(f'x_history must be [B,H,{HIST_COLS}] = [{B},{H},{HIST_COLS}], got {tuple(x_history.shape)}')
    if hist_article is not None and tuple(hist_article.shape) != (B, H):
        raise ValueError(f'hist_article must be [B,H] = [{B},{H}], got {tuple(hist_article.shape)}')
    for t in (s, x_history, hist_article):
        if t is not None and not t.is_cuda:
            raise _lib.NrmError('top_history runs on CUDA tensors only (no CPU fallback)')
        if t is not None and t.device != s.device:
            raise ValueError('scores and the pad-row source must be on the same device')
    s = s.to(torch.float32).contiguous()
    xh = x_history.to(torch.float64).contiguous() if x_history is not None else None
    ha = hist_article.to(torch.int32).contiguous() if hist_article is not None else None
    dev = s.device
    idx = torch.empty(2, B, C, k, dtype=torch.int32, device=dev)
    val = torch.empty(2, B, C, k, dtype=torch.float32, device=dev)
    p = engine._ptr
    _lib.check(_lib.load().nrm_history_topk(p(s), B, C, H, k, p(xh), p(ha), p(idx), p(val), _stream(dev)), 'nrm_history_topk')
    idx = idx.to(torch.int64)
    return HistoryTopK(idx[0], val[0], idx[1], val[1])
