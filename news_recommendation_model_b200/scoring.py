"""Scoring epilogue and submission text on the GPU — the host side of `test.py`'s scoring loop.

The reference finishes every scoring batch on the host (`test.py:58-71`): ensemble mean of the per-model softmax,
a second softmax over the rows that still hold pad candidates, one `.cpu().numpy()` per impression, and later
(`test.py:118-132`) `thread_num` worker processes that sort each score list in Python to build the rank string.
Here the whole batch stays on the device until ONE copy back:

    scores, ranks = nrm.scoring.ensemble_scores(model_list, x_history, x_inview, x_global, empty_num)
    text = nrm.scoring.submission_text(impression_id, ranks, empty_num)      # bytes of predictions.txt for the batch

`model_test` mirrors `test.py:model_test` (same arguments, same queue records, same id list) and
`write_submission_file` mirrors `test.py:write_submission_file` without the worker processes."""
from __future__ import annotations

import queue as _queue
import zipfile
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .engine import _ptr, _stream


def score_epilogue(logits: torch.Tensor, empty_num: Optional[torch.Tensor] = None, want_ranks: bool = True
                   ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """logits: [M,B,C] (or [B,C]) eval-mode outputs of the M ensemble members on the GPU; empty_num: [B] pad candidates
    left at the end of each row.  Returns (scores float32 [B,C], ranks int32 [B,C] or None) as `test.py:58-70` and
    `test.py:124-127` define them; pad entries hold score 0 and rank -1."""
    if logits.dim() == 2:
        logits = logits.unsqueeze(0)
    if logits.dim() != 3:
        raise ValueError('logits must be [M, B, C] or [B, C]')
    if not logits.is_cuda:
        raise _lib.NrmError('score_epilogue runs on CUDA tensors only (no CPU fallback)')
    x = logits.detach().to(torch.float32).contiguous()
    M, B, C = x.shape
    dev = x.device
    en = None
    if empty_num is not None:
        en = empty_num.detach().to(device=dev, dtype=torch.int64).contiguous()
        if en.shape != (B,):
            raise ValueError('empty_num must be [B]')
    scores = torch.empty(B, C, dtype=torch.float32, device=dev)
    ranks = torch.empty(B, C, dtype=torch.int32, device=dev) if want_ranks else None
    if B == 0 or C == 0:
        return scores, ranks
    _lib.check(_lib.load().nrm_score_epilogue(_ptr(x), M, x.stride(0), x.stride(1), B, C, _ptr(en), _ptr(scores), _ptr(ranks), _stream(dev)),
               'nrm_score_epilogue')
    return scores, ranks


def bucket_plan(n: torch.Tensor, C: int, groups: int = 8, min_group: int = 128):
    """Host-side plan of `ensemble_logits`: `n` [B] = real candidates per impression (CPU int64), C = columns of the batch.
    Returns [(indices, width)]: the impressions sorted by candidate count (stable, descending) cut into up to `groups`
    groups with even boundaries (the kernels work on impression pairs); `width` = longest list of the group + 1 pad column,
    capped at C.  Every impression appears exactly once; an impression with pads always has a pad column inside `width`."""
    B = int(n.numel())
    order = torch.argsort(n, descending=True, stable=True)
    G = max(1, min(int(groups), B // max(1, int(min_group))))
    edges = [((B * g // G) + 1) // 2 * 2 for g in range(G)] + [B]
    plan = []
    for g in range(G):
        lo, hi = edges[g], edges[g + 1]
        if hi > lo:
            idx = order[lo:hi]
            plan.append((idx, min(int(C), int(n[idx].max()) + 1)))
    return plan


@torch.no_grad()
def ensemble_logits(model_list: Sequence[torch.nn.Module], x_history, x_inview, x_global, empty_num=None, groups: int = 8,
                    min_group: int = 128) -> torch.Tensor:
    """Eval-mode logits [M,B,C] of every ensemble member, as `model(x_history, x_inview, x_global)` gives them.

    Pad candidates are all-zero rows (`process_data.py:214-222`), so all pads of an impression have the SAME logit, and
    candidate lists are ragged (median 11, maximum ~100): computing every column of the batch spends most of the time on
    copies of one number.  With `empty_num` given, the impressions are therefore sorted by their number of real candidates
    and scored in up to `groups` groups, each only as wide as its longest list plus one pad column; the pad logit is then
    replicated into the remaining columns.  The result is bit-identical to scoring the full rectangle (rows are independent
    in eval mode; `tests/test_gpu_scoring.py` checks it), so `test.py`'s softmax-over-pads quirk is reproduced exactly."""
    B, C = int(x_inview.shape[0]), int(x_inview.shape[1])
    M = len(model_list)
    dev = x_history.device
    if empty_num is None or B < 2 * min_group or C < 8:
        return torch.stack([m(x_history, x_inview, x_global) for m in model_list], 0)
    n = (C - empty_num.detach().to('cpu', torch.int64)).clamp_(0, C)                # real candidates per impression
    out = torch.empty(M, B, C, dtype=torch.float32, device=dev)
    for idx_cpu, cg in bucket_plan(n, C, groups, min_group):
        idx = idx_cpu.to(dev)
        xh_g = x_history.index_select(0, idx)
        xt_g = x_inview.index_select(0, idx)[:, :cg]
        xg_g = x_global.index_select(0, idx)[:, :cg]
        if cg < C:
            pad_col = n[idx_cpu].to(dev).unsqueeze(1)                               # first pad column of every impression (< cg)
        for mi, m in enumerate(model_list):
            lg = m(xh_g, xt_g, xg_g)
            if cg < C:
                lg = torch.cat((lg, lg.gather(1, pad_col).expand(-1, C - cg)), 1)
            out[mi].index_copy_(0, idx, lg)
    return out


@torch.no_grad()
def ensemble_scores(model_list: Sequence[torch.nn.Module], x_history, x_inview, x_global, empty_num=None, want_ranks: bool = True,
                    groups: int = 8):
    """`test.py:58-70` for one batch: every model's eval forward (ragged-aware, see `ensemble_logits`), then the fused
    epilogue.  `groups=1` scores the full rectangle."""
    logits = ensemble_logits(model_list, x_history, x_inview, x_global, empty_num if groups > 1 else None, groups)
    return score_epilogue(logits, empty_num, want_ranks)


def submission_lines(impression_id: torch.Tensor, ranks: torch.Tensor, empty_num: Optional[torch.Tensor] = None
                     ) -> Tuple[bytes, np.ndarray]:
    """The lines `test.py:129-130` formats, for a whole batch: returns (text, offsets) where line b is
    text[offsets[b]:offsets[b+1]] == b"{impression_id} [{r0},{r1},...]\\n"."""
    if not ranks.is_cuda:
        raise _lib.NrmError('submission_lines runs on CUDA tensors only (no CPU fallback)')
    dev = ranks.device
    rk = ranks.detach().to(torch.int32).contiguous()
    B, C = rk.shape
    if B == 0:
        return b'', np.zeros(1, np.int64)
    ids = impression_id.detach().to(device=dev, dtype=torch.int64).contiguous()
    if ids.shape != (B,):
        raise ValueError('impression_id must be [B]')
    en = None
    if empty_num is not None:
        en = empty_num.detach().to(device=dev, dtype=torch.int64).contiguous()
    lib = _lib.load()
    if C == 0:
        raise ValueError('ranks must have at least one candidate column')
    cap = int(lib.nrm_rank_strings_capacity(B, C))
    out = torch.empty(cap, dtype=torch.uint8, device=dev)
    offsets = torch.empty(B + 1, dtype=torch.int64, device=dev)
    _lib.check(lib.nrm_rank_strings(_ptr(ids), _ptr(rk), _ptr(en), B, C, _ptr(offsets), _ptr(out), cap, _stream(dev)), 'nrm_rank_strings')
    off = offsets.cpu().numpy()
    total = int(off[-1])
    if total > cap:
        raise _lib.NrmError('nrm_rank_strings: text does not fit the buffer')
    return out[:total].cpu().numpy().tobytes(), off


def submission_text(impression_id, ranks, empty_num=None) -> bytes:
    return submission_lines(impression_id, ranks, empty_num)[0]


class SubmissionRing:
    """Pinned result ring for the submission text (`test.py:118-132`) of a scoring loop.  `push` formats one batch on the GPU and
    enqueues the device-to-host copies of the text and its line offsets into the next pinned slot WITHOUT synchronising, so the
    host goes straight on to the next batch; the (text, offsets) of an older batch comes back from `push` once the ring wraps
    (`depth - 1` batches late), the rest from `drain()` — always in push order.  `submission_lines` is the blocking one-batch form."""

    def __init__(self, max_batch: int, max_candidates: int, depth: int = 4, device='cuda'):
        if depth < 2:
            raise ValueError('SubmissionRing needs at least 2 slots')
        self.lib = _lib.load()
        self.dev = torch.device(device)
        self.depth, self.max_batch, self.max_candidates = depth, max_batch, max_candidates
        cap = int(self.lib.nrm_rank_strings_capacity(max_batch, max_candidates))
        self._dtext = [torch.empty(cap, dtype=torch.uint8, device=self.dev) for _ in range(depth)]
        self._doff = [torch.empty(max_batch + 1, dtype=torch.int64, device=self.dev) for _ in range(depth)]
        self._htext = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in range(depth)]
        self._hoff = [torch.empty(max_batch + 1, dtype=torch.int64).pin_memory() for _ in range(depth)]
        self._event = [torch.cuda.Event() for _ in range(depth)]
        self._rows = [0] * depth                      # 0 = slot free
        self._caps = [0] * depth
        self._head = 0                                # next slot to fill
        self._tail = 0                                # oldest slot not yet collected

    def _collect(self) -> Tuple[bytes, np.ndarray]:
        slot = self._tail % self.depth
        self._event[slot].synchronize()
        B = self._rows[slot]
        off = self._hoff[slot][:B + 1].numpy().copy()
        total = int(off[-1])
        if total > self._caps[slot]:
            raise _lib.NrmError('nrm_rank_strings: text does not fit the buffer')
        text = self._htext[slot][:total].numpy().tobytes()
        self._rows[slot] = 0
        self._tail += 1
        return text, off

    def push(self, impression_id: torch.Tensor, ranks: torch.Tensor, empty_num: Optional[torch.Tensor] = None
             ) -> Optional[Tuple[bytes, np.ndarray]]:
        if not ranks.is_cuda:
            raise _lib.NrmError('SubmissionRing runs on CUDA tensors only (no CPU fallback)')
        rk = ranks.detach().to(torch.int32).contiguous()
        B, C = rk.shape
        if B == 0 or C == 0 or B > self.max_batch or C > self.max_candidates:
            raise ValueError(f'ranks [{B},{C}] outside the ring\'s [1..{self.max_batch}, 1..{self.max_candidates}]')
        done = self._collect() if self._head - self._tail == self.depth else None
        slot = self._head % self.depth
        ids = impression_id.detach().to(device=self.dev, dtype=torch.int64, non_blocking=True).contiguous()
        if ids.shape != (B,):
            raise ValueError('impression_id must be [B]')
        en = None if empty_num is None else empty_num.detach().to(device=self.dev, dtype=torch.int64, non_blocking=True).contiguous()
        cap = int(self.lib.nrm_rank_strings_capacity(B, C))
        _lib.check(self.lib.nrm_rank_strings(_ptr(ids), _ptr(rk), _ptr(en), B, C, _ptr(self._doff[slot]), _ptr(self._dtext[slot]), cap,
                                             _stream(self.dev)), 'nrm_rank_strings')
        self._hoff[slot][:B + 1].copy_(self._doff[slot][:B + 1], non_blocking=True)
        self._htext[slot][:cap].copy_(self._dtext[slot][:cap], non_blocking=True)      # the whole capacity: its length is not known on the host yet
        self._event[slot].record(torch.cuda.current_stream(self.dev))
        self._rows[slot], self._caps[slot] = B, cap
        self._head += 1
        return done

    def drain(self) -> List[Tuple[bytes, np.ndarray]]:
        out = []
        while self._tail < self._head:
            out.append(self._collect())
        return out


@torch.no_grad()
def model_test(model_list, test_data, device='cuda', prediction_queue=None, id_list=None, batch_size=1, text_sink: Optional[List[bytes]] = None):
    """Mirror of `test.py:model_test` (`test.py:31-74`): same arguments, the same records
    `[impression_id, user_id, scores (numpy float32, pads dropped), label_id (numpy, pads dropped)]` on `prediction_queue`
    and the same "{impression_id}_{user_id}" strings in `id_list`, in the same order.  Per batch there is one device
    epilogue launch and one copy back instead of one `.cpu()` per impression.  If `text_sink` is a list, the formatted
    submission lines of every batch (`test.py:118-132`) are appended to it as bytes."""
    loader = torch.utils.data.DataLoader(dataset=test_data, batch_size=batch_size, shuffle=False)
    for model in model_list:
        model.eval()
        model.to(device)
    if prediction_queue is None:
        prediction_queue = _queue.Queue()
    if id_list is None:
        id_list = []
    ring = None
    for data in loader:
        impression_id, user_id, x_history, x_inview, x_global, _, label_id, empty_num = data
        trim = int(torch.min(empty_num))
        x_history = x_history.to(device)
        x_inview = x_inview.to(device)
        x_global = x_global.to(device)
        if trim > 0:                                               # test.py:52-56
            x_inview = x_inview[:, 0:-trim]
            x_global = x_global[:, 0:-trim]
            label_id = label_id[:, 0:-trim]
            empty_num = empty_num - trim
        scores, ranks = ensemble_scores(model_list, x_history, x_inview, x_global, empty_num, want_ranks=text_sink is not None)
        if text_sink is not None:                                  # the text comes back through a pinned ring, a few batches late
            if ring is None or ranks.shape[0] > ring.max_batch or ranks.shape[1] > ring.max_candidates:
                if ring is not None:
                    text_sink.extend(t for t, _ in ring.drain())
                ring = SubmissionRing(max(ranks.shape[0], batch_size), max(ranks.shape[1], 64), device=ranks.device)
            done = ring.push(impression_id, ranks, empty_num)
            if done is not None:
                text_sink.append(done[0])
        host = scores.cpu().numpy()
        for d_i in range(host.shape[0]):
            n = host.shape[1] - int(empty_num[d_i])
            prediction_queue.put([impression_id[d_i], user_id[d_i], host[d_i, :n].copy(), label_id[d_i, :n].numpy()])
            id_list.append('{}_{}'.format(int(impression_id[d_i]), int(user_id[d_i])))
    if ring is not None:
        text_sink.extend(t for t, _ in ring.drain())
    return prediction_queue, id_list


@torch.no_grad()
def model_validation(model_list, validation_data, device='cuda', batch_size=1):
    """Mirror of `verify.py:model_validation` (`verify.py:19-42`): returns `[auc, tpr]` = mean per-impression ROC AUC
    (`tool/evaluation.py:3-5`, ties averaged) of the ensemble scores and the fraction of impressions whose best-scored
    candidate is the clicked one (`verify.py:32`, `tool/evaluation.py:16-17`).  Scores, AUC and hits are computed on the
    GPU per batch (`ensemble_scores`, `metrics.batch_metrics`); one number pair comes back at the end instead of one
    sklearn call per impression."""
    from . import metrics
    loader = torch.utils.data.DataLoader(dataset=validation_data, batch_size=batch_size, shuffle=False)
    for model in model_list:
        model.eval()
        model.to(device)
    auc_sum = torch.zeros((), dtype=torch.float64, device=device)
    hit_sum = torch.zeros((), dtype=torch.float64, device=device)
    count = 0
    for data in loader:
        _, _, x_history, x_inview, x_global, label, _, empty_num = data
        trim = int(torch.min(empty_num))
        x_history, x_inview, x_global, label = x_history.to(device), x_inview.to(device), x_global.to(device), label.to(device)
        if trim > 0:                                               # test.py:52-56
            x_inview, x_global, label = x_inview[:, 0:-trim], x_global[:, 0:-trim], label[:, 0:-trim]
            empty_num = empty_num - trim
        scores, _ = ensemble_scores(model_list, x_history, x_inview, x_global, empty_num, want_ranks=False)
        n_valid = (scores.shape[1] - empty_num).to(device)
        m = metrics.batch_metrics(scores, label, n_valid)
        auc_sum += m['auc'].double().sum()
        hit_sum += m['hit'].double().sum()
        count += int(scores.shape[0])
    return [float(auc_sum) / max(count, 1), float(hit_sum) / max(count, 1)]


def write_submission_file(text_chunks: Sequence[bytes], path: str, name: str = 'predictions') -> str:
    """`test.py:write_submission_file` (`test.py:76-116`) for text that `model_test(text_sink=...)` already formatted:
    writes `path + "predictions.txt"` and zips it to `path + name + ".zip"`."""
    file_path = path + 'predictions.txt'
    zip_path = path + '{}.zip'.format(name)
    with open(file_path, 'wb') as f:
        for chunk in text_chunks:
            f.write(chunk)
    with zipfile.ZipFile(zip_path, 'w', zipfile.ZIP_DEFLATED) as z:
        z.write(file_path, arcname=file_path.split('/')[-1])
    return zip_path
