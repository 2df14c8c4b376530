"""Pipelined training step: the train.py:66-75 loop body as one replayable unit.

`train.py` runs, per batch: H2D of the float64 features, `model(...)`, `model.loss(...)`,
`loss.backward()`, `optimizer.step()`, `optimizer.zero_grad()`, then reads `loss.item()`.
Driven from Python that is ~60 kernel launches through autograd plus a device sync per
step.  `FusedTrainStep` keeps the same arithmetic (the same C-ABI calls in the same order on
the same flat buffers) but

  * stages the batch into one of two static device slots on a copy stream, so the H2D of
    batch i+1 overlaps the compute of batch i;
  * captures the five calls (forward, loss, loss backward, backward, Adam) of each slot in a
    CUDA graph and replays it with a single launch;
  * returns the loss through a pinned host ring, read one step late, so the host never
    stalls the pipeline.

Under data parallelism the graph is split around the gradient all-reduce.
"""
from __future__ import annotations

import ctypes
import struct
from typing import List, Optional

import torch

from . import _lib, engine
from .config import HIST_COLS, TGT_COLS, GLOBAL_COLS

_p = engine._ptr


class _Slot:
    def __init__(self, B, H, C, dev):
        self.xh = torch.empty(B, H, HIST_COLS, dtype=torch.float64, device=dev)
        self.xt = torch.empty(B, C, TGT_COLS, dtype=torch.float64, device=dev)
        self.xg = torch.empty(B, C, GLOBAL_COLS, dtype=torch.float64, device=dev)
        self.label = torch.empty(B, C, dtype=torch.float64, device=dev)
        self.uid = torch.empty(B, dtype=torch.int64, device=dev)
        self.ready = torch.cuda.Event()        # H2D of this slot finished
        self.consumed = torch.cuda.Event()     # compute that read this slot finished
        self.graph_fb: Optional[torch.cuda.CUDAGraph] = None
        self.graph_adam: Optional[torch.cuda.CUDAGraph] = None
        self.used = False
        self.compact = None                    # device CompactBatch staging buffers (wire.py), allocated on first use
        self.wire = 'packed'                   # what the last load() put into this slot
        self.rows = B                          # impressions the last load() put into this slot (< B: ragged last batch)
        self.graph_wire = None                 # wire format the captured graph was recorded for


class LossHandle:
    """Result of one step; `.item()` waits for that step only.  The values live in a pinned ring of `ring` (default 8)
    entries: read a handle before `ring` more steps have been enqueued."""

    def __init__(self, host_slot: torch.Tensor, event: torch.cuda.Event):
        self._host, self._event = host_slot, event

    def item(self) -> float:
        self._event.synchronize()
        return float(self._host.item())


class FusedTrainStep:
    SYNC_BN = True          # DataParallel(sync_bn=True) is supported on this path (tests/dp_check.py looks at this flag)
    SPARSE_DELTA_MIN = 65536

    def __init__(self, model, B: int, H: int, C: int, *, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-5,
                 alpha=0.95, use_graph=True, ring=8, nslots=2, articles=None):
        """`articles`: a device `wire.ArticleTable`; with it `load()` also accepts `wire.CompactBatch`es (ids instead of
        packed float64 rows) and the step starts with the expansion kernel."""
        self.model, self.B, self.H, self.C, self.alpha = model, B, H, C, float(alpha)
        self.articles = articles
        self.flat = model.flat_parameters()
        dev = self.flat.device
        self.dev, self.lib = dev, _lib.load()
        self.dp = model._dp
        world = self.dp.world if self.dp is not None else 1
        self.precision = model._precision_code()
        self.mode = engine.MODE_BN_BATCH_STATS | engine.MODE_KEEP_FOR_BWD
        # compact batches go straight into the row kernels (no expansion to the packed float64 tensors) in the tensor-core precisions;
        # the FFMA attention of precision fp32 reads the packed rows, so it gets nrm_expand_compact in front
        self.compact_direct = self.precision != 0
        n = self.flat.total
        # data parallel: the flat gradient buffer in symmetric (peer-mapped) memory, so that the Adam kernel of every rank can read
        # all of them (dp.PeerContext); None -> NCCL all-reduce between two graphs
        # user tables beyond SPARSE_DELTA_MIN entries: delta's gradient (<= B non-zeros per rank) travels as (user id, value) lists
        self.sparse_delta = self.dp is not None and self.flat.delta_numel >= self.SPARSE_DELTA_MIN
        self.peer = None
        if self.dp is not None:
            self.peer = self.dp.peer_context(n, dev, B, self.flat.fixed, self.flat.delta_numel if self.sparse_delta else 0)
        self.sparse_delta = self.sparse_delta and self.peer is not None
        self.grads = self.peer.grads if self.peer is not None else torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        # AdamDeviceState: int64 step | lr, beta1, beta2, eps, wd, grad_scale, step_size, bc2_sqrt
        raw = struct.pack('<q8f', 0, lr, betas[0], betas[1], eps, weight_decay, 1.0, 0.0, 0.0)
        self.adam_state = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
        ws_bytes = int(self.lib.nrm_workspace_bytes(B, H, C, self.mode))
        self.ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        ls_bytes = int(self.lib.nrm_loss_scratch_bytes(B, C))
        self.loss_scratch = torch.zeros(ls_bytes, dtype=torch.uint8, device=dev)    # zero once: holds an arrival counter
        self.logits = torch.empty(B, C, dtype=torch.float32, device=dev)
        self.dlogits = torch.empty(B, C, dtype=torch.float32, device=dev)
        self.one = torch.ones((), dtype=torch.float32, device=dev)
        self.loss_dev = torch.zeros(ring, dtype=torch.float32, device=dev)
        self.loss_host = torch.zeros(ring, dtype=torch.float32).pin_memory()
        self.ring, self.count = ring, 0
        self.slots: List[_Slot] = [_Slot(B, H, C, dev) for _ in range(nslots)]
        self.loaded = 0
        self.copy_stream = torch.cuda.Stream(dev)
        # NCCL collectives between the halves of a synchronised-BatchNorm step are issued eagerly: no graph on that (fallback) path
        self.use_graph = use_graph and not (self.dp is not None and self.dp.sync_bn and self.peer is None)
        self.one_graph = self.dp is None or self.peer is not None
        self.world = world
        self._tail_scratch = {}
        self._warmup()

    def _warmup(self):
        """Run every kernel of the step once on scratch state (zero inputs, cloned BatchNorm buffers
        and optimizer state) so that module loading and function attributes are settled before
        the first graph capture.  Leaves the model, the gradients and Adam untouched."""
        lib, m, f, s = self.lib, self.model, self.flat, self.slots[0]
        for t in (s.xh, s.xt, s.xg, s.label, s.uid):
            t.zero_()
        saved = (m.bn.running_mean.clone(), m.bn.running_var.clone(), m.bn.num_batches_tracked.clone())
        scratch_loss = self.loss_dev.new_zeros(())
        n0 = lib.nrm_launch_count()
        self._warming = True                  # no cross-rank flags during the warm-up pass: their epochs belong to real steps
        self._forward_backward(s, scratch_loss)
        self._warming = False
        if self.peer is not None:
            _lib.check(lib.nrm_peer_preload(), 'nrm_peer_preload')      # load the peer kernels outside any graph capture
        self.launches_per_step = int(lib.nrm_launch_count() - n0) + 2      # + Adam prepare / update
        with torch.no_grad():
            m.bn.running_mean.copy_(saved[0]); m.bn.running_var.copy_(saved[1]); m.bn.num_batches_tracked.copy_(saved[2])
        self.grads.zero_()
        st = self.adam_state.clone()
        tiny = [torch.zeros(4, dtype=torch.float32, device=self.dev) for _ in range(4)]
        _lib.check(lib.nrm_adam_step_device(_p(tiny[0]), _p(tiny[1]), _p(tiny[2]), _p(tiny[3]), 4, _p(st),
                                            engine._stream(self.dev)), 'nrm_adam_step_device')
        torch.cuda.synchronize(self.dev)

    # ---- the five C-ABI calls of one step (train.py:69-75) --------------------------------
    def _forward_backward(self, s: _Slot, loss_out: torch.Tensor, B: Optional[int] = None, loss_scratch: Optional[torch.Tensor] = None):
        """B < self.B: a ragged last batch in the first B rows of the slot (eager only; its own zeroed loss scratch)."""
        lib, m, f = self.lib, self.model, self.flat
        st = engine._stream(self.dev)
        H, C = self.H, self.C
        B = self.B if B is None else B
        loss_scratch = self.loss_scratch if loss_scratch is None else loss_scratch
        warming = getattr(self, '_warming', False)
        sync_bn = self.dp is not None and self.dp.sync_bn and not warming
        direct = s.wire == 'compact' and self.compact_direct          # the slot's compact batch is the input itself
        cb = ctypes.byref(s.cstruct) if direct else None
        if not sync_bn:
            if direct:
                _lib.check(lib.nrm_forward_compact(cb, B, H, C, _p(f.buf), _p(m.bn.running_mean), _p(m.bn.running_var),
                                                   _p(m.bn.num_batches_tracked), self.mode, self.precision, _p(self.logits), _p(self.ws),
                                                   self.ws.numel(), st), 'nrm_forward_compact')
            else:
                _lib.check(lib.nrm_forward(_p(s.xh), _p(s.xt), C * TGT_COLS, _p(s.xg), C * GLOBAL_COLS, B, H, C, _p(f.buf),
                                           _p(m.bn.running_mean), _p(m.bn.running_var), _p(m.bn.num_batches_tracked), self.mode,
                                           self.precision, _p(self.logits), _p(self.ws), self.ws.numel(), st), 'nrm_forward')
        else:
            # synchronised BatchNorm: the two halves of the forward around the exchange of the column sums (2 x 264 doubles);
            # N ranks x B impressions then reproduce one process on N * B
            sums = self._bn_sums(0)
            if direct:
                _lib.check(lib.nrm_forward_encoder_compact(cb, B, H, C, _p(f.buf), self.mode, self.precision, _p(sums), _p(self.ws),
                                                           self.ws.numel(), st), 'nrm_forward_encoder_compact')
            else:
                _lib.check(lib.nrm_forward_encoder(_p(s.xh), _p(s.xt), C * TGT_COLS, _p(s.xg), C * GLOBAL_COLS, B, H, C, _p(f.buf), self.mode,
                                                   self.precision, _p(sums), _p(self.ws), self.ws.numel(), st), 'nrm_forward_encoder')
            gsums = self._exchange_stats(0, sums, B * C)
            _lib.check(lib.nrm_forward_head(B, H, C, _p(f.buf), _p(m.bn.running_mean), _p(m.bn.running_var), _p(m.bn.num_batches_tracked),
                                            self.mode, self.precision, _p(gsums), B * C * self.world, _p(self.logits), _p(self.ws), self.ws.numel(), st),
                       'nrm_forward_head')
        delta = f.buf[f.fixed:f.fixed + f.delta_numel]
        _lib.check(lib.nrm_loss_forward(_p(self.logits), _p(delta), f.delta_numel, _p(s.uid), _p(s.label), B, C, self.alpha, _p(loss_out),
                                        _p(loss_scratch), loss_scratch.numel(), st), 'nrm_loss_forward')
        if self.peer is not None and not warming:
            # before anything of this step is written into the gradient buffer: every peer has consumed the previous step's
            _lib.check(lib.nrm_peer_wait_consumed(_p(self.adam_state), _p(self.peer.ctx), st), 'nrm_peer_wait_consumed')
        if self.sparse_delta and not warming:
            _lib.check(lib.nrm_loss_backward_sparse(_p(s.uid), B, C, _p(self.one), _p(self.dlogits), f.delta_numel, _p(self.peer.sparse_uid),
                                                    _p(self.peer.sparse_val), _p(loss_scratch), loss_scratch.numel(), st), 'nrm_loss_backward_sparse')
        else:
            ddelta = self.grads[f.fixed:f.fixed + f.delta_numel]
            _lib.check(lib.nrm_loss_backward(_p(s.uid), B, C, _p(self.one), _p(self.dlogits), _p(ddelta), f.delta_numel,
                                             _p(loss_scratch), loss_scratch.numel(), st), 'nrm_loss_backward')
        if not sync_bn:
            if direct:
                _lib.check(lib.nrm_backward_compact(cb, B, H, C, _p(f.buf), self.mode, self.precision, _p(self.dlogits), _p(self.grads),
                                                    _p(self.ws), self.ws.numel(), st), 'nrm_backward_compact')
            else:
                _lib.check(lib.nrm_backward(_p(s.xh), _p(s.xt), C * TGT_COLS, _p(s.xg), C * GLOBAL_COLS, B, H, C, _p(f.buf), self.mode,
                                            self.precision, _p(self.dlogits), _p(self.grads), _p(self.ws), self.ws.numel(), st),
                           'nrm_backward')
        else:
            sums = self._bn_sums(1)
            # head weight gradients stay on the library's side stream until the encoder backward has been enqueued
            _lib.check(lib.nrm_backward_head_deferred(B, H, C, _p(f.buf), self.precision, _p(self.dlogits), _p(self.grads), _p(sums), _p(self.ws),
                                                      self.ws.numel(), st), 'nrm_backward_head_deferred')
            gsums = self._exchange_stats(1, sums, B * C)
            if direct:
                _lib.check(lib.nrm_backward_encoder_compact(cb, B, H, C, _p(f.buf), self.mode, self.precision, _p(gsums), B * C * self.world,
                                                            _p(self.grads), _p(self.ws), self.ws.numel(), st), 'nrm_backward_encoder_compact')
            else:
                _lib.check(lib.nrm_backward_encoder(_p(s.xh), _p(s.xt), C * TGT_COLS, _p(s.xg), C * GLOBAL_COLS, B, H, C, _p(f.buf), self.mode,
                                                    self.precision, _p(gsums), B * C * self.world, _p(self.grads), _p(self.ws), self.ws.numel(), st),
                           'nrm_backward_encoder')

    def _bn_sums(self, which: int) -> torch.Tensor:
        if self.peer is not None:
            return self.peer.stats_local[which]
        if not hasattr(self, '_sums_local'):
            self._sums_local = torch.zeros(2, 528, dtype=torch.float64, device=self.dev)
        return self._sums_local[which]

    def _exchange_stats(self, which: int, sums: torch.Tensor, local_rows: int) -> torch.Tensor:
        """Sum the BatchNorm statistics over the ranks: one small kernel over peer memory (graph-safe), else an NCCL all-reduce."""
        if self.peer is not None:
            out = self.peer.stats_out[which]
            _lib.check(self.lib.nrm_peer_allsum_stats(_p(sums), which, _p(out), _p(self.adam_state), _p(self.peer.ctx),
                                                      engine._stream(self.dev)), 'nrm_peer_allsum_stats')
            return out
        self.dp.all_reduce_stats(sums, local_rows)
        return sums

    def _adam(self):
        if self.peer is not None:            # gradient average over the ranks fused into the update (peer memory)
            _lib.check(self.lib.nrm_adam_step_allreduce(_p(self.flat.buf), _p(self.exp_avg), _p(self.exp_avg_sq), self.flat.total,
                                                        _p(self.adam_state), _p(self.peer.ctx), _p(self.peer.ticket), engine._stream(self.dev)),
                       'nrm_adam_step_allreduce')
            return
        _lib.check(self.lib.nrm_adam_step_device(_p(self.flat.buf), _p(self.grads), _p(self.exp_avg), _p(self.exp_avg_sq),
                                                 self.flat.total, _p(self.adam_state), engine._stream(self.dev)),
                   'nrm_adam_step_device')

    # ---- optimizer state: what torch.optim.Adam + LambdaLR give the reference loop (train.py:48-49) --------------------
    _ADAM_FIELDS = ('lr', 'beta1', 'beta2', 'eps', 'weight_decay', 'grad_scale')

    def _adam_host(self):
        step, lr, b1, b2, eps, wd, gs, _, _ = struct.unpack('<q8f', bytes(self.adam_state.cpu().numpy().tobytes()))
        return {'step': step, 'lr': lr, 'beta1': b1, 'beta2': b2, 'eps': eps, 'weight_decay': wd, 'grad_scale': gs}

    def set_hyper(self, **kw):
        """Change lr / beta1 / beta2 / eps / weight_decay / grad_scale between steps (e.g. the 0.65 ** epoch schedule of
        train.py:49).  The captured graphs stay valid: the Adam kernel reads these values from device memory; the new values
        are written with one small async copy on the current stream, i.e. in order with the steps."""
        unknown = set(kw) - set(self._ADAM_FIELDS)
        if unknown:
            raise ValueError(f'unknown Adam hyper-parameter(s): {sorted(unknown)}')
        cur = self._adam_host() if len(kw) < len(self._ADAM_FIELDS) else {}
        cur.update({k: float(v) for k, v in kw.items()})
        raw = struct.pack('<6f', *[cur[k] for k in self._ADAM_FIELDS])
        host = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
        self.adam_state[8:32].copy_(host.to(self.dev, non_blocking=False))

    def set_lr(self, lr: float):
        self.set_hyper(lr=lr)

    def state_dict(self):
        """Optimizer state for checkpoint / resume: flat moments (same layout as the flat parameter buffer), step and the
        hyper-parameters.  Model weights and BatchNorm buffers are in model.state_dict() as usual."""
        torch.cuda.current_stream(self.dev).synchronize()
        return {'exp_avg': self.exp_avg.detach().clone(), 'exp_avg_sq': self.exp_avg_sq.detach().clone(), **self._adam_host(),
                'layout': [(name, off, n) for name, off, n, _ in self.flat.slots]}

    def load_state_dict(self, sd):
        if [tuple(x) for x in sd['layout']] != [(name, off, n) for name, off, n, _ in self.flat.slots]:
            raise _lib.NrmError('FusedTrainStep.load_state_dict: the saved moments use another parameter layout (user_num?)')
        self.exp_avg.copy_(sd['exp_avg']); self.exp_avg_sq.copy_(sd['exp_avg_sq'])
        raw = struct.pack('<q8f', int(sd['step']), sd['lr'], sd['beta1'], sd['beta2'], sd['eps'], sd['weight_decay'], sd['grad_scale'], 0.0, 0.0)
        self.adam_state.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(self.dev))

    # ---- pipeline -------------------------------------------------------------------------
    def _load_compact(self, s: _Slot, batch):
        from . import wire
        if self.articles is None:
            raise _lib.NrmError('FusedTrainStep: pass articles=ArticleTable to feed CompactBatches')
        b, bh, bc = batch.shape
        if b > self.B or (bh, bc) != (self.H, self.C):
            raise ValueError(f'CompactBatch of shape {batch.shape} does not fit this step (B <= {self.B}, H = {self.H}, C = {self.C})')
        if s.compact is None:
            s.compact = wire.CompactBatch(*[torch.zeros((self.B,) + tuple(getattr(batch, f).shape[1:]), dtype=getattr(batch, f).dtype, device=self.dev)
                                            for f in batch.__dataclass_fields__])
            c = s.compact
            s.cstruct = _lib.CompactBatchStruct(self.articles.rows.data_ptr(), int(self.articles.n), c.hist_article.data_ptr(),
                                                c.hist_time.data_ptr(), c.hist_click.data_ptr(), c.cand_article.data_ptr(),
                                                c.cand_time.data_ptr(), c.label.data_ptr(), s.label.data_ptr())
            self._expand(s)                                  # first launch of the kernel outside any graph capture
            # the zero fills / the expansion above run on the compute stream: the H2D copies below must not overtake them
            self.copy_stream.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self.copy_stream):
            if s.used:
                self.copy_stream.wait_event(s.consumed)
            fields = ('hist_article', 'hist_time', 'hist_click', 'cand_article', 'cand_time', 'label')
            if b == self.B:                                  # full batch: one multi-tensor copy call (host time, not bytes, is what counts here)
                torch._foreach_copy_([getattr(s.compact, f) for f in fields] + [s.uid], [getattr(batch, f) for f in fields] + [batch.user_id],
                                     non_blocking=True)
            else:
                for f in fields:
                    getattr(s.compact, f)[:b].copy_(getattr(batch, f), non_blocking=True)
                s.uid[:b].copy_(batch.user_id, non_blocking=True)
            s.ready.record(self.copy_stream)
        loader = getattr(batch, '_loader', None)
        if loader is not None:                               # wire.PrefetchLoader: its pinned ring slot is free once these copies are done
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
            loader.release(batch, ev)
        s.wire = 'compact'
        s.rows = b                                           # b < B: ragged last batch (expanded whole, trained on its first b rows)
        return s

    def _expand(self, s: _Slot):
        """Compact slot -> what the forward reads: nothing to do on the direct path (the row kernels read the compact batch; the
        labels are converted by the first of them), the packed float64 tensors otherwise."""
        from . import wire
        if self.compact_direct:
            return
        wire.expand_into(self.articles, s.compact, s.xh, s.xt, s.xg, s.label)

    def load(self, batch) -> _Slot:
        """Enqueue the H2D copy of a (pinned) host batch into the next slot (round robin).  `batch` is a packed
        `synthetic.Batch`-like object (x_history, x_target, x_global, label, user_id) or a `wire.CompactBatch`."""
        s = self.slots[self.loaded % len(self.slots)]
        self.loaded += 1
        if hasattr(batch, 'hist_article'):
            return self._load_compact(s, batch)
        s.wire = 'packed'
        b = int(batch.x_history.shape[0])
        if b > self.B or tuple(batch.x_history.shape[1:]) != (self.H, HIST_COLS) or tuple(batch.x_target.shape[1:]) != (self.C, TGT_COLS):
            raise ValueError(f'batch of shape {tuple(batch.x_history.shape)} / {tuple(batch.x_target.shape)} does not fit this step '
                             f'(B <= {self.B}, H = {self.H}, C = {self.C})')
        s.rows = b                                           # b < B: the ragged last batch of DataLoader(..., drop_last=False), train.py:40
        with torch.cuda.stream(self.copy_stream):
            if s.used:
                self.copy_stream.wait_event(s.consumed)      # do not overwrite a slot still being read
            if b == self.B:
                torch._foreach_copy_([s.xh, s.xt, s.xg, s.label, s.uid], [batch.x_history, batch.x_target, batch.x_global, batch.label, batch.user_id],
                                     non_blocking=True)
            else:
                s.xh[:b].copy_(batch.x_history, non_blocking=True)
                s.xt[:b].copy_(batch.x_target, non_blocking=True)
                s.xg[:b].copy_(batch.x_global, non_blocking=True)
                s.label[:b].copy_(batch.label, non_blocking=True)
                s.uid[:b].copy_(batch.user_id, non_blocking=True)
            s.ready.record(self.copy_stream)
        return s

    def run(self, s: _Slot) -> LossHandle:
        cur = torch.cuda.current_stream(self.dev)
        cur.wait_event(s.ready)
        k = self.count % self.ring
        loss_out = self.loss_dev[k:k + 1]
        if s.rows != self.B:
            # ragged last batch: the same five calls with the smaller B, eagerly (a graph per tail size would never be replayed)
            if self.dp is not None:
                raise _lib.NrmError('FusedTrainStep: ragged batches under data parallelism would bias the gradient average; '
                                    'drop or pad the tail')
            scratch = self._tail_scratch.get(s.rows)
            if scratch is None:
                scratch = self._tail_scratch[s.rows] = torch.zeros(int(self.lib.nrm_loss_scratch_bytes(s.rows, self.C)),
                                                                   dtype=torch.uint8, device=self.dev)
            if s.wire == 'compact':
                self._expand(s)
            self._forward_backward(s, loss_out, B=s.rows, loss_scratch=scratch)
            self._adam()
        elif self.use_graph:
            if s.graph_fb is None or s.graph_wire != s.wire:
                # eager warm-up pass is NOT wanted (it would be an extra optimizer step): capture directly
                s.graph_fb = torch.cuda.CUDAGraph()
                s.loss_slot = self.loss_dev.new_zeros(())
                with torch.cuda.graph(s.graph_fb, capture_error_mode='thread_local'):       # other threads (a loader) may call CUDA meanwhile
                    if s.wire == 'compact':
                        self._expand(s)
                    self._forward_backward(s, s.loss_slot)
                    if self.one_graph:
                        self._adam()                     # single process or peer-memory data parallel: the whole step is ONE graph
                s.graph_wire = s.wire
                if not self.one_graph:                   # NCCL data parallel: the gradient all-reduce sits between two graphs
                    s.graph_adam = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(s.graph_adam, capture_error_mode='thread_local'):
                        self._adam()
            s.graph_fb.replay()
            if not self.one_graph:
                self.dp.buckets.reduce(self.grads, 0, self.grads.numel())
                self.dp.buckets.wait()
                s.graph_adam.replay()
            loss_out = s.loss_slot.view(1)
        else:
            if s.wire == 'compact':
                self._expand(s)
            self._forward_backward(s, loss_out)
            if self.dp is not None and self.peer is None:
                self.dp.buckets.reduce(self.grads, 0, self.grads.numel())
                self.dp.buckets.wait()
            self._adam()
        s.consumed.record(cur)
        s.used = True
        self.loss_host[k:k + 1].copy_(loss_out, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(cur)
        self.count += 1
        return LossHandle(self.loss_host[k], ev)

    def step(self, batch) -> LossHandle:
        return self.run(self.load(batch))
