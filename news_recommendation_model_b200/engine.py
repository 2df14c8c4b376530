"""Host-side plumbing between the nn.Module mirror and libnrm_b200.

* one flat float32 buffer holds every trainable tensor (layout from the library);
  the modules' nn.Parameters are views into it, so kernels read weights with fixed
  offsets and the optimizer can update everything with one launch;
* every training forward gets a `StepToken` that owns its workspace and (lazily) one
  flat gradient buffer; the backward kernels write the gradients there and autograd
  receives views of it;
* torch is used for device memory, streams and autograd bookkeeping only.
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, NamedTuple, Optional, Tuple

import torch

from . import _lib
from .config import E_DIM, HIST_COLS, TGT_COLS, GLOBAL_COLS

MODE_EVAL = 0
MODE_BN_BATCH_STATS = 1
MODE_KEEP_FOR_BWD = 2
PRECISION = {'fp32': 0, 'bf16': 1, 'bf16x3': 2}

_LAYOUT: Optional[Tuple[List[Tuple[str, int, int]], int]] = None


def layout():
    global _LAYOUT
    if _LAYOUT is None:
        _LAYOUT = _lib.layout()
    return _LAYOUT


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _al4(n: int) -> int:
    return (n + 3) & ~3


class FlatParams:
    """The flat parameter buffer of one model and the views into it."""

    def __init__(self, named: Dict[str, torch.nn.Parameter]):
        entries, fixed = layout()
        dev = None
        for name, off, numel in entries:
            if name == 'delta' and name not in named:
                continue
            p = named[name]
            if dev is None:
                dev = p.device
            if p.device != dev:
                raise _lib.NrmError('all parameters of a model must live on one device')
            if p.dtype != torch.float32:
                raise _lib.NrmError(f'{name}: parameters must be float32 (got {p.dtype})')
            if numel >= 0 and p.numel() != numel:
                raise _lib.NrmError(f'{name}: expected {numel} elements, got {p.numel()}')
        self.device = dev
        self.delta_numel = named['delta'].numel() if 'delta' in named else 0
        self.fixed = fixed
        self.total = fixed + _al4(self.delta_numel)
        self.buf = torch.zeros(self.total, dtype=torch.float32, device=dev)
        self.slots: List[Tuple[str, int, int, torch.Size]] = []
        with torch.no_grad():
            for name, off, numel in entries:
                if name == 'delta' and name not in named:
                    continue
                p = named[name]
                n = p.numel()
                view = self.buf[off:off + n].view(p.shape)
                view.copy_(p.detach())
                p.data = view
                self.slots.append((name, off, n, p.shape))
        self.bn_weight_off = next(off for name, off, _, _ in self.slots if name == 'bn.weight')
        # the Parameter objects in layout order (without delta): the autograd inputs of every forward
        self.params = [named[name] for name, _, _, _ in self.slots if name != 'delta']

    def is_current(self, named: Dict[str, torch.nn.Parameter]) -> bool:
        base = self.buf.data_ptr()
        for name, off, n, _ in self.slots:
            p = named.get(name)
            if p is None or p.data_ptr() != base + 4 * off or p.numel() != n:
                return False
        return True

    def grad_views(self, gbuf: torch.Tensor, skip_delta: bool) -> List[torch.Tensor]:
        """Views of the flat gradient buffer with the parameters' shapes, in layout order: ONE split call (sizes include
        the alignment gaps between entries) instead of a slice per tensor."""
        plan = self.__dict__.get('_split_plan')
        if plan is None:
            sizes, pick, pos = [], [], 0
            for name, off, n, shape in self.slots:
                if off > pos:
                    sizes.append(off - pos)
                pick.append((len(sizes), name, shape if len(shape) != 1 else None))
                sizes.append(n)
                pos = off + n
            if self.total > pos:
                sizes.append(self.total - pos)
            plan = self._split_plan = (sizes, pick)
        sizes, pick = plan
        if gbuf.numel() != self.total:
            return [gbuf[off:off + n].view(shape) for name, off, n, shape in self.slots if not (skip_delta and name == 'delta')]
        parts = gbuf.split_with_sizes(sizes)
        return [parts[i] if shape is None else parts[i].view(shape) for i, name, shape in pick
                if not (skip_delta and name == 'delta')]


class StepToken:
    """Lives from one forward to the end of its backward(s)."""
    __slots__ = ('workspace', 'grad_buf', 'B', 'H', 'C', 'mode', 'inputs', 'total', 'device', 'done')

    def __init__(self, workspace, B, H, C, mode, inputs, total, device):
        self.workspace, self.B, self.H, self.C, self.mode = workspace, B, H, C, mode
        self.inputs, self.total, self.device = inputs, total, device
        self.grad_buf = None
        self.done = False

    def grads(self) -> torch.Tensor:
        if self.grad_buf is None:
            self.grad_buf = torch.zeros(self.total, dtype=torch.float32, device=self.device)
        return self.grad_buf


class Runtime:
    """Per-model cache of device scratch (never pickled with the model)."""

    def __init__(self):
        self.flat: Optional[FlatParams] = None
        self.eval_ws: Optional[torch.Tensor] = None
        self.train_ws: Optional[torch.Tensor] = None
        self.train_ws_token: Optional[StepToken] = None
        self.loss_scratch: Optional[torch.Tensor] = None
        self.loss_scratch_busy = False

    def workspace(self, B, H, C, mode, device) -> torch.Tensor:
        need = int(_lib.load().nrm_workspace_bytes(B, H, C, mode))
        if mode & MODE_KEEP_FOR_BWD:
            busy = self.train_ws_token is not None and not self.train_ws_token.done
            if self.train_ws is None or self.train_ws.numel() < need or self.train_ws.device != device or busy:
                self.train_ws = torch.empty(need, dtype=torch.uint8, device=device)
            return self.train_ws
        if self.eval_ws is None or self.eval_ws.numel() < need or self.eval_ws.device != device:
            self.eval_ws = torch.empty(need, dtype=torch.uint8, device=device)
        return self.eval_ws


class Packed(NamedTuple):
    """A batch of packed float64 rows as the packed entry points take it (`nrm_forward(xh, xt, xt_bs, xg, xg_bs, B, H, C, ...)`)."""
    xh: torch.Tensor
    xt: torch.Tensor
    xt_bs: int              # batch strides in elements
    xg: torch.Tensor
    xg_bs: int
    suffix = ''

    @property
    def args(self) -> tuple:
        return _ptr(self.xh), _ptr(self.xt), self.xt_bs, _ptr(self.xg), self.xg_bs


def packed(xh: torch.Tensor, xt: torch.Tensor, xg: torch.Tensor) -> Packed:
    """The binding of packed tensors whose impressions are dense rows.  B = 1: a size-1 dimension may carry any stride, so the
    library gets the dense one."""
    B, C = xt.shape[0], xt.shape[1]
    return Packed(xh, xt, xt.stride(0) if B > 1 else C * TGT_COLS, xg, xg.stride(0) if B > 1 else C * GLOBAL_COLS)


class Compact(NamedTuple):
    """A device `wire.CompactBatch` and its `ArticleTable` as the `_compact` entry points take them
    (`nrm_forward_compact(&batch, B, H, C, ...)`): the row kernels read the article ids directly."""
    struct: _lib.CompactBatchStruct
    keep: tuple             # the tensors `struct` points into
    suffix = '_compact'

    @property
    def args(self) -> tuple:
        return (ctypes.byref(self.struct),)


def compact(table, cb, label64: Optional[torch.Tensor] = None) -> Compact:
    """`label64`: a float64 [B,C] buffer the first row kernel converts `cb.label` into (what the loss reads); None: no labels."""
    label32 = cb.label if label64 is not None else None
    struct = _lib.CompactBatchStruct(table.rows.data_ptr(), table.n, cb.hist_article.data_ptr(), cb.hist_time.data_ptr(),
                                     cb.hist_click.data_ptr(), cb.cand_article.data_ptr(), cb.cand_time.data_ptr(),
                                     label32.data_ptr() if label32 is not None else None,
                                     label64.data_ptr() if label64 is not None else None)
    return Compact(struct, (table, cb, label64))


def call(inputs, entry: str, *rest) -> None:
    """`entry` in the variant for `inputs`' wire format, with `inputs`' arguments first."""
    name = entry + inputs.suffix
    _lib.check(getattr(_lib.load(), name)(*inputs.args, *rest), name)


def prepare_inputs(x_history, x_target, x_global) -> Packed:
    """Validate the packed float64 feature tensors (SURVEY.md 8b input conventions) and
    return their binding."""
    if x_history.dim() != 3 or x_history.shape[2] != HIST_COLS:
        raise ValueError(f'x_history must be [B,H,{HIST_COLS}], got {tuple(x_history.shape)}')
    if x_target.dim() != 3 or x_target.shape[2] != TGT_COLS:
        raise ValueError(f'x_target must be [B,C,{TGT_COLS}], got {tuple(x_target.shape)}')
    if x_global.dim() != 3 or x_global.shape[2] != GLOBAL_COLS or x_global.shape[:2] != x_target.shape[:2]:
        raise ValueError(f'x_global must be [B,C,{GLOBAL_COLS}], got {tuple(x_global.shape)}')
    if x_history.shape[0] != x_target.shape[0]:
        raise ValueError('x_history and x_target disagree on the batch size')
    if not x_history.is_cuda:
        raise _lib.NrmError('news_recommendation_model_b200 runs on CUDA devices only (no CPU fallback): '
                            'move the model and its inputs to a B200 first')
    dev = x_history.device
    out = []
    for t, cols in ((x_history, HIST_COLS), (x_target, TGT_COLS), (x_global, GLOBAL_COLS)):
        if t.device != dev:
            raise ValueError('all inputs must be on the same device')
        if t.dtype != torch.float64:
            t = t.to(torch.float64)
        # rows of one impression must be dense; the batch stride may be larger (test.py:53-54)
        if t.stride(2) != 1 or t.stride(1) != cols or (t.shape[0] > 1 and t.stride(0) < t.shape[1] * cols):
            t = t.contiguous()
        out.append(t)
    xh, xt, xg = out
    if not xh.is_contiguous():
        xh = xh.contiguous()
    return packed(xh, xt, xg)


def forward(inputs, B, H, C, params, bn_mean, bn_var, bn_nbt, mode, precision, logits, ws, stream, bn_sums=None, exchange=None):
    """Encoder and head forward of one batch.  `exchange` None: one call.  Otherwise the two halves of a synchronised-BatchNorm
    forward: the encoder writes this rank's BatchNorm column sums into `bn_sums`, and `exchange(bn_sums)` returns the sums and the
    row count the head normalises with."""
    if exchange is None:
        call(inputs, 'nrm_forward', B, H, C, _ptr(params), _ptr(bn_mean), _ptr(bn_var), _ptr(bn_nbt), mode, precision, _ptr(logits),
             _ptr(ws), ws.numel(), stream)
        return
    call(inputs, 'nrm_forward_encoder', B, H, C, _ptr(params), mode, precision, _ptr(bn_sums), _ptr(ws), ws.numel(), stream)
    sums, rows = exchange(bn_sums)
    _lib.check(_lib.load().nrm_forward_head(B, H, C, _ptr(params), _ptr(bn_mean), _ptr(bn_var), _ptr(bn_nbt), mode, precision, _ptr(sums),
                                            rows, _ptr(logits), _ptr(ws), ws.numel(), stream), 'nrm_forward_head')


def backward(inputs, B, H, C, params, mode, precision, dlogits, grads, ws, stream, bn_sums=None, exchange=None, defer_wgrad=True):
    """Head and encoder backward of one batch into `grads`.  `exchange` None: one call.  Otherwise the two halves, and
    `exchange(bn_sums)` runs between them and returns the BatchNorm backward sums and row count the encoder combines with
    (`bn_sums` None: this rank's own).  `defer_wgrad` False: the head's weight gradients are complete when `exchange` runs;
    True: the encoder backward enqueues them beside its own tail."""
    if exchange is None:
        call(inputs, 'nrm_backward', B, H, C, _ptr(params), mode, precision, _ptr(dlogits), _ptr(grads), _ptr(ws), ws.numel(), stream)
        return
    head = 'nrm_backward_head_deferred' if defer_wgrad else 'nrm_backward_head'
    _lib.check(getattr(_lib.load(), head)(B, H, C, _ptr(params), precision, _ptr(dlogits), _ptr(grads), _ptr(bn_sums), _ptr(ws), ws.numel(),
                                          stream), head)
    sums, rows = exchange(bn_sums)
    call(inputs, 'nrm_backward_encoder', B, H, C, _ptr(params), mode, precision, _ptr(sums), rows, _ptr(grads), _ptr(ws), ws.numel(), stream)


def forward_logits(rt: Runtime, flat: FlatParams, bn_mean, bn_var, bn_nbt, x_history, x_target, x_global,
                   mode: int, precision: int, dp=None):
    """Run the forward (`forward`); returns (logits [B,C], token or None)."""
    inputs = prepare_inputs(x_history, x_target, x_global)
    B, H, C = inputs.xh.shape[0], inputs.xh.shape[1], inputs.xt.shape[1]
    dev = inputs.xh.device
    if flat.device != dev:
        raise _lib.NrmError(f'model is on {flat.device} but inputs are on {dev}')
    ws = rt.workspace(B, H, C, mode, dev)
    logits = torch.empty(B, C, dtype=torch.float32, device=dev)
    sums = exchange = None
    if dp is not None and dp.sync_bn and (mode & MODE_BN_BATCH_STATS):
        sums = torch.empty(2 * E_DIM, dtype=torch.float64, device=dev)
        exchange = lambda s: (s, dp.all_reduce_stats(s, B * C))              # noqa: E731
    forward(inputs, B, H, C, flat.buf, bn_mean, bn_var, bn_nbt, mode, precision, logits, ws, _stream(dev), sums, exchange)
    token = None
    if mode & MODE_KEEP_FOR_BWD:
        token = StepToken(ws, B, H, C, mode, inputs, flat.total, dev)
        rt.train_ws_token = token
    return logits, token


def backward_params(flat: FlatParams, token: StepToken, dlogits: torch.Tensor, precision: int, dp=None) -> torch.Tensor:
    """Run the backward (`backward`) for `token`; returns the flat gradient buffer."""
    if token.done:
        raise _lib.NrmError('backward called twice for the same forward (activations already released)')
    B, H, C, dev = token.B, token.H, token.C, token.device
    g = token.grads()
    dl = dlogits.contiguous()
    if dl.dtype != torch.float32:
        dl = dl.float()
    args = (token.inputs, B, H, C, flat.buf, token.mode, precision, dl, g, token.workspace, _stream(dev))
    if dp is None:
        backward(*args)
    else:
        sync = dp.sync_bn and (token.mode & MODE_BN_BATCH_STATS)

        def exchange(sums):
            rows = dp.all_reduce_stats(sums, B * C) if sync else 0
            dp.reduce_head_bucket(g, flat)          # overlaps with the encoder backward
            return sums, rows
        sums = torch.empty(2 * E_DIM, dtype=torch.float64, device=dev) if sync else None
        backward(*args, sums, exchange, defer_wgrad=False)
        dp.reduce_encoder_bucket(g, flat)
        dp.wait()
    token.done = True
    token.inputs = None
    return g


class _ForwardFn(torch.autograd.Function):
    """UserModel.forward (user_model.py:27-35) with the hand-written backward."""

    @staticmethod
    def forward(ctx, model, x_history, x_target, x_global, mode, *params):
        rt = model._runtime()
        logits, token = forward_logits(rt, rt.flat, model.bn.running_mean, model.bn.running_var,
                                       model.bn.num_batches_tracked, x_history, x_target, x_global, mode,
                                       model._precision_code(), model._dp)
        ctx.model, ctx.token = model, token
        ctx.set_materialize_grads(False)
        logits._nrm_token = token
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        model, token = ctx.model, ctx.token
        flat = model._runtime().flat
        if dlogits is None:
            dlogits = torch.zeros(token.B, token.C, dtype=torch.float32, device=token.device)
        g = backward_params(flat, token, dlogits, model._precision_code(), model._dp)
        return (None, None, None, None, None) + tuple(flat.grad_views(g, skip_delta=True))


class _LossFn(torch.autograd.Function):
    """UserModel.loss (user_model.py:37-43) with the hand-written backward."""

    @staticmethod
    def forward(ctx, model, token, user_id, label, alpha, out, delta):
        lib = _lib.load()
        rt = model._runtime()
        B, C = out.shape
        dev = out.device
        need = int(lib.nrm_loss_scratch_bytes(B, C))
        # zero-filled once (it holds an arrival counter); reused from step to step unless a backward is still pending on it
        scratch = rt.loss_scratch
        if scratch is None or scratch.numel() != need or scratch.device != dev or rt.loss_scratch_busy:
            scratch = torch.zeros(need, dtype=torch.uint8, device=dev)
            if not rt.loss_scratch_busy:
                rt.loss_scratch = scratch
        if scratch is rt.loss_scratch and any(ctx.needs_input_grad):
            rt.loss_scratch_busy = True                    # until the backward has been enqueued
        loss = torch.empty((), dtype=torch.float32, device=dev)
        uid = user_id.to(device=dev, dtype=torch.int64).contiguous()
        lab = label.to(device=dev, dtype=torch.float64).contiguous()
        o = out.detach().contiguous()
        _lib.check(lib.nrm_loss_forward(_ptr(o), _ptr(delta.detach()), delta.numel(), _ptr(uid), _ptr(lab), B, C, float(alpha), _ptr(loss),
                                        _ptr(scratch), need, _stream(dev)), 'nrm_loss_forward')
        ctx.model, ctx.token, ctx.uid, ctx.scratch, ctx.shape = model, token, uid, scratch, (B, C)
        ctx.delta_numel = delta.numel()
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        lib = _lib.load()
        B, C = ctx.shape
        dev = ctx.scratch.device
        flat = ctx.model._runtime().flat
        token = ctx.token
        gl = grad_loss.detach().to(torch.float32).contiguous()
        dlogits = torch.empty(B, C, dtype=torch.float32, device=dev)
        if token is not None and not token.done and flat is not None and flat.delta_numel == ctx.delta_numel:
            g = token.grads()
            ddelta = g[flat.fixed:flat.fixed + ctx.delta_numel]
        else:
            ddelta = torch.empty(ctx.delta_numel, dtype=torch.float32, device=dev)
        _lib.check(lib.nrm_loss_backward(_ptr(ctx.uid), B, C, _ptr(gl), _ptr(dlogits), _ptr(ddelta), ctx.delta_numel,
                                         _ptr(ctx.scratch), ctx.scratch.numel(), _stream(dev)), 'nrm_loss_backward')
        rt = ctx.model._runtime()
        if ctx.scratch is rt.loss_scratch:
            rt.loss_scratch_busy = False
        dp = ctx.model._dp
        if dp is not None:
            # Data parallel: average the delta gradient HERE, before autograd sees it.  AccumulateGrad(delta) runs as soon as
            # this function returns -- a view that is all-reduced later (with the head bucket) would be accumulated into an
            # existing .grad (zero_grad(set_to_none=False), gradient accumulation) with its un-reduced, rank-local values and
            # the replicas would drift apart.  The head bucket therefore ends in front of delta (dp.reduce_head_bucket), and
            # the gradient stays the flat buffer's view so that FusedAdam keeps its one-launch path.
            dp.reduce_delta(ddelta)                            # in place, in stream order: still the flat buffer's view
        return None, None, None, None, None, dlogits, ddelta


def adam_step(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, *, lr, beta1,
              beta2, eps, weight_decay, step, grad_scale=1.0) -> None:
    lib = _lib.load()
    _lib.check(lib.nrm_adam_step(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq), param.numel(), float(lr),
                                 float(beta1), float(beta2), float(eps), float(weight_decay), int(step), float(grad_scale),
                                 _stream(param.device)), 'nrm_adam_step')


# ---------------------------------------------------------------------------------------
# stand-alone encoder (UserInvariantInterestModel / UserInstantInterestModel used outside
# a UserModel): packs the given tensors into a scratch flat buffer and runs
# nrm_forward_encoder.  Inference-only convenience; training goes through UserModel.
# ---------------------------------------------------------------------------------------
def standalone_encoder(named: Dict[str, torch.Tensor], x_history, x_target, x_global) -> torch.Tensor:
    lib = _lib.load()
    inputs = prepare_inputs(x_history, x_target, x_global)
    if any(p.requires_grad for p in named.values()) and torch.is_grad_enabled():
        raise _lib.NrmError('stand-alone encoder modules are inference-only (wrap the call in torch.no_grad()); '
                            'training runs through UserModel.forward')
    dev = inputs.xh.device
    entries, fixed = layout()
    buf = torch.zeros(fixed, dtype=torch.float32, device=dev)
    for name, off, numel in entries:
        if name in named:
            buf[off:off + numel].copy_(named[name].detach().reshape(-1))
    B, H, C = inputs.xh.shape[0], inputs.xh.shape[1], inputs.xt.shape[1]
    need = int(lib.nrm_workspace_bytes(B, H, C, MODE_EVAL))
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    call(inputs, 'nrm_forward_encoder', B, H, C, _ptr(buf), MODE_EVAL, 0, None, _ptr(ws), need, _stream(dev))
    off_e = int(lib.nrm_workspace_e_offset(B, H, C, MODE_EVAL))
    e = ws[off_e:off_e + 4 * B * C * E_DIM].view(torch.float32).view(B, C, E_DIM)
    return e.clone()


def _round256(n: int) -> int:
    return (n + 255) & ~255
