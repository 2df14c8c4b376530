"""The eval-mode forward and the frozen-BatchNorm backward, stage by stage, against a float64 evaluation of the same stage fed the
GPU's own upstream buffers (tests/test_gpu_stagewise.py does the same for the training step).

Two modes run only here:

* eval forward (MODE_EVAL: model.eval() under torch.no_grad(), what recommend, scoring and the attention-score export read):
  the head's BatchNorm normalises with the running statistics, the head keeps no activations (keep = 0) and the row kernel
  writes no sort keys.  xh and e are read from the eval workspace, the logits are compared with head_forward(training=False)
  fed the GPU e and the model's float32 running statistics (exactly converted to float64).
* frozen-BatchNorm backward (MODE_KEEP_FOR_BWD alone: model.eval() with gradients enabled, fine-tuning with frozen statistics):
  the head forward keeps its activations, bn_bwd_combine_kernel takes its training == 0 branch (de += rstd * gamma * dz, with
  the gate product of the tensor-core head) and the bn.weight / bn.bias gradients use the running-statistics xhat.  The same
  forward must give the eval logits bit for bit (keep only adds stores) and leave running_mean, running_var and
  num_batches_tracked untouched through the backward.

Every case runs with both shipped checkpoints: `train` (running variances down to about 3.4e-4) and `validation` (near-dead
channels whose 1 / sqrt(var + eps) reaches about 316, which amplifies the head's input rounding).  A row passes when
|gpu - ref| <= rtol * max|ref over its impression| + atol * max|ref over the buffer|, atol = rtol / 100; a parameter gradient
when |gpu - ref| <= rtol * max|ref| of that tensor.  A failure names the buffer, precision, mode, checkpoint, case regime and
the (b, c | h, column) of the worst element.

Tolerances.  The floor of a buffer is the worst err / max|ref over the impression| over every case and both checkpoints, with the
case (b2 = b2_h1_c1, b1 = b1_h50_c5, b1h1 = b1_h1_c1, the others by batch size) and checkpoint (t / v) it came from; the forward
buffers are the same kernels and the same values in both modes (the logits bit for bit).  Measured on one B200 at a 1000 W power
limit, nvcc 12.9:

    buffer          fp32                  bf16x3                bf16
    xh              4.4e-07 (b2000 t)     4.4e-07 (b2000 t)     4.4e-07 (b2000 t)
    e_label         1.3e-06 (b2000 t)     3.7e-05 (b160 v)      1.0e-02 (b160 v)
    e_textimg       5.6e-07 (b5 t)        1.3e-05 (b2000 v)     8.3e-03 (b2000 v)
    e_direct        1.5e-07 (b2000 t)     1.5e-07 (b2000 t)     1.5e-07 (b2000 t)
    logits          1.7e-06 (b2000 t)     1.4e-05 (b2000 t)     5.0e-05 (b2000 t)
    de              4.0e-06 (b2000 t)     2.1e-05 (b2000 t)     8.1e-05 (b2000 t)
    dtp_label       -                     1.2e-05 (b2000 v)     1.0e-02 (b2000 v)
    dtp_textimg     -                     3.3e-05 (b2000 t)     4.4e-02 (b2000 v)
    dxh             2.2e-06 (b160 t)      1.8e-05 (b2000 t)     5.3e-03 (b2000 t)
    dxt             4.0e-07 (b160 v)      4.2e-06 (b160 v)      3.1e-03 (b160 v)
    dxin_h          5.4e-07 (b2000 t)     1.7e-05 (b2000 t)     5.4e-03 (b2000 v)
    grad_head       1.8e-06 (b2 v)        4.1e-05 (b2 v)        2.7e-02 (b2 v)
    grad_attention  3.0e-06 (b2000 v)     2.6e-05 (b1 t)        1.2e-02 (b1 t)
    grad_w1         8.6e-07 (b160 v)      1.2e-05 (b1h1 t)      4.6e-03 (b1h1 t)
    grad_embed      1.0e-06 (b160 t)      7.3e-07 (b160 t)      9.1e-07 (b2000 v)
    e_label, H = 1  4.2e-05 (b2 t)        7.0e-05 (b2 t)        1.5e-01 (b2 t)

Each rtol is 3x its floor, rounded up to one significant digit; atol is rtol / 100.  The small batches need no table of their own
here: with frozen statistics no BatchNorm runs over 1, 2 or 5 rows, and their head and gradient floors sit with the large ones
(fp32 grad_embed at most 1e-6 in every case, against 1.5e-4 at B = 1 in training mode).  What stays ill-conditioned is the label
attention with a single history row (H = 1: the pooled vector is one score, a sum of 64 gelu terms that nearly cancel, times the
row), so e_label of the H = 1 cases gets its own rtol, the one the training file gives the smallest batches.  dxt is 3-12x its
training floor at b160 in every precision: with frozen statistics the attention part of dL/dxt outweighs the direct path
de[:, 136:200] more than with batch statistics, and carries the attention's rounding (the bf16 pair products).

Set NRM_STAGEWISE_FLOORS=<path> to write the floors measured by a run as JSON (keys mode/precision/buffer/checkpoint/case; the
training file's floors, when it runs in the same session, keep their precision/buffer/case keys).
"""
import warnings

import pytest
import torch

from news_recommendation_model_b200 import engine
from stagewise_gpu import (CASES, DEV, PRECISIONS, DtpNotWritten, batch, check_grad, check_rows, cotangent, model, params64,
                           report_floors, ws_fields)
from stagewise_ref import grad_stage, stage_references

pytestmark = pytest.mark.gpu

CHECKPOINTS = ('train', 'validation')
MODE_FROZEN_BN = engine.MODE_KEEP_FOR_BWD

# the training matrix plus the shapes only eval mode reaches or that the pool and ranking consumers run
EVAL_CASES = CASES + [
    ('b1_h1_c1', 1, 1, 1, {}, 'B * C = 1: one head row, allowed in eval mode only'),
    ('b64_h50_c200', 64, 50, 200, {}, 'pool-shaped batch: R = 12800 over many head tiles, G = 25'),
    ('b5_h65_c9', 5, 65, 9, {}, 'C = 8 + 1 with H = 64 + 1: a last group of one candidate and a last history chunk of one row'),
]
EVAL_CASE = {c[0]: c for c in EVAL_CASES}
FROZEN_CASE_IDS = ['b2_h1_c1', 'b1_h50_c5', 'b1_h1_c1', 'b160_h129_c17', 'b2000_h20_c5']
H1_CASES = ('b2_h1_c1', 'b1_h1_c1')

# rtol per precision and buffer, both modes (see the module docstring for the floors they come from); E_LABEL_H1 for e_label of the
# cases with a single history row
RTOL = {
    'fp32': dict(xh=2e-6, e_label=4e-6, e_textimg=2e-6, e_direct=5e-7, logits=5e-6, de=2e-5, dxh=7e-6, dxt=2e-6, dxin_h=2e-6,
                 grad_head=6e-6, grad_attention=9e-6, grad_w1=3e-6, grad_embed=4e-6),
    'bf16x3': dict(xh=2e-6, e_label=2e-4, e_textimg=4e-5, e_direct=5e-7, logits=5e-5, de=7e-5, dtp_label=4e-5, dtp_textimg=1e-4,
                   dxh=6e-5, dxt=2e-5, dxin_h=6e-5, grad_head=2e-4, grad_attention=8e-5, grad_w1=4e-5, grad_embed=3e-6),
    'bf16': dict(xh=2e-6, e_label=4e-2, e_textimg=3e-2, e_direct=5e-7, logits=2e-4, de=3e-4, dtp_label=4e-2, dtp_textimg=2e-1,
                 dxh=2e-2, dxt=1e-2, dxin_h=2e-2, grad_head=9e-2, grad_attention=4e-2, grad_w1=2e-2, grad_embed=3e-6),
}
E_LABEL_H1 = {'fp32': 2e-4, 'bf16x3': 3e-4, 'bf16': 5e-1}


def _table(name, case_id):
    """The tolerance entry a (buffer, case) is checked against."""
    return 'e_label, H = 1' if name == 'e_label' and case_id in H1_CASES else name


def rtol_for(precision, name, case_id):
    return E_LABEL_H1[precision] if _table(name, case_id) != name else RTOL[precision][name]


FLOORS = {}            # (mode, precision, buffer, checkpoint, case id) -> worst err / impression scale seen by this run


@pytest.fixture(scope='module', autouse=True)
def _report_floors():
    yield
    report_floors(FLOORS, lambda k: (k[1], _table(k[2], k[4])), lambda g: f'{g[0]:7s} {g[1]:15s}',
                  lambda k: rtol_for(k[1], k[2], k[4]), where=lambda k: f'{k[4]}, {k[3]}, {k[0]}')


def _stats64(m):
    return m.bn.running_mean.detach().double(), m.bn.running_var.detach().double()


class _Checks:
    """The per-row and per-tensor checks of one (mode, checkpoint, precision, case) run."""

    def __init__(self, mode, checkpoint, precision, case):
        self.mode, self.checkpoint, self.precision, self.case = mode, checkpoint, precision, case
        self.label = f'{precision}, {mode}, {checkpoint} checkpoint, {case[0]}: {case[5]}'
        self.failures = []

    def _key(self, name):
        return (self.mode, self.precision, name, self.checkpoint, self.case[0])

    def rows(self, name, got, ref):
        _, B, H, C, _, _ = self.case
        n = H if name in ('xh', 'dxh', 'dxin_h') else C
        check_rows(name, got.reshape(B, n, -1), ref.reshape(B, n, -1), rtol_for(self.precision, name, self.case[0]),
                   self.label, FLOORS, self._key(name), self.failures)

    def forward(self, bufs, logits, ref):
        self.rows('xh', bufs['xh'], ref['xh'])
        self.rows('e_label', bufs['e'][:, 0:64], ref['e'][:, 0:64])
        self.rows('e_textimg', bufs['e'][:, 64:128], ref['e'][:, 64:128])
        self.rows('e_direct', bufs['e'][:, 128:], ref['e'][:, 128:])
        self.rows('logits', logits, ref['logits'])

    def grad(self, k, got, ref):
        name = 'grad_' + grad_stage(k)
        check_grad(name, k, got, ref, rtol_for(self.precision, name, self.case[0]), self.label, FLOORS, self._key(name),
                   self.failures)


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('checkpoint', CHECKPOINTS)
@pytest.mark.parametrize('case_id', list(EVAL_CASE))
def test_eval_forward_against_float64(case_id, checkpoint, precision):
    case = EVAL_CASE[case_id]
    _, B, H, C, _, _ = case
    d = batch(case).to(DEV)
    m = model(precision, checkpoint).eval()
    with torch.no_grad():
        logits = m(d.x_history, d.x_target, d.x_global)
        torch.cuda.synchronize()
        bufs = ws_fields(m, B, H, C, engine.MODE_EVAL, ('xh', 'e'))
        up = {k: v.double() for k, v in bufs.items()}
        ref, _ = stage_references(params64(checkpoint), d.x_history, d.x_target, d.x_global, None, gpu=up, training=False,
                                  stats=_stats64(m))
    chk = _Checks('eval', checkpoint, precision, case)
    chk.forward(bufs, logits, ref)
    assert not chk.failures, '\n'.join(chk.failures)


def frozen_bn_step(case, checkpoint, precision):
    """model.eval(): the no_grad logits, then a forward with gradients enabled and out.backward(G) with the seeded cotangent.
    Returns the logits of both forwards, the BatchNorm buffers before, after the forward and after the backward, the training
    workspace buffers and the parameter gradients, all cloned."""
    _, B, H, C, _, _ = case
    d = batch(case).to(DEV)
    G = cotangent(B, C).to(DEV)
    m = model(precision, checkpoint).eval()
    bn = lambda: [t.detach().clone() for t in (m.bn.running_mean, m.bn.running_var, m.bn.num_batches_tracked)]
    with torch.no_grad():
        eval_logits = m(d.x_history, d.x_target, d.x_global).clone()
    res = dict(eval_logits=eval_logits, bn_before=bn())
    m.zero_grad(set_to_none=True)
    out = m(d.x_history, d.x_target, d.x_global)
    assert out.requires_grad and out._nrm_token.mode == MODE_FROZEN_BN
    torch.cuda.synchronize()
    res.update(logits=out.detach().clone(), bn_forward=bn())
    out.backward(G)
    torch.cuda.synchronize()
    res.update(bn_backward=bn(), bufs=ws_fields(m, B, H, C, MODE_FROZEN_BN), stats=_stats64(m),
               grads={k: v.grad.detach().clone() for k, v in m.named_parameters() if v.grad is not None})
    return res


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('case_id', FROZEN_CASE_IDS)
def test_eval_forward_with_gradients_enabled(case_id, precision):
    """The frozen-BatchNorm forward stores the head's activations and nothing else changes: its logits equal the no_grad eval
    logits bit for bit, and the BatchNorm buffers stay as they were through the forward and the backward."""
    res = frozen_bn_step(EVAL_CASE[case_id], 'validation', precision)
    same = res['logits'] == res['eval_logits']
    assert bool(same.all()), (f'[{precision}, {case_id}] logits with gradients enabled differ from the no_grad eval logits at '
                              f'(b, c) {torch.nonzero(~same)[:8].tolist()}')
    for when in ('bn_forward', 'bn_backward'):
        for name, before, after in zip(('running_mean', 'running_var', 'num_batches_tracked'), res['bn_before'], res[when]):
            assert torch.equal(before, after), f'[{precision}, {case_id}] bn.{name} changed by the eval-mode {when[3:]}'


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('checkpoint', CHECKPOINTS)
@pytest.mark.parametrize('case_id', FROZEN_CASE_IDS)
def test_frozen_bn_backward_against_float64(case_id, checkpoint, precision):
    case = EVAL_CASE[case_id]
    _, B, H, C, _, _ = case
    res = frozen_bn_step(case, checkpoint, precision)
    b = batch(case).to(DEV)
    bufs = {k: v.to(DEV) for k, v in res['bufs'].items()}
    up = {k: bufs[k].double() for k in ('xh', 'e', 'de', 'dxh', 'dxt', 'dxin_h')}
    with torch.no_grad():
        ref, grads = stage_references(params64(checkpoint), b.x_history, b.x_target, b.x_global, cotangent(B, C).to(DEV).double(),
                                      gpu=up, training=False, stats=res['stats'])
    chk = _Checks('frozen-bn', checkpoint, precision, case)
    chk.forward(bufs, res['logits'], ref)
    chk.rows('de', bufs['de'], ref['de'])
    if precision == 'fp32':
        warnings.warn(f'dtp not compared [fp32, {case_id}]: the FFMA backward keeps dL/dtp in registers and never writes the buffer',
                      DtpNotWritten)
    else:
        chk.rows('dtp_label', bufs['dtp'][0], ref['dtp'][0])
        chk.rows('dtp_textimg', bufs['dtp'][1], ref['dtp'][1])
    chk.rows('dxh', bufs['dxh'], ref['dxh'])
    chk.rows('dxt', bufs['dxt'], ref['dxt'])
    chk.rows('dxin_h', bufs['dxin_h'], ref['dxin_h'])
    assert {k for k in grads if k != 'delta'} <= res['grads'].keys()
    for k, r in grads.items():
        if k != 'delta':
            chk.grad(k, res['grads'][k].to(DEV), r)
    assert not chk.failures, '\n'.join(chk.failures)
