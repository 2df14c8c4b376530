"""Every stage of the training step against a float64 evaluation of the same stage, fed the GPU's own upstream buffers.

tests/test_gpu_parity.py checks a step at its ends: logits, loss and each parameter gradient to 2e-4 of that gradient's largest
element.  A parameter gradient sums over all B*H or B*C rows, so one wrong impression or one wrong (candidate, history) pair is
diluted by about 1/B there.  Here one training forward runs per case, its backward is driven by a seeded random cotangent G of
the logits (out.backward(G): it reaches every candidate row, and has none of the softmax shift invariance of the loss), and the
workspace buffers are read back by name (nrm_debug_ws_field):

    buffer            compared per          reference fed with (tests/stagewise_ref.py)
    xh                history row           the packed inputs (embedding + w1)
    e_label/e_textimg candidate row         GPU xh, GPU e[:, 136:200] (t), the history pca / GPU e[:, 200:264]
    e_direct          candidate row         the packed inputs (e[:, 128:264]: instant interest, target embedding, pca)
    logits            candidate row         GPU e (BatchNorm statistics recomputed in float64 from it)
    de                candidate row         GPU e, G
    dtp_label/_textimg candidate row        GPU xh, t, pca, GPU de[:, 0:64] / de[:, 64:128]  (tensor-core precisions: the FFMA
                                            backward of fp32 keeps dL/dtp in registers and never writes the buffer)
    dxh               history row           same as dtp (label branch)
    dxt               candidate row         same, plus the direct path de[:, 136:200]
    dxin_h            history row           GPU dxh
    grad_<stage>      whole tensor          each stage's GPU inputs, as above (head: GPU e, G; attention: GPU de; w1: GPU dxh;
                                            embed: GPU dxin_h, dxt, de[:, 128:136])

A row passes when |gpu - ref| <= rtol * max|ref over its impression| + atol * max|ref over the buffer|; a parameter gradient when
|gpu - ref| <= rtol * max|ref| of that tensor.  A failure names the buffer, the precision, the case's regime and the (b, c | h, column)
of the worst element.

Tolerances.  The floor of a buffer is the worst err / max|ref over the impression| over the cases of the matrix below (and over
runs of the since-removed item-tile attention kernels), with the case it came from; measured on one B200 at a 1000 W power limit,
nvcc 12.9.  Cases with B >= 7 (RTOL):

    buffer          fp32              bf16x3            bf16
    xh              4.4e-07 (b2000)   4.4e-07 (b2000)   4.4e-07 (b2000)
    e_label         1.3e-06 (b2000)   2.6e-05 (b160)    7.8e-03 (b160)
    e_textimg       5.1e-07 (b150)    1.2e-05 (b2000)   7.7e-03 (b2000)
    e_direct        1.5e-07 (b2000)   1.5e-07 (b2000)   1.5e-07 (b2000)
    logits          3.6e-06 (b300)    1.6e-05 (b2000)   5.0e-05 (b2000)
    de              3.2e-06 (b2000)   1.6e-05 (b2000)   6.8e-05 (b2000)
    dtp_label       -                 1.6e-05 (b150)    8.0e-03 (b2000)
    dtp_textimg     -                 4.1e-05 (b160)    3.0e-02 (b2000)
    dxh             3.8e-06 (b150)    1.8e-05 (b2000)   8.1e-03 (b2000)
    dxt             1.3e-07 (b160)    5.9e-07 (b160)    2.5e-04 (b160)
    dxin_h          5.3e-07 (b300)    1.1e-05 (b2000)   5.0e-03 (b300)
    grad_head       2.3e-06 (b160)    2.0e-05 (b160)    8.3e-03 (b160)
    grad_attention  2.6e-06 (b150)    5.0e-05 (b150)    2.1e-02 (b150)
    grad_w1         1.4e-06 (b160)    5.9e-06 (b2000)   2.0e-03 (b160)
    grad_embed      4.0e-06 (b40)     1.6e-06 (b2000)   1.8e-06 (b40)

The two smallest batches, B = 2, H = 1, C = 1 and B = 1, H = 50, C = 5 (SMALL_CASES, RTOL_SMALL):

    buffer          fp32              bf16x3            bf16
    xh              1.8e-07 (b1)      1.8e-07 (b1)      1.8e-07 (b1)
    e_label         4.2e-05 (b2)      7.0e-05 (b2)      1.5e-01 (b2)
    e_textimg       3.5e-07 (b1)      6.1e-06 (b1)      3.3e-03 (b2)
    e_direct        4.9e-08 (b1)      4.9e-08 (b1)      4.9e-08 (b1)
    logits          1.3e-05 (b2)      3.5e-05 (b2)      7.6e-05 (b2)
    de              2.1e-06 (b2)      5.0e-06 (b2)      5.5e-06 (b2)
    dtp_label       -                 4.4e-06 (b2)      3.1e-03 (b2)
    dtp_textimg     -                 8.8e-06 (b1)      4.8e-03 (b1)
    dxh             4.7e-05 (b2)      3.7e-05 (b2)      1.9e-01 (b2)
    dxt             4.5e-08 (b1)      4.6e-08 (b1)      4.9e-06 (b1)
    dxin_h          3.3e-07 (b1)      6.6e-06 (b1)      3.4e-03 (b1)
    grad_head       4.6e-06 (b2)      8.7e-05 (b2)      2.8e-02 (b2)
    grad_attention  3.1e-06 (b1)      6.6e-05 (b1)      2.8e-02 (b1)
    grad_w1         2.0e-07 (b1)      1.0e-05 (b2)      3.8e-03 (b2)
    grad_embed      1.5e-04 (b1)      3.6e-05 (b1)      7.1e-05 (b1)

Each rtol is 3x its floor in its own table, rounded up to one significant digit; atol is rtol / 100.  The small batches get their
own table because they are ill-conditioned.  With B = 2, H = 1, C = 1 a pooled vector is one score times one history row, and the
score is a sum of 64 gelu terms that nearly cancel, so the rounding of those terms is the whole relative error of the impression;
in bf16 (8-bit operands in the pair product) that reaches 15-19 % of e_label and dxh.  BatchNorm over 2 (B = 2) or 5 (B = 1) rows
has near-constant channels whose rstd multiplies the same rounding in the head and in the gradients downstream of it (fp32
grad_embed 1.5e-4 at B = 1, against 4e-6 with B >= 7).  The bf16 rtols of the B >= 7 table (1e-2 order for the pair-product
buffers) follow from 8-bit operands; the fp32 ones are a few 1e-6.

The FFMA backward of fp32 never writes dtp; each fp32 case says so with a DtpNotWritten warning.

Set NRM_STAGEWISE_FLOORS=<path> to write the floors measured by a run as JSON.
"""
import ctypes
import json
import os
import warnings

import numpy as np
import pytest
import torch

import news_recommendation_model_b200 as nrm
from news_recommendation_model_b200 import _lib
from fixtures import load_weights
from news_recommendation_model_b200.synthetic import make_batch
from oracle import reference_port as O
from stagewise_ref import grad_stage, stage_references

pytestmark = pytest.mark.gpu

DEV = 'cuda'
USERS = 50
PRECISIONS = ('fp32', 'bf16x3', 'bf16')

# (id, B, H, C, make_batch options, regime)
CASES = [
    ('b2_h1_c1', 2, 1, 1, {}, 'smallest training batch'),
    ('b1_h50_c5', 1, 50, 5, {}, 'B = 1: batch-stride branch of engine.forward_logits'),
    ('b7_h65_c8', 7, 65, 8, {}, 'G = 1 with a full group of 8; history chunks of 64 + 1 rows'),
    ('b150_h50_c9', 150, 50, 9, dict(variable_candidates=True),
     'G = 2, 300 units over 148 CTAs: atomic dxh, groups of one impression on different CTAs, last group of 1'),
    ('b160_h129_c17', 160, 129, 17, dict(variable_history=True),
     'G = 3, B > 148: CTAs holding two impressions on the read-modify-write dxh path; chunks of 64 + 64 + 1 rows'),
    ('b40_h64_c40', 40, 64, 40, {}, 'G = 5: 8 x 64 = 512 stacked rows, exactly 4 tiles per chunk'),
    ('b300_h37_c5', 300, 37, 5, {}, 'G = 1 with several units per CTA; FFMA persistent backward with B > 148'),
    ('b2000_h20_c5', 2000, 20, 5, {}, 'R = 10000 > 148 * 64: tensor-core head CTAs with several tiles, last-CTA BatchNorm sums'),
]
CASE_IDS = [c[0] for c in CASES]
CASE = {c[0]: c for c in CASES}

# rtol per buffer and precision (see the module docstring for the floors they come from): RTOL for every case with B >= 7, RTOL_SMALL
# for the two ill-conditioned smallest batches (SMALL_CASES)
RTOL = {
    'fp32': dict(xh=2e-6, e_label=4e-6, e_textimg=2e-6, e_direct=5e-7, logits=2e-5, de=1e-5, dxh=2e-5, dxt=4e-7, dxin_h=2e-6,
                 grad_head=7e-6, grad_attention=8e-6, grad_w1=5e-6, grad_embed=2e-5),
    'bf16x3': dict(xh=2e-6, e_label=8e-5, e_textimg=4e-5, e_direct=5e-7, logits=5e-5, de=5e-5, dtp_label=5e-5, dtp_textimg=2e-4,
                   dxh=6e-5, dxt=2e-6, dxin_h=4e-5, grad_head=7e-5, grad_attention=2e-4, grad_w1=2e-5, grad_embed=5e-6),
    'bf16': dict(xh=2e-6, e_label=3e-2, e_textimg=3e-2, e_direct=5e-7, logits=2e-4, de=3e-4, dtp_label=3e-2, dtp_textimg=1e-1,
                 dxh=3e-2, dxt=8e-4, dxin_h=2e-2, grad_head=3e-2, grad_attention=7e-2, grad_w1=7e-3, grad_embed=6e-6),
}
SMALL_CASES = ('b2_h1_c1', 'b1_h50_c5')
RTOL_SMALL = {
    'fp32': dict(xh=6e-7, e_label=2e-4, e_textimg=2e-6, e_direct=2e-7, logits=4e-5, de=7e-6, dxh=2e-4, dxt=2e-7, dxin_h=1e-6,
                 grad_head=2e-5, grad_attention=1e-5, grad_w1=6e-7, grad_embed=5e-4),
    'bf16x3': dict(xh=6e-7, e_label=3e-4, e_textimg=2e-5, e_direct=2e-7, logits=2e-4, de=2e-5, dtp_label=2e-5, dtp_textimg=3e-5,
                   dxh=2e-4, dxt=2e-7, dxin_h=2e-5, grad_head=3e-4, grad_attention=2e-4, grad_w1=3e-5, grad_embed=2e-4),
    'bf16': dict(xh=6e-7, e_label=5e-1, e_textimg=1e-2, e_direct=2e-7, logits=3e-4, de=2e-5, dtp_label=1e-2, dtp_textimg=2e-2,
                 dxh=6e-1, dxt=2e-5, dxin_h=2e-2, grad_head=9e-2, grad_attention=9e-2, grad_w1=2e-2, grad_embed=3e-4),
}


def rtol_for(precision, name, case_id):
    return (RTOL_SMALL if case_id in SMALL_CASES else RTOL)[precision][name]


ATOL_FRACTION = 0.01   # atol = rtol / 100, for impressions whose own scale is near zero
FLOORS = {}            # (precision, buffer, case id) -> worst err / impression scale seen by this run

class DtpNotWritten(UserWarning):
    """The precision under test does not write the dtp workspace buffer, so it is not compared."""


WS_FIELDS = ('xh', 'e', 'de', 'dtp', 'dxh', 'dxt', 'dxin_h')
MODE_TRAIN = 3         # MODE_BN_BATCH_STATS | MODE_KEEP_FOR_BWD


def _batch(case):
    _, B, H, C, kw, _ = case
    return make_batch(B, H, C, seed=B * 1000 + H * 10 + C, user_num=USERS, fp32_exact=True, **kw)


def _cotangent(B, C):
    return torch.randn(B, C, generator=torch.Generator().manual_seed(B * 7 + C), dtype=torch.float32)


def _model(precision):
    model = nrm.UserModel(USERS)
    model.load_state_dict(load_weights('train'), strict=False)
    return model.to(DEV).train().set_precision(precision)


def _ws_fields(model, B, H, C):
    lib = _lib.load()
    ws = model._runtime().train_ws
    out = {}
    for f in WS_FIELDS:
        nb = ctypes.c_longlong()
        off = lib.nrm_debug_ws_field(B, H, C, MODE_TRAIN, f.encode(), ctypes.byref(nb))
        assert off >= 0, f
        out[f] = ws[off:off + nb.value].view(torch.float32).clone()
    R, NH = B * C, B * H
    out['xh'] = out['xh'].view(NH, 64); out['dxh'] = out['dxh'].view(NH, 64); out['dxin_h'] = out['dxin_h'].view(NH, 66)
    out['e'] = out['e'].view(R, 264); out['de'] = out['de'].view(R, 264); out['dxt'] = out['dxt'].view(R, 64)
    out['dtp'] = out['dtp'].view(2, R, 64)
    return out


def gpu_step(model, x_history, x_target, x_global, G):
    """One training forward + out.backward(G) -> (logits, workspace buffers, parameter gradients), all cloned."""
    model.zero_grad(set_to_none=True)
    out = model(x_history, x_target, x_global)
    out.backward(G)
    torch.cuda.synchronize()
    B, H, C = x_history.shape[0], x_history.shape[1], x_target.shape[1]
    grads = {k: v.grad.detach().clone() for k, v in model.named_parameters() if v.grad is not None}
    return out.detach().clone(), _ws_fields(model, B, H, C), grads


def run_case(case_id, precision):
    case = CASE[case_id]
    b = _batch(case)
    d = b.to(DEV)
    G = _cotangent(case[1], case[3]).to(DEV)
    logits, bufs, grads = gpu_step(_model(precision), d.x_history, d.x_target, d.x_global, G)
    return dict(logits=logits, bufs=bufs, grads=grads)


def _params64():
    p = O.load_params(load_weights('train'), dtype=torch.float64, user_num=USERS)
    return {k: v.to(DEV) for k, v in p.items()}


def _check_rows(name, got, ref, precision, case, failures):
    """got / ref [B, n, k]; per impression scale."""
    rtol = rtol_for(precision, name, case[0])
    got, ref = got.double(), ref.double()
    err = torch.nan_to_num((got - ref).abs(), nan=float('inf'))
    imp = ref.abs().amax(dim=(1, 2))
    buf = ref.abs().max()
    ratio = err / imp.clamp_min(1e-30)[:, None, None]
    key = (precision, name, case[0])
    FLOORS[key] = max(FLOORS.get(key, 0.0), float(ratio.max()))
    allowed = rtol * imp[:, None, None] + ATOL_FRACTION * rtol * buf
    over = err / allowed.clamp_min(1e-30)
    if float(over.max()) > 1.0:
        b, n, k = np.unravel_index(int(over.argmax()), tuple(over.shape))
        idx = 'h' if name in ('xh', 'dxh', 'dxin_h') else 'c'
        failures.append(f'{name} [{precision}, {case[0]}: {case[5]}]: worst at b={b} {idx}={n} col={k}: gpu {float(got[b, n, k]):.6e} '
                        f'ref {float(ref[b, n, k]):.6e}, err / impression scale {float(ratio[b, n, k]):.2e} > rtol {rtol:.1e}')


def check_step(case, precision, res, failures):
    """Compare one GPU step (run_case) with the stage references fed its own buffers."""
    _, B, H, C, _, _ = case
    R = B * C
    b = _batch(case)
    bufs = {k: v.to(DEV) for k, v in res['bufs'].items()}
    G = _cotangent(B, C).to(DEV)
    up = {k: bufs[k].double() for k in ('xh', 'e', 'de', 'dxh', 'dxt', 'dxin_h')}
    with torch.no_grad():
        ref, grads = stage_references(_params64(), b.x_history.to(DEV), b.x_target.to(DEV), b.x_global.to(DEV), G.double(), gpu=up)
    rows_h = lambda t: t.reshape(B, H, -1)
    rows_c = lambda t: t.reshape(B, C, -1)
    chk = lambda name, g, r: _check_rows(name, g, r, precision, case, failures)
    chk('xh', rows_h(bufs['xh']), rows_h(ref['xh']))
    chk('e_label', rows_c(bufs['e'][:, 0:64]), rows_c(ref['e'][:, 0:64]))
    chk('e_textimg', rows_c(bufs['e'][:, 64:128]), rows_c(ref['e'][:, 64:128]))
    chk('e_direct', rows_c(bufs['e'][:, 128:]), rows_c(ref['e'][:, 128:]))
    chk('logits', rows_c(res['logits'].to(DEV)), rows_c(ref['logits']))
    chk('de', rows_c(bufs['de']), rows_c(ref['de']))
    if precision == 'fp32':
        warnings.warn(f'dtp not compared [fp32, {case[0]}]: the FFMA backward keeps dL/dtp in registers and never writes the buffer',
                      DtpNotWritten)
    else:
        chk('dtp_label', rows_c(bufs['dtp'][0]), rows_c(ref['dtp'][0]))
        chk('dtp_textimg', rows_c(bufs['dtp'][1]), rows_c(ref['dtp'][1]))
    chk('dxh', rows_h(bufs['dxh']), rows_h(ref['dxh']))
    chk('dxt', rows_c(bufs['dxt']), rows_c(ref['dxt']))
    chk('dxin_h', rows_h(bufs['dxin_h']), rows_h(ref['dxin_h']))
    for k, r in grads.items():
        if k == 'delta':
            continue
        name = 'grad_' + grad_stage(k)
        g = res['grads'][k].to(DEV).double()
        err = float(torch.nan_to_num((g - r).abs(), nan=float('inf')).max())
        scale = max(float(r.abs().max()), 1e-30)
        key = (precision, name, case[0])
        FLOORS[key] = max(FLOORS.get(key, 0.0), err / scale)
        rtol = rtol_for(precision, name, case[0])
        if err > rtol * scale:
            failures.append(f'{name} {k} [{precision}, {case[0]}: {case[5]}]: max err {err:.3e} = {err / scale:.2e} of max|ref| {scale:.3e} '
                            f'> rtol {rtol:.1e}')


@pytest.fixture(scope='module', autouse=True)
def _report_floors():
    yield
    if not FLOORS:
        return
    worst = {}
    for (prec, name, cid), v in FLOORS.items():
        key = (cid in SMALL_CASES, prec, name)
        if v >= worst.get(key, (-1.0, ''))[0]:
            worst[key] = (v, cid)
    lines = ['measured floors (worst err / impression scale over the cases run):']
    for (small, prec, name), (v, cid) in sorted(worst.items()):
        lines.append(f'  {"small" if small else "B >= 7":6s} {prec:7s} {name:15s} {v:.3e} ({cid})   rtol {rtol_for(prec, name, cid):.1e}')
    print('\n'.join(lines))
    path = os.environ.get('NRM_STAGEWISE_FLOORS')
    if path:
        with open(path, 'w') as f:
            json.dump({f'{p}/{n}/{c}': v for (p, n, c), v in sorted(FLOORS.items())}, f, indent=1)


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('case_id', CASE_IDS)
def test_stagewise_against_float64(case_id, precision):
    case = CASE[case_id]
    failures = []
    check_step(case, precision, run_case(case_id, precision), failures)
    assert not failures, '\n'.join(failures)


@pytest.mark.parametrize('precision', PRECISIONS)
def test_trimmed_candidate_views_bit_identical(precision):
    """x_target[:, :C-k] / x_global[:, :C-k] views (batch stride of the untrimmed tensor, as test.py:52-56 makes them) give the
    same logits and gradients, bit for bit, as .contiguous() copies.  C - k = 17 candidates: three groups on the row-stacked path."""
    B, H, C, keep = 20, 30, 20, 17
    b = make_batch(B, H, C, seed=404, user_num=USERS, variable_candidates=True).to(DEV)
    xt, xg = b.x_target[:, :keep], b.x_global[:, :keep]
    assert xt.stride(0) == C * xt.shape[2] and not xt.is_contiguous()
    G = _cotangent(B, keep).to(DEV)
    model = _model(precision)
    l_view, _, g_view = gpu_step(model, b.x_history, xt, xg, G)
    l_copy, _, g_copy = gpu_step(model, b.x_history, xt.contiguous(), xg.contiguous(), G)
    assert torch.equal(l_view, l_copy)
    assert g_view.keys() == g_copy.keys()
    for k in g_view:
        assert torch.equal(g_view[k], g_copy[k]), k


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('case_id', ['b150_h50_c9', 'b160_h129_c17'])
def test_dxh_bit_identical_run_to_run(case_id, precision):
    """G = 2 (atomic adds of two groups into a zeroed dxh) and G = 3 (read-modify-write across the groups of a CTA): two runs of
    the same step write the same dxh and dxt bit for bit.  At G = 2 each dxh element receives exactly two atomic adds into zero,
    and 0 + a + b == 0 + b + a, so the kernels as they stand cannot fail that case: it guards the accumulation scheme, and fails as
    soon as an element gets a third addend in run-dependent order (more groups, or chunks of one group added separately)."""
    case = CASE[case_id]
    b = _batch(case).to(DEV)
    G = _cotangent(case[1], case[3]).to(DEV)
    model = _model(precision)
    _, first, _ = gpu_step(model, b.x_history, b.x_target, b.x_global, G)
    _, second, _ = gpu_step(model, b.x_history, b.x_target, b.x_global, G)
    for f in ('dxh', 'dxt'):
        same = first[f] == second[f]
        assert bool(same.all()), (f, case[5], 'differing rows', torch.nonzero(~same.all(dim=-1)).flatten()[:16].tolist())
