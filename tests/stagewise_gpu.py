"""GPU side of the stagewise float64 checks, shared by tests/test_gpu_stagewise.py (the training step) and
tests/test_gpu_stagewise_eval.py (the eval forward and the frozen-BatchNorm backward): the case table of the attention kernels'
work-split regimes, the seeded batches, cotangents and models, workspace buffers read back by name (nrm_debug_ws_field), the
per-row and per-tensor comparisons, and the report of the measured floors."""
import ctypes
import json
import os

import numpy as np
import torch

import news_recommendation_model_b200 as nrm
from news_recommendation_model_b200 import _lib, engine
from fixtures import load_weights
from news_recommendation_model_b200.synthetic import make_batch
from oracle import reference_port as O

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

ATOL_FRACTION = 0.01   # atol = rtol / 100, for impressions whose own scale is near zero
WS_FIELDS = ('xh', 'e', 'de', 'dtp', 'dxh', 'dxt', 'dxin_h')
ROWS_H = ('xh', 'dxh', 'dxin_h')                     # buffers with one row per history row; the others have one per candidate
MODE_TRAIN = engine.MODE_BN_BATCH_STATS | engine.MODE_KEEP_FOR_BWD
ALL_FLOORS = {}        # the floors of every module run in this session, written to NRM_STAGEWISE_FLOORS


class DtpNotWritten(UserWarning):
    """The precision under test does not write the dtp workspace buffer, so it is not compared."""


def batch(case):
    _, B, H, C, kw, _ = case
    return make_batch(B, H, C, seed=B * 1000 + H * 10 + C, user_num=USERS, fp32_exact=True, **kw)


def cotangent(B, C):
    return torch.randn(B, C, generator=torch.Generator().manual_seed(B * 7 + C), dtype=torch.float32)


def model(precision, checkpoint='train'):
    m = nrm.UserModel(USERS)
    m.load_state_dict(load_weights(checkpoint), strict=False)
    return m.to(DEV).train().set_precision(precision)


def params64(checkpoint='train'):
    p = O.load_params(load_weights(checkpoint), dtype=torch.float64, user_num=USERS)
    return {k: v.to(DEV) for k, v in p.items()}


def ws_fields(model, B, H, C, mode=MODE_TRAIN, fields=WS_FIELDS):
    """Clones of the named buffers of the workspace the last forward of `mode` used (the training workspace when the mode keeps
    activations for the backward, the eval workspace otherwise), shaped [rows, columns]."""
    lib = _lib.load()
    rt = model._runtime()
    ws = rt.train_ws if mode & engine.MODE_KEEP_FOR_BWD else rt.eval_ws
    cols = dict(xh=64, dxh=64, dxin_h=66, e=264, de=264, dxt=64, dtp=64)
    out = {}
    for f in fields:
        nb = ctypes.c_longlong()
        off = lib.nrm_debug_ws_field(B, H, C, mode, f.encode(), ctypes.byref(nb))
        assert off >= 0, f
        out[f] = ws[off:off + nb.value].view(torch.float32).clone()
        out[f] = out[f].view(2, B * C, 64) if f == 'dtp' else out[f].view(-1, cols[f])
    return out


def check_rows(name, got, ref, rtol, label, floors, key, failures):
    """got / ref [B, n, k]: one impression per leading index.  An element passes when |got - ref| <= rtol * max|ref over its
    impression| + ATOL_FRACTION * rtol * max|ref over the buffer|; floors[key] keeps the worst err / impression scale."""
    got, ref = got.double(), ref.double()
    err = torch.nan_to_num((got - ref).abs(), nan=float('inf'))
    imp = ref.abs().amax(dim=(1, 2))
    buf = ref.abs().max()
    ratio = err / imp.clamp_min(1e-30)[:, None, None]
    floors[key] = max(floors.get(key, 0.0), float(ratio.max()))
    allowed = rtol * imp[:, None, None] + ATOL_FRACTION * rtol * buf
    over = err / allowed.clamp_min(1e-30)
    if float(over.max()) > 1.0:
        b, n, k = np.unravel_index(int(over.argmax()), tuple(over.shape))
        idx = 'h' if name in ROWS_H else 'c'
        failures.append(f'{name} [{label}]: worst at b={b} {idx}={n} col={k}: gpu {float(got[b, n, k]):.6e} '
                        f'ref {float(ref[b, n, k]):.6e}, err / impression scale {float(ratio[b, n, k]):.2e} > rtol {rtol:.1e}')


def check_grad(name, k, got, ref, rtol, label, floors, key, failures):
    """A whole parameter gradient: |got - ref| <= rtol * max|ref| of that tensor."""
    err = float(torch.nan_to_num((got.double() - ref).abs(), nan=float('inf')).max())
    scale = max(float(ref.abs().max()), 1e-30)
    floors[key] = max(floors.get(key, 0.0), err / scale)
    if err > rtol * scale:
        failures.append(f'{name} {k} [{label}]: max err {err:.3e} = {err / scale:.2e} of max|ref| {scale:.3e} > rtol {rtol:.1e}')


def report_floors(floors, group, columns, rtol_of, where=lambda key: key[-1]):
    """Print the worst floor of each tolerance group (group(key) -> sort key of the group; columns(group) -> its printed
    columns; rtol_of(key) -> the rtol the key is checked against; where(key) -> the case it came from), and write every floor
    measured in this session as JSON to $NRM_STAGEWISE_FLOORS when set."""
    if not floors:
        return
    worst = {}
    for key, v in floors.items():
        g = group(key)
        if v >= worst.get(g, (-1.0, None))[0]:
            worst[g] = (v, key)
    lines = ['measured floors (worst err / impression scale over the cases run):']
    for g, (v, key) in sorted(worst.items()):
        lines.append(f'  {columns(g)} {v:.3e} ({where(key)})   rtol {rtol_of(key):.1e}')
    print('\n'.join(lines))
    ALL_FLOORS.update(floors)
    path = os.environ.get('NRM_STAGEWISE_FLOORS')
    if path:
        with open(path, 'w') as f:
            json.dump({'/'.join(k): v for k, v in sorted(ALL_FLOORS.items())}, f, indent=1)
