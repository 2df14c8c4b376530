"""bf16 tensor-core path (tcgen05): building-block self test and forward parity at bf16 tolerance."""
import ctypes

import numpy as np
import pytest
import torch

from news_recommendation_model_b200 import _lib
from fixtures import load_weights
from news_recommendation_model_b200.synthetic import make_batch
from oracle import reference_port as O
import parity as P

pytestmark = pytest.mark.gpu

# bf16 operands (8-bit mantissa) in the pair GEMM, fp32 accumulation and fp32 everywhere else.
TOL_LOGITS_BF16 = 3e-2


@pytest.mark.parametrize('mode', [0, 1, 2])
@pytest.mark.parametrize('split', [1, 3])
def test_umma_building_blocks(mode, split):
    """tcgen05 descriptors (K-major and MN-major views of one tile), half-lane accumulator pairing, hi/lo split."""
    lib = _lib.load()
    torch.manual_seed(0)
    mats = [torch.randn(64, 64, device='cuda') for _ in range(4)]
    out = torch.full((2, 64, 64), float('nan'), device='cuda')
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    _lib.check(lib.nrm_debug_umma_selftest(p(mats[0]), p(mats[1]), p(mats[2]), p(mats[3]), p(out), mode, split, None), 'selftest')
    torch.cuda.synchronize()
    for q in range(2):
        a, b = mats[q].double(), mats[2 + q].double()
        if split == 1:
            a, b = mats[q].bfloat16().double(), mats[2 + q].bfloat16().double()
        ref = {0: a @ b.t(), 1: a.t() @ b, 2: a @ b}[mode]
        err = (out[q].double() - ref).abs().max().item()
        tol = 1e-3 if split == 1 else 2e-4          # split 3: ~2^-16 relative per product, 64 products of magnitude ~1
        assert err < tol, (mode, split, q, err, out[q][:2, :4], ref[:2, :4])


@pytest.mark.parametrize('B,H,C,kw', [(16, 50, 5, {}), (5, 13, 4, dict(variable_history=True)),
                                      (3, 130, 3, dict(variable_history=True)), (4, 64, 19, dict(variable_candidates=True))])
def test_bf16_forward_close_to_oracle(B, H, C, kw):
    b = make_batch(B, H, C, seed=B * 100 + H, user_num=40, **kw)
    model, p = P.build_models(load_weights('train'), 40)
    model.set_precision('bf16').eval()
    d = b.to('cuda')
    with torch.no_grad():
        out = model(d.x_history, d.x_target, d.x_global).cpu()
        ref = O.user_model_forward(p, b.x_history, b.x_target, b.x_global, training=False)
    err = (out - ref).abs().max().item()
    assert err <= TOL_LOGITS_BF16, err
    # and it must really be a different (rounded) computation from the fp32 path, not a silent alias
    model.set_precision('fp32')
    with torch.no_grad():
        out32 = model(d.x_history, d.x_target, d.x_global).cpu()
    assert (out32 - ref).abs().max().item() <= 5e-4
    assert (out32 - out).abs().max().item() > 0


def test_bf16_training_step_runs_and_is_close():
    b = make_batch(32, 50, 5, seed=8, user_num=40)
    model, p = P.build_models(load_weights('train'), 40)
    model.set_precision('bf16')
    rep = P.compare_step(model, p, b, training=True)
    assert rep['logits'] <= TOL_LOGITS_BF16, P.format_report(rep)
    assert rep['loss'] <= 5e-3, P.format_report(rep)
    for k, (err, scale) in rep['grads'].items():
        if k in P.NOISE_KEYS:
            continue
        assert err <= 0.05 * scale + 1e-6, (k, err, scale)


# ---- bf16x3: the tensor-core path must meet the SAME tolerances as the fp32 FFMA path -------------------
@pytest.mark.parametrize('B,H,C,kw', [
    (64, 50, 5, {}),
    (7, 13, 4, dict(variable_history=True)),
    (3, 130, 3, dict(variable_history=True)),
    (5, 64, 19, dict(variable_candidates=True)),
    (33, 50, 15, dict(variable_candidates=True)),
])
def test_bf16x3_training_step_meets_fp32_tolerance(B, H, C, kw):
    b = make_batch(B, H, C, seed=B * 1000 + H, user_num=40, **kw)
    delta0 = torch.from_numpy(np.random.default_rng(3).normal(0, 0.3, 41).astype(np.float32))
    model, p = P.build_models(load_weights('train'), 40, delta0)
    model.set_precision('bf16x3')
    rep = P.compare_step(model, p, b, training=True)
    assert rep['logits'] <= P.TOL_LOGITS, P.format_report(rep)
    assert rep['loss'] <= P.TOL_LOSS, P.format_report(rep)
    assert not P.grad_failures(rep), P.format_report(rep)


def test_bf16x3_eval_forward_meets_fp32_tolerance():
    b = make_batch(9, 200, 12, seed=77, user_num=40, variable_history=True, variable_candidates=True)
    model, p = P.build_models(load_weights('validation'), 40)
    model.set_precision('bf16x3').eval()
    d = b.to('cuda')
    with torch.no_grad():
        out = model(d.x_history, d.x_target, d.x_global).cpu()
        ref = O.user_model_forward(p, b.x_history, b.x_target, b.x_global, training=False)
    assert (out - ref).abs().max().item() <= P.TOL_LOGITS
