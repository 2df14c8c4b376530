"""CPU-side checks of the drop-in boundary: module surface, state_dict contract, seeded
initialisation, C-ABI exports.  No kernel is launched here."""
import ctypes
import os
import pickle
import re
import sys

import pytest
import torch

import news_recommendation_model_b200 as nrm
from news_recommendation_model_b200 import _lib, engine
from fixtures import load_weights
from oracle import reference_port as O
from oracle.make_ref import reference_root

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = reference_root()


def test_state_dict_contract():
    m = nrm.UserModel(7)
    sd = m.state_dict()
    assert list(sd.keys()) == ['delta'] + [k for k, _ in O.STATE_KEYS]
    for k, shape in O.STATE_KEYS:
        assert tuple(sd[k].shape) == shape, k
    assert sd['delta'].shape == (8,)
    assert [k for k, _ in m.named_parameters()][0] == 'delta'            # train.py:96 pops it by name
    res = m.load_state_dict(load_weights('train'), strict=False)         # test.py:160
    assert res.missing_keys == ['delta'] and res.unexpected_keys == []
    assert int(m.bn.num_batches_tracked) == 3000
    assert m.bn.num_features == 264 and m.instant_interest_model.output_dim == 8
    assert m.invariant_interest_model.embed_setting == [32, 16, 8, 8]


def test_model_survives_pickle_and_deepcopy():
    import copy
    m = nrm.UserModel(3)
    m2 = pickle.loads(pickle.dumps(m))                                   # test.py:177 ships models to a child process
    m3 = copy.deepcopy(m)
    for a, b, c in zip(m.parameters(), m2.parameters(), m3.parameters()):
        assert torch.equal(a, b) and torch.equal(a, c)


def test_cpu_forward_fails_loudly():
    from news_recommendation_model_b200.synthetic import make_batch
    b = make_batch(2, 3, 2)
    m = nrm.UserModel(5)
    with pytest.raises(nrm.NrmError, match='CUDA'):
        m(b.x_history, b.x_target, b.x_global)


@pytest.mark.skipif(REF is None, reason="the original project's source is not in the tree (baseline/_ref, oracle/make_ref.py)")
def test_seeded_init_matches_reference(tmp_path):
    """train.py:42-46: torch.manual_seed(seed); UserModel(max_user_id) -- same constructors in the
    same order must leave the same initial weights."""
    import subprocess
    code = ("import sys, torch; sys.path.insert(0, %r); sys.dont_write_bytecode = True\n"
            "from models.user_model import UserModel\n"
            "torch.manual_seed(1234); m = UserModel(11)\n"
            "torch.save(m.state_dict(), sys.argv[1])\n") % REF
    path = str(tmp_path / 'ref_init.pth')
    subprocess.run([sys.executable, '-c', code, path], check=True, cwd=str(tmp_path))
    ref = torch.load(path)
    torch.manual_seed(1234)
    ours = nrm.UserModel(11).state_dict()
    assert list(ref.keys()) == list(ours.keys())
    for k in ref:
        assert torch.equal(ref[k], ours[k]), k


def test_shipped_checkpoints_load_unchanged(tmp_path):
    """test.py:159-160 loads ckpt/ckpt_ebnerd_large_{train,validation}_final.pth.  Every tensor of those checkpoints is stored,
    in checkpoint order, in tests/golden/weights_*.npz (make_golden.py:dump_weights); written back as a .pth and loaded the way
    test.py loads it, each reaches the model unchanged."""
    for name in ('train', 'validation'):
        path = tmp_path / f'ckpt_ebnerd_large_{name}_final.pth'
        torch.save(load_weights(name), path)
        sd = torch.load(path, map_location='cpu')
        m = nrm.UserModel()
        res = m.load_state_dict(sd, strict=False)
        assert res.missing_keys == ['delta'] and res.unexpected_keys == []
        gold = load_weights(name)
        for k, v in m.state_dict().items():
            if k != 'delta':
                assert torch.equal(v, gold[k]), k


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, 'include', 'nrm_b200.h')).read()
    declared = set(re.findall(r'\b(nrm_[a-z0-9_]+)\s*\(', header))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _lib.load().nrm_version() >= 100


def test_ctypes_bindings_have_the_parameter_count_of_the_header():
    """Every prototype of include/nrm_b200.h against the ctypes signature `_lib` binds: same number of parameters (a drifted
    binding passes garbage instead of failing)."""
    header = open(os.path.join(ROOT, 'include', 'nrm_b200.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    protos = re.findall(r'\b(nrm_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;', header)
    assert len(protos) == len(_lib.SIGNATURES)
    for name, params in protos:
        params = params.strip()
        n = 0 if params in ('', 'void') else len(params.split(','))
        assert n == len(_lib.SIGNATURES[name][1]), (name, n, len(_lib.SIGNATURES[name][1]))


def test_flat_layout_matches_reference_keys():
    entries, fixed = engine.layout()
    names = [n for n, _, _ in entries]
    assert names == list(O.TRAINABLE_KEYS) + ['delta']
    shapes = dict(O.STATE_KEYS)
    end = 0
    for name, off, numel in entries[:-1]:
        n = 1
        for d in shapes[name]:
            n *= d
        assert numel == n and off % 4 == 0 and off >= end, name
        end = off + numel
    assert entries[-1][1] == fixed and fixed % 4 == 0 and fixed >= end
    lib = _lib.load()
    assert lib.nrm_workspace_bytes(0, 1, 1, 0) == 0
    small, big = lib.nrm_workspace_bytes(4, 5, 3, 0), lib.nrm_workspace_bytes(4, 5, 3, 3)
    assert 0 < small < big


def test_argument_errors_are_reported_without_a_gpu():
    lib = _lib.load()
    rc = lib.nrm_adam_step(None, None, None, None, 10, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, 1.0, None)
    assert rc == -1 and b'nrm_adam_step' in lib.nrm_last_error()
    rc = lib.nrm_forward(None, None, 0, None, 0, 0, 1, 1, None, None, None, None, 0, 0, None, None, 0, None)
    assert rc == -1


def test_gelu_approximation_restated_in_numpy():
    """csrc/nrm_common.cuh evaluates Phi(x) with Abramowitz-Stegun 7.1.26 (float32 FMAs, approximate rcp / ex2).
    Restated here in float32 numpy against scipy's erf in float64: the kernels' GELU and GELU' stay well
    inside the parity tolerances (torch's own float32 GELU is accurate to ~1e-6)."""
    import numpy as np
    from scipy.special import erf
    f = np.float32
    x = np.linspace(-12, 12, 480001).astype(f)
    z = np.abs(x) * f(0.70710678118654752440)
    t = f(1.0) / (f(0.3275911) * z + f(1.0))
    poly = t * f(1.061405429) + f(-1.453152027)
    poly = t * poly + f(1.421413741)
    poly = t * poly + f(-0.284496736)
    poly = t * poly + f(0.254829592)
    poly = poly * t
    w = np.abs(x) * f(0.84932180028801904272)                   # exp(-x^2/2) = 2^(-w^2): the kernels use ex2.approx
    ex = np.exp2((w * -w).astype(f)).astype(f)
    half = f(0.5) * poly * ex
    gelu = (-np.abs(x)) * half + np.maximum(x, f(0))            # gelu_f
    cdf = f(0.5) + np.copysign(f(0.5) - half, x)                # gelu_both
    grad = x * f(0.39894228040143267794) * ex + cdf
    assert np.abs(x * cdf - gelu).max() < 1e-6
    xd = x.astype(np.float64)
    cdf_ref = 0.5 * (1.0 + erf(xd / np.sqrt(2.0)))
    gelu_ref = xd * cdf_ref
    grad_ref = cdf_ref + xd * np.exp(-0.5 * xd * xd) / np.sqrt(2.0 * np.pi)
    assert np.abs(gelu - gelu_ref).max() < 1e-6
    assert np.abs(grad - grad_ref).max() < 1e-6


def test_models_shim_shadows_the_reference_package():
    """shim/ first on sys.path: the reference scripts' `from models.user_model import UserModel` gets this implementation."""
    import subprocess
    code = ("import sys; sys.path[:0] = [%r, %r]; from models.user_model import UserModel; from models.attention_model import MLP, "
            "PointwiseAttentionExpanded; from configs.model_config import config; import news_recommendation_model_b200 as n; "
            "assert UserModel is n.UserModel and MLP is n.MLP and config['pca_vector'] == 64; print('ok')") % (os.path.join(ROOT, 'shim'), ROOT)
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert out.returncode == 0 and 'ok' in out.stdout, out.stderr[-2000:]


def test_flat_params_views_and_gradient_split_plan_on_cpu():
    """engine.FlatParams is plain tensor plumbing (no kernels): the parameters become views of ONE buffer in layout order,
    and grad_views() (one split_with_sizes call) returns exactly the slices the layout describes."""
    import torch
    import news_recommendation_model_b200 as nrm
    from news_recommendation_model_b200 import engine
    m = nrm.UserModel(7)
    named = dict(m.named_parameters())
    flat = engine.FlatParams(named)
    assert flat.is_current(named) and flat.total % 4 == 0
    base = flat.buf.data_ptr()
    for name, off, n, shape in flat.slots:
        p = named[name]
        assert p.data_ptr() == base + 4 * off and p.numel() == n and tuple(p.shape) == tuple(shape)
    assert [id(p) for p in flat.params] == [id(named[name]) for name, _, _, _ in flat.slots if name != 'delta']
    g = torch.arange(flat.total, dtype=torch.float32)
    for skip in (False, True):
        views = flat.grad_views(g, skip)
        slots = [sl for sl in flat.slots if not (skip and sl[0] == 'delta')]
        assert len(views) == len(slots)
        for v, (name, off, n, shape) in zip(views, slots):
            assert tuple(v.shape) == tuple(shape) and v.data_ptr() == g.data_ptr() + 4 * off
            assert float(v.reshape(-1)[0]) == float(off) and float(v.reshape(-1)[-1]) == float(off + n - 1)
    # a buffer of another length falls back to plain slicing
    g2 = torch.zeros(flat.total + 8)
    assert len(flat.grad_views(g2, False)) == len(flat.slots)
