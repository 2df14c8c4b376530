"""Helpers shared by the tests: golden-fixture loading and input regeneration."""
import hashlib
import os

import numpy as np
import torch

from news_recommendation_model_b200.synthetic import Batch, make_batch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def load_weights(name: str):
    """name in {'train', 'validation'} -> reference state_dict (37 tensors, no delta)."""
    z = np.load(os.path.join(GOLDEN, f'weights_{name}_final.npz'))
    return {k: torch.from_numpy(z[k].copy()) for k in z.files}


def load_case(name: str):
    return np.load(os.path.join(GOLDEN, name + '.npz'))


def stored(case, key, a):
    """`a`, a whole tensor, at the elements the case stores for `key`: all of them, or the fixed sample in sample/<key>
    (tests/golden/make_golden.py:sample_large)."""
    a = np.asarray(a)
    return a.reshape(-1)[case['sample/' + key]] if 'sample/' + key in case.files else a


def grad_scale(case, key):
    """Largest |gradient| of the whole tensor (the stored gradient may be a sample)."""
    return float(case['gradmax/' + key]) if 'gradmax/' + key in case.files else float(np.abs(case['grad/' + key]).max())


def _sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def case_batch(case, **regen_kwargs) -> Batch:
    """Inputs of a golden case: stored (float32, lossless) or regenerated from the seed and
    checked against the stored SHA-256 of the float64 bytes."""
    B, H, C, user_num, seed = [int(v) for v in case['meta']]
    if 'x_history' in case.files:
        t = torch.from_numpy
        b = Batch(t(case['impression_id'].copy()), t(case['user_id'].copy()),
                  t(case['x_history'].astype(np.float64)), t(case['x_target'].astype(np.float64)),
                  t(case['x_global'].astype(np.float64)), t(case['label'].astype(np.float64)),
                  torch.zeros(B, C, dtype=torch.float64), t(case['empty_num'].copy()))
    else:
        b = make_batch(B, H, C, seed=seed, user_num=user_num, fp32_exact=True, **regen_kwargs)
    got = _sha(b.x_history.numpy(), b.x_target.numpy(), b.x_global.numpy(), b.label.numpy(), b.user_id.numpy())
    assert got == str(case['input_sha256']), 'golden inputs do not match their recorded checksum'
    return b
