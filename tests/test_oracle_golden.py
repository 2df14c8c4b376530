"""Pin the oracle (oracle/reference_port.py) against what the UNMODIFIED reference computed
(tests/golden/*.npz, produced by tests/golden/make_golden.py in the build container)."""
import numpy as np
import pytest
import torch

from fixtures import case_batch, grad_scale, load_case, load_weights, stored
from oracle import reference_port as O

# identical ATen kernels on the same host give bit-equal results; leave a little room for
# other CPUs (different vector widths change summation order inside at::mm / at::sum)
TOL = 2e-6


def _train_step(case_name, weights='train'):
    case = load_case(case_name)
    b = case_batch(case)
    user_num = int(case['meta'][3])
    p = O.load_params(load_weights(weights), user_num=user_num)
    p['delta'] = torch.from_numpy(case['delta0'].copy())
    leaves = {k: p[k].requires_grad_(True) for k in O.TRAINABLE_KEYS + ('delta',)}
    out = O.user_model_forward(p, b.x_history, b.x_target, b.x_global, training=True)
    loss = O.user_model_loss(p['delta'], b.user_id, out, b.label)
    loss.backward()
    return case, p, leaves, out, loss


def test_train_step_matches_reference_b16():
    case, p, leaves, out, loss = _train_step('case_train_b16')
    assert np.abs(out.detach().numpy() - case['logits']).max() <= TOL
    assert abs(loss.item() - float(case['loss'])) <= TOL
    for k, leaf in leaves.items():
        ref = case['grad/' + k]
        err = np.abs(stored(case, k, leaf.grad.numpy()) - ref).max()
        tol = TOL * max(1.0, grad_scale(case, k))
        assert err <= tol, (k, err)
        if 'gradnorm/' + k in case.files:     # a sampled tensor: its whole gradient through the norm
            n_err = abs(leaf.grad.double().norm().item() - float(case['gradnorm/' + k]))
            assert n_err <= tol * np.sqrt(leaf.numel()), (k, n_err)
    # BN buffers after the training forward (momentum 0.1, unbiased running_var)
    for k in ('bn.running_mean', 'bn.running_var'):
        ref = case['after/' + k]
        assert np.abs(p[k].detach().numpy() - ref).max() <= TOL * max(1.0, np.abs(ref).max()), k
    assert int(p['bn.num_batches_tracked']) == int(case['after/bn.num_batches_tracked'])
    # one Adam step (train.py:48,74): first step => m = (1-b1) g, v = (1-b2) g^2.  It is fed the reference's gradient (checked
    # above): an element whose gradient is near eps moves by up to lr when that gradient changes in its last bits.  Fed the
    # oracle's own gradient, invariant_interest_model.text_img_attention.mlp.fc1.weight came out 8.5e-6 from the reference's
    # on the Intel Xeon host of a B200 machine (ATen AVX512 kernels), while another Xeon host with the same kernels matched
    with torch.no_grad():
        for k, leaf in leaves.items():
            param = torch.from_numpy(stored(case, k, leaf.detach().numpy()).copy())
            grad = torch.from_numpy(case['grad/' + k].copy())
            O.adam_step(param, grad, torch.zeros_like(param), torch.zeros_like(param), 1)
            ref = case['after/' + k]
            assert np.abs(param.numpy() - ref).max() <= TOL * max(1.0, np.abs(ref).max()), k


def test_config1_b64_matches_reference():
    case, p, leaves, out, loss = _train_step('case_cfg1_b64')
    assert np.abs(out.detach().numpy() - case['logits']).max() <= TOL
    assert abs(loss.item() - float(case['loss'])) <= TOL
    for k, leaf in leaves.items():
        ref = float(case['gradnorm/' + k])
        assert abs(leaf.grad.double().norm().item() - ref) <= 1e-5 * max(1.0, ref), k


def test_scoring_matches_reference_ragged_candidates():
    case = load_case('case_eval_b8')
    b = case_batch(case)
    sets = [O.load_params(load_weights(n)) for n in ('train', 'validation')]
    with torch.no_grad():
        for n, p in enumerate(sets):
            logits = O.user_model_forward(p, b.x_history, b.x_target, b.x_global, training=False)
            assert np.abs(logits.numpy() - case[f'eval_logits/{n}']).max() <= 2e-5   # 316x BN gain on dead channels
        B = int(case['meta'][0])
        rows = []
        for s in range(0, B, 4):          # make_golden scored with batch_size=4 (test.py trims per batch)
            rows += O.score_batch(sets, b.x_history[s:s + 4], b.x_target[s:s + 4], b.x_global[s:s + 4],
                                  b.empty_num[s:s + 4])
    for i, score in enumerate(rows):
        ref = case[f'score/{i}']
        assert score.shape[0] == ref.shape[0]
        assert np.abs(score.numpy() - ref).max() <= TOL
        assert O.rank_string(score.numpy()) == str(case['ranks'][i])
        assert abs(O.auc(b.label[i].numpy()[:len(ref)], score.numpy()) - case['auc'][i]) <= 1e-9


def test_state_key_table_matches_checkpoint():
    sd = load_weights('train')
    assert list(sd.keys()) == [k for k, _ in O.STATE_KEYS]
    for k, shape in O.STATE_KEYS:
        assert tuple(sd[k].shape) == shape
    assert sum(v.numel() for v in sd.values()) == 223860
