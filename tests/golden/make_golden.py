#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED reference.

Runs only in the build container, where the reference is mounted read-only at
/root/reference (it does not exist on the GPU box).  It imports the reference's
own `models.user_model.UserModel`, loads the two shipped checkpoints, feeds it
seeded synthetic EB-NeRD-shaped batches (news_recommendation_model_b200.synthetic)
and stores what the reference computed:

  weights_*.npz          the 37 tensors of ckpt/ckpt_ebnerd_large_*_final.pth
  case_train_b16.npz     train-mode logits, loss, all 37 gradients (incl. dense
                         delta), post-Adam parameters and BN buffers for one
                         train.py:69-75 step (B=16,H=50,C=5,user_num=1000);
                         tensors of more than SAMPLE elements are stored at a
                         fixed seeded sample of them (sample_large), inputs
                         regenerated from the seed
  case_cfg1_b64.npz      BASELINE config 1 (B=64,H=50,C=5): train-mode logits,
                         loss, gradient norms (inputs regenerated from the seed)
  case_eval_b8.npz       test.py:31-74 scoring of ragged-candidate impressions
                         (H=200) with the 2-model ensemble: scores, ranks, AUC

Usage:  python tests/golden/make_golden.py     (from the repo root)
"""
import hashlib
import os
import queue
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = '/root/reference'
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)

from news_recommendation_model_b200.synthetic import make_batch  # noqa: E402


def import_reference():
    """Import the reference package tree without touching our own modules."""
    sys.path.insert(0, REF)
    # tool/process_data.py imports zstandard, absent here and irrelevant to the path
    sys.modules.setdefault('zstandard', types.ModuleType('zstandard'))
    from models.user_model import UserModel
    import test as ref_test                    # /root/reference/test.py (model_test)
    from tool.evaluation import auc_score
    return UserModel, ref_test, auc_score


SAMPLE = 8192          # keeps every fixture file under 1 MB


def sample_large(d):
    """For every gradient of more than SAMPLE elements: keep it and the updated tensor at a fixed seeded sample of SAMPLE
    flat indices (sample/<key>), plus the largest magnitude and the norm of the whole gradient (gradmax/, gradnorm/)."""
    for key in [k for k in d if k.startswith('grad/')]:
        k, g = key[len('grad/'):], d[key]
        if g.size <= SAMPLE:
            continue
        idx = np.sort(np.random.default_rng(0).choice(g.size, SAMPLE, replace=False)).astype(np.int64)
        d['sample/' + k] = idx
        d['gradmax/' + k] = np.array(np.abs(g).max(), dtype=np.float64)
        d['gradnorm/' + k] = np.array(np.linalg.norm(g.astype(np.float64)))
        d[key] = g.reshape(-1)[idx]
        d['after/' + k] = d['after/' + k].reshape(-1)[idx]
    return d


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def dump_weights(name):
    sd = torch.load(f'{REF}/ckpt/ckpt_ebnerd_large_{name}_final.pth', map_location='cpu')
    np.savez_compressed(f'{HERE}/weights_{name}_final.npz', **{k: v.numpy() for k, v in sd.items()})
    return sd


def batch_arrays(b, store_inputs):
    d = {'input_sha256': np.array(sha(b.x_history.numpy(), b.x_target.numpy(), b.x_global.numpy(),
                                      b.label.numpy(), b.user_id.numpy()))}
    if store_inputs:   # fp32_exact batches: float32 storage is lossless
        d.update(x_history=b.x_history.numpy().astype(np.float32), x_target=b.x_target.numpy().astype(np.float32),
                 x_global=b.x_global.numpy().astype(np.float32), label=b.label.numpy().astype(np.float32),
                 user_id=b.user_id.numpy(), empty_num=b.empty_num.numpy(), impression_id=b.impression_id.numpy())
    return d


def train_case(UserModel, sd, path, *, B, H, C, user_num, seed, store_inputs, full):
    torch.manual_seed(0)
    b = make_batch(B, H, C, seed=seed, user_num=user_num, fp32_exact=True)
    model = UserModel(user_num)
    model.load_state_dict(sd, strict=False)
    with torch.no_grad():     # non-zero delta so the personalised term differs from the plain one
        model.delta.copy_(torch.from_numpy(np.random.default_rng(seed + 1).normal(0, 0.3, user_num + 1).astype(np.float32)))
    delta0 = model.delta.detach().clone()
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)
    out = model(b.x_history, b.x_target, b.x_global)         # train.py:69
    loss = model.loss(b.user_id, out, b.label)               # train.py:71
    loss.backward()                                          # train.py:73
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
    opt.step()                                               # train.py:74
    d = batch_arrays(b, store_inputs)
    d.update(meta=np.array([B, H, C, user_num, seed]), logits=out.detach().numpy(), loss=np.array(loss.item(), dtype=np.float64),
             loss_f32=loss.detach().numpy(), delta0=delta0.numpy())
    if full:
        for k, g in grads.items():
            d['grad/' + k] = g.numpy()
        for k, v in model.state_dict().items():
            d['after/' + k] = v.numpy()
        sample_large(d)
    else:
        for k, g in grads.items():
            d['gradnorm/' + k] = np.array(g.double().norm().item())
            d['gradsum/' + k] = np.array(g.double().sum().item())
    np.savez_compressed(path, **d)
    print(path, 'loss', loss.item(), 'max|logit|', out.abs().max().item())


def eval_case(UserModel, ref_test, auc_score, sds, path, *, B, H, C, seed):
    b = make_batch(B, H, C, seed=seed, user_num=1000, variable_history=True, variable_candidates=True, fp32_exact=True)
    models = []
    for sd in sds:
        m = UserModel()
        m.load_state_dict(sd, strict=False)
        models.append(m)
    records = [[b.impression_id[i].numpy(), b.user_id[i].numpy(), b.x_history[i].numpy(), b.x_target[i].numpy(),
                b.x_global[i].numpy(), b.label[i].numpy(), b.label_id[i].numpy(), b.empty_num[i].numpy()] for i in range(B)]
    q, ids = ref_test.model_test(models, records, torch.device('cpu'), queue.Queue(), [], batch_size=4)   # test.py:31-74
    d = batch_arrays(b, True)
    d['meta'] = np.array([B, H, C, 1000, seed])
    aucs, ranks = [], []
    for i in range(B):
        _, _, score, _ = q.get()
        d[f'score/{i}'] = np.asarray(score)
        aucs.append(auc_score(b.label[i].numpy()[0:len(score)], score))      # verify.py:30
        order = sorted(enumerate(score), key=lambda x: x[1], reverse=True)   # test.py:124-127
        rk = ['-1'] * len(score)
        for r_i, (j, _) in enumerate(order):
            rk[j] = str(r_i + 1)
        ranks.append(','.join(rk))
    d['auc'] = np.array(aucs)
    d['ranks'] = np.array(ranks)
    # single-model eval logits (UserModel.forward in eval mode) for each checkpoint
    with torch.no_grad():
        for n, m in enumerate(models):
            m.eval()
            d[f'eval_logits/{n}'] = m(b.x_history, b.x_target, b.x_global).numpy()
    np.savez_compressed(path, **d)
    print(path, 'mean auc', float(np.mean(aucs)))


def main():
    UserModel, ref_test, auc_score = import_reference()
    sd_t = dump_weights('train')
    sd_v = dump_weights('validation')
    train_case(UserModel, sd_t, f'{HERE}/case_train_b16.npz', B=16, H=50, C=5, user_num=1000, seed=1234,
               store_inputs=False, full=True)
    train_case(UserModel, sd_t, f'{HERE}/case_cfg1_b64.npz', B=64, H=50, C=5, user_num=1000, seed=4321,
               store_inputs=False, full=False)
    eval_case(UserModel, ref_test, auc_score, [sd_t, sd_v], f'{HERE}/case_eval_b8.npz', B=8, H=200, C=24, seed=99)


if __name__ == '__main__':
    main()
