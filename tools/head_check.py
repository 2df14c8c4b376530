#!/usr/bin/env python
"""Full-size (B=1024, H=50, C=5) training step against the oracle: per-tensor gradient error / tolerance, in precision bf16x3 or
the one given as the fourth argument (fp32: the FFMA head, attention and w1 kernels; bf16 / bf16x3: the tensor-core ones)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import parity as P
from fixtures import load_weights
from news_recommendation_model_b200.synthetic import make_batch
from oracle import reference_port as O

B = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
H = int(sys.argv[2]) if len(sys.argv) > 2 else 50
C = int(sys.argv[3]) if len(sys.argv) > 3 else 5
PRECISION = sys.argv[4] if len(sys.argv) > 4 else 'bf16x3'
U = 1000
b = make_batch(B, H, C, seed=2024, user_num=U)
delta0 = torch.from_numpy(np.random.default_rng(11).normal(0, 0.3, U + 1).astype(np.float32))
model, p = P.build_models(load_weights('train'), U, delta0)
model.train().set_precision(PRECISION)
leaves = {k: p[k].requires_grad_(True) for k in O.TRAINABLE_KEYS + ('delta',)}
out_o = O.user_model_forward(p, b.x_history, b.x_target, b.x_global, training=True)
loss_o = O.user_model_loss(p['delta'], b.user_id, out_o, b.label)
loss_o.backward()
g_o = {k: v.grad.detach().clone() for k, v in leaves.items()}
d = b.to('cuda')
out = model(d.x_history, d.x_target, d.x_global)
loss = model.loss(d.user_id, out, d.label)
loss.backward()
g_c = {k: v.grad.detach().cpu().clone() for k, v in model.named_parameters()}
print(PRECISION, 'B', B, 'H', H, 'C', C,
      'logits err %.2e' % (out.detach().cpu() - out_o.detach()).abs().max().item(), 'loss err %.2e' % abs(float(loss) - float(loss_o)))
for k, go in g_o.items():
    scale = go.abs().max().item()
    tol = P.TOL_GRAD_ABS if k in P.NOISE_KEYS else P.TOL_GRAD_REL * scale + P.TOL_GRAD_ABS
    err = (g_c[k] - go).abs().max().item()
    print(f'  {k:62s} err {err:.2e}  scale {scale:.2e}  err/tol {err / tol:6.2f}' + ('   <-- FAIL' if err > tol else ''))
