"""ORACLE (test infrastructure, NOT product code): the kernels' algebra on the CPU.

`reference_port.py` restates the reference as written.  The CUDA kernels do not
compute it that way: they use the reduced form of the pairwise attention MLP and
hand-derived backward formulas (DESIGN.md §3).  This file states that algebra
once, in plain tensor ops with an explicit manual backward, so that it can be
checked against autograd of the as-written port on the CPU (tests/
test_reduced_algebra.py) before the same formulas are transliterated to CUDA.

Reduced attention (reference: attention_model.py:81-92).  With fc1 weight split in
four 64x64 blocks W = [Wa|Wb|Wc|Wd] over the concat [h, t, t-h, t*h]:

    fc1(concat)[c,h,:] = W_c h + tp_c,   W_c = Wd diag(t_c) + (Wa - Wc),
                                         tp_c = (Wb + Wc) t_c + b1

so one candidate's hidden tile is a plain GEMM of the history tile with a
candidate-specific 64x64 matrix, and no [B,C,H,256] tensor exists.
"""
from __future__ import annotations

import math
from typing import Dict, Tuple

import torch

from .reference_port import II

T = torch.Tensor


def gelu(x: T) -> T:
    return 0.5 * x * (1.0 + torch.erf(x * (1.0 / math.sqrt(2.0))))


def gelu_grad(x: T) -> T:
    return 0.5 * (1.0 + torch.erf(x * (1.0 / math.sqrt(2.0)))) + x * torch.exp(-0.5 * x * x) * (1.0 / math.sqrt(2.0 * math.pi))


# ---------------------------------------------------------------------------
# feature rows  (user_invariant_interest_model.py:58-79)
# ---------------------------------------------------------------------------

def decode_rows(x: T, dtype) -> Dict[str, T]:
    """x: [N, 80|78] float64 packed rows -> integer ids and float columns."""
    xf = x.to(dtype)
    d = dict(time=xf[:, 0:4].to(torch.int64), pca=xf[:, 4:68], cat=xf[:, 68].to(torch.int64),
             sub=xf[:, 69:74].to(torch.int64), sent=xf[:, 74:77], typ=xf[:, 77].to(torch.int64))
    if x.shape[1] == 80:
        d['extra'] = xf[:, 78:80]
    return d


def embed_rows(p, d) -> T:
    """-> xin [N, 64(+2)] = [cat+mean(sub) 32 | relu(sent) 16 | type 8 | time 8 | read_time, scroll]."""
    tab = p[II + 'category_embedding.0.weight']
    both = tab[d['cat']] + tab[d['sub']].sum(1) / 5.0
    sent = torch.relu(d['sent'] @ p[II + 'sentiment_embedding.0.weight'].t() + p[II + 'sentiment_embedding.0.bias'])
    typ = p[II + 'type_embedding.0.weight'][d['typ']]
    tm = (p[II + 'year_embedding.0.weight'][d['time'][:, 0]] + p[II + 'month_embedding.0.weight'][d['time'][:, 1]]
          + p[II + 'day_embedding.0.weight'][d['time'][:, 2]] + p[II + 'hour_embedding.0.weight'][d['time'][:, 3]])
    cols = [both, sent, typ, tm]
    if 'extra' in d:
        cols.append(d['extra'])
    return torch.cat(cols, dim=1)


def embed_rows_backward(p, d, xin: T, dxin: T, grads: Dict[str, T]) -> None:
    """Accumulate table / sentiment gradients from d(xin)[:, 0:64]."""
    def acc(key, idx, val):
        grads[key].index_add_(0, idx, val)
    acc(II + 'category_embedding.0.weight', d['cat'], dxin[:, 0:32])
    for s in range(5):
        acc(II + 'category_embedding.0.weight', d['sub'][:, s], dxin[:, 0:32] / 5.0)
    dpre = dxin[:, 32:48] * (xin[:, 32:48] > 0).to(dxin.dtype)
    grads[II + 'sentiment_embedding.0.weight'] += dpre.t() @ d['sent']
    grads[II + 'sentiment_embedding.0.bias'] += dpre.sum(0)
    acc(II + 'type_embedding.0.weight', d['typ'], dxin[:, 48:56])
    for i, name in enumerate(('year', 'month', 'day', 'hour')):
        acc(II + name + '_embedding.0.weight', d['time'][:, i], dxin[:, 56:64])


# ---------------------------------------------------------------------------
# reduced pairwise attention + pooling, forward and backward
# ---------------------------------------------------------------------------

def derived_weights(p, prefix) -> Tuple[T, T, T, T, T, T]:
    W = p[prefix + 'mlp.fc1.weight']
    Wa, Wb, Wc, Wd = W[:, 0:64], W[:, 64:128], W[:, 128:192], W[:, 192:256]
    return Wa - Wc, Wb + Wc, Wd, p[prefix + 'mlp.fc1.bias'], p[prefix + 'mlp.fc2.weight'][0], p[prefix + 'mlp.fc2.bias'][0]


def attention_forward(p, prefix, t: T, h: T):
    """t [B,C,64], h [B,H,64] -> pooled [B,C,64], (hid, s) for the backward."""
    A, Bm, Wd, b1, w2, b2 = derived_weights(p, prefix)
    tp = t @ Bm.t() + b1                                              # [B,C,64]
    Wc = Wd[None, None] * t[:, :, None, :] + A[None, None]            # [B,C,64j,64k]
    hid = torch.einsum('bcjk,bhk->bchj', Wc, h) + tp[:, :, None, :]   # [B,C,H,64]
    s = gelu(hid) @ w2 + b2                                           # [B,C,H]
    pooled = torch.einsum('bch,bhk->bck', s, h)
    return pooled, (Wc, hid, s)


def attention_backward(p, prefix, t: T, h: T, saved, dP: T, grads, need_input_grads: bool):
    """dP [B,C,64] -> (dt, dh, Gt): dt, dh are None for the text/img branch whose inputs are data; Gt [B,C,64] = dL/dtp
    (the sum of dhid over the history rows).  fc1/fc2 gradients are accumulated into `grads`."""
    A, Bm, Wd, b1, w2, b2 = derived_weights(p, prefix)
    Wc, hid, s = saved
    ds = torch.einsum('bck,bhk->bch', dP, h)
    act = gelu(hid)
    grads[prefix + 'mlp.fc2.weight'] += torch.einsum('bch,bchj->j', ds, act)[None]
    grads[prefix + 'mlp.fc2.bias'] += ds.sum().reshape(1)
    dhid = ds[..., None] * w2 * gelu_grad(hid)                        # [B,C,H,64j]
    Gt = dhid.sum(2)                                                  # [B,C,64j]
    S = torch.einsum('bchj,bhk->bcjk', dhid, h)                       # [B,C,64j,64k]
    dA = S.sum((0, 1))
    dWd = torch.einsum('bcjk,bck->jk', S, t)
    dBm = torch.einsum('bcj,bck->jk', Gt, t)
    grads[prefix + 'mlp.fc1.bias'] += Gt.sum((0, 1))
    grads[prefix + 'mlp.fc1.weight'] += torch.cat([dA, dBm, dBm - dA, dWd], dim=1)
    if not need_input_grads:
        return None, None, Gt
    dt = Gt @ Bm + torch.einsum('bcjk,jk->bck', S, Wd)
    dh = torch.einsum('bch,bck->bhk', s, dP) + torch.einsum('bchj,bcjk->bhk', dhid, Wc)
    return dt, dh, Gt


# ---------------------------------------------------------------------------
# stages of the training step.  Each takes its inputs as arguments, so that a test can feed one stage the
# upstream buffers of another implementation (tests/test_gpu_stagewise.py feeds the GPU's own).
# ---------------------------------------------------------------------------

def grad_buffers(p) -> Dict[str, T]:
    return {k: torch.zeros_like(v) for k, v in p.items() if v.dtype.is_floating_point and not k.startswith('bn.running')}


def w1_forward(p, xin_h: T) -> T:
    """xh = w1(xin_h)   (user_invariant_interest_model.py:78)"""
    return xin_h @ p[II + 'w1.weight'].t() + p[II + 'w1.bias']


def w1_backward(p, xin_h: T, dxh: T, grads) -> T:
    """-> dxin_h; w1 gradients accumulated into `grads`."""
    grads[II + 'w1.weight'] += dxh.t() @ xin_h
    grads[II + 'w1.bias'] += dxh.sum(0)
    return dxh @ p[II + 'w1.weight']


def instant_forward(p, x_global: T, dtype) -> Tuple[T, T]:
    """-> (g [R,3], eu_l [R,8] = relu(out_fc(g)))   (user_instant_interest_model.py)"""
    g = x_global.reshape(-1, 3).to(dtype)
    Wi, bi = p['instant_interest_model.out_fc.0.weight'], p['instant_interest_model.out_fc.0.bias']
    return g, torch.relu(g @ Wi.t() + bi)


def instant_backward(g: T, eu_l: T, de_l: T, grads) -> None:
    """de_l = de[:, 128:136]"""
    dpre = de_l * (eu_l > 0).to(de_l.dtype)
    grads['instant_interest_model.out_fc.0.weight'] += dpre.t() @ g
    grads['instant_interest_model.out_fc.0.bias'] += dpre.sum(0)


def head_forward(p, e: T, training: bool = True, stats: Tuple[T, T] = None):
    """e [R,264] -> (logits [R], saved).  training: BatchNorm over the batch's own (biased) statistics, computed from e; else
    `stats` = (mean, var), the running statistics when None.  (user_model.py:31-35)"""
    if training:
        mean = e.mean(0)
        var = ((e - mean) ** 2).mean(0)                               # biased, used for normalisation
    elif stats is not None:
        mean, var = stats
    else:
        mean, var = p['bn.running_mean'], p['bn.running_var']
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    xhat = (e - mean) * rstd
    z = xhat * p['bn.weight'] + p['bn.bias']
    G1, c1, G2, c2 = p['gate.fc1.weight'], p['gate.fc1.bias'], p['gate.fc2.weight'], p['gate.fc2.bias']
    M1, d1, M2, d2 = p['mlp.fc1.weight'], p['mlp.fc1.bias'], p['mlp.fc2.weight'], p['mlp.fc2.bias']
    O1, f1, O2, f2 = p['out_mlp.fc1.weight'], p['out_mlp.fc1.bias'], p['out_mlp.fc2.weight'], p['out_mlp.fc2.bias']
    a1 = z @ G1.t() + c1; u1 = gelu(a1)
    gate = u1 @ G2.t() + c2
    x = gate * e
    a2 = x @ M1.t() + d1; u2 = gelu(a2)
    y = u2 @ M2.t() + d2
    a3 = y @ O1.t() + f1; u3 = gelu(a3)
    r = (u3 @ O2.t() + f2).reshape(-1)
    saved = dict(e=e, mean=mean, var=var, rstd=rstd, xhat=xhat, z=z, a1=a1, u1=u1, gate=gate, x=x, a2=a2, u2=u2, y=y, a3=a3, u3=u3,
                 training=training)
    return r, saved


def head_backward(p, saved, dlogits: T, grads) -> T:
    """dlogits [R] -> de [R,264]; the head's weight gradients (bn, gate, mlp, out_mlp) accumulated into `grads`."""
    s = saved
    G1, G2, M1, M2, O1, O2 = (p[k] for k in ('gate.fc1.weight', 'gate.fc2.weight', 'mlp.fc1.weight', 'mlp.fc2.weight',
                                             'out_mlp.fc1.weight', 'out_mlp.fc2.weight'))
    dr = dlogits.reshape(-1, 1)
    grads['out_mlp.fc2.weight'] += dr.t() @ s['u3']
    grads['out_mlp.fc2.bias'] += dr.sum(0)
    da3 = (dr @ O2) * gelu_grad(s['a3'])
    grads['out_mlp.fc1.weight'] += da3.t() @ s['y']; grads['out_mlp.fc1.bias'] += da3.sum(0)
    dy = da3 @ O1
    grads['mlp.fc2.weight'] += dy.t() @ s['u2']; grads['mlp.fc2.bias'] += dy.sum(0)
    da2 = (dy @ M2) * gelu_grad(s['a2'])
    grads['mlp.fc1.weight'] += da2.t() @ s['x']; grads['mlp.fc1.bias'] += da2.sum(0)
    dx = da2 @ M1
    dgate = dx * s['e']
    de = dx * s['gate']
    grads['gate.fc2.weight'] += dgate.t() @ s['u1']; grads['gate.fc2.bias'] += dgate.sum(0)
    da1 = (dgate @ G2) * gelu_grad(s['a1'])
    grads['gate.fc1.weight'] += da1.t() @ s['z']; grads['gate.fc1.bias'] += da1.sum(0)
    dz = da1 @ G1
    xhat, rstd = s['xhat'], s['rstd']
    grads['bn.weight'] += (dz * xhat).sum(0); grads['bn.bias'] += dz.sum(0)
    dxhat = dz * p['bn.weight']
    if s['training']:
        return de + rstd * (dxhat - dxhat.mean(0) - xhat * (dxhat * xhat).mean(0))
    return de + rstd * dxhat


def loss_backward(p, r: T, user_id, label, grads, *, alpha=0.95, dtype=torch.float32) -> Tuple[T, T]:
    """r [B,C] -> (loss, dlogits [B,C]); the delta gradient accumulated into `grads`.  (user_model.py:37-43)"""
    B, C = r.shape
    yl = label.to(dtype)
    N = float(B * C)

    def bce_softmax(logits):
        pr = torch.softmax(logits, dim=1)
        lo = -(yl * torch.clamp(torch.log(pr), min=-100.0) + (1 - yl) * torch.clamp(torch.log(1 - pr), min=-100.0)).sum() / N
        dpr = (pr - yl) / torch.clamp((1 - pr) * pr, min=1e-12) / N
        dlog = pr * (dpr - (dpr * pr).sum(1, keepdim=True))
        return lo, dlog
    l1, dl1 = bce_softmax(r)
    l2, dl2 = bce_softmax(r + p['delta'][user_id][:, None])
    grads['delta'].index_add_(0, user_id, alpha * dl2.sum(1))
    return (1 - alpha) * l1 + alpha * l2, (1 - alpha) * dl1 + alpha * dl2


# ---------------------------------------------------------------------------
# whole training step in kernel form
# ---------------------------------------------------------------------------

def forward_backward(p, x_history, x_target, x_global, user_id, label, *, training=True, alpha=0.95,
                     dtype=torch.float32):
    """Returns (logits, loss, grads dict incl. 'delta', bn batch stats)."""
    B, H, _ = x_history.shape
    C = x_target.shape[1]
    R = B * C
    grads = grad_buffers(p)

    # ---- encoder forward
    dh_ = decode_rows(x_history.reshape(B * H, -1), dtype)
    dt_ = decode_rows(x_target.reshape(R, -1), dtype)
    xin_h = embed_rows(p, dh_)                                        # [BH,66]
    xt = embed_rows(p, dt_)                                           # [R,64]
    xh = w1_forward(p, xin_h)                                         # [BH,64]
    lab_P, lab_saved = attention_forward(p, II + 'label_attention.', xt.view(B, C, 64), xh.view(B, H, 64))
    ti_P, ti_saved = attention_forward(p, II + 'text_img_attention.', dt_['pca'].view(B, C, 64), dh_['pca'].view(B, H, 64))
    g, eu_l = instant_forward(p, x_global, dtype)
    e = torch.cat([lab_P.reshape(R, 64), ti_P.reshape(R, 64), eu_l, xt, dt_['pca']], dim=1)   # [R,264]

    # ---- head forward, loss forward + backward, head backward
    r, head_saved = head_forward(p, e, training)
    r = r.reshape(B, C)
    loss, dr = loss_backward(p, r, user_id, label, grads, alpha=alpha, dtype=dtype)
    de = head_backward(p, head_saved, dr.reshape(R), grads)

    # ---- encoder backward
    instant_backward(g, eu_l, de[:, 128:136], grads)
    dt_lab, dh_lab, _ = attention_backward(p, II + 'label_attention.', xt.view(B, C, 64), xh.view(B, H, 64), lab_saved,
                                           de[:, 0:64].reshape(B, C, 64), grads, True)
    attention_backward(p, II + 'text_img_attention.', dt_['pca'].view(B, C, 64), dh_['pca'].view(B, H, 64), ti_saved,
                       de[:, 64:128].reshape(B, C, 64), grads, False)
    dxt = dt_lab.reshape(R, 64) + de[:, 136:200]
    dxin_h = w1_backward(p, xin_h, dh_lab.reshape(B * H, 64), grads)
    embed_rows_backward(p, dh_, xin_h, dxin_h, grads)
    embed_rows_backward(p, dt_, xt, dxt, grads)
    return r, loss, grads, (head_saved['mean'], head_saved['var'])
