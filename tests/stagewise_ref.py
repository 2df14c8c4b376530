"""Float64 references of every stage of one training step (oracle/reduced_mirror.py stage functions), each fed either by the
previous reference stage (`gpu=None`: the plain chained reference) or by another implementation's own upstream buffers
(`gpu` = dict of that implementation's buffers in float64).  Fed the GPU's buffers, each stage's reference differs from the
kernel only by the kernel's own rounding, not by the noise that piles up upstream of it.

Buffer names follow the training workspace (nrm_debug_ws_field): xh [B*H,64], e [R,264], de [R,264], dxh [B*H,64],
dxt [R,64], dxin_h [B*H,66], dtp [2,R,64] (dL/dtp of the label and the text/img branch), plus logits [R]."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from oracle import reduced_mirror as M
from oracle.reference_port import II

LAB, TI = II + 'label_attention.', II + 'text_img_attention.'
HEAD_PREFIXES = ('bn.', 'gate.', 'mlp.', 'out_mlp.')


def grad_stage(key: str) -> str:
    """Which stage of the backward writes the gradient of parameter `key`."""
    if key.startswith(HEAD_PREFIXES):
        return 'head'
    if key.startswith(LAB) or key.startswith(TI):
        return 'attention'
    if key.startswith(II + 'w1.'):
        return 'w1'
    return 'embed'            # embedding tables, sentiment and instant-interest Linear layers


def stage_references(p, x_history, x_target, x_global, G, gpu: Optional[Dict[str, torch.Tensor]] = None,
                     dtype=torch.float64):
    """p: parameters (dtype, on the inputs' device); x_*: packed rows; G [B,C]: the cotangent of the logits.
    Returns (ref, grads): ref = dict of reference buffers (names as above), grads = parameter gradients by key."""
    B, H, _ = x_history.shape
    C = x_target.shape[1]
    R = B * C
    up = (lambda name, own: gpu[name]) if gpu is not None else (lambda name, own: own)
    grads = M.grad_buffers(p)
    ref = {}

    dh_ = M.decode_rows(x_history.reshape(B * H, -1), dtype)
    dt_ = M.decode_rows(x_target.reshape(R, -1), dtype)
    xin_h = M.embed_rows(p, dh_)
    xt = M.embed_rows(p, dt_)
    ref['xh'] = M.w1_forward(p, xin_h)
    g, eu_l = M.instant_forward(p, x_global, dtype)
    pca_h, pca_t = dh_['pca'].reshape(B, H, 64), dt_['pca']

    # attention forward: t = e[:, 136:200] (label) / e[:, 200:264] (text/img), h = xh (label) / pca of the history rows
    xh_in = up('xh', ref['xh']).reshape(B, H, 64)
    e_own = torch.cat([torch.zeros(R, 128, dtype=dtype, device=xt.device), eu_l, xt, pca_t], dim=1)
    t_lab = up('e', e_own)[:, 136:200].reshape(B, C, 64)
    t_ti = up('e', e_own)[:, 200:264].reshape(B, C, 64)
    lab_P, lab_saved = M.attention_forward(p, LAB, t_lab, xh_in)
    ti_P, ti_saved = M.attention_forward(p, TI, t_ti, pca_h)
    ref['e'] = torch.cat([lab_P.reshape(R, 64), ti_P.reshape(R, 64), eu_l, xt, pca_t], dim=1)

    # head: BatchNorm statistics recomputed from the e it is fed
    r, head_saved = M.head_forward(p, up('e', ref['e']), training=True)
    ref['logits'] = r
    ref['de'] = M.head_backward(p, head_saved, G.reshape(R).to(dtype), grads)

    # encoder backward
    de_in = up('de', ref['de'])
    M.instant_backward(g, eu_l, de_in[:, 128:136], grads)
    dt_lab, dh_lab, gt_lab = M.attention_backward(p, LAB, t_lab, xh_in, lab_saved, de_in[:, 0:64].reshape(B, C, 64), grads, True)
    _, _, gt_ti = M.attention_backward(p, TI, t_ti, pca_h, ti_saved, de_in[:, 64:128].reshape(B, C, 64), grads, False)
    ref['dtp'] = torch.stack([gt_lab.reshape(R, 64), gt_ti.reshape(R, 64)])
    ref['dxh'] = dh_lab.reshape(B * H, 64)
    ref['dxt'] = dt_lab.reshape(R, 64) + de_in[:, 136:200]
    ref['dxin_h'] = M.w1_backward(p, xin_h, up('dxh', ref['dxh']), grads)
    M.embed_rows_backward(p, dh_, xin_h, up('dxin_h', ref['dxin_h']), grads)
    M.embed_rows_backward(p, dt_, xt, up('dxt', ref['dxt']), grads)
    return ref, grads
