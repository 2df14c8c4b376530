"""Host restatements for the attention-score tests: the reference's scores (oracle/reference_port.pairwise_attention, the
as-written concat) and the top-k as a stable sort, plus the score tolerances (measured in test_explain_host.py)."""
import math

import torch
import torch.nn.functional as F

from oracle import reference_port as O

# max |s_as_written - s_reduced| / max |s| in float32 on the golden inputs of case_cfg1_b64 (train and validation weights,
# both branches): 7.31e-7 (label_attention, train weights; text_img_attention 3.3e-7).  The re-association floor of the
# score itself, as test_reduced_algebra.py measures the one of the logits.
SCORE_FLOOR_REL = 7.4e-7
# GPU tolerances, relative to max |s| of the batch: fp32 (FFMA) and bf16x3 (hi/lo split, 2^-16 operand error) at 200 times the
# floor; bf16 (8-bit operand mantissa, 2^-9) at 2e-2, the relative size of the bf16 logits tolerance of test_gpu_tensorcore.py.
SCORE_TOL_REL = {'fp32': 200 * SCORE_FLOOR_REL, 'bf16x3': 200 * SCORE_FLOOR_REL, 'bf16': 2e-2}


def oracle_scores(p, x_history, x_target, dtype=torch.float32):
    """(s_label, s_ti) [B,C,H] of user_invariant_interest_model.py:83-87, through the as-written pairwise attention."""
    time_h, pca_h, cat_h, sub_h, sent_h, typ_h, read_h, scroll_h = O.split_row(x_history.to(dtype), 8)
    time_t, pca_t, cat_t, sub_t, sent_t, typ_t = O.split_row(x_target.to(dtype), 6)
    lab_h = torch.cat((O.feature_embedding(p, cat_h, sub_h, sent_h, typ_h), O.time_embedding(p, time_h), read_h, scroll_h), dim=2)
    lab_h = F.linear(lab_h.reshape(-1, lab_h.shape[2]), p[O.II + 'w1.weight'], p[O.II + 'w1.bias']).reshape(lab_h.shape[0], lab_h.shape[1], -1)
    lab_t = torch.cat((O.feature_embedding(p, cat_t, sub_t, sent_t, typ_t), O.time_embedding(p, time_t)), dim=2)
    s_lab = O.pairwise_attention(p, O.II + 'label_attention.', lab_t, lab_h)[..., 0]
    s_ti = O.pairwise_attention(p, O.II + 'text_img_attention.', pca_t, pca_h)[..., 0]
    return s_lab, s_ti, (lab_t, lab_h), (pca_t, pca_h)


def host_topk(scores, real, k):
    """scores [B,C,H] (host), real [B,H] bool -> (idx [B,C,k] int64, val [B,C,k] float32): the positions of the real rows in
    Python's stable sorted(..., reverse=True) order of their scores, padded with -1 / NaN."""
    B, C, H = scores.shape
    idx = torch.full((B, C, k), -1, dtype=torch.int64)
    val = torch.full((B, C, k), math.nan, dtype=torch.float32)
    s = scores.tolist()
    for b in range(B):
        rows = [h for h in range(H) if real[b, h]]
        for c in range(C):
            order = sorted(rows, key=lambda h: s[b][c][h], reverse=True)[:k]
            for j, h in enumerate(order):
                idx[b, c, j] = h
                val[b, c, j] = scores[b, c, h]
    return idx, val
