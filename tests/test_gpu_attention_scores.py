"""Attention scores exported by the fused forward (nrm_forward_scores[_compact]) and the top-k "why this article" kernel
(nrm_history_topk), through news_recommendation_model_b200.explain, in every precision."""
import ctypes

import pytest
import torch

import parity as P
from explain_ref import SCORE_TOL_REL, host_topk, oracle_scores
from fixtures import case_batch, load_case, load_weights
from news_recommendation_model_b200 import _lib, explain, wire
from news_recommendation_model_b200.synthetic import make_batch

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp32', 'bf16', 'bf16x3']


def _model(precision, weights='train', user_num=1000):
    model, p = P.build_models(load_weights(weights), user_num)
    return model.set_precision(precision), p


def _check_against_oracle(model, p, b, precision):
    d = b.to('cuda')
    s = explain.attention_scores(model, d.x_history, d.x_target, d.x_global)
    with torch.no_grad():
        s_lab, s_ti, _, _ = oracle_scores(p, b.x_history, b.x_target)
    for name, got, ref in (('label', s.label, s_lab), ('text_img', s.text_img, s_ti)):
        assert got.shape == ref.shape
        err = (got.cpu() - ref).abs().max().item()
        scale = ref.abs().max().item()
        assert err <= SCORE_TOL_REL[precision] * scale, (precision, name, err, scale, err / scale)
    return s


@pytest.mark.parametrize('precision', PRECISIONS)
def test_scores_match_the_oracle_on_the_golden_inputs(precision):
    case = load_case('case_cfg1_b64')
    model, p = _model(precision, user_num=int(case['meta'][3]))
    _check_against_oracle(model, p, case_batch(case), precision)


@pytest.mark.parametrize('precision', PRECISIONS)
def test_scores_match_the_oracle_with_variable_history(precision):
    model, p = _model(precision, 'validation', user_num=40)
    _check_against_oracle(model, p, make_batch(6, 200, 11, seed=17, user_num=40, variable_history=True), precision)


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('B,H,C,trim', [(9, 50, 5, 0), (1, 1, 1, 0), (3, 20, 104, 4), (2, 256, 3, 0)])
def test_logits_are_those_of_the_eval_forward(precision, B, H, C, trim):
    """Bit-identical to model.eval()(...) in the same precision; trim > 0: column-trimmed x_target / x_global views (test.py:53-54)."""
    model, _ = _model(precision, user_num=40)
    d = make_batch(B, H, C, seed=B + H + C, user_num=40, variable_history=True).to('cuda')
    xt, xg = d.x_target[:, :C - trim], d.x_global[:, :C - trim]
    s = explain.attention_scores(model, d.x_history, xt, xg)
    model.eval()
    with torch.no_grad():
        ref = model(d.x_history, xt, xg)
    assert s.logits.shape == (B, C - trim) and s.label.shape == (B, C - trim, H) and s.text_img.shape == (B, C - trim, H)
    assert torch.equal(s.logits, ref)
    assert torch.isfinite(s.label).all() and torch.isfinite(s.text_img).all()


@pytest.mark.parametrize('precision', PRECISIONS)
def test_batchnorm_statistics_are_untouched_in_training_mode(precision):
    model, _ = _model(precision, user_num=40)
    model.train()
    before = {k: v.clone() for k, v in model.bn.state_dict().items()}
    d = make_batch(8, 30, 6, seed=3, user_num=40).to('cuda')
    s = explain.attention_scores(model, d.x_history, d.x_target, d.x_global)
    torch.cuda.synchronize()
    assert model.training
    for k, v in model.bn.state_dict().items():
        assert torch.equal(v, before[k]), k
    model.eval()
    with torch.no_grad():
        assert torch.equal(s.logits, model(d.x_history, d.x_target, d.x_global))


@pytest.mark.parametrize('precision', PRECISIONS)
def test_compact_input_gives_the_same_bits_as_the_expanded_one(precision):
    model, _ = _model(precision, user_num=40)
    table = wire.make_article_table(3000, seed=5).to('cuda')
    cb = wire.make_compact_batch(table, 7, 70, 12, seed=9, user_num=40, variable_history=True, variable_candidates=True).to('cuda')
    sc = explain.attention_scores_compact(model, table, cb)
    b = wire.expand(table, cb)
    se = explain.attention_scores(model, b.x_history, b.x_target, b.x_global)
    for name in ('logits', 'label', 'text_img'):
        assert torch.equal(getattr(sc, name), getattr(se, name)), name


def _with_ties(b):
    """History rows 3 and 7 of every impression copy row 0: equal scores, exactly, in both branches."""
    xh = b.x_history.clone()
    xh[:, 3] = xh[:, 0]
    xh[:, 7] = xh[:, 0]
    return b.__class__(b.impression_id, b.user_id, xh, b.x_target, b.x_global, b.label, b.label_id, b.empty_num)


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('k', [1, 5, 40])
def test_top_history_is_a_stable_descending_sort_without_pad_rows(precision, k):
    model, _ = _model(precision, user_num=40)
    b = _with_ties(make_batch(6, 40, 7, seed=23, user_num=40, variable_history=True))
    d = b.to('cuda')
    s = explain.attention_scores(model, d.x_history, d.x_target, d.x_global)
    top = explain.top_history(s, k, x_history=d.x_history)
    real = b.x_history.abs().sum(2) > 0
    assert (~real).any()
    if k == 40:
        assert (real.sum(1) < k).any()                  # some rows end in -1 / NaN slots
    for scores, idx, val in ((s.label, top.label_idx, top.label_score), (s.text_img, top.text_img_idx, top.text_img_score)):
        sc = scores.cpu()
        assert torch.equal(sc[:, :, 3], sc[:, :, 0]) and torch.equal(sc[:, :, 7], sc[:, :, 0])   # the ties are there
        ref_idx, ref_val = host_topk(sc, real, k)
        assert idx.dtype == torch.int64 and idx.shape == (6, 7, k) and val.shape == (6, 7, k)
        assert torch.equal(idx.cpu(), ref_idx)
        assert torch.allclose(val.cpu(), ref_val, rtol=0, atol=0, equal_nan=True)
        i = idx.cpu()
        assert not ((i >= 0) & ~real.gather(1, i.clamp(min=0).view(6, -1)).view(6, 7, k)).any()   # never a pad row
        assert torch.isnan(val.cpu()[i < 0]).all()


@pytest.mark.parametrize('precision', ['bf16', 'bf16x3'])
def test_top_history_reads_pad_rows_from_the_compact_batch(precision):
    model, _ = _model(precision, user_num=40)
    table = wire.make_article_table(3000, seed=5).to('cuda')
    cb = wire.make_compact_batch(table, 5, 64, 6, seed=4, user_num=40, variable_history=True).to('cuda')
    s = explain.attention_scores_compact(model, table, cb)
    k = 64
    top = explain.top_history(s, k, hist_article=cb.hist_article)
    real = (cb.hist_article != 0).cpu()
    b = wire.expand(table, cb)
    top_x = explain.top_history(s, k, x_history=b.x_history)
    for idx, val, idx_x, val_x, sc in ((top.label_idx, top.label_score, top_x.label_idx, top_x.label_score, s.label),
                                       (top.text_img_idx, top.text_img_score, top_x.text_img_idx, top_x.text_img_score, s.text_img)):
        ref_idx, ref_val = host_topk(sc.cpu(), real, k)
        assert torch.equal(idx.cpu(), ref_idx) and torch.equal(idx, idx_x)
        assert torch.allclose(val.cpu(), ref_val, rtol=0, atol=0, equal_nan=True)
        assert torch.allclose(val, val_x, rtol=0, atol=0, equal_nan=True)
    # without a pad-row source every row takes part
    top_all = explain.top_history(s, k)
    assert (top_all.label_idx >= 0).all()


def test_train_mode_call_into_the_c_entry_point_is_rejected():
    lib = _lib.load()
    model, _ = _model('bf16x3', user_num=40)
    d = make_batch(2, 10, 3, seed=1, user_num=40).to('cuda')
    B, H, C = 2, 10, 3
    flat = model.flat_parameters()
    ws = torch.empty(int(lib.nrm_workspace_bytes(B, H, C, 3)), dtype=torch.uint8, device='cuda')
    logits = torch.empty(B, C, device='cuda')
    scores = torch.empty(2, B, C, H, device='cuda')
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    for mode in (1, 2, 3):
        rc = lib.nrm_forward_scores(p(d.x_history), p(d.x_target), C * 78, p(d.x_global), C * 3, B, H, C, p(flat.buf),
                                    p(model.bn.running_mean), p(model.bn.running_var), p(model.bn.num_batches_tracked), mode, 2,
                                    p(logits), p(scores), p(ws), ws.numel(), None)
        assert rc == -1, (mode, rc)                 # NRM_EINVAL


def test_k_larger_than_h_raises_value_error():
    s = torch.zeros(2, 1, 1, 3, device='cuda')
    with pytest.raises(ValueError):
        explain.top_history(s, 4)
