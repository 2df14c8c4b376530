"""Attention-score export (news_recommendation_model_b200.explain) on the host: the re-association floor of the scores that sets
the GPU tolerances, and the argument checks that need no device."""
import pytest
import torch

from fixtures import case_batch, load_case, load_weights
from explain_ref import SCORE_FLOOR_REL, oracle_scores
from news_recommendation_model_b200 import NrmError, explain
from oracle import reduced_mirror as M
from oracle import reference_port as O


@pytest.mark.parametrize('weights', ['train', 'validation'])
def test_score_reassociation_floor_in_float32(weights):
    """max |s_as_written - s_reduced| / max |s| in float32 on the golden inputs of case_cfg1_b64: the kernels compute the
    reduced form (oracle/reduced_mirror.py), so this is the least difference a correct fp32 kernel can show.  Measured:
    label_attention 7.31e-7 (train) / 6.25e-7 (validation), text_img_attention 3.25e-7 / 2.95e-7 (SCORE_FLOOR_REL = 7.4e-7;
    the bound below leaves a factor 2 for hosts whose float32 libraries round differently)."""
    b = case_batch(load_case('case_cfg1_b64'))
    p = O.load_params(load_weights(weights))
    with torch.no_grad():
        s_lab, s_ti, lab, pca = oracle_scores(p, b.x_history, b.x_target)
        for prefix, s_ref, (t, h) in (('label_attention.', s_lab, lab), ('text_img_attention.', s_ti, pca)):
            _, (_, _, s_red) = M.attention_forward(p, O.II + prefix, t, h)
            rel = ((s_ref - s_red).abs().max() / s_ref.abs().max()).item()
            assert 0 < rel <= 2 * SCORE_FLOOR_REL, (prefix, rel)


def test_top_history_checks_its_arguments_before_the_device():
    s = torch.zeros(2, 1, 1, 3)
    with pytest.raises(ValueError):
        explain.top_history(s, 4)                    # k > H
    with pytest.raises(ValueError):
        explain.top_history(s, 0)
    with pytest.raises(ValueError):
        explain.top_history(torch.zeros(3, 1, 1, 3), 1)
    with pytest.raises(ValueError):
        explain.top_history(torch.zeros(2, 1, 1, 70), 65)   # k > 64
    with pytest.raises(ValueError):
        explain.top_history(s, 1, x_history=torch.zeros(1, 3, 80), hist_article=torch.zeros(1, 3, dtype=torch.int32))
    with pytest.raises(NrmError):
        explain.top_history(s, 2)                    # CPU tensors: no fallback


def test_attention_scores_refuses_cpu_inputs():
    model = torch.nn.Module()                        # never reached: the inputs are checked first
    with pytest.raises(ValueError):
        explain.attention_scores(model, torch.zeros(1, 3, 79, dtype=torch.float64), torch.zeros(1, 2, 78, dtype=torch.float64),
                                 torch.zeros(1, 2, 3, dtype=torch.float64))
    with pytest.raises(NrmError):
        explain.attention_scores(model, torch.zeros(1, 3, 80, dtype=torch.float64), torch.zeros(1, 2, 78, dtype=torch.float64),
                                 torch.zeros(1, 2, 3, dtype=torch.float64))
