"""The stage references of tests/stagewise_ref.py, chained on themselves in float64, against autograd of the as-written port
(oracle/reference_port.py), for a random cotangent of the logits: logits, e, every parameter gradient, and the intermediate
gradients the GPU test compares, taken from the port's own intermediates with retain_grad:
de = dL/de, dxh = dL/d(w1 output), dxt = dL/d(target embedding), dxin_h[:, 0:64] = dL/d(history embedding columns), and
dtp = dL/d(attention fc1 pre-activation) summed over the history rows.  tests/test_gpu_stagewise.py feeds the same stages the
GPU's own buffers."""
import pytest
import torch

from fixtures import load_weights
from news_recommendation_model_b200.synthetic import make_batch
from oracle import reference_port as O
from stagewise_ref import grad_stage, stage_references


def _capture(monkeypatch):
    """Wrap the port's building blocks so that the tensors whose gradients the stage references produce keep them."""
    cap = {'emb': [], 'time': [], 'att': {}, 'pre': {}}
    fe, te, pa, mlp, ec = O.feature_embedding, O.time_embedding, O.pairwise_attention, O.mlp, O.e_concat

    def keep(t):
        t.retain_grad()
        return t

    monkeypatch.setattr(O, 'feature_embedding', lambda *a: cap['emb'].append(keep(fe(*a))) or cap['emb'][-1])
    monkeypatch.setattr(O, 'time_embedding', lambda *a: cap['time'].append(keep(te(*a))) or cap['time'][-1])

    def pairwise(p, prefix, target, history):
        if prefix.startswith(O.II + 'label_attention'):
            cap['att'] = dict(t=keep(target), h=keep(history))
        return pa(p, prefix, target, history)

    def mlp_pre(p, prefix, x):
        if 'attention' not in prefix:
            return mlp(p, prefix, x)
        pre = keep(torch.nn.functional.linear(x, p[prefix + 'fc1.weight'], p[prefix + 'fc1.bias']))
        cap['pre'][prefix] = pre
        return torch.nn.functional.linear(torch.nn.functional.gelu(pre), p[prefix + 'fc2.weight'], p[prefix + 'fc2.bias'])

    monkeypatch.setattr(O, 'pairwise_attention', pairwise)
    monkeypatch.setattr(O, 'mlp', mlp_pre)
    monkeypatch.setattr(O, 'e_concat', lambda *a, **k: cap.setdefault('e', keep(ec(*a, **k))))
    return cap


@pytest.mark.parametrize('B,H,C,kw', [(5, 13, 9, dict(variable_history=True, variable_candidates=True)), (2, 1, 1, {})])
def test_chained_stages_equal_autograd_in_float64(B, H, C, kw, monkeypatch):
    b = make_batch(B, H, C, seed=11 + B, user_num=20, **kw)
    p = O.load_params(load_weights('train'), dtype=torch.float64, user_num=20)
    G = torch.randn(B, C, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    leaves = {k: p[k].clone().requires_grad_(True) for k in O.TRAINABLE_KEYS}
    pa = dict(p, **leaves)
    cap = _capture(monkeypatch)
    out = O.user_model_forward(pa, b.x_history, b.x_target, b.x_global, training=True, dtype=torch.float64,
                               update_running_stats=False)
    out.backward(G)
    monkeypatch.undo()
    ref, grads = stage_references(p, b.x_history, b.x_target, b.x_global, G)

    def same(name, got, want):
        assert got.shape == want.shape, name
        assert (got - want).abs().max() <= 1e-10 * max(1.0, want.abs().max().item()), name

    R = B * C
    same('logits', ref['logits'], out.detach().reshape(-1))
    same('e', ref['e'], cap['e'].detach().reshape(R, -1))
    same('de', ref['de'], cap['e'].grad.reshape(R, -1))
    same('dxh', ref['dxh'], cap['att']['h'].grad.reshape(B * H, 64))
    same('dxt', ref['dxt'], cap['att']['t'].grad.reshape(R, 64))
    emb_h, time_h = cap['emb'][0], cap['time'][0]              # the history rows are embedded first (invariant_interest)
    same('dxin_h', ref['dxin_h'][:, 0:64], torch.cat([emb_h.grad, time_h.grad], dim=2).reshape(B * H, 64))
    for i, prefix in enumerate((O.II + 'label_attention.mlp.', O.II + 'text_img_attention.mlp.')):
        same('dtp', ref['dtp'][i], cap['pre'][prefix].grad.reshape(B, C, H, 64).sum(2).reshape(R, 64))
    for k, leaf in leaves.items():
        assert grad_stage(k) in ('head', 'attention', 'w1', 'embed')
        same(k, grads[k], leaf.grad)
