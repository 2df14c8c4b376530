"""GPU parity (run on the B200 box with -m gpu): the CUDA path, called through the
nn.Module mirror -> C ABI, against the oracle port and the golden fixtures."""
import numpy as np
import pytest
import torch

import news_recommendation_model_b200 as nrm
from fixtures import case_batch, grad_scale, load_case, load_weights, stored
from news_recommendation_model_b200.synthetic import make_batch
from oracle import reference_port as O
import parity as P

pytestmark = pytest.mark.gpu


def _check(rep):
    assert rep['logits'] <= P.TOL_LOGITS, P.format_report(rep)
    assert rep['loss'] <= P.TOL_LOSS, P.format_report(rep)
    bad = P.grad_failures(rep)
    assert not bad, P.format_report(rep)


def test_train_step_against_golden_reference_outputs():
    """case_train_b16: logits / loss / every gradient the UNMODIFIED reference produced."""
    case = load_case('case_train_b16')
    b = case_batch(case)
    model, _ = P.build_models(load_weights('train'), int(case['meta'][3]), torch.from_numpy(case['delta0'].copy()))
    model.train()
    out, loss, grads = P.cuda_step(model, b)
    assert np.abs(out.numpy() - case['logits']).max() <= P.TOL_LOGITS
    assert abs(float(loss) - float(case['loss'])) <= P.TOL_LOSS
    for k, g in grads.items():
        ref = case['grad/' + k]
        scale = grad_scale(case, k)
        tol = P.TOL_GRAD_ABS if k in P.NOISE_KEYS else P.TOL_GRAD_REL * scale + P.TOL_GRAD_ABS
        err = np.abs(stored(case, k, g.numpy()) - ref).max()
        assert err <= tol, (k, err, scale)
        if 'gradnorm/' + k in case.files:     # a sampled tensor: its whole gradient through the norm
            n_err = abs(g.double().norm().item() - float(case['gradnorm/' + k]))
            assert n_err <= tol * np.sqrt(g.numel()), (k, n_err, scale)
    # BatchNorm buffers after the training forward
    sd = model.state_dict()
    for k in ('bn.running_mean', 'bn.running_var'):
        ref = case['after/' + k]
        assert np.abs(sd[k].cpu().numpy() - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), k
    assert int(sd['bn.num_batches_tracked']) == int(case['after/bn.num_batches_tracked'])


def test_adam_step_against_golden_reference_outputs():
    case = load_case('case_train_b16')
    b = case_batch(case)
    model, _ = P.build_models(load_weights('train'), int(case['meta'][3]), torch.from_numpy(case['delta0'].copy()))
    model.train()
    opt = nrm.FusedAdam(model.parameters(), lr=1e-3, weight_decay=1e-5)      # train.py:48
    d = b.to('cuda')
    out = model(d.x_history, d.x_target, d.x_global)
    model.loss(d.user_id, out, d.label).backward()
    opt.step()
    opt.zero_grad()
    for k, v in model.named_parameters():
        if k in P.NOISE_KEYS:      # gradient is rounding noise; Adam turns its sign into +-lr
            continue
        ref = case['after/' + k]
        before = stored(case, k, case['delta0'] if k == 'delta' else load_weights('train')[k].numpy())
        moved = np.abs(ref - before).max()
        err = np.abs(stored(case, k, v.detach().cpu().numpy()) - ref).max()
        # first Adam step moves every touched weight by ~lr (g / (|g| + eps)): elements whose gradient is ~eps are
        # sensitive to 1e-9 differences in g, so allow 5% of that movement
        assert err <= 0.05 * max(moved, 1e-3) + 1e-7, (k, err, moved)


@pytest.mark.parametrize('B,H,C,kw', [
    (64, 50, 5, {}),                                 # BASELINE config 1
    (7, 13, 4, dict(variable_history=True)),         # ragged sizes, padded history
    (3, 130, 3, dict(variable_history=True)),        # history spans several 64-row tiles
    (5, 64, 19, dict(variable_candidates=True)),     # more candidates than one 8-wide chunk, pad candidates
    (1, 1, 1, {}),                                   # degenerate
])
def test_train_step_matches_oracle(B, H, C, kw):
    b = make_batch(B, H, C, seed=B * 1000 + H, user_num=40, **kw)
    delta0 = torch.from_numpy(np.random.default_rng(3).normal(0, 0.3, 41).astype(np.float32))
    model, p = P.build_models(load_weights('train'), 40, delta0)
    if B * C == 1:
        return   # BatchNorm1d refuses a single row in training mode (reference raises too)
    _check(P.compare_step(model, p, b, training=True))


def test_non_fp32_representable_inputs_round_like_the_reference():
    b = make_batch(9, 21, 5, seed=77, user_num=40, fp32_exact=False)
    model, p = P.build_models(load_weights('validation'), 40)
    _check(P.compare_step(model, p, b, training=True))


def test_duplicate_users_share_one_delta_row():
    b = make_batch(32, 10, 5, seed=5, user_num=3)            # 32 impressions over 4 users
    delta0 = torch.tensor([0.5, -0.25, 0.1, 0.0])
    model, p = P.build_models(load_weights('train'), 3, delta0)
    _check(P.compare_step(model, p, b, training=True))


def test_eval_scoring_against_golden_reference_outputs():
    """case_eval_b8: test.py:31-74 scores, ranks and AUC of the 2-model ensemble on ragged candidate lists."""
    case = load_case('case_eval_b8')
    b = case_batch(case)
    models = []
    for name in ('train', 'validation'):
        m = nrm.UserModel()
        m.load_state_dict(load_weights(name), strict=False)
        models.append(m.to('cuda').eval())
    d = b.to('cuda')
    with torch.no_grad():
        for n, m in enumerate(models):
            logits = m(d.x_history, d.x_target, d.x_global).cpu().numpy()
            assert np.abs(logits - case[f'eval_logits/{n}']).max() <= 5e-4      # dead BN channels amplify 316x
        B = int(case['meta'][0])
        i = 0
        for s in range(0, B, 4):                     # the reference scored with batch_size=4
            xh, xt, xg, en = d.x_history[s:s + 4], d.x_target[s:s + 4], d.x_global[s:s + 4], b.empty_num[s:s + 4]
            trim = int(en.min())
            if trim > 0:                             # test.py:52-56: non-contiguous column slices
                xt, xg, en = xt[:, 0:-trim], xg[:, 0:-trim], en - trim
            out = sum(torch.softmax(m(xh, xt, xg), dim=1) for m in models) / len(models)
            for r in range(out.shape[0]):
                z = int(en[r])
                score = (torch.softmax(out[r:r + 1, 0:-z], dim=1).squeeze(0) if z > 0 else out[r]).cpu().numpy()
                ref = case[f'score/{i}']
                assert score.shape == ref.shape
                assert np.abs(score - ref).max() <= 1e-5
                assert O.rank_string(score) == str(case['ranks'][i])
                assert abs(O.auc(b.label[i].numpy()[:len(ref)], score) - case['auc'][i]) <= 1e-4
                i += 1


def test_eval_mode_forward_leaves_bn_buffers_alone_and_train_mode_updates_them():
    b = make_batch(16, 20, 5, seed=11).to('cuda')
    m = nrm.UserModel().to('cuda')
    m.load_state_dict(load_weights('train'), strict=False)
    before = {k: v.clone() for k, v in m.state_dict().items() if k.startswith('bn.running') or k.endswith('tracked')}
    m.eval()
    with torch.no_grad():
        m(b.x_history, b.x_target, b.x_global)
    for k, v in before.items():
        assert torch.equal(m.state_dict()[k], v)
    m.train()
    with torch.no_grad():
        m(b.x_history, b.x_target, b.x_global)
    assert int(m.bn.num_batches_tracked) == int(before['bn.num_batches_tracked']) + 1
    assert not torch.equal(m.bn.running_mean, before['bn.running_mean'])


def test_backward_is_run_to_run_deterministic():
    b = make_batch(48, 50, 5, seed=21, user_num=10)
    model, _ = P.build_models(load_weights('train'), 10)
    model.train()
    _, _, g1 = P.cuda_step(model, b)
    _, _, g2 = P.cuda_step(model, b)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


def test_fused_adam_matches_torch_adam_over_several_steps():
    torch.manual_seed(0)
    n = 10007
    p0 = torch.randn(n, device='cuda')
    pa, pb = torch.nn.Parameter(p0.clone()), torch.nn.Parameter(p0.clone())
    oa = nrm.FusedAdam([pa], lr=1e-3, weight_decay=1e-5)
    ob = torch.optim.Adam([pb], lr=1e-3, weight_decay=1e-5)
    for step in range(5):
        g = torch.randn(n, device='cuda') * (10.0 ** (step - 2))
        pa.grad, pb.grad = g.clone(), g.clone()
        oa.step(); ob.step()
        assert (pa - pb).abs().max().item() <= 2e-6, step


def test_full_size_properties_config2():
    """B=1024,H=50,C=5 (BASELINE config 2): size-independent properties -- the batch is the
    small batch tiled, so per-impression encoder outputs repeat and gradients scale exactly."""
    small = make_batch(64, 50, 5, seed=9, user_num=100)
    reps = 16
    big = type(small)(*[torch.cat([getattr(small, f)] * reps) for f in small.__dataclass_fields__])
    model, _ = P.build_models(load_weights('train'), 100)
    model.train()
    out_s, loss_s, g_s = P.cuda_step(model, small)
    out_b, loss_b, g_b = P.cuda_step(model, big)
    # BatchNorm statistics of a tiled batch equal those of the base batch -> identical logits / loss
    assert (out_b[:64] - out_s).abs().max() <= 2e-5
    assert (out_b.view(reps, 64, 5) - out_b[:64]).abs().max() <= 1e-6
    assert abs(float(loss_b) - float(loss_s)) <= 1e-6
    for k in g_s:
        if k in P.NOISE_KEYS:
            continue
        scale = float(g_s[k].abs().max())
        assert float((g_b[k] - g_s[k]).abs().max()) <= 2e-4 * scale + 1e-7, k


@pytest.mark.parametrize('use_graph', [False, True])
def test_fused_train_step_equals_module_path(use_graph):
    """FusedTrainStep (pipelined C-ABI calls, optionally CUDA-graph replayed) must leave exactly the
    weights that the train.py-style loop (autograd + FusedAdam) leaves."""
    B, H, C, U = 32, 50, 5, 30
    batches = [make_batch(B, H, C, seed=300 + i, user_num=U) for i in range(4)]
    w = load_weights('train')
    ma, _ = P.build_models(w, U)
    mb, _ = P.build_models(w, U)
    ma.train(); mb.train()
    opt = nrm.FusedAdam(ma.parameters(), lr=1e-3, weight_decay=1e-5)
    losses_a = []
    for b in batches:
        d = b.to('cuda')
        out = ma(d.x_history, d.x_target, d.x_global)
        loss = ma.loss(d.user_id, out, d.label)
        loss.backward(); opt.step(); opt.zero_grad()
        losses_a.append(loss.item())
    tr = nrm.FusedTrainStep(mb, B, H, C, lr=1e-3, weight_decay=1e-5, use_graph=use_graph)
    losses_b = [tr.step(b.pin()).item() for b in batches]
    torch.cuda.synchronize()
    assert np.allclose(losses_a, losses_b, rtol=0, atol=1e-6), (losses_a, losses_b)
    for (k, pa), (_, pb) in zip(ma.named_parameters(), mb.named_parameters()):
        assert torch.equal(pa, pb), k
    for k in ('running_mean', 'running_var', 'num_batches_tracked'):
        assert torch.equal(getattr(ma.bn, k), getattr(mb.bn, k)), k


def test_helper_methods_of_the_invariant_interest_model_match_the_oracle():
    """slice_x / feature_embedding / time_embedding (user_invariant_interest_model.py:50-71) keep the reference's signatures;
    the embeddings run through the fused row kernel."""
    b = make_batch(5, 9, 4, seed=17, user_num=10)
    model, p = P.build_models(load_weights('train'), 10)
    inv = model.invariant_interest_model
    xt = b.x_target.to('cuda')
    parts = inv.slice_x(xt.to(torch.float32), 6)
    ref_parts = O.split_row(b.x_target.to(torch.float32), 6)
    assert [tuple(a.shape) for a in parts] == [tuple(r.shape) for r in ref_parts]
    for a, r in zip(parts, ref_parts):
        assert torch.equal(a.cpu(), r)
    t, _, cat, sub, sent, typ = parts
    rt, _, rcat, rsub, rsent, rtyp = ref_parts
    with torch.no_grad():
        fe = inv.feature_embedding(cat, sub, sent, typ).cpu()
        te = inv.time_embedding(t).cpu()
    assert fe.shape == (5, 4, 56) and te.shape == (5, 4, 8)
    assert (fe - O.feature_embedding(p, rcat, rsub, rsent, rtyp)).abs().max().item() <= 1e-6
    assert (te - O.time_embedding(p, rt)).abs().max().item() <= 1e-6


def test_out_of_range_user_id_gives_a_nan_loss_instead_of_reading_out_of_bounds():
    """The reference raises IndexError for delta[id] with id > user_num (user_model.py:38); the kernel cannot raise, so the loss
    of that step is NaN and nothing is read outside delta."""
    b = make_batch(8, 5, 3, seed=3, user_num=10)
    model, _ = P.build_models(load_weights('train'), 10)
    model.train()
    d = b.to('cuda')
    out = model(d.x_history, d.x_target, d.x_global)
    good = model.loss(d.user_id, out, d.label)
    uid = d.user_id.clone()
    uid[3] = 11
    bad = model.loss(uid, out, d.label)
    uid[3] = -1
    bad2 = model.loss(uid, out, d.label)
    assert torch.isfinite(good) and torch.isnan(bad) and torch.isnan(bad2)
