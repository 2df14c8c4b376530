"""Recommendation from a shared article pool (nrm_forward_pool, nrm_pool_topk) through news_recommendation_model_b200.recommend,
in every precision: the pool logits against the eval forward on the pool replicated per user, chunk invariance, BatchNorm left
alone, and the selection against its host restatement (tests/recommend_ref.py)."""
import ctypes

import numpy as np
import pytest
import torch

import parity as P
from fixtures import load_weights
from recommend_ref import host_top_articles
from news_recommendation_model_b200 import _lib, engine, recommend, wire

pytestmark = pytest.mark.gpu

PRECISIONS = ['fp32', 'bf16', 'bf16x3']
N_ARTICLES = 3000


def _model(precision, weights='train'):
    model, _ = P.build_models(load_weights(weights), 40)
    return model.set_precision(precision)


_TABLE = {}


def _table():
    if 't' not in _TABLE:
        _TABLE['t'] = wire.make_article_table(N_ARTICLES - 1, seed=5).to('cuda')
    return _TABLE['t']


def _users(B, H, seed):
    cb = wire.make_compact_batch(_table(), B, H, 1, seed=seed, user_num=40, variable_history=True).to('cuda')
    return cb.hist_article, cb.hist_time, cb.hist_click


def _pool(N, seed):
    rng = np.random.default_rng(seed)
    pa = rng.integers(1, N_ARTICLES, N).astype(np.int32)
    pt = wire.pack_time(np.array([1, 6, 17, 9]))                          # one time for every pool article
    return torch.from_numpy(pa).cuda(), torch.full((N,), int(pt.view(np.int32)), dtype=torch.int32, device='cuda')


def _expanded_logits(model, users, pool):
    """model.eval()(...) on the compact batch whose candidates are the pool replicated to [B,N]."""
    ha, ht, hc = users
    pa, pt = pool
    B, N = ha.shape[0], pa.shape[0]
    cb = wire.CompactBatch(torch.zeros(B, dtype=torch.int64, device='cuda'), torch.zeros(B, dtype=torch.int64, device='cuda'),
                           ha, ht, hc, pa.expand(B, N).contiguous(), pt.expand(B, N).contiguous(),
                           torch.zeros(B, N, device='cuda'), torch.zeros(B, dtype=torch.int64, device='cuda'))
    b = wire.expand(_table(), cb)
    model.eval()
    with torch.no_grad():
        return model(b.x_history, b.x_target, b.x_global)


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('B', [1, 7])
@pytest.mark.parametrize('H', [1, 50, 200])
def test_pool_logits_are_those_of_the_eval_forward_on_the_replicated_pool(precision, B, H):
    model = _model(precision)
    users, pool = _users(B, H, seed=B * 1000 + H), _pool(300, seed=H)
    got = recommend.pool_logits(model, _table(), *users, pool[1], pool_article=pool[0], chunk=64)
    assert got.shape == (B, 300) and got.dtype == torch.float32
    assert torch.equal(got, _expanded_logits(model, users, pool))


@pytest.mark.parametrize('precision', PRECISIONS)
def test_pool_logits_do_not_depend_on_the_chunk(precision):
    model = _model(precision)
    users, (pa, pt) = _users(5, 60, seed=11), _pool(300, seed=12)
    ref = recommend.pool_logits(model, _table(), *users, pt, pool_article=pa)             # chunk=None
    for chunk in (8, 64, 296, 304):
        assert torch.equal(recommend.pool_logits(model, _table(), *users, pt, pool_article=pa, chunk=chunk), ref), chunk


@pytest.mark.parametrize('precision', PRECISIONS)
def test_default_pool_is_every_real_article(precision):
    model = _model(precision)
    users = _users(2, 20, seed=3)
    n = N_ARTICLES - 1
    pt = torch.zeros(n, dtype=torch.int32, device='cuda')
    full = recommend.pool_logits(model, _table(), *users, pt)
    pa = torch.arange(1, N_ARTICLES, dtype=torch.int32, device='cuda')
    assert full.shape == (2, n)
    assert torch.equal(full, recommend.pool_logits(model, _table(), *users, pt, pool_article=pa, chunk=1000))


@pytest.mark.parametrize('precision', PRECISIONS)
def test_batchnorm_statistics_are_untouched_in_training_mode(precision):
    model = _model(precision)
    model.train()
    before = {k: v.clone() for k, v in model.bn.state_dict().items()}
    users, (pa, pt) = _users(4, 30, seed=5), _pool(100, seed=6)
    recommend.top_articles(model, _table(), *users, pt, 10, pool_article=pa, chunk=32)
    torch.cuda.synchronize()
    assert model.training
    for k, v in model.bn.state_dict().items():
        assert torch.equal(v, before[k]), k


def _check_against_host(rec, logits, pa, k, hist_article):
    pos, val = host_top_articles(logits.cpu().numpy(), pa.cpu().numpy(), N_ARTICLES, k,
                                 hist_article.cpu().numpy() if hist_article is not None else None)
    assert rec.position.dtype == torch.int64 and rec.article.dtype == torch.int64 and rec.score.dtype == torch.float32
    assert torch.equal(rec.position.cpu(), torch.from_numpy(pos))
    assert torch.allclose(rec.score.cpu().double(), torch.from_numpy(val), rtol=0, atol=0, equal_nan=True)
    pa_c = pa.cpu().long()
    art = torch.where(rec.position.cpu() >= 0, pa_c[rec.position.cpu().clamp(min=0)], torch.full_like(rec.position.cpu(), -1))
    assert torch.equal(rec.article.cpu(), art)
    return pos


@pytest.mark.parametrize('precision', PRECISIONS)
def test_top_articles_leave_out_clicked_pad_and_out_of_range_ids(precision):
    model = _model(precision)
    ha, ht, hc = _users(6, 40, seed=8)
    pa, pt = _pool(200, seed=9)
    pa[3], pa[4], pa[5], pa[6] = 0, N_ARTICLES, -7, N_ARTICLES + 100
    pa[10:30] = ha[2, :20]                                                   # user 2's history (pad ids 0 included)
    pa[40:45] = ha[0, 0]                                                     # duplicates of a clicked id
    logits = recommend.pool_logits(model, _table(), ha, ht, hc, pt, pool_article=pa)
    for exclude in (True, False):
        rec = recommend.top_articles(model, _table(), ha, ht, hc, pt, 200, pool_article=pa, exclude_clicked=exclude, chunk=48)
        pos = _check_against_host(rec, logits, pa, 200, ha if exclude else None)
        assert (pos == -1).any()                                             # k = N: never all eligible
        assert not np.isin(rec.position.cpu().numpy(), [3, 4, 5, 6]).any()
        hit = np.isin(rec.article[2].cpu().numpy(), ha[2].cpu().numpy()[ha[2].cpu().numpy() != 0])
        assert hit.any() != exclude


@pytest.mark.parametrize('precision', PRECISIONS)
def test_ties_nan_and_short_pools_against_the_host_selection(precision):
    model = _model(precision)
    ha, ht, hc = _users(5, 25, seed=13)
    pa, pt = _pool(70, seed=14)
    logits = recommend.pool_logits(model, _table(), ha, ht, hc, pt, pool_article=pa)
    tied = logits.clone()
    tied[:, [5, 9, 17, 64]] = tied[:, [2]]                                   # exact ties across chunks of 8
    tied[1, 30:40] = tied[1, 0]
    tied[3, 11] = float('nan')
    tied[4, 12] = -0.0
    tied[4, 13] = 0.0
    for k in (1, 8, 33, 70):
        rec = recommend.select(tied, k, pa, N_ARTICLES, hist_article=ha)
        _check_against_host(rec, tied, pa, k, ha)
    # fewer eligible positions than k: all but 6 positions are pad ids
    short = pa.clone()
    short[6:] = 0
    rec = recommend.select(logits, 30, short, N_ARTICLES)
    _check_against_host(rec, logits, short, 30, None)
    assert (rec.position[:, 6:] == -1).all() and torch.isnan(rec.score[:, 6:]).all() and (rec.article[:, 6:] == -1).all()


@pytest.mark.parametrize('precision', PRECISIONS)
def test_one_user_one_article(precision):
    model = _model(precision)
    ha, ht, hc = _users(1, 1, seed=15)
    pa, pt = _pool(1, seed=16)
    rec = recommend.top_articles(model, _table(), ha, ht, hc, pt, 1, pool_article=pa, exclude_clicked=False)
    logits = recommend.pool_logits(model, _table(), ha, ht, hc, pt, pool_article=pa)
    assert rec.position.tolist() == [[0]] and rec.article.tolist() == [[int(pa[0])]]
    assert torch.equal(rec.score, logits)


@pytest.mark.parametrize('precision', PRECISIONS)
def test_ensemble_scores_are_the_masked_softmax_mean(precision):
    models = [_model(precision, 'train'), _model(precision, 'validation')]
    ha, ht, hc = _users(4, 50, seed=17)
    pa, pt = _pool(300, seed=18)
    pa[:30] = ha[1, :30]
    N = 300
    rec = recommend.top_articles(models, _table(), ha, ht, hc, pt, N, pool_article=pa)
    x = torch.stack([recommend.pool_logits(m, _table(), ha, ht, hc, pt, pool_article=pa) for m in models]).double().cpu()
    pa_c = pa.cpu()
    ok = torch.ones(4, N, dtype=torch.bool)
    for b in range(4):
        ok[b] = (pa_c >= 1) & (pa_c < N_ARTICLES) & ~torch.isin(pa_c, ha[b].cpu()[ha[b].cpu() != 0])
    ref = torch.zeros(4, N, dtype=torch.float64)
    for xm in x:
        ref += torch.softmax(xm.masked_fill(~ok, float('-inf')), dim=1)
    ref /= len(models)
    pos, score = rec.position.cpu(), rec.score.cpu()
    n_ok = ok.sum(1)
    for b in range(4):
        p, s = pos[b, :n_ok[b]], score[b, :n_ok[b]].double()
        assert (p >= 0).all() and (pos[b, n_ok[b]:] == -1).all()
        assert torch.equal(p.sort().values, torch.nonzero(ok[b]).view(-1))  # every eligible position exactly once
        rel = ((s - ref[b, p]).abs() / ref[b, p]).max().item()
        assert rel <= 1e-6, (b, rel)
        host = sorted(range(len(p)), key=lambda j: (s[j].item(), -p[j].item()), reverse=True)
        assert [p[j].item() for j in host] == p.tolist()                      # stable descending order of the returned scores


@pytest.mark.parametrize('precision', PRECISIONS)
def test_scale_against_the_host_selection(precision):
    model = _model(precision)
    ha, ht, hc = _users(64, 200, seed=19)
    pa, pt = _pool(20000, seed=20)
    pa[::97] = 0
    logits = recommend.pool_logits(model, _table(), ha, ht, hc, pt, pool_article=pa)
    rec = recommend.top_articles(model, _table(), ha, ht, hc, pt, 100, pool_article=pa)
    _check_against_host(rec, logits, pa, 100, ha)


@pytest.mark.parametrize('precision', PRECISIONS)
def test_bad_chunk_and_k_return_einval(precision):
    lib = _lib.load()
    model = _model(precision)
    ha, ht, hc = _users(2, 10, seed=21)
    pa, pt = _pool(2000, seed=22)
    B, H, N = 2, 10, 2000
    table = _table()
    users = engine.compact(table, wire.CompactBatch(None, None, ha, ht, hc, pa, pt, None, None))
    flat = model.flat_parameters()
    ws = torch.empty(int(lib.nrm_pool_workspace_bytes(B, H, N, 16)), dtype=torch.uint8, device='cuda')
    logits = torch.zeros(B, N, device='cuda')
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    code = model._precision_code()
    assert lib.nrm_forward_pool(*users.args, B, H, N, 12, p(flat.buf), p(model.bn.running_mean), p(model.bn.running_var), code,
                                p(logits), p(ws), ws.numel(), None) == -1
    assert lib.nrm_forward_pool(*users.args, B, H, N, 16, p(flat.buf), p(model.bn.running_mean), p(model.bn.running_var), code,
                                p(logits), p(ws), ws.numel(), None) == 0
    pos = torch.empty(B, 1025, dtype=torch.int32, device='cuda')
    val = torch.empty(B, 1025, device='cuda')
    assert lib.nrm_pool_topk(p(logits), 1, B * N, B, N, 1025, p(pa), table.n, p(ha), H, p(pos), p(val), None) == -1
    assert b'1024' in lib.nrm_last_error()
    assert lib.nrm_pool_topk(p(logits), 1, B * N, B, N, 1024, p(pa), table.n, p(ha), H, p(pos), p(val), None) == 0
    torch.cuda.synchronize()
