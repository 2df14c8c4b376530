"""Pool evaluation (news_recommendation_model_b200.recommend.rank_targets / pool_metrics / evaluate) on the host: the float64
restatement (tests/pool_eval_ref.py) against a naive per-target count and sklearn, pool_metrics' count formulas against the
restatement's metrics, and the argument checks that need no device."""
import numpy as np
import pytest
import torch
from sklearn.metrics import roc_auc_score

from pool_eval_ref import edge_case, host_pool_metrics, host_rank_targets
from recommend_ref import eligible, host_top_articles, scores
from news_recommendation_model_b200 import NrmError, recommend, wire

CASES = [dict(M=1, seed=1), dict(M=2, seed=2), dict(M=3, seed=3), dict(M=1, seed=4, N=8), dict(M=2, seed=5, B=1),
         dict(M=1, seed=6, N=200, P=40)]


def _case(c):
    return edge_case(c['M'], c['seed'], B=c.get('B', 6), N=c.get('N', 60), P=c.get('P', 12))


def _naive(logits, targets, pool, n_articles, hist):
    """Per target, one comparison with every pool position: rank = #{eligible m: s_m > s or (s_m == s and m < n)}."""
    ok = eligible(logits, pool, n_articles, hist)
    s = scores(logits, ok)
    B, P = targets.shape
    res = np.full((B, P, 3), -1, dtype=np.int64)
    for b in range(B):
        for p in range(P):
            t = targets[b, p]
            if t in targets[b, :p] or not 1 <= t < n_articles or t not in pool:
                continue
            n = int(np.flatnonzero(pool == t)[0])
            if not ok[b, n]:
                continue
            e = ok[b]
            res[b, p] = (np.sum(e & ((s[b] > s[b, n]) | ((s[b] == s[b, n]) & (np.arange(pool.size) < n)))),
                         np.sum(e & (s[b] > s[b, n])), np.sum(e & (s[b] == s[b, n])) - 1)
    return res


@pytest.mark.parametrize('case', CASES, ids=str)
@pytest.mark.parametrize('exclude', [True, False])
def test_restatement_against_a_naive_count_and_sklearn(case, exclude):
    logits, pool, hist, targets, n_articles = _case(case)
    ha = hist if exclude else None
    r = host_rank_targets(logits, targets, pool, n_articles, ha)
    naive = _naive(logits, targets, pool, n_articles, ha)
    assert np.array_equal(np.stack([r['rank'], r['greater'], r['equal']], -1), naive)
    ok = eligible(logits, pool, n_articles, ha)
    assert np.array_equal(r['n_eligible'], ok.sum(1))
    # rank < k exactly for the targets among the recommender's top k, at index rank
    N = pool.size
    for k in (1, 5, N):
        pos, _ = host_top_articles(logits, pool, n_articles, k, ha)
        for b in range(targets.shape[0]):
            assert {int(n): i for i, n in enumerate(pos[b]) if n >= 0 and n in r['position'][b]} == \
                {int(n): int(q) for n, q in zip(r['position'][b], r['rank'][b]) if 0 <= q < k}
    m = host_pool_metrics(r, ks=(1, 5))
    for b in range(targets.shape[0]):
        rankable = set(int(n) for n in r['position'][b] if n >= 0)
        elig = np.flatnonzero(ok[b])
        y = np.array([n in rankable for n in elig])
        if 0 < y.sum() < y.size:
            assert abs(m['auc'][b] - roc_auc_score(y, r['scores'][b, elig])) <= 1e-12
        else:
            assert np.isnan(m['auc'][b])
    if case['seed'] == 1:                                                   # the edge cases are present
        assert r['rank'][5].max() == -1 and np.isnan(m['rr'][5]) and np.isnan(m['recall@5'][5])
        assert (r['rank'][:, 2] == -1).all()                                  # slot 2 repeats slot 1
        assert (r['equal'] > 0).any()


def _ranks_of(r):
    t = lambda a: torch.from_numpy(np.asarray(a))
    return recommend.TargetRanks(t(r['position']), t(r['rank']), t(r['greater']), t(r['equal']), t(r['score']).float(),
                                 t(r['n_eligible']))


@pytest.mark.parametrize('case', CASES, ids=str)
def test_pool_metrics_against_their_definitions(case):
    logits, pool, hist, targets, n_articles = _case(case)
    r = host_rank_targets(logits, targets, pool, n_articles, hist)
    ks = (1, 3, 10, 1000)
    ref = host_pool_metrics(r, ks)
    got = recommend.pool_metrics(_ranks_of(r), ks)
    assert set(got) == set(ref)
    for name, v in got.items():
        assert v.shape == (targets.shape[0],)
        if name == 'n_targets':
            assert v.dtype == torch.int64 and np.array_equal(v.numpy(), ref[name])
        else:
            assert v.dtype == torch.float32
            assert np.allclose(v.double().numpy(), ref[name], rtol=0, atol=1e-6, equal_nan=True), name


def test_pool_metrics_by_hand():
    # one user, 10 eligible positions, targets ranked 0 and 3 with no ties; a second user without targets
    r = recommend.TargetRanks(torch.tensor([[4, 7, -1], [-1, -1, -1]]), torch.tensor([[0, 3, -1], [-1, -1, -1]]),
                              torch.tensor([[0, 3, -1], [-1, -1, -1]]), torch.tensor([[0, 0, -1], [-1, -1, -1]]),
                              torch.tensor([[2.0, 1.0, float('nan')], [float('nan')] * 3]), torch.tensor([10, 10]))
    m = recommend.pool_metrics(r, ks=(1, 2, 5))
    assert m['hit@1'][0] == 1 and m['recall@1'][0] == 0.5 and m['recall@5'][0] == 1
    assert abs(m['ndcg@2'][0].item() - 1 / (1 + 1 / np.log2(3))) < 1e-6
    assert abs(m['ndcg@5'][0].item() - (1 + 1 / np.log2(5)) / (1 + 1 / np.log2(3))) < 1e-6
    assert m['rr'][0] == 1 and abs(m['auc'][0].item() - (8 + 6) / 16) < 1e-7           # 8 negatives: 8 and 6 below
    assert all(torch.isnan(m[k][1]) for k in m if k != 'n_targets') and m['n_targets'].tolist() == [2, 0]


def test_rank_targets_checks_its_arguments_before_the_device():
    pa = torch.arange(1, 6, dtype=torch.int32)
    tg = torch.ones(2, 3, dtype=torch.int32)
    x = torch.zeros(2, 5)
    for bad in (torch.ones(2, 1025, dtype=torch.int32), torch.ones(2, 0, dtype=torch.int32), tg.long(), torch.ones(3, 3, dtype=torch.int32),
                torch.ones(6, dtype=torch.int32)):
        with pytest.raises(ValueError):
            recommend.rank_targets(x, bad, pa, 10)
    with pytest.raises(ValueError):
        recommend.rank_targets(x, tg, torch.tensor([1, 2, 3, 2, 5], dtype=torch.int32), 10)       # repeated pool id
    with pytest.raises(ValueError):
        recommend.rank_targets(x.double(), tg, pa, 10)
    with pytest.raises(ValueError):
        recommend.rank_targets(torch.zeros(17, 2, 5), tg, pa, 10)
    with pytest.raises(ValueError):
        recommend.rank_targets(x, tg, pa.long(), 10)
    with pytest.raises(ValueError):
        recommend.rank_targets(x, tg, pa, 10, hist_article=torch.zeros(3, 4, dtype=torch.int32))
    with pytest.raises(NrmError):
        recommend.rank_targets(x, tg, torch.tensor([0, 0, 12, 12, 5], dtype=torch.int32), 10)    # pads / out-of-range ids may repeat
    with pytest.raises(NrmError):
        recommend.rank_targets(x, tg, pa, 10)
    for ks in ((), (0,), (2.0,), (True,)):
        with pytest.raises(ValueError):
            recommend.pool_metrics(_ranks_of(host_rank_targets(x.numpy(), tg.numpy(), pa.numpy(), 10)), ks)


def test_evaluate_checks_its_arguments_before_the_device():
    table = wire.ArticleTable(torch.zeros(6, wire.ARTICLE_COLS))
    ha = torch.ones(2, 3, dtype=torch.int32)
    ht, hc = torch.zeros(2, 3, dtype=torch.int32), torch.zeros(2, 3, 2)
    pa, pt = torch.arange(1, 6, dtype=torch.int32), torch.zeros(5, dtype=torch.int32)
    tg = torch.ones(2, 4, dtype=torch.int32)
    model = torch.nn.Module()                                                # never reached
    for bad in (torch.ones(2, 1025, dtype=torch.int32), tg.long(), torch.ones(3, 4, dtype=torch.int32), torch.ones(4, 2, dtype=torch.int32).t()):
        with pytest.raises(ValueError):
            recommend.evaluate(model, table, ha, ht, hc, pt, bad, pool_article=pa)
    with pytest.raises(ValueError):
        recommend.evaluate(model, table, ha, ht, hc, pt, tg, pool_article=torch.tensor([1, 2, 3, 4, 4], dtype=torch.int32))
    with pytest.raises(ValueError):
        recommend.evaluate(model, table, ha, ht, hc, pt, tg, pool_article=pa, ks=(0,))
    with pytest.raises(ValueError):
        recommend.evaluate(model, table, ha, ht, hc, pt, tg, pool_article=pa, chunk=12)
    with pytest.raises(ValueError):
        recommend.evaluate([model] * 17, table, ha, ht, hc, pt, tg, pool_article=pa)
    with pytest.raises(NrmError):
        recommend.evaluate(model, table, ha, ht, hc, pt, tg, pool_article=pa)
