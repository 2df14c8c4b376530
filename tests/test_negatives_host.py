"""Pool negatives without a GPU: the reference's Philox against Random123's known answers, the reference's rules on hand-built
impressions, and the argument checks of NegativeSampler and nrm_sample_negatives."""
import ctypes

import pytest
import torch

import negatives_ref as R
from news_recommendation_model_b200 import _lib, negatives, wire


@pytest.mark.parametrize('ctr, key, out', [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_reproduces_the_random123_known_answers(ctr, key, out):
    assert R.philox4x32_10(ctr, key) == out


def _one(hist, cand, label, pool, weights=None, n=100, k=4, seed=3, step=0, times=None):
    times = times if times is not None else [10 + c for c in range(len(cand))]
    ids, t, lab = R.sample([hist], [cand], [times], [label], pool, weights, n, k, seed, step)
    return ids[0], t[0], lab[0]


def test_exhausted_pool_leaves_pads():
    # the only pool ids not in the history or the candidates are 5 and 6
    ids, t, lab = _one([1, 2, 0], [3, 4], [0.0, 1.0], [1, 2, 3, 4, 5, 6], k=4)
    assert sorted(ids[:2]) == [5, 6] and ids[2:] == [0, 0]
    assert t == [11, 11, 0, 0] and lab == [0.0] * 4
    # every pool id excluded: all pads
    assert _one([1, 2], [3], [1.0], [1, 2, 3], k=3)[0] == [0, 0, 0]


def test_impression_without_a_positive_gets_pads():
    assert _one([1], [2, 3], [0.0, 0.0], list(range(1, 50)), k=5) == ([0] * 5, [0] * 5, [0.0] * 5)


def test_negatives_take_the_time_of_the_first_positive():
    ids, t, _ = _one([], [7, 8, 9], [0.0, 1.0, 1.0], list(range(1, 90)), k=6, times=[100, 200, 300])
    assert all(i > 0 for i in ids) and t == [200] * 6


def test_zero_weights_and_out_of_range_ids_are_never_drawn():
    pool = [0, -3, 100, 5, 6, 7, 250]
    for seed in range(20):
        ids, _, _ = _one([], [1], [1.0], pool, weights=[9, 9, 9, 1, 0, 1, 9], n=100, k=2, seed=seed)
        assert sorted(ids) == [5, 7]
    assert R.pool_cdf(pool, [9, 9, 9, 1, 0, 1, 9], 100) == [0, 0, 0, 1, 1, 2, 2]


def test_repeated_pool_ids_are_accepted_once():
    for seed in range(20):
        ids, _, _ = _one([], [1], [1.0], [7, 7, 7, 7, 9], k=3, seed=seed)
        assert sorted(ids) == [0, 7, 9]


def test_attempts_are_resolved_in_order_with_the_philox_draws():
    pool = list(range(1, 41))
    cdf = R.pool_cdf(pool, None, 100)
    seed, step, row = 11, 5, 2
    expect, seen = [], {3}
    for a in range(64):
        i = pool[R.draw(cdf, seed, step, row, a)]
        if i not in seen and len(expect) < 2:
            expect.append(i)
            seen.add(i)
    hist = [[0], [0], [0]]
    ids, _, _ = R.sample(hist, [[3]] * 3, [[1]] * 3, [[1.0]] * 3, pool, None, 100, 2, seed, step)
    assert ids[row] == expect
    # draws depend on the step and the row
    assert R.sample(hist, [[3]] * 3, [[1]] * 3, [[1.0]] * 3, pool, None, 100, 2, seed, step + 1)[0] != ids
    assert R.sample(hist, [[3]] * 3, [[1]] * 3, [[1.0]] * 3, pool, None, 100, 2, seed, step, row_offset=1)[0][:2] == ids[1:]


def test_draw_follows_the_weights():
    cdf = [1, 1, 4]                       # weights 1, 0, 3
    counts = [0, 0, 0]
    for a in range(4000):
        counts[R.draw(cdf, 1, 0, 0, a)] += 1
    assert counts[1] == 0 and 800 < counts[0] < 1200


def test_sampler_builds_the_reference_cdf_and_checks_its_arguments():
    table = wire.ArticleTable(torch.zeros(10, wire.ARTICLE_COLS))
    s = negatives.NegativeSampler(table, k=3, seed=2 ** 64 - 1)
    assert s.N == 9 and s.total == 9 and s.cdf.tolist() == list(range(1, 10))
    pool = torch.tensor([0, 3, 12, 3, 9], dtype=torch.int32)
    w = torch.tensor([5, 2, 7, 0, 1])
    s = negatives.NegativeSampler(table, k=1, pool_article=pool, weights=w)
    assert s.cdf.tolist() == R.pool_cdf(pool.tolist(), w.tolist(), 10) == [0, 2, 2, 2, 3]
    for kw, msg in (({'k': 0}, 'k must'), ({'k': 65}, 'k must'), ({'seed': -1}, 'seed'), ({'seed': 1 << 64}, 'seed'),
                    ({'pool_article': pool.long()}, 'int32'), ({'weights': w.float(), 'pool_article': pool}, 'integer'),
                    ({'weights': w[:3], 'pool_article': pool}, r'\[N\]'), ({'weights': -w, 'pool_article': pool}, 'non-negative'),
                    ({'weights': torch.zeros(5, dtype=torch.int64), 'pool_article': pool}, 'total weight'),
                    ({'pool_article': torch.tensor([0, 10, 11], dtype=torch.int32)}, 'total weight'),
                    ({'weights': torch.full((5,), 1 << 61), 'pool_article': torch.tensor([1, 2, 3, 4, 5], dtype=torch.int32)}, '2\\^62')):
        with pytest.raises(ValueError, match=msg):
            negatives.NegativeSampler(table, **kw)
    negatives.NegativeSampler(table, weights=torch.tensor([1 << 59] * 8 + [0]))             # exactly 2^62
    cb = wire.make_compact_batch(table, 2, 3, 2, seed=1)
    with pytest.raises(_lib.NrmError, match='CUDA'):
        negatives.NegativeSampler(table, k=2).sample(cb)


def test_c_abi_refuses_bad_arguments_without_a_gpu():
    lib = _lib.load()
    p = ctypes.c_void_p(256)

    def call(hist=p, H=3, B=2, C=6, C0=2, N=10, n=10, row_offset=0, step=p):
        return lib.nrm_sample_negatives(hist, H, p, p, p, B, C, C0, p, p, N, n, 0, step, row_offset, None)
    for kw in ({'hist': None}, {'step': None}, {'B': 0}, {'H': 0}, {'C0': 0}, {'N': 0}, {'n': 0}, {'C': 2}, {'C': 2 + 65},
               {'H': 16384 - 5}, {'row_offset': -1}, {'row_offset': 2 ** 31 - 2}):
        assert call(**kw) == -1, kw
        assert b'nrm_sample_negatives' in lib.nrm_last_error()
