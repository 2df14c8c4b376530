"""Cost of ranking held-out targets against the whole pool: nrm_pool_rank (recommend.rank_targets / evaluate).

    python tools/pool_eval_bench.py [--reps 7] [--out FILE.json]

On precomputed logits (seeded random numbers, 205 MB per model: larger than the L2) at B = 1024 users, N = 50 000 pool articles
with distinct ids, exclusion on (H = 200 clicked pool articles per user), P in {16, 1024} targets per user drawn from the pool and
M in {1, 2} models:
  * nrm_pool_rank;
  * nrm_pool_topk with k = 100 on the same logits, for scale (it reads the same logits, with one pass per radix digit);
  * for M = 1, a plain torch baseline for scale: the masked scores, then each target's count of larger scores,
    (s[:, None, :] > s_target[:, :, None]).sum(-1), in chunks of users that keep its [chunk, P, N] comparison under 1 GiB.  It
    gives `greater` only (no stable rank, no ensemble), and is checked against nrm_pool_rank's `greater`.
The C entry points are called directly on preallocated buffers; CUDA events around `iters` back-to-back calls, variants of one
group alternated `--reps` times in this one process, the median per call reported with the card name and power limit read in the
same run."""
import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from news_recommendation_model_b200 import _lib, engine  # noqa: E402
from recommend_bench import HBM_BYTES_PER_S, card, stream, time_variants  # noqa: E402

N_ARTICLES = 125541                                     # EB-NeRD large


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--out', default=None, help='also write the results as JSON to this file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('pool_eval_bench.py measures on a CUDA device; none is visible')
    name, power = card()
    out = {'card': name, 'power_limit': power, 'reps': args.reps, 'runs': []}
    print(f'# {name}, power limit {power}; median of {args.reps} alternated runs')
    lib = _lib.load()
    p = engine._ptr
    B, N, H, k = 1024, 50000, 200, 100
    rng = np.random.default_rng(7)
    pool = rng.permutation(np.arange(1, N_ARTICLES))[:N].astype(np.int32)
    pa = torch.from_numpy(pool).cuda()
    ha = torch.from_numpy(rng.choice(pool, (B, H)).astype(np.int32)).cuda()
    inv = torch.full((N_ARTICLES,), -1, dtype=torch.int64, device='cuda')
    inv[pa.long()] = torch.arange(N, device='cuda')
    clicked = torch.zeros(B, N, dtype=torch.bool, device='cuda')      # the torch baseline's mask, built once, outside the timing
    clicked.scatter_(1, inv[ha.long()], True)
    g = torch.Generator(device='cuda').manual_seed(5)
    for M in (1, 2):
        logits = torch.randn(M, B, N, device='cuda', generator=g)
        pos = torch.empty(B, k, dtype=torch.int32, device='cuda')
        val = torch.empty(B, k, device='cuda')

        def topk():
            _lib.check(lib.nrm_pool_topk(p(logits), M, B * N, B, N, k, p(pa), N_ARTICLES, p(ha), H, p(pos), p(val), stream()), 'nrm_pool_topk')
        masked = logits[0].masked_fill(clicked, float('-inf')) if M == 1 else None
        for P in (16, 1024):
            tg = torch.from_numpy(rng.choice(pool, (B, P)).astype(np.int32)).cuda()
            outs = [torch.empty(B, P, dtype=torch.int32, device='cuda') for _ in range(4)]
            score = torch.empty(B, P, device='cuda')
            n_elig = torch.empty(B, dtype=torch.int32, device='cuda')

            def rank():
                _lib.check(lib.nrm_pool_rank(p(logits), M, B * N, B, N, p(pa), N_ARTICLES, p(ha), H, p(tg), P, *(p(o) for o in outs),
                                             p(score), p(n_elig), stream()), 'nrm_pool_rank')
            fns = {'nrm_pool_rank': rank, 'nrm_pool_topk_k100': topk}
            if M == 1:
                tpos = inv[tg.long()]
                chunk = max(1, (1 << 30) // (P * N))
                greater = torch.empty(B, P, dtype=torch.int64, device='cuda')

                def torch_baseline():
                    st = masked.gather(1, tpos)
                    for b0 in range(0, B, chunk):
                        greater[b0:b0 + chunk] = (masked[b0:b0 + chunk, None, :] > st[b0:b0 + chunk, :, None]).sum(-1)
                fns['torch_greater'] = torch_baseline
            t = time_variants(fns, args.reps, 5)
            torch.cuda.synchronize()
            r = dict(M=M, B=B, N=N, P=P, H=H, rank_us=t['nrm_pool_rank']['median_us'], topk_k100_us=t['nrm_pool_topk_k100']['median_us'],
                     hbm_bound_us=M * B * N * 4 / HBM_BYTES_PER_S * 1e6, rankable=int((outs[1] >= 0).sum()), timings=t)
            line = (f'M={M} B={B} N={N} P={P:4d}: nrm_pool_rank {r["rank_us"]:.0f} us, nrm_pool_topk(k=100) {r["topk_k100_us"]:.0f} us, '
                    f'HBM bound {r["hbm_bound_us"]:.0f} us')
            if M == 1:
                ok = outs[1] >= 0
                r['torch_us'] = t['torch_greater']['median_us']
                r['torch_greater_matches'] = bool(torch.equal(greater[ok], outs[2].long()[ok]))
                line += f', torch greater {r["torch_us"]:.0f} us (same counts: {r["torch_greater_matches"]})'
            out['runs'].append(r)
            print(line)
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
