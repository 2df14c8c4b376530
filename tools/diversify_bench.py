"""Cost and effect of re-ranking pool recommendations for diversity: nrm_pool_diversify (recommend.diversify / diverse_articles).

    python tools/diversify_bench.py [--reps 7] [--out FILE.json]

On precomputed logits (seeded random numbers, 205 MB: larger than the L2) at B = 1024 users, N = 50 000 pool articles with distinct
ids, exclusion on (H = 200 clicked pool articles per user), the synthetic EB-NeRD-large article table (about 3 000 categories), as
tools/pool_eval_bench.py:
  * nrm_pool_topk(K') for K' in {128, 512}, which produces the candidates, and nrm_pool_diversify on them for k in {10, 100},
    lam in {1, 0.7}, without a cap and with max_per_category = 2;
  * a plain torch MMR loop on the same candidates (per step: gains, masked argmax, gather of the pick's vector, batched dot, max;
    one Python iteration per pick), timed the same way, with the fraction of users whose list equals the kernel's;
  * on a real-model pool (validation weights, bf16x3, B = 256, H = 200, N = 20 000 pool articles of that table), the mean
    list_diversity (intra-list diversity and distinct categories) at k = 10 of `select` against `diversify` on the pool logits,
    i.e. of what top_articles and diverse_articles return (tests/test_gpu_diversify.py checks that identity).
The C entry points are called directly on preallocated buffers; CUDA events around `iters` back-to-back calls, variants of one
group alternated `--reps` times in this one process, the median per call reported with the card name and power limit read in the
same run."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import news_recommendation_model_b200 as nrm  # noqa: E402
from news_recommendation_model_b200 import _lib, engine, recommend, wire  # noqa: E402
from recommend_bench import card, stream, time_variants, users_and_pool  # noqa: E402


def torch_mmr(cpos, cval, pa, rows, k, lam, q):
    """Greedy MMR over [B,K'] candidates in plain torch: one Python iteration per pick.  -> [B,k] int64 pool positions."""
    valid = cpos >= 0
    ids = pa[cpos.clamp(min=0)].long()
    v = rows[ids, :64]
    norm = v.norm(dim=-1, keepdim=True)
    u = torch.where(norm > 0, v / norm.clamp(min=1e-30), torch.zeros_like(v))
    cat = rows[ids, 64].long()
    s = cval
    fin = valid & torch.isfinite(s)
    hi = torch.where(fin, s, torch.full_like(s, -float('inf'))).amax(1, keepdim=True)
    lo = torch.where(fin, s, torch.full_like(s, float('inf'))).amin(1, keepdim=True)
    rel = torch.where(hi > lo, (s - lo) / (hi - lo), torch.ones_like(s))
    m = torch.zeros_like(s)
    live = valid.clone()
    count = torch.zeros_like(cat)
    picks = []
    for t in range(k):
        gain = lam * rel - (1.0 - lam) * m
        j = torch.where(live, gain, torch.full_like(gain, -float('inf'))).argmax(1, keepdim=True)
        picks.append(j)
        live.scatter_(1, j, False)
        sim = (u * u.gather(1, j[:, :, None].expand(-1, 1, 64))).sum(-1)
        m = sim if t == 0 else torch.maximum(m, sim)
        if q > 0:
            count += cat == cat.gather(1, j)
            live &= count < q
    return cpos.gather(1, torch.cat(picks, 1)).long()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--out', default=None, help='also write the results as JSON to this file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('diversify_bench.py measures on a CUDA device; none is visible')
    name, power = card()
    out = {'card': name, 'power_limit': power, 'reps': args.reps, 'runs': [], 'model_pool': []}
    print(f'# {name}, power limit {power}; median of {args.reps} alternated runs')
    lib = _lib.load()
    p = engine._ptr
    table = wire.make_article_table().to('cuda')
    n_articles = table.n
    rows = table.rows
    B, N, H = 1024, 50000, 200
    rng = np.random.default_rng(7)
    pool = rng.permutation(np.arange(1, n_articles))[:N].astype(np.int32)
    pa = torch.from_numpy(pool).cuda()
    ha = torch.from_numpy(rng.choice(pool, (B, H)).astype(np.int32)).cuda()
    g = torch.Generator(device='cuda').manual_seed(5)
    logits = torch.randn(B, N, device='cuda', generator=g)
    for kc in (128, 512):
        cpos = torch.empty(B, kc, dtype=torch.int32, device='cuda')
        cval = torch.empty(B, kc, device='cuda')

        def topk():
            _lib.check(lib.nrm_pool_topk(p(logits), 1, B * N, B, N, kc, p(pa), n_articles, p(ha), H, p(cpos), p(cval), stream()),
                       'nrm_pool_topk')
        topk()
        for k in (10, 100):
            for lam in (1.0, 0.7):
                for q in (0, 2):
                    pos = torch.empty(B, k, dtype=torch.int32, device='cuda')
                    val, gain = torch.empty(B, k, device='cuda'), torch.empty(B, k, device='cuda')

                    def div():
                        _lib.check(lib.nrm_pool_diversify(p(cpos), p(cval), B, kc, k, lam, q, p(pa), N, p(rows), n_articles, p(pos),
                                                          p(val), p(gain), stream()), 'nrm_pool_diversify')

                    def tmmr():
                        return torch_mmr(cpos, cval, pa, rows, k, lam, q)
                    t = time_variants({'nrm_pool_diversify': div, f'nrm_pool_topk_k{kc}': topk, 'torch_mmr': tmmr}, args.reps, 3)
                    torch.cuda.synchronize()
                    agree = float((tmmr() == pos.long()).all(1).float().mean())
                    r = dict(B=B, N=N, candidates=kc, k=k, lam=lam, max_per_category=q, diversify_us=t['nrm_pool_diversify']['median_us'],
                             topk_us=t[f'nrm_pool_topk_k{kc}']['median_us'], torch_us=t['torch_mmr']['median_us'],
                             torch_same_list_fraction=agree, timings=t)
                    out['runs'].append(r)
                    print(f"K'={kc:3d} k={k:3d} lam={lam} cap={q}: nrm_pool_diversify {r['diversify_us']:.0f} us, "
                          f"nrm_pool_topk(K') {r['topk_us']:.0f} us, torch MMR loop {r['torch_us']:.0f} us "
                          f"(same list for {100 * agree:.1f} % of users)")
    del logits
    torch.cuda.empty_cache()

    # a real-model pool: what the re-ranking buys
    from fixtures import load_weights
    model = nrm.UserModel(1000)
    model.load_state_dict(load_weights('validation'), strict=False)
    model.to('cuda').eval().set_precision('bf16x3')
    Bm, Hm, Nm, k = 256, 200, 20000, 10
    cb, pa_m, pt = users_and_pool(table, Bm, Hm, Nm, seed=41)
    x = recommend.pool_logits(model, table, cb.hist_article, cb.hist_time, cb.hist_click, pt, pool_article=pa_m)
    top = recommend.select(x, k, pa_m, n_articles, hist_article=cb.hist_article)
    lists = {'top_articles': top}
    for lam, q in ((0.7, None), (0.5, None), (0.7, 2)):
        lists[f'diverse lam={lam} cap={q}'] = recommend.diversify(x, k, pa_m, table, lam=lam, max_per_category=q, hist_article=cb.hist_article)
    for label, rec in lists.items():
        ild, ncat = recommend.list_diversity(table, rec.article)
        r = dict(list=label, B=Bm, N=Nm, k=k, mean_ild=float(torch.nanmean(ild)), mean_categories=float(ncat.double().mean()),
                 mean_score=float(torch.nanmean(rec.score)))
        out['model_pool'].append(r)
        print(f"model pool B={Bm} N={Nm} k={k} {label:28s}: intra-list diversity {r['mean_ild']:.4f}, "
              f"categories {r['mean_categories']:.2f}, mean logit {r['mean_score']:.3f}")
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
