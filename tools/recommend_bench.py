"""Cost of recommending from a shared article pool: nrm_forward_pool and nrm_pool_topk.

    python tools/recommend_bench.py [--reps 7] [--out FILE.json]

Validation-checkpoint weights, H = 200 with variable history length, an article table of 125 541 articles (EB-NeRD large):
  * chunking overhead (bf16x3, B = 64, N = 4096): one nrm_forward on the batch whose candidates are the pool replicated to [64,4096]
    against nrm_forward_pool in one chunk and in the chunks pool_logits picks by default (workspace under 1 GiB);
  * throughput (bf16x3 and bf16): nrm_forward_pool at B = 256, N = 20 000 and B = 1024, N = 4096 in (user, article, history row)
    pairs per second, with the default chunk; `chunk_fixed_us` is one call at N = 8, i.e. what every chunk spends on the history
    side (embedding, w1 projection, weight preparation), which the chunked forward recomputes per chunk;
  * selection (B = 1024, N = 50 000, k = 100, exclusion on, M = 1 and 2 models): nrm_pool_topk against torch (masked_fill, for M = 2
    the softmax mean, then torch.topk), and its fraction of the HBM bound M * B * N * 4 bytes / 7.7 TB/s.  The logits are seeded
    random numbers, 205 MB per model: larger than the L2.
The C entry points are called directly on preallocated buffers; CUDA events around `iters` back-to-back calls, variants of one
group alternated `--reps` times in this one process, the median per call reported with the card name and power limit read in the
same run."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import news_recommendation_model_b200 as nrm  # noqa: E402
from news_recommendation_model_b200 import _lib, engine, recommend, wire  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(',')]
        return name, power
    except Exception:                                   # noqa: BLE001 -- reported as unknown, the timings stay valid
        return torch.cuda.get_device_name(), 'unknown'


def time_variants(fns, reps, iters):
    for fn in fns.values():                             # warm-up: module load, shared-memory attributes, side stream
        fn()
    torch.cuda.synchronize()
    res = {name: [] for name in fns}
    for _ in range(reps):
        for name, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            e1.synchronize()
            res[name].append(e0.elapsed_time(e1) * 1e3 / iters)
    return {name: dict(median_us=statistics.median(v), min_us=min(v), max_us=max(v)) for name, v in res.items()}


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def users_and_pool(table, B, H, N, seed):
    cb = wire.make_compact_batch(table, B, H, 1, seed=seed, user_num=1000, variable_history=True).to('cuda')
    rng = np.random.default_rng(seed + 1)
    pa = torch.from_numpy(rng.integers(1, table.n, N).astype(np.int32)).cuda()
    pt = torch.full((N,), int(wire.pack_time(np.array([1, 6, 17, 9])).view(np.int32)), dtype=torch.int32, device='cuda')
    return cb, pa, pt


def pool_call(model, table, cb, pa, pt, chunk):
    """A closure running nrm_forward_pool on preallocated buffers."""
    lib = _lib.load()
    B, H = cb.hist_article.shape
    N = pa.shape[0]
    ws = torch.empty(int(lib.nrm_pool_workspace_bytes(B, H, N, chunk)), dtype=torch.uint8, device='cuda')
    logits = torch.empty(B, N, device='cuda')
    users = engine.compact(table, wire.CompactBatch(None, None, cb.hist_article, cb.hist_time, cb.hist_click, pa, pt, None, None))
    p = engine._ptr
    flat = model.flat_parameters()
    args = (*users.args, B, H, N, chunk, p(flat.buf), p(model.bn.running_mean), p(model.bn.running_var), model._precision_code(),
            p(logits), p(ws), ws.numel(), stream())

    def run():
        _lib.check(lib.nrm_forward_pool(*args), 'nrm_forward_pool')
    run.logits, run.users = logits, users
    return run


def replicated_forward_call(model, table, cb, pa, pt):
    """nrm_forward on the expanded batch whose candidates are the pool replicated per user."""
    lib = _lib.load()
    B, N = cb.hist_article.shape[0], pa.shape[0]
    rep = wire.CompactBatch(cb.impression_id, cb.user_id, cb.hist_article, cb.hist_time, cb.hist_click, pa.expand(B, N).contiguous(),
                            pt.expand(B, N).contiguous(), torch.zeros(B, N, device='cuda'), cb.empty_num)
    b = wire.expand(table, rep)
    xh, xt, xg = b.x_history, b.x_target, b.x_global
    H = xh.shape[1]
    ws = torch.empty(int(lib.nrm_workspace_bytes(B, H, N, engine.MODE_EVAL)), dtype=torch.uint8, device='cuda')
    logits = torch.empty(B, N, device='cuda')
    p = engine._ptr
    flat = model.flat_parameters()
    args = (p(xh), p(xt), xt.stride(0), p(xg), xg.stride(0), B, H, N, p(flat.buf), p(model.bn.running_mean), p(model.bn.running_var),
            p(model.bn.num_batches_tracked), engine.MODE_EVAL, model._precision_code(), p(logits), p(ws), ws.numel(), stream())

    def run():
        _lib.check(lib.nrm_forward(*args), 'nrm_forward')
    run.logits = logits
    return run


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--out', default=None, help='also write the results as JSON to this file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('recommend_bench.py measures on a CUDA device; none is visible')
    from fixtures import load_weights
    name, power = card()
    out = {'card': name, 'power_limit': power, 'reps': args.reps}
    print(f'# {name}, power limit {power}; median of {args.reps} alternated runs')
    table = wire.make_article_table().to('cuda')
    model = nrm.UserModel(1000)
    model.load_state_dict(load_weights('validation'), strict=False)
    model.to('cuda').eval()

    # chunking overhead
    model.set_precision('bf16x3')
    B, H, N = 64, 200, 4096
    cb, pa, pt = users_and_pool(table, B, H, N, seed=31)
    chunk = recommend.default_chunk(B, H, N)
    fns = {'forward_replicated': replicated_forward_call(model, table, cb, pa, pt), 'pool_one_chunk': pool_call(model, table, cb, pa, pt, 4096),
           'pool_default_chunk': pool_call(model, table, cb, pa, pt, chunk)}
    t = time_variants(fns, args.reps, 5)
    torch.cuda.synchronize()
    same = all(torch.equal(fns['forward_replicated'].logits, fns[v].logits) for v in ('pool_one_chunk', 'pool_default_chunk'))
    f = t['forward_replicated']['median_us']
    out['overhead'] = dict(B=B, H=H, N=N, precision='bf16x3', default_chunk=chunk, bit_identical=same, **t)
    print(f'overhead  B={B} H={H} N={N} bf16x3: nrm_forward on the replicated pool {f:.0f} us; pool, one chunk '
          f'{t["pool_one_chunk"]["median_us"]:.0f} us ({100 * (t["pool_one_chunk"]["median_us"] / f - 1):+.1f} %); pool, chunk {chunk} '
          f'{t["pool_default_chunk"]["median_us"]:.0f} us ({100 * (t["pool_default_chunk"]["median_us"] / f - 1):+.1f} %); bit-identical: {same}')
    del fns
    torch.cuda.empty_cache()

    # throughput
    out['throughput'] = []
    for precision in ('bf16x3', 'bf16'):
        model.set_precision(precision)
        for B, N in ((256, 20000), (1024, 4096)):
            cb, pa, pt = users_and_pool(table, B, H, N, seed=32)
            chunk = recommend.default_chunk(B, H, N)
            fns = {'pool': pool_call(model, table, cb, pa, pt, chunk), 'chunk_fixed': pool_call(model, table, cb, pa[:8], pt[:8], 8)}
            t = time_variants(fns, args.reps, 2)
            us = t['pool']['median_us']
            pairs = B * N * H
            n_chunks = -(-N // chunk)
            r = dict(precision=precision, B=B, H=H, N=N, chunk=chunk, chunks=n_chunks, pairs=pairs, pairs_per_s=pairs / (us * 1e-6),
                     pool_us=us, chunk_fixed_us=t['chunk_fixed']['median_us'])
            out['throughput'].append(r)
            print(f'pool      {precision:6s} B={B} H={H} N={N} chunk={chunk} ({n_chunks} chunks): {us / 1e3:.1f} ms, '
                  f'{r["pairs_per_s"]:.3g} pairs/s; history side per chunk {r["chunk_fixed_us"]:.0f} us '
                  f'({100 * n_chunks * r["chunk_fixed_us"] / us:.1f} % of the call)')
            del fns
            torch.cuda.empty_cache()

    # selection
    lib = _lib.load()
    B, N, k, Hs = 1024, 50000, 100, 200
    g = torch.Generator(device='cuda').manual_seed(5)
    cb, pa, _ = users_and_pool(table, B, Hs, N, seed=33)
    ha = cb.hist_article
    clicked = torch.zeros(B, N, dtype=torch.bool, device='cuda')      # the torch baseline's [B,N] mask, built once, outside the timing
    for b in range(B):
        clicked[b] = torch.isin(pa, ha[b][ha[b] != 0])
    mask = ((pa < 1) | (pa >= table.n))[None, :] | clicked
    out['selection'] = []
    p = engine._ptr
    for M in (1, 2):
        logits = torch.randn(M, B, N, device='cuda', generator=g)
        pos = torch.empty(B, k, dtype=torch.int32, device='cuda')
        val = torch.empty(B, k, device='cuda')

        def kernel():
            _lib.check(lib.nrm_pool_topk(p(logits), M, B * N, B, N, k, p(pa), table.n, p(ha), Hs, p(pos), p(val), stream()), 'nrm_pool_topk')

        def torch_baseline():
            if M == 1:
                return torch.topk(logits[0].masked_fill(mask, float('-inf')), k, dim=1)
            s = torch.softmax(logits.masked_fill(mask, float('-inf')), dim=2).mean(0)
            return torch.topk(s, k, dim=1)
        t = time_variants({'nrm_pool_topk': kernel, 'torch': torch_baseline}, args.reps, 10)
        us = t['nrm_pool_topk']['median_us']
        bound_us = M * B * N * 4 / HBM_BYTES_PER_S * 1e6
        ref = torch_baseline()
        same = bool(torch.equal(pos.long(), ref.indices)) if M == 1 else None
        r = dict(M=M, B=B, N=N, k=k, H=Hs, kernel_us=us, torch_us=t['torch']['median_us'], hbm_bound_us=bound_us,
                 fraction_of_hbm_bound=bound_us / us, same_positions_as_torch=same)
        out['selection'].append(r)
        print(f'select    M={M} B={B} N={N} k={k}: nrm_pool_topk {us:.0f} us, torch {r["torch_us"]:.0f} us, HBM bound {bound_us:.0f} us '
              f'({100 * r["fraction_of_hbm_bound"]:.0f} %)' + (f'; same positions as torch.topk: {same}' if M == 1 else ''))
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
