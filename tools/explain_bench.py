"""Cost of the attention-score export: eval nrm_forward against nrm_forward_scores against nrm_forward_scores + nrm_history_topk.

    python tools/explain_bench.py [--reps 15] [--iters 20] [--k 5] [--out FILE.json]

Validation-checkpoint weights, precisions bf16x3 and fp32, two shapes:
  * the scoring shape of bench.py: batch 80, H = 200 with variable history length, candidate lists ~ clipped lognormal [5, 100]
    padded to the batch maximum (the common pad tail trimmed as test.py:52-56);
  * B = 1024, H = 200 (variable length), C = 15: the shape of a training batch.
The C entry points are called directly on preallocated buffers (no Python work inside the timed loops), CUDA events around
`--iters` back-to-back calls, the three variants alternated `--reps` times in this one process; the median per call is
reported with the card name and power limit read in the same run."""
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

import torch  # noqa: E402

import news_recommendation_model_b200 as nrm  # noqa: E402
from news_recommendation_model_b200 import _lib, engine  # noqa: E402
from news_recommendation_model_b200.synthetic import make_batch  # noqa: E402


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(',')]
        return name, power
    except Exception:                                   # noqa: BLE001 -- reported as unknown, the timings stay valid
        return torch.cuda.get_device_name(), 'unknown'


def setup(model, b, k):
    lib = _lib.load()
    keep = b.x_target.shape[1] - int(b.empty_num.min())
    xh, xt, xg = engine.prepare_inputs(b.x_history, b.x_target[:, :keep], b.x_global[:, :keep])
    B, H, C = xh.shape[0], xh.shape[1], xt.shape[1]
    dev = xh.device
    flat = model.flat_parameters()
    ws = torch.empty(int(lib.nrm_workspace_bytes(B, H, C, engine.MODE_EVAL)), dtype=torch.uint8, device=dev)
    logits = torch.empty(B, C, device=dev)
    scores = torch.empty(2, B, C, H, device=dev)
    idx = torch.empty(2, B, C, k, dtype=torch.int32, device=dev)
    val = torch.empty(2, B, C, k, device=dev)
    p = engine._ptr
    prec = model._precision_code()
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    common = (p(xh), p(xt), xt.stride(0), p(xg), xg.stride(0), B, H, C, p(flat.buf), p(model.bn.running_mean), p(model.bn.running_var),
              p(model.bn.num_batches_tracked), engine.MODE_EVAL, prec, p(logits))

    def forward():
        _lib.check(lib.nrm_forward(*common, p(ws), ws.numel(), st), 'nrm_forward')

    def forward_scores():
        _lib.check(lib.nrm_forward_scores(*common, p(scores), p(ws), ws.numel(), st), 'nrm_forward_scores')

    def forward_scores_topk():
        forward_scores()
        _lib.check(lib.nrm_history_topk(p(scores), B, C, H, k, p(xh), None, p(idx), p(val), st), 'nrm_history_topk')
    return (B, H, C), {'forward': forward, 'forward_scores': forward_scores, 'forward_scores_topk': forward_scores_topk}


def time_variants(fns, reps, iters):
    for fn in fns.values():                             # warm-up: module load, shared-memory attributes, side stream
        for _ in range(3):
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


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--reps', type=int, default=15)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--k', type=int, default=5)
    ap.add_argument('--out', default=None, help='also write the results as JSON to this file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('explain_bench.py measures on a CUDA device; none is visible')
    from fixtures import load_weights
    dev = torch.device('cuda')
    name, power = card()
    model = nrm.UserModel(1000)
    model.load_state_dict(load_weights('validation'), strict=False)
    model.to(dev).eval()
    shapes = {'scoring_b80': make_batch(80, 200, 100, seed=777, user_num=1000, variable_history=True, variable_candidates=True),
              'train_b1024_c15': make_batch(1024, 200, 15, seed=778, user_num=1000, variable_history=True)}
    out = {'card': name, 'power_limit': power, 'k': args.k, 'reps': args.reps, 'iters': args.iters, 'results': []}
    print(f'# {name}, power limit {power}; median of {args.reps} alternated runs of {args.iters} calls, k = {args.k}')
    print(f'{"shape":16s} {"precision":9s} {"B,H,C":14s} {"forward us":>11s} {"+scores us":>11s} {"+topk us":>11s} {"scores %":>9s} {"topk %":>7s}')
    for precision in ('bf16x3', 'fp32'):
        model.set_precision(precision)
        for shape, b in shapes.items():
            (B, H, C), fns = setup(model, b.to(dev), args.k)
            t = time_variants(fns, args.reps, args.iters)
            f, s, k = (t[v]['median_us'] for v in ('forward', 'forward_scores', 'forward_scores_topk'))
            out['results'].append(dict(shape=shape, precision=precision, B=B, H=H, C=C, **{v: t[v] for v in t}))
            print(f'{shape:16s} {precision:9s} {f"{B},{H},{C}":14s} {f:11.1f} {s:11.1f} {k:11.1f} {100 * (s / f - 1):8.1f}% {100 * (k / f - 1):6.1f}%')
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
