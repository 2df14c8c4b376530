"""Cost of drawing pool negatives: nrm_sample_negatives (negatives.NegativeSampler) alone and inside FusedTrainStep.

    python tools/negatives_bench.py [--reps 7] [--steps 50] [--out FILE.json]

At B = 1024 impressions, the pool is every article of the synthetic EB-NeRD-large table (125 541 articles, uniform weights), for
(H, C0, k) in {(50, 1, 4), (200, 5, 20)}:
  * the sampler kernel alone on a preallocated [B, C0 + k] batch (CUDA events around `iters` back-to-back launches);
  * FusedTrainStep (bf16x3, CUDA graph) with negatives= fed [B, C0] batches, against the same step without a sampler fed
    batches pre-sampled to the same width C0 + k: the difference is what sampling adds to a training step.  Batches are
    resident on the device, so both variants copy the same bytes per step.
Variants of one group are alternated `--reps` times in this one process; the median per call or step is reported with the card
name and power limit read in the same run."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

import news_recommendation_model_b200 as nrm  # noqa: E402
from news_recommendation_model_b200 import negatives, wire  # noqa: E402
from fixtures import load_weights  # noqa: E402
from recommend_bench import card, time_variants  # noqa: E402

B = 1024
SHAPES = ((50, 1, 4), (200, 5, 20))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--steps', type=int, default=50, help='training steps per timed window')
    ap.add_argument('--out', default=None, help='also write the results as JSON to this file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('negatives_bench.py measures on a CUDA device; none is visible')
    name, power = card()
    out = {'card': name, 'power_limit': power, 'reps': args.reps, 'B': B, 'kernel': [], 'train_step': []}
    print(f'# {name}, power limit {power}; median of {args.reps} alternated runs')
    table = wire.make_article_table().to('cuda')
    for H, C0, k in SHAPES:
        s = negatives.NegativeSampler(table, k=k, seed=1)
        cb = wire.make_compact_batch(table, B, H, C0, seed=3, user_num=1000, variable_history=True).to('cuda')
        wide = s.sample(cb)
        step = torch.zeros(1, dtype=torch.int64, device='cuda')
        r = time_variants({'kernel': lambda: s.sample_into(wide, C0, step)}, args.reps, 200)['kernel']
        out['kernel'].append(dict(H=H, C0=C0, k=k, **r))
        print(f'kernel  H={H:3d} C0={C0} k={k:2d}: {r["median_us"]:8.2f} us  [{r["min_us"]:.2f}-{r["max_us"]:.2f}]')

        cbs = [wire.make_compact_batch(table, B, H, C0, seed=10 + i, user_num=1000, variable_history=True).to('cuda') for i in range(2)]
        pre = [s.sample(c, step=i) for i, c in enumerate(cbs)]
        steps = {}
        for variant in ('sampled', 'pre_sampled'):
            m = nrm.UserModel(1000)
            m.load_state_dict(load_weights('train'), strict=False)
            m.to('cuda').train().set_precision('bf16x3')
            tr = nrm.FusedTrainStep(m, B, H, C0 + k, articles=table, negatives=s if variant == 'sampled' else None)
            feed = cbs if variant == 'sampled' else pre
            state = {'i': 0}

            def window(tr=tr, feed=feed, state=state):
                for _ in range(args.steps):
                    tr.step(feed[state['i'] % 2])
                    state['i'] += 1
            steps[variant] = window
        r = time_variants(steps, args.reps, 1)
        for variant, v in r.items():
            v = {key: val / args.steps for key, val in v.items()}
            out['train_step'].append(dict(H=H, C0=C0, k=k, variant=variant, **v))
            print(f'step    H={H:3d} C0={C0} k={k:2d} {variant:11s}: {v["median_us"]:8.2f} us  [{v["min_us"]:.2f}-{v["max_us"]:.2f}]')
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            json.dump(out, fh, indent=1)


if __name__ == '__main__':
    main()
