#!/usr/bin/env python
"""Headline benchmark: training-step throughput of the EB-NeRD recommender hot path.

  python bench.py --gpus 1 --steps K --warmup W            (our CUDA path)
  python bench.py --impl reference --steps K --warmup W    (the unmodified reference's CPU path from baseline/_ref)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (data parallel)

One "step" = train.py:69-75 on one batch of synthetic EB-NeRD-shaped impressions:
forward -> loss -> backward -> Adam -> zero_grad.  Workload = BASELINE.json configs[1]
(B=1024 impressions per GPU, history 50, 1 positive + 4 negatives, fp32), weights from the
shipped train checkpoint.  Prints ONE JSON line (see DESIGN.md section 6 for every field).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

D = 64
N_POOL = 6            # distinct batches rotated through: 6 x 36 MB of inputs > the 126 MB L2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=1024, help='impressions per GPU per step')
    ap.add_argument('--history', type=int, default=50)
    ap.add_argument('--candidates', type=int, default=5)
    ap.add_argument('--user-num', type=int, default=1000)
    ap.add_argument('--precision', default='bf16x3', choices=['fp32', 'bf16', 'bf16x3'],
                    help='pair products: bf16x3 = tcgen05 with hi/lo split operands (fp32-grade, default), fp32 = FFMA, bf16 = tcgen05 bf16')
    ap.add_argument('--no-variants', action='store_true', help='skip the short resident runs of the other two precisions')
    ap.add_argument('--sync-bn', action='store_true', help='all-reduce BatchNorm statistics across ranks')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='FusedTrainStep issues the C-ABI calls eagerly instead of replaying a CUDA graph')
    ap.add_argument('--cpu-steps', type=int, default=60, help='train steps of the CPU port timed for cpu_baseline (about 15 s on 16 cores)')
    ap.add_argument('--no-scoring', action='store_true', help='skip the scoring (configs[2]) leg')
    ap.add_argument('--no-loader', action='store_true', help='skip the record-list -> loader -> loss leg')
    ap.add_argument('--no-large-users', action='store_true', help='skip the user_num = 2 000 000 leg')
    ap.add_argument('--no-long-history', action='store_true', help='skip the configs[4] leg (B=4096, H=256)')
    ap.add_argument('--no-dp-check', action='store_true', help='skip the N-rank vs single-process numerical pre-flight (world > 1)')
    ap.add_argument('--no-affinity', action='store_true', help='do not bind each rank to the CPU cores local to its GPU')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps write what the last of them computed (loss, logits, '
                                                          'gradients, model state after the update) as DIR/<name>.npy; see dump_outputs')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or int(os.environ.get('WORLD_SIZE', '1')) > 1):
        ap.error('--dump-outputs writes the outputs of --impl ours in one process')
    return args


def load_weights():
    from fixtures import load_weights as lw
    return lw('train')


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=float(p['hbm_gbs']), tensor=float(p.get('bf16_tflops_sustained', p['bf16_tflops'])), source='measured')
    return dict(hbm=6650.0, tensor=1400.0, source='fallback')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(',')]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx = max(mx, float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(names, parts[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU path (baseline/_ref; oracle/reference_port.py only when that copy is absent)
# ------------------------------------------------------------------------------------------
def cpu_reference_rate(args, steps, warmup):
    """Time train.py:69-75 on the host cores.  Preferred: the UNMODIFIED reference `models.user_model.UserModel`
    from baseline/_ref (byte copy made by oracle/make_ref.py; kind "reference").  Fallback when that copy is absent:
    the oracle port (kind "port").  -> (impressions/s, ms/step, cores, kind)"""
    from news_recommendation_model_b200.synthetic import make_batch
    from oracle.make_ref import reference_modules, reference_root
    torch.set_num_threads(os.cpu_count())
    batches = [make_batch(args.batch, args.history, args.candidates, seed=100 + i, user_num=args.user_num) for i in range(2)]
    times = []
    if reference_root() is not None:
        kind = 'reference'
        with reference_modules(with_scripts=False) as ref:
            model = ref.UserModel(args.user_num)               # train.py:46
            model.load_state_dict(load_weights(), strict=False)
            model.train()
            opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)   # train.py:48
            for i in range(warmup + steps):
                b = batches[i % len(batches)]
                t0 = time.perf_counter()
                out = model(b.x_history, b.x_target, b.x_global)                 # train.py:69
                loss = model.loss(b.user_id, out, b.label)                         # train.py:71
                loss.backward()                                                    # train.py:73-75
                opt.step()
                opt.zero_grad()
                dt = time.perf_counter() - t0
                if i >= warmup:
                    times.append(dt)
    else:
        kind = 'port'
        from oracle import reference_port as O
        p = O.load_params(load_weights(), user_num=args.user_num)
        leaves = [p[k].requires_grad_(True) for k in O.TRAINABLE_KEYS + ('delta',)]
        opt = torch.optim.Adam(leaves, lr=1e-3, weight_decay=1e-5)
        for i in range(warmup + steps):
            b = batches[i % len(batches)]
            t0 = time.perf_counter()
            out = O.user_model_forward(p, b.x_history, b.x_target, b.x_global, training=True)
            loss = O.user_model_loss(p['delta'], b.user_id, out, b.label)
            loss.backward()
            opt.step()
            opt.zero_grad()
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    total = float(np.sum(times))
    return args.batch * steps / total, total / steps * 1e3, os.cpu_count(), kind


def _cpu_sample_text(kind, steps, warmup, batch):
    what = ('the unmodified reference models.user_model.UserModel (baseline/_ref, byte copy of /root/reference) driven as train.py:69-75'
            if kind == 'reference' else 'oracle/reference_port.py (baseline/_ref absent)')
    return f'{steps} full train steps (B={batch}) of {what} on the host CPU, {warmup} warm-up'


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps, warmup = args.steps, max(1, min(args.warmup, 5))
    rate, ms, cores, kind = cpu_reference_rate(args, steps, warmup)
    line = {
        'impl': 'reference', 'metric': 'train_impressions_per_sec', 'value': rate, 'unit': 'impressions/s',
        'n_gpus': args.gpus, 'steps': steps, 'warmup': warmup, 'ms_per_step': ms, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, 1),
        'cpu_baseline': {'value': rate, 'unit': 'impressions/s', 'cores': cores, 'kind': kind,
                         'sample': _cpu_sample_text(kind, steps, warmup, args.batch)},
        'e2e': {'value': rate, 'unit': 'impressions/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {'workload': f'train step (fwd+loss+bwd+Adam), B={args.batch}/GPU, H={args.history}, C={args.candidates} '
                        f'(1 pos + {args.candidates - 1} neg), user_num={args.user_num}, ckpt_ebnerd_large_train_final weights',
            'global_batch': args.batch * world, 'history': args.history, 'candidates': args.candidates,
            'parallelism': f'dp{world}', 'precision': args.precision, 'sync_bn': bool(args.sync_bn),
            'l2_policy': f'{N_POOL} distinct input batches rotated (~{N_POOL * 36} MB of inputs > 126 MB L2)'}



# ------------------------------------------------------------------------------------------
# kernel timing + roofline helpers
# ------------------------------------------------------------------------------------------
def timed_kernels(lib, fn, n):
    """Run fn(i) n times with the library's per-kernel-group CUDA events enabled (events on the launch stream of every group,
    nrm_timing_enable); -> {group: ms per call of fn}."""
    import ctypes
    from news_recommendation_model_b200 import _lib
    lib.nrm_timing_enable(1)
    for i in range(n):
        fn(i)
    torch.cuda.synchronize()
    cbuf = ctypes.create_string_buffer(16384)
    _lib.check(lib.nrm_timing_report(cbuf, 16384), 'nrm_timing_report')
    lib.nrm_timing_enable(0)
    kern = {}
    for ln in cbuf.value.decode().strip().splitlines():
        name, cnt, tot = ln.split()[:3]
        kern[name] = {'launch_groups': int(cnt), 'ms': float(tot) / n}
    return kern


ROWSTACKED = set() if os.environ.get('NRM_ATT_ITEM_TILES') else {'attention_input_grad_label'}


def algorithmic_work(B, H, C, total_params):
    """Algorithmic FLOPs / bytes of every timed kernel group of one training step (SURVEY 8d per-impression figures x B;
    DESIGN.md section 4).  EVERY group is a roofline candidate: the dominant one is whichever takes longest."""
    P, R, NH = B * C * H, B * C, B * H
    N = NH + R
    head = 2.0 * 87186 * R                                       # 5 x (264 x 66) + 66 MACs per candidate row
    return {
        'attention_forward_label': ('tensor', 2.0 * P * D * D), 'attention_forward_textimg': ('tensor', 2.0 * P * D * D),
        'attention_forward': ('tensor', 2 * 2.0 * P * D * D),    # both branches in one launch (tensor-core paths)
        # backward products per pair: hid recompute + weight gradient (both branches); + input gradient (label branch: its own
        # kernel on the row-stacked path, inside attention_backward_label on the item-tile path)
        'attention_backward_label': ('tensor', (2 if 'attention_input_grad_label' in ROWSTACKED else 3) * 2.0 * P * D * D),
        'attention_input_grad_label': ('tensor', 2.0 * P * D * D),
        'attention_backward_textimg': ('tensor', 2 * 2.0 * P * D * D),
        'head_forward': ('tensor', head), 'head_backward': ('tensor', head), 'head_wgrad': ('tensor', head),   # dgrad chain | weight gradients
        'w1_backward': ('tensor', 2 * 2.0 * 66 * 64 * NH),
        'embed_rows': ('hbm', 8.0 * (80 * NH + 81 * R) + 4.0 * (66 * NH + 64 * NH + 136 * R)),
        'w1_forward': ('hbm', 4.0 * (66 + 64) * NH),
        'bn_statistics': ('hbm', 4.0 * 264 * R),
        'attention_finish': ('hbm', 4.0 * 2 * (64 + 64 + 264) * R),
        'small_linear_grads': ('hbm', 4.0 * (19 + 16) * N + 8.0 * 6 * N),
        'table_l1': ('hbm', 4.0 * (6 * 32 + 5 * 8) * N + 4.0 * 11 * N), 'table_l2': ('hbm', 4.0 * (6 * 32 + 5 * 8) * N / 128),
        'adam': ('hbm', 28.0 * total_params),
    }


# Groups the library launches on its side stream, concurrently with main-stream kernels that fill the SMs (the text/img attention
# backward, the table gradients): their event-to-event time is mostly waiting for SMs, so they are reported (kernels_ms_per_step,
# roofline_fraction_by_kernel) but are not candidates for the DOMINANT kernel; profiles/ holds their stand-alone ncu durations.
SIDE_STREAM_GROUPS = {'w1_backward', 'small_linear_grads', 'head_wgrad'}


def pick_roofline(kern, work, pk, precision, traffic_table=None):
    cand = {k: v for k, v in kern.items() if k in work and k not in SIDE_STREAM_GROUPS}
    if not cand:
        return None
    top = max(cand, key=lambda k: cand[k]['ms'])
    bound, w = work[top]
    dur = kern[top]['ms'] / 1e3
    traffic = (traffic_table or {}).get(top)
    if bound == 'tensor':
        ach = w / dur / 1e12
        return {'kernel': top, 'bound': 'tensor', 'achieved': ach, 'peak': pk['tensor'], 'unit': 'TFLOP/s', 'frac': ach / pk['tensor'],
                'traffic': traffic, 'peak_source': pk['source'] + ' bf16 sustained (cuBLAS)', 'algorithmic_flops_per_launch': w,
                'launch_ms': dur * 1e3,
                'note': {'fp32': 'FFMA path: the products run on the CUDA cores',
                         'bf16': 'tcgen05 tiles, bf16 operands',
                         'bf16x3': 'attention: tcgen05 tiles, 3 MMAs issued per algorithmic product (hi/lo split); bound by the GELU / '
                                   'operand-build work on the CUDA cores (issue slots), see DESIGN.md section 4.  head forward / dgrad: tcgen05 M = 64 tiles, '
                                   'six part products (three-part bf16 split, fp32-grade); w1 backward: tcgen05; head weight gradients: FFMA'}[precision]}
    ach = w / dur / 1e9
    return {'kernel': top, 'bound': 'hbm', 'achieved': ach, 'peak': pk['hbm'], 'unit': 'GB/s', 'frac': ach / pk['hbm'], 'traffic': traffic,
            'peak_source': pk['source'], 'algorithmic_bytes_per_launch': w, 'launch_ms': dur * 1e3}


def all_fractions(kern, work, pk):
    """{group: fraction of its roofline}: the whole table, so that a regression anywhere is visible."""
    out = {}
    for k, v in kern.items():
        if k in work and v['ms'] > 0:
            bound, w = work[k]
            out[k] = round(w / (v['ms'] / 1e3) / (pk['tensor'] * 1e12 if bound == 'tensor' else pk['hbm'] * 1e9), 4)
    return out


def scoring_cpu_baseline(host_batch, user_num):
    """The reference's own scoring loop (test.py:31-74 model_test, unmodified, baseline/_ref) on the host cores: one batch-80
    sample of the bench's scoring workload, 2-model ensemble (test.py:150-152)."""
    import queue
    from fixtures import load_weights as lw
    from oracle.make_ref import reference_modules, reference_root
    if reference_root() is None:
        return None
    torch.set_num_threads(os.cpu_count())
    b = host_batch
    n = int(b.x_history.shape[0])
    records = [[b.impression_id[i].numpy(), b.user_id[i].numpy(), b.x_history[i].numpy(), b.x_target[i].numpy(), b.x_global[i].numpy(),
                b.label[i].numpy(), b.label_id[i].numpy(), b.empty_num[i].numpy()] for i in range(n)]
    with reference_modules() as ref:
        models = []
        for name in ('train', 'validation'):
            m = ref.UserModel(user_num)
            m.load_state_dict(lw(name), strict=False)
            models.append(m)
        ref.model_test(models, records[:16], torch.device('cpu'), queue.Queue(), [], batch_size=16)     # warm-up
        t0 = time.perf_counter()
        ref.model_test(models, records, torch.device('cpu'), queue.Queue(), [], batch_size=80)          # test.py:138 batch size
        dt = time.perf_counter() - t0
    return {'value': n / dt, 'unit': 'impressions/s', 'cores': os.cpu_count(), 'kind': 'reference', 'ms_per_batch': dt * 1e3,
            'sample': f'one batch of {n} impressions (H=200, ragged candidates) through the unmodified reference test.py:model_test on the host CPU, '
                      '2-model ensemble'}


DUMP_ELEMENTS = 1 << 20       # per array: logits or delta of a large --batch / --user-num are stored as a fixed seeded sample


def dump_outputs(out_dir, tr, model, loss):
    """What the last timed FusedTrainStep step of a single process computed, as out_dir/<name>.npy: loss, logits,
    grad.<parameter> (the gradient the update used) and state.<key> (model.state_dict() after the update), float32 (float64 for integer buffers).  An array
    of more than DUMP_ELEMENTS elements keeps the same seeded sample of its flattened values in every run, so two builds run
    with the same arguments compare array for array."""
    arrays = {'loss': torch.tensor([loss.item()]), 'logits': tr.logits}
    arrays.update({'grad.' + name: tr.grads[off:off + n].view(shape) for name, off, n, shape in tr.flat.slots})
    arrays.update({'state.' + k: v for k, v in model.state_dict().items()})
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if a.size > DUMP_ELEMENTS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_ELEMENTS, replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), a)
        total += a.nbytes
    assert total <= 64 << 20, f'{total} bytes of outputs'


def make_records(n, H, C, seed, user_num):
    """Synthetic impressions in the reference's record-list layout (tool/process_data.py:252; what import_processed_data returns)."""
    from news_recommendation_model_b200.synthetic import make_batch
    b = make_batch(n, H, C, seed=seed, user_num=user_num, fp32_exact=True)
    return [[b.impression_id[i].numpy(), b.user_id[i].numpy(), b.x_history[i].numpy(), b.x_target[i].numpy(), b.x_global[i].numpy(),
             b.label[i].numpy(), b.label_id[i].numpy(), b.empty_num[i].numpy()] for i in range(n)]


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import news_recommendation_model_b200 as nrm
    from news_recommendation_model_b200 import _lib
    from news_recommendation_model_b200.dp import DataParallel
    from news_recommendation_model_b200.synthetic import make_batch

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    from news_recommendation_model_b200.dp import bind_to_local_cpus
    cpus = None if args.no_affinity else bind_to_local_cpus(local)     # before any pinned buffer is allocated
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.load()

    model = nrm.UserModel(args.user_num)
    model.load_state_dict(load_weights(), strict=False)
    model.to(dev).train()
    model.set_precision(args.precision)
    if world > 1:
        DataParallel(model, sync_bn=args.sync_bn)

    # pre-flight under data parallelism: N ranks vs one process on the same batch, identical replicas (tests/dp_check.py)
    dp_parity = None
    if world > 1 and not args.no_dp_check:
        import dp_check
        ok, rep = dp_check.run_check(dev, rank, world, precision=args.precision)
        dp_parity = {'status': 'ok' if ok else 'FAILED', **{k: (round(v, 9) if isinstance(v, float) else v) for k, v in rep.items()}}

    B, H, C = args.batch, args.history, args.candidates
    host = [make_batch(B, H, C, seed=1234 + 97 * rank + i, user_num=args.user_num).pin() for i in range(N_POOL)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    K, W = args.steps, max(3, args.warmup)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    # ---- A. the pipelined public API (news_recommendation_model_b200.FusedTrainStep): the five
    #         C-ABI calls of train.py:69-75 per step, CUDA-graph replayed, N_POOL input slots.
    from news_recommendation_model_b200 import wire
    table_host = wire.make_article_table()
    table = table_host.to(dev)                    # 125 541 articles x 320 B = 40 MB, resident in HBM for the compact wire format
    tr = nrm.FusedTrainStep(model, B, H, C, lr=1e-3, weight_decay=1e-5, nslots=N_POOL, use_graph=not args.no_graph, articles=table)
    slots = [tr.load(hb) for hb in host]          # all slots resident in HBM
    torch.cuda.synchronize()
    for i in range(max(W, N_POOL)):               # every slot replays its own CUDA graph: capture all of them before timing
        tr.run(slots[i % N_POOL])
    barrier()
    with ClockSampler(local) as clk:
        e0.record()
        for i in range(K):
            last = tr.run(slots[i % N_POOL])
        e1.record()
        barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    value = world * B * K / (ms_total / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tr, model, last)     # before the legs below train the same model further

    # ---- B. end to end through the same API: every step copies its batch from pinned host memory
    #         into a device slot (copy stream, one batch ahead) and the host reads every step's loss.
    def e2e_loop(n, host=host):
        nxt = tr.load(host[0])
        prev, last = None, 0.0
        for i in range(n):
            cur = nxt
            if i + 1 < n:
                nxt = tr.load(host[(i + 1) % N_POOL])
            h = tr.run(cur)
            if prev is not None:
                last = prev.item()                # D2H result of the previous step (never stalls the GPU)
            prev = h
        return prev.item()
    e2e_loop(3)
    barrier()
    e0.record()
    e2e_loop(K)
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * B * K / (e2e_ms / 1e3)
    h2d = host[0].input_bytes()
    # the copies alone (same pinned buffers, same copy stream, nothing else running): the floor of the end-to-end step
    torch.cuda.synchronize()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(tr.copy_stream):
        c0.record()
        for i in range(10):
            tr.load(host[i % N_POOL])
        c1.record()
    torch.cuda.synchronize()
    h2d_ms = max_over_ranks(c0.elapsed_time(c1) / 10)

    # ---- B2. the same loop fed in the compact wire format (wire.py, the additional entry point of SURVEY section 8f N3):
    #          ids into the resident article table instead of packed float64 rows; the step starts with the expansion kernel
    host_c = [wire.make_compact_batch(table_host, B, H, C, seed=4321 + 97 * rank + i, user_num=args.user_num).pin() for i in range(N_POOL)]
    e2e_loop(max(3, N_POOL), host_c)              # re-captures every slot's graph with the expansion in front
    barrier()
    e0.record()
    e2e_loop(K, host_c)
    e1.record()
    barrier()
    e2ec_ms = max_over_ranks(e0.elapsed_time(e1))
    e2ec = {'value': world * B * K / (e2ec_ms / 1e3), 'unit': 'impressions/s', 'h2d_bytes_per_step': host_c[0].input_bytes(),
            'd2h_bytes_per_step': 4, 'ms_per_step': e2ec_ms / K,
            'note': 'same FusedTrainStep fed wire.CompactBatch (article ids + click features, article table resident in HBM); '
                    'NOT the reference wire format - e2e above is'}

    # ---- C. the drop-in nn.Module path driven exactly like train.py (autograd + FusedAdam), device-resident
    opt = nrm.FusedAdam(model.parameters(), lr=1e-3, weight_decay=1e-5)
    pool = [b.to(dev) for b in host]

    def step(b):
        out = model(b.x_history, b.x_target, b.x_global)
        loss = model.loss(b.user_id, out, b.label)
        loss.backward()
        opt.step()
        opt.zero_grad()
        return loss
    for i in range(W):
        step(pool[i % N_POOL])
    barrier()
    e0.record()
    for i in range(K):
        step(pool[i % N_POOL])
    e1.record()
    barrier()
    mod_ms = max_over_ranks(e0.elapsed_time(e1))
    launches = tr.launches_per_step                  # kernels of ours per step (counted while the step was recorded)

    # ---- per-kernel timing pass (CUDA events on the launch stream inside the library)
    kt_steps = min(K, 8)
    kern = timed_kernels(lib, lambda i: step(pool[i % N_POOL]), kt_steps)
    pk = peaks()
    total_params = model.flat_parameters().total
    work = algorithmic_work(B, H, C, total_params)
    traffic_table = None
    for tname in ('r02_traffic.json', 'r01_traffic.json'):
        tpath = os.path.join(ROOT, 'profiles', tname)
        if os.path.exists(tpath):
            traffic_table = json.load(open(tpath)).get(args.precision, {})
            break
    roofline = pick_roofline(kern, work, pk, args.precision, traffic_table)
    roofline_all = all_fractions(kern, work, pk)

    # ---- A2. loader leg (SURVEY 8f N4): from the reference's record list to the loss.  wire.from_records converts the records once
    #          (timed, reported), wire.PrefetchLoader's background thread gathers shuffled batches into its fixed pinned ring and
    #          FusedTrainStep trains on them; the timed region is whole epochs of that loop, every loss read by the host.
    loader_leg = None
    if not args.no_loader:
        n_rec = B * 8
        t0 = time.perf_counter()
        records = make_records(n_rec, H, C, 31337 + rank, args.user_num)
        t_gen = time.perf_counter() - t0
        t0 = time.perf_counter()
        ds = wire.from_records(records, pin=True)
        t_conv = time.perf_counter() - t0
        del records
        tr_l = nrm.FusedTrainStep(model, B, H, C, lr=1e-3, weight_decay=1e-5, nslots=3, use_graph=not args.no_graph, articles=ds.table.to(dev))

        loader = wire.PrefetchLoader(ds, B, shuffle=True, drop_last=True, depth=4)      # the pinned ring is allocated once

        def epoch(seed):
            prev, last = None, 0.0
            for cb in loader.set_epoch(seed):
                h = tr_l.step(cb)
                if prev is not None:
                    last = prev.item()
                prev = h
            return prev.item()
        epoch(0)                                            # captures the graphs of the three slots
        barrier()
        n_ep = max(1, (K + 7) // 8)
        e0.record()
        for ep in range(n_ep):
            epoch(1 + ep)
        e1.record()
        barrier()
        l_ms = max_over_ranks(e0.elapsed_time(e1))
        loader_leg = {'value': world * B * 8 * n_ep / (l_ms / 1e3), 'unit': 'impressions/s', 'ms_per_step': l_ms / (8 * n_ep), 'steps': 8 * n_ep,
                      'records': n_rec, 'from_records_s': round(t_conv, 3), 'articles_in_table': ds.table.n,
                      'h2d_bytes_per_step': next(iter(ds.batches(B, pin=False))).input_bytes(),
                      'note': 'record list (process_data.py:252 layout) -> wire.from_records (once) -> PrefetchLoader thread + fixed pinned '
                              'ring -> FusedTrainStep (compact wire format); shuffled epochs, drop_last, every loss read by the host'}
        del tr_l, ds, loader

    # ---- D. scoring (BASELINE configs[2]; test.py:31-74 + 118-132): 2-model ensemble (train + validation checkpoints), eval mode,
    #         H = 200 (the ETL's pad length), ragged candidate lists padded to the batch maximum, pads trimmed per batch as
    #         test.py:52-56, epilogue + stable ranks + submission text on the GPU (scoring.py).  Batch 80 as test.py:138 and a
    #         large-batch variant; resident inputs and end to end (pinned host float64 inputs in, text bytes out).
    scoring = None
    if not args.no_scoring:
        from fixtures import load_weights as lw
        model.set_precision(args.precision)
        m_val = nrm.UserModel(args.user_num)
        m_val.load_state_dict(lw('validation'), strict=False)
        m_val.to(dev).eval().set_precision(args.precision)
        model.eval()
        ens = [model, m_val]
        scoring = {'unit': 'impressions/s', 'config': 'eval, 2-model ensemble, H=200 (variable length), candidates ~ clipped lognormal [5,100] padded to the '
                   'batch maximum, softmax / pad re-softmax / stable ranks / submission text on the GPU'}
        for Bs, reps in ((80, 20), (1024, 4)):
            hb = [make_batch(Bs, 200, 100, seed=777 + 31 * rank + i, user_num=args.user_num, variable_history=True, variable_candidates=True).pin()
                  for i in range(2)]
            trims = [int(b.empty_num.min()) for b in hb]
            db = [b.to(dev) for b in hb]

            ring = nrm.scoring.SubmissionRing(Bs, 100, depth=4, device=dev)       # pinned result ring: the text comes back a few batches late

            def score(b, trim, text):
                keep = b.x_target.shape[1] - trim
                with torch.no_grad():
                    sc, rk = nrm.scoring.ensemble_scores(ens, b.x_history, b.x_target[:, :keep], b.x_global[:, :keep], b.empty_num - trim)
                if not text:
                    return sc
                done = ring.push(b.impression_id, rk, b.empty_num - trim)
                return done[0] if done is not None else b''
            for i in range(2):
                score(db[i], trims[i], False)
            barrier()
            e0.record()
            for i in range(reps):
                score(db[i % 2], trims[i % 2], False)
            e1.record()
            barrier()
            ms_res = max_over_ranks(e0.elapsed_time(e1)) / reps
            # end to end: batch i + 1 travels on a copy stream while batch i is scored; every batch's text bytes come back through
            # scoring.SubmissionRing (pinned, asynchronous: no blocking copy per batch)
            cs = torch.cuda.Stream(dev)
            NSLOT = 3                                    # fixed device staging slots (no allocation inside the timed loop)
            stage = [hb[0].to(dev) for _ in range(NSLOT)]
            done_ev = [None] * NSLOT                     # compute that read the slot has finished

            def fetch(i):
                k = i % NSLOT
                with torch.cuda.stream(cs):
                    if done_ev[k] is not None:
                        cs.wait_event(done_ev[k])
                    src, dst = hb[i % 2], stage[k]
                    for f in src.__dataclass_fields__:
                        getattr(dst, f).copy_(getattr(src, f), non_blocking=True)
                    ev = torch.cuda.Event(); ev.record(cs)
                return dst, ev, k

            def e2e_scoring(n):
                total = 0
                nxt = fetch(0)
                for i in range(n):
                    cur, ev, k = nxt
                    if i + 1 < n:
                        nxt = fetch(i + 1)
                    torch.cuda.current_stream(dev).wait_event(ev)
                    total += len(score(cur, trims[i % 2], True))
                    done_ev[k] = torch.cuda.Event(); done_ev[k].record(torch.cuda.current_stream(dev))
                return total + sum(len(t) for t, _ in ring.drain())          # every batch's text is on the host when the loop ends
            e2e_scoring(2)
            barrier()
            e0.record()
            nbytes = e2e_scoring(reps)
            e1.record()
            barrier()
            ms_e2e = max_over_ranks(e0.elapsed_time(e1)) / reps
            # the same loop fed in the compact wire format (ids into the resident article table, wire.expand on the GPU)
            hc = [wire.make_compact_batch(table_host, Bs, 200, 100, seed=555 + 31 * rank + i, user_num=args.user_num, variable_history=True,
                                          variable_candidates=True).pin() for i in range(2)]
            trims_c = [int(b.empty_num.min()) for b in hc]

            cstage = [hc[0].to(dev) for _ in range(NSLOT)]                # fixed device slots: compact batch + its expansion
            xstage = [wire.expand(table, c) for c in cstage]
            cdone = [None] * NSLOT

            def fetch_c(i):
                k = i % NSLOT
                with torch.cuda.stream(cs):
                    if cdone[k] is not None:
                        cs.wait_event(cdone[k])
                    src, dst = hc[i % 2], cstage[k]
                    for f in src.__dataclass_fields__:
                        getattr(dst, f).copy_(getattr(src, f), non_blocking=True)
                    ev = torch.cuda.Event(); ev.record(cs)
                return ev, k

            def e2e_scoring_compact(n):
                total = 0
                nxt = fetch_c(0)
                for i in range(n):
                    ev, k = nxt
                    if i + 1 < n:
                        nxt = fetch_c(i + 1)
                    torch.cuda.current_stream(dev).wait_event(ev)
                    x = xstage[k]
                    wire.expand_into(table, cstage[k], x.x_history, x.x_target, x.x_global, x.label)
                    x.impression_id, x.empty_num = cstage[k].impression_id, cstage[k].empty_num
                    total += len(score(x, trims_c[i % 2], True))
                    cdone[k] = torch.cuda.Event(); cdone[k].record(torch.cuda.current_stream(dev))
                return total + sum(len(t) for t, _ in ring.drain())
            e2e_scoring_compact(2)
            barrier()
            e0.record()
            e2e_scoring_compact(reps)
            e1.record()
            barrier()
            ms_e2ec = max_over_ranks(e0.elapsed_time(e1)) / reps
            scoring[f'batch_{Bs}'] = {'value': world * Bs / (ms_res / 1e3), 'ms_per_batch': ms_res,
                                      'e2e': {'value': world * Bs / (ms_e2e / 1e3), 'ms_per_batch': ms_e2e,
                                              'h2d_bytes_per_batch': hb[0].input_bytes(), 'd2h_bytes_per_batch': nbytes // reps},
                                      'e2e_compact': {'value': world * Bs / (ms_e2ec / 1e3), 'ms_per_batch': ms_e2ec,
                                                      'h2d_bytes_per_batch': hc[0].input_bytes()},
                                      'candidate_columns': hb[0].x_target.shape[1] - trims[0]}
            if Bs == 80:
                # roofline of the scoring leg: its dominant kernel (one launch per model and batch at batch 80), timed by the library's
                # CUDA events, against the algorithmic FLOPs of the pair products of that batch
                ks = timed_kernels(lib, lambda i: score(db[i % 2], trims[i % 2], False), 4)
                keep = hb[0].x_target.shape[1] - trims[0]
                pairs = 0.5 * sum(Bs * (b.x_target.shape[1] - t) * 200 for b, t in zip(hb, trims))     # mean of the two batches
                if 'attention_forward' in ks:
                    per_launch_ms = ks['attention_forward']['ms'] / len(ens)
                    ach = 2 * 2.0 * pairs * D * D / (per_launch_ms / 1e3) / 1e12
                    scoring['roofline'] = {'kernel': 'attention_forward (batch 80, per model)', 'bound': 'tensor', 'achieved': ach, 'peak': pk['tensor'],
                                           'unit': 'TFLOP/s', 'frac': ach / pk['tensor'], 'launch_ms': per_launch_ms, 'traffic': None,
                                           'algorithmic_flops_per_launch': 2 * 2.0 * pairs * D * D,
                                           'kernels_ms_per_batch': {k: round(v['ms'], 4) for k, v in ks.items()}}
                if world == 1 and rank == 0 and not args.no_cpu_baseline:
                    scoring['cpu_baseline'] = scoring_cpu_baseline(hb[0], args.user_num)
        model.train()

    # ---- E. long-history stress (BASELINE configs[4]): B = 4096 impressions, H = 256 with variable length (zero-padded rows, as the
    #         ETL pads), C = 5; one resident batch: training step (FusedTrainStep, CUDA-graph replay) and eval forward; roofline of
    #         its dominant kernel.  0.67 GB of float64 inputs per batch: resident only.
    long_history = None
    if not args.no_long_history:
        Bl, Hl, Cl = 4096, 256, 5
        hbl = make_batch(Bl, Hl, Cl, seed=555 + rank, user_num=args.user_num, variable_history=True)
        dbl = hbl.to(dev)
        trl = nrm.FusedTrainStep(model, Bl, Hl, Cl, lr=1e-3, weight_decay=1e-5, nslots=1, use_graph=not args.no_graph)
        sl = trl.load(hbl)
        torch.cuda.synchronize()
        for i in range(3):
            trl.run(sl)
        barrier()
        nl = 5
        e0.record()
        for i in range(nl):
            trl.run(sl)
        e1.record()
        barrier()
        ms_l = max_over_ranks(e0.elapsed_time(e1)) / nl
        model.eval()
        with torch.no_grad():
            for i in range(2):
                model(dbl.x_history, dbl.x_target, dbl.x_global)
            barrier()
            e0.record()
            for i in range(nl):
                model(dbl.x_history, dbl.x_target, dbl.x_global)
            e1.record()
            barrier()
        ms_le = max_over_ranks(e0.elapsed_time(e1)) / nl
        model.train()

        def lstep(i):
            out = model(dbl.x_history, dbl.x_target, dbl.x_global)
            model.loss(dbl.user_id, out, dbl.label).backward()
            model.zero_grad(set_to_none=True)
        lstep(0)
        kl = timed_kernels(lib, lstep, 3)
        wl = algorithmic_work(Bl, Hl, Cl, total_params)
        long_history = {'workload': f'B={Bl}/GPU, H={Hl} (variable length, zero-padded rows), C={Cl}, user_num={args.user_num}',
                        'train': {'value': world * Bl / (ms_l / 1e3), 'unit': 'impressions/s', 'ms_per_step': ms_l},
                        'eval_forward': {'value': world * Bl / (ms_le / 1e3), 'unit': 'impressions/s', 'ms_per_batch': ms_le},
                        'roofline': pick_roofline(kl, wl, pk, args.precision), 'roofline_fraction_by_kernel': all_fractions(kl, wl, pk),
                        'kernels_ms_per_step': {k: round(v['ms'], 4) for k, v in kl.items()},
                        'l2_policy': 'one batch: 0.67 GB of inputs > 126 MB L2'}
        del trl, sl, dbl, hbl
        torch.cuda.empty_cache()

    # ---- F. large user table (SURVEY 8d / 8e: user_num = 2 000 000 -> delta holds 8 MB, its gradient <= B non-zeros per rank):
    #         resident FusedTrainStep; under data parallelism the sparse (user id, value) exchange against the dense one
    large_users = None
    if not args.no_large_users:
        UL = 2_000_000
        large_users = {'user_num': UL}
        hl = [make_batch(B, H, C, seed=4242 + 97 * rank + i, user_num=UL).pin() for i in range(2)]
        for label_, smin in (('sparse_delta_exchange', nrm.FusedTrainStep.SPARSE_DELTA_MIN), ('dense_delta_exchange', 1 << 40)):
            if world == 1 and label_ == 'sparse_delta_exchange':
                continue                                    # one process: nothing to exchange, the dense Adam pass is all there is
            mL = nrm.UserModel(UL)
            mL.load_state_dict(load_weights(), strict=False)
            mL.to(dev).train().set_precision(args.precision)
            if world > 1:
                DataParallel(mL, sync_bn=args.sync_bn)
            old_min = nrm.FusedTrainStep.SPARSE_DELTA_MIN
            nrm.FusedTrainStep.SPARSE_DELTA_MIN = smin
            try:
                trL = nrm.FusedTrainStep(mL, B, H, C, lr=1e-3, weight_decay=1e-5, nslots=2, use_graph=not args.no_graph)
            finally:
                nrm.FusedTrainStep.SPARSE_DELTA_MIN = old_min
            sL = [trL.load(b) for b in hl]
            torch.cuda.synchronize()
            for i in range(4):
                trL.run(sL[i % 2])
            barrier()
            e0.record()
            for i in range(10):
                trL.run(sL[i % 2])
            e1.record()
            barrier()
            msL = max_over_ranks(e0.elapsed_time(e1)) / 10
            large_users[label_ if world > 1 else 'single_process'] = {'value': world * B / (msL / 1e3), 'ms_per_step': msL,
                                                                      'sparse': bool(trL.sparse_delta)}
            del trL, sL, mL
        torch.cuda.empty_cache()

    # short resident runs of the other precisions (same step, same data), for context
    variants = {}
    if not args.no_variants:
        for prec in ('fp32', 'bf16', 'bf16x3'):
            if prec == args.precision:
                continue
            model.set_precision(prec)
            trv = nrm.FusedTrainStep(model, B, H, C, lr=1e-3, weight_decay=1e-5, nslots=N_POOL, use_graph=not args.no_graph)
            sl = [trv.load(hb) for hb in host]
            torch.cuda.synchronize()
            for i in range(N_POOL):
                trv.run(sl[i % N_POOL])
            barrier()
            e0.record()
            for i in range(10):
                trv.run(sl[i % N_POOL])
            e1.record()
            barrier()
            msv = max_over_ranks(e0.elapsed_time(e1))
            variants[prec] = {'value': world * B * 10 / (msv / 1e3), 'ms_per_step': msv / 10}
            del trv, sl
        model.set_precision(args.precision)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rate, ms, cores, kind = cpu_reference_rate(args, args.cpu_steps, 2)
        cpu = {'value': rate, 'unit': 'impressions/s', 'cores': cores, 'kind': kind, 'ms_per_step': ms,
               'sample': _cpu_sample_text(kind, args.cpu_steps, 2, B)}
    line = {
        'metric': 'train_impressions_per_sec', 'value': value, 'unit': 'impressions/s', 'n_gpus': world, 'steps': K,
        'warmup': W, 'ms_per_step': ms_total / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': {'fp32': 'f32', 'bf16x3': 'f32 (pair products as 3 x bf16 tcgen05 MMAs, fp32 accumulate; meets the fp32 tolerances)', 'bf16': 'bf16'}[args.precision],
        'data': 'synthetic', 'config': workload_config(args, world),
        'clocks': clk.summary(),
        'e2e': {'value': e2e_value, 'unit': 'impressions/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                'ms_per_step': e2e_ms / K, 'h2d_only_ms_per_step': h2d_ms,
                'host_cpu_binding': (f'{len(cpus)} cores local to the GPU (NVML affinity)' if cpus else 'none')},
        'e2e_compact': e2ec,
        'gpu_launches': int(launches) * K, 'gpu_launches_per_step': int(launches),
        'module_path': {'value': world * B * K / (mod_ms / 1e3), 'unit': 'impressions/s', 'ms_per_step': mod_ms / K,
                        'note': 'drop-in nn.Module path driven like train.py:69-75 (autograd + FusedAdam), device-resident'},
        'api': 'FusedTrainStep (CUDA-graph replay of the 5 C-ABI calls)' if not args.no_graph else 'FusedTrainStep (eager C-ABI calls)',
        'dp_transport': (None if world == 1 else ('peer memory: gradient average fused into the Adam kernel over NVLink (one CUDA graph per step)'
                                                  if tr.peer is not None else f'NCCL all-reduce between two graphs ({model._dp.peer_error})')),
        'roofline': roofline, 'roofline_fraction_by_kernel': roofline_all, 'side_stream_groups': sorted(SIDE_STREAM_GROUPS),
        'kernels_ms_per_step': {k: round(v['ms'], 4) for k, v in kern.items()},
        'e2e_loader': loader_leg, 'long_history': long_history, 'large_user_table': large_users,
        'cpu_baseline': cpu, 'precision_variants': variants, 'scoring': scoring, 'dp_parity': dp_parity,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit('bench.py --impl ours needs a CUDA device (there is no CPU fallback)')
        run_ours(args)


if __name__ == '__main__':
    main()
