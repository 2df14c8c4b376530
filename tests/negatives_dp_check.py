"""torchrun check of pool negatives under data parallelism (tests/test_gpu_negatives_dp.py launches it on >= 2 GPUs).

Every rank trains FusedTrainStep(negatives=...) with DataParallel(sync_bn=True) on its shard of B impressions for three steps.
The negatives a rank draws must be bit-identical to rows [rank * B, (rank + 1) * B) of what one process on the whole N * B
batch draws, the replicas must stay bit-identical, and the weights must follow the single process within the fp32 tolerances
of tests/dp_check.py (a synchronised BatchNorm sums its statistics in another order)."""
import os
import sys

import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import news_recommendation_model_b200 as nrm          # noqa: E402
from news_recommendation_model_b200 import negatives, wire   # noqa: E402
from news_recommendation_model_b200.dp import DataParallel   # noqa: E402
from fixtures import load_weights                      # noqa: E402
from dp_check import _same_on_all_ranks                # noqa: E402
import parity as P                                     # noqa: E402


def run_check(dev, rank: int, world: int):
    B, H, C0, K, U = 64, 50, 5, 4, 100
    table = wire.make_article_table(3000, seed=5).to(dev)
    full = [wire.make_compact_batch(table, B * world, H, C0, seed=90 + i, user_num=U, variable_history=True).to(dev) for i in range(3)]
    shard = [wire.CompactBatch(*[getattr(cb, f)[rank * B:(rank + 1) * B].contiguous() for f in cb.__dataclass_fields__]) for cb in full]
    sampler = negatives.NegativeSampler(table, k=K, seed=77)

    def fresh():
        m = nrm.UserModel(U)
        m.load_state_dict(load_weights('train'), strict=False)
        return m.to(dev).train().set_precision('bf16x3')
    rep, ok = {}, True
    md = fresh()
    DataParallel(md, sync_bn=True)
    td = nrm.FusedTrainStep(md, B, H, C0 + K, lr=1e-3, weight_decay=1e-5, articles=table, negatives=sampler, nslots=1)
    m1 = fresh()
    t1 = nrm.FusedTrainStep(m1, B * world, H, C0 + K, lr=1e-3, weight_decay=1e-5, articles=table, negatives=sampler, nslots=1)
    same_draws = True
    for cb, cbs in zip(full, shard):
        td.step(cbs).item()
        t1.step(cb).item()
        torch.cuda.synchronize()
        mine = td.slots[0].compact.cand_article[:, C0:]
        same_draws = same_draws and torch.equal(mine, t1.slots[0].compact.cand_article[rank * B:(rank + 1) * B, C0:])
    flag = torch.tensor([1.0 if same_draws else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    rep['draws_equal_single_process_rows'] = bool(flag.item() == 1.0)
    rep['replicas_identical'] = _same_on_all_ranks(md.flat_parameters().buf)
    ok = rep['draws_equal_single_process_rows'] and rep['replicas_identical']
    a, b = md.flat_parameters(), m1.flat_parameters()
    ref = {name: b.buf[off:off + n].detach().cpu() for name, off, n, _ in b.slots}
    got = [(name, a.buf[off:off + n].detach().cpu()) for name, off, n, _ in a.slots]
    try:
        P.assert_weights_follow(got, ref, 3)
        rep['weights_follow_single_process'] = 'ok'
    except AssertionError as ex:
        rep['weights_follow_single_process'] = f'FAILED {ex}'
        ok = False
    return ok, rep


def main():
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    ok, rep = run_check(dev, rank, world)
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = bool(flag.item() == 1.0)
    if rank == 0:
        print(f'negatives_dp_check world={world}: {rep} -> {"OK" if ok else "FAILED"}', flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == '__main__':
    main()
