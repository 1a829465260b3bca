"""Cost of synchronised BatchNorm (--sync-bn): images/s of the data-parallel IQN training step with and without it.

    python -m torch.distributed.run --nproc-per-node N tools/bench_sync_bn.py [--batch 256] [--rounds 3]

Strong scaling like `bench.py --strong`: a global batch of --batch images, --batch / N per rank, config '128', bf16,
CUDA graphs, inputs resident in HBM.  Two trainers are built from the same seed, one per arm, and timed alternately
(--rounds times each, --steps steps per timing) so that both see the same machine state.  Also counts, on the host, the
BatchNorm all-reduces one training step issues (during the graph capture of the synchronised arm).  Prints the card name
and power limit, then one JSON line.  Needs at least 2 GPUs: on one process --sync-bn does nothing.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _card(index):
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', str(index)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ''
    return out or torch.cuda.get_device_name(index)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=256, help='global batch')
    ap.add_argument('--config', default='128')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    args = ap.parse_args()
    rank, local, world = (int(os.environ.get(k, d)) for k, d in (('RANK', 0), ('LOCAL_RANK', 0), ('WORLD_SIZE', 1)))
    if world < 2:
        raise SystemExit('bench_sync_bn: run it under torch.distributed.run with at least 2 processes')
    if args.batch % world:
        raise SystemExit(f'bench_sync_bn: global batch {args.batch} is not divisible by {world} ranks')
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from tartangan_b200 import ops
    from tartangan_b200.parallel import shutdown
    from tartangan_b200.trainers.gan import make_trainer
    from tartangan_b200.trainers.iqn import IQNTrainer
    from tartangan_b200.trainers.trainer import tartan_batch
    b = args.batch // world
    arms = {}
    for sync in (False, True):
        torch.manual_seed(0)
        arms[sync] = make_trainer(IQNTrainer, config=args.config, batch_size=b, cuda_graph=True, sync_bn=sync)
    imgs = tartan_batch(1234 + rank, b, arms[False].g.max_size).cuda()
    # graph capture happens at the first step of each arm, with ops.state.bn_group as that arm needs it
    reduces = {'n': 0}
    real = ops._bn_all_reduce

    def counting(sums, group):
        reduces['n'] += 1
        return real(sums, group)
    torch.manual_seed(1000 + rank)
    for sync, t in arms.items():
        ops.state.bn_group = dist.group.WORLD if sync else None
        ops._bn_all_reduce = counting if sync else real
        t.train_batch(imgs, as_floats=False)
        ops._bn_all_reduce = real
        for _ in range(args.warmup):
            t.train_batch(imgs, as_floats=False)
    # the first graphed step runs two eager warm-up steps and the capture of one step (GanTrainer._capture); the
    # replays run no Python
    assert reduces['n'] % 3 == 0, reduces
    per_step = reduces['n'] // 3
    times = {False: [], True: []}
    for _ in range(args.rounds):
        for sync, t in arms.items():
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                t.train_batch(imgs, as_floats=False)
            torch.cuda.synchronize()
            dist.barrier()
            times[sync].append(time.perf_counter() - t0)
    ops.state.bn_group = None
    if rank == 0:
        rate = {s: [args.batch * args.steps / x for x in v] for s, v in times.items()}
        print(f'card: {_card(local)}', flush=True)
        print(json.dumps({'config': args.config, 'world': world, 'global_batch': args.batch,
                          'img_s_local_bn': [round(r, 1) for r in rate[False]],
                          'img_s_sync_bn': [round(r, 1) for r in rate[True]],
                          'bn_all_reduces_per_step': per_step}), flush=True)
    shutdown(list(arms.values()))
    os._exit(0)


if __name__ == '__main__':
    main()
