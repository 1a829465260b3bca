"""Worker of tests/test_gpu_sync_bn_dist.py (run under `python -m torch.distributed.run --nproc-per-node 2`).

Synchronised BatchNorm end to end: every rank trains the CNN trainer (config '32') on its shard of b images with
--sync-bn, and rank 0 replays the step on the CPU oracle at the UNSHARDED global batch of world * b images, whose z draws
are each rank's z draws concatenated in rank order.  With BatchNorm statistics over the global batch, the data-parallel
step is that single step: the mean of the ranks' losses, the averaged gradients and the BatchNorm running statistics
must match it.  Also checked: the running statistics are bitwise equal across ranks, and so are the parameters after
two steps.

argv: precision (fp32 | bf16), mode (eager | graph), [control]: `control` trains WITHOUT --sync-bn and requires the
running statistics to miss the global-batch oracle, which shows that the comparison can tell the two apart.
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _cos(a, b):
    a, b = a.detach().float().cpu().flatten(), b.detach().float().cpu().flatten()
    return float(torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-30))


def _bn_buffers(t):
    out = {}
    for net, mod in (('g', t.g), ('d', t.d)):
        for k, v in mod.state_dict().items():
            if k.endswith('running_mean') or k.endswith('running_var'):
                out[f'{net}.{k}'] = v.detach().float()
    return out


def _oracle_step(O, orc, shards, seeds, b):
    """One oracle step at the global batch; z of the D and the G step = the ranks' draws concatenated."""
    zs = [[], []]
    for s in seeds:
        torch.manual_seed(s)
        for i in range(2):                        # the trainer draws z(D step) then z(G step) from the CPU generator
            zs[i].append(torch.randn(b, orc.spec.latent_dims))
    queue = [torch.cat(z) for z in zs]
    orc._fake = lambda n: O.generator(orc.g, orc.spec, queue.pop(0), orc.norm, orc.g_base)
    out = orc.train_batch(torch.cat(shards))
    assert not queue
    return out


def main():
    precision, graph = sys.argv[1], sys.argv[2] == 'graph'
    control = len(sys.argv) > 3 and sys.argv[3] == 'control'
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', rank)))
    dist.init_process_group('nccl', device_id=torch.device('cuda', torch.cuda.current_device()))
    from oracle import tartan_oracle as O
    from tartangan_b200 import ops
    from tartangan_b200.trainers.cnn import CNNTrainer
    from tartangan_b200.trainers.gan import make_trainer
    config, b = '32', 4
    torch.manual_seed(0)
    t = make_trainer(CNNTrainer, config=config, batch_size=b, precision=precision, cuda_graph=graph,
                     sync_bn=not control)
    assert t.sync_bn == (not control) and (ops.state.bn_group is not None) == (not control)
    cpu = lambda m: {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    orc = O.OracleTrainer('cnn', O.SPECS[config], cpu(t.g), cpu(t.target_g), cpu(t.d), world * b) if rank == 0 else None
    tol_loss, tol_cos, tol_bn = (3e-3, 0.9995, 1e-3) if precision == 'fp32' else (5e-2, 0.97, 1e-1)
    ok = True
    for step in range(2):
        shards = [O.tartan_batch(100 + step * world + r, b, 32) for r in range(world)]
        seeds = [500 + step * world + r for r in range(world)]
        torch.manual_seed(seeds[rank])
        got = t.train_batch(shards[rank])
        torch.cuda.synchronize()
        mine = torch.tensor([got['d_loss'], got['gp'], got['g_loss']], device='cuda')
        dist.all_reduce(mine)
        mine /= world
        bufs = _bn_buffers(t)
        flat = torch.cat([v.reshape(-1) for v in bufs.values()])
        ref = flat.clone()
        dist.broadcast(ref, 0)
        same = torch.tensor([float(torch.equal(flat, ref))], device='cuda')
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        if rank == 0:
            want = _oracle_step(O, orc, shards, seeds, b)
            if step == 0 and not control:
                tol = tol_loss
                for i, name in enumerate(('d_loss', 'gp', 'g_loss')):
                    val, r = float(mine[i]), want[name]
                    if abs(val - r) > tol * max(1.0, abs(r)):
                        print(f'MISMATCH step {step} {name}: mean over ranks {val} vs global-batch oracle {r}'); ok = False
                for net, mod in (('d', t.d), ('g', t.g)):
                    params = dict(mod.named_parameters())
                    ref_g = orc.last_grads[net]
                    scale = max(float(v.abs().max()) for v in ref_g.values())
                    worst = 1.0
                    for k, v in ref_g.items():
                        if k.endswith('.bias') and float(v.abs().max()) < max(2e-3 * scale, 5e-5):
                            continue                      # analytically zero gradients (bias before BatchNorm)
                        c = _cos(params[k].grad, v)
                        worst = min(worst, c)
                        if not c >= (tol_cos if v.numel() >= 64 else tol_cos - 0.07):
                            print(f'MISMATCH averaged gradient {net}.{k}: cosine {c:.5f}'); ok = False
                    print(f'[sync bn] {precision} {"graph" if graph else "eager"}: {net} averaged gradients, '
                          f'worst cosine {worst:.5f}')
            if float(same) != 1.0 and not control:
                print(f'MISMATCH step {step}: BatchNorm running statistics differ across ranks'); ok = False
            if step == 0:
                oref = {f'{net}.{k}': v for net, sd in (('g', orc.g), ('d', orc.d)) for k, v in sd.items()
                        if k.endswith('running_mean') or k.endswith('running_var')}
                assert set(oref) == set(bufs), sorted(set(oref) ^ set(bufs))
                worst, where = 0.0, None
                for k, v in bufs.items():
                    e = float((v.cpu() - oref[k]).abs().max() / oref[k].abs().max().clamp_min(1e-6))
                    if e > worst:
                        worst, where = e, k
                print(f'[sync bn] {precision} {"graph" if graph else "eager"}{" control" if control else ""}: '
                      f'running statistics vs global-batch oracle, worst relative error {worst:.3g} ({where}), '
                      f'bar {tol_bn:g}')
                if control and not worst > 10 * tol_bn:
                    print(f'MISMATCH control: local statistics come within {worst:.3g} of the global-batch oracle'); ok = False
                if not control and not worst <= tol_bn:
                    print('MISMATCH running statistics vs global-batch oracle'); ok = False
    flat = torch.cat([p.detach().reshape(-1) for p in list(t.d.parameters()) + list(t.g.parameters())])
    ref = flat.clone()
    dist.broadcast(ref, 0)
    same = torch.tensor([float(torch.equal(flat, ref))], device='cuda')
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    if rank == 0:
        if float(same) != 1.0:
            print('MISMATCH: ranks hold different parameters after the steps'); ok = False
        print('SYNC_BN_OK' if ok else 'SYNC_BN_FAILED', flush=True)
    dist.barrier()
    from tartangan_b200.parallel import shutdown
    clean = shutdown([t])
    if rank == 0:
        print('clean NCCL shutdown' if clean else 'NCCL shutdown timed out (process exits anyway)', flush=True)
    sys.stdout.flush()
    os._exit(0)


if __name__ == '__main__':
    main()
