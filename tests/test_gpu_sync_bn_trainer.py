"""Synchronised BatchNorm at the trainer level on one GPU.

* --sync-bn on a single process is accepted and changes nothing: losses, parameter gradients and parameters are bitwise
  those of the default in fp32 mode, eager and CUDA graph, with the same kernel count per step.
* The synchronised code path of ops.py, forced on with a one-rank NCCL group: reduce -> all-reduce -> apply with
  count = M and param_scale = 1 computes exactly what the combined entry points compute, so an fp32 step is bitwise
  that of the default path."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _trainer(sync_bn, graph, config='32', b=4):
    from tartangan_b200.trainers.cnn import CNNTrainer
    from tartangan_b200.trainers.gan import make_trainer
    torch.manual_seed(0)
    return make_trainer(CNNTrainer, config=config, batch_size=b, precision='fp32', cuda_graph=graph, sync_bn=sync_bn)


def _run(t, steps=2, force_group=None):
    from tartangan_b200 import _lib, ops
    from oracle import tartan_oracle as O
    if force_group is not None:
        ops.state.bn_group, t.sync_bn = force_group, True
    out = []
    try:
        for step in range(steps):
            imgs = O.tartan_batch(100 + step, t.args.batch_size, 32)
            torch.manual_seed(500 + step)
            k0 = _lib.Counters.kernels
            losses = t.train_batch(imgs)
            torch.cuda.synchronize()
            out.append(dict(losses=losses, kernels=_lib.Counters.kernels - k0,
                            grads=[o._ensure_flat().grad.clone() for o in (t.optimizer_d, t.optimizer_g)],
                            params=[p.detach().clone() for p in list(t.d.parameters()) + list(t.g.parameters())],
                            buffers=[v.clone() for m in (t.g, t.d) for k, v in m.state_dict().items() if 'running' in k]))
    finally:
        if force_group is not None:
            ops.state.bn_group = None
    return out


def _assert_same(a, b):
    for sa, sb in zip(a, b):
        assert sa['losses'] == sb['losses']
        assert sa['kernels'] == sb['kernels']
        for key in ('grads', 'params', 'buffers'):
            for x, y in zip(sa[key], sb[key]):
                assert torch.equal(x, y), key


@pytest.mark.parametrize('graph', [False, True])
def test_sync_bn_on_one_process_changes_nothing(graph):
    from tartangan_b200 import ops
    ref = _run(_trainer(False, graph))
    t = _trainer(True, graph)
    assert t.sync_bn is False and ops.state.bn_group is None
    _assert_same(_run(t), ref)


def test_sync_path_with_one_rank_is_bitwise_the_local_path(tmp_path):
    import torch.distributed as dist
    from tartangan_b200 import _lib
    ref = _run(_trainer(False, False))
    dist.init_process_group('nccl', init_method=f'file://{tmp_path}/store', rank=0, world_size=1,
                            device_id=torch.device('cuda', torch.cuda.current_device()))
    try:
        t = _trainer(False, False)
        calls = {}
        real_call = _lib.call

        def counting(name, *args):
            calls[name] = calls.get(name, 0) + 1
            return real_call(name, *args)
        from tartangan_b200 import ops
        ops.call = counting
        try:
            got = _run(t, force_group=dist.group.WORLD)
        finally:
            ops.call = real_call
    finally:
        dist.destroy_process_group()
    for name in ('ttg_bn_act_fwd_stats_n', 'ttg_bn_act_bwd_reduce', 'ttg_bn_act_bwd_apply', 'ttg_bn_act_bwd2_reduce',
                 'ttg_bn_act_bwd2_apply'):
        assert calls.get(name, 0) > 0, (name, calls)
    for name in ('ttg_bn_act_fwd_stats', 'ttg_bn_act_bwd', 'ttg_bn_act_bwd_acc', 'ttg_bn_act_bwd2_acc'):
        assert calls.get(name, 0) == 0, (name, calls)
    for sa, sb in zip(got, ref):
        sa['kernels'] = sb['kernels']             # (the split entry points are counted per call)
    _assert_same(got, ref)
