"""GPU parity of the round-1 fast paths that the small-shape operator tests do not reach:

* bulk-copy (TMA 1-D) pipelined channel kernels  -> tensors above the size threshold (chanops.cuh: cb_ok)
* streaming conv kernel with compile-time channel counts (128 -> 128, 128 -> 64, 64 -> 128) and wgrad at those sizes
* conv epilogue / residual-join BatchNorm statistics (ttg_conv2d_tc_stats, ttg_*_stats, ttg_bn_finalize)
* 8-channel staging of the RGB layers (ttg_pad_channels8 / ttg_unpad_channels8)
* all filters of a model packed in one launch (ttg_pack_weights_multi)

Oracle: the same op in PyTorch fp32 on the CPU (operands rounded to bf16 where the kernel rounds them).
Tolerances: bf16 outputs 2e-2 relative L2; fp32 reductions 2e-3 relative.
"""
import math

import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def rel_l2(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-6))


def _internal(x):
    from tartangan_b200 import ops
    return ops.to_internal(x.cuda(), BF)


@pytest.fixture(autouse=True)
def _bf16_mode():
    import tartangan_b200 as tb
    tb.set_precision('bf16')
    yield
    tb.set_precision('bf16')


# ------------------------------------------------------------------ bulk-pipelined BatchNorm kernels
@pytest.mark.parametrize('c,hw,n', [(16, 64, 16), (64, 32, 12), (128, 16, 24), (256, 8, 48)])
def test_bn_act_large_fwd_bwd_double(c, hw, n):
    """Sizes above the bulk-kernel threshold (>= 148 * 512 * 8 elements); forward, backward and double backward."""
    from tartangan_b200 import ops
    from tartangan_b200.models.layers import BatchNorm2d
    torch.manual_seed(3)
    assert n * c * hw * hw >= 8 * 512 * 148
    x = (torch.randn(n, c, hw, hw) * 1.3 + 0.2).to(BF).float().requires_grad_()
    ref = torch.nn.BatchNorm2d(c)
    with torch.no_grad():
        ref.weight.uniform_(0.5, 1.5)
        ref.bias.uniform_(-0.5, 0.5)
    bn = BatchNorm2d(c).cuda()
    bn.load_state_dict(ref.state_dict())
    y = F.leaky_relu(ref(x), 0.2)
    g = torch.randn_like(y).to(BF).float()
    gx, = torch.autograd.grad(y, x, g, create_graph=True)
    v = torch.randn_like(x).to(BF).float()
    ggx, = torch.autograd.grad((gx * v).sum(), x)

    xd = x.detach().cuda().requires_grad_()
    yd = ops.bn_act(ops.to_internal(xd, BF), bn, 0.2)
    assert rel_l2(yd, y) < 2e-2
    gxd, = torch.autograd.grad(yd, xd, _internal(g), create_graph=True)
    assert rel_l2(gxd, gx) < 2e-2
    ggxd, = torch.autograd.grad(ops.DotFn.apply(ops.to_internal(gxd, BF), _internal(v)), xd)
    assert rel_l2(ggxd, ggx) < 4e-2
    assert rel_l2(bn.running_mean, ref.running_mean) < 2e-3 and rel_l2(bn.running_var, ref.running_var) < 2e-3


def test_axpby_and_channel_sum_large():
    from tartangan_b200 import ops
    torch.manual_seed(4)
    a, b = torch.randn(8, 32, 64, 64).to(BF), torch.randn(8, 32, 64, 64).to(BF)
    out = ops.AxpbyFn.apply(_internal(a.float()), _internal(b.float()), 1.0, 0.5)
    assert rel_l2(out, a.float() + 0.5 * b.float()) < 1e-2
    s = ops.ChannelSumFn.apply(_internal(a.float()))
    want = a.float().sum(dim=(0, 2, 3))
    assert float((s.cpu() - want).abs().max() / want.abs().max()) < 2e-3


# ------------------------------------------------------------------ streaming / static conv kernels
@pytest.mark.parametrize('cin,cout,hw,n', [(128, 128, 16, 6), (128, 128, 8, 10), (128, 64, 16, 6), (64, 128, 16, 6),
                                           (64, 64, 32, 3), (32, 32, 32, 5), (16, 16, 64, 2)])
def test_conv_static_kernels(cin, cout, hw, n):
    """fprop, dgrad and wgrad at the channel counts that select the compile-time (static) kernels; more tiles than
    SMs in the persistent loops for the small-channel cases."""
    from tartangan_b200 import ops
    torch.manual_seed(5)
    x = torch.randn(n, cin, hw, hw).to(BF).float().requires_grad_()
    w = (torch.randn(cout, cin, 3, 3) / math.sqrt(cin * 9)).requires_grad_()
    b = torch.randn(cout, requires_grad=True)
    wq = w.detach().to(BF).float().requires_grad_()
    y = F.conv2d(x, wq, b, padding=1)
    gy = torch.randn_like(y).to(BF).float()
    gx, gw, gb = torch.autograd.grad(y, (x, wq, b), gy)
    xd, wd, bd = x.detach().cuda().requires_grad_(), w.detach().cuda().requires_grad_(), b.detach().cuda().requires_grad_()
    yd = ops.conv2d(ops.to_internal(xd, BF), wd, bd)
    assert rel_l2(yd, y) < 1e-2
    gxd, gwd, gbd = torch.autograd.grad(yd, (xd, wd, bd), _internal(gy))
    assert rel_l2(gxd, gx) < 1e-2 and rel_l2(gwd, gw) < 1e-2 and rel_l2(gbd, gb) < 1e-2


# ------------------------------------------------------------------ producer statistics
@pytest.mark.parametrize('cin,cout,hw,n,k', [(16, 16, 32, 4, 3), (32, 64, 20, 3, 3), (128, 128, 16, 4, 3), (64, 32, 16, 2, 1)])
def test_conv_epilogue_statistics(cin, cout, hw, n, k):
    from tartangan_b200 import ops
    torch.manual_seed(6)
    x = _internal(torch.randn(n, cin, hw, hw))
    w = (torch.randn(cout, cin, k, k) / math.sqrt(cin * k * k)).cuda()
    b = torch.randn(cout).cuda()
    assert ops.conv_stats_ok(w, 0, BF)
    y = ops.conv2d(x, w, b, stats=True)
    pending = ops.state.producer_stats
    assert pending is not None and pending[0].data_ptr() == y.data_ptr()
    sums = ops.take_producer_stats(y)
    assert sums is not None and ops.take_producer_stats(y) is None          # consumed once
    yf = y.float().cpu()
    want = torch.cat([yf.sum(dim=(0, 2, 3)), (yf * yf).sum(dim=(0, 2, 3))]).double()
    got = sums.cpu()
    assert float((got - want).abs().max() / want.abs().max()) < 1e-4       # statistics of the STORED bf16 values
    y_plain = ops.conv2d(x, w, b)
    assert torch.equal(y_plain, y)                                          # same conv, bit for bit


def test_bn_consumes_producer_statistics():
    """conv(stats) -> bn_act and join(stats) -> bn_act give the same result as the two-pass BatchNorm."""
    from tartangan_b200 import ops
    from tartangan_b200.models.layers import BatchNorm2d
    torch.manual_seed(7)
    x = _internal(torch.randn(4, 32, 16, 16))
    w = (torch.randn(32, 32, 3, 3) / 17.0).cuda()
    bn1, bn2 = BatchNorm2d(32).cuda(), BatchNorm2d(32).cuda()
    a1 = ops.bn_act(ops.conv2d(x, w, None, stats=True), bn1, 0.2)
    a2 = ops.bn_act(ops.conv2d(x, w, None), bn2, 0.2)
    assert rel_l2(a1, a2) < 1e-3 and rel_l2(bn1.running_var, bn2.running_var) < 1e-4
    h, s = _internal(torch.randn(4, 32, 16, 16)), _internal(torch.randn(4, 32, 8, 8))
    for join, args in ((ops.add_up2, (h, s)), (ops.avg_pool2_add, (h, s))):
        bn1, bn2 = BatchNorm2d(32).cuda(), BatchNorm2d(32).cuda()
        a1 = ops.bn_act(join(*args, stats=True), bn1, 0.2)
        a2 = ops.bn_act(join(*args, stats=False), bn2, 0.2)
        assert rel_l2(a1, a2) < 1e-3 and rel_l2(bn1.running_mean, bn2.running_mean) < 1e-4


def test_stale_producer_statistics_are_dropped():
    from tartangan_b200 import ops
    from tartangan_b200.models.layers import BatchNorm2d
    torch.manual_seed(8)
    x = _internal(torch.randn(2, 16, 16, 16))
    w = (torch.randn(16, 16, 3, 3) / 12.0).cuda()
    ops.conv2d(x, w, None, stats=True)                   # statistics pending for a tensor nobody normalises
    other = _internal(torch.randn(2, 16, 16, 16) * 3 + 1)
    bn = BatchNorm2d(16).cuda()
    ref = torch.nn.BatchNorm2d(16)
    got = ops.bn_act(other, bn, 0.2)
    want = F.leaky_relu(ref(other.float().cpu()), 0.2)
    assert rel_l2(got, want) < 2e-2 and ops.state.producer_stats is None


# ------------------------------------------------------------------ RGB staging, multi-pack
def test_pad_unpad_channels8_roundtrip():
    from tartangan_b200 import ops
    from tartangan_b200._lib import call, ptr
    torch.manual_seed(9)
    x = _internal(torch.randn(3, 3, 9, 7))
    x8 = ops._pad8(x)
    assert x8.shape == (3, 8, 9, 7) and torch.equal(x8[:, :3], x) and float(x8[:, 3:].abs().max()) == 0.0
    back = ops.empty_nhwc(3, 3, 9, 7, BF, 'cuda')
    call('ttg_unpad_channels8', ptr(x8), ptr(back), 3 * 9 * 7, 3)
    assert torch.equal(back, x)


def test_pack_weights_multi_matches_single_pack():
    from tartangan_b200 import ops
    from tartangan_b200.optim import FlatParams
    torch.manual_seed(10)
    shapes = [(16, 3, 3, 3), (32, 16, 3, 3), (32, 16, 1, 1), (3, 16, 1, 1), (64, 64, 3, 3)]
    params = [torch.nn.Parameter(torch.randn(*s, device='cuda')) for s in shapes] + \
             [torch.nn.Parameter(torch.randn(7, device='cuda'))]
    singles = {(i, m): ops._packed(p, m, 'tc').clone() for i, p in enumerate(params[:-1]) for m in (0, 1)}
    flat = FlatParams(params)
    pm = ops.PackedModel(flat)
    pm.repack()
    for i, p in enumerate(params[:-1]):
        for m in (0, 1):
            assert torch.equal(ops._packed(p, m, 'tc'), singles[(i, m)]), (i, m)


def test_device_image_stack_matches_host_pipeline(tmp_path):
    """SURVEY 8 f-3: uint8 stack in HBM, crop + normalise in one kernel == the host pipeline of NpzImageDataset
    (image_bytes_dataset.py:44-49: crop, ToTensor, Normalize(0.5, 0.5)) bit for bit in fp32; ragged crop origins,
    the last row / column of the image included; and one trainer epoch over an .npz runs through it."""
    import numpy as np
    import tartangan_b200 as tb
    from tartangan_b200 import ops
    from tartangan_b200.trainers.trainer import DeviceImageStack
    rng = np.random.RandomState(0)
    imgs = rng.randint(0, 256, size=(7, 40, 52, 3), dtype=np.uint8)
    ds = DeviceImageStack(imgs, 32, 'cuda', seed=3)
    index = torch.tensor([6, 0, 3, 3, 5]); oy = torch.tensor([8, 0, 3, 8, 1]); ox = torch.tensor([20, 0, 7, 19, 20])
    got = ds.crop(index, oy, ox)
    ref = torch.stack([torch.from_numpy(np.ascontiguousarray(imgs[i, y:y + 32, x:x + 32])).permute(2, 0, 1).float() / 127.5 - 1.0
                       for i, y, x in zip(index.tolist(), oy.tolist(), ox.tolist())])
    assert got.shape == (5, 3, 32, 32) and got.dtype == torch.float32
    assert torch.equal(got.cpu(), ref)                            # same IEEE operations as the host pipeline
    tb.set_precision('bf16')
    internal = ds.crop(index, oy, ox, internal=True)
    assert torch.equal(ops.from_internal(internal).cpu(), ref.bfloat16().float()) or \
        float((ops.from_internal(internal).cpu() - ref).abs().max()) < 8e-3
    batches = list(ds.epoch(3))
    assert len(batches) == 2 and all(b.shape == (3, 3, 32, 32) for b in batches)      # drop_last
    assert all(float(b.min()) >= -1.0 and float(b.max()) <= 1.0 for b in batches)
    # end to end: the trainer loop over an .npz with --device-dataset
    from tartangan_b200.trainers.iqn import IQNTrainer
    from tartangan_b200.trainers.gan import make_trainer
    np.savez(tmp_path / 'imgs.npz', images=rng.randint(0, 256, size=(9, 36, 36, 3), dtype=np.uint8))
    torch.manual_seed(0)
    t = make_trainer(IQNTrainer, config='32', batch_size=4, model_scale=0.25, output=str(tmp_path), device_dataset=True,
                     quiet_logs=True, epochs=1)
    t.args.data_path = str(tmp_path / 'imgs.npz')
    logs = t.train(max_steps=2)
    assert len(logs['d_loss']) == 2 and all(v == v for v in logs['d_loss'])
    # f-2: the progress sampler (image_sampler.py) rendered target_g / g samples and the slerp grid at step 0 and at the end
    samples = sorted(os.listdir(os.path.join(t.output_root, 'samples')))
    assert samples == ['grid_sample_0.png', 'grid_sample_2.png', 'sample_0.png', 'sample_2.png'], samples
    imgs, grid = t.sampler.render()
    assert imgs.shape == (32, 3, 32, 32) and grid.shape == (25, 3, 32, 32) and float(imgs.abs().max()) <= 1.0
    g = t.sampler._latent_grid_samples.cpu()
    assert torch.allclose(g[0], g[0]) and g.shape == (25, t.gan_config.latent_dims)
    n = g.norm(dim=1)                           # slerp between (almost) equal-norm gaussians keeps the norm in their range
    assert float(n.min()) > 0.5 * float(n.max())


def test_generator_head_fused_kernel():
    """ops.RgbHeadFn (ttg_rgb_head_fwd / _bwd): tanh(conv1x1(a) + b) -> fp32 NCHW and its three gradients against torch
    on the bf16-rounded input, at the three supported widths; the trainer-level path is covered by the parity tests."""
    from tartangan_b200 import ops
    import tartangan_b200 as tb
    tb.set_precision('bf16')
    torch.manual_seed(11)
    for cin, n, hw in ((16, 3, 24), (8, 2, 16), (32, 2, 12)):
        a = (torch.randn(n, cin, hw, hw) * 0.7).bfloat16().float()
        w = (torch.randn(3, cin, 1, 1) / math.sqrt(cin)).requires_grad_()
        b = (torch.randn(3) * 0.1).requires_grad_()
        ar = a.clone().requires_grad_()
        y = torch.tanh(F.conv2d(ar, w, b))
        g = torch.randn_like(y)
        ga, gw, gb = torch.autograd.grad(y, (ar, w, b), g)
        ad = ops.to_internal(a.cuda()).requires_grad_()
        wd, bd = w.detach().cuda().requires_grad_(), b.detach().cuda().requires_grad_()
        yd = ops.RgbHeadFn.apply(ad, wd, bd)
        assert yd.dtype == torch.float32 and yd.is_contiguous() and yd.shape == y.shape
        assert float((yd.cpu() - y).abs().max()) < 2e-5
        gad, gwd, gbd = torch.autograd.grad(yd, (ad, wd, bd), g.cuda())
        assert rel_l2(gad.float().cpu(), ga) < 1e-2           # bf16 output
        assert rel_l2(gwd.cpu(), gw) < 2e-4 and rel_l2(gbd.cpu(), gb) < 2e-4
