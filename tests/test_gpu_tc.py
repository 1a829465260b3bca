"""tcgen05 convolution kernels (fprop / dgrad / wgrad) against fp32 torch on bf16-rounded operands."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SHAPES = [  # cin, cout, k, h, w, n, up
    (16, 16, 3, 16, 8, 1, 0), (16, 16, 3, 32, 32, 2, 0), (32, 16, 1, 16, 16, 2, 0), (16, 32, 3, 12, 20, 3, 0),
    (64, 64, 3, 8, 8, 2, 0), (128, 128, 3, 16, 16, 2, 0), (256, 256, 3, 8, 8, 1, 0), (128, 64, 1, 8, 8, 2, 0),
    (64, 32, 3, 16, 16, 2, 1), (32, 32, 3, 4, 4, 3, 0), (256, 128, 3, 16, 16, 1, 0),
    (3, 16, 3, 32, 24, 2, 0), (16, 3, 1, 16, 16, 2, 0), (3, 32, 1, 16, 16, 2, 0), (32, 3, 3, 20, 12, 1, 0),
    # layers of the '256' / '512' configs (BASELINE configs 4 and 5): 256-channel 1x1 projections and 3x3 convs
    (256, 128, 1, 16, 16, 2, 0), (128, 256, 1, 16, 16, 2, 0), (128, 256, 3, 16, 16, 1, 0), (256, 256, 3, 16, 16, 2, 1),
    (256, 256, 1, 8, 8, 2, 0), (8, 8, 3, 32, 32, 1, 0), (16, 8, 3, 32, 32, 2, 1), (16, 8, 1, 32, 32, 2, 0),
    # full-width rows of the headline layers (config '128': 128x128 and 64x64 feature maps) through the DEFAULT
    # TMA-fed fprop / dgrad / wgrad kernels, several images so that CTAs loop over more than one tile
    (16, 16, 3, 128, 128, 3, 0), (3, 16, 3, 128, 128, 2, 0), (16, 3, 1, 128, 128, 2, 0), (32, 16, 3, 128, 128, 2, 1),
    (32, 32, 3, 64, 64, 3, 0), (16, 32, 3, 64, 64, 2, 0), (64, 32, 3, 64, 64, 2, 1), (32, 16, 1, 128, 128, 1, 0),
    (64, 64, 3, 32, 32, 3, 0), (32, 64, 3, 32, 32, 2, 0), (16, 32, 1, 32, 32, 2, 0), (64, 32, 3, 40, 24, 2, 0),
]


def _rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-6)), float((a - b).abs().max() / b.abs().max().clamp_min(1e-6))


@pytest.mark.parametrize('cin,cout,k,h,w,n,up', SHAPES)
def test_tc_conv(cin, cout, k, h, w, n, up):
    import tartangan_b200 as tb
    from tartangan_b200 import ops
    tb.set_precision('bf16')
    assert ops.state.use_tc
    torch.manual_seed(cin * 7 + cout + k + h)
    r = lambda t: t.bfloat16().float()
    x = r(torch.randn(n, cin, h >> up, w >> up))
    wt = r(torch.randn(cout, cin, k, k) / math.sqrt(cin * k * k))
    b = torch.randn(cout)
    xu = F.interpolate(x, scale_factor=2, mode='nearest') if up else x
    xu = xu.clone().requires_grad_()
    wr = wt.clone().requires_grad_()
    y = F.conv2d(xu, wr, b, padding=k // 2)
    gy = r(torch.randn_like(y))
    gx, gw = torch.autograd.grad(y, (xu, wr), gy)
    if up:
        gx = F.avg_pool2d(gx, 2) * 4

    xd = ops.to_internal(x.cuda()).requires_grad_()
    wd = wt.cuda().requires_grad_()
    bd = b.cuda()
    yd = ops.conv2d(xd, wd, bd, up)
    l2, mx = _rel(yd, y)
    assert l2 < 6e-3 and mx < 2e-2, ('fprop', l2, mx)
    gxd, gwd = torch.autograd.grad(yd, (xd, wd), ops.to_internal(gy.cuda()))
    l2, mx = _rel(gxd, gx)
    assert l2 < 6e-3 and mx < 2e-2, ('dgrad', l2, mx)
    l2, mx = _rel(gwd, gw)
    assert l2 < 6e-3 and mx < 2e-2, ('wgrad', l2, mx)
