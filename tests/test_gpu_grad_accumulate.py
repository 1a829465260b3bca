"""In-place parameter gradients (ops.direct_param_grads) against float64 references.

Inside `ops.direct_param_grads()` the conv and BatchNorm parameter gradients are ADDED to `p.grad` (a view of the
optimiser's flat buffer) by dedicated entry points: ttg_conv2d_wgrad_tc_acc, ttg_channel_sum_acc, ttg_bn_act_bwd_acc,
ttg_bn_act_bwd2_acc and ttg_rgb_head_bwd(accumulate = 1).  Their flag bit 0 means "add", bit 1 "the workspace is
already zero" (ops.ZeroArena).  The training step reaches only these; the operator tests, which differentiate with
torch.autograd.grad, reach only the overwriting variants.

Every operator case here
  * prefills `.grad` with a random G0 on the gradient's own scale, so an add that overwrites fails;
  * records the entry points that ran and their flags, so a shape that falls back to autograd's path fails;
  * compares `p.grad - G0` (float64) with torch in float64 on the CPU, computed from the bf16 operands the kernels
    received, read back from the device (for the BatchNorm the mean / invstd it saved as well).
So the only error left is the kernels' fp32 summation; the bars are set from that, not from bf16 rounding.  One pixel
dropped out of K changes a sum by about 1/sqrt(K), 1e-2 at these sizes.

The LeakyReLU mask of the BatchNorm backward flips where the pre-activation is within rounding of zero, and which
way it flips is not part of the contract: the cotangents are zeroed there (and, for the R1 case, in the 3x3
neighbourhood the following conv spreads them over), so the reference does not depend on it.

Measured on one NVIDIA B200 at a 1000 W power limit, worst relative L2 / max error over all cases [bar]:
  conv weight (test_conv_wgrad_acc, test_conv_shared_weight)   5.6e-7 / 9.6e-7   [3e-6 / 5e-6]
  conv bias, fused into the wgrad kernel or ttg_channel_sum_acc  1.0e-6 / 1.6e-6   [5e-6 / 1e-5]
  BatchNorm gamma / beta                                         1.1e-7 / 1.4e-7   [5e-7 / 1e-6]
  generator head weight / bias                                   1.2e-7 / 1.6e-7   [5e-7 / 1e-6]
The trainer-level test compares the in-place path with autograd's AccumulateGrad path (ops._NO_DIRECT) over one
D and one G backward of the benchmarked configurations, with the learning rates at 0 so that both half-steps start
from the same weights.  Both arms run the same kernels except for the final add, so they differ by the run-to-run
spread of the fp32 atomics only, which the test measures itself (two runs of each arm).  The largest spreads are
those of the conv biases that feed a BatchNorm (analytically zero gradients); the worst difference seen was 0.31 of
its bar.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# index of the flags argument of each in-place entry point (ops.call(name, *args))
FLAG_ARG = {'ttg_conv2d_wgrad_tc_acc': 12, 'ttg_channel_sum_acc': 4, 'ttg_bn_act_bwd_acc': 12,
            'ttg_bn_act_bwd2_acc': 13, 'ttg_rgb_head_bwd': 10}
# entry points that overwrite their output: never reached under direct_param_grads()
OVERWRITING = {'ttg_conv2d_wgrad_tc_ex', 'ttg_conv2d_wgrad_bias_tc_ex', 'ttg_conv2d_wgrad_direct_det', 'ttg_channel_sum',
               'ttg_bn_act_bwd', 'ttg_bn_act_bwd2'}

# (relative L2, max |error| / max |ref|)
WGRAD_BAR = (3e-6, 5e-6)
BIAS_BAR = (5e-6, 1e-5)
BN_BAR = (5e-7, 1e-6)
RGB_BAR = (5e-7, 1e-6)


def _ops():
    import tartangan_b200 as tb
    from tartangan_b200 import ops
    tb.set_precision('bf16')
    assert ops.state.use_tc
    return ops


@pytest.fixture
def calls(monkeypatch):
    """[(entry point, args)] of every ops.call while the test runs."""
    ops = _ops()
    seen, real = [], ops.call

    def record(name, *args):
        seen.append((name, args))
        return real(name, *args)
    monkeypatch.setattr(ops, 'call', record)
    monkeypatch.setattr(ops.state, 'arena', None)
    real_ws = ops._ws
    # ordinary workspaces are torch.empty: make sure they are not zero already, so that a kernel which skips clearing
    # one shows
    monkeypatch.setattr(ops, '_ws', lambda nbytes, device: real_ws(nbytes, device).fill_(2.0 ** 20))
    return seen


@pytest.fixture(params=['memset', 'arena'])
def workspace(request, calls):
    """Flag bit 1 of the in-place entry points.  'memset': no arena, every kernel clears the (non-zero, see `calls`)
    workspace it is handed.  'arena': a ZeroArena whose earlier period and current period both wrote their slices
    before the kernels take theirs.  -> the expected flag bit."""
    ops = _ops()
    if request.param == 'memset':
        return 0
    arena = ops.ZeroArena(torch.device('cuda'), nbytes=32 << 20)
    for sizes in ((3 << 20, 4096), (1000, 777)):
        arena.reset()
        for nbytes in sizes:
            arena.take(nbytes).fill_(0x41)
    ops.state.arena = arena            # (the `calls` fixture restores None)
    return 2


def _check_calls(calls, expected, flag_bit=0):
    """Each entry point of `expected` ({name: count}) ran that often with flag bit 0 set and bit 1 == flag_bit; no
    overwriting variant ran."""
    names = [n for n, _ in calls]
    assert not OVERWRITING & set(names), names
    for name, count in expected.items():
        assert names.count(name) == count, (name, names)
    for name, args in calls:
        if name in FLAG_ARG:
            flags = args[FLAG_ARG[name]]
            assert flags & 1 and (flags & 2) == flag_bit, (name, flags)


def _dev(t):
    """float tensor -> bf16 NHWC on the device (logical NCHW)."""
    return t.to(torch.bfloat16).cuda().contiguous(memory_format=torch.channels_last)


def _host(t):
    return t.detach().double().cpu()


def _params(*tensors):
    """nn.Parameters on the device, re-homed into an optim.FlatParams with .grad attached."""
    from tartangan_b200.optim import FlatParams
    ps = [torch.nn.Parameter(t.float().cuda()) for t in tensors]
    FlatParams(ps).attach_grads()
    return ps


def _prefill(refs):
    """p.grad = G0, random on the scale of the expected gradient -> {p: G0 as float64}."""
    g0 = {}
    for p, ref in refs.items():
        p.grad.copy_(torch.randn(ref.shape, dtype=torch.float64) * float(ref.std()))
        g0[p] = _host(p.grad)
    return g0


def _err(got, ref):
    d = got - ref
    return float(d.norm() / ref.norm()), float(d.abs().max() / ref.abs().max())


def _compare(tag, g0, refs, bars, got=None):
    """got (default: the current .grad) minus G0 against refs; every error is printed before any is asserted."""
    errs = {}
    for p, ref in refs.items():
        what, bar = bars[p]
        cur = got[p] if got is not None else _host(p.grad)
        errs[what] = _err(cur - g0[p], ref), bar
        print(f'[grad-acc] {tag} {what}: rel-L2 {errs[what][0][0]:.2e}, max {errs[what][0][1]:.2e}')
    for what, ((l2, mx), (bl2, bmx)) in errs.items():
        assert l2 <= bl2 and mx <= bmx, (tag, what, l2, mx)


def _wgrad_ref(x, gy, k):
    return torch.nn.grad.conv2d_weight(_host(x), (gy.shape[1], x.shape[1], k, k), _host(gy), padding=k // 2)


# ---------------------------------------------------------------------------------------------- conv weight gradient
# Every branch of wgrad_tc_core (csrc/conv_tc.cu).  H and W are not multiples of the 16x8 tile, and each shape has
# more tiles than the kernel launches CTAs, so that CTAs loop over several tiles.
WGRAD_SHAPES = [  # cin, cout, k, n, h, w
    (16, 16, 3, 3, 100, 260),     # persistent, mfold (fuse 3)
    (64, 32, 3, 3, 69, 230),      # persistent, mfold, Cin 64
    (32, 64, 3, 3, 69, 230),      # persistent, fuse 1
    (64, 128, 3, 3, 69, 85),      # persistent, fuse 1
    (128, 128, 3, 2, 69, 85),     # persistent, fuse 0, 3x3
    (64, 128, 1, 4, 69, 230),     # persistent, fuse 0, 1x1
    (128, 256, 3, 2, 69, 85),     # persistent, halves = 2
    (64, 256, 1, 3, 69, 85),      # persistent, halves = 2, 1x1
    (256, 128, 3, 2, 53, 45),     # conv_wgrad_tc_kernel (nbuf < 2): atomics into gw, bias by ttg_channel_sum_acc
    (256, 128, 1, 4, 100, 130),   # conv_wgrad_tc_kernel, 1x1
    (256, 256, 3, 1, 37, 45),     # conv_wgrad_tc_kernel, halves = 2
    (16, 8, 3, 3, 100, 260),      # Cout 8: padded gy, bias by a separate ttg_channel_sum_acc
    (8, 16, 3, 3, 100, 260),      # Cin 8: padded x
    (16, 8, 1, 6, 69, 230),       # Cout 8, 1x1
    (8, 32, 1, 6, 69, 230),       # Cin 8, 1x1
]


@pytest.mark.parametrize('bias', [True, False], ids=['bias', 'nobias'])
@pytest.mark.parametrize('cin,cout,k,n,h,w', WGRAD_SHAPES)
def test_conv_wgrad_acc(cin, cout, k, n, h, w, bias, workspace, calls):
    ops = _ops()
    torch.manual_seed(cin * 31 + cout * 7 + k)
    x = _dev(torch.randn(n, cin, h, w))
    ps = _params(torch.randn(cout, cin, k, k) / math.sqrt(cin * k * k), torch.randn(cout))
    wt, b = ps[0], (ps[1] if bias else None)
    y = ops.conv2d(x, wt, b)
    gy = _dev(torch.randn(n, cout, h, w))
    refs = {wt: _wgrad_ref(x, gy, k)}
    if bias:
        refs[b] = _host(gy).sum((0, 2, 3))
    g0 = _prefill(refs)
    with ops.direct_param_grads():
        y.backward(gy)
    _check_calls(calls, {'ttg_conv2d_wgrad_tc_acc': 1, 'ttg_channel_sum_acc': int(bias and cout < 16)}, workspace)
    _compare(f'wgrad {cin}->{cout} k{k} {n}x{h}x{w}', g0, refs, {wt: ('w', WGRAD_BAR), b: ('b', BIAS_BAR)})


# ---------------------------------------------------------------------------- several contributions to one .grad
@pytest.mark.parametrize('streams', [1, 2])
@pytest.mark.parametrize('cin,cout,k', [(64, 64, 3), (256, 128, 1), (16, 8, 3)])
def test_conv_shared_weight(cin, cout, k, streams, calls):
    """One weight (and bias) in two convs of one backward; with streams = 2 the second conv runs on another stream,
    the way GanTrainer.d_forward_backward runs D(fake), so its backward chain runs there too; the in-place weight
    gradients of both chains must still go to the one weight-gradient stream, since the wgrad unpack and
    ttg_channel_sum_acc add with a plain read-modify-write.  `.grad` is read right after the `with` block, without a
    device synchronise: join_all_streams() must have ordered every contribution before it."""
    ops = _ops()
    torch.manual_seed(cin + cout + streams)
    n, h, w = 2, 37, 45
    xs = [_dev(torch.randn(n, cin, h, w)) for _ in range(2)]
    gys = [_dev(torch.randn(n, cout, h, w)) for _ in range(2)]
    wt, b = _params(torch.randn(cout, cin, k, k) / math.sqrt(cin * k * k), torch.randn(cout))
    refs = {wt: _wgrad_ref(xs[0], gys[0], k) + _wgrad_ref(xs[1], gys[1], k),
            b: _host(gys[0]).sum((0, 2, 3)) + _host(gys[1]).sum((0, 2, 3))}
    g0 = _prefill(refs)
    main = torch.cuda.current_stream()
    ys = [ops.conv2d(xs[0], wt, b)]
    if streams == 2:
        side = torch.cuda.Stream()
        side.wait_stream(main)
        ops.state.pending_streams.add(side)
        with torch.cuda.stream(side):
            ys.append(ops.conv2d(xs[1], wt, b))
        main.wait_stream(side)
    else:
        ys.append(ops.conv2d(xs[1], wt, b))
    with ops.direct_param_grads():
        torch.autograd.backward(ys, gys)
    got = {wt: wt.grad.clone(), b: b.grad.clone()}          # on the launching stream, no synchronise before
    got = {p: _host(t) for p, t in got.items()}
    _check_calls(calls, {'ttg_conv2d_wgrad_tc_acc': 2, 'ttg_channel_sum_acc': 2 * int(cout < 16)})
    _compare(f'shared {cin}->{cout} k{k} streams {streams}', g0, refs, {wt: ('w', WGRAD_BAR), b: ('b', BIAS_BAR)}, got)


# ------------------------------------------------------------------------------------ BatchNorm + LeakyReLU
def _bn_ambiguous(a, tol=1e-4):
    """-> (x, gamma, beta, mean, invstd as float64 from what BnActFn saved, mask of the elements whose pre-activation
    is within `tol` of zero, where the LeakyReLU slope the kernel applies depends on its rounding)."""
    x, gamma, beta, mean, invstd = (_host(t) for t in a.grad_fn.saved_tensors)
    v = lambda t: t.view(1, -1, 1, 1)
    y = v(gamma) * (x - v(mean)) * v(invstd) + v(beta)
    return (x, gamma, beta, mean, invstd), y.abs() < tol * (1 + v(beta).abs())


def _bn_first_order(saved, ga, slope):
    """(d gamma, d beta) of lrelu(batch_norm(x)) for the cotangent ga, with the kernel's batch statistics."""
    x, gamma, beta, mean, invstd = saved
    v = lambda t: t.view(1, -1, 1, 1)
    xhat = (x - v(mean)) * v(invstd)
    d = ga * torch.where(v(gamma) * xhat + v(beta) > 0, 1.0, slope)
    return (d * xhat).sum((0, 2, 3)), d.sum((0, 2, 3))


def _bn_second_order_gamma(saved, ga, u, slope):
    """d/d gamma of <gx, u>, gx = the input gradient of lrelu(batch_norm(x)) for ga (the R1 term; the statistics
    do not depend on gamma and the mask is piecewise constant)."""
    x, gamma, beta, mean, invstd = saved
    v = lambda t: t.view(1, -1, 1, 1)
    xhat = (x - v(mean)) * v(invstd)
    d = ga * torch.where(v(gamma) * xhat + v(beta) > 0, 1.0, slope)
    mu = lambda t: t.mean((0, 2, 3), keepdim=True)
    return invstd * (u * (d - mu(d) - xhat * mu(d * xhat))).sum((0, 2, 3))


def _bn_module(c):
    bn = torch.nn.BatchNorm2d(c).cuda()
    bn.weight, bn.bias = _params(1 + 0.3 * torch.randn(c), 0.3 * torch.randn(c))
    return bn


@pytest.mark.parametrize('n,c,h,w', [(4, 16, 33, 35), (8, 32, 16, 16), (2, 64, 19, 23), (3, 256, 9, 11)])
def test_bn_act_param_grads_acc(n, c, h, w, workspace, calls):
    ops = _ops()
    torch.manual_seed(c + h)
    bn = _bn_module(c)
    x = _dev(0.5 + 2 * torch.randn(n, c, h, w))
    a = ops.bn_act(x, bn)
    saved, amb = _bn_ambiguous(a)
    ga = _dev(torch.randn(n, c, h, w).masked_fill(amb, 0))
    ref_gamma, ref_beta = _bn_first_order(saved, _host(ga), ops.SLOPE)
    refs = {bn.weight: ref_gamma, bn.bias: ref_beta}
    g0 = _prefill(refs)
    with ops.direct_param_grads():
        a.backward(ga)
    _check_calls(calls, {'ttg_bn_act_bwd_acc': 1}, workspace)
    _compare(f'bn_act C{c} {n}x{h}x{w}', g0, refs, {bn.weight: ('gamma', BN_BAR), bn.bias: ('beta', BN_BAR)})


# ----------------------------------------------------------------------------------------- R1 second order
def test_r1_second_order_acc(workspace, calls, monkeypatch):
    """conv + bias -> bn_act -> conv + bias, the layer pattern of D.  Like GanTrainer.d_forward_backward: the input
    gradient is taken with create_graph inside ops.inputs_only_grads(), then ONE backward of the first-order objective
    and of a penalty on that gradient runs under direct_param_grads().  Each conv weight then receives a first-order
    contribution (Conv2dFn.backward) and an R1 one (ConvDgradFn.backward); gamma a first-order one
    (ttg_bn_act_bwd_acc) and an R1 one (ttg_bn_act_bwd2_acc).  The references sum the float64 contributions of the
    operands each call received."""
    ops = _ops()
    torch.manual_seed(5)
    n, c0, c1, c2, h, w = 4, 16, 32, 16, 21, 27
    x = _dev(torch.randn(n, c0, h, w)).requires_grad_()
    w1, b1, w2, b2 = _params(torch.randn(c1, c0, 3, 3) / math.sqrt(9 * c0), 0.1 * torch.randn(c1),
                             torch.randn(c2, c1, 3, 3) / math.sqrt(9 * c1), 0.1 * torch.randn(c2))
    bn = _bn_module(c1)
    a = ops.bn_act(ops.conv2d(x, w1, b1), bn)
    out = ops.conv2d(a, w2, b2)
    saved, amb = _bn_ambiguous(a)
    # zero the output cotangents wherever the 3x3 conv after the BatchNorm would carry them to an ambiguous element
    amb = F.max_pool2d(amb.any(1, keepdim=True).double(), 3, 1, 1) > 0
    g_in, g_out = (_dev(torch.randn(n, c2, h, w).masked_fill(amb, 0)) for _ in range(2))
    u = _dev(torch.randn(n, c0, h, w))
    with ops.inputs_only_grads():
        gx, = torch.autograd.grad(out, x, g_in, create_graph=True)

    wgrads, bn1, bn2 = [], [], []
    real_wgrad, real_bwd, real_bwd2 = ops._wgrad_direct, ops.BnActFn.backward, ops.BnActBwdFn.backward

    def wgrad(x_, gy, w_, bias, up, want_b):
        done = real_wgrad(x_, gy, w_, bias, up, want_b)
        if done:
            wgrads.append((w_, bias if want_b else None, x_, gy))
        return done

    def bwd(ctx, ga):
        if ops.state.direct_grads:
            bn1.append(_host(ga))
        return real_bwd(ctx, ga)

    def bwd2(ctx, u_, *rest):
        if ops.state.direct_grads:
            bn2.append((_host(ctx.saved_tensors[1]), _host(u_)))
        return real_bwd2(ctx, u_, *rest)
    monkeypatch.setattr(ops, '_wgrad_direct', wgrad)
    monkeypatch.setattr(ops.BnActFn, 'backward', staticmethod(bwd))
    monkeypatch.setattr(ops.BnActBwdFn, 'backward', staticmethod(bwd2))

    g0 = {p: _host(p.grad) for p in (w1, b1, w2, b2, bn.weight, bn.bias)}
    calls.clear()                        # (the create_graph pass above ran the overwriting BatchNorm backward)
    with ops.direct_param_grads():
        torch.autograd.backward([out, gx], [g_out, u])
    got = {p: _host(p.grad) for p in g0}
    _check_calls(calls, {'ttg_conv2d_wgrad_tc_acc': 4, 'ttg_bn_act_bwd_acc': 1, 'ttg_bn_act_bwd2_acc': 1}, workspace)
    assert len(bn1) == 1 and len(bn2) == 1 and len(wgrads) == 4

    refs = {p: torch.zeros_like(g0[p]) for p in g0}
    for w_, bias, x_, gy in wgrads:
        refs[w_] += _wgrad_ref(x_, gy, w_.shape[2])
        if bias is not None:
            refs[bias] += _host(gy).sum((0, 2, 3))
    assert {id(w_) for w_, *_ in wgrads} == {id(w1), id(w2)}
    assert sorted(id(b) for _, b, _, _ in wgrads if b is not None) == sorted([id(b1), id(b2)])
    d_gamma, d_beta = _bn_first_order(saved, bn1[0], ops.SLOPE)
    refs[bn.weight] += d_gamma + _bn_second_order_gamma(saved, *bn2[0], ops.SLOPE)
    refs[bn.bias] += d_beta
    # b1 feeds the BatchNorm: its gradient is analytically zero, so the pixel sums cancel and their relative error
    # is larger (measured 1.4e-6 / 2.8e-6)
    bars = {w1: ('w1', WGRAD_BAR), w2: ('w2', WGRAD_BAR), b1: ('b1', (2e-5, 5e-5)), b2: ('b2', BIAS_BAR),
            bn.weight: ('gamma', BN_BAR), bn.bias: ('beta', BN_BAR)}
    _compare('r1', g0, refs, bars, got)


# -------------------------------------------------------------------------------------------- generator head
@pytest.mark.parametrize('bias', [True, False], ids=['bias', 'nobias'])
@pytest.mark.parametrize('cin', [8, 16, 32])
def test_rgb_head_acc(cin, bias, calls):
    """ops.RgbHeadFn (conv1x1 C -> 3 + tanh, fp32 NCHW out) adds its weight and bias gradients to .grad."""
    ops = _ops()
    torch.manual_seed(cin)
    n, h, w = 3, 37, 45
    a = _dev(torch.randn(n, cin, h, w))
    wt, b = _params(0.3 * torch.randn(3, cin, 1, 1), 0.1 * torch.randn(3))
    b = b if bias else None
    y = ops.RgbHeadFn.apply(a, wt, b)
    g = torch.randn(y.shape, device='cuda')
    gpre = _host(g) * (1 - _host(y) ** 2)
    refs = {wt: torch.einsum('nohw,nihw->oi', gpre, _host(a)).view(3, cin, 1, 1)}
    if bias:
        refs[b] = gpre.sum((0, 2, 3))
    g0 = _prefill(refs)
    with ops.direct_param_grads():
        y.backward(g)
    _check_calls(calls, {'ttg_rgb_head_bwd': 1})
    _compare(f'rgb_head C{cin}', g0, refs, {wt: ('w', RGB_BAR), b: ('b', RGB_BAR)})


# ------------------------------------------------------------------------- trainer: in-place against autograd
def _step_grads(t, imgs):
    torch.manual_seed(300)
    t.train_batch(imgs)
    torch.cuda.synchronize()
    return {(net, k): _host(p.grad) for net, mod in (('d', t.d), ('g', t.g)) for k, p in mod.named_parameters()}


def _rel(a, b, floor):
    """Relative L2 difference; a tensor whose gradient is below `floor` per element (conv biases that feed a
    BatchNorm: analytically zero, rounding noise) is measured on that scale instead."""
    return float((a - b).norm() / max(float(b.norm()), floor * math.sqrt(b.numel())))


@pytest.mark.parametrize('graph', [False, True], ids=['eager', 'graph'])
@pytest.mark.parametrize('config,batch', [('64', 64), ('128', 32)])
def test_trainer_direct_matches_autograd(config, batch, graph, monkeypatch):
    """One D and one G half-step (train_batch with both learning rates 0) with the in-place path and with
    AccumulateGrad (ops._NO_DIRECT): every parameter gradient agrees to within a few times the run-to-run spread."""
    from oracle import tartan_oracle as O
    from tartangan_b200 import ops
    from tartangan_b200.trainers.gan import make_trainer
    from tartangan_b200.trainers.iqn import IQNTrainer
    imgs = O.tartan_batch(1234, batch, int(config))
    runs, state = {}, None
    for arm in ('direct', 'autograd'):
        monkeypatch.setattr(ops, '_NO_DIRECT', arm == 'autograd')
        torch.manual_seed(0)
        t = make_trainer(IQNTrainer, config=config, batch_size=batch, precision='bf16', cuda_graph=graph,
                         lr_d=0.0, lr_g=0.0)
        if state is None:
            state = [{k: v.detach().clone() for k, v in m.state_dict().items()} for m in (t.g, t.target_g, t.d)]
        else:
            for m, sd in zip((t.g, t.target_g, t.d), state):
                m.load_state_dict(sd)
            t.parameters_changed()
        runs[arm] = [_step_grads(t, imgs) for _ in range(2)]
        del t
    for net in ('d', 'g'):
        keys = [k for k in runs['direct'][0] if k[0] == net]
        ref = runs['autograd'][0]
        floor = 2e-3 * max(float(ref[k].abs().max()) for k in keys)
        spread = {k: max(_rel(r[0][k], r[1][k], floor) for r in runs.values()) for k in keys}
        diff = {k: _rel(runs['direct'][0][k], ref[k], floor) for k in keys}
        bar = {k: max(4 * spread[k], 1e-5) for k in keys}
        ks, kd = max(spread, key=spread.get), max(diff, key=lambda k: diff[k] / bar[k])
        print(f'[grad-acc] trainer {config} {"graph" if graph else "eager"} {net}: {len(keys)} gradients, worst spread '
              f'{ks[1]} {spread[ks]:.2e}, worst direct-vs-autograd relative to its bar {kd[1]} {diff[kd]:.2e} '
              f'(spread {spread[kd]:.2e}, bar {bar[kd]:.2e})')
        bad = [(k[1], diff[k], spread[k]) for k in keys if not diff[k] <= bar[k]]
        assert not bad, bad
