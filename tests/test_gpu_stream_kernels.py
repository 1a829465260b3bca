"""The streaming kernels (channel-wise drivers, BatchNorm, resampling, joins, layout, max-pool) against float64.

Every case calls the C ABI directly (`_lib.call`), so that it controls which kernel the dispatcher picks, and asserts by
name (torch.profiler, CUDA activity only) that this kernel ran.  A view that starts one element into a slightly larger
buffer breaks the 16-byte alignment and selects the scalar paths; no pointer or size reaches outside an allocation.
Outputs are prefilled with NaN, so an element a kernel skips fails.  References are float64 on the CPU, computed from
the bf16 / fp32 operands the kernels received.

Bars (u = 2^-24, the fp32 unit roundoff; `A` = the sum of the absolute values of the terms of the fp32 expression the
kernel evaluates, i.e. the expression with every operand replaced by its magnitude):
  * pure data movement is bit-exact: upsample2 at scale 1, the layout kernels (fp32 -> bf16 must round to nearest
    even, like torch's cast), spatial_bcast, max-pool forward / scatter / gather;
  * an output the kernel computes as one fp32 expression of its operands and rounds once: |err| <= half an ulp of the
    output dtype at the float64 value + 8 u A (at most 8 fp32 roundings per expression); for bf16 outputs this is one
    bf16 ulp in practice.  Bilinear adds 8 u max(H, W) max|x|: its source coordinate o * (in - 1) / (out - 1) is
    formed in fp32, so each weight may be off by 2 u in;
  * reductions: every fp32 partial sum of these kernels collects at most L = 64 terms at the sizes used here (grid-
    stride loops over one full wave; the bulk kernel: 2 units per chunk and <= 30 chunks per block), and partial
    sums are combined in fp64, so |err| <= 64 u sum|terms|.  spatial_sum is one thread per (image, channel) walking
    all HW pixels: L = HW;
  * BatchNorm statistics: mean +- 64 u E|x|, var = E[x^2] - mean^2 +- 64 u (E[x^2] + 2 |mean| E|x|), and invstd,
    the running statistics from those by first-order propagation (+ a few u for their own fp32 arithmetic);
  * BatchNorm backward and double backward outputs: half an ulp + 64 u A, where A is built from the magnitudes of
    the terms that cancel (d, mean(d), xhat * mean(d xhat), ...), not from the result, and the reduced per-channel
    means enter A through their absolute sums.  These references run float64 autograd through a BatchNorm whose
    statistics have the kernel's values (`_bn_ref`), so that the fp32 error of the statistics, checked on its own,
    does not enter the output bars a second time.

The LeakyReLU mask flips where the pre-activation is within rounding of zero; which way is not part of the contract,
so the cotangents are zeroed there and the one output that is multiplied by the mask itself (d/d ga of the double
backward) is not compared there.

Coverage (kernel -> cases):
  chan_reduce_bulk_kernel / chan_map_bulk_kernel     test_bn_chain[bulk-*, wrap-*, mean16], test_eltwise[*-bulk]
  chan_reduce_c3_kernel / chan_map_c3_kernel         test_bn_chain[c3-*]
  chan_reduce_kernel<T, V> / chan_map_kernel<T, V>   test_bn_chain[reg-*], test_eltwise[*-reg, *-f32]
  chan_reduce_kernel<T, 1> / chan_map_kernel<T, 1>   test_bn_chain[scalar-*, misaligned-*], test_eltwise[*-odd, *-mis]
  bn_finalize_kernel, count_mult, producer sums      test_bn_statistics;  bn_eval_stats_kernel: test_bn_eval
  pool2_bf16x8 / pool2<T, V> / pool2<T, 1>           test_pool2_upsample2 (bf16 pool2<T, 8> needs >= 2^31 units)
  upsample2_bf16x8 / upsample2<T, V> / <T, 1>        test_pool2_upsample2
  bilinear_down_kernel, bilinear_down_bwd_kernel     test_bilinear, test_bilinear_candidate_sweep, ..._smem_limit
  add_up2_kernel / pool2_add_kernel (+ stats)        test_joins, test_join_stats, test_join_stats_fallback
  nchw_to_nhwc (elem, rgb, per pixel), nhwc_to_nchw  test_layout;  spatial_sum / spatial_bcast: test_spatial
  maxpool2_fwd / scatter / gather                    test_maxpool_ties, test_maxpool_nan
"""
import math
import re

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
L_SUM = 64                 # longest fp32 partial-sum chain at these sizes (see the module docstring)
K_EXPR = 8                 # fp32 roundings per output expression
F32, BF16 = 0, 1
TORCH_DT = {F32: torch.float32, BF16: torch.bfloat16}
TNAME = {F32: 'float', BF16: '__nv_bfloat16'}
VN = {F32: 4, BF16: 8}     # elements per 16-byte vector
EPS, MOM, SLOPE = 1e-5, 0.1, 0.2
NAN = float('nan')


def _lib():
    import tartangan_b200  # noqa: F401
    from tartangan_b200 import _lib as lib
    lib.lib.load()
    return lib


def _call(name, *args):
    _lib().call(name, *args)


def _p(t):
    return None if t is None else t.data_ptr()


@pytest.fixture(scope='module')
def kernels():
    """run(fn) -> names of the CUDA kernels that fn launched."""
    from torch.profiler import ProfilerActivity, profile

    def run(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events()]
    run(lambda: torch.zeros(8, device='cuda').add_(1))     # (first use initialises the tracer)
    return run


def _ran(names, *patterns):
    for pat in patterns:
        assert any(re.search(pat, n) for n in names), (pat, sorted(set(names)))


def _not_ran(names, *patterns):
    for pat in patterns:
        assert not any(re.search(pat, n) for n in names), (pat, sorted(set(names)))


# ------------------------------------------------------------------------------------------------------- buffers
def _buf(n, dt, misalign=False, fill=NAN):
    """n elements on the device, NaN-filled; misalign: the view starts one element into a larger buffer."""
    base = torch.full((n + 16,), fill, dtype=TORCH_DT[dt] if isinstance(dt, int) else dt, device='cuda')
    off = 1 if misalign else 0
    return base[off:off + n]


def _q(host, dt):
    """host values rounded to the kernel dtype, as float64."""
    return host.to(TORCH_DT[dt]).double()


def _dev(host, dt, misalign=False):
    d = _buf(host.numel(), dt, misalign)
    d.copy_(host.reshape(-1).to(TORCH_DT[dt]))
    return d


def _host(t, shape=None):
    h = t.detach().double().cpu()
    return h.view(shape) if shape is not None else h


def _half_ulp(ref, dt):
    """half an ulp of the output dtype at |ref| (0 where ref == 0)."""
    _, e = torch.frexp(ref)
    h = torch.ldexp(torch.ones_like(ref), e - (9 if dt == BF16 else 25))
    return torch.where(ref == 0, torch.zeros_like(ref), h)


def _bar(ref, dt, A, k=K_EXPR):
    return _half_ulp(ref, dt) + k * U * A


def _check(group, tag, got, ref, bar, mask=None):
    got, ref, bar = (t.reshape(-1).double().cpu() for t in (got, ref, bar))
    if mask is not None:
        m = mask.reshape(-1).cpu()
        got, ref, bar = got[m], ref[m], bar[m]
    err = (got - ref).abs()
    bad = ~(err <= bar)
    ratio = float((err / bar.clamp_min(1e-300)).max()) if err.numel() else 0.0
    print(f'[stream] {group} {tag}: worst |err|/bar {ratio:.3g}, max |err| {float(err.max()) if err.numel() else 0:.3g}')
    if bad.any():
        i = int(bad.nonzero()[0])
        raise AssertionError(f'{group} {tag}: {int(bad.sum())} of {got.numel()} outside the bar; first at {i}: '
                             f'got {float(got[i])}, ref {float(ref[i])}, bar {float(bar[i])}')


def _exact(group, tag, got, ref):
    got, ref = got.reshape(-1).double().cpu(), ref.reshape(-1).double().cpu()
    bad = ~((got == ref) | (got.isnan() & ref.isnan()))
    print(f'[stream] {group} {tag}: exact, {int(bad.sum())} differ')
    if bad.any():
        i = int(bad.nonzero()[0])
        raise AssertionError(f'{group} {tag}: {int(bad.sum())} of {got.numel()} differ; first at {i}: '
                             f'got {float(got[i])}, ref {float(ref[i])}')


# ------------------------------------------------------------------------------------------ channel-wise dispatch
def _branch(n, C, dt, aligned):
    """The kernel launch_chan_reduce / launch_chan_map pick (csrc/chanops.cuh)."""
    if C == 3 and aligned and n % (3 * VN[dt]) == 0:
        return 'c3'
    g = C // 8
    if dt == BF16 and C % 8 == 0 and g & (g - 1) == 0 and g <= 32 and aligned and n >= 8 * 512 * 148:
        return 'bulk'
    if C % VN[dt] == 0 and aligned:
        return 'vec'
    return 'scalar'


def _reduce_pat(branch, dt):
    return {'c3': r'chan_reduce_c3_kernel<', 'bulk': r'chan_reduce_bulk_kernel<',
            'vec': rf'chan_reduce_kernel<{TNAME[dt]}, {VN[dt]}, ', 'scalar': rf'chan_reduce_kernel<{TNAME[dt]}, 1, '}[branch]


def _map_pat(branch, dt):
    return {'c3': r'chan_map_c3_kernel<', 'bulk': r'chan_map_bulk_kernel<',
            'vec': rf'chan_map_kernel<{TNAME[dt]}, {VN[dt]}, ', 'scalar': rf'chan_map_kernel<{TNAME[dt]}, 1, '}[branch]


# ------------------------------------------------------------------------------------------------- BatchNorm
def _bn_input(M, C, dt, mean_ratio=0.3, seed=0):
    g = torch.Generator().manual_seed(seed)
    std = 0.5 + 1.5 * torch.rand(C, generator=g, dtype=torch.float64)
    sign = torch.where(torch.rand(C, generator=g) < 0.5, -1.0, 1.0).double()
    x = torch.randn(M, C, generator=g, dtype=torch.float64) * std + sign * mean_ratio * std
    return _q(x, dt)


def _stats_bars(x, mean_ref, Mu, rm0, rv0, k=L_SUM):
    """-> bars of (mean, invstd, running_mean, running_var) for statistics reduced from x (see the docstring)."""
    M = x.shape[0]
    ea, e2 = x.abs().mean(0), (x * x).mean(0)
    var_ref = x.var(0, unbiased=False)
    dm = k * U * ea + 2 * U * mean_ref.abs()
    dvar = k * U * (e2 + 2 * mean_ref.abs() * ea) + 1e-15 * e2
    r = (var_ref + EPS).rsqrt()
    dr = 0.5 * r ** 3 * dvar + 4 * U * r
    f = Mu / (Mu - 1) if Mu > 1 else 1.0
    drm = MOM * dm + 4 * U * (rm0.abs() + mean_ref.abs())
    drv = MOM * f * dvar + 4 * U * (rv0.abs() + var_ref * f)
    return dm, dr, drm, drv


def _check_stats(group, tag, x, mean, invstd, rm, rv, rm0, rv0, count_mult=1, k=L_SUM):
    """mean / invstd / running statistics against float64 F.batch_norm (running var: unbiased over M * count_mult)."""
    M = x.shape[0]
    Mu = M * count_mult
    mean_ref, var_ref = x.mean(0), x.var(0, unbiased=False)
    rm_ref, rv_ref = rm0.clone(), rv0.clone()
    if count_mult == 1:
        F.batch_norm(x, rm_ref, rv_ref, training=True, momentum=MOM, eps=EPS)
    else:
        rm_ref = (1 - MOM) * rm0 + MOM * mean_ref
        rv_ref = (1 - MOM) * rv0 + MOM * var_ref * Mu / (Mu - 1)
    dm, dr, drm, drv = _stats_bars(x, mean_ref, Mu, rm0, rv0, k)
    _check(group, f'{tag} mean', _host(mean), mean_ref, dm)
    _check(group, f'{tag} invstd', _host(invstd), (var_ref + EPS).rsqrt(), dr)
    _check(group, f'{tag} running_mean', _host(rm), rm_ref, drm)
    _check(group, f'{tag} running_var', _host(rv), rv_ref, drv)


def _bn_ref(x, mk, rk, gamma, beta, ga, u):
    """float64 autograd of lrelu(batch_norm(x)) in train mode, with the statistics pinned to the kernel's values
    (mk, rk) but their derivatives those of the batch mean and the biased batch variance:
    -> y, (gx, d gamma, d beta) for ga, (d/dx, d/dga, d/dgamma of <gx, u>)."""
    xr, g, b, gar = (t.clone().requires_grad_() for t in (x, gamma, beta, ga))
    mt = xr.mean(0)
    vt = ((xr - mt) ** 2).mean(0)
    m = mk + (mt - mt.detach())
    v = (rk.pow(-2) - EPS) + (vt - vt.detach())
    a = F.leaky_relu(g * (xr - m) * (v + EPS).rsqrt() + b, SLOPE)
    gx, gg, gb = torch.autograd.grad(a, (xr, g, b), gar, create_graph=True)
    g_x, g_ga, gg2 = torch.autograd.grad(gx, (xr, gar, g), u)
    return a.detach(), (gx.detach(), gg.detach(), gb.detach()), (g_x, g_ga, gg2)


class _BnDev:
    """Device operands of one BatchNorm case."""

    def __init__(self, M, C, dt, misalign, seed):
        g = torch.Generator().manual_seed(seed + 1)
        self.gamma = (1 + 0.3 * torch.randn(C, generator=g, dtype=torch.float64)).float().double()
        self.beta = (0.3 * torch.randn(C, generator=g, dtype=torch.float64)).float().double()
        self.rm0 = torch.randn(C, generator=g, dtype=torch.float64).float().double()
        self.rv0 = (0.5 + torch.rand(C, generator=g, dtype=torch.float64)).float().double()
        f = lambda t: t.float().cuda()
        self.d_gamma, self.d_beta = f(self.gamma), f(self.beta)
        self.rm, self.rv = f(self.rm0), f(self.rv0)
        self.mean, self.invstd = _buf(C, torch.float32), _buf(C, torch.float32)
        self.nb = torch.full((1,), 7, dtype=torch.int64, device='cuda')
        self.ws = torch.full((5 * C,), 1e30, dtype=torch.float64, device='cuda')   # reduce kernels must clear it


# (M rows, C, dtype, misaligned, per-channel |mean| / std)
def _rows(n_elem, C, extra=3):
    return -(-n_elem // C) + extra


BN_CASES = {}
for _C in (8, 16, 32, 64, 128, 256):
    BN_CASES[f'bulk-C{_C}'] = (_rows(8 * 512 * 148, _C), _C, BF16, False, 0.3)     # just above the bulk threshold
    BN_CASES[f'reg-C{_C}'] = (_rows(300_000, _C), _C, BF16, False, 0.3)              # shuffle group counts 1..32
BN_CASES.update({
    # The two wrap cases (about 17 M elements) are the slowest: their float64 double-backward reference holds a few
    # GB of host memory at its peak.  They keep the backward passes, because the 2- and 3-input bulk kernels run
    # fewer blocks per SM, so their rings wrap more often than the statistics pass does.
    'wrap-C16': (1_100_003, 16, BF16, False, 0.3),      # 4297 chunks > 4 x 148 x 7, partial last chunk
    'wrap-C128': (133_001, 128, BF16, False, 0.3),      # 4157 chunks
    'mean16-C32': (20_003, 32, BF16, False, 16.0),      # bulk, |mean| = 16 std: var = E[x^2] - mean^2 cancels
    'mean16-reg-C64': (4_001, 64, BF16, False, 16.0),
    'reg-C120': (2_501, 120, BF16, False, 0.3),         # 15 groups (512thin-test)
    'reg-C200': (1_501, 200, BF16, False, 0.3),         # 25 groups (test256)
    'reg-C512': (601, 512, BF16, False, 0.3),           # 64 groups (128big)
    'reg-C1024': (301, 1024, BF16, False, 0.3),         # 128 groups (1024)
    'scalar-C100': (3_001, 100, BF16, False, 0.3),      # 512thin-test
    'scalar-C180': (1_701, 180, BF16, False, 0.3),      # test256
    'scalar-C4': (40_001, 4, BF16, False, 0.3),         # test128
    'misaligned-C16': (20_001, 16, BF16, True, 0.3),
    'misaligned-bulksize-C16': (_rows(8 * 512 * 148, 16), 16, BF16, True, 0.3),
    'c3-bf16': (65_536, 3, BF16, False, 0.3),
    'scalar-C3': (65_537, 3, BF16, False, 0.3),         # n not a multiple of 24
    'misaligned-C3': (65_536, 3, BF16, True, 0.3),
    'f32-C16': (20_001, 16, F32, False, 0.3),
    'f32-C100': (3_001, 100, F32, False, 0.3),
    'f32-c3': (65_536, 3, F32, False, 0.3),
    'f32-scalar-C6': (20_001, 6, F32, False, 0.3),
    'f32-misaligned-C16': (20_001, 16, F32, True, 0.3),
})


@pytest.mark.parametrize('case', list(BN_CASES))
def test_bn_chain(case, kernels):
    """ttg_bn_act_fwd_stats (statistics reduced here), ttg_bn_act_fwd, ttg_channel_sum, ttg_bn_act_bwd (with and
    without gx) and ttg_bn_act_bwd2 on one tensor, each on the branch `_branch` predicts."""
    M, C, dt, mis, mean_ratio = BN_CASES[case]
    n = M * C
    br = _branch(n, C, dt, not mis)
    group = f'bn/{br}'
    seed = M + C
    x = _bn_input(M, C, dt, mean_ratio, seed)
    d = _BnDev(M, C, dt, mis, seed)
    dx = _dev(x, dt, mis)
    y = _buf(n, dt, mis)

    names = kernels(lambda: _call('ttg_bn_act_fwd_stats', _p(dx), _p(y), M, C, None, _p(d.d_gamma), _p(d.d_beta),
                                  EPS, MOM, SLOPE, _p(d.mean), _p(d.invstd), _p(d.rm), _p(d.rv), _p(d.nb), 1,
                                  _p(d.ws), dt))
    _ran(names, _reduce_pat(br, dt), _map_pat(br, dt))
    assert int(d.nb) == 8
    _check_stats(group, case, x, d.mean, d.invstd, d.rm, d.rv, d.rm0, d.rv0)
    mk, rk = _host(d.mean), _host(d.invstd)

    # forward apply, with the kernel's statistics
    a = d.gamma * rk
    y_ref = F.leaky_relu(x * a + (d.beta - mk * a), SLOPE)
    A_y = (x * a).abs() + (mk * a).abs() + d.beta.abs()
    _check(group, f'{case} y (fwd_stats)', _host(y, (M, C)), y_ref, _bar(y_ref, dt, A_y))
    y2 = _buf(n, dt, mis)
    names = kernels(lambda: _call('ttg_bn_act_fwd', _p(dx), _p(y2), M, C, _p(d.mean), _p(d.invstd), _p(d.d_gamma),
                                  _p(d.d_beta), SLOPE, dt))
    _ran(names, _map_pat(br, dt))
    _check(group, f'{case} y (fwd)', _host(y2, (M, C)), y_ref, _bar(y_ref, dt, A_y))

    # per-channel sum (conv bias gradient)
    cs = _buf(C, torch.float32)
    names = kernels(lambda: _call('ttg_channel_sum', _p(dx), M, C, _p(cs), _p(d.ws), dt))
    _ran(names, _reduce_pat(br, dt))
    _check(group, f'{case} channel_sum', _host(cs), x.sum(0), L_SUM * U * x.abs().sum(0))

    # backward; cotangents zeroed where the LeakyReLU mask depends on rounding
    g = torch.Generator().manual_seed(seed + 2)
    pre = x * a + (d.beta - mk * a)
    amb = pre.abs() <= 1e-5 * A_y
    ga = _q(torch.randn(M, C, generator=g, dtype=torch.float64).masked_fill(amb, 0), dt)
    u = _q(torch.randn(M, C, generator=g, dtype=torch.float64), dt)
    _, (gx_ref, gg_ref, gb_ref), (g_x_ref, g_ga_ref, gg2_ref) = _bn_ref(x, mk, rk, d.gamma, d.beta, ga, u)
    dga, du = _dev(ga, dt, mis), _dev(u, dt, mis)
    gx, gg, gb = _buf(n, dt, mis), _buf(C, torch.float32), _buf(C, torch.float32)
    names = kernels(lambda: _call('ttg_bn_act_bwd', _p(dx), _p(dga), _p(gx), M, C, _p(d.mean), _p(d.invstd),
                                  _p(d.d_gamma), _p(d.d_beta), SLOPE, _p(gg), _p(gb), _p(d.ws), dt))
    _ran(names, _reduce_pat(br, dt), _map_pat(br, dt))
    X = (x.abs() + mk.abs()) * rk                    # bounds |xhat| and scales the fp32 error of forming it
    gr = (d.gamma * rk).abs()
    gaa, ua = ga.abs(), u.abs()
    mean = lambda t: t.mean(0)
    A_Pd = gaa + mean(gaa) + X * mean(gaa * X)
    A_Pu = ua + mean(ua) + X * mean(ua * X)
    _check(group, f'{case} gx', _host(gx, (M, C)), gx_ref, _bar(gx_ref, dt, gr * A_Pd, L_SUM))
    _check(group, f'{case} d gamma', _host(gg), gg_ref, L_SUM * U * (gaa * X).sum(0) + U * gg_ref.abs())
    _check(group, f'{case} d beta', _host(gb), gb_ref, L_SUM * U * gaa.sum(0) + U * gb_ref.abs())

    gg_, gb_ = _buf(C, torch.float32), _buf(C, torch.float32)
    names = kernels(lambda: _call('ttg_bn_act_bwd', _p(dx), _p(dga), None, M, C, _p(d.mean), _p(d.invstd),
                                  _p(d.d_gamma), _p(d.d_beta), SLOPE, _p(gg_), _p(gb_), _p(d.ws), dt))
    _ran(names, _reduce_pat(br, dt), r'bn_param_grads_kernel')
    _not_ran(names, r'chan_map')
    _check(group, f'{case} d gamma (no gx)', _host(gg_), gg_ref, L_SUM * U * (gaa * X).sum(0) + U * gg_ref.abs())
    _check(group, f'{case} d beta (no gx)', _host(gb_), gb_ref, L_SUM * U * gaa.sum(0) + U * gb_ref.abs())

    # backward of backward (R1)
    g_ga, g_x, gg2 = _buf(n, dt, mis), _buf(n, dt, mis), _buf(C, torch.float32)
    names = kernels(lambda: _call('ttg_bn_act_bwd2', _p(dx), _p(dga), _p(du), _p(g_ga), _p(g_x), M, C, _p(d.mean),
                                  _p(d.invstd), _p(d.d_gamma), _p(d.d_beta), SLOPE, _p(gg2), _p(d.ws), dt))
    _ran(names, _reduce_pat(br, dt), _map_pat(br, dt))
    _check(group, f'{case} bwd2 d ga', _host(g_ga, (M, C)), g_ga_ref, _bar(g_ga_ref, dt, gr * A_Pu, L_SUM), mask=~amb)
    A_k = X * (mean(gaa * X) * mean(ua * X) + mean(ua * gaa) + mean(ua) * mean(gaa))
    A_gx2 = gr * rk * (A_k + mean(ua * X) * A_Pd + mean(gaa * X) * A_Pu)
    _check(group, f'{case} bwd2 d x', _host(g_x, (M, C)), g_x_ref, _bar(g_x_ref, dt, A_gx2, L_SUM))
    A_gg2 = rk * M * (mean(ua * gaa) + mean(ua) * mean(gaa) + mean(gaa * X) * mean(ua * X))
    _check(group, f'{case} bwd2 d gamma', _host(gg2), gg2_ref, L_SUM * U * A_gg2 + U * gg2_ref.abs())


@pytest.mark.parametrize('count_mult', [1, 4])
@pytest.mark.parametrize('C,dt', [(16, BF16), (3, BF16), (32, F32)])
def test_bn_statistics(C, dt, count_mult, kernels):
    """ttg_bn_stats (bn_finalize_kernel) and ttg_bn_act_fwd_stats with producer sums: mean, invstd, running mean and
    unbiased running var over M * count_mult (count_mult = 4: the BatchNorm on the low-resolution source of an
    upsample), num_batches + 1 per call.  The producer sums are exact float64 sums, so the finalisation is checked
    at fp32 resolution."""
    M = 2 * 8 * 8
    x = _bn_input(M, C, dt, 2.0, seed=C + count_mult)
    d = _BnDev(M, C, dt, False, C)
    dx = _dev(x, dt)
    names = kernels(lambda: _call('ttg_bn_stats', _p(dx), M, C, EPS, MOM, _p(d.mean), _p(d.invstd), _p(d.rm),
                                  _p(d.rv), _p(d.nb), _p(d.ws), count_mult, dt))
    _ran(names, _reduce_pat(_branch(M * C, C, dt, True), dt), r'bn_finalize_kernel')
    assert int(d.nb) == 8
    _check_stats('bn/stats', f'bn_stats C{C} x{count_mult}', x, d.mean, d.invstd, d.rm, d.rv, d.rm0, d.rv0, count_mult)

    d = _BnDev(M, C, dt, False, C)
    sums = torch.cat([x.sum(0), (x * x).sum(0)]).cuda()
    y = _buf(M * C, dt)
    names = kernels(lambda: _call('ttg_bn_act_fwd_stats', _p(dx), _p(y), M, C, _p(sums), _p(d.d_gamma),
                                  _p(d.d_beta), EPS, MOM, SLOPE, _p(d.mean), _p(d.invstd), _p(d.rm), _p(d.rv),
                                  _p(d.nb), count_mult, None, dt))
    _not_ran(names, r'chan_reduce')
    assert int(d.nb) == 8
    _check_stats('bn/stats', f'producer sums C{C} x{count_mult}', x, d.mean, d.invstd, d.rm, d.rv, d.rm0, d.rv0,
                 count_mult, k=1)


def test_bn_eval(kernels):
    """Eval mode: ttg_bn_eval_stats + ttg_bn_act_fwd against F.batch_norm(training=False)."""
    M, C, dt = 4096, 64, BF16
    x = _bn_input(M, C, dt)
    d = _BnDev(M, C, dt, False, 3)
    dx, y = _dev(x, dt), _buf(M * C, dt)

    def run():
        _call('ttg_bn_eval_stats', _p(d.rm), _p(d.rv), EPS, C, _p(d.mean), _p(d.invstd))
        _call('ttg_bn_act_fwd', _p(dx), _p(y), M, C, _p(d.mean), _p(d.invstd), _p(d.d_gamma), _p(d.d_beta), SLOPE, dt)
    _ran(kernels(run), r'bn_eval_stats_kernel', _map_pat('vec', dt))
    r_ref = (d.rv0 + EPS).rsqrt()
    _exact('bn/eval', 'mean', _host(d.mean), d.rm0)
    _check('bn/eval', 'invstd', _host(d.invstd), r_ref, 4 * U * r_ref)   # rsqrtf: <= 2 ulp
    y_ref = F.leaky_relu(F.batch_norm(x, d.rm0, d.rv0, d.gamma, d.beta, training=False, eps=EPS), SLOPE)
    a = d.gamma * r_ref
    A = (x * a).abs() + (d.rm0 * a).abs() + d.beta.abs()
    _check('bn/eval', 'y', _host(y, (M, C)), y_ref, _bar(y_ref, dt, A, 2 * K_EXPR))


# ------------------------------------------------------------------------------------------ element-wise maps
ELU = (1.0, 1.0)
SELU = (1.6732632423543772, 1.0507009873554805)


def _elu_f(x, ab):
    alpha, scale = (float(torch.tensor(v, dtype=torch.float32)) for v in ab)
    return F.selu(x) if ab is SELU else scale * F.elu(x, alpha)


EW_SIZES = {'bulk': (8 * 512 * 148 + 24, BF16, False), 'reg': (8000, BF16, False), 'odd': (8001, BF16, False),
            'mis': (8000, BF16, True), 'f32': (8000, F32, False), 'f32odd': (8001, F32, False)}
EW_OPS = ['lrelu_fwd', 'lrelu_bwd', 'elu_fwd', 'elu_bwd', 'elu_bwd2', 'selu_bwd2', 'axpby']


@pytest.mark.parametrize('size', list(EW_SIZES))
@pytest.mark.parametrize('op', EW_OPS)
def test_eltwise(op, size, kernels):
    """ttg_lrelu_*, ttg_elu_* and ttg_axpby: launch_chan_map with C = 8 (n % 8 == 0) or 1, against torch float64."""
    n, dt, mis = EW_SIZES[size]
    g = torch.Generator().manual_seed(n + len(op))
    x, gg, u = (_q(2 * torch.randn(n, generator=g, dtype=torch.float64), dt) for _ in range(3))
    dx, dg, du, out = _dev(x, dt, mis), _dev(gg, dt, mis), _dev(u, dt, mis), _buf(n, dt, mis)
    xr = x.clone().requires_grad_()
    ab = SELU if op.startswith('selu') else ELU
    abf = [float(torch.tensor(v, dtype=torch.float32)) for v in ab]
    expk = 1 + 4 * x.abs()                      # __expf: 2 + 1.2 |x| ulp
    if op == 'lrelu_fwd':
        fn = lambda: _call('ttg_lrelu_fwd', _p(dx), _p(out), n, SLOPE, dt)
        ref, A = F.leaky_relu(x, SLOPE), x.abs()
    elif op == 'lrelu_bwd':
        fn = lambda: _call('ttg_lrelu_bwd', _p(dx), _p(dg), _p(out), n, SLOPE, dt)
        ref, = torch.autograd.grad(F.leaky_relu(xr, SLOPE), xr, gg)
        A = gg.abs()
    elif op == 'elu_fwd':
        fn = lambda: _call('ttg_elu_fwd', _p(dx), _p(out), n, abf[0], abf[1], dt)
        ref = _elu_f(x, ab)
        A = 4 * ref.abs() + 4 * abf[0] * abf[1] * x.abs().clamp_max(1)
    elif op == 'elu_bwd':
        fn = lambda: _call('ttg_elu_bwd', _p(dx), _p(dg), _p(out), n, abf[0], abf[1], dt)
        ref, = torch.autograd.grad(_elu_f(xr, ab), xr, gg)
        A = expk * ref.abs()
    else:                                         # d/dx of <g f'(x), u> = g u f''(x)
        fn = lambda: _call('ttg_elu_bwd2', _p(dx), _p(dg), _p(du), _p(out), n, abf[0], abf[1], dt)
        gr = gg.clone().requires_grad_()
        gx, = torch.autograd.grad(_elu_f(xr, ab), xr, gr, create_graph=True)
        ref, = torch.autograd.grad(gx, xr, u)
        A = expk * ref.abs()
    if op == 'axpby':
        al, be = 0.75, -1.25
        fn = lambda: _call('ttg_axpby', _p(dx), _p(dg), _p(out), n, al, be, dt)
        ref, A = al * x + be * gg, (al * x).abs() + (be * gg).abs()
    names = kernels(fn)
    aligned = not mis
    if op == 'axpby' and (dt == F32 or not aligned or n % 8):
        _ran(names, rf'axpby_kernel<{TNAME[dt]}, {VN[dt] if aligned and n % VN[dt] == 0 else 1}>')
    else:
        _ran(names, _map_pat(_branch(n, 8 if n % 8 == 0 else 1, dt, aligned), dt))
    _check(f'eltwise/{op}', size, _host(out), ref, _bar(ref, dt, A))


# ------------------------------------------------------------------------------------------------- resampling
def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _img(N, H, W, C, dt, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return _q(scale * torch.randn(N, H, W, C, generator=g, dtype=torch.float64), dt)


def _vec_pat(kernel, dt, aligned_vec):
    return rf'{kernel}<{TNAME[dt]}, {VN[dt] if aligned_vec else 1}[,>]'


# (N, H, W, C, dtype, misaligned): H, W of the larger side
RS_CASES = {'x8-C16': (2, 32, 32, 16, BF16, False), 'x8-C128': (2, 16, 16, 128, BF16, False),
            'x8-C256': (1, 8, 8, 256, BF16, False), 'scalar-C3': (2, 64, 64, 3, BF16, False),
            'scalar-mis-C16': (2, 32, 32, 16, BF16, True), 'f32-vec-C16': (2, 32, 32, 16, F32, False),
            'f32-scalar-C3': (2, 64, 64, 3, F32, False), 'f32-scalar-mis-C16': (2, 16, 16, 16, F32, True)}


@pytest.mark.parametrize('scale', [1.0, 0.25, 0.7])
@pytest.mark.parametrize('case', list(RS_CASES))
def test_pool2_upsample2(case, scale, kernels):
    """ttg_pool2_sum (scale * 2x2 sum) against F.avg_pool2d, ttg_upsample2 against F.interpolate(nearest)."""
    N, H, W, C, dt, mis = RS_CASES[case]
    aligned_vec = not mis and C % VN[dt] == 0
    x8 = dt == BF16 and aligned_vec
    x = _img(N, H, W, C, dt, H + C)
    dx, y = _dev(x, dt, mis), _buf(N * H * W * C // 4, dt, mis)
    names = kernels(lambda: _call('ttg_pool2_sum', _p(dx), _p(y), N, H // 2, W // 2, C, scale, dt))
    _ran(names, r'pool2_bf16x8_kernel' if x8 else _vec_pat('pool2_kernel', dt, aligned_vec))
    ref = _nhwc(F.avg_pool2d(_nchw(x), 2)) * 4 * scale
    A = _nhwc(F.avg_pool2d(_nchw(x.abs()), 2)) * 4 * scale
    _check(f'resample/pool2{"-x8" if x8 else ""}', f'{case} scale {scale}', _host(y), ref, _bar(ref, dt, A))

    s = _img(N, H // 2, W // 2, C, dt, H + C + 1)
    ds, y = _dev(s, dt, mis), _buf(N * H * W * C, dt, mis)
    names = kernels(lambda: _call('ttg_upsample2', _p(ds), _p(y), N, H // 2, W // 2, C, scale, dt))
    _ran(names, r'upsample2_bf16x8_kernel' if x8 else _vec_pat('upsample2_kernel', dt, aligned_vec))
    ref = _nhwc(F.interpolate(_nchw(s), scale_factor=2, mode='nearest')) * scale
    if scale == 1.0:
        _exact('resample/upsample2', f'{case} scale 1', _host(y), ref)
    else:
        _check('resample/upsample2', f'{case} scale {scale}', _host(y), ref, _bar(ref, dt, ref.abs()))


def _bil_ref(x, Ho, Wo):
    return _nhwc(F.interpolate(_nchw(x), size=(Ho, Wo), mode='bilinear', align_corners=True))


def _bil_bwd_ref(gy, H, W):
    """B^T gy: the vector-Jacobian product of the align_corners bilinear resize H x W -> H/2 x W/2."""
    xr = torch.zeros(gy.shape[0], gy.shape[3], H, W, dtype=torch.float64, requires_grad=True)
    yr = F.interpolate(xr, size=(H // 2, W // 2), mode='bilinear', align_corners=True)
    g, = torch.autograd.grad(yr, xr, _nchw(gy))
    return _nhwc(g)


BIL_CASES = {  # (N, H, W, C, dtype, misaligned, bwd work item)
    'vec-pixel-C16': (2, 32, 32, 16, BF16, False, 'pixel'), 'vec-vector-C64': (2, 16, 16, 64, BF16, False, 'vector'),
    'vec-vector-C256': (1, 8, 8, 256, BF16, False, 'vector'), 'scalar-pixel-C3': (2, 64, 64, 3, BF16, False, 'pixel'),
    'scalar-pixel-mis-C16': (2, 16, 16, 16, BF16, True, 'pixel'),
    'scalar-vector-mis-C32': (2, 16, 16, 32, BF16, True, 'vector'),
    'f32-vec-pixel-C16': (2, 16, 16, 16, F32, False, 'pixel'), 'f32-vec-vector-C64': (2, 16, 16, 64, F32, False, 'vector'),
    'f32-scalar-vector-C18': (2, 16, 16, 18, F32, False, 'vector'), 'rect-C16': (2, 12, 40, 16, BF16, False, 'pixel')}


@pytest.mark.parametrize('add', [False, True], ids=['plain', 'add'])
@pytest.mark.parametrize('case', list(BIL_CASES))
def test_bilinear(case, add, kernels):
    """ttg_bilinear_down_fwd against F.interpolate(bilinear, align_corners=True); ttg_bilinear_down_bwd_add (the D
    block's gradient fan-in: add + B^T gy) against add + the vector-Jacobian product of that interpolate."""
    N, H, W, C, dt, mis, item = BIL_CASES[case]
    aligned_vec = not mis and C % VN[dt] == 0
    assert (C >= 32 if aligned_vec else C > 16) == (item == 'vector')
    x = _img(N, H, W, C, dt, H * C)
    dx, y = _dev(x, dt, mis), _buf(N * H * W * C // 4, dt, mis)
    names = kernels(lambda: _call('ttg_bilinear_down_fwd', _p(dx), _p(y), N, H, W, C, dt))
    _ran(names, _vec_pat('bilinear_down_kernel', dt, aligned_vec))
    ref = _bil_ref(x, H // 2, W // 2)
    A = _bil_ref(x.abs(), H // 2, W // 2) + max(H, W) * x.abs().max()
    if not add:
        _check('resample/bilinear-fwd', case, _host(y), ref, _bar(ref, dt, A))

    gy = _img(N, H // 2, W // 2, C, dt, H * C + 1)
    ad = _img(N, H, W, C, dt, H * C + 2) if add else None
    dgy, dad, gx = _dev(gy, dt, mis), (_dev(ad, dt, mis) if add else None), _buf(N * H * W * C, dt, mis)
    names = kernels(lambda: _call('ttg_bilinear_down_bwd_add', _p(dgy), _p(dad), _p(gx), N, H, W, C, dt))
    _ran(names, _vec_pat('bilinear_down_bwd_kernel', dt, aligned_vec))
    ref = _bil_bwd_ref(gy, H, W) + (ad if add else 0)
    A = _bil_bwd_ref(gy.abs(), H, W) + (ad.abs() if add else 0) + 9 * max(H, W) * gy.abs().max()
    _check(f'resample/bilinear-bwd-{item}', f'{case} {"add" if add else "plain"}', _host(gx), ref, _bar(ref, dt, A))


@pytest.mark.parametrize('rows', [True, False], ids=['H-sweep', 'W-sweep'])
def test_bilinear_candidate_sweep(rows, kernels):
    """The per-row / per-column candidate tables of the transpose, at every even size 2..256 of one side."""
    C, dt, fixed = 8, BF16, 6
    worst = 0.0
    for s in range(2, 257, 2):
        H, W = (s, fixed) if rows else (fixed, s)
        gy = _img(1, H // 2, W // 2, C, dt, s)
        dgy, gx = _dev(gy, dt), _buf(H * W * C, dt)
        _call('ttg_bilinear_down_bwd_add', _p(dgy), None, _p(gx), 1, H, W, C, dt)
        ref = _bil_bwd_ref(gy, H, W)
        A = _bil_bwd_ref(gy.abs(), H, W) + 9 * max(H, W) * gy.abs().max()
        got, bar = _host(gx), _bar(ref, dt, A)
        err = (got - ref.reshape(-1)).abs()
        worst = max(worst, float((err / bar.reshape(-1).clamp_min(1e-300)).max()))
        assert bool((err <= bar.reshape(-1)).all()), (H, W, int((err > bar.reshape(-1)).sum()))
    print(f'[stream] resample/bilinear-sweep {"H" if rows else "W"} 2..256: worst |err|/bar {worst:.3g}')
    _ran(kernels(lambda: _call('ttg_bilinear_down_bwd_add', _p(dgy), None, _p(gx), 1, H, W, C, dt)),
         _vec_pat('bilinear_down_bwd_kernel', dt, True))


def test_bilinear_smem_limit():
    """Candidate tables larger than 48 KB are refused with an error; the largest size that fits still works."""
    from tartangan_b200 import _lib as lib
    C, dt = 8, BF16
    H, W = 1024, 340                                          # (H + W) * 36 = 49104 <= 49152
    gy = _img(1, H // 2, W // 2, C, dt, 1)
    dgy, gx = _dev(gy, dt), _buf(H * W * C, dt)
    _call('ttg_bilinear_down_bwd_add', _p(dgy), None, _p(gx), 1, H, W, C, dt)
    ref = _bil_bwd_ref(gy, H, W)
    A = _bil_bwd_ref(gy.abs(), H, W) + 9 * max(H, W) * gy.abs().max()
    _check('resample/bilinear-bwd-pixel', f'{H}x{W}', _host(gx), ref, _bar(ref, dt, A))
    W = 342                                                   # 49176 bytes
    # operands sized for this shape, so that the call stays in bounds even if the size check were lost
    dgy2, gx2 = _buf(H // 2 * (W // 2) * C, dt, fill=0.0), _buf(H * W * C, dt)
    with pytest.raises(RuntimeError, match='too large'):
        _call('ttg_bilinear_down_bwd_add', _p(dgy2), None, _p(gx2), 1, H, W, C, dt)
    torch.cuda.synchronize()
    assert bool(gx2.isnan().all()), 'a refused call must not write'
    assert lib.last_error()


# ---------------------------------------------------------------------------------------------------------- joins
JOIN_CASES = {'vec-C128': (2, 8, 8, 128, BF16, False), 'vec-C16': (2, 32, 32, 16, BF16, False),
              'vec-C64': (2, 16, 16, 64, BF16, False), 'scalar-C3': (2, 32, 32, 3, BF16, False),
              'scalar-C100': (2, 16, 16, 100, BF16, False), 'scalar-mis-C16': (2, 16, 16, 16, BF16, True),
              'f32-vec-C16': (2, 16, 16, 16, F32, False), 'f32-scalar-C6': (2, 16, 16, 6, F32, False)}


def _join(kind, N, Ho, Wo, C, dt, seed):
    """-> (h, s, reference, A) of add_up2 (h + up(s), at Ho x Wo) or pool2_add (0.25 sum4(h) + s)."""
    if kind == 'add_up2':
        h, s = _img(N, Ho, Wo, C, dt, seed), _img(N, Ho // 2, Wo // 2, C, dt, seed + 1)
        up = _nhwc(F.interpolate(_nchw(s), scale_factor=2, mode='nearest'))
        return h, s, h + up, h.abs() + up.abs()
    h, s = _img(N, 2 * Ho, 2 * Wo, C, dt, seed), _img(N, Ho, Wo, C, dt, seed + 1)
    return h, s, _nhwc(F.avg_pool2d(_nchw(h), 2)) + s, _nhwc(F.avg_pool2d(_nchw(h.abs()), 2)) + s.abs()


@pytest.mark.parametrize('kind', ['add_up2', 'pool2_add'])
@pytest.mark.parametrize('case', list(JOIN_CASES))
def test_joins(kind, case, kernels):
    N, Ho, Wo, C, dt, mis = JOIN_CASES[case]
    aligned_vec = not mis and C % VN[dt] == 0
    h, s, ref, A = _join(kind, N, Ho, Wo, C, dt, Ho * C)
    dh, ds, y = _dev(h, dt, mis), _dev(s, dt, mis), _buf(N * Ho * Wo * C, dt, mis)
    args = (N, Ho, Wo, C) + ((0.25,) if kind == 'pool2_add' else ()) + (dt,)
    names = kernels(lambda: _call(f'ttg_{kind}', _p(dh), _p(ds), _p(y), *args))
    _ran(names, rf'{kind}_kernel<{TNAME[dt]}, {VN[dt] if aligned_vec else 1}, false>')
    _check(f'join/{kind}', case, _host(y), ref, _bar(ref, dt, A))


@pytest.mark.parametrize('kind', ['add_up2', 'pool2_add'])
@pytest.mark.parametrize('C', [8, 16, 32, 64, 128, 256])
def test_join_stats(kind, C, kernels):
    """The joins that also reduce the BatchNorm sums of their output: the sums are those of the STORED bf16 values."""
    dt, N, Ho, Wo = BF16, 2, 32, 32
    h, s, ref, A = _join(kind, N, Ho, Wo, C, dt, C)
    dh, ds, y = _dev(h, dt), _dev(s, dt), _buf(N * Ho * Wo * C, dt)
    sums = torch.full((2 * C,), 1e30, dtype=torch.float64, device='cuda')
    args = (N, Ho, Wo, C) + ((0.25,) if kind == 'pool2_add' else ()) + (_p(sums), dt)
    names = kernels(lambda: _call(f'ttg_{kind}_stats', _p(dh), _p(ds), _p(y), *args))
    _ran(names, rf'{kind}_kernel<{TNAME[dt]}, 8, true>')
    got = _host(y, (-1, C))
    _check(f'join/{kind}', f'stats C{C} y', got, ref.reshape(-1, C), _bar(ref.reshape(-1, C), dt, A.reshape(-1, C)))
    sm = _host(sums)
    _check(f'join/{kind}-stats', f'C{C} sum', sm[:C], got.sum(0), L_SUM * U * got.abs().sum(0))
    _check(f'join/{kind}-stats', f'C{C} sum of squares', sm[C:], (got * got).sum(0), L_SUM * U * (got * got).sum(0))


@pytest.mark.parametrize('kind', ['add_up2', 'pool2_add'])
@pytest.mark.parametrize('C', [120, 512])
def test_join_stats_fallback(kind, C, kernels):
    """A width ttg_join_stats_supported rejects: ops runs the plain join, leaves no producer statistics, and the
    following BatchNorm reduces its own (two passes)."""
    import tartangan_b200 as tb
    from tartangan_b200 import ops
    tb.set_precision('bf16')
    dt, N, Ho, Wo = BF16, 2, 8, 8
    h, s, ref, A = _join(kind, N, Ho, Wo, C, dt, C)
    to = lambda t: t.to(torch.bfloat16).cuda().permute(0, 3, 1, 2)       # NHWC memory, logical NCHW
    assert not ops._join_stats_ok(to(s))
    bn = torch.nn.BatchNorm2d(C).cuda()
    out = {}

    def run():
        ops.state.producer_stats = None
        y = ops.add_up2(to(h), to(s)) if kind == 'add_up2' else ops.avg_pool2_add(to(h), to(s))
        assert ops.state.producer_stats is None
        out['y'] = y
        out['a'] = ops.bn_act(y, bn)
    names = kernels(run)
    _ran(names, rf'{kind}_kernel<{TNAME[dt]}, 8, false>', _reduce_pat('vec', dt), _map_pat('vec', dt))
    _not_ran(names, rf'{kind}_kernel<[^>]*true>')
    y = _host(out['y'].permute(0, 2, 3, 1))
    _check(f'join/{kind}', f'fallback C{C}', y, ref, _bar(ref, dt, A))
    yq = y.reshape(-1, C)
    a_ref = F.leaky_relu(F.batch_norm(yq, None, None, training=True, eps=bn.eps), SLOPE)
    # (statistics in float64 here: compared at the bf16 output resolution plus the statistics' fp32 bound)
    A = (yq - yq.mean(0)).abs() * (yq.var(0, unbiased=False) + bn.eps).rsqrt() + 1
    _check(f'join/{kind}', f'fallback C{C} bn_act', _host(out['a'].permute(0, 2, 3, 1)).reshape(-1, C), a_ref,
           _bar(a_ref, dt, A, 4 * L_SUM))


# --------------------------------------------------------------------------------------------------------- layout
LAYOUT_CASES = {'elem-C128': (4, 128, 16, BF16), 'elem-C16-f32': (2, 16, 256, F32), 'rgb': (2, 3, 64 * 64, BF16),
                'pixel-C3-f32': (2, 3, 32 * 32, F32), 'pixel-C3-odd': (2, 3, 33 * 31, BF16),
                'pixel-C16-large': (2, 16, 32 * 32, BF16), 'pixel-C8': (2, 8, 16 * 16, BF16)}


@pytest.mark.parametrize('case', list(LAYOUT_CASES))
def test_layout(case, kernels):
    """ttg_nchw_to_nhwc (fp32 NCHW -> NHWC, rounding like torch's cast) and ttg_nhwc_to_nchw: bit-exact."""
    N, C, HW, dt = LAYOUT_CASES[case]
    g = torch.Generator().manual_seed(HW + C)
    x = torch.randn(N, C, HW, generator=g, dtype=torch.float32) * 3       # fp32: many values not exact in bf16
    dx, y = x.cuda(), _buf(N * HW * C, dt)
    names = kernels(lambda: _call('ttg_nchw_to_nhwc', _p(dx), _p(y), N, C, HW, dt))
    rgb = C == 3 and HW % 8 == 0 and dt == BF16
    pat = (r'nchw_to_nhwc_elem_kernel<' if C >= 16 and HW <= 256 else
           r'nchw_to_nhwc_rgb_bf16_kernel' if rgb else rf'nchw_to_nhwc_kernel<{TNAME[dt]}>')
    _ran(names, pat)
    ref = x.permute(0, 2, 1).to(TORCH_DT[dt])
    _exact('layout', f'{case} to nhwc', _host(y), ref.double())

    z = _buf(N * C * HW, torch.float32)
    names = kernels(lambda: _call('ttg_nhwc_to_nchw', _p(y), _p(z), N, C, HW, dt))
    _ran(names, r'nhwc_to_nchw_rgb_bf16_kernel' if rgb else rf'nhwc_to_nchw_kernel<{TNAME[dt]}>')
    _exact('layout', f'{case} to nchw', _host(z), ref.permute(0, 2, 1).double())


@pytest.mark.parametrize('C,dt', [(128, BF16), (16, BF16), (3, BF16), (64, F32)])
def test_spatial(C, dt, kernels):
    """ttg_spatial_sum (sum over H, W; fp32 out) and ttg_spatial_bcast (its adjoint; a cast, bit-exact)."""
    N, HW = 3, 16 * 16
    x = _img(N, 16, 16, C, dt, C).reshape(N, HW, C)
    dx, out = _dev(x, dt), _buf(N * C, torch.float32)
    _ran(kernels(lambda: _call('ttg_spatial_sum', _p(dx), _p(out), N, HW, C, dt)), rf'spatial_sum_kernel<{TNAME[dt]}>')
    _check('layout/spatial_sum', f'C{C}', _host(out, (N, C)), x.sum(1), HW * U * x.abs().sum(1))
    g = torch.randn(N, C, dtype=torch.float32) * 3
    dg, gx = g.cuda(), _buf(N * HW * C, dt)
    _ran(kernels(lambda: _call('ttg_spatial_bcast', _p(dg), _p(gx), N, HW, C, dt)),
         rf'spatial_bcast_kernel<{TNAME[dt]}>')
    _exact('layout/spatial_bcast', f'C{C}', _host(gx), g.to(TORCH_DT[dt]).double()[:, None, :].expand(N, HW, C))


# ------------------------------------------------------------------------------------------------------- max-pool
def _maxpool_case(x, dt, kernels, tag):
    """x: NHWC float64 (values exact in dt).  fwd / scatter / gather against F.max_pool2d with indices and its
    first and second derivatives, all bit-exact."""
    N, H, W, C = x.shape
    Ho, Wo = H // 2, W // 2
    dx, y, idx = _dev(x, dt), _buf(N * Ho * Wo * C, dt), torch.full((N * Ho * Wo * C,), 255, dtype=torch.uint8,
                                                                     device='cuda')
    _ran(kernels(lambda: _call('ttg_maxpool2_fwd', _p(dx), _p(y), _p(idx), N, Ho, Wo, C, dt)),
         rf'maxpool2_fwd_kernel<{TNAME[dt]}>')
    xr = _nchw(x).contiguous().requires_grad_()
    y_ref, i_ref = F.max_pool2d(xr, 2, return_indices=True)
    _exact('maxpool', f'{tag} fwd', _host(y), _nhwc(y_ref.detach()))
    # torch's flat index h * W + w -> the kernel's window position (dy * 2 + dx)
    win = (i_ref // W % 2) * 2 + i_ref % W % 2
    _exact('maxpool', f'{tag} argmax', _host(idx), _nhwc(win))

    g = torch.Generator().manual_seed(N * H)
    gy, v = (_q(torch.randn(N, Ho, Wo, C, generator=g, dtype=torch.float64), dt) for _ in range(2))
    dgy, gx = _dev(gy, dt), _buf(N * H * W * C, dt)
    _ran(kernels(lambda: _call('ttg_maxpool2_scatter', _p(dgy), _p(idx), _p(gx), N, Ho, Wo, C, dt)),
         rf'maxpool2_scatter_kernel<{TNAME[dt]}>')
    gyr = _nchw(gy).contiguous().requires_grad_()
    gx_ref, = torch.autograd.grad(y_ref, xr, gyr, create_graph=True)
    _exact('maxpool', f'{tag} scatter', _host(gx), _nhwc(gx_ref.detach()))
    # the second derivative: d/d gy of <gx, u> gathers u at the argmax
    u = _q(torch.randn(N, H, W, C, generator=g, dtype=torch.float64), dt)
    du, z = _dev(u, dt), _buf(N * Ho * Wo * C, dt)
    _ran(kernels(lambda: _call('ttg_maxpool2_gather', _p(du), _p(idx), _p(z), N, Ho, Wo, C, dt)),
         rf'maxpool2_gather_kernel<{TNAME[dt]}>')
    z_ref, = torch.autograd.grad(gx_ref, gyr, _nchw(u).contiguous())
    _exact('maxpool', f'{tag} gather', _host(z), _nhwc(z_ref))


@pytest.mark.parametrize('N,H,W,C,dt', [(2, 16, 16, 64, BF16), (2, 32, 32, 16, F32), (2, 8, 8, 3, BF16)])
def test_maxpool_ties(N, H, W, C, dt, kernels):
    """Integer-valued inputs: most windows tie; the first maximum in window order wins, as in torch."""
    g = torch.Generator().manual_seed(C)
    x = torch.randint(-2, 3, (N, H, W, C), generator=g).double()
    _maxpool_case(x, dt, kernels, f'ties {N}x{H}x{W}x{C}')


@pytest.mark.parametrize('dt', [BF16, F32], ids=['bf16', 'f32'])
def test_maxpool_nan(dt, kernels):
    """A NaN in any window position propagates to the output and takes the index, as in torch; windows with two
    NaNs take the last one (torch tests `v > max || isnan(v)`)."""
    N, H, W, C = 2, 8, 8, 16
    g = torch.Generator().manual_seed(5)
    x = torch.randint(-2, 3, (N, H, W, C), generator=g).double()
    for c in range(C):              # channel c: a NaN at window position c % 4, and for c >= 8 a second one
        pos = [c % 4] + ([(c % 4 + 1 + c % 3) % 4] if c >= 8 else [])
        for p in pos:
            x[0, p // 2::2, p % 2::2, c] = NAN
    _maxpool_case(x, dt, kernels, f'nan {TNAME[dt]}')
