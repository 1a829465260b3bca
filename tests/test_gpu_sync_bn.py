"""The split BatchNorm + LeakyReLU entry points of synchronised BatchNorm (--sync-bn), on one GPU.

A batch of M rows is cut into k equal shards.  Each shard runs the reduce entry point on its own rows; the shards' fp64
sums are added on the device, which is what the all-reduce over k ranks computes; then each shard runs the apply entry
point with the global count and param_scale = 1 / k.  The concatenated outputs, and the parameter gradients summed over
the shards (what the gradient all-reduce computes), are compared with float64 on the CPU over the WHOLE batch, from the
bf16 / fp32 operands the kernels received.  With k = 1 the split entry points must reproduce the combined ones bit for bit.

Bars are those of tests/test_gpu_stream_kernels.py (fp32 partial sums of at most 64 terms, combined in fp64; see its
docstring) over the global batch.  The k per-shard parameter gradients each round once (param_scale * global sum) and
are then added in fp32, hence (k + 2) u of the result on top.
"""
import pytest
import torch
import torch.nn.functional as F

import test_gpu_stream_kernels as S
from test_gpu_stream_kernels import BF16, EPS, F32, L_SUM, MOM, TORCH_DT, U, _buf, _call, _dev, _host, _p

pytestmark = pytest.mark.gpu


def _rows(C):
    # not a multiple of the bulk kernels' 4096-element chunk; C = 3 needs M % 8 == 0 for the c3 kernels; at C >= 64 a
    # bf16 shard is above the bulk threshold (8 * 512 * 148 elements)
    return 9480 if C == 3 else 9475


def _stats_check(tag, x, mean, invstd, rm, rv, rm0, rv0, count_mult, extra=0.0):
    """S._check_stats with count_mult 1 or 4; extra: relative slack of sums taken before rounding to the dtype."""
    Mu = x.shape[0] * count_mult
    mean_ref, var_ref = x.mean(0), x.var(0, unbiased=False)
    rm_ref = (1 - MOM) * rm0 + MOM * mean_ref
    rv_ref = (1 - MOM) * rv0 + MOM * var_ref * Mu / (Mu - 1)
    dm, dr, drm, drv = S._stats_bars(x, mean_ref, Mu, rm0, rv0)
    if extra:
        ea, e2 = x.abs().mean(0), (x * x).mean(0)
        dvar = extra * (e2 + 2 * mean_ref.abs() * ea)
        r = (var_ref + EPS).rsqrt()
        dm, dr = dm + extra * ea, dr + 0.5 * r ** 3 * dvar
        drm, drv = drm + MOM * extra * ea, drv + MOM * dvar * Mu / (Mu - 1)
    S._check('sync', f'{tag} mean', _host(mean), mean_ref, dm)
    S._check('sync', f'{tag} invstd', _host(invstd), (var_ref + EPS).rsqrt(), dr)
    S._check('sync', f'{tag} running_mean', _host(rm), rm_ref, drm)
    S._check('sync', f'{tag} running_var', _host(rv), rv_ref, drv)


def _same(tag, tensors):
    for t in tensors[1:]:
        assert torch.equal(t, tensors[0]), f'{tag}: shards disagree'


def _ws(n, zero):
    """fp64 workspace of n sums: pre-zeroed (flag 2) or full of garbage the reduce must clear (flag 0)."""
    return (torch.zeros(n, dtype=torch.float64, device='cuda'), 2) if zero else \
        (torch.full((n,), 1e30, dtype=torch.float64, device='cuda'), 0)


def _forward(x, dx, Ms, k, C, dt, slope, count_mult, sums_of, tag, extra=0.0):
    """Sharded forward: per-shard sums (sums_of(r)), added, then ttg_bn_act_fwd_stats_n per shard.  -> (mean, invstd)."""
    M = k * Ms
    tot = sum(sums_of(r) for r in range(k))
    g = torch.Generator().manual_seed(C + k)
    gamma = (1 + 0.3 * torch.randn(C, generator=g, dtype=torch.float64)).float().double()
    beta = (0.3 * torch.randn(C, generator=g, dtype=torch.float64)).float().double()
    rm0 = torch.randn(C, generator=g, dtype=torch.float64).float().double()
    rv0 = (0.5 + torch.rand(C, generator=g, dtype=torch.float64)).float().double()
    y = _buf(M * C, dt)
    d_gamma, d_beta = gamma.float().cuda(), beta.float().cuda()
    outs = []
    for r in range(k):
        mean, invstd = _buf(C, torch.float32), _buf(C, torch.float32)
        rm, rv = rm0.float().cuda(), rv0.float().cuda()
        nb = torch.full((1,), 7, dtype=torch.int64, device='cuda')
        _call('ttg_bn_act_fwd_stats_n', _p(dx[r * Ms * C:]), _p(y[r * Ms * C:]), Ms, C, M, _p(tot),
              _p(d_gamma), _p(d_beta), EPS, MOM, slope, _p(mean), _p(invstd), _p(rm), _p(rv),
              _p(nb), count_mult, None, dt)
        assert int(nb) == 8
        outs.append((mean, invstd, rm, rv))
    for i, name in enumerate(('mean', 'invstd', 'running_mean', 'running_var')):
        _same(f'{tag} {name}', [o[i] for o in outs])
    mean, invstd, rm, rv = outs[0]
    _stats_check(tag, x, mean, invstd, rm, rv, rm0, rv0, count_mult, extra)
    mk, rk = _host(mean), _host(invstd)
    a = gamma * rk
    y_ref = F.leaky_relu(x * a + (beta - mk * a), slope)
    A_y = (x * a).abs() + (mk * a).abs() + beta.abs()
    S._check('sync', f'{tag} y', _host(y, (M, C)), y_ref, S._bar(y_ref, dt, A_y))
    return mean, invstd, gamma, beta


def _bn_ref(x, mk, rk, gamma, beta, ga, u, slope):
    """S._bn_ref with a LeakyReLU slope argument."""
    xr, g, b, gar = (t.clone().requires_grad_() for t in (x, gamma, beta, ga))
    mt = xr.mean(0)
    vt = ((xr - mt) ** 2).mean(0)
    m = mk + (mt - mt.detach())
    v = (rk.pow(-2) - EPS) + (vt - vt.detach())
    a = F.leaky_relu(g * (xr - m) * (v + EPS).rsqrt() + b, slope)
    gx, gg, gb = torch.autograd.grad(a, (xr, g, b), gar, create_graph=True)
    g_x, g_ga, gg2 = torch.autograd.grad(gx, (xr, gar, g), u)
    return (gx.detach(), gg.detach(), gb.detach()), (g_x, g_ga, gg2)


@pytest.mark.parametrize('k', [2, 3])
@pytest.mark.parametrize('slope', [0.2, 1.0])
@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('C', [3, 16, 64, 128])
def test_sharded_bn(C, dt, slope, k):
    Ms = _rows(C)
    M = k * Ms
    x = S._bn_input(M, C, dt, 0.3, seed=C + 7 * k)
    dx = _dev(x, dt)
    tag = f'C{C} {"bf16" if dt == BF16 else "f32"} slope {slope} k{k}'

    def bn_sums(r):
        ws, flag = _ws(2 * C, zero=r > 0)
        _call('ttg_bn_sums', _p(dx[r * Ms * C:]), Ms, C, _p(ws), flag, dt)
        return ws
    for cm in (1, 4):
        mean, invstd, gamma, beta = _forward(x, dx, Ms, k, C, dt, slope, cm, bn_sums, f'{tag} x{cm}')
    mk, rk = _host(mean), _host(invstd)
    d_gamma, d_beta = gamma.float().cuda(), beta.float().cuda()

    # backward: cotangents zeroed where the LeakyReLU mask depends on rounding
    g = torch.Generator().manual_seed(M + C)
    a = gamma * rk
    pre = x * a + (beta - mk * a)
    A_y = (x * a).abs() + (mk * a).abs() + beta.abs()
    amb = pre.abs() <= 1e-5 * A_y
    ga = S._q(torch.randn(M, C, generator=g, dtype=torch.float64).masked_fill(amb, 0), dt)
    u = S._q(torch.randn(M, C, generator=g, dtype=torch.float64), dt)
    (gx_ref, gg_ref, gb_ref), (g_x_ref, g_ga_ref, gg2_ref) = _bn_ref(x, mk, rk, gamma, beta, ga, u, slope)
    dga, du = _dev(ga, dt), _dev(u, dt)
    bn = (_p(mean), _p(invstd), _p(d_gamma), _p(d_beta), slope)

    sums = []
    for r in range(k):
        ws, flag = _ws(2 * C, zero=r % 2 == 1)
        _call('ttg_bn_act_bwd_reduce', _p(dx[r * Ms * C:]), _p(dga[r * Ms * C:]), Ms, C, *bn, _p(ws), flag, dt)
        sums.append(ws)
    tot = sum(sums)
    gx = _buf(M * C, dt)
    G0 = torch.randn(2, C, generator=g).cuda()
    acc = G0.clone()                                          # accumulate = 1: every shard adds its share
    over = [(_buf(C, torch.float32), _buf(C, torch.float32)) for _ in range(k)]      # accumulate = 0
    nogx = G0.clone()                                         # gx NULL: parameter gradients only
    for r in range(k):
        _call('ttg_bn_act_bwd_apply', _p(dx[r * Ms * C:]), _p(dga[r * Ms * C:]), _p(gx[r * Ms * C:]), Ms, C, M,
              _p(tot), *bn, _p(acc[0]), _p(acc[1]), 1.0 / k, 1, dt)
        _call('ttg_bn_act_bwd_apply', _p(dx[r * Ms * C:]), _p(dga[r * Ms * C:]), _p(gx[r * Ms * C:]), Ms, C, M,
              _p(tot), *bn, _p(over[r][0]), _p(over[r][1]), 1.0 / k, 0, dt)
        _call('ttg_bn_act_bwd_apply', None, None, None, Ms, C, M, _p(tot), *bn, _p(nogx[0]), _p(nogx[1]), 1.0 / k, 1, dt)
    X = (x.abs() + mk.abs()) * rk
    gr = (gamma * rk).abs()
    gaa, ua = ga.abs(), u.abs()
    mean_ = lambda t: t.mean(0)
    A_Pd = gaa + mean_(gaa) + X * mean_(gaa * X)
    A_Pu = ua + mean_(ua) + X * mean_(ua * X)
    S._check('sync', f'{tag} gx', _host(gx, (M, C)), gx_ref, S._bar(gx_ref, dt, gr * A_Pd, L_SUM))
    bar_g = L_SUM * U * (gaa * X).sum(0) + (k + 2) * U * gg_ref.abs()
    bar_b = L_SUM * U * gaa.sum(0) + (k + 2) * U * gb_ref.abs()
    G0h = _host(G0)
    for name, gg_, gb_, base in (('accumulate', acc[0], acc[1], G0h), ('overwrite', sum(o[0] for o in over),
                                 sum(o[1] for o in over), torch.zeros_like(G0h)), ('no gx', nogx[0], nogx[1], G0h)):
        S._check('sync', f'{tag} d gamma ({name})', _host(gg_) - base[0], gg_ref, bar_g + (k + 1) * U * base[0].abs())
        S._check('sync', f'{tag} d beta ({name})', _host(gb_) - base[1], gb_ref, bar_b + (k + 1) * U * base[1].abs())

    # double backward (R1)
    sums = []
    for r in range(k):
        ws, flag = _ws(5 * C, zero=r % 2 == 0)
        _call('ttg_bn_act_bwd2_reduce', _p(dx[r * Ms * C:]), _p(dga[r * Ms * C:]), _p(du[r * Ms * C:]), Ms, C, *bn,
              _p(ws), flag, dt)
        sums.append(ws)
    tot = sum(sums)
    g_ga, g_x = _buf(M * C, dt), _buf(M * C, dt)
    acc2 = G0[0].clone()
    over2 = [_buf(C, torch.float32) for _ in range(k)]
    for r in range(k):
        rows = lambda t: _p(t[r * Ms * C:])
        _call('ttg_bn_act_bwd2_apply', rows(dx), rows(dga), rows(du), rows(g_ga), rows(g_x), Ms, C, M, _p(tot), *bn,
              _p(acc2), 1.0 / k, 1, dt)
        _call('ttg_bn_act_bwd2_apply', rows(dx), rows(dga), rows(du), rows(g_ga), rows(g_x), Ms, C, M, _p(tot), *bn,
              _p(over2[r]), 1.0 / k, 0, dt)
    S._check('sync', f'{tag} bwd2 d ga', _host(g_ga, (M, C)), g_ga_ref, S._bar(g_ga_ref, dt, gr * A_Pu, L_SUM),
             mask=~amb)
    A_k = X * (mean_(gaa * X) * mean_(ua * X) + mean_(ua * gaa) + mean_(ua) * mean_(gaa))
    A_gx2 = gr * rk * (A_k + mean_(ua * X) * A_Pd + mean_(gaa * X) * A_Pu)
    S._check('sync', f'{tag} bwd2 d x', _host(g_x, (M, C)), g_x_ref, S._bar(g_x_ref, dt, A_gx2, L_SUM))
    A_gg2 = rk * M * (mean_(ua * gaa) + mean_(ua) * mean_(gaa) + mean_(gaa * X) * mean_(ua * X))
    bar = L_SUM * U * A_gg2 + (k + 2) * U * gg2_ref.abs()
    S._check('sync', f'{tag} bwd2 d gamma (accumulate)', _host(acc2) - G0h[0], gg2_ref, bar + (k + 1) * U * G0h[0].abs())
    S._check('sync', f'{tag} bwd2 d gamma (overwrite)', _host(sum(over2)), gg2_ref, bar)


@pytest.mark.parametrize('k', [2, 3])
@pytest.mark.parametrize('cout', [64, 128])
def test_sharded_bn_conv_sums(cout, k):
    """Forward statistics from the sums the tensor-core conv epilogue produces (ttg_conv2d_tc_stats), one conv per
    shard, against float64 statistics of the bf16 conv outputs."""
    from tartangan_b200 import ops
    ops.set_precision('bf16')
    n, hw, cin = 3, 16, 32
    g = torch.Generator().manual_seed(cout + k)
    w = (torch.randn(cout, cin, 3, 3, generator=g) / 12).cuda()
    assert ops.conv_stats_ok(w, 0, torch.bfloat16)
    ys, sums = [], []
    for r in range(k):
        xr = ops.to_internal(torch.randn(n, cin, hw, hw, generator=g).cuda())
        y = ops.conv2d(xr, w, None, stats=True)
        s = ops.take_producer_stats(y)
        assert s is not None
        ys.append(ops.nhwc(y).permute(0, 2, 3, 1).reshape(-1, cout))
        sums.append(s)
    Ms = n * hw * hw
    dy = torch.cat(ys).contiguous().view(-1)
    x = _host(dy, (k * Ms, cout))
    # the epilogue may sum the fp32 accumulators before their rounding to bf16: half a bf16 ulp of slack per moment
    _forward(x, dy, Ms, k, cout, BF16, 0.2, 1, lambda r: sums[r], f'conv sums C{cout} k{k}', extra=2.0 ** -8)


@pytest.mark.parametrize('dt', [F32, BF16])
@pytest.mark.parametrize('C', [3, 16, 64, 128])
def test_split_matches_combined_bitwise(C, dt):
    """k = 1: reduce + apply with count = M and param_scale = 1 give exactly what the combined entry points give."""
    M = _rows(C)
    x = S._bn_input(M, C, dt, 0.3, seed=C)
    dx = _dev(x, dt)
    g = torch.Generator().manual_seed(C + 1)
    ga, u = (_dev(S._q(torch.randn(M, C, generator=g, dtype=torch.float64), dt), dt) for _ in range(2))
    gamma = (1 + 0.3 * torch.randn(C, generator=g)).cuda()
    beta = (0.3 * torch.randn(C, generator=g)).cuda()
    G0 = torch.randn(3, C, generator=g).cuda()

    def run(split):
        o = dict(y=_buf(M * C, dt), mean=_buf(C, torch.float32), invstd=_buf(C, torch.float32),
                 rm=torch.zeros(C, device='cuda'), rv=torch.ones(C, device='cuda'),
                 nb=torch.zeros(1, dtype=torch.int64, device='cuda'), gx=_buf(M * C, dt), g=G0.clone(),
                 g_ga=_buf(M * C, dt), g_x=_buf(M * C, dt))
        st = (EPS, MOM, 0.2, _p(o['mean']), _p(o['invstd']), _p(o['rm']), _p(o['rv']), _p(o['nb']), 4)
        ws = torch.zeros(5 * C, dtype=torch.float64, device='cuda')
        if split:
            _call('ttg_bn_sums', _p(dx), M, C, _p(ws), 0, dt)
            _call('ttg_bn_act_fwd_stats_n', _p(dx), _p(o['y']), M, C, M, _p(ws), _p(gamma), _p(beta), *st, None, dt)
        else:
            _call('ttg_bn_act_fwd_stats', _p(dx), _p(o['y']), M, C, None, _p(gamma), _p(beta), *st, _p(ws), dt)
        bn = (_p(o['mean']), _p(o['invstd']), _p(gamma), _p(beta), 0.2)
        ws.zero_()
        if split:
            _call('ttg_bn_act_bwd_reduce', _p(dx), _p(ga), M, C, *bn, _p(ws), 2, dt)
            _call('ttg_bn_act_bwd_apply', _p(dx), _p(ga), _p(o['gx']), M, C, M, _p(ws), *bn, _p(o['g'][0]),
                  _p(o['g'][1]), 1.0, 1, dt)
            _call('ttg_bn_act_bwd2_reduce', _p(dx), _p(ga), _p(u), M, C, *bn, _p(ws), 0, dt)
            _call('ttg_bn_act_bwd2_apply', _p(dx), _p(ga), _p(u), _p(o['g_ga']), _p(o['g_x']), M, C, M, _p(ws), *bn,
                  _p(o['g'][2]), 1.0, 1, dt)
        else:
            _call('ttg_bn_act_bwd_acc', _p(dx), _p(ga), _p(o['gx']), M, C, *bn, _p(o['g'][0]), _p(o['g'][1]), 3,
                  _p(ws), dt)
            _call('ttg_bn_act_bwd2_acc', _p(dx), _p(ga), _p(u), _p(o['g_ga']), _p(o['g_x']), M, C, *bn,
                  _p(o['g'][2]), 1, _p(ws), dt)
        torch.cuda.synchronize()
        return o
    a, b = run(False), run(True)
    for key in a:
        assert torch.equal(a[key].view(torch.uint8) if a[key].dtype != torch.int64 else a[key],
                           b[key].view(torch.uint8) if b[key].dtype != torch.int64 else b[key]), key


def test_split_rejects_bad_counts():
    """count < M, and sums = NULL with a count other than M, are argument errors (no kernel runs)."""
    M, C = 64, 16
    x = _buf(M * C, F32, fill=0.0)
    y = _buf(M * C, F32)
    ws = torch.zeros(5 * C, dtype=torch.float64, device='cuda')
    v = torch.ones(C, device='cuda')
    st = (_p(v), _p(v), EPS, MOM, 0.2, _p(v.clone()), _p(v.clone()), None, None, None, 1)
    with pytest.raises(RuntimeError, match='bad arguments'):
        _call('ttg_bn_act_fwd_stats_n', _p(x), _p(y), M, C, M - 1, _p(ws), *st, None, F32)
    with pytest.raises(RuntimeError, match='count == M'):
        _call('ttg_bn_act_fwd_stats_n', _p(x), _p(y), M, C, 2 * M, None, *st, _p(ws), F32)
    with pytest.raises(RuntimeError, match='bad arguments'):
        _call('ttg_bn_act_bwd_apply', _p(x), _p(x), _p(y), M, C, M - 1, _p(ws), _p(v), _p(v), _p(v), _p(v), 0.2,
              None, None, 1.0, 0, F32)
    with pytest.raises(RuntimeError, match='bad arguments'):
        _call('ttg_bn_act_bwd2_apply', _p(x), _p(x), _p(x), _p(y), _p(y), M, C, M - 1, _p(ws), _p(v), _p(v), _p(v),
              _p(v), 0.2, None, 1.0, 0, F32)
