"""Micro-benchmark of single kernels through the C ABI (CUDA events, L2 flushed between runs).
    python tools/kbench.py conv 256 128 128 16 16 3 [reps]
    python tools/kbench.py wgrad 256 128 128 16 16 3
    python tools/kbench.py bn 4194304 16
"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from tartangan_b200 import ops, _lib
from tartangan_b200._lib import call, ptr

def timeit(fn, reps=10):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0]

def main():
    kind = sys.argv[1]
    a = [int(v) for v in sys.argv[2:]]
    bf = torch.bfloat16
    if kind in ('conv', 'wgrad', 'convd'):
        n, h, w, cin, cout, k = a[:6]
        reps = a[6] if len(a) > 6 else 10
        x = ops.empty_nhwc(n, cin, h, w, bf, 'cuda'); x.normal_()
        wt = torch.randn(cout, cin, k, k, device='cuda') * 0.05
        nbytes = n * h * w * (cin + cout) * 2
        flops = 2.0 * n * h * w * cin * cout * k * k
        if kind == 'conv':
            wp = ops._packed(wt, 0, 'tc')
            y = ops.empty_nhwc(n, cout, h, w, bf, 'cuda')
            fn = lambda: call('ttg_conv2d_tc', ptr(x), ptr(wp), None, ptr(y), n, h, w, cin, cout, k, _lib.BF16)
        elif kind == 'convd':
            wp = ops._packed(wt, 0, 'direct')
            y = ops.empty_nhwc(n, cout, h, w, bf, 'cuda')
            fn = lambda: call('ttg_conv2d_direct', ptr(x), ptr(wp), None, ptr(y), n, h, w, cin, cout, k, 0, _lib.BF16, _lib.BF16)
        else:
            gy = ops.empty_nhwc(n, cout, h, w, bf, 'cuda'); gy.normal_()
            gw = torch.empty(cout, cin, k, k, device='cuda')
            ws = torch.empty(_lib.lib.ttg_conv2d_wgrad_tc_workspace_bytes(cin, cout, k) // 4 + 4, device='cuda')
            fn = lambda: call('ttg_conv2d_wgrad_tc', ptr(x), ptr(gy), ptr(gw), n, h, w, cin, cout, k, ptr(ws))
        med, best = timeit(fn, reps)
        print(f'{kind} N{n} {h}x{w} {cin}->{cout} k{k}: median {med*1e3:.1f} us  best {best*1e3:.1f} us  '
              f'{nbytes/med/1e6:.0f} GB/s  {flops/med/1e9:.1f} TFLOP/s')
    elif kind == 'rgb':
        # RGB layers through the Python operator (pad8 staging + TMA kernels): fprop 3->16, dgrad 16->3, wgrad 3->16
        n, h, w, k = a[:4]
        x3 = ops.empty_nhwc(n, 3, h, w, bf, 'cuda'); x3.normal_()
        g16 = ops.empty_nhwc(n, 16, h, w, bf, 'cuda'); g16.normal_()
        wt = torch.randn(16, 3, k, k, device='cuda') * 0.05
        for name, fn in (('fprop 3->16', lambda: ops._conv_raw(x3, wt, None, 0, 0)),
                         ('dgrad 16->3', lambda: ops._conv_raw(g16, wt, None, 1, 0)),
                         ('wgrad 3->16', lambda: ops.ConvWgradFn.apply(x3, g16, k, 0))):
            med, best = timeit(fn)
            print(f'rgb {name} N{n} {h}x{w} k{k}: median {med*1e3:.1f} us best {best*1e3:.1f} us')
    elif kind == 'bn':
        m, c = a[:2]
        x = torch.randn(m, c, device='cuda').to(bf)
        mean = torch.zeros(c, device='cuda'); inv = torch.ones(c, device='cuda')
        ws = torch.empty(5 * c, dtype=torch.float64, device='cuda')
        y = torch.empty_like(x)
        fn = lambda: call('ttg_bn_stats', ptr(x), m, c, 1e-5, 0.1, ptr(mean), ptr(inv), None, None, None, ptr(ws), 1, _lib.BF16)
        med, best = timeit(fn)
        print(f'bn_stats M{m} C{c}: {med*1e3:.1f} us {m*c*2/med/1e6:.0f} GB/s')
        fn = lambda: call('ttg_bn_act_fwd', ptr(x), ptr(y), m, c, ptr(mean), ptr(inv), ptr(inv), ptr(mean), 0.2, _lib.BF16)
        med, best = timeit(fn)
        print(f'bn_act_fwd M{m} C{c}: {med*1e3:.1f} us {m*c*4/med/1e6:.0f} GB/s')
        g = torch.empty(c, device='cuda')
        fn = lambda: call('ttg_bn_act_bwd', ptr(x), ptr(y), ptr(y), m, c, ptr(mean), ptr(inv), ptr(inv), ptr(mean), 0.2, ptr(g), ptr(g), ptr(ws), _lib.BF16)
        med, best = timeit(fn)
        print(f'bn_act_bwd M{m} C{c}: {med*1e3:.1f} us {m*c*10/med/1e6:.0f} GB/s')



def iqn(rows_b, c=128, nq=8):
    """IQN head + quantile-Huber forward/backward at B rows (asymptotic GB/s at >= 2^20 quantile rows)."""
    b = rows_b
    feats = torch.randn(b, c, device='cuda'); taus = torch.rand(b * nq, device='cuda')
    we = torch.randn(c, 20, device='cuda') * .3; be = torch.zeros(c, device='cuda'); wo = torch.randn(c, device='cuda'); bo = torch.zeros(1, device='cuda')
    p = torch.empty(b * nq, device='cuda'); tgt = torch.ones(b, device='cuda'); loss = torch.empty((), device='cuda')
    g = torch.randn(b * nq, device='cuda'); gf = torch.empty(b, c, device='cuda')
    gwe = torch.empty(c, 20, device='cuda'); gbe = torch.empty(c, device='cuda'); gwo = torch.empty(c, device='cuda'); gbo = torch.empty(1, device='cuda')
    fwd = lambda: (call('ttg_iqn_head_fwd', ptr(feats), ptr(taus), ptr(we), ptr(be), ptr(wo), ptr(bo), ptr(p), None, b, nq, c, 20),
                   call('ttg_quantile_huber_fwd', ptr(p), ptr(tgt), ptr(taus), ptr(loss), b, nq, 1.0))
    bwd = lambda: call('ttg_iqn_head_bwd', ptr(g), ptr(feats), ptr(taus), ptr(we), ptr(be), ptr(wo), ptr(gf), ptr(gwe), ptr(gbe), ptr(gwo), ptr(gbo), b, nq, c, 20)
    # algorithmic bytes: feats read once per quantile row in the unfused reference = rows*C*4; fused kernel reads feats B*C*4 + taus + writes p
    med, best = timeit(fwd)
    nb = b * c * 4 + b * nq * 8
    print(f'iqn_head+huber fwd B={b} nq={nq} C={c}: {med*1e3:.1f} us  fused bytes {nb/1e6:.1f} MB -> {nb/med/1e6:.0f} GB/s; '
          f'unfused reference traffic (x.repeat + emb + mix) {(3*b*nq*c*4)/1e6:.0f} MB -> equivalent {(3*b*nq*c*4)/med/1e6:.0f} GB/s')
    med, best = timeit(bwd)
    nb = 2 * b * c * 4 + b * nq * 8
    print(f'iqn_head bwd B={b}: {med*1e3:.1f} us  {nb/med/1e6:.0f} GB/s (fused bytes)')


def iqn_fused(b, c=128, nq=8):
    """The single-kernel IQN head (+ quantile mean + quantile-Huber loss) forward and backward at B batch rows
    (B * nq quantile rows).  Algorithmic bytes: feats B*C*4 + taus / p_tau 2*B*nq*4 + p_mean / target 2*B*4 (forward);
    feats + gf 2*B*C*4 + taus / p_tau (backward).  Arithmetic: B*nq*C*(2*E + ~12) fp32 flop + B*nq*C tanh (MUFU)."""
    feats = torch.randn(b, c, device='cuda'); taus = torch.rand(b * nq, device='cuda')
    we = torch.randn(c, 20, device='cuda') * .3; be = torch.zeros(c, device='cuda'); wo = torch.randn(c, device='cuda'); bo = torch.zeros(1, device='cuda')
    p = torch.empty(b * nq, device='cuda'); pm = torch.empty(b, device='cuda'); tgt = torch.ones(b, device='cuda'); loss = torch.empty((), device='cuda')
    gpm = torch.randn(b, device='cuda'); gl = torch.ones(1, device='cuda'); gf = torch.empty(b, c, device='cuda')
    gwe = torch.empty(c, 20, device='cuda'); gbe = torch.empty(c, device='cuda'); gwo = torch.empty(c, device='cuda'); gbo = torch.empty(1, device='cuda')
    fwd = lambda: call('ttg_iqn_head_loss_fwd', ptr(feats), ptr(taus), ptr(we), ptr(be), ptr(wo), ptr(bo), ptr(tgt), ptr(p), ptr(pm), ptr(loss), b, nq, c, 20, 1.0)
    bwd = lambda: call('ttg_iqn_head_loss_bwd', ptr(gpm), ptr(gl), ptr(p), ptr(tgt), ptr(feats), ptr(taus), ptr(we), ptr(be), ptr(wo), ptr(gf), ptr(gwe), ptr(gbe), ptr(gwo), ptr(gbo), b, nq, c, 20, 1.0)
    flop = b * nq * c * (2 * 20 + 12.0)
    for name, fn, nb in (('fwd', fwd, b * c * 4 + 2 * b * nq * 4 + 2 * b * 4), ('bwd', bwd, 2 * b * c * 4 + 2 * b * nq * 4 + b * 4)):
        med, best = timeit(fn)
        print(f'iqn_head_loss {name} B={b} nq={nq} C={c} ({b*nq} quantile rows): median {med*1e3:.1f} us  algorithmic {nb/1e6:.2f} MB -> '
              f'{nb/med/1e6:.0f} GB/s ({nb/med/1e6/6473.9*100:.1f} % of 6473.9)  fp32 {flop*(1 if name == "fwd" else 2.5)/med/1e9:.1f} TFLOP/s  '
              f'tanh {b*nq*c/med/1e6:.0f} G/s')


def spectral(rows, cols):
    """Single-launch spectral-norm power iteration + scaling (ttg_spectral_norm) and its backward at one filter size."""
    w = torch.randn(rows, cols, device='cuda') * 0.05
    u = torch.nn.functional.normalize(torch.randn(rows, device='cuda'), dim=0)
    v = torch.nn.functional.normalize(torch.randn(cols, device='cuda'), dim=0)
    out = torch.empty_like(w); sigma = torch.empty(1, device='cuda'); g = torch.randn_like(w); gw = torch.empty_like(w)
    ws = torch.empty(_lib.lib.ttg_spectral_norm_workspace_floats(rows, cols), device='cuda')
    fwd = lambda: call('ttg_spectral_norm', ptr(w), ptr(u), ptr(v), ptr(out), ptr(sigma), rows, cols, 1, 1e-12, ptr(ws))
    bwd = lambda: call('ttg_spectral_norm_bwd', ptr(g), ptr(out), ptr(u), ptr(v), ptr(sigma), ptr(gw), rows, cols, ptr(ws))
    for name, fn, passes in (('fwd (W^T u, W v, sigma, W / sigma: 4 passes over W)', fwd, 5), ('bwd (dot + update: 2 passes)', bwd, 5)):
        med, best = timeit(fn)
        nb = rows * cols * 4 * passes
        print(f'spectral_norm {name} {rows}x{cols}: median {med*1e3:.1f} us  ({nb/1e6:.2f} MB of L2-resident traffic, -> {nb/med/1e6:.0f} GB/s)')


if sys.argv[1] == 'sn':
    spectral(int(sys.argv[2]), int(sys.argv[3]))
elif sys.argv[1] == 'iqnf':
    iqn_fused(int(sys.argv[2]), int(sys.argv[3]) if len(sys.argv) > 3 else 128, int(sys.argv[4]) if len(sys.argv) > 4 else 8)
elif sys.argv[1] == 'iqn':
    iqn(int(sys.argv[2]), int(sys.argv[3]) if len(sys.argv) > 3 else 128)
else:
    main()
