"""Per-entry-point device timing with CUDA events on the launching stream (bench / tuning aid).

    with KernelProfiler() as prof:
        trainer.train_batch(...)
    prof.summary()  -> rows sorted by total device time, with algorithmic bytes / flops where modelled
"""
from collections import defaultdict

import torch

from . import _lib


def _conv_key(args):
    # (x, wp, bias, y, N, H, W, Cin, Cout, k, up, ...)
    n, h, w, cin, cout, k, up = args[4:11]
    return f'N{n} {h}x{w} {cin}->{cout} k{k} up{up}'


def _conv_bytes_flops(args, elt=2):
    n, h, w, cin, cout, k, up = args[4:11]
    pix_out = n * h * w
    pix_in = pix_out >> (2 * up)
    return (pix_in * cin + pix_out * cout) * elt, 2.0 * pix_out * cin * cout * k * k


def _wgrad_key(args):
    n, h, w, cin, cout, k, up = args[3:10]
    return f'N{n} {h}x{w} {cin}->{cout} k{k} up{up}'


def _wgrad_bytes_flops(args, elt=2):
    n, h, w, cin, cout, k, up = args[3:10]
    pix_out = n * h * w
    return ((pix_out >> (2 * up)) * cin + pix_out * cout) * elt, 2.0 * pix_out * cin * cout * k * k


def _elt(code):
    return 2 if code == _lib.BF16 else 4


# algorithmic HBM bytes of the streaming kernels (each tensor read or written once), keyed by entry point
_STREAM_MODELS = {
    # (x, y, N, Hi, Wi, C, scale, dtype): 1 low-res read + 4 writes
    'ttg_upsample2': lambda a: (f'N{a[2]} {a[3]}x{a[4]} C{a[5]}', a[2] * a[3] * a[4] * a[5] * _elt(a[7]) * 5),
    # (x, y, N, Ho, Wo, C, scale, dtype): 4 reads + 1 write
    'ttg_pool2_sum': lambda a: (f'N{a[2]} {a[3]}x{a[4]} C{a[5]}', a[2] * a[3] * a[4] * a[5] * _elt(a[7]) * 5),
    # (h, s, y, N, Ho, Wo, C, [sums,] dtype): h + y at full resolution, s at a quarter
    'ttg_add_up2': lambda a: (f'N{a[3]} {a[4]}x{a[5]} C{a[6]}', int(a[3] * a[4] * a[5] * a[6] * _elt(a[7]) * 2.25)),
    'ttg_add_up2_stats': lambda a: (f'N{a[3]} {a[4]}x{a[5]} C{a[6]}', int(a[3] * a[4] * a[5] * a[6] * _elt(a[8]) * 2.25)),
    # (h, s, y, N, Ho, Wo, C, scale, [sums,] dtype): h at 4x the output resolution, s + y at the output resolution
    'ttg_pool2_add': lambda a: (f'N{a[3]} {a[4]}x{a[5]} C{a[6]}', a[3] * a[4] * a[5] * a[6] * _elt(a[8]) * 6),
    'ttg_pool2_add_stats': lambda a: (f'N{a[3]} {a[4]}x{a[5]} C{a[6]}', a[3] * a[4] * a[5] * a[6] * _elt(a[9]) * 6),
    # (x, y, N, Hi, Wi, C, dtype): full-resolution tensor + quarter-resolution tensor
    'ttg_bilinear_down_fwd': lambda a: (f'N{a[2]} {a[3]}x{a[4]} C{a[5]}', int(a[2] * a[3] * a[4] * a[5] * _elt(a[6]) * 1.25)),
    'ttg_bilinear_down_bwd': lambda a: (f'N{a[2]} {a[3]}x{a[4]} C{a[5]}', int(a[2] * a[3] * a[4] * a[5] * _elt(a[6]) * 1.25)),
    # (gy, add, gx, N, Hi, Wi, C, dtype): + the full-resolution addend
    'ttg_bilinear_down_bwd_add': lambda a: (f'N{a[3]} {a[4]}x{a[5]} C{a[6]}', int(a[3] * a[4] * a[5] * a[6] * _elt(a[7]) * (2.25 if a[1] else 1.25))),
    # (a, b, out, n, alpha, beta, dtype)
    'ttg_axpby': lambda a: (f'n{a[3]}', a[3] * _elt(a[6]) * (2 if a[0] == a[1] else 3)),
    # (x, y8, npix, c_real): bf16
    'ttg_pad_channels8': lambda a: (f'npix{a[2]} c{a[3]}', a[2] * (a[3] + 8) * 2),
    'ttg_unpad_channels8': lambda a: (f'npix{a[2]} c{a[3]}', a[2] * (a[3] + 8) * 2),
    # (x, y, N, C, HW, dtype): fp32 on the NCHW side
    'ttg_nchw_to_nhwc': lambda a: (f'N{a[2]} C{a[3]} HW{a[4]}', a[2] * a[3] * a[4] * (4 + _elt(a[5]))),
    'ttg_nhwc_to_nchw': lambda a: (f'N{a[2]} C{a[3]} HW{a[4]}', a[2] * a[3] * a[4] * (4 + _elt(a[5]))),
    # (p, g, m, v, ema, n, ...): p, m, v read + written, g read, ema read + written when present
    'ttg_adam_flat': lambda a: (f'n{a[5]}', a[5] * 4 * (7 + (2 if a[4] else 0))),
    # (a, w, bias, y, N, HW, Cin) / (a, w, y, g, ga, gw, gb, N, HW, Cin, ...): bf16 NHWC activations, fp32 NCHW image
    'ttg_rgb_head_fwd': lambda a: (f'N{a[4]} HW{a[5]} C{a[6]}', a[4] * a[5] * (a[6] * 2 + 12)),
    'ttg_rgb_head_bwd': lambda a: (f'N{a[7]} HW{a[8]} C{a[9]}', a[7] * a[8] * (a[9] * 4 + 24)),
    # (x, src_dtype, y, dst_dtype, n)
    'ttg_cast': lambda a: (f'n{a[4]}', a[4] * (_elt(a[1]) + _elt(a[3]))),
}


class KernelProfiler:
    def __init__(self):
        self.events = []

    def __enter__(self):
        _lib.Counters.profiler = self
        return self

    def __exit__(self, *a):
        _lib.Counters.profiler = None

    def record(self, name, args, e0, e1):
        key, nbytes, flops = '', 0, 0.0
        # the tensor-core entry points have no `up` argument (always 0); it is inserted to share the direct conv's layout
        if name == 'ttg_conv2d_direct':
            key = _conv_key(args)
            nbytes, flops = _conv_bytes_flops(args)
        elif name in ('ttg_conv2d_tc', 'ttg_conv2d_tc_stats'):     # (x, wp, bias, y, N, H, W, Cin, Cout, k, ...)
            a = list(args[:10]) + [0]
            key = _conv_key(a)
            nbytes, flops = _conv_bytes_flops(a)
            name = 'ttg_conv2d_tc'
        elif name == 'ttg_conv2d_tc_ex':        # (x, wp, bias, y, N, H, W, CinP, CoutP, cin, cout, k, ...)
            a = list(args[:4]) + list(args[4:7]) + [args[9], args[10], args[11], 0]
            key = _conv_key(a)
            nbytes, flops = _conv_bytes_flops(a)
            name = 'ttg_conv2d_tc'
        elif name == 'ttg_conv2d_wgrad_tc_ex':  # (x, gy, gw, N, H, W, CinP, CoutP, cin, cout, k, ws)
            a = list(args[:3]) + list(args[3:6]) + [args[8], args[9], args[10], 0]
            key = _wgrad_key(a)
            nbytes, flops = _wgrad_bytes_flops(a)
            name = 'ttg_conv2d_wgrad_tc'
        elif name == 'ttg_conv2d_wgrad_tc':     # (x, gy, gw, N, H, W, Cin, Cout, k, ws)
            a = list(args[:9]) + [0]
            key = _wgrad_key(a)
            nbytes, flops = _wgrad_bytes_flops(a)
        elif name in ('ttg_conv2d_wgrad_direct', 'ttg_conv2d_wgrad_direct_det'):
            key = _wgrad_key(args)
            nbytes, flops = _wgrad_bytes_flops(args)
        elif name in ('ttg_bn_stats',):
            key = f'M{args[1]} C{args[2]}'
            nbytes = args[1] * args[2] * 2
        elif name == 'ttg_bn_act_fwd':
            key = f'M{args[2]} C{args[3]}'
            nbytes = args[2] * args[3] * 2 * 2
        elif name == 'ttg_bn_act_fwd_stats':       # (x, y, M, C, sums, ...): statistics pass only when sums is NULL
            key = f'M{args[2]} C{args[3]}'
            nbytes = args[2] * args[3] * 2 * (2 if args[4] else 3)
            name = 'ttg_bn_act_fwd'
        elif name in ('ttg_conv2d_wgrad_tc_acc', 'ttg_conv2d_wgrad_bias_tc_ex'):   # (x, gy, gw, gbias, N, H, W, CinP, CoutP, cin, cout, k, ...)
            a = list(args[:3]) + list(args[4:7]) + [args[9], args[10], args[11], 0]
            key = _wgrad_key(a)
            nbytes, flops = _wgrad_bytes_flops(a)
            name = 'ttg_conv2d_wgrad_tc'
        elif name == 'ttg_bn_act_bwd_acc':
            key = f'M{args[3]} C{args[4]}'
            nbytes = args[3] * args[4] * 2 * 5
            name = 'ttg_bn_act_bwd'
        elif name == 'ttg_bn_act_bwd2_acc':
            key = f'M{args[5]} C{args[6]}'
            nbytes = args[5] * args[6] * 2 * 8
            name = 'ttg_bn_act_bwd2'
        elif name == 'ttg_bn_act_bwd':
            key = f'M{args[3]} C{args[4]}'
            nbytes = args[3] * args[4] * 2 * 5          # reduce reads x,ga; apply reads x,ga writes gx
        elif name == 'ttg_bn_act_bwd2':
            key = f'M{args[5]} C{args[6]}'
            nbytes = args[5] * args[6] * 2 * 8          # reduce reads 3; apply reads 3 writes 2
        elif name in _STREAM_MODELS:              # resampling / joins / layout / optimiser: bytes in + bytes out
            key, nbytes = _STREAM_MODELS[name](args)
        self.events.append((name, key, nbytes, flops, e0, e1))

    def summary(self):
        torch.cuda.synchronize()
        agg = defaultdict(lambda: [0, 0.0, 0, 0.0])
        for name, key, nbytes, flops, e0, e1 in self.events:
            a = agg[(name, key)]
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
            a[2] += nbytes
            a[3] += flops
        rows = [dict(name=n, key=k, calls=v[0], ms=v[1], bytes=v[2], flops=v[3]) for (n, k), v in agg.items()]
        rows.sort(key=lambda r: -r['ms'])
        return rows

    def by_name(self):
        rows = self.summary()
        agg = defaultdict(lambda: dict(calls=0, ms=0.0, bytes=0, flops=0.0))
        for r in rows:
            a = agg[r['name']]
            a['calls'] += r['calls']
            a['ms'] += r['ms']
            a['bytes'] += r['bytes']
            a['flops'] += r['flops']
        out = [dict(name=k, **v) for k, v in agg.items()]
        out.sort(key=lambda r: -r['ms'])
        return out
