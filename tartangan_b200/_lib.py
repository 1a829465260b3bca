"""ctypes binding of libttg_b200.so (the C ABI declared in include/ttg_b200.h).

The argument types are parsed from the header itself, so the header is the single
source of truth.  There is no fallback: if the library is missing or a call fails,
a RuntimeError is raised.
"""
import ctypes
import os
import re

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(_HERE), 'include', 'ttg_b200.h')
LIB_PATH = os.environ.get('TTG_B200_LIB') or os.path.join(_HERE, 'lib', 'libttg_b200.so')

F32, BF16 = 0, 1
_DTYPE_CODE = {torch.float32: F32, torch.bfloat16: BF16}


def dtype_code(dt):
    try:
        return _DTYPE_CODE[dt]
    except KeyError:
        raise RuntimeError(f'tartangan_b200: unsupported activation dtype {dt}') from None


def _ctype(decl):
    decl = decl.strip()
    if '*' in decl:
        return ctypes.c_void_p
    base = re.sub(r'\b(const|unsigned)\b', '', decl).split()
    base = ' '.join(base[:-1]) if len(base) > 1 else base[0]
    return {'int': ctypes.c_int, 'float': ctypes.c_float, 'long long': ctypes.c_longlong,
            'size_t': ctypes.c_size_t, 'void': None}[base]


def parse_header(path=HEADER):
    """-> {name: (restype, [argtypes])} for every `ttg_*` prototype."""
    text = open(path).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    protos = {}
    for m in re.finditer(r'([\w\s\*]+?)\b(ttg_\w+)\s*\(([^)]*)\)\s*;', text):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        if '*' in ret:
            restype = ctypes.c_char_p
        else:
            restype = {'int': ctypes.c_int, 'size_t': ctypes.c_size_t}[ret]
        argtypes = [] if args in ('', 'void') else [_ctype(a) for a in args.split(',')]
        protos[name] = (restype, argtypes)
    return protos


class _Lib:
    def __init__(self):
        self._dll = None
        self.protos = parse_header()

    def load(self):
        if self._dll is None:
            if not os.path.isfile(LIB_PATH):
                raise RuntimeError(
                    f'tartangan_b200: {LIB_PATH} is missing. Build it with '
                    '`python -m tartangan_b200.build` (nvcc, sm_100a). There is no CPU fallback.')
            dll = ctypes.CDLL(LIB_PATH)
            for name, (restype, argtypes) in self.protos.items():
                fn = getattr(dll, name)       # AttributeError if the header and the library disagree
                fn.restype, fn.argtypes = restype, argtypes
            self._dll = dll
        return self._dll

    def __getattr__(self, name):
        if name.startswith('ttg_'):
            return getattr(self.load(), name)
        raise AttributeError(name)


lib = _Lib()


def last_error():
    return lib.ttg_last_error().decode()


def check(rc, what=''):
    if rc != 0:
        raise RuntimeError(f'tartangan_b200 kernel call failed ({what}): {last_error()}')


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError('tartangan_b200: tensor is not on a CUDA device; there is no CPU path')
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


# kernels launched per entry point (for the bench's gpu_launches counter)
KERNELS_PER_CALL = {
    'ttg_bn_stats': 2, 'ttg_rgb_head_bwd': 2, 'ttg_conv2d_wgrad_direct_det': 2, 'ttg_bn_act_bwd': 2, 'ttg_bn_act_bwd2': 2, 'ttg_channel_sum': 2, 'ttg_sqsum_f32': 2,
    'ttg_dot_f32out': 2, 'ttg_adam_flat': 2, 
    'ttg_attn_bwd': 3, 'ttg_conv2d_wgrad_tc_acc': 2, 'ttg_bn_act_bwd_acc': 2, 'ttg_bn_act_bwd2_acc': 2, 'ttg_channel_sum_acc': 2, 'ttg_conv2d_wgrad_tc': 2, 'ttg_conv2d_wgrad_tc_ex': 2, 'ttg_conv2d_wgrad_bias_tc_ex': 2,
}


class Counters:
    calls = 0
    kernels = 0
    profiler = None      # optional object with .record(name, args, start_event, end_event)


def call(name, *args):
    """Invoke an `int ttg_*(..., stream)` entry point on the current stream."""
    Counters.calls += 1
    Counters.kernels += KERNELS_PER_CALL.get(name, 1)
    prof = Counters.profiler
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    rc = getattr(lib, name)(*args, stream())
    if rc != 0:
        raise RuntimeError(f'tartangan_b200: {name} failed: {last_error()}')
    if prof is not None:
        e1.record()
        prof.record(name, args, e0, e1)
