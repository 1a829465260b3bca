"""Differentiable operators over the C ABI (include/ttg_b200.h).

Every operator is a ``torch.autograd.Function`` whose forward launches the
hand-written kernels through ``_lib.call`` and whose backward is itself written in
terms of these operators, never ``once_differentiable`` where the R1 penalty
(reference models/losses.py:17-30, ``create_graph=True``) needs a second backward:
conv fprop/dgrad/wgrad, BatchNorm+LeakyReLU, pooling, bilinear, sum-pool, Linear,
the IQN head, max-pool, bmm and softmax are all closed under differentiation here.

Activation tensors keep the reference's logical NCHW shape but live in NHWC memory
(``torch.channels_last`` strides); their dtype (fp32 or bf16) is the precision mode.
PyTorch is used for allocation, streams and autograd bookkeeping only.
"""
import weakref

import torch
from torch.autograd import Function

from . import _lib
from ._lib import call, ptr, dtype_code

SLOPE = 0.2
# development switches (A/B runs): TTG_NO_DIRECT=1 keeps autograd's AccumulateGrad path, TTG_NO_ARENA=1 the per-call memsets
import os as _os
_NO_DIRECT = _os.environ.get('TTG_NO_DIRECT', '0') == '1'
_NO_ARENA = _os.environ.get('TTG_NO_ARENA', '0') == '1'
# TTG_SKIP_STREAM=0: the skip branch of a residual block stays on the launching stream (A/B; see skip_branch below)
_SKIP_STREAM = _os.environ.get('TTG_SKIP_STREAM', '1') == '1'


class _State:
    act_dtype = torch.bfloat16     # precision mode for activations ('bf16' default)
    inputs_only = False            # set by gradient_penalty: skip parameter gradients
    use_tc = True                  # tensor-core conv kernels when shapes allow
    launches = 0                   # kernels launched through the C ABI (bench counter)
    pack_generation = 0            # bumped to invalidate every packed-weight cache (CUDA-graph capture)
    producer_stats = None          # (tensor, float64 sums) left by a producer kernel (conv / residual join) for bn_act
    fused_attention = True         # tcgen05 attention kernels when the shape allows (else bmm / softmax / bmm)
    direct_grads = False           # inside direct_param_grads(): parameter gradients are added to p.grad by the kernels
    arena = None                   # ZeroArena of the running trainer (pre-zeroed workspaces), or None
    wgrad_stream = None            # side stream of the in-place weight-gradient kernels (_wgrad_direct)
    wgrad_pending = False          # kernels were launched on it since the last join_side_streams()
    pending_streams = set()        # other streams that carry parts of the running step (the trainer's D(fake) stream)
    bn_group = None                # process group of synchronised BatchNorm (--sync-bn, world > 1), or None: local statistics


state = _State()


def set_precision(mode):
    """'bf16' (bf16 activations / tensor-core convs) or 'fp32' (exact CUDA-core path)."""
    state.act_dtype = {'bf16': torch.bfloat16, 'fp32': torch.float32}[mode]


def get_precision():
    return 'bf16' if state.act_dtype == torch.bfloat16 else 'fp32'


class inputs_only_grads:
    """Context: backward passes inside compute gradients w.r.t. activations only
    (the R1 penalty differentiates w.r.t. the real images, models/losses.py:23-26)."""

    def __enter__(self):
        self.prev, state.inputs_only = state.inputs_only, True

    def __exit__(self, *a):
        state.inputs_only = self.prev


class local_batchnorm:
    """Context: train-mode BatchNorm inside uses the statistics of the local batch even when synchronised BatchNorm is
    on.  For work outside the training step (progress samples, FID): it is not part of the global batch, and a caller
    may run it on one rank only, where a collective would wait for ranks that never issue it."""

    def __enter__(self):
        self.prev, state.bn_group = state.bn_group, None
        return self

    def __exit__(self, *a):
        state.bn_group = self.prev
        return False


class ZeroArena:
    """One pre-zeroed device buffer that hands out the zero-initialised workspaces of a training step (partial-sum
    images of the wgrad kernels, fp64 reduction slots of the BatchNorm backward passes).  The kernels are told that
    their workspace is already clear (flag bit 1 of the ttg_*_acc entry points), so the ~120 per-call memsets of a
    step become ONE clear of the used prefix at `reset()` (start of the D and of the G half-step).  Slices are
    bump-allocated, 256-byte aligned, never reused within a period; a request that does not fit returns None and
    the caller falls back to an ordinary workspace + memset."""

    def __init__(self, device, nbytes=128 << 20):
        self.buf = torch.zeros(nbytes, dtype=torch.uint8, device=device)
        self.offset = 0            # bump pointer of the current period
        self.dirty = 0             # prefix that may hold non-zero data (high-water mark since the buffer was created)
        self.clean_from = 0        # takes below this offset are guaranteed zero in the current period

    def reset(self):
        self.dirty = max(self.dirty, self.offset)
        if self.dirty:
            self.buf[:self.dirty].zero_()
        self.offset = 0
        self.clean_from = self.dirty

    def take(self, nbytes):
        start = (self.offset + 255) & ~255
        if start + nbytes > self.buf.numel():
            return None
        self.offset = start + nbytes
        out = self.buf[start:start + nbytes]
        # beyond the prefix cleared by reset() the buffer has never been written (torch.zeros at creation), unless an
        # earlier period reached further than the last reset knew: then clear explicitly
        if self.offset > self.clean_from and start < self.dirty:
            out.zero_()
        return out


def _ws_zero(nbytes, device):
    """(workspace, flag): a zeroed arena slice and 2 (= 'workspace is already zero'), or an ordinary one and 0."""
    arena = state.arena
    if arena is not None and arena.buf.device == torch.device(device):
        t = arena.take(nbytes)
        if t is not None:
            return t, 2
    return _ws(nbytes, device), 0


def join_side_streams():
    """The launching stream waits for the weight-gradient kernels on the side stream (before anything reads `.grad`:
    the optimiser, a gradient all-reduce, the arena reset of the next half-step)."""
    if state.wgrad_pending:
        torch.cuda.current_stream().wait_stream(state.wgrad_stream)
        state.wgrad_pending = False


class skip_branch:
    """Context for the skip branch of a residual block (1x1 projection of the resampled input, generator.py:59-60,
    discriminator.py:92-94): it is independent of the conv branch until the residual add, so it runs on a companion
    stream of the launching stream and its small kernels fill SMs the conv branch leaves idle; autograd runs its
    backward (the projection's dgrad) on that stream as well.  `join(out)` before the add.  bf16 mode only (the fp32
    parity path stays on one stream)."""
    _streams = {}

    def __init__(self, *inputs):
        self.inputs = [t for t in inputs if torch.is_tensor(t) and t.is_cuda]
        self.side = None
        if _SKIP_STREAM and self.inputs and state.act_dtype == torch.bfloat16:
            self.cur = torch.cuda.current_stream()
            key = (self.cur.device.index, self.cur.cuda_stream)
            side = skip_branch._streams.get(key)
            if side is None:
                side = skip_branch._streams[key] = torch.cuda.Stream(device=self.cur.device)
            self.side = side

    def __enter__(self):
        if self.side is not None:
            self.side.wait_stream(self.cur)
            if torch.is_grad_enabled():            # its backward (and that of the branch point) runs there too
                state.pending_streams.add(self.side)
                state.pending_streams.add(self.cur)
            for t in self.inputs:
                t.record_stream(self.side)
            self._ctx = torch.cuda.stream(self.side)
            self._ctx.__enter__()
        return self

    def __exit__(self, *a):
        if self.side is not None:
            self._ctx.__exit__(*a)
        return False

    def join(self, out):
        if self.side is not None:
            self.cur.wait_stream(self.side)
            out.record_stream(self.cur)
        return out


def join_all_streams(clear=True):
    """The launching stream waits for EVERY stream that may hold contributions to `.grad` or unfinished parts of the
    step: the weight-gradient stream, the D(fake) stream, the early-G stream, the skip-branch companions and the stream
    that called backward (`state.pending_streams`).  Called when a backward pass ends (clear=True) and, by the
    data-parallel hooks, before every gradient all-reduce (clear=False: later buckets must wait for the same streams).
    The in-place kernels return no tensor to autograd, so the engine inserts no synchronisation for them; and a hook
    runs on whichever chain's stream finished last on the HOST, which says nothing about the other chains' kernels."""
    if not state.wgrad_pending and not state.pending_streams:
        return                                    # (nothing forked: also the CPU-only host-logic tests)
    cur = torch.cuda.current_stream()
    if state.wgrad_pending:
        cur.wait_stream(state.wgrad_stream)
        if clear:
            state.wgrad_pending = False
    for st in list(state.pending_streams):
        if st != cur:
            cur.wait_stream(st)
    if clear:
        state.pending_streams.clear()


class direct_param_grads:
    """Context for `loss.backward()`: conv / BatchNorm parameter gradients are ADDED to `p.grad` by the producing
    kernels (ttg_*_acc) and the backward returns None for them, so autograd launches no AccumulateGrad / gradient
    fan-in add kernel per parameter (~190 launches per training step).  Only leaf parameters whose `.grad` is a
    pre-attached contiguous fp32 buffer (optim.FlatParams.attach_grads) take this path, and never under
    `create_graph`.  Not for `torch.autograd.grad(..., params)`: that must not touch `.grad`."""

    def __enter__(self):
        self.prev, state.direct_grads = state.direct_grads, not _NO_DIRECT

    def __exit__(self, *a):
        state.direct_grads = self.prev
        join_all_streams()


def _direct(p):
    """The buffer to accumulate p's gradient into, or None when the ordinary autograd path must be used."""
    if (state.direct_grads and p is not None and not torch.is_grad_enabled() and p.is_leaf and p.requires_grad
            and p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous()
            and p.grad.shape == p.shape):
        return p.grad
    return None


def _wgrad_direct(x, gy, w, bias, up, want_b):
    """gw (and gb) of a tensor-core conv added straight into w.grad (bias.grad).  True if done."""
    cout, cin, k, _ = w.shape
    dw = _direct(w)
    db = _direct(bias) if want_b else None
    if (dw is None or (want_b and db is None) or up != 0 or cin < 8 or cout < 8 or gy.dtype != torch.bfloat16
            or x.dtype != torch.bfloat16 or not _tc_ok(x.dtype, cin, cout)):
        return False
    x, gy = nhwc(x), nhwc(gy)
    n, _, h, wd_ = gy.shape
    # The weight gradient only feeds `.grad`: nothing later in backward depends on it, so it runs on a SIDE stream and
    # the dgrad / BatchNorm-backward chain on the launching stream does not wait for it.  The layers below 32x32 launch
    # 32-128 CTAs on 148 SMs (section 7b of DESIGN.md); their wgrad kernels now fill the SMs the chain leaves idle.
    # All in-place weight-gradient kernels share the one side stream, which is also what keeps them correct: the
    # unpack of the partial sums and ttg_channel_sum_acc add to .grad with a plain read-modify-write, and the D(real)
    # and D(fake) chains run on two streams.  join_side_streams() orders the optimiser / all-reduce / next arena
    # reset after them.
    side = state.wgrad_stream
    if side is None:
        side = state.wgrad_stream = torch.cuda.Stream(device=x.device)
    side.wait_stream(torch.cuda.current_stream())              # x, gy (and the cleared arena) are ready
    x.record_stream(side)
    gy.record_stream(side)
    state.wgrad_pending = True
    with torch.cuda.stream(side):
        ws, z = _ws_zero(_lib.lib.ttg_conv2d_wgrad_tc_workspace_bytes(cin, cout, k), x.device)
        fused_bias = want_b and cout >= 16
        call('ttg_conv2d_wgrad_tc_acc', ptr(x), ptr(gy), ptr(dw), ptr(db) if fused_bias else None, n, h, wd_, _pad16(cin),
             _pad16(cout), cin, cout, k, 1 | z, ptr(ws))
        if want_b and not fused_bias:
            ws2, z2 = _ws_zero(_lib.lib.ttg_bn_workspace_bytes(cout), x.device)
            call('ttg_channel_sum_acc', ptr(gy), n * h * wd_, cout, ptr(db), 1 | z2, ptr(ws2), dtype_code(gy.dtype))
    return True


# --------------------------------------------------------------------------- helpers
def _is_nhwc(x):
    return x.dim() == 4 and x.permute(0, 2, 3, 1).is_contiguous()


def nhwc(x):
    """Return x in NHWC memory (logical NCHW).  Gradients produced by these ops already are."""
    if _is_nhwc(x):
        return x
    return x.contiguous(memory_format=torch.channels_last) if x.dim() == 4 else x.contiguous()


def empty_nhwc(n, c, h, w, dtype, device):
    return torch.empty((n, h, w, c), dtype=dtype, device=device).permute(0, 3, 1, 2)


def _empty_like(x):
    if x.dim() == 4:
        n, c, h, w = x.shape
        return empty_nhwc(n, c, h, w, x.dtype, x.device)
    return torch.empty(x.shape, dtype=x.dtype, device=x.device)


def _ws(nbytes, device):
    return torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=device)


def _flat(x):
    return x if x.is_contiguous() else x.contiguous()


# --------------------------------------------------------------------------- layout boundary
class ToInternal(Function):
    """fp32 NCHW (reference layout, trainers/trainer.py:57-61) -> NHWC activation dtype."""

    @staticmethod
    def forward(ctx, x, dtype):
        ctx.dtype = dtype
        n, c, h, w = x.shape
        x = x.float() if x.dtype != torch.float32 else x
        y = empty_nhwc(n, c, h, w, dtype, x.device)
        if _is_nhwc(x) and not x.is_contiguous():
            call('ttg_cast', ptr(x), _lib.F32, ptr(y), dtype_code(dtype), x.numel())
        else:
            call('ttg_nchw_to_nhwc', ptr(x.contiguous()), ptr(y), n, c, h * w, dtype_code(dtype))
        return y

    @staticmethod
    def backward(ctx, g):
        return FromInternal.apply(g), None


class FromInternal(Function):
    """NHWC activation -> fp32 NCHW contiguous."""

    @staticmethod
    def forward(ctx, x):
        ctx.dtype = x.dtype
        x = nhwc(x)
        n, c, h, w = x.shape
        y = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
        call('ttg_nhwc_to_nchw', ptr(x), ptr(y), n, c, h * w, dtype_code(x.dtype))
        return y

    @staticmethod
    def backward(ctx, g):
        return ToInternal.apply(g, ctx.dtype)


def to_internal(x, dtype=None):
    return ToInternal.apply(x, dtype or state.act_dtype)


def from_internal(x):
    return FromInternal.apply(x)


# --------------------------------------------------------------------------- convolution
def _packed(w, mode, kind):
    """Packed copy of a conv weight.  The cache lives ON the weight tensor (so it dies with it) and
    is validated by (_version, _ttg_epoch, data_ptr): _version catches in-place torch updates,
    _ttg_epoch is bumped by FusedAdam, whose kernel writes the flat buffer behind autograd's back."""
    ver = (w._version, getattr(w, '_ttg_epoch', 0), w.data_ptr(), state.pack_generation)
    cache = getattr(w, '_ttg_pack', None)
    if cache is None:
        cache = {}
        try:
            w._ttg_pack = cache
        except AttributeError:
            pass
    hit = cache.get((kind, mode))
    if hit is not None and hit[0] == ver:
        return hit[1]
    cout, cin, k, _ = w.shape
    wd = w.detach()
    wd = wd if wd.is_contiguous() else wd.contiguous()
    if kind == 'direct':
        wp = torch.empty(k * k * cin * cout, dtype=torch.float32, device=w.device)
        call('ttg_pack_weight_direct', ptr(wd), ptr(wp), cout, cin, k, mode)
    else:
        coutp, cinp = _pad16(cout), _pad16(cin)
        nbytes = _lib.lib.ttg_pack_weight_tc_bytes(coutp, cinp, k)
        wp = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
        if (coutp, cinp) == (cout, cin):
            call('ttg_pack_weight_tc', ptr(wd), ptr(wp), cout, cin, k, mode)
        else:
            call('ttg_pack_weight_tc_pad', ptr(wd), ptr(wp), cout, cin, coutp, cinp, k, mode)
    cache[(kind, mode)] = (ver, wp)
    return wp


class PackedModel:
    """Packed (bf16, UMMA operand image) copies of every tensor-core-eligible conv filter of one flat
    parameter buffer, refreshed by ONE kernel launch (`repack`) after each optimiser update.  The
    per-tensor caches that `_packed` consults are pointed at views of the shared buffer."""

    def __init__(self, flat):
        self.flat = flat
        rows, self.slots, dst, blocks = [], [], 0, 0
        for p, off in zip(flat.params, flat.offsets):
            if p.dim() != 4 or p.shape[2] != p.shape[3] or p.shape[2] not in (1, 3):
                continue
            cout, cin, k, _ = p.shape
            if not _tc_ok(torch.bfloat16, cin, cout):
                continue
            coutp, cinp = _pad16(cout), _pad16(cin)
            nbytes = coutp * cinp * k * k * 2
            for mode in (0, 1):
                rows.append([off, dst, cout, cin, coutp, cinp, k, mode, blocks])
                self.slots.append((p, mode, dst, nbytes))
                dst += (nbytes + 255) // 256 * 256
                blocks += (cout * cin * k * k + 255) // 256
        dev = flat.data.device
        self.buf = torch.zeros(max(dst, 16), dtype=torch.uint8, device=dev)      # zero: channel padding stays zero
        self.table = torch.tensor(rows, dtype=torch.int64, device=dev).reshape(-1, 9) if rows else None
        self.blocks = blocks

    def repack(self):
        if self.table is None or state.act_dtype != torch.bfloat16:
            return
        call('ttg_pack_weights_multi', ptr(self.flat.data), ptr(self.buf), ptr(self.table), self.table.shape[0], self.blocks)
        for p, mode, dst, nbytes in self.slots:
            cache = getattr(p, '_ttg_pack', None)
            if cache is None:
                cache = p._ttg_pack = {}
            ver = (p._version, getattr(p, '_ttg_epoch', 0), p.data_ptr(), state.pack_generation)
            cache[('tc', mode)] = (ver, self.buf[dst:dst + nbytes])


def _pad8(x):
    """8-channel staging copy (channels >= C zero) of a bf16 NHWC tensor with C < 8 channels."""
    n, c, h, w = x.shape
    y = empty_nhwc(n, 8, h, w, x.dtype, x.device)
    call('ttg_pad_channels8', ptr(x), ptr(y), n * h * w, c)
    return y


def _pad16(c):
    """Channel counts <= 8 (the RGB layers) are zero-padded to 16 inside the tensor-core kernels."""
    return 16 if c <= 8 else c


def _tc_ok(dtype, cin, cout):
    ok = lambda c: c <= 8 or (c % 16 == 0 and c <= 256)
    return state.use_tc and dtype == torch.bfloat16 and ok(cin) and ok(cout)


def conv_stats_ok(w, up, dtype):
    """True when conv2d(..., stats=True) can return the BatchNorm statistics of its output from the conv epilogue."""
    cout, cin, k, _ = w.shape
    return (not up and dtype == torch.bfloat16 and state.use_tc and cin % 16 == 0 and cout % 16 == 0
            and bool(_lib.lib.ttg_conv2d_tc_stats_supported(cin, cout, k)))


def _conv_raw(x, w, bias, mode, up, out_dtype=None, stats=None):
    """y = conv(x) with w packed in `mode` (0 fprop: w is OIHW; 1 dgrad: roles swapped).
    stats: optional float64[2*Cout] that receives sum / sum of squares of the output (fprop, TMA kernels only)."""
    x = nhwc(x)
    n, cx, hi, wi = x.shape
    cout, cin, k, _ = w.shape
    c_in_eff, c_out_eff = (cin, cout) if mode == 0 else (cout, cin)
    assert cx == c_in_eff, f'conv: input has {cx} channels, weight expects {c_in_eff}'
    h, wd_ = hi << up, wi << up
    out_dtype = out_dtype or x.dtype
    y = empty_nhwc(n, c_out_eff, h, wd_, out_dtype, x.device)
    if _tc_ok(x.dtype, cin, cout) and out_dtype in (torch.bfloat16, torch.float32):
        assert up == 0, 'tensor-core conv: conv2d() materialises the upsample first'
        wp = _packed(w, mode, 'tc')
        if stats is not None:
            call('ttg_conv2d_tc_stats', ptr(x), ptr(wp), ptr(bias), ptr(y), n, h, wd_, c_in_eff, c_out_eff, k, ptr(stats))
            return y
        # RGB layers: stage the <= 8-channel tensor as 8-channel pixels so the layer runs on the TMA kernels
        stage8 = out_dtype == torch.bfloat16
        xin, cin_mem = (_pad8(x), 8) if (stage8 and c_in_eff < 8) else (x, c_in_eff)
        yout, cout_mem = (empty_nhwc(n, 8, h, wd_, out_dtype, x.device), 8) if (stage8 and c_out_eff < 8) else (y, c_out_eff)
        call('ttg_conv2d_tc_ex', ptr(xin), ptr(wp), ptr(bias), ptr(yout), n, h, wd_, _pad16(c_in_eff), _pad16(c_out_eff),
             cin_mem, cout_mem, k, dtype_code(out_dtype))
        if yout is not y:
            call('ttg_unpad_channels8', ptr(yout), ptr(y), n * h * wd_, c_out_eff)
    else:
        wp = _packed(w, mode, 'direct')
        call('ttg_conv2d_direct', ptr(x), ptr(wp), ptr(bias), ptr(y), n, h, wd_, c_in_eff, c_out_eff, k, up,
             dtype_code(x.dtype), dtype_code(out_dtype))
    return y


class Conv2dFn(Function):
    """nn.Conv2d(k in {1,3}, padding=k//2) with optional nearest x2 upsample of the input folded in."""

    @staticmethod
    def forward(ctx, x, w, bias, up, out_dtype, stats=None):
        ctx.save_for_backward(x, w)
        ctx.up, ctx.has_bias, ctx.in_dtype = up, bias is not None, x.dtype
        ctx.bias = bias            # only its .grad buffer is touched (direct_param_grads)
        return _conv_raw(x, w, bias, 0, up, out_dtype, stats)

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        gx = gw = gb = None
        if gy.dtype != ctx.in_dtype:
            gy = CastFn.apply(gy, ctx.in_dtype)
        if ctx.needs_input_grad[0]:
            gx = ConvDgradFn.apply(gy, w, ctx.up)
        if not state.inputs_only:
            want_w, want_b = ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
            if want_w and _wgrad_direct(x, gy, w, ctx.bias, ctx.up, want_b):
                pass                                                    # added to w.grad / bias.grad by the kernel
            elif (want_w and want_b and ctx.up == 0 and gy.dtype == torch.bfloat16 and w.shape[0] >= 16
                    and _tc_ok(x.dtype, w.shape[1], w.shape[0])):
                gw, gb = ConvWgradBiasFn.apply(x, gy, w.shape[2])      # one pass over gy for both
            else:
                if want_w:
                    gw = ConvWgradFn.apply(x, gy, w.shape[2], ctx.up)
                if want_b:
                    gb = ChannelSumFn.apply(gy)
        return gx, gw, gb, None, None, None


class ConvDgradFn(Function):
    """gx = conv(gy, flipped/transposed w); with up=1 followed by the adjoint of nearest upsample."""

    @staticmethod
    def forward(ctx, gy, w, up):
        ctx.save_for_backward(gy, w)
        ctx.up = up
        gx = _conv_raw(gy, w, None, 1, 0)
        if up:
            gx = _pool2(gx, 1.0)
        return gx

    @staticmethod
    def backward(ctx, ggx):
        gy, w = ctx.saved_tensors
        g_gy = g_w = None
        if ctx.needs_input_grad[0]:
            g_gy = Conv2dFn.apply(ggx, w, None, ctx.up, None)
        if ctx.needs_input_grad[1] and not state.inputs_only and not _wgrad_direct(ggx, gy, w, None, ctx.up, False):
            g_w = ConvWgradFn.apply(ggx, gy, w.shape[2], ctx.up)
        return g_gy, g_w, None


class ConvWgradFn(Function):
    """gw[co,ci,ky,kx] = sum_pixels gy[p,co] * x[p+tap,ci]  (fp32, OIHW)."""

    @staticmethod
    def forward(ctx, x, gy, k, up):
        ctx.save_for_backward(x, gy)
        ctx.k, ctx.up = k, up
        x, gy = nhwc(x), nhwc(gy)
        n, cout, h, w = gy.shape
        cin = x.shape[1]
        gw = torch.empty((cout, cin, k, k), dtype=torch.float32, device=x.device)
        if _tc_ok(x.dtype, cin, cout) and gy.dtype == torch.bfloat16:
            assert up == 0, 'tensor-core wgrad: conv2d() materialises the upsample first'
            ws = _ws(_lib.lib.ttg_conv2d_wgrad_tc_workspace_bytes(cin, cout, k), x.device)
            if cin < 8 or cout < 8:
                # RGB layers: 8-channel staging copies of the narrow operand(s); the extra rows / columns of the
                # 8-channel weight gradient are zero and are dropped
                xin, cin_mem = (_pad8(x), 8) if cin < 8 else (x, cin)
                gin, cout_mem = (_pad8(gy), 8) if cout < 8 else (gy, cout)
                gw8 = torch.empty((cout_mem, cin_mem, k, k), dtype=torch.float32, device=x.device)
                call('ttg_conv2d_wgrad_tc_ex', ptr(xin), ptr(gin), ptr(gw8), n, h, w, _pad16(cin), _pad16(cout), cin_mem,
                     cout_mem, k, ptr(ws))
                gw.copy_(gw8[:cout, :cin])
            else:
                call('ttg_conv2d_wgrad_tc_ex', ptr(x), ptr(gy), ptr(gw), n, h, w, _pad16(cin), _pad16(cout), cin, cout, k,
                     ptr(ws))
        else:
            ws = _ws(_lib.lib.ttg_conv2d_wgrad_direct_workspace_bytes(n, h, w, cin, cout, k), x.device)
            call('ttg_conv2d_wgrad_direct_det', ptr(x), ptr(gy), ptr(gw), n, h, w, cin, cout, k, up,
                 dtype_code(x.dtype), dtype_code(gy.dtype), ptr(ws))
        return gw

    @staticmethod
    def backward(ctx, ggw):
        x, gy = ctx.saved_tensors
        g_x = g_gy = None
        if ctx.needs_input_grad[0]:
            g_x = ConvDgradFn.apply(gy, ggw, ctx.up)
        if ctx.needs_input_grad[1]:
            g_gy = Conv2dFn.apply(x, ggw, None, ctx.up, None)
        return g_x, g_gy, None, None


class ConvWgradBiasFn(Function):
    """(gw, gb): weight gradient and bias gradient (sum over pixels of gy) of a tensor-core conv in one kernel
    (ttg_conv2d_wgrad_bias_tc_ex): the warps that are idle while TMA feeds the tensor cores add up the gy tiles."""

    @staticmethod
    def forward(ctx, x, gy, k):
        ctx.save_for_backward(x, gy)
        ctx.k = k
        x, gy = nhwc(x), nhwc(gy)
        n, cout, h, w = gy.shape
        cin = x.shape[1]
        gb = torch.empty(cout, dtype=torch.float32, device=x.device)
        ws = _ws(_lib.lib.ttg_conv2d_wgrad_tc_workspace_bytes(cin, cout, k), x.device)
        if cin < 8:           # RGB input: 8-channel staging copy, the extra columns of the gradient are dropped
            gw8 = torch.empty((cout, 8, k, k), dtype=torch.float32, device=x.device)
            call('ttg_conv2d_wgrad_bias_tc_ex', ptr(_pad8(x)), ptr(gy), ptr(gw8), ptr(gb), n, h, w, 16, cout, 8, cout, k,
                 ptr(ws))
            gw = gw8[:, :cin].contiguous()
        else:
            gw = torch.empty((cout, cin, k, k), dtype=torch.float32, device=x.device)
            call('ttg_conv2d_wgrad_bias_tc_ex', ptr(x), ptr(gy), ptr(gw), ptr(gb), n, h, w, _pad16(cin), cout, cin, cout, k,
                 ptr(ws))
        return gw, gb

    @staticmethod
    def backward(ctx, ggw, ggb):
        x, gy = ctx.saved_tensors
        g_x = g_gy = None
        if ggw is not None:
            if ctx.needs_input_grad[0]:
                g_x = ConvDgradFn.apply(gy, ggw, 0)
            if ctx.needs_input_grad[1]:
                g_gy = Conv2dFn.apply(x, ggw, None, 0, None)
        if ggb is not None and ctx.needs_input_grad[1]:
            n, c, h, w = gy.shape
            bc = ggb.to(gy.dtype).view(1, c, 1, 1).expand(n, c, h, w)
            g_gy = bc if g_gy is None else g_gy + bc
        return g_x, g_gy, None


def conv2d(x, w, bias=None, up=0, out_dtype=None, stats=False):
    if up and x.dtype == torch.bfloat16 and _tc_ok(x.dtype, w.shape[1], w.shape[0]):
        # tensor-core path: materialise the nearest x2 upsample (one streaming pass) so that fprop AND wgrad fetch
        # their tiles with TMA; measured 2-3x faster than gathering (y>>1, x>>1) with cp.async inside the conv
        # (32->16 @128^2: 197 us -> ~105 us).  The fp32 path keeps the upsample folded into the conv.
        x, up = upsample2(x), 0
    if stats and conv_stats_ok(w, up, x.dtype) and out_dtype in (None, torch.bfloat16):
        # the conv epilogue also accumulates the BatchNorm statistics of y; bn_act() picks them up (same tensor object)
        sums = torch.empty(2 * w.shape[0], dtype=torch.float64, device=x.device)
        y = Conv2dFn.apply(x, w, bias, up, out_dtype, sums)
        state.producer_stats = (y, sums)
        return y
    return Conv2dFn.apply(x, w, bias, up, out_dtype)


def take_producer_stats(x):
    """Statistics left by the kernel that produced x (or None).  Consumed at most once (by the first bn_act after the
    producer) and only for the same memory: the producer's output is kept alive until then, so its address cannot
    have been recycled for another tensor."""
    ps, state.producer_stats = state.producer_stats, None
    if ps is not None and ps[0].data_ptr() == x.data_ptr() and ps[0].shape == x.shape and ps[0].dtype == x.dtype \
            and ps[0].stride() == x.stride():
        return ps[1]
    return None


def _join_stats_ok(t):
    return (t.dtype == torch.bfloat16 and t.dim() == 4
            and bool(_lib.lib.ttg_join_stats_supported(t.shape[1])))


class ChannelSumFn(Function):
    @staticmethod
    def forward(ctx, x):
        x = nhwc(x)
        ctx.shape, ctx.dtype = x.shape, x.dtype
        n, c, h, w = x.shape
        out = torch.empty(c, dtype=torch.float32, device=x.device)
        call('ttg_channel_sum', ptr(x), n * h * w, c, ptr(out), ptr(_ws(8 * c, x.device)), dtype_code(x.dtype))
        return out

    @staticmethod
    def backward(ctx, g):
        n, c, h, w = ctx.shape
        return g.to(ctx.dtype).view(1, c, 1, 1).expand(n, c, h, w)


class CastFn(Function):
    @staticmethod
    def forward(ctx, x, dtype):
        ctx.src = x.dtype
        x = nhwc(x) if x.dim() == 4 else _flat(x)
        y = torch.empty_like(x, dtype=dtype)
        call('ttg_cast', ptr(x), dtype_code(x.dtype), ptr(y), dtype_code(dtype), x.numel())
        return y

    @staticmethod
    def backward(ctx, g):
        return CastFn.apply(g, ctx.src), None


# --------------------------------------------------------------------------- BatchNorm + LeakyReLU
def _bn_world(group):
    import torch.distributed as dist
    return dist.get_world_size(group)


def _bn_all_reduce(sums, group):
    """Sum the fp64 channel sums of every rank (synchronised BatchNorm), in place, ordered on the current stream."""
    import torch.distributed as dist
    dist.all_reduce(sums, group=group)


def _bn_sync_ws(n, device):
    """(fp64 [n] workspace for the sums, flag) from the arena, as _ws_zero."""
    ws, z = _ws_zero(8 * n, device)
    return ws.view(torch.float64)[:n], z


def _bn_bwd_sync(x, ga, gx, mean, invstd, gamma, beta, slope, ggamma, gbeta, accumulate, group):
    """Backward of synchronised BatchNorm + LeakyReLU: local reduce, all-reduce of the 2C sums, apply over the global
    count.  Every rank writes 1/world of the global gamma / beta gradients; the gradient all-reduce adds them up."""
    n, c, h, w = x.shape
    world = _bn_world(group)
    sums, z = _bn_sync_ws(2 * c, x.device)
    call('ttg_bn_act_bwd_reduce', ptr(x), ptr(ga), n * h * w, c, ptr(mean), ptr(invstd), ptr(gamma), ptr(beta), slope,
         ptr(sums), z, dtype_code(x.dtype))
    _bn_all_reduce(sums, group)
    call('ttg_bn_act_bwd_apply', ptr(x), ptr(ga), ptr(gx), n * h * w, c, world * n * h * w, ptr(sums), ptr(mean),
         ptr(invstd), ptr(gamma), ptr(beta), slope, ptr(ggamma), ptr(gbeta), 1.0 / world, accumulate, dtype_code(x.dtype))


class BnActFn(Function):
    """lrelu(batch_norm(x)) with batch statistics (train) or running statistics (eval)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, num_batches, training, momentum, eps, slope, count_mult=1,
                sums=None):
        x = nhwc(x)
        n, c, h, w = x.shape
        m = n * h * w
        dev = x.device
        mean = torch.empty(c, dtype=torch.float32, device=dev)
        invstd = torch.empty(c, dtype=torch.float32, device=dev)
        y = _empty_like(x)
        group = state.bn_group if training else None
        if group is not None:
            # synchronised: the local sums (from the producer or reduced here) are summed over the ranks, and the
            # statistics and running-statistics update use the global pixel count
            if sums is None:
                sums, z = _bn_sync_ws(2 * c, dev)
                call('ttg_bn_sums', ptr(x), m, c, ptr(sums), z, dtype_code(x.dtype))
            _bn_all_reduce(sums, group)
            call('ttg_bn_act_fwd_stats_n', ptr(x), ptr(y), m, c, _bn_world(group) * m, ptr(sums), ptr(gamma), ptr(beta),
                 eps, momentum, slope, ptr(mean), ptr(invstd), ptr(running_mean), ptr(running_var), ptr(num_batches),
                 count_mult, None, dtype_code(x.dtype))
        elif training:
            # statistics (already reduced by the producing conv / join kernel when `sums` is given), their
            # finalisation and the apply pass: one entry point, one or two launches
            ws = None if sums is not None else _ws(_lib.lib.ttg_bn_workspace_bytes(c), dev)
            call('ttg_bn_act_fwd_stats', ptr(x), ptr(y), m, c, ptr(sums), ptr(gamma), ptr(beta), eps, momentum, slope,
                 ptr(mean), ptr(invstd), ptr(running_mean), ptr(running_var), ptr(num_batches), count_mult, ptr(ws),
                 dtype_code(x.dtype))
        else:
            call('ttg_bn_eval_stats', ptr(running_mean), ptr(running_var), eps, c, ptr(mean), ptr(invstd))
            call('ttg_bn_act_fwd', ptr(x), ptr(y), m, c, ptr(mean), ptr(invstd), ptr(gamma), ptr(beta), slope,
                 dtype_code(x.dtype))
        ctx.save_for_backward(x, gamma, beta, mean, invstd)
        ctx.slope, ctx.training = slope, training
        return y

    @staticmethod
    def backward(ctx, ga):
        if not ctx.training:
            raise NotImplementedError('tartangan_b200: backward through eval-mode BatchNorm is not on the '
                                      'reference path (D/G are always in train mode) and is not implemented')
        x, gamma, beta, mean, invstd = ctx.saved_tensors
        dg, db = _direct(gamma), _direct(beta)
        if (dg is not None and db is not None and not state.inputs_only and ctx.needs_input_grad[1]
                and ctx.needs_input_grad[2]):
            x, ga = nhwc(x), nhwc(ga)
            n, c, h, w = x.shape
            gx = _empty_like(x)
            if state.bn_group is not None:
                _bn_bwd_sync(x, ga, gx, mean, invstd, gamma, beta, ctx.slope, dg, db, 1, state.bn_group)
                return gx, None, None, None, None, None, None, None, None, None, None, None
            ws, z = _ws_zero(_lib.lib.ttg_bn_workspace_bytes(c), x.device)
            call('ttg_bn_act_bwd_acc', ptr(x), ptr(ga), ptr(gx), n * h * w, c, ptr(mean), ptr(invstd), ptr(gamma),
                 ptr(beta), ctx.slope, ptr(dg), ptr(db), 1 | z, ptr(ws), dtype_code(x.dtype))
            return gx, None, None, None, None, None, None, None, None, None, None, None
        gx, ggamma, gbeta = BnActBwdFn.apply(x, ga, gamma, beta, mean, invstd, ctx.slope)
        if state.inputs_only:
            ggamma = gbeta = None
        return gx, ggamma, gbeta, None, None, None, None, None, None, None, None, None


class BnActBwdFn(Function):
    @staticmethod
    def forward(ctx, x, ga, gamma, beta, mean, invstd, slope):
        x, ga = nhwc(x), nhwc(ga)
        n, c, h, w = x.shape
        dev = x.device
        gx = _empty_like(x)
        ggamma = torch.empty(c, dtype=torch.float32, device=dev)
        gbeta = torch.empty(c, dtype=torch.float32, device=dev)
        if state.bn_group is not None:
            _bn_bwd_sync(x, ga, gx, mean, invstd, gamma, beta, slope, ggamma, gbeta, 0, state.bn_group)
        else:
            ws = _ws(_lib.lib.ttg_bn_workspace_bytes(c), dev)
            call('ttg_bn_act_bwd', ptr(x), ptr(ga), ptr(gx), n * h * w, c, ptr(mean), ptr(invstd), ptr(gamma), ptr(beta),
                 slope, ptr(ggamma), ptr(gbeta), ptr(ws), dtype_code(x.dtype))
        ctx.save_for_backward(x, ga, gamma, beta, mean, invstd)
        ctx.slope = slope
        ctx.set_materialize_grads(False)
        return gx, ggamma, gbeta

    @staticmethod
    def backward(ctx, u, u_gamma, u_beta):
        if u_gamma is not None or u_beta is not None:
            raise NotImplementedError('tartangan_b200: differentiating BatchNorm parameter gradients is not '
                                      'supported (only d(input grad) is needed by the R1 penalty)')
        if u is None:
            return (None,) * 7
        x, ga, gamma, beta, mean, invstd = ctx.saved_tensors
        u = nhwc(u)
        n, c, h, w = x.shape
        dev = x.device
        g_ga, g_x = _empty_like(x), _empty_like(x)
        dg = None if state.inputs_only or not ctx.needs_input_grad[2] else _direct(gamma)
        g_gamma = None if (state.inputs_only or dg is not None) else torch.empty(c, dtype=torch.float32, device=dev)
        group = state.bn_group
        if group is not None:
            # synchronised: g_gamma is not linear in the per-rank sums, so it too comes from the global ones
            world = _bn_world(group)
            sums, z = _bn_sync_ws(5 * c, dev)
            call('ttg_bn_act_bwd2_reduce', ptr(x), ptr(ga), ptr(u), n * h * w, c, ptr(mean), ptr(invstd), ptr(gamma),
                 ptr(beta), ctx.slope, ptr(sums), z, dtype_code(x.dtype))
            _bn_all_reduce(sums, group)
            call('ttg_bn_act_bwd2_apply', ptr(x), ptr(ga), ptr(u), ptr(g_ga), ptr(g_x), n * h * w, c, world * n * h * w,
                 ptr(sums), ptr(mean), ptr(invstd), ptr(gamma), ptr(beta), ctx.slope,
                 ptr(dg if dg is not None else g_gamma), 1.0 / world, 1 if dg is not None else 0, dtype_code(x.dtype))
            return g_x, g_ga, g_gamma, None, None, None, None
        ws, z = _ws_zero(_lib.lib.ttg_bn_workspace_bytes(c), dev)
        call('ttg_bn_act_bwd2_acc', ptr(x), ptr(ga), ptr(u), ptr(g_ga), ptr(g_x), n * h * w, c, ptr(mean), ptr(invstd),
             ptr(gamma), ptr(beta), ctx.slope, ptr(dg if dg is not None else g_gamma), (1 if dg is not None else 0) | z,
             ptr(ws), dtype_code(x.dtype))
        return g_x, g_ga, g_gamma, None, None, None, None


def bn_act(x, bn, slope=SLOPE, count_mult=1):
    """x -> lrelu(bn(x)) for an nn.BatchNorm2d-compatible module `bn` (or identity norm if None).
    count_mult=4: x is the low-resolution source of a nearest x2 upsample; statistics are identical,
    only the unbiased running-variance correction uses the upsampled element count."""
    sums = take_producer_stats(x)
    if bn is None:
        return leaky_relu(x, slope)
    return BnActFn.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.num_batches_tracked,
                         bn.training or bn.running_mean is None, bn.momentum, bn.eps, slope, count_mult, sums)


class LeakyReluFn(Function):
    @staticmethod
    def forward(ctx, x, slope):
        x = nhwc(x) if x.dim() == 4 else _flat(x)
        ctx.save_for_backward(x)
        ctx.slope = slope
        y = _empty_like(x)
        call('ttg_lrelu_fwd', ptr(x), ptr(y), x.numel(), slope, dtype_code(x.dtype))
        return y

    @staticmethod
    def backward(ctx, g):
        x, = ctx.saved_tensors
        return LeakyReluMaskFn.apply(x, g, ctx.slope), None


class LeakyReluMaskFn(Function):
    """out = g * lrelu'(x); linear in g, piecewise constant in x."""

    @staticmethod
    def forward(ctx, x, g, slope):
        g = (nhwc(g) if g.dim() == 4 else _flat(g))
        ctx.save_for_backward(x)
        ctx.slope = slope
        out = _empty_like(x)
        call('ttg_lrelu_bwd', ptr(x), ptr(g), ptr(out), x.numel(), slope, dtype_code(x.dtype))
        return out

    @staticmethod
    def backward(ctx, u):
        x, = ctx.saved_tensors
        return None, LeakyReluMaskFn.apply(x, u, ctx.slope), None


def leaky_relu(x, slope=SLOPE):
    return LeakyReluFn.apply(x, slope)


SELU_ALPHA, SELU_SCALE = 1.6732632423543772848170429916717, 1.0507009873554804934193349852946


class EluFn(Function):
    """scale * (x > 0 ? x : alpha * (exp(x) - 1)): nn.ELU (alpha, 1) / nn.SELU (SELU_ALPHA, SELU_SCALE) — the other two
    choices of --activation (reference trainers/cnn.py:41-45)."""

    @staticmethod
    def forward(ctx, x, alpha, scale):
        x = nhwc(x) if x.dim() == 4 else _flat(x)
        ctx.save_for_backward(x)
        ctx.alpha, ctx.scale = alpha, scale
        y = _empty_like(x)
        call('ttg_elu_fwd', ptr(x), ptr(y), x.numel(), alpha, scale, dtype_code(x.dtype))
        return y

    @staticmethod
    def backward(ctx, g):
        x, = ctx.saved_tensors
        return EluBwdFn.apply(x, g, ctx.alpha, ctx.scale), None, None


class EluBwdFn(Function):
    """out = g * f'(x).  Linear in g; its x-cotangent g * u * f''(x) is what the R1 penalty differentiates through."""

    @staticmethod
    def forward(ctx, x, g, alpha, scale):
        g = nhwc(g) if g.dim() == 4 else _flat(g)
        ctx.save_for_backward(x, g)
        ctx.alpha, ctx.scale = alpha, scale
        out = _empty_like(x)
        call('ttg_elu_bwd', ptr(x), ptr(g), ptr(out), x.numel(), alpha, scale, dtype_code(x.dtype))
        return out

    @staticmethod
    def backward(ctx, u):
        x, g = ctx.saved_tensors
        gx = gg = None
        u = nhwc(u) if u.dim() == 4 else _flat(u)
        if ctx.needs_input_grad[0]:
            gx = _empty_like(x)
            call('ttg_elu_bwd2', ptr(x), ptr(g), ptr(u), ptr(gx), x.numel(), ctx.alpha, ctx.scale, dtype_code(x.dtype))
        if ctx.needs_input_grad[1]:
            gg = EluBwdFn.apply(x, u, ctx.alpha, ctx.scale)
        return gx, gg, None, None


def elu(x, alpha=1.0, scale=1.0):
    return EluFn.apply(x, float(alpha), float(scale))


def selu(x):
    return EluFn.apply(x, SELU_ALPHA, SELU_SCALE)


# --------------------------------------------------------------------------- resampling
def _pool2(x, scale):
    x = nhwc(x)
    n, c, h, w = x.shape
    y = empty_nhwc(n, c, h // 2, w // 2, x.dtype, x.device)
    call('ttg_pool2_sum', ptr(x), ptr(y), n, h // 2, w // 2, c, scale, dtype_code(x.dtype))
    return y


def _up2(x, scale):
    x = nhwc(x)
    n, c, h, w = x.shape
    y = empty_nhwc(n, c, h * 2, w * 2, x.dtype, x.device)
    call('ttg_upsample2', ptr(x), ptr(y), n, h, w, c, scale, dtype_code(x.dtype))
    return y


class Pool2Fn(Function):
    """scale * 2x2 sum (AvgPool2d(2) when scale=0.25)."""

    @staticmethod
    def forward(ctx, x, scale):
        ctx.scale = scale
        return _pool2(x, scale)

    @staticmethod
    def backward(ctx, g):
        return Up2Fn.apply(g, ctx.scale), None


class Up2Fn(Function):
    """scale * nearest x2 upsample."""

    @staticmethod
    def forward(ctx, x, scale):
        ctx.scale = scale
        return _up2(x, scale)

    @staticmethod
    def backward(ctx, g):
        return Pool2Fn.apply(g, ctx.scale), None


class AddUp2Fn(Function):
    """h + nearest_up2(s): the generator's residual join with the upsample of the skip folded in."""

    @staticmethod
    def forward(ctx, h, s, sums=None):
        h, s = nhwc(h), nhwc(s)
        n, c, ho, wo = h.shape
        y = _empty_like(h)
        if sums is not None:
            call('ttg_add_up2_stats', ptr(h), ptr(s), ptr(y), n, ho, wo, c, ptr(sums), dtype_code(h.dtype))
        else:
            call('ttg_add_up2', ptr(h), ptr(s), ptr(y), n, ho, wo, c, dtype_code(h.dtype))
        return y

    @staticmethod
    def backward(ctx, g):
        return g, Pool2Fn.apply(g, 1.0), None


class Pool2AddFn(Function):
    """scale * pool2sum(h) + s: the discriminator's residual join with AvgPool2d(2) folded in."""

    @staticmethod
    def forward(ctx, h, s, scale, sums=None):
        ctx.scale = scale
        h, s = nhwc(h), nhwc(s)
        n, c, ho, wo = s.shape
        y = _empty_like(s)
        if sums is not None:
            call('ttg_pool2_add_stats', ptr(h), ptr(s), ptr(y), n, ho, wo, c, scale, ptr(sums), dtype_code(h.dtype))
        else:
            call('ttg_pool2_add', ptr(h), ptr(s), ptr(y), n, ho, wo, c, scale, dtype_code(h.dtype))
        return y

    @staticmethod
    def backward(ctx, g):
        return Up2Fn.apply(g, ctx.scale), g, None, None


def add_up2(h, s, stats=True):
    """stats: also reduce the BatchNorm statistics of the result (the next block / the output layer starts with a
    BatchNorm over exactly this tensor); bn_act() picks them up."""
    if stats and _join_stats_ok(h):
        sums = torch.empty(2 * h.shape[1], dtype=torch.float64, device=h.device)
        y = AddUp2Fn.apply(h, s, sums)
        state.producer_stats = (y, sums)
        return y
    return AddUp2Fn.apply(h, s)


def avg_pool2_add(h, s, stats=True):
    if stats and _join_stats_ok(s):
        sums = torch.empty(2 * s.shape[1], dtype=torch.float64, device=s.device)
        y = Pool2AddFn.apply(h, s, 0.25, sums)
        state.producer_stats = (y, sums)
        return y
    return Pool2AddFn.apply(h, s, 0.25)


def avg_pool2(x):
    return Pool2Fn.apply(x, 0.25)


def upsample2(x):
    return Up2Fn.apply(x, 1.0)


class BilinearDownFn(Function):
    @staticmethod
    def forward(ctx, x):
        x = nhwc(x)
        n, c, h, w = x.shape
        y = empty_nhwc(n, c, h // 2, w // 2, x.dtype, x.device)
        call('ttg_bilinear_down_fwd', ptr(x), ptr(y), n, h, w, c, dtype_code(x.dtype))
        return y

    @staticmethod
    def backward(ctx, g):
        return BilinearDownTFn.apply(g)


class BilinearDownTFn(Function):
    @staticmethod
    def forward(ctx, g):
        g = nhwc(g)
        n, c, ho, wo = g.shape
        gx = empty_nhwc(n, c, ho * 2, wo * 2, g.dtype, g.device)
        call('ttg_bilinear_down_bwd', ptr(g), ptr(gx), n, ho * 2, wo * 2, c, dtype_code(g.dtype))
        return gx

    @staticmethod
    def backward(ctx, u):
        return BilinearDownFn.apply(u)


def bilinear_down(x):
    return BilinearDownFn.apply(x)


class BilinearDownTAddFn(Function):
    """other + B^T g (one kernel): the input-gradient fan-in of a residual D block."""

    @staticmethod
    def forward(ctx, g, other):
        g, other = nhwc(g), nhwc(other)
        n, c, ho, wo = g.shape
        gx = _empty_like(other)
        call('ttg_bilinear_down_bwd_add', ptr(g), ptr(other), ptr(gx), n, ho * 2, wo * 2, c, dtype_code(g.dtype))
        return gx

    @staticmethod
    def backward(ctx, u):
        return BilinearDownFn.apply(u), u


class ForkDownFn(Function):
    """x -> (x, bilinear_down(x)): the two branches of a residual D block (discriminator.py:90-95).  The backward
    adds the conv branch's gradient and the transposed-bilinear of the skip branch's gradient in ONE pass."""

    @staticmethod
    def forward(ctx, x):
        x = nhwc(x)
        n, c, h, w = x.shape
        y = empty_nhwc(n, c, h // 2, w // 2, x.dtype, x.device)
        call('ttg_bilinear_down_fwd', ptr(x), ptr(y), n, h, w, c, dtype_code(x.dtype))
        return x.view_as(x), y

    @staticmethod
    def backward(ctx, g_main, g_skip):
        if g_skip is None:
            return g_main
        if g_main is None:
            return BilinearDownTFn.apply(g_skip)
        if g_main.dtype != g_skip.dtype:
            return AxpbyFn.apply(g_main, BilinearDownTFn.apply(g_skip).to(g_main.dtype), 1.0, 1.0)
        return BilinearDownTAddFn.apply(g_skip, g_main)


def fork_bilinear_down(x):
    return ForkDownFn.apply(x)


class AxpbyFn(Function):
    """alpha*a + beta*b (same shape/dtype)."""

    @staticmethod
    def forward(ctx, a, b, alpha, beta):
        ctx.alpha, ctx.beta = alpha, beta
        if a.dim() == 4:
            a, b = nhwc(a), nhwc(b)
        else:
            a, b = _flat(a), _flat(b)
        out = _empty_like(a)
        call('ttg_axpby', ptr(a), ptr(b), ptr(out), a.numel(), alpha, beta, dtype_code(a.dtype))
        return out

    @staticmethod
    def backward(ctx, g):
        ga = g if ctx.alpha == 1.0 else ScaleFn.apply(g, ctx.alpha)
        gb = g if ctx.beta == 1.0 else ScaleFn.apply(g, ctx.beta)
        return ga, gb, None, None


class ScaleFn(Function):
    @staticmethod
    def forward(ctx, x, s):
        ctx.s = s
        x = nhwc(x) if x.dim() == 4 else _flat(x)
        out = _empty_like(x)
        call('ttg_axpby', ptr(x), ptr(x), ptr(out), x.numel(), s, 0.0, dtype_code(x.dtype))
        return out

    @staticmethod
    def backward(ctx, g):
        return ScaleFn.apply(g, ctx.s), None


def add(a, b):
    return AxpbyFn.apply(a, b, 1.0, 1.0)


def scale(x, s):
    return ScaleFn.apply(x, float(s))


class ForkFn(Function):
    """Identity with two consumers; the backward adds the two gradients with our own kernel
    instead of autograd's implicit accumulation."""

    @staticmethod
    def forward(ctx, x):
        return x.view_as(x), x.view_as(x)

    @staticmethod
    def backward(ctx, g1, g2):
        if g1 is None:
            return g2
        if g2 is None:
            return g1
        return AxpbyFn.apply(g1, g2, 1.0, 1.0)


def fork(x):
    return ForkFn.apply(x)


class SpatialSumFn(Function):
    """(N,C,H,W) -> fp32 (N,C): torch.sum(feats, [2,3])."""

    @staticmethod
    def forward(ctx, x):
        x = nhwc(x)
        ctx.shape, ctx.dtype = x.shape, x.dtype
        n, c, h, w = x.shape
        out = torch.empty((n, c), dtype=torch.float32, device=x.device)
        call('ttg_spatial_sum', ptr(x), ptr(out), n, h * w, c, dtype_code(x.dtype))
        return out

    @staticmethod
    def backward(ctx, g):
        return SpatialBcastFn.apply(g, ctx.shape, ctx.dtype)


class SpatialBcastFn(Function):
    @staticmethod
    def forward(ctx, g, shape, dtype):
        n, c, h, w = shape
        g = _flat(g)
        out = empty_nhwc(n, c, h, w, dtype, g.device)
        call('ttg_spatial_bcast', ptr(g), ptr(out), n, h * w, c, dtype_code(dtype))
        return out

    @staticmethod
    def backward(ctx, u):
        return SpatialSumFn.apply(u), None, None


def spatial_sum(x):
    return SpatialSumFn.apply(x)


class TanhFn(Function):
    @staticmethod
    def forward(ctx, x):
        x = nhwc(x) if x.dim() == 4 else _flat(x)
        y = _empty_like(x)
        call('ttg_tanh_fwd', ptr(x), ptr(y), x.numel())
        ctx.save_for_backward(y)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        y, = ctx.saved_tensors
        g = nhwc(g) if g.dim() == 4 else _flat(g)
        gx = _empty_like(y)
        call('ttg_tanh_bwd', ptr(y), ptr(g), ptr(gx), y.numel())
        return gx


def tanh(x):
    return TanhFn.apply(x)


class RgbHeadFn(Function):
    """tanh(conv1x1(a, w) + bias) -> fp32 NCHW image: the generator's output layer (generator.py:120-129) as one
    streaming kernel forward and one backward (ttg_rgb_head_fwd / _bwd)."""

    @staticmethod
    def forward(ctx, a, w, bias):
        a = nhwc(a)
        n, cin, h, wd_ = a.shape
        y = torch.empty((n, w.shape[0], h, wd_), dtype=torch.float32, device=a.device)
        wf = _flat(w.detach()).view(w.shape[0], cin)
        call('ttg_rgb_head_fwd', ptr(a), ptr(wf), ptr(bias), ptr(y), n, h * wd_, cin)
        ctx.save_for_backward(a, w, y)
        ctx.bias = bias
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        a, w, y = ctx.saved_tensors
        n, cin, h, wd_ = a.shape
        g = g.contiguous()
        ga = _empty_like(a)
        bias = ctx.bias
        dw, db = _direct(w), (_direct(bias) if bias is not None else None)
        direct = dw is not None and (bias is None or db is not None) and not state.inputs_only
        gw = dw if direct else torch.empty_like(w, dtype=torch.float32)
        gb = (db if direct else torch.empty(w.shape[0], dtype=torch.float32, device=a.device)) if bias is not None else None
        ws = _ws(_lib.lib.ttg_rgb_head_workspace_bytes(cin), a.device)
        call('ttg_rgb_head_bwd', ptr(a), ptr(_flat(w.detach())), ptr(y), ptr(g), ptr(ga), ptr(gw), ptr(gb), n, h * wd_, cin,
             1 if direct else 0, ptr(ws))
        if direct:
            return ga, None, None
        return ga, gw, gb


def rgb_head_ok(conv, x):
    w = conv.weight if hasattr(conv, 'weight') and isinstance(conv.weight, torch.nn.Parameter) else None
    return (w is not None and x.dtype == torch.bfloat16 and x.dim() == 4 and w.shape[2] == 1 and w.shape[3] == 1
            and bool(_lib.lib.ttg_rgb_head_supported(w.shape[1], w.shape[0])))


# --------------------------------------------------------------------------- fp32 matmul / Linear
def _mm(a, b, bias, ta, tb):
    a, b = _flat(a), _flat(b)
    m = a.shape[1] if ta else a.shape[0]
    k = a.shape[0] if ta else a.shape[1]
    n = b.shape[0] if tb else b.shape[1]
    kb = b.shape[1] if tb else b.shape[0]
    assert k == kb, (a.shape, b.shape, ta, tb)
    out = torch.empty((m, n), dtype=torch.float32, device=a.device)
    call('ttg_matmul_f32', ptr(a), ptr(b), ptr(bias), ptr(out), m, n, k, int(ta), int(tb))
    return out


class MatmulFn(Function):
    """C = op(A) op(B) in fp32; closed under differentiation through the transpose flags."""

    @staticmethod
    def forward(ctx, a, b, ta, tb):
        ctx.save_for_backward(a, b)
        ctx.ta, ctx.tb = ta, tb
        return _mm(a, b, None, ta, tb)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        ta, tb = ctx.ta, ctx.tb
        ga = gb = None
        if ctx.needs_input_grad[0]:
            ga = MatmulFn.apply(g, b, False, not tb) if not ta else MatmulFn.apply(b, g, tb, True)
        if ctx.needs_input_grad[1]:
            gb = MatmulFn.apply(a, g, not ta, False) if not tb else MatmulFn.apply(g, a, True, ta)
        return ga, gb, None, None


class ColsumFn(Function):
    """out[n] = scale * sum_m x[m,n]."""

    @staticmethod
    def forward(ctx, x, scale):
        x = _flat(x)
        ctx.m, ctx.scale = x.shape[0], scale
        out = torch.empty(x.shape[1], dtype=torch.float32, device=x.device)
        call('ttg_colsum_f32', ptr(x), ptr(out), x.shape[0], x.shape[1], scale)
        return out

    @staticmethod
    def backward(ctx, g):
        return RowBcastFn.apply(g, ctx.m, ctx.scale), None


class RowBcastFn(Function):
    """out[m,n] = scale * g[n]."""

    @staticmethod
    def forward(ctx, g, m, scale):
        g = _flat(g)
        ctx.scale = scale
        out = torch.empty((m, g.shape[0]), dtype=torch.float32, device=g.device)
        call('ttg_rowbcast_f32', ptr(g), ptr(out), m, g.shape[0], scale)
        return out

    @staticmethod
    def backward(ctx, u):
        return ColsumFn.apply(u, ctx.scale), None, None


class LinearFn(Function):
    """y = x W^T + b (nn.Linear), fp32."""

    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        ctx.has_bias = b is not None
        return _mm(x, w, b, False, True)

    @staticmethod
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = MatmulFn.apply(g, w, False, False)
        if not state.inputs_only:
            if ctx.needs_input_grad[1]:
                gw = MatmulFn.apply(g, x, True, False)
            if ctx.has_bias and ctx.needs_input_grad[2]:
                gb = ColsumFn.apply(g, 1.0)
        return gx, gw, gb


def linear(x, w, b=None):
    return LinearFn.apply(x, w, b)


# --------------------------------------------------------------------------- IQN head and losses
class IqnHeadFn(Function):
    """p_tau[r] for rows r = q*B + b (models/iqn.py:91-103 + Linear(C->1))."""

    @staticmethod
    def forward(ctx, feats, taus, we, be, wo, bo, nq):
        feats, taus = _flat(feats), _flat(taus)
        b, c = feats.shape
        e = we.shape[1]
        p_tau = torch.empty(b * nq, dtype=torch.float32, device=feats.device)
        call('ttg_iqn_head_fwd', ptr(feats), ptr(taus), ptr(_flat(we)), ptr(be), ptr(_flat(wo)), ptr(bo), ptr(p_tau),
             None, b, nq, c, e)
        ctx.save_for_backward(feats, taus, we, be, wo)
        ctx.nq = nq
        return p_tau

    @staticmethod
    def backward(ctx, g):
        feats, taus, we, be, wo = ctx.saved_tensors
        gf, gwe, gbe, gwo, gbo = IqnHeadBwdFn.apply(g, feats, taus, we, be, wo, ctx.nq)
        if state.inputs_only:
            gwe = gbe = gwo = gbo = None
        return gf, None, gwe, gbe, gwo, gbo, None


class IqnHeadBwdFn(Function):
    @staticmethod
    def forward(ctx, g, feats, taus, we, be, wo, nq):
        g = _flat(g)
        b, c = feats.shape
        e = we.shape[1]
        dev = feats.device
        gf = torch.empty((b, c), dtype=torch.float32, device=dev)
        gwe = torch.empty((c, e), dtype=torch.float32, device=dev)
        gbe = torch.empty(c, dtype=torch.float32, device=dev)
        gwo = torch.empty(wo.shape, dtype=torch.float32, device=dev)
        gbo = torch.empty(1, dtype=torch.float32, device=dev)
        call('ttg_iqn_head_bwd', ptr(g), ptr(feats), ptr(taus), ptr(_flat(we)), ptr(be), ptr(_flat(wo)), ptr(gf),
             ptr(gwe), ptr(gbe), ptr(gwo), ptr(gbo), b, nq, c, e)
        ctx.save_for_backward(g, taus, we, be, wo)
        ctx.nq = nq
        ctx.set_materialize_grads(False)
        return gf, gwe, gbe, gwo, gbo

    @staticmethod
    def backward(ctx, ggf, ggwe, ggbe, ggwo, ggbo):
        if any(t is not None for t in (ggwe, ggbe, ggwo, ggbo)):
            raise NotImplementedError('tartangan_b200: second derivatives of IQN-head parameter gradients are '
                                      'not supported (the R1 penalty only differentiates d p / d feats)')
        if ggf is None:
            return (None,) * 7
        # gf = sum_q g * e(We,be,tau) * wo is independent of feats and has the same form as the forward
        # with feats := ggf: d/dg is the forward itself (no bias), d/d(We,be,wo) is the backward.
        g, taus, we, be, wo = ctx.saved_tensors
        ggf = _flat(ggf)
        b, c = ggf.shape
        e = we.shape[1]
        dev = ggf.device
        cot_g = torch.empty(b * ctx.nq, dtype=torch.float32, device=dev)
        call('ttg_iqn_head_fwd', ptr(ggf), ptr(taus), ptr(_flat(we)), ptr(be), ptr(_flat(wo)), None, ptr(cot_g), None,
             b, ctx.nq, c, e)
        gwe = gbe = gwo = None
        if not state.inputs_only:
            gwe = torch.empty((c, e), dtype=torch.float32, device=dev)
            gbe = torch.empty(c, dtype=torch.float32, device=dev)
            gwo = torch.empty(wo.shape, dtype=torch.float32, device=dev)
            call('ttg_iqn_head_bwd', ptr(g), ptr(ggf), ptr(taus), ptr(_flat(we)), ptr(be), ptr(_flat(wo)), None,
                 ptr(gwe), ptr(gbe), ptr(gwo), None, b, ctx.nq, c, e)
        return cot_g, None, None, gwe, gbe, gwo, None


class IqnHeadLossFn(Function):
    """The whole IQN head in one launch (blocks/discriminator.py:164-178): (feats, taus, head parameters, target) ->
    (p_target = mean over quantiles [B], quantile-Huber loss).  target=None: no loss (returned as None)."""

    @staticmethod
    def forward(ctx, feats, taus, we, be, wo, bo, target, nq, k):
        feats, taus = _flat(feats), _flat(taus).reshape(-1)
        b, c = feats.shape
        e = we.shape[1]
        dev = feats.device
        p_tau = torch.empty(b * nq, dtype=torch.float32, device=dev)
        p_mean = torch.empty(b, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev) if target is not None else None
        tgt = _flat(target).reshape(-1).float() if target is not None else None
        call('ttg_iqn_head_loss_fwd', ptr(feats), ptr(taus), ptr(_flat(we)), ptr(be), ptr(_flat(wo)), ptr(bo), ptr(tgt),
             ptr(p_tau), ptr(p_mean), ptr(loss), b, nq, c, e, float(k))
        ctx.save_for_backward(feats, taus, we, be, wo, tgt, p_tau)
        ctx.nq, ctx.k, ctx.has_loss = nq, float(k), target is not None
        ctx.set_materialize_grads(False)
        if loss is None:
            return p_mean.view(b, 1)
        return p_mean.view(b, 1), loss

    @staticmethod
    def backward(ctx, g_pmean, g_loss=None):
        feats, taus, we, be, wo, tgt, p_tau = ctx.saved_tensors
        gf, gwe, gbe, gwo, gbo = IqnHeadLossBwdFn.apply(g_pmean, g_loss, feats, taus, we, be, wo, tgt, p_tau, ctx.nq, ctx.k)
        if state.inputs_only:
            gwe = gbe = gwo = gbo = None
        return gf, None, gwe, gbe, gwo, gbo, None, None, None


class IqnHeadLossBwdFn(Function):
    """One kernel: cotangents of (p_target, loss) -> gradients of feats and the head parameters.  Differentiable once
    more w.r.t. the p_target path (the R1 penalty, models/losses.py:23-26): d p_target / d feats does not depend on
    feats, so the second backward re-uses the forward (feats := cotangent) and this kernel."""

    @staticmethod
    def forward(ctx, g_pmean, g_loss, feats, taus, we, be, wo, tgt, p_tau, nq, k):
        b, c = feats.shape
        e = we.shape[1]
        dev = feats.device
        gp = _flat(g_pmean).reshape(-1).float() if g_pmean is not None else None
        gl = _flat(g_loss).reshape(-1).float() if g_loss is not None else None
        gf = torch.empty((b, c), dtype=torch.float32, device=dev)
        gwe = torch.empty((c, e), dtype=torch.float32, device=dev)
        gbe = torch.empty(c, dtype=torch.float32, device=dev)
        gwo = torch.empty(wo.shape, dtype=torch.float32, device=dev)
        gbo = torch.empty(1, dtype=torch.float32, device=dev)
        call('ttg_iqn_head_loss_bwd', ptr(gp), ptr(gl), ptr(p_tau), ptr(tgt), ptr(feats), ptr(taus), ptr(_flat(we)), ptr(be),
             ptr(_flat(wo)), ptr(gf), ptr(gwe), ptr(gbe), ptr(gwo), ptr(gbo), b, nq, c, e, float(k))
        ctx.save_for_backward(gp, taus, we, be, wo)
        ctx.nq, ctx.loss_path = nq, g_loss is not None
        ctx.set_materialize_grads(False)
        return gf, gwe, gbe, gwo, gbo

    @staticmethod
    def backward(ctx, ggf, ggwe, ggbe, ggwo, ggbo):
        if any(t is not None for t in (ggwe, ggbe, ggwo, ggbo)):
            raise NotImplementedError('tartangan_b200: second derivatives of IQN-head parameter gradients are '
                                      'not supported (the R1 penalty only differentiates d p / d feats)')
        if ggf is None:
            return (None,) * 11
        if ctx.loss_path:
            raise NotImplementedError('tartangan_b200: differentiating the IQN loss gradient a second time is not on the '
                                      'reference path (the R1 penalty differentiates p_target only)')
        gp, taus, we, be, wo = ctx.saved_tensors
        ggf = _flat(ggf)
        b, c = ggf.shape
        e = we.shape[1]
        dev = ggf.device
        # gf[b, :] = (gp[b] / nq) * sum_q e(tau_qb) * wo  is linear in gp and independent of feats:
        #   cot(gp)[b] = mean_q <ggf[b], e(tau_qb) * wo>  = the forward's quantile mean with feats := ggf (no bias, no loss)
        scratch = torch.empty(b * ctx.nq, dtype=torch.float32, device=dev)
        cot_gp = torch.empty(b, dtype=torch.float32, device=dev)
        call('ttg_iqn_head_loss_fwd', ptr(ggf), ptr(taus), ptr(_flat(we)), ptr(be), ptr(_flat(wo)), None, None, ptr(scratch),
             ptr(cot_gp), None, b, ctx.nq, c, e, 1.0)
        gwe = gbe = gwo = None
        if not state.inputs_only:
            gwe = torch.empty((c, e), dtype=torch.float32, device=dev)
            gbe = torch.empty(c, dtype=torch.float32, device=dev)
            gwo = torch.empty(wo.shape, dtype=torch.float32, device=dev)
            call('ttg_iqn_head_loss_bwd', ptr(gp), None, None, None, ptr(ggf), ptr(taus), ptr(_flat(we)), ptr(be), ptr(_flat(wo)),
                 None, ptr(gwe), ptr(gbe), ptr(gwo), None, b, ctx.nq, c, e, 1.0)
        return cot_gp.view(-1, 1) if gp is not None else None, None, None, None, gwe, gbe, gwo, None, None, None, None


class QuantileHuberFn(Function):
    """iqn_loss (models/iqn.py:111-130)."""

    @staticmethod
    def forward(ctx, p_tau, target, taus, nq, k):
        p_tau, target, taus = _flat(p_tau), _flat(target), _flat(taus)
        b = target.numel()
        loss = torch.empty((), dtype=torch.float32, device=p_tau.device)
        call('ttg_quantile_huber_fwd', ptr(p_tau), ptr(target), ptr(taus), ptr(loss), b, nq, k)
        ctx.save_for_backward(p_tau, target, taus)
        ctx.nq, ctx.k = nq, k
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gloss):
        p_tau, target, taus = ctx.saved_tensors
        gp = torch.empty_like(p_tau)
        call('ttg_quantile_huber_bwd', ptr(p_tau), ptr(target), ptr(taus), ptr(_flat(gloss)), ptr(gp),
             target.numel(), ctx.nq, ctx.k)
        return gp, None, None, None, None


class BceLogitsFn(Function):
    """nn.BCEWithLogitsLoss() (mean)."""

    @staticmethod
    def forward(ctx, x, y):
        x, y = _flat(x), _flat(y)
        loss = torch.empty((), dtype=torch.float32, device=x.device)
        call('ttg_bce_logits_fwd', ptr(x), ptr(y), ptr(loss), x.numel())
        ctx.save_for_backward(x, y)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gloss):
        x, y = ctx.saved_tensors
        gx = torch.empty_like(x)
        call('ttg_bce_logits_bwd', ptr(x), ptr(y), ptr(_flat(gloss)), ptr(gx), x.numel())
        return gx, None


class SqsumFn(Function):
    """scale * sum(x^2) over an fp32 tensor (R1 reduction, models/losses.py:27-29)."""

    @staticmethod
    def forward(ctx, x, scale):
        x = _flat(x)
        out = torch.empty((), dtype=torch.float32, device=x.device)
        call('ttg_sqsum_f32', ptr(x), x.numel(), scale, ptr(out), ptr(_ws(8, x.device)))
        ctx.save_for_backward(x)
        ctx.scale = scale
        return out

    @staticmethod
    def backward(ctx, g):
        x, = ctx.saved_tensors
        return ScaleByDevFn.apply(x, g, 2.0 * ctx.scale), None


class ScaleByDevFn(Function):
    """x * (host * s) with s a device scalar (fp32 tensors)."""

    @staticmethod
    def forward(ctx, x, s, host):
        x = _flat(x)
        out = torch.empty_like(x)
        call('ttg_scale_f32', ptr(x), ptr(out), x.numel(), host, ptr(_flat(s)))
        ctx.save_for_backward(s)
        ctx.host = host
        return out

    @staticmethod
    def backward(ctx, u):
        s, = ctx.saved_tensors
        if ctx.needs_input_grad[1]:
            raise NotImplementedError('tartangan_b200: gradient w.r.t. the scalar of ScaleByDevFn')
        return ScaleByDevFn.apply(u, s, ctx.host), None, None


# --------------------------------------------------------------------------- attention primitives
class MaxPool2Fn(Function):
    @staticmethod
    def forward(ctx, x):
        x = nhwc(x)
        n, c, h, w = x.shape
        y = empty_nhwc(n, c, h // 2, w // 2, x.dtype, x.device)
        idx = torch.empty(n * (h // 2) * (w // 2) * c, dtype=torch.uint8, device=x.device)
        call('ttg_maxpool2_fwd', ptr(x), ptr(y), ptr(idx), n, h // 2, w // 2, c, dtype_code(x.dtype))
        ctx.save_for_backward(idx)
        ctx.mark_non_differentiable(idx)
        return y

    @staticmethod
    def backward(ctx, g):
        idx, = ctx.saved_tensors
        return MaxPoolScatterFn.apply(g, idx)


class MaxPoolScatterFn(Function):
    @staticmethod
    def forward(ctx, g, idx):
        g = nhwc(g)
        n, c, ho, wo = g.shape
        gx = empty_nhwc(n, c, ho * 2, wo * 2, g.dtype, g.device)
        call('ttg_maxpool2_scatter', ptr(g), ptr(idx), ptr(gx), n, ho, wo, c, dtype_code(g.dtype))
        ctx.save_for_backward(idx)
        return gx

    @staticmethod
    def backward(ctx, u):
        idx, = ctx.saved_tensors
        return MaxPoolGatherFn.apply(u, idx), None


class MaxPoolGatherFn(Function):
    @staticmethod
    def forward(ctx, x, idx):
        x = nhwc(x)
        n, c, h, w = x.shape
        y = empty_nhwc(n, c, h // 2, w // 2, x.dtype, x.device)
        call('ttg_maxpool2_gather', ptr(x), ptr(idx), ptr(y), n, h // 2, w // 2, c, dtype_code(x.dtype))
        ctx.save_for_backward(idx)
        return y

    @staticmethod
    def backward(ctx, g):
        idx, = ctx.saved_tensors
        return MaxPoolScatterFn.apply(g, idx), None


def max_pool2(x):
    return MaxPool2Fn.apply(x)


def _bmm(a, b, ta, tb):
    a, b = _flat(a), _flat(b)
    bt = a.shape[0]
    m = a.shape[2] if ta else a.shape[1]
    k = a.shape[1] if ta else a.shape[2]
    n = b.shape[1] if tb else b.shape[2]
    out = torch.empty((bt, m, n), dtype=a.dtype, device=a.device)
    call('ttg_bmm', ptr(a), ptr(b), ptr(out), bt, m, n, k, int(ta), int(tb), dtype_code(a.dtype))
    return out


class BmmFn(Function):
    """Batched op(A) op(B) on (batch, rows, cols) tensors, fp32 accumulate."""

    @staticmethod
    def forward(ctx, a, b, ta, tb):
        ctx.save_for_backward(a, b)
        ctx.ta, ctx.tb = ta, tb
        return _bmm(a, b, ta, tb)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        ta, tb = ctx.ta, ctx.tb
        ga = gb = None
        if ctx.needs_input_grad[0]:
            ga = BmmFn.apply(g, b, False, not tb) if not ta else BmmFn.apply(b, g, tb, True)
        if ctx.needs_input_grad[1]:
            gb = BmmFn.apply(a, g, not ta, False) if not tb else BmmFn.apply(g, a, True, ta)
        return ga, gb, None, None


class SoftmaxFn(Function):
    @staticmethod
    def forward(ctx, x):
        x = _flat(x)
        y = torch.empty_like(x)
        call('ttg_softmax_fwd', ptr(x), ptr(y), x.numel() // x.shape[-1], x.shape[-1], dtype_code(x.dtype))
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, g):
        y, = ctx.saved_tensors
        return SoftmaxBwdFn.apply(y, g)


class SoftmaxBwdFn(Function):
    @staticmethod
    def forward(ctx, y, g):
        g = _flat(g)
        gx = torch.empty_like(y)
        call('ttg_softmax_bwd', ptr(y), ptr(g), ptr(gx), y.numel() // y.shape[-1], y.shape[-1], dtype_code(y.dtype))
        ctx.save_for_backward(y, g)
        return gx

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, w):
        y, g = ctx.saved_tensors
        w = _flat(w)
        cot_g, cot_y = torch.empty_like(y), torch.empty_like(y)
        call('ttg_softmax_bwd2', ptr(y), ptr(g), ptr(w), ptr(cot_g), ptr(cot_y), y.numel() // y.shape[-1],
             y.shape[-1], dtype_code(y.dtype))
        return cot_y, cot_g


def _attention_unfused(q, k, v):
    """softmax(q k^T) v with beta materialised: every step is a differentiable op of this file."""
    beta = SoftmaxFn.apply(BmmFn.apply(q, k, False, True))
    return BmmFn.apply(beta, v, False, False)


def attention_fused_ok(q, k, v):
    return (state.fused_attention and q.dtype == torch.bfloat16 and q.dim() == 3 and
            bool(_lib.lib.ttg_attn_supported(q.shape[1], k.shape[1], q.shape[2], v.shape[2])))


class FusedAttentionFn(Function):
    """o = softmax(q k^T) v per image on the tcgen05 kernels (reference attention.py:25-34), beta never stored.

    backward: the fused recompute kernel; under ``create_graph`` (the R1 penalty differentiates D's attention
    twice, models/losses.py:23) the gradients are rebuilt from the differentiable bmm / softmax ops instead, so
    the second backward sees an ordinary graph."""

    @staticmethod
    def forward(ctx, q, k, v):
        q, k, v = _flat(q), _flat(k), _flat(v)
        bt, nq, dk = q.shape
        nk, dv = k.shape[1], v.shape[2]
        o = torch.empty((bt, nq, dv), dtype=q.dtype, device=q.device)
        lse = torch.empty((bt, nq), dtype=torch.float32, device=q.device)
        call('ttg_attn_fwd', ptr(q), ptr(k), ptr(v), ptr(o), ptr(lse), bt, nq, nk, dk, dv)
        ctx.save_for_backward(q, k, v, o, lse)
        ctx.mark_non_differentiable(lse)
        return o

    @staticmethod
    def backward(ctx, go):
        q, k, v, o, lse = ctx.saved_tensors
        go = _flat(go)
        if torch.is_grad_enabled():
            beta = SoftmaxFn.apply(BmmFn.apply(q, k, False, True))
            gv = BmmFn.apply(beta, go, True, False)
            gs = SoftmaxBwdFn.apply(beta, BmmFn.apply(go, v, False, True))
            return BmmFn.apply(gs, k, False, False), BmmFn.apply(gs, q, True, False), gv
        bt, nq, dk = q.shape
        nk, dv = k.shape[1], v.shape[2]
        gq, gk, gv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        ws = _ws(_lib.lib.ttg_attn_bwd_workspace_bytes(bt, nq, dk), q.device)
        call('ttg_attn_bwd', ptr(q), ptr(k), ptr(v), ptr(o), ptr(go), ptr(lse), ptr(gq), ptr(gk), ptr(gv), bt, nq, nk,
             dk, dv, ptr(ws))
        return gq, gk, gv


def attention_core(q, k, v):
    """(batch, Nq, dk), (batch, Nk, dk), (batch, Nk, dv) -> (batch, Nq, dv)."""
    if attention_fused_ok(q, k, v):
        return FusedAttentionFn.apply(q, k, v)
    return _attention_unfused(q, k, v)


class ScaleDevFn(Function):
    """x * s with s a one-element fp32 device tensor (attention gamma)."""

    @staticmethod
    def forward(ctx, x, s):
        x = nhwc(x) if x.dim() == 4 else _flat(x)
        out = _empty_like(x)
        call('ttg_scale_dev', ptr(x), ptr(out), x.numel(), ptr(s), dtype_code(x.dtype))
        ctx.save_for_backward(x, s)
        return out

    @staticmethod
    def backward(ctx, g):
        x, s = ctx.saved_tensors
        gx = ScaleDevFn.apply(g, s) if ctx.needs_input_grad[0] else None
        gs = None
        if ctx.needs_input_grad[1] and not state.inputs_only:
            gs = DotFn.apply(g, x).reshape(s.shape)
        return gx, gs


class DotFn(Function):
    """sum(a*b) -> fp32 scalar."""

    @staticmethod
    def forward(ctx, a, b):
        a = nhwc(a) if a.dim() == 4 else _flat(a)
        b = nhwc(b) if b.dim() == 4 else _flat(b)
        out = torch.empty((), dtype=torch.float32, device=a.device)
        call('ttg_dot_f32out', ptr(a), ptr(b), ptr(out), a.numel(), ptr(_ws(8, a.device)), dtype_code(a.dtype))
        ctx.save_for_backward(a, b)
        return out

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g = g.reshape(1)
        ga = ScaleDevFn.apply(b, g) if ctx.needs_input_grad[0] else None
        gb = ScaleDevFn.apply(a, g) if ctx.needs_input_grad[1] else None
        return ga, gb


def ensure_internal(x):
    """Accept the reference's fp32 NCHW tensors at any module boundary."""
    if x.dim() != 4:
        return x
    if x.dtype == state.act_dtype and _is_nhwc(x):
        return x
    return ToInternal.apply(x, state.act_dtype)


class SpectralNormFn(Function):
    """w / sigma(w) with `n_iter` power-iteration steps updating u, v in place (torch.nn.utils.spectral_norm).
    Backward treats u, v as constants: g_w = (g - <g, w_out> u v^T) / sigma."""

    @staticmethod
    def forward(ctx, w, u, v, n_iter, eps):
        wd = _flat(w.detach())
        rows, cols = w.shape[0], w[0].numel()
        w_out = torch.empty_like(wd)
        sigma = torch.empty(1, dtype=torch.float32, device=w.device)
        ws = torch.empty(_lib.lib.ttg_spectral_norm_workspace_floats(rows, cols), dtype=torch.float32, device=w.device)
        if n_iter > 0:
            call('ttg_spectral_norm', ptr(wd), ptr(u), ptr(v), ptr(w_out), ptr(sigma), rows, cols, n_iter, eps, ptr(ws))
        else:       # eval: sigma = u^T W v with the stored vectors, no update
            uu, vv = u.clone(), v.clone()
            call('ttg_spectral_norm_sigma', ptr(wd), ptr(uu), ptr(vv), ptr(w_out), ptr(sigma), rows, cols, ptr(ws))
        ctx.save_for_backward(w_out, u.clone(), v.clone(), sigma)
        return w_out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        w_out, u, v, sigma = ctx.saved_tensors
        g = _flat(g)
        rows, cols = w_out.shape[0], w_out[0].numel()
        gw = torch.empty_like(w_out)
        call('ttg_spectral_norm_bwd', ptr(g), ptr(w_out), ptr(u), ptr(v), ptr(sigma), ptr(gw), rows, cols,
             ptr(_ws(4 * _lib.lib.ttg_spectral_norm_workspace_floats(rows, cols), g.device)))
        return gw, None, None, None, None
