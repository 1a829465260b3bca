"""Shared body of CNNTrainer / IQNTrainer: model construction from the factory seam and the
D-step / G-step / EMA schedule of reference trainers/cnn.py:29-165 and trainers/iqn.py:30-156.
"""
import functools
import os

import numpy as np
import torch
from torch import nn

from .. import ops
from ..models.blocks import (GeneratorInputMLP, GeneratorOutput, ResidualDiscriminatorBlock,
                             ResidualGeneratorBlock, TiledZGeneratorInput)
from ..models.layers import ELU, SELU, BatchNorm2d, LeakyReLU, SpectralNormConv2d
from ..models.losses import gradient_penalty
from ..models.pluggan import GAN_CONFIGS, Generator
from ..optim import FlatParams, FusedAdam
from .trainer import Trainer
from .utils import toggle_grad

_EARLY_GEN = os.environ.get('TTG_EARLY_GEN', '0') == '1'      # development switch, see _stage_inputs
_FAKE_STREAM = os.environ.get('TTG_FAKE_STREAM', '1') == '1'   # A/B switch, see d_forward_backward
_EARLY_GFWD = os.environ.get('TTG_EARLY_GFWD', '1') == '1'     # A/B switch, see early_g_forward
_GEN_ASYNC = os.environ.get('TTG_GEN_ASYNC', '1') == '1'       # A/B switch, see _capture (generator-sample graph on its own stream)


class GanTrainer(Trainer):
    discriminator_cls = None          # set by subclasses
    d_output_cls = None

    # ------------------------------------------------------------------ construction
    def build_models(self):
        args = self.args
        ops.set_precision(getattr(args, 'precision', 'bf16'))
        cfg = GAN_CONFIGS[args.config]
        if getattr(args, 'attention', None):
            cfg = cfg._replace(attention=tuple(int(i) for i in str(args.attention).split(',') if i != ''))
        self.gan_config = cfg.scale_model(args.model_scale)
        norm_factory = {'id': nn.Identity, 'bn': BatchNorm2d}[args.norm]
        g_input_factory = {'mlp': GeneratorInputMLP, 'tiledz': TiledZGeneratorInput}[args.g_base]
        activation_factory = {'relu': functools.partial(LeakyReLU, 0.2), 'selu': SELU, 'elu': ELU}[args.activation]
        # additive flag --spectral-norm {none,d,g,gd}: binds the blocks' conv_factory seam (reference generator.py:34,
        # discriminator.py:28,52 — never bound by the reference trainers) to the power-iteration conv
        sn = getattr(args, 'spectral_norm', 'none') or 'none'
        g_conv = dict(conv_factory=SpectralNormConv2d) if 'g' in sn and sn != 'none' else {}
        d_conv = dict(conv_factory=SpectralNormConv2d) if 'd' in sn and sn != 'none' else {}
        g_factories = dict(
            input_factory=functools.partial(g_input_factory, activation_factory=activation_factory),
            block_factory=functools.partial(ResidualGeneratorBlock, norm_factory=norm_factory,
                                            activation_factory=activation_factory, **g_conv),
            output_factory=functools.partial(GeneratorOutput, norm_factory=norm_factory,
                                             activation_factory=activation_factory, **g_conv))
        self.g = Generator(self.gan_config, **g_factories).to(self.device)
        self.target_g = Generator(self.gan_config, **g_factories).to(self.device)
        self.d = self.discriminator_cls(
            self.gan_config,
            block_factory=functools.partial(ResidualDiscriminatorBlock, norm_factory=norm_factory,
                                            activation_factory=activation_factory, **d_conv),
            output_factory=functools.partial(self.d_output_cls, norm_factory=norm_factory,
                                             activation_factory=activation_factory),
            **(dict(input_factory=functools.partial(self.discriminator_cls.default_input, **d_conv))
               if d_conv and getattr(self.discriminator_cls, 'default_input', None) is not None else {}),
        ).to(self.device)
        nq = getattr(args, 'num_quantiles', None)
        if nq and hasattr(self.d, 'to_output') and hasattr(self.d.to_output, 'iqn'):
            self.d.to_output.iqn.num_quantiles = nq
        if args.activation == 'selu':
            self.init_params_selu(self.g.parameters())
            self.init_params_selu(self.d.parameters())
        self.optimizer_g = FusedAdam(self.g.parameters(), lr=args.lr_g, betas=(0., 0.999))
        self.optimizer_d = FusedAdam(self.d.parameters(), lr=args.lr_d, betas=(0., 0.999))
        self.update_target_generator(1.)       # NB: like the reference this is an EMA step, not a copy (B.1)
        self._target_flat = None
        self.world_size, self.rank = 1, 0
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.world_size, self.rank = torch.distributed.get_world_size(), torch.distributed.get_rank()
            self.broadcast_parameters()
        # --sync-bn: BatchNorm statistics over the global batch.  The BatchNorm passes then issue collectives, which
        # every rank must issue in the same order: the step runs the single-stream schedule (see _single_stream)
        self.sync_bn = bool(getattr(args, 'sync_bn', False)) and self.world_size > 1 and args.norm == 'bn'
        ops.state.bn_group = torch.distributed.group.WORLD if self.sync_bn else None

    def init_params_selu(self, params):
        """trainers/cnn.py:96-105 / trainers/iqn.py:94-102: vectors zeroed, matrices / filters N(0, 1/fan_in).  The draws
        come from the CPU generator (like the reference, whose models are initialised before .to(device)), in
        parameter order, so a seed gives the reference's values."""
        for p in params:
            d = p.data
            if d.dim() == 1:
                d.zero_()
            else:
                fan_in, _ = nn.init._calculate_fan_in_and_fan_out(d)
                d.copy_(torch.empty(d.shape).normal_(std=float(np.sqrt(1. / fan_in))))

    def broadcast_parameters(self):
        """Data parallel start-up: every rank adopts rank 0's parameters and buffers."""
        for m in (self.g, self.target_g, self.d):
            for t in list(m.parameters()) + list(m.buffers()):
                torch.distributed.broadcast(t.data, 0)

    # ------------------------------------------------------------------ losses (subclass hooks)
    def d_real(self, real):
        """-> (p_real, loss of the real half)"""
        raise NotImplementedError

    def d_fake(self, fake):
        """-> loss of the fake half"""
        raise NotImplementedError

    def d_combine(self, l_real, l_fake):
        raise NotImplementedError

    def d_losses(self, real, fake):
        """-> (p_real, d_loss without penalty)"""
        p_real, l_real = self.d_real(real)
        return p_real, self.d_combine(l_real, self.d_fake(fake))

    def g_loss(self, fake):
        raise NotImplementedError

    # ------------------------------------------------------------------ one optimisation step
    def _reducer(self, optimizer):
        """Bucketed all-reduce over the optimiser's flat gradient buffer (data parallel only)."""
        if self.world_size == 1:
            return None
        flat = optimizer._ensure_flat()
        red = getattr(optimizer, '_ttg_reducer', None)
        if red is None or red.flat_grad is not flat.grad:
            from ..parallel import BucketedAllReduce
            red = BucketedAllReduce(flat.params, flat.offsets, flat.grad, num_buckets=2)
            optimizer._ttg_reducer = red
        return red

    def _reset_arena(self):
        """Start a new period of the pre-zeroed workspace arena (ops.ZeroArena): one clear per half-step."""
        if ops._NO_ARENA:
            return
        arena = getattr(self, '_arena', None)
        if arena is None:
            arena = self._arena = ops.ZeroArena(self.device)
        ops.state.arena = arena        # (the arena of the trainer that is stepping)
        arena.reset()

    def _backward(self, loss, optimizer, overlap=True):
        """loss.backward(); in data parallel the loss is scaled by 1/world so the SUMMED gradients are the
        global-batch average, and (eager mode) the exchange is overlapped with the rest of backward."""
        if loss.is_cuda and ops.state.pending_streams:
            ops.state.pending_streams.add(torch.cuda.current_stream())     # (a bucket hook may run on another chain's stream)
        if self.world_size == 1:
            with ops.direct_param_grads():      # conv / BatchNorm parameter gradients land in the flat .grad buffer
                loss.backward()
            return
        red = self._reducer(optimizer) if overlap else None
        if red is not None:
            red.begin()
        with ops.direct_param_grads():          # (the grad hooks still fire: AccumulateGrad runs with an undefined grad)
            loss.backward(torch.full_like(loss, 1.0 / self.world_size))
        if red is not None:
            red.finish()

    # The step is cut into four segments so that the same code runs eagerly or as CUDA graphs
    # (one graph on a single GPU; three graphs with the two gradient exchanges between them otherwise).
    def d_forward_backward(self, imgs, overlap=True, fake=None):
        """fake: the generator sample for this D step when it was produced ahead of time (graph mode generates it
        while the host batch is still being copied to the device)."""
        toggle_grad(self.g, False)
        toggle_grad(self.d, True)
        self.optimizer_d.zero_grad()
        self._reset_arena()
        if fake is None:
            with torch.no_grad():
                fake = self.sample_g(len(imgs))
        real = imgs
        if self.args.grad_penalty:
            real = imgs.detach().requires_grad_()
        gp = None
        if _FAKE_STREAM and self.args.grad_penalty and not self._single_stream():
            # The fake half of the D step (forward, and through autograd its whole backward chain) runs on a second
            # stream: D(fake) forward overlaps the R1 inner backward, the fake backward chain overlaps the real one and
            # the R1 double backward.  D's layers below 32x32 launch 32-128 CTAs on 148 SMs, so two chains fill what one
            # leaves idle.  Order kept: D(fake) forward starts after D(real) forward (the BatchNorm running statistics
            # are updated real first, then fake, like the reference); parameter gradients of the two chains meet in the
            # flat .grad buffer through the single weight-gradient stream and atomic BatchNorm accumulations.  bf16 mode
            # only: the fp32 parity path stays on one stream (fixed summation order).
            main = torch.cuda.current_stream()
            side = getattr(self, '_fake_stream', None)
            if side is None:
                side = self._fake_stream = torch.cuda.Stream(device=self.device)
                # (the head's Linear / embedding gradients reach AccumulateGrad from two streams by design; the engine
                # synchronises them, the advisory warning about it would be printed every step)
                warn_off = getattr(torch.autograd.graph, 'set_warn_on_accumulate_grad_stream_mismatch', None)
                if warn_off is not None:
                    warn_off(False)
            p_real, l_real = self.d_real(real)
            side.wait_stream(main)
            self._wait_gen_sample(side)
            ops.state.pending_streams.add(side)     # joined again when backward ends / before a gradient all-reduce
            fake.record_stream(side)
            with torch.cuda.stream(side):
                l_fake = self.d_fake(fake)
            gp = gradient_penalty(p_real, real)
            main.wait_stream(side)
            l_fake.record_stream(main)
            d_loss = self.d_combine(l_real, l_fake)
        else:
            self._wait_gen_sample(torch.cuda.current_stream())
            p_real, d_loss = self.d_losses(real, fake)
            if self.args.grad_penalty:
                gp = gradient_penalty(p_real, real)
        if gp is not None:
            d_loss = ops.AxpbyFn.apply(d_loss, gp, 1.0, float(self.args.grad_penalty))
        self._backward(d_loss, self.optimizer_d, overlap)
        return d_loss.detach(), (gp.detach() if gp is not None else None)

    def d_update(self):
        self.optimizer_d.step()

    def _single_stream(self):
        """The step keeps its BatchNorm work on one stream: in fp32 mode (fixed summation order) and under synchronised
        BatchNorm (each BatchNorm pass all-reduces its sums, so the ranks must reach them in one program order).  The
        skip-branch and weight-gradient side streams carry no BatchNorm and stay."""
        return ops.get_precision() != 'bf16' or getattr(self, 'sync_bn', False)

    def _wait_gen_sample(self, stream):
        """Graph mode with the generator-sample graph on its own stream: `stream` waits (an external event-wait node
        inside the step graph) until that graph has produced this step's sample."""
        ev = getattr(self, '_gen_done', None)
        st = getattr(self, '_st', None)
        if ev is not None and st is not None and st.get('active'):
            stream.wait_event(ev)

    def early_g_forward(self, n):
        """Graph mode: the generator forward of the G STEP, issued at the start of the step on its own stream.  It
        depends on nothing the D step produces (G's parameters change only at the end of the step, z1 is already
        staged), so it runs beside the D step; only D(fake_g) has to wait for D's update.  Order kept: it starts after
        the generator sample of the D step (G's BatchNorm running statistics: z0 pass first, then z1, like the
        reference).  Returns the sample for g_forward_backward(fake=...); None when switched off."""
        if not _EARLY_GFWD or self._single_stream():
            return None
        main = torch.cuda.current_stream()
        g2 = getattr(self, '_g_stream', None)
        if g2 is None:
            g2 = self._g_stream = torch.cuda.Stream(device=self.device)
        toggle_grad(self.g, True)               # the graph of this forward is what the G step differentiates
        g2.wait_stream(main)
        self._wait_gen_sample(g2)               # (G's BatchNorm running statistics: the z0 pass comes first)
        ops.state.pending_streams.add(g2)
        with torch.cuda.stream(g2):
            fake = self.sample_g(n)
        return fake

    def g_forward_backward(self, imgs, overlap=True, fake=None):
        toggle_grad(self.g, True)
        toggle_grad(self.d, False)
        self.optimizer_g.zero_grad()
        self._reset_arena()
        if fake is None:
            fake = self.sample_g(len(imgs))
        else:                                   # produced by early_g_forward on its own stream
            main = torch.cuda.current_stream()
            main.wait_stream(self._g_stream)
            fake.record_stream(main)
            ops.state.pending_streams.add(self._g_stream)       # its backward chain runs there too
        g_loss = self.g_loss(fake)
        self._backward(g_loss, self.optimizer_g, overlap)
        return g_loss.detach()

    def g_update(self):
        # Adam and the EMA of target_g (update_target_generator) are one kernel
        self.optimizer_g.ema_target = self._flat_target()
        self.optimizer_g.ema_lr = float(self.args.lr_target_g)
        self.optimizer_g.step()

    def d_step(self, imgs):
        out = self.d_forward_backward(imgs)
        self.d_update()
        return out

    def g_step(self, imgs):
        out = self.g_forward_backward(imgs)
        self.g_update()
        return out

    def train_batch(self, imgs, as_floats=True):
        if getattr(self, 'sync_bn', False) and len(imgs) != self.args.batch_size:
            # the statistics divide by world * (per-rank batch): shards must be equal
            raise ValueError(f'--sync-bn needs the same batch on every rank: got {len(imgs)} images, '
                             f'--batch-size is {self.args.batch_size}')
        self.g.train()
        self.d.train()
        if getattr(self.args, 'cuda_graph', False) and len(imgs) == self.args.batch_size:
            d_loss, gp, g_loss = self._train_batch_graphed(imgs)
        else:
            imgs = imgs.to(self.device, non_blocking=True)
            d_loss, gp = self.d_step(imgs)
            g_loss = self.g_step(imgs)
        if not as_floats:
            return dict(g_loss=g_loss, d_loss=d_loss, gp=gp)
        gp_val = float(gp) * self.args.grad_penalty if gp is not None else 0.
        return dict(g_loss=float(g_loss), d_loss=float(d_loss), gp=gp_val)

    # ------------------------------------------------------------------ CUDA-graph execution
    def _n_tau_draws(self):
        return 3 if hasattr(self.d, 'to_output') and hasattr(self.d.to_output, 'iqn') else 0

    def sample_z(self, n=None):
        st = getattr(self, '_st', None)
        if st is not None and st['active']:          # graph capture: read the static buffer
            z = st['z'][st['zi']]
            st['zi'] += 1
            return z
        return super().sample_z(n)

    def _static_taus(self, rows):
        st = self._st
        if not st['active']:
            return torch.rand(rows, 1).to(self.device)
        t = st['tau'][st['ti']]
        st['ti'] += 1
        return t

    def _stage_inputs(self, imgs, part=None):
        """Draw z / tau from the CPU generator in the reference's order (trainer.py:153-156, iqn.py:105-108:
        z, tau, tau, z, tau) into pinned buffers and copy them, with the images, into the static device
        buffers the graphs read.  part: None = everything; 'first' = z0 and the image copy only, 'rest' = the
        remaining draws (TTG_EARLY_GEN=1: the generator-sample graph, which reads only z0, is launched between
        the two parts so that the other CPU draws overlap it, and the image copy is issued before any draw; same
        draw order.  Measured at the end of round 2, `profiles/r2_bench_1gpu_split_staging.log`: 12.59 ms / step,
        end to end 18 573 images/s against 18 700 without it - no gain, the ~1.1 ms between the device-timed and
        the end-to-end step is the 50.9 MB pinned H2D copy in front of D(real), not the ~1 ms of CPU draws; off by
        default)."""
        st = self._st
        b, nq = self.args.batch_size, (self.d.to_output.iqn.num_quantiles if st['tau'] else 0)
        order = ['z0'] + (['t0', 't1'] if st['tau'] else []) + ['z1'] + (['t2'] if st['tau'] else [])
        if part == 'first':
            order = order[:1]
        elif part == 'rest':
            order = order[1:]
        # The pinned staging buffers are double-buffered: the host may run ahead of the GPU (as_floats=False), and
        # redrawing into a buffer whose asynchronous copy of the PREVIOUS step is still in flight would tear that
        # step's draws.  Slot k is reused only after the copies issued from it two steps ago have completed.
        if part != 'rest':
            st['slot'] ^= 1
            ev = st['pin_done'][st['slot']]
            if ev is not None:
                ev.synchronize()
        slot = st['slot']
        if part == 'first' and getattr(self, '_copy_stream', None) is not None:
            # split staging: the image batch starts travelling BEFORE the CPU draws (~1 ms per step at the headline
            # size), which then overlap the copy instead of preceding it
            cs = self._copy_stream
            cs.wait_stream(torch.cuda.current_stream())   # the previous step may still be reading the static buffer
            with torch.cuda.stream(cs):
                st['imgs'].copy_(imgs, non_blocking=True)
                self._imgs_ready.record(cs)
            imgs = None
        for key in order:
            i = int(key[1])
            if key[0] == 'z':
                torch.randn(b, self.gan_config.latent_dims, out=st['z_pin'][slot][i])
                st['z'][i].copy_(st['z_pin'][slot][i], non_blocking=True)
            else:
                torch.rand(b * nq, 1, out=st['tau_pin'][slot][i])
                st['tau'][i].copy_(st['tau_pin'][slot][i], non_blocking=True)
        if part != 'first':
            ev = st['pin_done'][slot] or torch.cuda.Event()
            ev.record()
            st['pin_done'][slot] = ev
        if part == 'rest' or imgs is None:
            return                                        # the images went with the first part
        cs = getattr(self, '_copy_stream', None)
        if cs is None:
            st['imgs'].copy_(imgs, non_blocking=True)
            return
        # the image batch travels on a copy stream while the first graph (the generator sample of the D step, which
        # does not need the images) runs; the second graph waits for `imgs_ready`
        cs.wait_stream(torch.cuda.current_stream())       # the previous step may still be reading the static buffer
        with torch.cuda.stream(cs):
            st['imgs'].copy_(imgs, non_blocking=True)
            self._imgs_ready.record(cs)

    def _capture(self, imgs):
        dev, b = self.device, self.args.batch_size
        nt = self._n_tau_draws()
        nq = self.d.to_output.iqn.num_quantiles if nt else 0
        self._st = st = dict(
            imgs=torch.empty((b,) + tuple(imgs.shape[1:]), dtype=torch.float32, device=dev),
            z=[torch.empty(b, self.gan_config.latent_dims, device=dev) for _ in range(2)],
            z_pin=[[torch.empty(b, self.gan_config.latent_dims).pin_memory() for _ in range(2)] for _ in range(2)],
            tau=[torch.empty(b * nq, 1, device=dev) for _ in range(nt)],
            tau_pin=[[torch.empty(b * nq, 1).pin_memory() for _ in range(nt)] for _ in range(2)],
            slot=0, pin_done=[None, None], zi=0, ti=0, active=False)
        # warm-up (eager, on a side stream as torch.cuda.graph requires): sets lazy kernel attributes, flattens
        # the parameter buffers, fills the packed-weight caches.  RNG state is restored afterwards so that the
        # first graphed step consumes the same draws an eager first step would have.
        rng = torch.get_rng_state()
        saved = [{k: v.clone() for k, v in m.state_dict().items()} for m in (self.g, self.target_g, self.d)]
        for opt in (self.optimizer_d, self.optimizer_g):
            opt._ensure_flat()
        opt_saved = [(o._m.clone(), o._v.clone(), o._step.clone()) for o in (self.optimizer_d, self.optimizer_g)]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            x = imgs.to(dev)
            for _ in range(2):
                self.d_step(x)
                self.g_step(x)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for m, sd in zip((self.g, self.target_g, self.d), saved):
            m.load_state_dict(sd)
        for opt, (m_, v_, s_) in zip((self.optimizer_d, self.optimizer_g), opt_saved):
            opt._m.copy_(m_); opt._v.copy_(v_); opt._step.copy_(s_)
        torch.set_rng_state(rng)
        ops.state.pack_generation += 1          # invalidate every per-tensor packed-weight cache ...
        for opt in (self.optimizer_d, self.optimizer_g):
            opt.repack()                        # ... and refill them (eagerly) from the shared buffers the graphs read
        # route z / tau draws to the static buffers while capturing
        if nt:
            self.d.to_output.iqn.tau_source = self._static_taus
        self._stage_inputs(imgs)
        st['zi'] = st['ti'] = 0
        st['active'] = True
        graphs, pool = [], None
        out = {}
        from .. import _lib
        k_before = _lib.Counters.kernels

        def seg(fn, own_pool=False):
            """own_pool: the segment gets a private memory pool of its own.  Segments that share a pool may alias each
            other's freed intermediates, which is only safe when they never run concurrently."""
            nonlocal pool
            g = torch.cuda.CUDAGraph()
            # Python's cyclic collector must not run inside a capture: collecting an OLDER trainer (its CUDA graphs and
            # their private memory pool) calls cudaFree / cudaGraphExecDestroy, which invalidates a capture in progress
            # ("operation failed due to a previous error during capture"; seen when several trainers are built in one
            # process, e.g. the test suite).  Collect before, keep the collector off while capturing.
            import gc
            gc.collect()
            ops.state.pending_streams.clear()      # (streams forked outside this capture must not be waited on inside it)
            ops.state.wgrad_pending = False
            was_enabled = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.graph(g, pool=None if own_pool else pool):
                    fn()
            finally:
                if was_enabled:
                    gc.enable()
            if not own_pool:
                pool = g.pool()
            graphs.append(g)

        # Data parallel: the bucketed NCCL all-reduces are captured INSIDE the graph.  They are launched from the
        # post-accumulate-grad hooks while backward is being captured; ProcessGroupNCCL forks its own stream off the
        # capture stream at that point and `finish()` joins it back, so in the instantiated graph each bucket's
        # exchange is a side branch that runs concurrently with the rest of backward (D: the R1 double backward and
        # the trunk below the bucket; G: the blocks below the bucket).  One graph per step on any world size.
        # TTG_DP_BLOCKING=1 keeps round 1's scheme (blocking all-reduce of the whole buffer between graph segments).
        blocking = self.world_size > 1 and os.environ.get('TTG_DP_BLOCKING', '0') == '1'
        overlap = not blocking
        def gen():
            with torch.no_grad():
                out['fake'] = self.sample_g(b)
        gen_async = _GEN_ASYNC and not blocking and not self._single_stream()
        # needs no images: runs while the host batch is still in flight (and, with gen_async, beside the step graph: then
        # its intermediates must not share memory with the step graph's)
        seg(gen, own_pool=gen_async)
        if not blocking:
            if self.world_size > 1:               # build the reducers (and their hooks) before capturing
                self._reducer(self.optimizer_d); self._reducer(self.optimizer_g)
            self._gen_done = self._gen_stream = None
            if gen_async:
                # The generator-sample graph (G forward of the D step, needs neither the images nor anything of this
                # step) is replayed on its OWN stream; the step graph waits for it through an external event-wait node
                # placed where the sample is first needed (D(fake) forward, the early G-step forward), so it overlaps
                # the image copy AND D(real) forward + the R1 inner backward.
                self._gen_stream = torch.cuda.Stream(device=self.device)
                self._gen_done = torch.cuda.Event(external=True)
                self._gen_done.record(torch.cuda.current_stream())

            def rest():
                early = self.early_g_forward(b)
                out['d_loss'], out['gp'] = self.d_forward_backward(st['imgs'], overlap, fake=out['fake'])
                self.d_update()
                out['g_loss'] = self.g_forward_backward(st['imgs'], overlap, fake=early)
                self.g_update()
            seg(rest)
            self._segments = [(graphs[0], 'imgs'), (graphs[1], None)]
        else:
            def s1():
                out['d_loss'], out['gp'] = self.d_forward_backward(st['imgs'], overlap, fake=out['fake'])
            def s2():
                self.d_update()
                out['g_loss'] = self.g_forward_backward(st['imgs'], overlap)
            seg(s1); seg(s2); seg(self.g_update)
            gd, gg = self.optimizer_d._ensure_flat().grad, self.optimizer_g._ensure_flat().grad
            self._segments = [(graphs[0], 'imgs'), (graphs[1], gd), (graphs[2], gg), (graphs[3], None)]
        self._copy_stream = torch.cuda.Stream()
        self._imgs_ready = torch.cuda.Event()
        self._graph_out = out
        self._graph_kernels = _lib.Counters.kernels - k_before      # kernels recorded in the graphs = launched per replay
        st['active'] = False
        torch.cuda.synchronize()
        # the capture pass itself executed nothing: restore nothing, the first replay is step 1

    def _train_batch_graphed(self, imgs):
        early = False
        if getattr(self, '_segments', None) is None:
            self._capture(imgs)
        elif _EARLY_GEN:
            self._stage_inputs(imgs, 'first')
            early = True
        else:
            self._stage_inputs(imgs)
        from .. import _lib
        _lib.Counters.kernels += self._graph_kernels
        gen_stream = getattr(self, '_gen_stream', None)
        for si, (graph, exchange) in enumerate(self._segments):
            if si == 0 and gen_stream is not None:
                main = torch.cuda.current_stream()
                gen_stream.wait_stream(main)              # the previous step (Adam of G, its BatchNorm buffers) is done
                with torch.cuda.stream(gen_stream):
                    graph.replay()
                    self._gen_done.record(gen_stream)
            else:
                graph.replay()
            if early and si == 0:
                self._stage_inputs(imgs, 'rest')          # CPU draws of tau / z1 while the generator sample runs
            if isinstance(exchange, str):         # 'imgs': the next graph reads the image batch
                if getattr(self, '_copy_stream', None) is not None:
                    torch.cuda.current_stream().wait_event(self._imgs_ready)
            elif exchange is not None:
                torch.distributed.all_reduce(exchange)
        # the replays changed every parameter behind Python's back (Adam, EMA of target_g): invalidate the per-tensor
        # packed-weight caches so that the next EAGER use of g / d / target_g (sampling, an eager step) repacks
        ops.state.pack_generation += 1
        o = self._graph_out
        return o['d_loss'], o['gp'], o['g_loss']

    def release_graphs(self):
        """Drop the captured CUDA graphs (the next graphed step re-captures).  Call before
        torch.distributed.destroy_process_group(): tearing the NCCL communicator down while instantiated graphs still
        hold its captured collectives hangs (measured on torch 2.11 / NCCL 2.28)."""
        torch.cuda.synchronize()
        self._segments = None
        self._graph_out = None
        import gc
        gc.collect()
        torch.cuda.synchronize()

    def parameters_changed(self):
        """Call after parameters were modified outside the optimiser (load_state_dict, manual edits): drops every
        packed-weight cache and refreshes the shared packed buffers the captured graphs read."""
        ops.state.pack_generation += 1
        for opt in (self.optimizer_d, self.optimizer_g):
            if getattr(opt, 'flat', None) is not None:
                opt.repack()

    def _flat_target(self):
        if self._target_flat is None or not self._target_flat.intact():
            self._target_flat = FlatParams(list(self.target_g.parameters()))
        return self._target_flat

    @torch.no_grad()
    def update_target_generator(self, lr=None):
        """target += (g - target) * lr_target_g over parameters only; like the reference the `lr`
        argument is ignored (trainers/cnn.py:158-165, Appendix B.1)."""
        for g_p, t_p in zip(self.g.parameters(), self.target_g.parameters()):
            src, dst = g_p.data.contiguous(), t_p.data
            ops.call('ttg_ema_flat', ops.ptr(dst), ops.ptr(src), dst.numel(), float(self.args.lr_target_g))


def make_trainer(cls, config='64', batch_size=16, gan_config=None, device='cuda', **overrides):
    """Build a trainer without the CLI / filesystem side effects (tests, bench, smoke).
    `gan_config` (a GANConfig) may be given instead of a GAN_CONFIGS key."""
    import argparse
    p = argparse.ArgumentParser()
    cls.add_args_to_parser(p)
    args = p.parse_args(['synthetic', '--batch-size', str(batch_size), '--config', str(config)])
    for k, v in overrides.items():
        if not hasattr(args, k):
            raise AttributeError(f'unknown trainer argument {k}')
        setattr(args, k, v)
    args.device = device
    if gan_config is not None:
        GAN_CONFIGS[f'_custom_{id(gan_config)}'] = gan_config
        args.config = f'_custom_{id(gan_config)}'
    t = cls.__new__(cls)
    t.args, t.steps, t.epoch, t.components, t.run_id = args, 0, 1, [], 'adhoc'
    t.build_models()
    return t
