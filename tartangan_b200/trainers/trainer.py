"""Trainer base — interface of tartangan/trainers/trainer.py: the same CLI flags (two-phase
argparse with @file support), epoch/batch loop, z / batch helpers, get_state/set_state and
the checkpoint layout of components/model_checkpoint.py.  The loop is the CALLER of the hot
path (train_batch); the observability side-cars of the reference (image sampler, FID, Katib /
Kubeflow / TensorBoard sinks) are out of scope (SURVEY.md §2 rows 9-10, §8f).
"""
import argparse
import json
import os
import random
import string
from collections import defaultdict
from datetime import datetime

import numpy as np
import torch

from .._lib import call, dtype_code, ptr
from .utils import set_device_from_args


def type_or_none(type_):
    def f(value):
        return None if value in (None, 'None', 'none', '') else type_(value)
    return f


class SyntheticTartanDataset(torch.utils.data.Dataset):
    """Deterministic tartan-shaped RGB images, fp32 CHW in [-1, 1] (SURVEY.md §8d)."""

    def __init__(self, size, length=4096, seed=1234):
        self.size, self.length, self.seed = size, length, seed

    def __len__(self):
        return self.length

    def __getitem__(self, i):
        return tartan_batch(self.seed + i, 1, self.size)[0]


def tartan_batch(seed, batch, size):
    g = torch.Generator().manual_seed(seed)
    ys, xs = torch.meshgrid(torch.arange(size), torch.arange(size), indexing='ij')
    twill = (((xs + ys) // 2) % 2).float()
    out = torch.empty(batch, 3, size, size)
    for i in range(batch):
        n = int(torch.randint(3, 9, (1,), generator=g))
        widths = torch.randint(1, max(2, size // 8) + 1, (n,), generator=g)
        colours = torch.rand(n, 3, generator=g)
        sett = torch.repeat_interleave(colours, widths, dim=0)
        sett = torch.cat([sett, sett.flip(0)])
        sett = sett.repeat(-(-size // sett.shape[0]), 1)[:size]
        warp = sett.t()[:, None, :].expand(3, size, size)
        weft = sett.t()[:, :, None].expand(3, size, size)
        out[i] = (twill * warp + (1 - twill) * weft) * 2 - 1
    return out


class NpzImageDataset(torch.utils.data.Dataset):
    """uint8 image stack stored in an .npz (key 'images' or first array), random-cropped to the
    generator's output size and mapped to [-1, 1] (contract of image_bytes_dataset.py:44-49).  The crop origin comes
    from Python's `random` module, row offset first: what RandomCrop does in torchvision 0.5.0, the version the
    reference pins (requirements.txt:7); torchvision >= 0.8 draws it from torch's global generator instead."""

    def __init__(self, path, size):
        data = np.load(path)
        key = 'images' if 'images' in data.files else data.files[0]
        self.images, self.size = data[key], size

    def __len__(self):
        return len(self.images)

    def __getitem__(self, i):
        img = self.images[i]
        h, w = img.shape[:2]
        y = random.randint(0, h - self.size)
        x = random.randint(0, w - self.size)
        crop = torch.from_numpy(np.ascontiguousarray(img[y:y + self.size, x:x + self.size]))
        return crop.permute(2, 0, 1).float() / 127.5 - 1.0


class DeviceImageStack:
    """Device-side input pipeline (SURVEY.md section 8 f-3): the uint8 image stack of an .npz lives in HBM and a
    batch is cropped + normalised by ONE kernel (ttg_u8_crop_normalize) instead of a per-image numpy / PIL loop and
    a host-to-device copy of fp32 pixels.  Same contract as NpzImageDataset + DataLoader(shuffle=True,
    drop_last=True): every epoch visits each image once in a random order, every visit takes a fresh uniform crop;
    batches are fp32 NCHW in [-1, 1] (what `train_batch` is given by the reference, trainers/trainer.py:84-86).
    Index / crop draws come from a CPU torch.Generator, like z and tau (trainer.py:153-156)."""

    def __init__(self, images, size, device='cuda', seed=None):
        images = torch.as_tensor(np.ascontiguousarray(images))
        if images.dtype != torch.uint8 or images.dim() != 4:
            raise ValueError('DeviceImageStack: expected a uint8 array of shape (M, H, W, C)')
        self.stack = images.to(device)
        self.size = size
        self.m, self.h, self.w, self.c = images.shape
        if size > self.h or size > self.w:
            raise ValueError(f'DeviceImageStack: crop {size} larger than the images ({self.h}x{self.w})')
        self.gen = torch.Generator()
        if seed is not None:
            self.gen.manual_seed(seed)

    def __len__(self):
        return self.m

    def crop(self, index, oy, ox, internal=False):
        """Batch for explicit (image index, crop origin) triples (int tensors of equal length)."""
        from .. import ops
        b = len(index)
        dev = self.stack.device
        # one packed host->device copy for the three int32 vectors
        meta = torch.stack([torch.as_tensor(index), torch.as_tensor(oy), torch.as_tensor(ox)]).to(torch.int32)
        meta = meta.pin_memory().to(dev, non_blocking=True) if dev.type == 'cuda' else meta
        if internal:
            out = ops.empty_nhwc(b, self.c, self.size, self.size, ops.state.act_dtype, dev)
        else:
            out = torch.empty((b, self.c, self.size, self.size), dtype=torch.float32, device=dev)
        call('ttg_u8_crop_normalize', ptr(self.stack), ptr(meta[0]), ptr(meta[1]), ptr(meta[2]), ptr(out), b, self.h,
             self.w, self.c, self.size, dtype_code(out.dtype), 0 if internal else 1)
        return out

    def epoch(self, batch_size):
        """Batches of one epoch (shuffled, drop_last)."""
        perm = torch.randperm(self.m, generator=self.gen)
        for s in range(0, self.m - batch_size + 1, batch_size):
            idx = perm[s:s + batch_size]
            oy = torch.randint(0, self.h - self.size + 1, (batch_size,), generator=self.gen)
            ox = torch.randint(0, self.w - self.size + 1, (batch_size,), generator=self.gen)
            yield self.crop(idx, oy, ox)


class Trainer:
    def __init__(self, args, components=()):
        self.args = args
        self.run_id = args.run_id if getattr(args, 'run_id', None) is not None else self._generate_run_id()
        os.makedirs(self.output_root, exist_ok=True)
        # one argument per line, so that `@{output}/{run_id}/config.args` feeds the same command line back through
        # fromfile_prefix_chars='@' (the contract of the reference's utils/cli.py:6-22 save_cli_arguments)
        argv = getattr(args, '_argv', None)
        with open(f'{self.output_root}/config.args', 'w') as f:
            f.write('\n'.join(argv if argv is not None else self._args_as_argv(args)) + '\n')
        self.components = list(components)
        self.steps = 0
        self.epoch = 1

    # ---- to be provided by CNNTrainer / IQNTrainer
    def build_models(self):
        raise NotImplementedError

    def train_batch(self, imgs):
        raise NotImplementedError

    # ---- data
    def prepare_dataset(self):
        size = self.g.max_size
        if self.args.data_path == 'synthetic':
            return SyntheticTartanDataset(size)
        if self.args.data_path.endswith('.npz'):
            if getattr(self.args, 'device_dataset', False):
                data = np.load(self.args.data_path)
                key = 'images' if 'images' in data.files else data.files[0]
                return DeviceImageStack(data[key], size, self.device)
            return NpzImageDataset(self.args.data_path, size)
        raise NotImplementedError('tartangan_b200: data_path must be "synthetic" or an .npz of uint8 images; the '
                                  'image-folder pipeline of the reference is outside the training-step scope')

    def train(self, max_steps=None):
        self.build_models()
        self.dataset = self.prepare_dataset()
        if isinstance(self.dataset, DeviceImageStack):
            class _Epochs:                       # re-iterable like a DataLoader
                def __iter__(it):
                    return self.dataset.epoch(self.args.batch_size)
            loader = _Epochs()
        else:
            loader = torch.utils.data.DataLoader(self.dataset, batch_size=self.args.batch_size, shuffle=True,
                                                 drop_last=True)
        logs = defaultdict(list)
        self._maybe_resume()
        fid = None
        if getattr(self.args, 'fid', False):
            from .fid import FIDEvaluator                 # needs --inception-moments and local Inception weights
            fid = self.fid_evaluator = FIDEvaluator(self)
        sampler = None
        if getattr(self.args, 'gen_freq', 0) and not getattr(self.args, 'no_samples', False):
            from .sampler import ImageSampler
            sampler = self.sampler = ImageSampler(self)
            sampler.on_train_begin(self.steps)          # draws the 32 progress latents (image_sampler.py:13-15)
        try:
            while self.epoch <= self.args.epochs:
                for images in loader:
                    metrics = self.train_batch(images)
                    for name, value in metrics.items():
                        logs[name].append(value)
                    # (a run resumed from step N must not immediately overwrite checkpoints/N with weights that are one
                    # step further on: the reference's `_loaded_from` guard, model_checkpoint.py:23-27)
                    if (self.steps and self.steps % self.args.checkpoint_freq == 0
                            and self.steps != getattr(self, '_loaded_from', None)):
                        self.save_checkpoint()
                    if sampler is not None:
                        sampler.on_batch_end(self.steps)
                    if fid is not None:
                        fid.on_batch_end(self.steps, logs)
                    if not self.args.quiet_logs or self.steps % self.args.log_iters == 0:
                        print(f'step {self.steps} ' + ' '.join(f'{k}={v:.4f}' for k, v in metrics.items()), flush=True)
                    self.steps += 1
                    if max_steps is not None and self.steps >= max_steps:
                        raise KeyboardInterrupt
                self.epoch += 1
        except KeyboardInterrupt:
            pass
        if sampler is not None:
            sampler.on_train_end(self.steps)
        self.save_checkpoint()
        return logs

    # ---- helpers on the hot path (trainers/trainer.py:153-176)
    def sample_z(self, n=None):
        """z ~ N(0, I) from the CPU generator, then copied to the device (trainer.py:153-156)."""
        if n is None:
            n = self.args.batch_size
        return torch.randn(n, self.gan_config.latent_dims).to(self.device)

    def sample_g(self, n=None, target_g=False, **g_kwargs):
        z = self.sample_z(n)
        return (self.target_g if target_g else self.g)(z, **g_kwargs)

    def make_adversarial_batch(self, real_data, **g_kwargs):
        generated = self.sample_g(len(real_data), **g_kwargs)
        batch = torch.cat([real_data, generated], dim=0)
        labels = torch.zeros(len(batch), 1, device=self.device)
        labels[:len(labels) // 2] = 1
        return batch, labels

    def make_generator_batch(self, real_data, **g_kwargs):
        generated = self.sample_g(len(real_data), **g_kwargs)
        return generated, torch.ones(len(generated), 1, device=self.device)

    # ---- state / checkpoints (components/model_checkpoint.py:32-74 layout)
    def get_state(self):
        return dict(epoch=self.epoch, steps=self.steps)

    def set_state(self, state):
        for key, value in state.items():
            setattr(self, key, value)

    @property
    def checkpoint_root(self):
        return f'{self.output_root}/checkpoints/{self.steps}'

    def save_checkpoint(self):
        """components/model_checkpoint.py:32-50.  --checkpoint-format reference (default): whole objects that the
        unmodified reference unpickles into ITS classes (its loader calls .state_dict() on them, :66);
        state_dict: plain state dicts (smaller; models with --spectral-norm, which have no reference twin)."""
        os.makedirs(self.checkpoint_root, exist_ok=True)
        fmt = getattr(self.args, 'checkpoint_format', 'reference')
        if fmt == 'reference' and getattr(self.args, 'spectral_norm', 'none') not in (None, 'none'):
            fmt = 'state_dict'
        for obj, name in ((self.g, 'g.pt'), (self.target_g, 'g_target.pt'), (self.d, 'd.pt'),
                          (self.optimizer_d, 'opt_d.pt'), (self.optimizer_g, 'opt_g.pt')):
            if fmt == 'reference':
                from ..checkpoint_compat import save_reference_object
                save_reference_object(obj, f'{self.checkpoint_root}/{name}')
            else:
                torch.save(obj.state_dict(), f'{self.checkpoint_root}/{name}')
        with open(f'{self.checkpoint_root}/trainer.json', 'w') as f:
            json.dump(self.get_state(), f)

    def load_checkpoint(self):
        """model_checkpoint.py:52-74.  Accepts whole objects written by the reference (its class paths resolve to the
        mirror classes through install_as_tartangan) or by save_checkpoint, and plain state dicts."""
        from .. import install_as_tartangan
        install_as_tartangan()
        for attr, name in (('g', 'g.pt'), ('target_g', 'g_target.pt'), ('d', 'd.pt'),
                           ('optimizer_d', 'opt_d.pt'), ('optimizer_g', 'opt_g.pt')):
            obj = torch.load(f'{self.checkpoint_root}/{name}', weights_only=False, map_location=self.device)
            sd = obj if isinstance(obj, dict) else obj.state_dict()     # reference saves whole objects
            getattr(self, attr).load_state_dict(sd)
        with open(f'{self.checkpoint_root}/trainer.json') as f:
            self.set_state(json.load(f))
        self._loaded_from = self.steps
        if hasattr(self, 'parameters_changed'):
            self.parameters_changed()

    def _maybe_resume(self):
        if getattr(self.args, 'resume_training_step', None):
            self.steps = self.args.resume_training_step
            self.load_checkpoint()
        elif getattr(self.args, 'resume_training_latest', False):
            root = f'{self.output_root}/checkpoints'
            ids = sorted(int(d) for d in os.listdir(root) if d.isdigit()) if os.path.isdir(root) else []
            if ids:
                self.steps = ids[-1]
                self.load_checkpoint()

    def _generate_run_id(self, suffix_len=6):
        now = datetime.now().strftime('%Y-%m-%d_%H-%M-%S')
        return f'{now}_' + ''.join(random.sample(string.ascii_letters, suffix_len))

    @property
    def device(self):
        return self.args.device

    @property
    def output_root(self):
        return f'{self.args.output}/{self.run_id}'

    # ---- CLI (trainer.py:236-313, model_checkpoint.py:110-117)
    @classmethod
    def get_component_classes(cls, args):
        return []

    @staticmethod
    def _args_as_argv(args):
        """A namespace built without a command line (tests, make_trainer) rendered as one: positional first."""
        out = [str(getattr(args, 'data_path', 'synthetic'))]
        for k, v in sorted(vars(args).items()):
            if k in ('data_path', 'device') or k.startswith('_') or v is None or v is False:
                continue
            flag = '--' + k.replace('_', '-')
            out += [flag] if v is True else [flag, str(v)]
        return out

    @classmethod
    def create_from_cli(cls, argv=None):
        import sys
        parser = argparse.ArgumentParser(description='TartanGAN trainer (B200)', fromfile_prefix_chars='@')
        cls.add_args_to_parser(parser)
        raw = list(sys.argv[1:] if argv is None else argv)
        args = parser.parse_args(raw)
        # what gets echoed to config.args: the command line with @files expanded
        expanded = []
        for a in raw:
            if a.startswith('@'):
                with open(a[1:]) as f:
                    expanded += [ln for ln in f.read().splitlines() if ln]
            else:
                expanded.append(a)
        args._argv = expanded
        set_device_from_args(args)
        print(f'Using device "{args.device}"')
        return cls(args, [])

    @classmethod
    def add_args_to_parser(cls, p):
        p.add_argument('data_path')
        p.add_argument('--batch-size', type=int, default=128)
        p.add_argument('--gen-freq', type=int, default=200, help='Output samples every N batches')
        p.add_argument('--lr-g', type=float, default=1e-4, help='Learning rate for the generator')
        p.add_argument('--lr-d', type=float, default=4e-4, help='Learning rate for the discriminator')
        p.add_argument('--lr-target-g', type=float, default=1e-3,
                       help='Exponential moving average factor for the target generator')
        p.add_argument('--no-cuda', action='store_true')
        p.add_argument('--epochs', type=int, default=10000)
        p.add_argument('--output', default='output')
        p.add_argument('--dataset-cache', default='cache/{root}_{size}.pkl')
        p.add_argument('--grad-penalty', type=float, default=5.,
                       help='Gradient penalty weight for discriminator on real data')
        p.add_argument('--config', default='64', help='Id of configuration to use. See pluggan.py.')
        p.add_argument('--model-scale', type=float, default=1.)
        p.add_argument('--cache-dataset', action='store_true')
        p.add_argument('--g-base', default='mlp')
        p.add_argument('--norm', default='bn', help='"bn" (batchnorm) or "id" (identity)')
        p.add_argument('--activation', default='relu', help='Activation function: "relu" (LeakyReLU 0.2), "selu" or "elu"')
        p.add_argument('--quiet-logs', action='store_true')
        p.add_argument('--log-iters', type=int, default=1000)
        p.add_argument('--log-progress-newlines', action='store_true')
        p.add_argument('--metrics-collector', default=None)
        p.add_argument('--run-id', type=type_or_none(str), default=None)
        p.add_argument('--fid', action='store_true')
        p.add_argument('--checkpoint-freq', type=int, default=100000)
        p.add_argument('--resume-training-step', type=type_or_none(int), default=None)
        p.add_argument('--resume-training-latest', action='store_true')
        # additive flags (defaults preserve the reference behaviour)
        p.add_argument('--precision', default='bf16', choices=('bf16', 'fp32'),
                       help='activation/conv-operand precision of the CUDA path')
        p.add_argument('--num-quantiles', type=int, default=8, help='IQN quantile count (reference: 8)')
        p.add_argument('--cuda-graph', action='store_true',
                       help='run the training step as CUDA graphs (static shapes; z/tau staged from the CPU generator)')
        p.add_argument('--device-dataset', action='store_true',
                       help='keep the uint8 .npz image stack in GPU memory; crop + normalise batches with one kernel')
        # components/metrics/fid.py:51-59 (enabled by --fid)
        p.add_argument('--inception-moments', type=type_or_none(str), default=None,
                       help='Path to pre-calculated inception moments (.npz with mu, sigma)')
        p.add_argument('--n-inception-imgs', default=1000, type=int)
        p.add_argument('--cleanup-inception-model', action='store_true')
        p.add_argument('--fid-freq', default=10000, type=int, help='Calculate test metrics every N batches')
        p.add_argument('--inception-weights', type=type_or_none(str), default=None,
                       help='local Inception-v3 state dict (no network: nothing is downloaded)')
        p.add_argument('--no-samples', action='store_true', help='do not render progress samples (no z draws for them)')
        p.add_argument('--checkpoint-format', default='reference', choices=('reference', 'state_dict'),
                       help='reference: whole pickled objects readable by the unmodified reference; state_dict: state dicts')
        p.add_argument('--spectral-norm', default='none', choices=('none', 'd', 'g', 'gd'),
                       help='spectral-normalised convolutions (power iteration, torch.nn.utils.spectral_norm '
                            'semantics) in the discriminator and / or the generator')
        p.add_argument('--attention', type=type_or_none(str), default=None,
                       help='comma-separated block indices with self-attention (overrides the config)')
        p.add_argument('--sync-bn', action='store_true',
                       help='data parallel: BatchNorm statistics over the global batch (all-reduced over the ranks) '
                            'instead of each rank\'s shard; the training step then runs on one stream')
