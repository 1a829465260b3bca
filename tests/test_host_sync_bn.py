"""Host side of synchronised BatchNorm (--sync-bn), without a GPU: the flag, and the local_batchnorm() context that
keeps work outside the training step (progress samples, FID) on local statistics."""
import argparse
import types

import numpy as np
import pytest
import torch

from tartangan_b200 import ops
from tartangan_b200.trainers.cnn import CNNTrainer
from tartangan_b200.trainers.iqn import IQNTrainer
from tartangan_b200.trainers.trainer import Trainer


@pytest.mark.parametrize('cls', [CNNTrainer, IQNTrainer])
def test_sync_bn_flag_parses_and_round_trips(cls, tmp_path):
    p = argparse.ArgumentParser(fromfile_prefix_chars='@')
    cls.add_args_to_parser(p)
    assert p.parse_args(['synthetic']).sync_bn is False
    args = p.parse_args(['synthetic', '--sync-bn', '--batch-size', '4'])
    assert args.sync_bn is True
    argv = Trainer._args_as_argv(args)
    assert '--sync-bn' in argv
    assert '--sync-bn' not in Trainer._args_as_argv(p.parse_args(['synthetic']))
    f = tmp_path / 'config.args'
    f.write_text('\n'.join(argv) + '\n')
    again = p.parse_args([f'@{f}'])
    assert vars(again) == vars(args)


class _Group:
    """Stands in for a process group: nothing here may issue a collective on it."""


def test_local_batchnorm_clears_and_restores():
    g = _Group()
    prev = ops.state.bn_group
    try:
        ops.state.bn_group = g
        with ops.local_batchnorm():
            assert ops.state.bn_group is None
        assert ops.state.bn_group is g
        with pytest.raises(KeyError):
            with ops.local_batchnorm():
                assert ops.state.bn_group is None
                raise KeyError('x')
        assert ops.state.bn_group is g
        ops.state.bn_group = None
        with ops.local_batchnorm():
            assert ops.state.bn_group is None
        assert ops.state.bn_group is None
    finally:
        ops.state.bn_group = prev


def _recording_trainer(seen, tmp_path):
    """A trainer whose generators record the BatchNorm group they run under."""
    def gen(z):
        seen.append(ops.state.bn_group)
        return torch.zeros(len(z), 3, 4, 4)
    t = types.SimpleNamespace(g=gen, target_g=gen, device='cpu', output_root=str(tmp_path),
                              args=types.SimpleNamespace(gen_freq=1, fid_freq=1, n_inception_imgs=8))
    t.sample_z = lambda n=None: torch.randn(n or 4, 8)
    t.sample_g = lambda n=None: gen(t.sample_z(n))
    return t


def test_sampler_and_fid_use_local_statistics(tmp_path):
    from tartangan_b200.trainers import fid as F_
    from tartangan_b200.trainers.sampler import ImageSampler
    g = _Group()
    prev = ops.state.bn_group
    seen = []
    t = _recording_trainer(seen, tmp_path)
    try:
        ops.state.bn_group = g
        s = ImageSampler(t)
        s.progress_samples = t.sample_z(32)
        s.render()
        assert seen and all(v is None for v in seen)
        assert ops.state.bn_group is g

        class Net(torch.nn.Module):
            def forward(self, x):
                f = x.flatten(1)[:, :16]
                return f, f[:, :10]
        np.savez(tmp_path / 'moments.npz', mu=np.zeros(16), sigma=np.eye(16))
        ev = F_.FIDEvaluator.__new__(F_.FIDEvaluator)
        ev.trainer = t
        ev.metrics = F_.InceptionMetrics(str(tmp_path / 'moments.npz'), 'cpu', net=Net())
        seen.clear()
        logs = {'fid': [], 'inception_score_mean': [], 'inception_score_std': []}
        ev.on_batch_end(1, logs)
        assert seen and all(v is None for v in seen)
        assert len(logs['fid']) == 1
        assert ops.state.bn_group is g
    finally:
        ops.state.bn_group = prev
