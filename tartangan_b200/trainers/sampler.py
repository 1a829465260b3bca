"""Progress samples from the generators — the inference side of the hot path (SURVEY.md section 8 f-2), interface of
tartangan/trainers/components/image_sampler.py:12-60: a fixed batch of 32 latents drawn once at train begin
(`progress_samples`), rendered through `target_g` and `g` every `--gen-freq` batches, plus a 5x5 spherical
interpolation grid between four fixed latents through `target_g`.  The z draws come from the CPU generator in the
reference's order (32 at train begin, 4 at the first render), so a seeded run consumes the same random stream.
"""
import os

import numpy as np
import torch


def slerp(val, low, high):
    """Spherical interpolation between two latent vectors (utils/slerp.py:5-15); linear when they are parallel."""
    cos = np.dot(low / np.linalg.norm(low), high / np.linalg.norm(high))
    omega = np.arccos(np.clip(cos, -1, 1))
    s = np.sin(omega)
    if s == 0:
        return (1.0 - val) * low + val * high
    return np.sin((1.0 - val) * omega) / s * low + np.sin(val * omega) / s * high


def slerp_grid(top_left, top_right, bottom_left, bottom_right, nrows, ncols):
    """utils/slerp.py:18-33: slerp down the two side columns, then across every row; (nrows*ncols, latent)."""
    tl, tr, bl, br = (np.asarray(t, dtype=np.float32) for t in (top_left, top_right, bottom_left, bottom_right))
    rows = []
    for a in np.linspace(0, 1, nrows):
        left, right = slerp(a, tl, bl), slerp(a, tr, br)
        rows.append(np.vstack([slerp(b, left, right) for b in np.linspace(0, 1, ncols)]))
    return torch.from_numpy(np.concatenate(rows, axis=0).astype(np.float32))      # (float32 like the reference's grid)


class ImageSampler:
    def __init__(self, trainer):
        self.trainer = trainer

    @property
    def sample_root(self):
        return f'{self.trainer.output_root}/samples'

    def on_train_begin(self, steps):
        os.makedirs(self.sample_root, exist_ok=True)
        self.progress_samples = self.trainer.sample_z(32)

    def on_batch_end(self, steps):
        if steps % self.trainer.args.gen_freq == 0:
            self.output_samples(f'{self.sample_root}/sample_{steps}.png')

    def on_train_end(self, steps):
        self.output_samples(f'{self.sample_root}/sample_{steps}.png')

    def render(self):
        """-> (progress images: 16 of target_g then 16 of g, 5x5 interpolation grid of target_g); fp32 NCHW in [-1, 1].
        Like the reference the modules stay in whatever mode the trainer left them in (train: batch statistics)."""
        from .. import ops
        t = self.trainer
        with torch.no_grad(), ops.local_batchnorm():     # not part of the global batch: BatchNorm over these latents only
            imgs = torch.cat([t.target_g(self.progress_samples)[:16], t.g(self.progress_samples)[:16]], dim=0)
            if not hasattr(self, '_latent_grid_samples'):
                self._latent_grid_samples = self.sample_latent_grid(5, 5)
            grid = t.target_g(self._latent_grid_samples)
        return imgs, grid

    def output_samples(self, filename):
        from torchvision.utils import save_image
        imgs, grid = self.render()
        save_image(imgs.float().cpu(), filename, normalize=True, value_range=(-1, 1), format='png')
        grid_filename = os.path.join(os.path.dirname(filename), f'grid_{os.path.basename(filename)}')
        save_image(grid.float().cpu(), grid_filename, nrow=5, normalize=True, value_range=(-1, 1), format='png')

    def sample_latent_grid(self, nrows, ncols):
        corners = [z.cpu().numpy() for z in self.trainer.sample_z(4)]
        return slerp_grid(*corners, nrows, ncols).to(self.trainer.device)
