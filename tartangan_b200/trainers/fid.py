"""Inception score / Frechet Inception Distance of generator samples — SURVEY.md section 8 row f-4, the interface
of tartangan/inception_utils.py:180-328 and trainers/components/metrics/fid.py:10-59.

What is here: the statistics (feature mean / covariance), the matrix square root by Newton-Schulz iteration, the
Frechet distance, the Inception score and the accumulation loop over `trainer.sample_g` (this package's kernels
produce the samples).  What is NOT here: the pretrained Inception-v3 weights.  The reference downloads them through
torchvision (`inception_v3(pretrained=True)`, inception_utils.py:268); there is no network in the build / bench
environment, so the feature network is loaded from a local state-dict file (`--inception-weights`, or a torchvision
checkpoint already present under $TORCH_HOME) and a missing file is a clear error, never a silent substitute.
Evaluation side-car: plain torch ops on the trainer's device, not part of the training step.
"""
import os

import numpy as np
import torch
import torch.nn.functional as F

# ImageNet normalisation the Inception wrapper applies to [0, 1] images (inception_utils.py:20-23 uses the same constants)
_MEAN = (0.485, 0.456, 0.406)
_STD = (0.229, 0.224, 0.225)


def torch_cov(m, rowvar=False):
    """Unbiased covariance of observations (rows when rowvar=False), like np.cov."""
    if m.dim() < 2:
        m = m.view(1, -1)
    if not rowvar and m.size(0) != 1:
        m = m.t()
    m = m - m.mean(dim=1, keepdim=True)
    return m.matmul(m.t()) / (m.size(1) - 1)


def sqrt_newton_schulz(a, iters=50):
    """Principal square root of a (batch of) square matrices by the coupled Newton-Schulz iteration
    Y <- Y T, Z <- T Z with T = (3 I - Z Y) / 2, started from Y = A / |A|_F, Z = I; sqrt(A) = Y sqrt(|A|_F)."""
    batched = a.dim() == 3
    a = a if batched else a.unsqueeze(0)
    n = a.shape[-1]
    norm = a.flatten(1).norm(dim=1).view(-1, 1, 1)
    y = a / norm
    eye = torch.eye(n, dtype=a.dtype, device=a.device).expand_as(a)
    z = eye.clone()
    for _ in range(iters):
        t = 0.5 * (3.0 * eye - z.bmm(y))
        y = y.bmm(t)
        z = t.bmm(z)
    out = y * norm.sqrt()
    return out if batched else out[0]


def frechet_distance(mu1, sigma1, mu2, sigma2, iters=50):
    """|mu1 - mu2|^2 + Tr(S1 + S2 - 2 sqrt(S1 S2)) between two Gaussians (inception_utils.py:206-235)."""
    assert mu1.shape == mu2.shape and sigma1.shape == sigma2.shape
    diff = mu1 - mu2
    covmean = sqrt_newton_schulz(sigma1.mm(sigma2), iters)
    return diff.dot(diff) + torch.trace(sigma1) + torch.trace(sigma2) - 2 * torch.trace(covmean)


def inception_score(probs, num_splits=10):
    """exp(mean KL(p(y|x) || p(y))) over `num_splits` chunks of softmax outputs -> (mean, std) (inception_utils.py:239-247)."""
    probs = probs.double()
    n = probs.shape[0] // num_splits
    scores = []
    for i in range(num_splits):
        chunk = probs[i * n:(i + 1) * n]
        kl = chunk * (chunk.clamp_min(1e-30).log() - chunk.mean(0, keepdim=True).clamp_min(1e-30).log())
        scores.append(float(kl.sum(1).mean().exp()))
    return float(np.mean(scores)), float(np.std(scores))


class InceptionFeatures(torch.nn.Module):
    """torchvision Inception-v3 returning (pool3 features [B, 2048], logits [B, 1000]) for images in [-1, 1]
    (what inception_utils.WrapInception computes, :33-81): map to [0, 1], ImageNet normalisation, resize to 299x299
    bilinear (align_corners=True), the trunk up to Mixed_7c, global average pool, fc."""

    def __init__(self, net):
        super().__init__()
        self.net = net
        self.register_buffer('mean', torch.tensor(_MEAN).view(1, 3, 1, 1))
        self.register_buffer('std', torch.tensor(_STD).view(1, 3, 1, 1))

    def forward(self, x):
        x = ((x + 1.) / 2.0 - self.mean) / self.std
        if x.shape[2] != 299 or x.shape[3] != 299:
            x = F.interpolate(x, size=(299, 299), mode='bilinear', align_corners=True)
        n = self.net
        for name in ('Conv2d_1a_3x3', 'Conv2d_2a_3x3', 'Conv2d_2b_3x3'):
            x = getattr(n, name)(x)
        x = F.max_pool2d(x, kernel_size=3, stride=2)
        x = n.Conv2d_4a_3x3(n.Conv2d_3b_1x1(x))
        x = F.max_pool2d(x, kernel_size=3, stride=2)
        for name in ('Mixed_5b', 'Mixed_5c', 'Mixed_5d', 'Mixed_6a', 'Mixed_6b', 'Mixed_6c', 'Mixed_6d', 'Mixed_6e',
                     'Mixed_7a', 'Mixed_7b', 'Mixed_7c'):
            x = getattr(n, name)(x)
        pool = x.mean((2, 3))
        logits = n.fc(F.dropout(pool, training=False))
        return pool, logits


def load_inception_net(weights_path=None):
    """Inception-v3 with weights from a LOCAL file.  Raises when there is none (no download is attempted)."""
    from torchvision.models import inception_v3
    candidates = [weights_path] if weights_path else []
    hub = os.path.join(os.environ.get('TORCH_HOME', os.path.expanduser('~/.cache/torch')), 'hub', 'checkpoints')
    if os.path.isdir(hub):
        candidates += [os.path.join(hub, f) for f in sorted(os.listdir(hub)) if f.startswith('inception_v3')]
    path = next((p for p in candidates if p and os.path.isfile(p)), None)
    if path is None:
        raise FileNotFoundError('FID / IS need pretrained Inception-v3 weights: pass --inception-weights <state-dict file> '
                                '(the reference downloads them with torchvision; this environment has no network)')
    net = inception_v3(weights=None, aux_logits=True, transform_input=False, init_weights=False)
    net.load_state_dict(torch.load(path, map_location='cpu'))
    return InceptionFeatures(net.eval())


def accumulate_activations(sample, net, num_images, reference_transform=True):
    """Run `sample()` (images in [-1, 1]) through `net` until `num_images` activations exist (inception_utils.py:250-264).
    reference_transform: the reference maps the samples to [0, 1] and applies the ImageNet normalisation HERE
    (:255-259) and then hands them to WrapInception, which does both AGAIN (:41-43).  Kept by default so that numbers are
    comparable with the reference's (its moments files went through the same path); False feeds [-1, 1] images once."""
    pool, probs, have = [], [], 0
    mean = std = None
    while have < num_images:
        with torch.no_grad():
            images = sample().float()
            if reference_transform:
                if mean is None:
                    mean = torch.tensor(_MEAN, device=images.device).view(1, 3, 1, 1)
                    std = torch.tensor(_STD, device=images.device).view(1, 3, 1, 1)
                images = ((images + 1) / 2. - mean) / std
            p, logits = net(images)
        pool.append(p.float())
        probs.append(F.softmax(logits.float(), 1))
        have += p.shape[0]
    return torch.cat(pool), torch.cat(probs)


class InceptionMetrics:
    """`get(sample, n)` -> (IS mean, IS std, FID) against pre-computed moments (an .npz with `mu`, `sigma`,
    inception_utils.py:284-291).  `net` may be given (tests use a small stand-in feature network)."""

    def __init__(self, moments_path, device, weights_path=None, net=None):
        data = np.load(moments_path)
        self.mu = torch.as_tensor(data['mu']).float().to(device)
        self.sigma = torch.as_tensor(data['sigma']).float().to(device)
        self.net = (net if net is not None else load_inception_net(weights_path)).to(device)

    def get(self, sample, num_images, num_splits=10):
        pool, probs = accumulate_activations(sample, self.net, num_images)
        is_mean, is_std = inception_score(probs, num_splits)
        mu, sigma = pool.mean(0), torch_cov(pool, rowvar=False)
        fid = float(frechet_distance(mu, sigma, self.mu, self.sigma))
        return is_mean, is_std, fid


class FIDEvaluator:
    """The trainer side (components/metrics/fid.py): every `--fid-freq` batches, IS / FID of `--n-inception-imgs`
    samples of `trainer.sample_g` are appended to the logs."""

    def __init__(self, trainer, net=None):
        a = trainer.args
        self.trainer = trainer
        self.metrics = InceptionMetrics(a.inception_moments, trainer.device, getattr(a, 'inception_weights', None), net=net)

    def on_batch_end(self, steps, logs):
        a = self.trainer.args
        if steps and steps % a.fid_freq == 0:
            from .. import ops
            with ops.local_batchnorm():          # not part of the global batch: BatchNorm over these samples only
                is_mean, is_std, fid = self.metrics.get(self.trainer.sample_g, a.n_inception_imgs, num_splits=5)
            logs['fid'].append(fid)
            logs['inception_score_mean'].append(is_mean)
            logs['inception_score_std'].append(is_std)
            print('Inception Score is %3.3f +/- %3.3f' % (is_mean, is_std))
            print('FID is %5.4f' % (fid,))
