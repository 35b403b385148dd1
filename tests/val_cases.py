"""Seeded label volumes for the validation tests: smooth random blobs (the argmax of upsampled noise fields), as ACDC's
structures are, plus the edge cases of medpy's metrics."""
import numpy as np
import scipy.ndimage as nd

ACDC_SHAPES = [(10, 256, 216), (8, 232, 256), (6, 154, 224), (12, 224, 224), (18, 181, 157)]


def blobs(shape, classes, seed, coarse=8, background=0.3):
    """[S,H,W] uint8 labels in [0, classes): argmax of `classes` smooth noise fields, background boosted by `background`."""
    rng = np.random.default_rng(seed)
    s, h, w = shape
    cs = (max(2, s // 3), max(2, h // coarse), max(2, w // coarse))
    f = rng.standard_normal((classes,) + cs)
    f = np.stack([nd.zoom(fc, (s / cs[0], h / cs[1], w / cs[2]), order=1)[:s, :h, :w] for fc in f])
    f[0] += background
    return f.argmax(0).astype(np.uint8)


def prediction_like(label, classes, seed, flip=0.02):
    """A plausible prediction of `label`: shifted by a voxel or two in-plane, with a few small blobs of other classes."""
    rng = np.random.default_rng(seed + 1)
    p = np.roll(label, (int(rng.integers(-2, 3)), int(rng.integers(-2, 3))), axis=(1, 2)).copy()
    noise = blobs(label.shape, classes, seed + 2, coarse=4, background=0.0)
    m = rng.random(label.shape) < flip
    m = nd.binary_dilation(m, iterations=1)
    p[m] = noise[m]
    return p
