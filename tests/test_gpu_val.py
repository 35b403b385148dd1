"""GPU (B200): validation on the device against the scipy / medpy transcription (oracle/val_ref.py).  Every comparison is
exact: the zoom is a gather, and the metrics are integers up to the host's last float64 operations."""
import numpy as np
import pytest
import scipy.ndimage as nd
import torch

import oracle
import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from hpfg_b200.validation import volume_metrics_raw
from oracle import val_ref
from tests.golden.common import make_predict_case
from tests.val_cases import ACDC_SHAPES, blobs, prediction_like

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PATCH = (224, 224)


def _sweep_pairs():
    pairs = [(a, b) for a in range(2, 520, 37) for b in range(2, 520, 41)]
    pairs += [(h, p) for _, h, w in ACDC_SHAPES for p in (224, 256)] + [(w, p) for _, h, w in ACDC_SHAPES for p in (224, 256)]
    pairs += [(1, 7), (7, 1), (1, 1)]
    return sorted(set(pairs + [(b, a) for a, b in pairs]))


@pytest.mark.parametrize("dtype", [np.float32, np.uint8, np.int64])
def test_zoom_kernel_matches_scipy(dtype):
    rng = np.random.default_rng(0)
    pairs = _sweep_pairs()
    cval = 0
    for k, (n_in, n_out) in enumerate(pairs):
        m_in, m_out = pairs[(k * 7) % len(pairs)]          # the other axis from elsewhere in the sweep
        fy, fx = n_out / n_in, m_out / m_in
        if int(round(n_in * fy)) != n_out or int(round(m_in * fx)) != m_out:
            continue
        a = (rng.random((3, n_in, m_in)) * 250 + 1).astype(dtype)
        ref = np.stack([nd.zoom(p, (fy, fx), order=0) for p in a])
        got = hb.zoom_nearest(torch.from_numpy(a).to(DEV), (n_out, m_out)).cpu().numpy()
        assert got.dtype == ref.dtype and np.array_equal(got, ref), (n_in, m_in, n_out, m_out)
        cval += int((ref == 0).sum())
    assert cval > 0                                          # the out-of-range (cval) case was exercised
    a = torch.from_numpy((rng.random((2, 256, 216)) * 9 + 1).astype(dtype)).to(DEV)
    back = hb.zoom_nearest(hb.zoom_nearest(a, PATCH), (256, 216)).cpu().numpy()
    assert (back[:, :, -1] == 0).all() and (back[:, :, :-1] != 0).all()      # 224 -> 216: c = 223.00000000000003 > 223


def _check_volume(pred, lab, classes):
    """Device integers == oracle integers, and the finished metrics == medpy's (or the same RuntimeError)."""
    p, g = torch.from_numpy(pred).to(DEV), torch.from_numpy(lab).to(DEV)
    block = volume_metrics_raw(p, g, classes).cpu().numpy()
    ref = np.array([val_ref.metric_ints(pred == i, lab == i) for i in range(1, classes)], dtype=np.int64)
    assert np.array_equal(block, ref), (block, ref)
    raises = any((pred == i).any() and not (lab == i).any() for i in range(1, classes))
    if raises:
        with pytest.raises(RuntimeError, match="second supplied array"):
            hb.volume_metrics(p, g, classes)
        with pytest.raises(RuntimeError, match="second supplied array"):
            val_ref.volume_metrics(pred, lab, classes)
        return
    got, want = hb.volume_metrics(p, g, classes), val_ref.volume_metrics(pred, lab, classes)
    assert [(float(a), float(b)) for a, b in got] == [(float(a), float(b)) for a, b in want]


@pytest.mark.parametrize("shape", ACDC_SHAPES + [(16, 512, 512)])
def test_volume_metrics_random_blobs(shape):
    lab = blobs(shape, 4, sum(shape))
    _check_volume(prediction_like(lab, 4, 3 * sum(shape)), lab, 4)


@pytest.mark.parametrize("classes", list(range(2, 10)))
def test_volume_metrics_class_counts(classes):
    lab = blobs((9, 96, 80), classes, 100 + classes, background=0.0)
    _check_volume(prediction_like(lab, classes, 200 + classes), lab, classes)


def test_volume_metrics_edge_cases():
    full = np.ones((4, 12, 10), np.uint8)                                           # touches every face of the volume
    _check_volume(np.pad(np.ones((4, 10, 8), np.uint8), ((0, 0), (1, 1), (1, 1))), full, 2)
    _check_volume(full, full, 2)
    lab = blobs((6, 40, 36), 3, 1)
    _check_volume(lab, lab, 3)                                                      # identical volumes: hd95 0, dice 1
    for shape in ((1, 64, 48), (1, 1, 30), (3, 1, 1)):                               # S = 1 (every voxel a border voxel) and lines
        lab = blobs(shape, 3, 2)
        _check_volume(prediction_like(lab, 3, 4), lab, 3)
    dot_l, dot_p = np.zeros((5, 16, 16), np.uint8), np.zeros((5, 16, 16), np.uint8)
    dot_l[2, 7, 9] = dot_p[4, 0, 15] = 1                                            # one-voxel objects
    dot_l[0, 0, 0] = 3                                                              # class 3 only in the label -> (0, 0)
    _check_volume(dot_p, dot_l, 4)
    dot_p[1, 3, 3] = 2                                                              # class 2 only in the prediction -> RuntimeError
    _check_volume(dot_p, dot_l, 4)
    _check_volume(np.zeros((3, 8, 8), np.uint8), np.zeros((3, 8, 8), np.uint8), 4)  # nothing at all: (0, 0) everywhere
    with pytest.raises(L.HpfgError):
        volume_metrics_raw(torch.zeros(2, 8, 8, dtype=torch.uint8, device=DEV), torch.zeros(2, 8, 8, dtype=torch.uint8, device=DEV), 1)


def _image(shape, seed):
    g = torch.Generator().manual_seed(seed)
    coarse = torch.rand(shape[0], 1, 4, 6, generator=g)
    vol = torch.nn.functional.interpolate(coarse, size=shape[1:], mode="bilinear", align_corners=True)[:, 0]
    return (vol + 0.05 * torch.rand(shape, generator=g)).contiguous()


def test_single_volume_unet_fp32_vs_oracle_pipeline():
    """The whole of val.py:268-281 with the library's fp32 UNet against scipy's zoom, the CPU oracle network slice by slice at
    batch 1 and the medpy transcription.  Labels agree wherever the reference's top-2 softmax margin exceeds 1e-3; the metrics of
    the device's own prediction are the oracle's exactly."""
    st, _ = make_predict_case(1, 4, 1, 8, 8, 5)
    net = hb.UNet(1, 4, precision="fp32")
    net.load_state_dict(st)
    net.to(DEV)
    shape = (7, 256, 216)
    image = _image(shape, 8)
    label = torch.from_numpy(blobs(shape, 4, 9))
    margins = []

    def predict_slice(sl):
        with torch.no_grad():
            p = torch.softmax(oracle.unet_forward(st, torch.from_numpy(sl)[None, None].float(), training=False), dim=1)[0]
        top = p.topk(2, dim=0).values
        margins.append((top[0] - top[1]).numpy())
        return p.argmax(0).numpy()

    want, ref_pred = val_ref.test_single_volume(image.numpy(), label.numpy(), predict_slice, 4, PATCH)
    got = hb.test_single_volume(image[None], label[None], net, 4, patch_size=list(PATCH))
    assert not net.training
    pred = hb.predict_single_volume(image[None], net, list(PATCH)).cpu().numpy()
    margin = val_ref.zoom_nearest(np.stack(margins), shape[1:])
    sure = margin > 1e-3
    assert sure.mean() > 0.5
    assert np.array_equal(pred[sure], ref_pred[sure])
    assert (pred == ref_pred).mean() > 0.999
    own = val_ref.volume_metrics(pred, label.numpy(), 4)
    assert [tuple(map(float, m)) for m in got] == [tuple(map(float, m)) for m in own]
    if (pred == ref_pred).all():
        assert [tuple(map(float, m)) for m in got] == [tuple(map(float, m)) for m in want]


class _BinNet(torch.nn.Module):
    """A network without near-ties: logits_c = -100 (x - c/4)^2 for an image whose values sit near the centres c/4."""

    def forward(self, x):
        c = torch.arange(4, device=x.device, dtype=torch.float32).view(1, 4, 1, 1) / 4
        return -100.0 * (x - c) ** 2


def test_single_volume_without_near_ties_equals_oracle_exactly():
    net = _BinNet()
    for k, shape in enumerate(ACDC_SHAPES[:4]):
        centres = blobs(shape, 4, 30 + k).astype(np.float32) / 4
        image = centres + 0.02 * np.random.default_rng(k).random(shape, dtype=np.float32)
        label = blobs(shape, 4, 40 + k) if k % 2 else np.where(np.roll(centres, 2, axis=1) > 0, (centres * 4).astype(np.uint8), 0)

        def predict_slice(sl):
            z = -100.0 * (sl[None] - np.arange(4, dtype=np.float32)[:, None, None] / 4) ** 2
            return z.argmax(0)

        want, ref_pred = val_ref.test_single_volume(image, label, predict_slice, 4, PATCH)
        got = hb.test_single_volume(torch.from_numpy(image)[None], torch.from_numpy(label)[None], net, 4, patch_size=list(PATCH))
        assert np.array_equal(hb.predict_single_volume(torch.from_numpy(image), net, list(PATCH)).cpu().numpy(), ref_pred)
        assert [tuple(map(float, m)) for m in got] == [tuple(map(float, m)) for m in want]


def test_validation_pass_keeps_one_plan_and_unet_plus_uses_val():
    """A validation over volumes of 6..21 slices leaves one plan per model (fixed chunks, zero-padded), and UNet_Plus's logits
    path gives the same metrics as a UNet with the same backbone."""
    st, _ = make_predict_case(1, 4, 1, 8, 8, 6)
    net = hb.UNet(1, 4, precision="bf16")
    net.load_state_dict(st)
    net.to(DEV)
    plus = hb.UNet_Plus(1, 4, precision="bf16").to(DEV)
    plus.load_state_dict(st, strict=False)
    results = []
    for k, s in enumerate((6, 10, 21, 13)):
        shape = (s,) + ACDC_SHAPES[k][1:]
        image, label = _image(shape, 60 + k), torch.from_numpy(blobs(shape, 4, 70 + k))
        a = hb.test_single_volume(image[None], label[None], net, 4, patch_size=list(PATCH))
        b = hb.test_single_volume(image[None], label[None], plus, 4, patch_size=list(PATCH))
        assert [tuple(map(float, m)) for m in a] == [tuple(map(float, m)) for m in b]
        results.append(a)
    assert list(net._plans) == [((hb.validation.VAL_CHUNK, 1) + PATCH, "bf16")] and len(net._plans[list(net._plans)[0]]) == 1
    assert len(plus._plans) == 1
    with pytest.raises(ValueError):
        hb.test_single_volume(image[None], label[None].float(), net, 4, patch_size=list(PATCH))
    with pytest.raises(ValueError):
        hb.test_single_volume(image[None], label[None].long() + 300, net, 4, patch_size=list(PATCH))
