"""Validation on the device: val.py:268-281 ``test_single_volume`` with scipy's order-0 zoom and medpy's Dice / HD95
(``calculate_metric_percase``, val.py:255-265; medpy 0.4.0) on the library's kernels (csrc/val.cu).

The metrics are integer computations up to the last few float operations (counts for Dice; exact squared distances and two
ranks for numpy.percentile's linear interpolation of HD95), so the device computes the integers and the host finishes them with
the same float64 operations numpy performs: the results equal the scipy / medpy ones bit for bit."""
import math

import numpy as np
import torch

from . import _lib as L

VAL_CHUNK = 16       # zoomed slices per network call; the last chunk is zero-padded so that one plan serves every volume
_ELEM = {torch.float32: 4, torch.int32: 4, torch.uint8: 1, torch.int8: 1, torch.bool: 1, torch.int64: 8, torch.float64: 8}


def zoom_nearest(x, size):
    """``scipy.ndimage.zoom(plane, (size[0]/H, size[1]/W), order=0)`` for every [H,W] plane of the CUDA tensor x [..., H, W]
    (fp32, fp64, int64, int32, uint8, int8 or bool), returned as [..., size[0], size[1]] of the same dtype.  scipy's rule per
    axis: f = (in-1)/(out-1), c = k*f in fp64; c > in-1 gives 0, otherwise x[floor(c + 0.5)] -- so a 216-wide slice zoomed to
    224 and back has 0 in its last column.  Note that scipy's own output size is round(H * zoom), which is not always the size
    the zoom factor was computed from; ``test_single_volume`` applies that rounding."""
    L.require_cuda(x, "zoom_nearest input")
    out = torch.empty(tuple(x.shape[:-2]) + (int(size[0]), int(size[1])), device=x.device, dtype=x.dtype)
    return zoom_nearest_into(x, out)


def zoom_nearest_into(x, out):
    """zoom_nearest(x, out.shape[-2:]) written into the contiguous tensor ``out`` of x's dtype and leading shape."""
    L.require_cuda(x, "zoom_nearest input")
    if x.dtype not in _ELEM:
        raise ValueError("zoom_nearest: unsupported dtype %s" % (x.dtype,))
    if not out.is_contiguous() or out.dtype != x.dtype or out.shape[:-2] != x.shape[:-2] or out.device != x.device:
        raise ValueError("zoom_nearest: output must be a contiguous %s tensor [%s, h, w] on %s"
                         % (x.dtype, ", ".join(map(str, x.shape[:-2])), x.device))
    x = x.contiguous()
    h, w = x.shape[-2], x.shape[-1]
    n = x.numel() // max(h * w, 1)
    if n == 0 or out.numel() == 0:
        return out
    L.check(L.lib().hpfg_zoom_nearest(L.ptr(x), n, h, w, out.shape[-2], out.shape[-1], _ELEM[x.dtype], L.ptr(out),
                                      L.stream_ptr(x.device)), "hpfg_zoom_nearest")
    return out


def metrics_from_ints(block):
    """calculate_metric_percase for every class from the device's int64 block [(C-1), 6] of {|P|, |G|, |P n G|, n, d2_lo, d2_hi}.

    val.py:255-265: (0, 0) when the prediction has no voxel of the class; medpy's RuntimeError when the label has none;
    otherwise dc = 2. * |P n G| / float(|P| + |G|) (medpy binary.dc) and hd95 = numpy.percentile(distances, 95) with the
    'linear' method: vi = (n-1)*0.95, g = vi - floor(vi), a / b the square roots of the d^2 at ranks lo / hi, and
    a + (b-a)*g for g < 0.5, else b - (b-a)*(1-g) (numpy's _lerp)."""
    out = []
    for cp, cg, ci, n, d2lo, d2hi in np.asarray(block, dtype=np.int64).reshape(-1, 6).tolist():
        if cp == 0:
            out.append((0, 0))
            continue
        if cg == 0:
            raise RuntimeError('The second supplied array does not contain any binary object.')
        dice = 2. * ci / float(cp + cg)
        vi = np.float64(n - 1) * np.float64(0.95)
        g = vi - np.float64(math.floor(vi))
        a, b = np.sqrt(np.float64(d2lo)), np.sqrt(np.float64(d2hi))
        diff = b - a
        hd = b - diff * (np.float64(1) - g) if g >= 0.5 else a + diff * g
        out.append((dice, np.float64(hd)))
    return out


def volume_metrics_raw(pred, label, classes):
    """Enqueue ``hpfg_volume_metrics`` on uint8 CUDA volumes [S,H,W]; returns the int64 [(classes-1), 6] device block (no sync)."""
    L.require_cuda(pred, "pred")
    L.require_cuda(label, "label")
    if pred.dtype != torch.uint8 or label.dtype != torch.uint8:
        raise ValueError("volume_metrics_raw: pred and label must be uint8")
    if pred.shape != label.shape or pred.dim() != 3:
        raise ValueError("volume_metrics_raw: pred and label must both be [S,H,W], got %s and %s"
                         % (tuple(pred.shape), tuple(label.shape)))
    s, h, w = pred.shape
    ws_bytes = L.lib().hpfg_volume_metrics_workspace_bytes(s, h, w, classes)
    if ws_bytes < 0:
        raise L.HpfgError("hpfg_volume_metrics_workspace_bytes: %s" % L.lib().hpfg_last_error().decode())
    ws = torch.empty(ws_bytes, device=pred.device, dtype=torch.uint8)
    out = torch.empty((classes - 1, 6), device=pred.device, dtype=torch.int64)
    L.check(L.lib().hpfg_volume_metrics(L.ptr(pred.contiguous()), L.ptr(label.contiguous()), s, h, w, classes, L.ptr(out),
                                        L.ptr(ws), L.stream_ptr(pred.device)), "hpfg_volume_metrics")
    return out


def _as_u8_labels(t, what):
    if t.dtype.is_floating_point or t.dtype.is_complex:
        raise ValueError("%s must hold integer classes, got %s" % (what, t.dtype))
    if t.dtype != torch.uint8 and t.numel() and (int(t.min()) < 0 or int(t.max()) > 255):
        raise ValueError("%s must hold classes in [0, 255]" % what)
    return t.to(torch.uint8)


def volume_metrics(pred, label, classes):
    """``[calculate_metric_percase(pred == i, label == i) for i in range(1, classes)]`` (val.py:278-280) for two CUDA label
    volumes [S,H,W] (or [1,S,H,W]) of integer classes in [0, 255]: a list of (dice, hd95), (0, 0) for a class the prediction
    lacks, RuntimeError (as medpy raises it) for a class the prediction has and the label lacks."""
    pred, label = pred.reshape(pred.shape[-3:]), label.reshape(label.shape[-3:])
    block = volume_metrics_raw(_as_u8_labels(pred, "pred").contiguous(), _as_u8_labels(label, "label").contiguous(), classes)
    return metrics_from_ints(block.cpu().numpy())


def _logits(net, x):
    # main.py validates UNet_Plus through its logits-only path
    val = getattr(net, "val", None)
    return val(x) if callable(val) else net(x)


def _volume(t, what):
    t = torch.as_tensor(t)
    t = t[0] if t.dim() == 4 else t
    if t.dim() != 3:
        raise ValueError("%s must be [1,S,H,W] or [S,H,W], got %s" % (what, tuple(t.shape)))
    return t


def predict_single_volume(image, net, patch_size=[256, 256]):
    """The prediction loop of val.py:270-277 for a whole volume: every slice of ``image`` [1,S,H,W] (or [S,H,W]) resampled to
    ``patch_size`` with scipy's order-0 zoom, labelled by the network (``argmax(softmax(net(x)), 1)`` in eval mode, which the
    network is left in, as the reference leaves it), and the labels resampled back.  Returns the uint8 [S,H,W] prediction on
    the network's device.

    The network runs on chunks of VAL_CHUNK zoomed slices with the last chunk zero-padded, so volumes of any slice count share
    one plan of the network; eval-mode slices are independent, so the padding changes no label."""
    from .losses import argmax_labels
    dev = net.flat_params.device if hasattr(net, "flat_params") else torch.device("cuda", torch.cuda.current_device())
    img = _volume(image, "image").to(dev).float().contiguous()
    s, h, w = img.shape
    ph, pw = int(round(h * (patch_size[0] / h))), int(round(w * (patch_size[1] / w)))   # scipy's output shape: round(in * zoom)
    if (int(round(ph * (h / patch_size[0]))), int(round(pw * (w / patch_size[1])))) != (h, w):
        raise ValueError("test_single_volume: a %dx%d slice zoomed to %s does not zoom back to %dx%d" % (h, w, tuple(patch_size), h, w))
    n_pad = -(-s // VAL_CHUNK) * VAL_CHUNK
    x = torch.zeros((n_pad, 1, ph, pw), device=dev, dtype=torch.float32)
    zoom_nearest_into(img, x[:s, 0])
    net.eval()
    pz = torch.empty((n_pad, ph, pw), device=dev, dtype=torch.uint8)
    with torch.no_grad():
        for c0 in range(0, n_pad, VAL_CHUNK):
            pz[c0:c0 + VAL_CHUNK] = argmax_labels(_logits(net, x[c0:c0 + VAL_CHUNK]), dtype=torch.uint8)
    return zoom_nearest(pz[:s], (h, w))


def test_single_volume(image, label, net, classes, patch_size=[256, 256]):
    """val.py:268-281 on the device: ``predict_single_volume`` and calculate_metric_percase for classes 1..classes-1 against
    ``label`` (integer classes in [0, 255]).  Returns the list of (dice, hd95), as the reference does.

    image / label may be CPU tensors (the data loader's), numpy arrays or CUDA tensors; each crosses to the device once, and the
    only device-to-host read is the (classes-1)*6 integer result block."""
    label = _volume(label, "label")
    image = _volume(image, "image")
    if tuple(label.shape) != tuple(image.shape):
        raise ValueError("test_single_volume: image %s and label %s differ in shape" % (tuple(image.shape), tuple(label.shape)))
    lab = _as_u8_labels(label, "label")
    pred = predict_single_volume(image, net, patch_size)
    lab = lab.to(pred.device).contiguous()
    return metrics_from_ints(volume_metrics_raw(pred, lab, classes).cpu().numpy())
