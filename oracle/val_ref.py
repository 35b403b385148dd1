"""scipy / numpy transcription of val.py's test_single_volume (val.py:268-281) and calculate_metric_percase
(val.py:255-265) with medpy 0.4.0's ``dc`` / ``hd95`` (the version requirements.txt pins).  Test infrastructure only.

medpy is not a dependency: its two functions are restated here from medpy/metric/binary.py (``dc``, ``hd95``,
``__surface_distances``) on the scipy.ndimage calls they make.  Besides the float results this module exposes the integers
the device computes (``metric_ints``), so that the finishing arithmetic can be checked on its own."""
import numpy as np
from scipy.ndimage import binary_erosion, distance_transform_edt, generate_binary_structure, zoom

PERCENTILE = 95


def zoom_index(n_in, n_out):
    """Source index of every output index of scipy.ndimage.zoom(order=0, mode='constant', grid_mode=False) on one axis, -1
    where scipy writes cval.  scipy/ndimage/_interpolation.py zoom(): zoom = (in-1)/(out-1) as one fp64 division (1 where
    out == 1); ni_interpolation.c NI_ZoomShift: coordinate k*zoom, out of range above in-1 -> cval, order 0 -> floor(c+0.5)."""
    f = (n_in - 1) / (n_out - 1) if n_out > 1 else 1.0
    c = np.arange(n_out, dtype=np.float64) * f
    return np.where(c > n_in - 1, -1, np.floor(c + 0.5)).astype(np.int64)


def zoom_nearest(a, size):
    """``zoom`` over the last two axes of ``a`` to ``size`` = (out_h, out_w) by the rule of zoom_index."""
    iy, ix = zoom_index(a.shape[-2], size[0]), zoom_index(a.shape[-1], size[1])
    out = a[..., np.maximum(iy, 0), :][..., np.maximum(ix, 0)].copy()
    out[..., iy < 0, :] = 0
    out[..., ix < 0] = 0
    return out


def zoom_size(n, patch):
    """Output length of zoom(x, patch / n) on an axis of length n: scipy rounds n * zoom with Python's round()."""
    return int(round(n * (patch / n)))


def border(x):
    """medpy __surface_distances: X ^ binary_erosion(X, generate_binary_structure(ndim, 1), iterations=1), border_value 0."""
    return x ^ binary_erosion(x, structure=generate_binary_structure(x.ndim, 1), iterations=1)


def surface_d2(a, b):
    """Exact squared distances sd(A,B)^2 = distance_transform_edt(~border(B))[border(A)]^2 as int64 (from the EDT's feature
    transform, so no square root is involved)."""
    ba, bb = border(a), border(b)
    _, idx = distance_transform_edt(~bb, return_indices=True)
    pos = np.indices(a.shape)
    d2 = ((idx - pos) ** 2).sum(axis=0)
    return d2[ba].astype(np.int64)


def metric_ints(pred, gt):
    """{|P|, |G|, |P n G|, n, d2_lo, d2_hi} of one class: the integers behind dc and hd95 (0 for d2 when either set is empty)."""
    p, g = pred.astype(bool), gt.astype(bool)
    cp, cg, ci = int(p.sum()), int(g.sum()), int((p & g).sum())
    if cp == 0 or cg == 0:
        n = int(border(p).sum()) + int(border(g).sum())
        return [cp, cg, ci, n, 0, 0]
    d2 = np.sort(np.concatenate([surface_d2(p, g), surface_d2(g, p)]))
    n = len(d2)
    vi = (n - 1) * (PERCENTILE / 100)
    lo = int(np.floor(vi))
    hi = min(lo + 1, n - 1)
    return [cp, cg, ci, n, int(d2[lo]), int(d2[hi])]


def dc(result, reference):
    """medpy.metric.binary.dc."""
    result, reference = np.atleast_1d(result.astype(bool)), np.atleast_1d(reference.astype(bool))
    intersection = np.count_nonzero(result & reference)
    size_i1, size_i2 = np.count_nonzero(result), np.count_nonzero(reference)
    try:
        return 2. * intersection / float(size_i1 + size_i2)
    except ZeroDivisionError:
        return 0.0


def _surface_distances(result, reference):
    """medpy.metric.binary.__surface_distances (voxelspacing None, connectivity 1)."""
    result, reference = np.atleast_1d(result.astype(bool)), np.atleast_1d(reference.astype(bool))
    if 0 == np.count_nonzero(result):
        raise RuntimeError('The first supplied array does not contain any binary object.')
    if 0 == np.count_nonzero(reference):
        raise RuntimeError('The second supplied array does not contain any binary object.')
    return distance_transform_edt(~border(reference))[border(result)]


def hd95(result, reference):
    """medpy.metric.binary.hd95."""
    hd1 = _surface_distances(result, reference)
    hd2 = _surface_distances(reference, result)
    return np.percentile(np.hstack((hd1, hd2)), PERCENTILE)


def calculate_metric_percase(pred, gt):
    """val.py:255-265."""
    pred = pred.astype(np.uint8)
    gt = gt.astype(np.uint8)
    pred[pred > 0] = 1
    gt[gt > 0] = 1
    if pred.sum() > 0:
        return dc(pred, gt), hd95(pred, gt)
    return 0, 0


def volume_metrics(prediction, label, classes):
    return [calculate_metric_percase(prediction == i, label == i) for i in range(1, classes)]


def test_single_volume(image, label, predict_slice, classes, patch_size=(256, 256)):
    """val.py:268-281 with the network abstracted: ``predict_slice(x)`` maps one zoomed fp32 slice [P0,P1] to its argmax labels
    [P0,P1] (the reference's argmax(softmax(net(x)), 1) in eval mode).  image, label: [S,H,W] numpy.  Returns the metric list and
    the prediction volume."""
    prediction = np.zeros_like(label)
    for ind in range(image.shape[0]):
        sl = image[ind, :, :]
        x, y = sl.shape[0], sl.shape[1]
        sl = zoom(sl, (patch_size[0] / x, patch_size[1] / y), order=0)
        out = predict_slice(sl)
        prediction[ind] = zoom(out, (x / patch_size[0], y / patch_size[1]), order=0)
    return volume_metrics(prediction, label, classes), prediction
