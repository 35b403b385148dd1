"""CPU: the scipy / numpy transcription of val.py's test_single_volume (oracle/val_ref.py) against scipy itself, and the
host-side finishing of hpfg_b200.validation against the oracle's integers -- bit for bit."""
import numpy as np
import pytest
import scipy.ndimage as nd
from scipy.ndimage import binary_erosion, distance_transform_edt, generate_binary_structure

from oracle import val_ref
from hpfg_b200.validation import metrics_from_ints
from tests.val_cases import ACDC_SHAPES, blobs, prediction_like


def _zoom_pairs():
    pairs = [(n_in, n_out) for n_in in range(2, 520, 23) for n_out in range(2, 520, 31)]
    pairs += [(224, 216), (216, 224), (256, 224), (224, 256), (154, 224), (224, 154), (232, 224), (224, 232), (181, 224),
              (224, 181), (1, 5), (5, 1), (1, 1)]
    return pairs


def test_zoom_rule_matches_scipy():
    cval_hits = 0
    for n_in, n_out in _zoom_pairs():
        fac = n_out / n_in
        if int(round(n_in * fac)) != n_out:        # scipy's output size is round(in * zoom)
            continue
        a = (np.arange(n_in, dtype=np.float64) + 1)[:, None] * np.ones((1, 2))
        z = nd.zoom(a, (fac, 1.0), order=0)[:, 0]
        idx = val_ref.zoom_index(n_in, n_out)
        cval_hits += int((idx < 0).sum())
        assert np.array_equal(z, np.where(idx < 0, 0.0, idx + 1.0)), (n_in, n_out)
    assert cval_hits > 0
    assert val_ref.zoom_index(224, 216)[-1] == -1                      # c = 223.00000000000003 > 223


@pytest.mark.parametrize("dtype", [np.float32, np.uint8, np.int64])
def test_zoom_nearest_matches_scipy_on_acdc_planes(dtype):
    rng = np.random.default_rng(3)
    for _, h, w in ACDC_SHAPES:
        for src, dst in (((h, w), (224, 224)), ((224, 224), (h, w))):
            a = (rng.random(src) * 200).astype(dtype)
            z = nd.zoom(a, (dst[0] / src[0], dst[1] / src[1]), order=0)
            assert z.dtype == a.dtype and np.array_equal(val_ref.zoom_nearest(a, dst), z)


def _direct(pred, gt):
    """calculate_metric_percase written straight from scipy (no oracle helpers)."""
    if pred.sum() == 0:
        return 0, 0
    fp = generate_binary_structure(3, 1)
    bp, bg = pred ^ binary_erosion(pred, structure=fp, iterations=1), gt ^ binary_erosion(gt, structure=fp, iterations=1)
    d = np.hstack((distance_transform_edt(~bg)[bp], distance_transform_edt(~bp)[bg]))
    return 2. * np.count_nonzero(pred & gt) / float(pred.sum() + gt.sum()), np.percentile(d, 95)


def _cases():
    out = []
    for k, shape in enumerate([(10, 64, 54), (6, 40, 56), (1, 48, 40), (3, 17, 23)]):
        lab = blobs(shape, 4, 10 + k)
        out.append((lab, prediction_like(lab, 4, 20 + k), 4))
    full = np.ones((4, 12, 10), np.uint8)                                 # an object touching every face
    out.append((full, np.pad(np.ones((4, 10, 8), np.uint8), ((0, 0), (1, 1), (1, 1))), 2))
    dot_l, dot_p = np.zeros((5, 16, 16), np.uint8), np.zeros((5, 16, 16), np.uint8)
    dot_l[2, 7, 9] = 1                                                     # one-voxel objects
    dot_p[4, 0, 15] = 1
    dot_p[1, 3, 3] = 2                                                     # class 2: in pred only -> RuntimeError
    dot_l[0, 0, 0] = 3                                                     # class 3: in label only -> (0, 0)
    out.append((dot_l, dot_p, 4))
    return out


def test_oracle_metrics_match_direct_scipy():
    for lab, pred, classes in _cases():
        for i in range(1, classes):
            p, g = pred == i, lab == i
            if p.sum() and not g.sum():
                with pytest.raises(RuntimeError, match="second supplied array"):
                    val_ref.calculate_metric_percase(p, g)
                continue
            got, ref = val_ref.calculate_metric_percase(p, g), _direct(p, g)
            assert got[0] == ref[0] and got[1] == ref[1], (i, got, ref)


def test_oracle_integers_are_the_surface_distances():
    lab = blobs((7, 50, 44), 3, 5)
    pred = prediction_like(lab, 3, 6)
    for i in (1, 2):
        p, g = pred == i, lab == i
        d = np.sort(np.hstack((val_ref._surface_distances(p, g), val_ref._surface_distances(g, p))))
        d2 = np.sort(np.concatenate([val_ref.surface_d2(p, g), val_ref.surface_d2(g, p)]))
        assert np.array_equal(np.sqrt(d2.astype(np.float64)), d)
        ints = val_ref.metric_ints(p, g)
        assert ints[:4] == [int(p.sum()), int(g.sum()), int((p & g).sum()), len(d)]


def test_finishing_reproduces_oracle_bit_for_bit():
    n_checked = 0
    for lab, pred, classes in _cases():
        block = np.array([val_ref.metric_ints(pred == i, lab == i) for i in range(1, classes)], dtype=np.int64)
        present = [(pred == i).any() and not (lab == i).any() for i in range(1, classes)]
        if any(present):
            with pytest.raises(RuntimeError, match="second supplied array"):
                metrics_from_ints(block)
            keep = [k for k, bad in enumerate(present) if not bad]
            got = metrics_from_ints(block[keep])
            ref = [val_ref.calculate_metric_percase(pred == i + 1, lab == i + 1) for i in keep]
        else:
            got, ref = metrics_from_ints(block), val_ref.volume_metrics(pred, lab, classes)
        assert len(got) == len(ref)
        for a, b in zip(got, ref):
            assert a[0] == b[0] and a[1] == b[1], (a, b)
            n_checked += 1
    assert n_checked >= 12
    assert metrics_from_ints(np.zeros((2, 6), np.int64)) == [(0, 0), (0, 0)]


def test_finishing_lerp_matches_numpy_percentile():
    rng = np.random.default_rng(1)
    for _ in range(500):
        n = int(rng.integers(1, 3000))
        d2 = np.sort(rng.integers(0, 5000, n))
        vi = (n - 1) * 0.95
        lo = int(np.floor(vi))
        hi = min(lo + 1, n - 1)
        (dice, hd), = metrics_from_ints([[3, 4, 2, n, d2[lo], d2[hi]]])
        assert hd == np.percentile(np.sqrt(d2.astype(np.float64)), 95) and dice == 2. * 2 / 7.
