"""GPU (B200): the fused loss kernels of csrc/loss.cu against fp64 references at every class count they are built for.

hpfg_ssl_loss (SUP, MT, CPS, UAMT), hpfg_ict_loss, hpfg_s4cv_loss and hpfg_dice_loss are templates on the class count and
accept C = 2..8; hpfg_softmax_mse accepts C = 1..8.  Every case compares the kernel with an fp64 reference of the same fp32
inputs: the oracle's restatements run on .double() tensors, gradients by autograd.  The shapes reach the kernels' edges: one
quad per image, 15 quads per image, labeled quads far beyond the one-launch Mean-Teacher grid, mostly unlabeled batches, and
an unlabeled batch larger than that grid holds at once.  Bars: 1e-5 relative on values, 1e-5 relative L2 on gradients (the
labeled and the unlabeled images each on their own), pseudo-labels and mask counts exact.  Each test prints its worst errors
(shown by pytest -rP).

Run as a script (``python -m tests.test_gpu_loss_classes OUT``) it writes the Mean-Teacher cases' kernel results to OUT: the
Mean-Teacher test runs it with HPFG_LOSS_MT_ONE=0, which the library reads once per process, to check the two-launch path."""
import os
import subprocess
import sys

import pytest
import torch

import oracle
import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from hpfg_b200.losses import dice_loss_raw
from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLASSES = list(range(2, 9))
# (n_l, n_u, H, W).  H x W: one quad per image, 15 quads, 196 quads.  With one unlabeled image of at most 196 quads the
# one-launch Mean-Teacher kernel runs one CTA; (8, 1) then gives its labeled phases 8x more quads than threads; (1, 12) is a
# batch of mostly unlabeled images.
CASES = [(n_l, n_u, h, w) for h, w in ((2, 2), (6, 10), (28, 28)) for n_l, n_u in ((1, 1), (3, 2), (8, 1), (1, 12))]
# Mean-Teacher at C = 4 and 8 only: 150528 unlabeled quads, more than the one-launch kernel's resident threads (at most
# 3 CTAs of 256 threads per SM), so its grid is capped and its unlabeled phase loops as well
BIG = (12, 12, 224, 224)
CE, DICE = 0.3, 0.9          # non-default Med_Sup_Loss coefficients of the SUP and MT cases
ONE_LAUNCH = os.environ.get("HPFG_LOSS_MT_ONE", "1").strip() != "0"


def _gen(salt, C, i):
    return torch.Generator().manual_seed(100000 * salt + 100 * C + i)


def _logits(g, n, C, h, w):
    return 2 * torch.randn(n, C, h, w, generator=g)


def _peer(g, n, C, h, w):
    """Logits whose argmax is read: integer steps plus 0.05*c, so that fp32 and fp64 softmaxes have the same maximum."""
    return torch.randint(-6, 7, (n, C, h, w), generator=g).float() + 0.05 * torch.arange(C).view(1, -1, 1, 1)


def _labels(g, n, C, h, w):
    """Class ids, about 10 % of them 255, with one class (drawn per case) in no label map: its Dice denominator is Z + smooth."""
    absent = int(torch.randint(0, C, (1,), generator=g))
    y = torch.randint(0, C - 1, (n, h, w), generator=g)
    y += (y >= absent).long()
    y[torch.rand(n, h, w, generator=g) < 0.1] = 255
    y.view(-1)[0] = (absent + 1) % C        # at least one pixel counts for CE
    return y


def _weights(C):
    return [0.4 + 0.25 * c for c in range(C)]


def _sup64(s, y, C, weight=None, ce=0.5, dice=0.5):
    """Med_Sup_Loss of fp64 logits, its Dice term weighted as DiceLoss(weight=): (loss, CE, Dice)."""
    ce_v = oracle.ce_loss(s, y)
    dice_v = oracle.dice_loss(torch.softmax(s, 1), y.unsqueeze(1), C, weight=weight)
    return ce * ce_v + dice * dice_v, ce_v, dice_v


def _dice64(p, target, n_cls):
    """DiceLoss (utils/loss/diceloss.py:155-191) in fp64: class c <=> target == c (the reference's one-hot on a float map)."""
    loss = 0.0
    for c in range(n_cls):
        t = (target == c).double()
        inter, y, z = (p[:, c] * t).sum(), (t * t).sum(), (p[:, c] * p[:, c]).sum()
        loss = loss + 1 - (2 * inter + 1e-5) / (z + y + 1e-5)
    return loss / n_cls


def _argmax32(z):
    """The first maximum of torch's fp32 softmax."""
    return torch.argmax(torch.softmax(z.float(), 1), 1)


def _n_valid(y):
    return float((y != 255).sum())


class _Worst:
    """Checks one test's values and gradients and keeps the largest relative errors, printed by report()."""

    def __init__(self, what):
        self.what, self.value, self.grad = what, 0.0, 0.0

    def scalars(self, got, want, exact=()):
        """got: the kernel's scalars; want: the reference's.  Entries in `exact` and zeros must match exactly."""
        for k, (a, b) in enumerate(zip(got.tolist(), want)):
            b = float(b)
            if k in exact or b == 0.0:
                assert a == b, (self.what, k, a, b)
                continue
            e = abs(a - b) / abs(b)
            assert e <= 1e-5, (self.what, k, a, b, e)
            self.value = max(self.value, e)

    def tensor(self, got, want, n_l=None, kind="grad"):
        """Relative L2 within 1e-5; with n_l, the first n_l images and the rest each on their own."""
        for part in ([slice(None)] if n_l is None else [slice(0, n_l), slice(n_l, None)]):
            e = rel_l2(got[part], want[part])
            assert e < 1e-5, (self.what, kind, part, e)
            setattr(self, kind, max(getattr(self, kind), e))

    def report(self):
        print("%s: worst value rel %.2e, worst gradient rel-l2 %.2e" % (self.what, self.value, self.grad))


def _same(a, b, keys):
    for k in keys:
        assert torch.equal(a[k], b[k]), k


def _dev(x):
    return torch.tensor(x, device=DEV, dtype=torch.float32)


# ------------------------------------------------------------------------------------------------------------ SUP
@pytest.mark.parametrize("C", CLASSES)
def test_sup_loss_matches_fp64(C):
    wst = _Worst("hpfg_ssl_loss SUP C=%d" % C)
    for i, (n_l, n_u, h, w) in enumerate(CASES):
        g = _gen(1, C, i)
        s, y = _logits(g, n_l + n_u, C, h, w), _labels(g, n_l, C, h, w)
        kw = dict(class_weights=_weights(C), ce_coef=CE, dice_coef=DICE)
        r = hb.ssl_loss_raw(L.LOSS_SUP, s.to(DEV), None, y.to(DEV), n_l, **kw)
        s64 = s.double().requires_grad_(True)
        loss, ce, dice = _sup64(s64[:n_l], y, C, _weights(C), CE, DICE)
        loss.backward()
        wst.scalars(r["scalars"], [loss, loss, 0, ce, dice, _n_valid(y), 0, 0], exact=(5,))
        wst.tensor(r["dstudent"], s64.grad, n_l)
        rd = hb.ssl_loss_raw(L.LOSS_SUP, s.to(DEV), None, y.to(DEV), n_l, cons_weight_dev=_dev([0.0]), **kw)
        _same(rd, r, ("scalars", "dstudent"))
    wst.report()


# ------------------------------------------------------------------------------------------------------------ MT
MT_W = 0.37


def _mt_cases(C):
    return CASES + ([BIG] if C in (4, 8) else [])


def _mt_inputs(C, i, case):
    n_l, n_u, h, w = case
    g = _gen(2, C, i)
    return _logits(g, n_l + n_u, C, h, w), _logits(g, n_u, C, h, w), _labels(g, n_l, C, h, w)


def _mt_kernel(C, s, t, y, n_l, **kw):
    """hpfg_ssl_loss in MT mode, and how many kernels it launched."""
    before = L.lib().hpfg_launch_count()
    r = hb.ssl_loss_raw(L.LOSS_MT, s.to(DEV), t.to(DEV), y.to(DEV), n_l, class_weights=_weights(C), ce_coef=CE,
                        dice_coef=DICE, **kw)
    return r, L.lib().hpfg_launch_count() - before


def _mt_two_launch_child(out):
    res = {}
    for C in CLASSES:
        for i, case in enumerate(_mt_cases(C)):
            s, t, y = _mt_inputs(C, i, case)
            r, launches = _mt_kernel(C, s, t, y, case[0], cons_weight=MT_W)
            res["%d,%d" % (C, i)] = dict(scalars=r["scalars"].cpu(), dstudent=r["dstudent"].cpu(), launches=launches)
    torch.save(res, out)


@pytest.fixture(scope="module")
def mt_two_launch(tmp_path_factory):
    """The MT cases through the reduce + gradient launches (the exact-global data-parallel mode's kernels), from a child
    process started with HPFG_LOSS_MT_ONE=0."""
    out = tmp_path_factory.mktemp("mt_two_launch") / "results.pt"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-m", "tests.test_gpu_loss_classes", str(out)]
    p = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, HPFG_LOSS_MT_ONE="0"), capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, (p.stdout[-2000:], p.stderr[-4000:])
    return torch.load(out, weights_only=True)


@pytest.mark.parametrize("C", CLASSES)
def test_mt_loss_matches_fp64_in_one_and_two_launches(C, mt_two_launch):
    wst = _Worst("hpfg_ssl_loss MT C=%d" % C)
    wst2 = _Worst("hpfg_ssl_loss MT, two launches, C=%d" % C)
    for i, case in enumerate(_mt_cases(C)):
        n_l, n_u, h, w = case
        if case == BIG:
            assert n_u * h * w // 4 > torch.cuda.get_device_properties(DEV).multi_processor_count * 3 * 256
        s, t, y = _mt_inputs(C, i, case)
        r, launches = _mt_kernel(C, s, t, y, n_l, cons_weight=MT_W)
        assert launches == (1 if ONE_LAUNCH else 2)
        s64 = s.double().requires_grad_(True)
        sup, ce, dice = _sup64(s64[:n_l], y, C, _weights(C), CE, DICE)
        cons = oracle.mt_consistency(s64[n_l:], t.double())
        loss = sup + MT_W * cons
        loss.backward()
        want = [loss, sup, cons, ce, dice, _n_valid(y), 0, 0]
        wst.scalars(r["scalars"], want, exact=(5,))
        wst.tensor(r["dstudent"], s64.grad, n_l)
        rd, _ = _mt_kernel(C, s, t, y, n_l, cons_weight_dev=_dev([MT_W]))
        _same(rd, r, ("scalars", "dstudent"))
        # the two-launch path: the same reference, and the one-launch results up to the order of its sums
        two = mt_two_launch["%d,%d" % (C, i)]
        assert two["launches"] == 2
        wst2.scalars(two["scalars"], want, exact=(5,))
        wst2.tensor(two["dstudent"], s64.grad, n_l)
        for k, (a, b) in enumerate(zip(two["scalars"].tolist(), r["scalars"].tolist())):
            assert abs(a - b) <= 1e-6 * abs(b), (k, a, b)
        assert rel_l2(two["dstudent"], r["dstudent"]) < 1e-6
    wst.report()
    wst2.report()


# ------------------------------------------------------------------------------------------------------------ CPS
@pytest.mark.parametrize("C", CLASSES)
def test_cps_loss_matches_fp64(C):
    wst = _Worst("hpfg_ssl_loss CPS C=%d" % C)
    cw = 0.45
    for i, (n_l, n_u, h, w) in enumerate(CASES):
        g = _gen(3, C, i)
        o1, o2, y = _peer(g, n_l + n_u, C, h, w), _peer(g, n_l + n_u, C, h, w), _labels(g, n_l, C, h, w)
        r = hb.ssl_loss_raw(L.LOSS_CPS, o1.to(DEV), o2.to(DEV), y.to(DEV), n_l, cons_weight=cw, want_pseudo=True)
        a64, b64 = o1.double().requires_grad_(True), o2.double().requires_grad_(True)
        sup, semi, pl1, pl2 = oracle.cps_losses(a64, b64, y, n_l, C)
        loss = sup + cw * semi
        loss.backward()
        _, ce1, dice1 = _sup64(a64[:n_l].detach(), y, C)
        wst.scalars(r["scalars"], [loss, sup, semi, ce1, dice1, _n_valid(y), 0, 0], exact=(5,))
        wst.tensor(r["dstudent"], a64.grad, n_l)
        wst.tensor(r["dother"], b64.grad, n_l)
        assert torch.equal(r["pseudo1"].cpu(), _argmax32(o1[n_l:])) and torch.equal(r["pseudo2"].cpu(), _argmax32(o2[n_l:]))
        assert torch.equal(pl1, _argmax32(o1[n_l:])) and torch.equal(pl2, _argmax32(o2[n_l:]))
        rd = hb.ssl_loss_raw(L.LOSS_CPS, o1.to(DEV), o2.to(DEV), y.to(DEV), n_l, cons_weight_dev=_dev([cw]), want_pseudo=True)
        _same(rd, r, ("scalars", "dstudent", "dother", "pseudo1", "pseudo2"))
    wst.report()


# ------------------------------------------------------------------------------------------------------------ UAMT
def _gap_threshold(unc):
    """An fp32 threshold in the widest gap between neighbouring sorted uncertainties from the 25th to the 55th percentile,
    so that the kernel's fp32 entropies and the fp64 ones fall on the same side of it."""
    v = unc.flatten().sort().values
    lo = int(0.25 * (v.numel() - 1))
    hi = max(int(0.55 * (v.numel() - 1)), lo + 1)
    k = int((v[lo + 1:hi + 1] - v[lo:hi]).argmax()) + lo
    thr = float(torch.tensor(float(v[k] + v[k + 1]) / 2, dtype=torch.float32))
    assert (unc - thr).abs().min().item() > 1e-4, "no gap of 2e-4 near the 40th percentile"
    return thr


@pytest.mark.parametrize("T", [1, 8])
@pytest.mark.parametrize("C", CLASSES)
def test_uamt_loss_matches_fp64(C, T):
    wst = _Worst("hpfg_ssl_loss UAMT T=%d C=%d" % (T, C))
    cw = 0.53
    for i, (n_l, n_u, h, w) in enumerate(CASES):
        g = _gen(40 + T, C, i)
        s, t, y = _logits(g, n_l + n_u, C, h, w), _logits(g, n_u, C, h, w), _labels(g, n_l, C, h, w)
        mc = t.repeat(T, 1, 1, 1) + 0.5 * torch.randn(T * n_u, C, h, w, generator=g)    # the teacher's T noisy passes
        # the mask keeps the pixels where the teacher is sure.  A student that mildly prefers the next class there keeps the
        # few masked pixels of the small cases well conditioned: (p - q)^2 is no square of a difference of nearly equal fp32
        # probabilities, and no softmax gradient is a cancellation at a saturated pixel
        s[n_l:] = 0.5 * t.roll(1, 1) + 0.3 * torch.randn(n_u, C, h, w, generator=g)
        s64, t64, mc64 = s.double().requires_grad_(True), t.double(), mc.double()
        _, unc, _ = oracle.uamt_consistency(s64[n_l:].detach(), t64, mc64, T, 0.0)
        thr = _gap_threshold(unc)
        kw = dict(mc_logits=mc.to(DEV), mc_passes=T)
        r = hb.ssl_loss_raw(L.LOSS_UAMT, s.to(DEV), t.to(DEV), y.to(DEV), n_l, cons_weight=cw, uamt_threshold=thr, **kw)
        sup, ce, dice = _sup64(s64[:n_l], y, C)
        cons, _, mask = oracle.uamt_consistency(s64[n_l:], t64, mc64, T, thr)
        loss = sup + cw * cons
        loss.backward()
        wst.scalars(r["scalars"], [loss, sup, cons, ce, dice, _n_valid(y), mask.sum(), 0], exact=(5, 6))
        wst.tensor(r["dstudent"], s64.grad, n_l)
        rd = hb.ssl_loss_raw(L.LOSS_UAMT, s.to(DEV), t.to(DEV), y.to(DEV), n_l, cons_weight_dev=_dev([cw]), uamt_threshold=0.0,
                             uamt_threshold_dev=_dev([thr]), **kw)
        _same(rd, r, ("scalars", "dstudent"))
    wst.report()


# ------------------------------------------------------------------------------------------------------------ ICT
@pytest.mark.parametrize("C", CLASSES)
def test_ict_loss_matches_fp64(C):
    wst = _Worst("hpfg_ict_loss C=%d" % C)
    cw = 0.41
    for i, (n_l, n_u, h, w) in enumerate(CASES):
        g = _gen(5, C, i)
        s, t, y = _logits(g, n_l + n_u, C, h, w), _logits(g, 2 * n_u, C, h, w), _labels(g, n_l, C, h, w)
        lam = torch.rand(n_u, generator=g)
        r = hb.ict_loss_raw(s.to(DEV), t.to(DEV), lam.to(DEV), y.to(DEV), n_l, cons_weight=cw)
        s64 = s.double().requires_grad_(True)
        sup, cons = oracle.ict_losses(s64, t.double(), lam, y, n_l, C)
        loss = sup + cw * cons
        loss.backward()
        _, ce, dice = _sup64(s64[:n_l].detach(), y, C)
        wst.scalars(r["scalars"], [loss, sup, cons, ce, dice, _n_valid(y), 0, 0], exact=(5,))
        wst.tensor(r["dstudent"], s64.grad, n_l)
        rd = hb.ict_loss_raw(s.to(DEV), t.to(DEV), lam.to(DEV), y.to(DEV), n_l, cons_weight_dev=_dev([cw]))
        _same(rd, r, ("scalars", "dstudent"))
    wst.report()


# ------------------------------------------------------------------------------------------------------------ S4CV
@pytest.mark.parametrize("teacher", [False, True], ids=["no_teacher", "teacher"])
@pytest.mark.parametrize("C", CLASSES)
def test_s4cv_loss_matches_fp64(C, teacher):
    wst = _Worst("hpfg_s4cv_loss %s C=%d" % ("teacher" if teacher else "no teacher", C))
    cps_w, mt_w = 0.7, 0.23
    for i, (n_l, n_u, h, w) in enumerate(CASES):
        g = _gen(6, C, 2 * i + teacher)
        o1, o2, y = _peer(g, n_l + n_u, C, h, w), _peer(g, n_l + n_u, C, h, w), _labels(g, n_l, C, h, w)
        t = _logits(g, n_u, C, h, w) if teacher else None
        r = hb.s4cv_loss_raw(o1.to(DEV), o2.to(DEV), t.to(DEV) if teacher else None, y.to(DEV), n_l, cps_weight=cps_w,
                             mt_weight=mt_w, want_pseudo=True)
        a64, b64 = o1.double().requires_grad_(True), o2.double().requires_grad_(True)
        t64 = t.double() if teacher else None
        loss, sup, semi, pl1, pl2 = oracle.s4cv_losses(a64, b64, t64, y, n_l, C, cps_w, mt_w)
        loss.backward()
        with torch.no_grad():
            _, ce1, dice1 = _sup64(a64[:n_l], y, C)
            p1, p2 = torch.softmax(a64[n_l:], 1), torch.softmax(b64[n_l:], 1)
            ps = oracle.dice_loss(p1, pl2.unsqueeze(1), C) + oracle.dice_loss(p2, pl1.unsqueeze(1), C)
            cl = 0.0
            if teacher:
                q = torch.softmax(t64, 1)
                cl = ((p1 - q) ** 2).mean() + ((p2 - q) ** 2).mean()
        wst.scalars(r["scalars"], [loss, sup, semi, ce1, dice1, _n_valid(y), ps, cl], exact=(5,))
        wst.tensor(r["dstudent"], a64.grad, n_l)
        wst.tensor(r["dother"], b64.grad, n_l)
        assert torch.equal(r["pseudo1"].cpu(), _argmax32(o1[n_l:])) and torch.equal(r["pseudo2"].cpu(), _argmax32(o2[n_l:]))
        assert torch.equal(pl1, _argmax32(o1[n_l:])) and torch.equal(pl2, _argmax32(o2[n_l:]))
        rd = hb.s4cv_loss_raw(o1.to(DEV), o2.to(DEV), t.to(DEV) if teacher else None, y.to(DEV), n_l,
                              weights_dev=_dev([cps_w, mt_w]), want_pseudo=True)
        _same(rd, r, ("scalars", "dstudent", "dother", "pseudo1", "pseudo2"))
    wst.report()


# ------------------------------------------------------------------------------------------------------------ Dice
@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("softmax", [0, 1])
@pytest.mark.parametrize("C", CLASSES)
def test_dice_loss_matches_fp64(C, softmax, weighted):
    wst = _Worst("hpfg_dice_loss softmax=%d %s C=%d" % (softmax, "weighted" if weighted else "unweighted", C))
    wts = _weights(C) if weighted else None
    for i, (n_l, n_u, h, w) in enumerate(CASES):
        n = n_l + n_u
        g = _gen(7, C, 4 * i + 2 * softmax + weighted)
        z, y = _logits(g, n, C, h, w), _labels(g, n, C, h, w)
        x = z if softmax else torch.softmax(z, 1)          # probabilities unless the kernel takes the softmax itself
        sc, dx = dice_loss_raw(x.to(DEV), y.to(DEV), softmax=bool(softmax), weight=wts)
        x64 = x.double().requires_grad_(True)
        loss = oracle.dice_loss(x64, y.unsqueeze(1), C, weight=wts, softmax=bool(softmax))
        loss.backward()
        with torch.no_grad():
            p = torch.softmax(x64, 1) if softmax else x64
            ratio = []
            for c in range(C):
                t = (y == c).double()
                ratio.append((2 * (p[:, c] * t).sum() + 1e-5) / ((p[:, c] ** 2).sum() + t.sum() + 1e-5))
        wst.scalars(sc, [loss] + ratio)
        wst.tensor(dx, x64.grad)
    wst.report()


@pytest.mark.parametrize("C", [3, 8])
def test_dice_loss_float_target_follows_the_reference_one_hot(C):
    """main.py hands DiceLoss a float map.  The reference's one-hot is ``target == c``: 1.5 and -0.5 are in no class,
    2.0 is class 2, 255.0 is in no class."""
    g = _gen(8, C, 0)
    p = torch.softmax(_logits(g, 2, C, 6, 10), 1)
    y = _labels(g, 2, C, 6, 10).float()
    y[0, 1, :4] = torch.tensor([1.5, -0.5, 2.0, 255.0])
    y[1, 3, 6:] = torch.tensor([-0.5, 1.5, 2.0, 255.0])
    p64 = p.double().requires_grad_(True)
    want = _dice64(p64, y, C)
    want.backward()
    pd = p.to(DEV).requires_grad_(True)
    loss = hb.DiceLoss(C)(pd, y.to(DEV).unsqueeze(1))
    loss.backward()
    assert abs(loss.item() - want.item()) <= 1e-5 * abs(want.item()), (loss.item(), want.item())
    assert rel_l2(pd.grad, p64.grad) < 1e-5


@pytest.mark.parametrize("C", [1, 9])
def test_class_counts_without_a_kernel_raise(C):
    """hpfg_ssl_loss and hpfg_dice_loss are built for 2..8 classes, hpfg_softmax_mse for 1..8."""
    s = torch.randn(2, C, 4, 4, device=DEV)
    y = torch.zeros(1, 4, 4, dtype=torch.int64, device=DEV)
    for mode, other in ((L.LOSS_SUP, None), (L.LOSS_MT, s[1:])):
        with pytest.raises(L.HpfgError):
            hb.ssl_loss_raw(mode, s, other, y, 1, cons_weight=0.1)
    with pytest.raises(L.HpfgError):
        dice_loss_raw(s, torch.zeros(2, 4, 4, dtype=torch.int64, device=DEV))
    if C == 9:
        with pytest.raises(L.HpfgError):
            hb.softmax_mse_loss(s, s.clone())


# ------------------------------------------------------------------------------------------------------------ softmax_mse_loss
def _mse64(a, b, sigmoid):
    if sigmoid:
        return (torch.sigmoid(a) - torch.sigmoid(b)) ** 2
    return oracle.softmax_mse(a, b)


@pytest.mark.parametrize("sigmoid", [False, True], ids=["softmax", "sigmoid"])
@pytest.mark.parametrize("C", list(range(1, 9)))
def test_softmax_mse_loss_matches_fp64(C, sigmoid):
    wst = _Worst("hpfg_softmax_mse %s C=%d" % ("sigmoid" if sigmoid else "softmax", C))
    for i, (n, h, w) in enumerate(((1, 2, 2), (3, 6, 10), (2, 28, 28))):
        g = _gen(9, C, 2 * i + sigmoid)
        a, b = _logits(g, n, C, h, w), _logits(g, n, C, h, w)
        gmap = torch.randn(n, C, h, w, generator=g)
        a64 = a.double().requires_grad_(True)
        ref = _mse64(a64, b.double(), sigmoid)
        ad, bd = a.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
        for up in ("map", "mean", "sum"):
            ad.grad = None
            out = hb.softmax_mse_loss(ad, bd, sigmoid=sigmoid)
            if up == "map":
                wst.tensor(out, ref, kind="value")
                out.backward(gmap.to(DEV))
                (want,) = torch.autograd.grad(ref, a64, gmap.double(), retain_graph=True)
            else:       # the upstream gradient of .mean() / .sum() is a stride-0 expansion of one value
                getattr(out, up)().backward()
                (want,) = torch.autograd.grad(getattr(ref, up)(), a64, retain_graph=True)
            wst.tensor(ad.grad, want)
            assert bd.grad is None                           # the target carries no gradient
    wst.report()


if __name__ == "__main__":
    _mt_two_launch_child(sys.argv[1])
