"""Loss classes with the reference's signatures (utils/loss/medloss.py:44-56 ``Med_Sup_Loss``,
utils/loss/diceloss.py:155-191 ``DiceLoss``, :64-81 ``softmax_mse_loss``) plus the fused whole-step SSL losses
of the Mean-Teacher / CPS / UAMT trainers, all running on the fused CUDA loss kernels (csrc/loss.cu).

Each fused call produces the loss value AND d loss / d logits in the same launch(es) (Mean-Teacher: one; other modes: two); the autograd
Function just hands the stored gradient back scaled by grad_output."""
import ctypes

import torch
import torch.nn as nn

from . import _lib as L


def _weights_arg(weight, n):
    if weight is None:
        return None
    assert len(weight) == n
    return (ctypes.c_float * n)(*[float(w) for w in weight])


def _workspace(mode, n_l, n_u, c, h, w, device):
    nbytes = L.lib().hpfg_ssl_loss_workspace_bytes(mode, n_l, n_u, c, h, w)
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def ssl_loss_raw(mode, student, other, labels, n_l, *, cons_weight=0.0, mc_logits=None, mc_passes=0,
                 uamt_threshold=0.0, class_weights=None, ce_coef=0.5, dice_coef=0.5, want_pseudo=False,
                 out=None, cons_weight_dev=None, uamt_threshold_dev=None):
    """Thin wrapper of hpfg_ssl_loss.  Returns dict(scalars[8], dstudent, dother, pseudo1, pseudo2)."""
    L.require_cuda(student, "logits")
    student = student.contiguous().float()
    n, c, h, w = student.shape
    n_u = n - n_l
    dev = student.device
    if labels is not None:
        labels = labels.contiguous().to(torch.int64)
        assert labels.shape == (n_l, h, w), "labels must be [n_l,H,W]"
    if other is not None:
        other = other.contiguous().float()
    dstudent = torch.empty_like(student)
    dother = torch.empty_like(other) if mode == L.LOSS_CPS else None
    scalars = torch.empty(8, device=dev, dtype=torch.float32)
    ws = _workspace(mode, n_l, n_u, c, h, w, dev)
    p1 = p2 = None
    if want_pseudo and mode == L.LOSS_CPS:
        p1 = torch.empty((n_u, h, w), device=dev, dtype=torch.int64)
        p2 = torch.empty((n_u, h, w), device=dev, dtype=torch.int64)
    if cons_weight_dev is not None:      # CUDA-graph replays: the consistency weight (and UAMT threshold, if given) on the device
        L.check(L.lib().hpfg_ssl_loss_dv(mode, L.ptr(student), L.ptr(other), L.ptr(mc_logits), mc_passes, L.ptr(labels),
                                         n_l, n_u, c, h, w, L.ptr(cons_weight_dev), float(uamt_threshold),
                                         L.ptr(uamt_threshold_dev), _weights_arg(class_weights, c), float(ce_coef),
                                         float(dice_coef), L.ptr(dstudent), L.ptr(dother), L.ptr(scalars), L.ptr(p1),
                                         L.ptr(p2), L.ptr(ws), L.stream_ptr(dev)), "hpfg_ssl_loss_dv")
        return dict(scalars=scalars, dstudent=dstudent, dother=dother, pseudo1=p1, pseudo2=p2)
    L.check(L.lib().hpfg_ssl_loss(mode, L.ptr(student), L.ptr(other), L.ptr(mc_logits), mc_passes, L.ptr(labels), n_l,
                                  n_u, c, h, w, float(cons_weight), float(uamt_threshold),
                                  _weights_arg(class_weights, c), float(ce_coef), float(dice_coef), L.ptr(dstudent),
                                  L.ptr(dother), L.ptr(scalars), L.ptr(p1), L.ptr(p2), L.ptr(ws), L.stream_ptr(dev)),
            "hpfg_ssl_loss")
    return dict(scalars=scalars, dstudent=dstudent, dother=dother, pseudo1=p1, pseudo2=p2)


class _SslLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, student, other, mode, labels, n_l, kw):
        r = ssl_loss_raw(mode, student, other.detach() if other is not None else None, labels, n_l, **kw)
        ctx.save_for_backward(r["dstudent"], r["dother"] if r["dother"] is not None else r["dstudent"].new_empty(0))
        ctx.has_other = r["dother"] is not None
        ctx.extras = r
        return r["scalars"][0].clone()

    @staticmethod
    def backward(ctx, g):
        ds, do = ctx.saved_tensors
        return ds * g, (do * g if ctx.has_other else None), None, None, None, None


class Med_Sup_Loss(nn.Module):
    """0.5*CE(ignore_index=255) + 0.5*Dice(softmax(logits), onehot(y))  (utils/loss/medloss.py:44-56)."""

    def __init__(self, num_classes, ce=0.5, dice=0.5):
        super().__init__()
        self.num_classes, self.ce, self.dice = num_classes, ce, dice

    def forward(self, outputs, target_label):
        assert outputs.shape[1] == self.num_classes
        return _SslLossFn.apply(outputs, None, L.LOSS_SUP, target_label, outputs.shape[0],
                                dict(ce_coef=self.ce, dice_coef=self.dice))


def dice_loss_raw(inputs, target, softmax=False, weight=None, want_grad=True):
    """Thin wrapper of hpfg_dice_loss: (scalars[1+C] = {loss, per-class dice}, d loss / d inputs or None).  inputs [n,C,H,W]
    probabilities (or logits with softmax=True), target any [n,(1,)H,W] tensor of class ids."""
    L.require_cuda(inputs, "DiceLoss inputs")
    x = inputs.contiguous().float()
    n, c, h, w = x.shape
    t = target.reshape(n, h, w).contiguous().to(torch.int64)
    dx = torch.empty_like(x) if want_grad else None
    scalars = torch.empty(1 + c, device=x.device, dtype=torch.float32)
    ws = torch.empty(2048, dtype=torch.uint8, device=x.device)
    L.check(L.lib().hpfg_dice_loss(L.ptr(x), L.ptr(t), n, c, h, w, int(bool(softmax)), _weights_arg(weight, c),
                                   L.ptr(dx), L.ptr(scalars), L.ptr(ws), L.stream_ptr(x.device)), "hpfg_dice_loss")
    return scalars, dx


class _DiceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inputs, target, n_classes, weight, softmax):
        scalars, dx = dice_loss_raw(inputs, target, softmax, weight, want_grad=inputs.requires_grad)
        if dx is not None:
            ctx.save_for_backward(dx)
        ctx.class_wise = scalars[1:]
        return scalars[0].clone()

    @staticmethod
    def backward(ctx, g):
        (dx,) = ctx.saved_tensors
        return dx * g, None, None, None, None


class DiceLoss(nn.Module):
    """``DiceLoss(n_classes)(inputs, target, weight=None, softmax=False)`` (utils/loss/diceloss.py:155-191).
    inputs [n,C,H,W] probabilities (or logits with softmax=True); target [n,1,H,W] class ids."""

    def __init__(self, n_classes):
        super().__init__()
        self.n_classes = n_classes

    def forward(self, inputs, target, weight=None, softmax=False):
        onehot_size = (target.shape[0], self.n_classes * target.shape[1]) + tuple(target.shape[2:])
        assert tuple(inputs.size()) == onehot_size, 'predict & target shape do not match'
        return _DiceFn.apply(inputs, target, self.n_classes, weight, softmax)


class _SoftmaxMseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, sigmoid):
        L.require_cuda(a, "softmax_mse_loss input")
        a32, b32 = a.contiguous().float(), b.detach().contiguous().float()
        n, c, h, w = a32.shape
        out = torch.empty_like(a32)
        L.check(L.lib().hpfg_softmax_mse(L.ptr(a32), L.ptr(b32), None, n, c, h, w, int(bool(sigmoid)), L.ptr(out),
                                         L.stream_ptr(a32.device)), "hpfg_softmax_mse")
        ctx.save_for_backward(a32, b32)
        ctx.sigmoid = bool(sigmoid)
        return out

    @staticmethod
    def backward(ctx, g):
        a32, b32 = ctx.saved_tensors
        n, c, h, w = a32.shape
        da = torch.empty_like(a32)
        L.check(L.lib().hpfg_softmax_mse(L.ptr(a32), L.ptr(b32), L.ptr(g.contiguous().float()), n, c, h, w, int(ctx.sigmoid),
                                         L.ptr(da), L.stream_ptr(a32.device)), "hpfg_softmax_mse")
        return da, None, None


def softmax_mse_loss(input_logits, target_logits, sigmoid=False):
    """Unreduced (softmax(a)-softmax(b))**2 over dim 1, or of the sigmoids (utils/loss/diceloss.py:64-81), on the
    `hpfg_softmax_mse` kernel (forward map and the gradient wrt ``input_logits``; the target is the no_grad teacher output
    in every trainer that calls this, 2019_07...:134-148, and carries no gradient here).  [N,C,H,W] CUDA logits, C <= 8."""
    assert input_logits.size() == target_logits.size()
    if input_logits.dim() != 4:
        raise L.HpfgError("softmax_mse_loss: expected [N,C,H,W] logits, got %s" % (tuple(input_logits.shape),))
    return _SoftmaxMseFn.apply(input_logits, target_logits, sigmoid)


# ---- fused whole-step losses (what the MT / CPS / UAMT trainers compute inline) ---------------------------
def mean_teacher_loss(student_logits, teacher_logits_u, labels, consistency_weight, ce=0.5, dice=0.5):
    """loss_sup + w*mean((softmax(s_u)-softmax(t_u))^2)  (2017_03_NIPS_Mean-Teacher_ACDC.py:97-106).
    student_logits [n_l+n_u,...]; teacher_logits_u [n_u,...] (the unlabeled slices only)."""
    n_l = labels.shape[0]
    return _SslLossFn.apply(student_logits, teacher_logits_u, L.LOSS_MT, labels, n_l,
                            dict(cons_weight=consistency_weight, ce_coef=ce, dice_coef=dice))


def cps_loss(logits1, logits2, labels, consistency_weight, ce=0.5, dice=0.5):
    """Cross pseudo supervision (2021_06_CVPR_CPS_ACDC.py:99-111); gradients flow to both networks."""
    n_l = labels.shape[0]
    return _SslLossFn.apply(logits1, logits2, L.LOSS_CPS, labels, n_l,
                            dict(cons_weight=consistency_weight, ce_coef=ce, dice_coef=dice))


def uamt_loss(student_logits, teacher_logits_u, mc_logits, labels, consistency_weight, threshold, T=8, ce=0.5,
              dice=0.5):
    """Uncertainty-aware MT (2019_07_MICCAI_Uncertainty_Aware_ACDC.py:145-162)."""
    n_l = labels.shape[0]
    return _SslLossFn.apply(student_logits, teacher_logits_u, L.LOSS_UAMT, labels, n_l,
                            dict(cons_weight=consistency_weight, mc_logits=mc_logits.contiguous().float(), mc_passes=T,
                                 uamt_threshold=threshold, ce_coef=ce, dice_coef=dice))


# ---- SURVEY 8f.4: ICT-MedSeg and S4CVNet step losses (same two kernels, extra modes) ----------------------
def ict_mix_inputs(ux0, ux1, mix_factors):
    """batch_ux_mixed = ux0*(1-l) + ux1*l  (2022_02_ISBI_ICT-MedSeg_ACDC.py:115-117); mix_factors: [n] or [n,1,1,1]."""
    L.require_cuda(ux0, "ICT inputs")
    a, b = ux0.contiguous().float(), ux1.contiguous().float()
    assert a.shape == b.shape
    lam = mix_factors.reshape(-1).to(device=a.device, dtype=torch.float32).contiguous()
    assert lam.numel() == a.shape[0]
    out = torch.empty_like(a)
    L.check(L.lib().hpfg_ict_mix(L.ptr(a), L.ptr(b), L.ptr(lam), a.shape[0], a[0].numel(), L.ptr(out),
                                 L.stream_ptr(a.device)), "hpfg_ict_mix")
    return out


def ict_loss_raw(student, teacher_u, mix_factors, labels, n_l, *, cons_weight=0.0, cons_weight_dev=None,
                 class_weights=None, ce_coef=0.5, dice_coef=0.5):
    """Thin wrapper of hpfg_ict_loss.  student [n_l+n_m,...], teacher_u [2*n_m,...] (ux0 half then ux1 half)."""
    L.require_cuda(student, "logits")
    student = student.contiguous().float()
    n, c, h, w = student.shape
    n_m = n - n_l
    dev = student.device
    teacher_u = teacher_u.contiguous().float()
    assert teacher_u.shape == (2 * n_m, c, h, w), "teacher logits must cover both un-mixed halves"
    lam = mix_factors.reshape(-1).to(device=dev, dtype=torch.float32).contiguous()
    assert lam.numel() == n_m
    labels = labels.contiguous().to(torch.int64)
    assert labels.shape == (n_l, h, w), "labels must be [n_l,H,W]"
    dstudent = torch.empty_like(student)
    scalars = torch.empty(8, device=dev, dtype=torch.float32)
    ws = _workspace(L.LOSS_ICT, n_l, n_m, c, h, w, dev)
    L.check(L.lib().hpfg_ict_loss(L.ptr(student), L.ptr(teacher_u), L.ptr(lam), L.ptr(labels), n_l, n_m, c, h, w,
                                  float(cons_weight), L.ptr(cons_weight_dev), _weights_arg(class_weights, c),
                                  float(ce_coef), float(dice_coef), L.ptr(dstudent), L.ptr(scalars), L.ptr(ws),
                                  L.stream_ptr(dev)), "hpfg_ict_loss")
    return dict(scalars=scalars, dstudent=dstudent, dother=None)


def s4cv_loss_raw(logits1, logits2, teacher_u, labels, n_l, *, cps_weight=0.0, mt_weight=0.0, weights_dev=None,
                  class_weights=None, ce_coef=0.5, dice_coef=0.5, want_pseudo=False):
    """Thin wrapper of hpfg_s4cv_loss.  teacher_u None = the reference's `cur_itrs < 1000` branch (no MSE terms)."""
    L.require_cuda(logits1, "logits")
    o1, o2 = logits1.contiguous().float(), logits2.contiguous().float()
    assert o1.shape == o2.shape
    n, c, h, w = o1.shape
    n_u = n - n_l
    dev = o1.device
    if teacher_u is not None:
        teacher_u = teacher_u.contiguous().float()
        assert teacher_u.shape == (n_u, c, h, w)
    labels = labels.contiguous().to(torch.int64)
    assert labels.shape == (n_l, h, w), "labels must be [n_l,H,W]"
    d1, d2 = torch.empty_like(o1), torch.empty_like(o2)
    scalars = torch.empty(8, device=dev, dtype=torch.float32)
    ws = _workspace(L.LOSS_S4CV, n_l, n_u, c, h, w, dev)
    p1 = p2 = None
    if want_pseudo:
        p1 = torch.empty((n_u, h, w), device=dev, dtype=torch.int64)
        p2 = torch.empty((n_u, h, w), device=dev, dtype=torch.int64)
    L.check(L.lib().hpfg_s4cv_loss(L.ptr(o1), L.ptr(o2), L.ptr(teacher_u), L.ptr(labels), n_l, n_u, c, h, w,
                                   float(cps_weight), float(mt_weight), L.ptr(weights_dev),
                                   _weights_arg(class_weights, c), float(ce_coef), float(dice_coef), L.ptr(d1), L.ptr(d2),
                                   L.ptr(scalars), L.ptr(p1), L.ptr(p2), L.ptr(ws), L.stream_ptr(dev)), "hpfg_s4cv_loss")
    return dict(scalars=scalars, dstudent=d1, dother=d2, pseudo1=p1, pseudo2=p2)


class _RawLossFn(torch.autograd.Function):
    """autograd shim over a *_raw call that already produced d loss / d logits for up to two logit tensors."""

    @staticmethod
    def forward(ctx, a, b, fn):
        r = fn(a.detach(), b.detach() if b is not None else None)
        ctx.save_for_backward(r["dstudent"], r["dother"] if r["dother"] is not None else r["dstudent"].new_empty(0))
        ctx.has_other = r["dother"] is not None
        ctx.extras = r
        return r["scalars"][0].clone()

    @staticmethod
    def backward(ctx, g):
        ds, do = ctx.saved_tensors
        return ds * g, (do * g if ctx.has_other else None), None


def ict_loss(student_logits, teacher_logits_u, mix_factors, labels, consistency_weight, ce=0.5, dice=0.5):
    """supervised_loss + w*mean((softmax(s_mixed) - mix(softmax(t(ux0)), softmax(t(ux1))))^2)
    (2022_02_ISBI_ICT-MedSeg_ACDC.py:121-137).  teacher_logits_u = cat([ema(ux0), ema(ux1)])."""
    n_l = labels.shape[0]
    t = teacher_logits_u.detach()
    return _RawLossFn.apply(student_logits, None, lambda s, _: ict_loss_raw(
        s, t, mix_factors, labels, n_l, cons_weight=consistency_weight, ce_coef=ce, dice_coef=dice))


def s4cvnet_loss(logits1, logits2, teacher_logits_u, labels, cps_weight, mt_weight, ce=0.5, dice=0.5):
    """loss_sup + loss_semi of 2022_08_CVPR_S4CVNet_ACDC.py:124-156 for any two segmentation networks' logits
    (gradients flow to both).  cps_weight = 7*consistency_weight_cps; teacher_logits_u None or mt_weight applied to
    consistency_loss1 + consistency_loss2 (pass None while cur_itrs < 1000, :143-145)."""
    n_l = labels.shape[0]
    t = teacher_logits_u.detach() if teacher_logits_u is not None else None
    return _RawLossFn.apply(logits1, logits2, lambda a, b: s4cv_loss_raw(
        a, b, t, labels, n_l, cps_weight=cps_weight, mt_weight=mt_weight, ce_coef=ce, dice_coef=dice))


def argmax_labels(logits, dtype=torch.int64):
    """torch.argmax(torch.softmax(logits, dim=1), dim=1) in one launch (val.py:275); int64 (default) or uint8 labels."""
    L.require_cuda(logits, "logits")
    z = logits.contiguous().float()
    n, c, h, w = z.shape
    assert dtype in (torch.int64, torch.uint8)
    out = torch.empty((n, h, w), device=z.device, dtype=dtype)
    L.check(L.lib().hpfg_argmax_labels(L.ptr(z), n, c, h, w, L.ptr(out) if dtype == torch.int64 else None,
                                       L.ptr(out) if dtype == torch.uint8 else None, L.stream_ptr(z.device)),
            "hpfg_argmax_labels")
    return out


class _ContrastFn(torch.autograd.Function):
    """Dense_Loss.contrastive_loss on ``hpfg_dense_contrastive`` (csrc/neck.cu): value, and the gradient wrt out_1 computed by
    the same call when out_1 needs it."""

    @staticmethod
    def forward(ctx, out_1, out_2, temperature):
        L.require_cuda(out_1, "Dense_Loss input")
        L.require_cuda(out_2, "Dense_Loss input")
        a, b = out_1.contiguous().float(), out_2.detach().contiguous().float()
        batch, dim = a.shape[0], a.shape[1]
        positions = a[0, 0].numel()
        lib = L.lib()
        work = torch.empty(lib.hpfg_dense_contrastive_workspace_floats(batch, dim, positions), device=a.device, dtype=torch.float32)
        loss = torch.empty((), device=a.device, dtype=torch.float32)
        d_a = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        L.check(lib.hpfg_dense_contrastive(L.ptr(a), L.ptr(b), batch, dim, positions, float(temperature), L.ptr(loss), L.ptr(d_a),
                                           L.ptr(work), L.stream_ptr(a.device)), "hpfg_dense_contrastive")
        ctx.save_for_backward(d_a)
        return loss

    @staticmethod
    def backward(ctx, g):
        (d_a,) = ctx.saved_tensors
        return (d_a * g if d_a is not None else None), None, None


class Dense_Loss(nn.Module):
    """``Dense_Loss(batch_size, device, temperature)(x, y)`` (utils/loss/dense_loss.py:5-40): SimCLR-style contrastive loss
    on the (global vector, dense map) pairs the projection necks return; ``y`` is the detached teacher side.  Each
    ``contrastive_loss`` is one ``hpfg_dense_contrastive`` call (normalise, [2B,2B] similarities, masked row sums, loss and
    the gradient wrt the first argument); CUDA tensors only."""

    def __init__(self, batch_size=32, device=None, temperature=0.7):
        super().__init__()
        self.device, self.batch_size, self.temperature = device, batch_size, temperature

    def contrastive_loss(self, out_1, out_2):
        """-log(exp(s_i,pos / t) / sum_{j != i} exp(s_ij / t)) averaged over the 2B rows, s = <z_i, z_j> of the
        channel-normalised, flattened features (utils/loss/dense_loss.py:18-34); out_1, out_2: [B,D] or [B,D,S]."""
        if out_1.shape != out_2.shape or out_1.dim() < 2:
            raise RuntimeError("Dense_Loss: expected two [B,D(,S)] tensors of one shape, got %s and %s"
                               % (tuple(out_1.shape), tuple(out_2.shape)))
        if out_1.shape[0] != self.batch_size:        # the reference builds its mask from the constructor's batch size
            raise RuntimeError("Dense_Loss was built for batch %d, got %d" % (self.batch_size, out_1.shape[0]))
        return _ContrastFn.apply(out_1, out_2, self.temperature)

    def forward(self, x, y):
        x1, x2 = x
        y1, y2 = y
        return 0.5 * (self.contrastive_loss(x1, y1.detach()) + self.contrastive_loss(x2, y2.detach()))
