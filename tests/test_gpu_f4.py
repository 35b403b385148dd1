"""GPU parity tests (B200) for the SURVEY 8f.3 / 8f.4 rows: the ICT-MedSeg and S4CVNet step losses, the ICT step driver
and the batched inference path, against golden vectors produced by the REAL reference (tests/golden/make_golden.py f4)
and against the CPU oracle on seeded inputs.  Tolerances as in test_gpu_parity.py."""
import pytest
import torch

import oracle
import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from tests.golden.common import make_state, make_masks, make_batch, make_predict_case
from tests.helpers import load_golden, check_summary, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _model(st, in_ch, n_cls, precision):
    m = hb.UNet(in_ch, n_cls, precision=precision)
    m.load_state_dict(st)
    return m.to(DEV)


@pytest.mark.parametrize("tag", ["c4", "c2"])
def test_ict_and_s4cv_losses_vs_reference_golden(tag):
    g = load_golden("f4_losses.pt")[tag]
    n_l, n_m, C, H, W = g["shape"]
    ict = g["ict"]
    s = ict["student"].to(DEV).requires_grad_(True)
    l = hb.ict_loss(s, ict["teacher"].to(DEV), ict["mix"].to(DEV), ict["y"].to(DEV), ict["w"])
    (gr,) = torch.autograd.grad(l, s)
    assert abs(l.item() - ict["loss"]) / abs(ict["loss"]) < 1e-5
    assert rel_l2(gr, ict["grad"]) < 1e-5
    r = hb.ict_loss_raw(s.detach(), ict["teacher"].to(DEV), ict["mix"].to(DEV), ict["y"].to(DEV), n_l, cons_weight=ict["w"])
    assert abs(r["scalars"][1].item() - ict["sup"]) / ict["sup"] < 1e-5
    assert abs(r["scalars"][2].item() - ict["cons"]) / ict["cons"] < 1e-5
    wdev = torch.tensor([ict["w"]], device=DEV, dtype=torch.float32)          # device-value variant (graph replay)
    r2 = hb.ict_loss_raw(s.detach(), ict["teacher"].to(DEV), ict["mix"].to(DEV), ict["y"].to(DEV), n_l, cons_weight_dev=wdev)
    assert torch.equal(r2["dstudent"], r["dstudent"]) and torch.equal(r2["scalars"], r["scalars"])
    s4 = g["s4cv"]
    y = s4["y"].to(DEV)
    for branch in ("early", "late"):
        b = s4[branch]
        o1, o2 = s4["logits1"].to(DEV).requires_grad_(True), s4["logits2"].to(DEV).requires_grad_(True)
        t = s4["teacher"].to(DEV) if b["cur_itrs"] >= 1000 else None
        l = hb.s4cvnet_loss(o1, o2, t, y, b["cps_weight"], b["mt_weight"])
        g1, g2 = torch.autograd.grad(l, [o1, o2])
        assert abs(l.item() - b["loss"]) / abs(b["loss"]) < 1e-5
        assert rel_l2(g1, b["grad1"]) < 1e-5 and rel_l2(g2, b["grad2"]) < 1e-5
        r = hb.s4cv_loss_raw(o1.detach(), o2.detach(), t, y, n_l, cps_weight=b["cps_weight"], mt_weight=b["mt_weight"],
                             want_pseudo=True)
        assert torch.equal(r["pseudo1"].cpu(), b["pl1"]) and torch.equal(r["pseudo2"].cpu(), b["pl2"])
        assert abs(r["scalars"][1].item() - b["sup"]) / b["sup"] < 1e-5
        assert abs(r["scalars"][2].item() - b["semi"]) / b["semi"] < 1e-5
        wdev = torch.tensor([b["cps_weight"], b["mt_weight"]], device=DEV, dtype=torch.float32)
        r2 = hb.s4cv_loss_raw(o1.detach(), o2.detach(), t, y, n_l, weights_dev=wdev)
        assert torch.equal(r2["dstudent"], r["dstudent"]) and torch.equal(r2["dother"], r["dother"])


def test_ict_mix_and_argmax_kernels_exact():
    g = torch.Generator().manual_seed(11)
    a, b = torch.rand(5, 1, 224, 224, generator=g), torch.rand(5, 1, 224, 224, generator=g)
    lam = torch.rand(5, 1, 1, 1, generator=g)
    got = hb.ict_mix_inputs(a.to(DEV), b.to(DEV), lam.to(DEV))
    assert torch.equal(got.cpu(), a * (1.0 - lam) + b * lam)                  # 2022_02...:117, bit-exact
    for C in range(2, 9):                                                      # every class count the kernel is built for
        z = 3 * torch.randn(3, C, 32, 40, generator=g)
        z[0, :, :4] = 0.25                                                      # exact ties -> first maximum
        z[1, 1:, 5] = z[1, :1, 5]
        ref = torch.argmax(torch.softmax(z, dim=1), dim=1)
        assert torch.equal(hb.argmax_labels(z.to(DEV)).cpu(), ref)
        assert torch.equal(hb.argmax_labels(z.to(DEV), dtype=torch.uint8).cpu().long(), ref)
    with pytest.raises(L.HpfgError):
        hb.argmax_labels(torch.zeros(1, 9, 8, 8, device=DEV))                  # more classes than the kernels carry


def test_ict_loss_full_size_properties():
    """At the YAML shape (8 labeled + 24 unlabeled -> 8 + 12 mixed, 4x224x224): against the oracle on the same seeded
    logits, plus the size-independent properties that every pixel's gradient sums to zero over classes and that
    lambda = 0 / 1 reduce the ICT term to the Mean-Teacher term against one teacher half."""
    g = torch.Generator().manual_seed(6)
    n_l, n_m = 8, 12
    s = 2 * torch.randn(n_l + n_m, 4, 224, 224, generator=g)
    t = 2 * torch.randn(2 * n_m, 4, 224, 224, generator=g)
    y = torch.randint(0, 4, (n_l, 224, 224), generator=g)
    lam = torch.rand(n_m, generator=g)
    sr = s.clone().requires_grad_(True)
    sup, cons = oracle.ict_losses(sr, t, lam, y, n_l, 4)
    lo = sup + 0.05 * cons
    (go,) = torch.autograd.grad(lo, sr)
    sd, td, yd = s.to(DEV), t.to(DEV), y.to(DEV)
    r = hb.ict_loss_raw(sd, td, lam.to(DEV), yd, n_l, cons_weight=0.05)
    assert abs(r["scalars"][0].item() - lo.item()) / lo.item() < 1e-5
    assert rel_l2(r["dstudent"], go) < 1e-5
    assert r["dstudent"].sum(dim=1).abs().max().item() < 1e-9
    for v, half in ((0.0, td[:n_m]), (1.0, td[n_m:])):
        ri = hb.ict_loss_raw(sd, td, torch.full((n_m,), v, device=DEV), yd, n_l, cons_weight=0.05)
        rm = hb.ssl_loss_raw(L.LOSS_MT, sd, half, yd, n_l, cons_weight=0.05)
        assert rel_l2(ri["dstudent"], rm["dstudent"]) < 1e-6
        assert abs(ri["scalars"][0].item() - rm["scalars"][0].item()) < 1e-6


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_ict_steps_vs_reference_golden(precision):
    g = load_golden("ict_steps_acdc.pt")
    c = g["cfg"]
    f32 = precision == "fp32"
    student = _model(make_state(c["in_ch"], c["n_cls"], c["seed"]), c["in_ch"], c["n_cls"], precision)
    teacher = _model(make_state(c["in_ch"], c["n_cls"], c["seed"] + 7), c["in_ch"], c["n_cls"], precision)
    step = hb.ICTStep(student, teacher)
    n_m = c["n_u"] // 2
    for i, rec in enumerate(g["steps"]):
        it = i + 1
        x_l, x_u, y = make_batch(c["n_l"], c["n_u"], c["in_ch"], c["n_cls"], c["h"], c["w"], c["seed"] + 100 * it)
        student.set_dropout_masks(make_masks(c["n_l"] + n_m, c["h"], c["w"], c["seed"] + 100 * it + 1))
        teacher.set_dropout_masks(make_masks(n_m, c["h"], c["w"], c["seed"] + 100 * it + 2))
        lam = torch.rand(n_m, 1, 1, 1, generator=torch.Generator().manual_seed(c["seed"] + 100 * it + 3))
        loss = step.step(torch.cat([x_l, x_u]).to(DEV), y.to(DEV), lam)
        assert abs(loss.item() - rec["loss"]) / rec["loss"] < (1e-5 if f32 else 1e-3)
        assert step.last["lr"] == pytest.approx(rec["lr"], rel=1e-12) and step.last["w"] == pytest.approx(rec["w"], rel=1e-12)
        sc = step.last["scalars"]
        assert abs(sc[2].item() - rec["cons"]) / rec["cons"] < (1e-4 if f32 else 1e-1)
        check_summary(step.last["logits"], rec["logits"], rtol=1e-5 if f32 else 3e-2, what="logits")
        check_summary(step.last["teacher_logits"], rec["teacher_logits"], rtol=1e-5 if f32 else 3e-2, what="teacher logits")
        if f32:
            sd, td = student.state_dict(), teacher.state_dict()
            assert torch.allclose(sd["decoder.out_conv.weight"].cpu(), rec["student_out_conv"], atol=2e-6)
            assert torch.allclose(td["decoder.out_conv.weight"].cpu(), rec["teacher_out_conv"], atol=2e-6)
            assert torch.allclose(td["encoder.in_conv.conv_conv.1.running_mean"].cpu(), rec["teacher_rm"], atol=1e-6)
            assert abs(float(student.flat_params.double().sum()) - rec["student_sum"]) < 1e-3
            assert abs(float(teacher.flat_params.double().sum()) - rec["teacher_sum"]) < 1e-3
    assert int(teacher.bn_counters[0]) == 2 * len(g["steps"])                 # two teacher forwards per step (:123-124)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_predict_volume_vs_reference_golden(precision):
    """val.py:268-281: slice-by-slice eval-mode argmax labels of the real reference vs one batched predict_volume call."""
    g = load_golden("predict_acdc.pt")
    c = g["cfg"]
    st, vol = make_predict_case(c["in_ch"], c["n_cls"], c["n"], c["h"], c["w"], c["seed"])
    st.update(g["buffers"])
    m = _model(st, c["in_ch"], c["n_cls"], precision)
    m.train()
    labels = hb.predict_volume(m, vol.to(DEV))
    assert not m.training and labels.dtype == torch.int64 and tuple(labels.shape) == (c["n"], c["h"], c["w"])
    ref, margin = g["labels"].long(), g["margin"].float()
    agree = (labels.cpu() == ref).float().mean().item()
    if precision == "fp32":
        assert torch.equal(labels.cpu()[margin > 1e-3], ref[margin > 1e-3]) and agree > 0.999
    else:
        assert agree > 0.95, agree                   # bf16 activations under a x40 output conv: near-ties may flip
        sure = margin > 0.1                      # top-2 softmax gap of the reference; ~10 % of this fixture's pixels
        assert sure.sum().item() > 500
        sure_agree = (labels.cpu()[sure] == ref[sure]).float().mean().item()
        print("bf16 predict_volume agreement: all pixels %.4f, margin>0.1 %.4f" % (agree, sure_agree))
        assert sure_agree > 0.98, sure_agree
    chunked = hb.predict_volume(m, vol.to(DEV), max_batch=2, dtype=torch.uint8)   # chunking does not change eval labels
    assert (chunked.long() == labels).float().mean().item() > 0.9999


def _oracle_plus_grads(c, dtype):
    """All 98 gradients of the fixture's loss from the CPU oracle in the given precision."""
    from tests.golden.common import make_plus_state
    cast = lambda d: {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in d.items()}
    st, te = cast(make_plus_state(c["in_ch"], c["n_cls"], c["seed"])), cast(make_plus_state(c["in_ch"], c["n_cls"], c["seed"] + 9))
    x, _, y = make_batch(c["n"], 0, c["in_ch"], c["n_cls"], c["h"], c["w"], c["seed"] + 7)
    x = x.to(dtype)
    names = [n for n, _ in oracle.unet_param_spec(c["in_ch"], c["n_cls"])] + [n for n, _ in oracle.unet_plus_neck_spec(c["n_cls"])]
    leaves = {n: st[n].clone().requires_grad_(True) for n in names}
    view = dict(st)
    view.update(leaves)
    out, h1, h2 = oracle.unet_plus_forward(view, x, True, make_masks(c["n"], c["h"], c["w"], c["seed"] + 11))
    with torch.no_grad():
        _, e1, e2 = oracle.unet_plus_forward(te, x, True, make_masks(c["n"], c["h"], c["w"], c["seed"] + 12))
    loss = oracle.med_sup_loss(out, y, c["n_cls"]) + c["weight"] * (oracle.dense_loss(h1, e1) + oracle.dense_loss(h2, e2))
    return dict(zip(names, torch.autograd.grad(loss, [leaves[n] for n in names])))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_unet_plus_and_dense_loss_vs_reference_golden(precision):
    """SURVEY 8f.2 (model/unet.py:178-206, utils/loss/dense_loss.py, main.py:151-170): the UNet_Plus drop-in through plain
    autograd -- logits, both projection necks, loss, and every one of the 98 parameter gradients (the bottleneck gradient
    of the high neck enters the plan through hpfg_unet_backward_ex)."""
    from tests.golden.common import make_plus_state
    g = load_golden("unet_plus_acdc.pt")
    c = g["cfg"]
    f32 = precision == "fp32"
    model2 = hb.build_model(type("A", (), dict(model="unet_plus", in_channels=c["in_ch"], num_classes=c["n_cls"], precision=precision))())
    assert isinstance(model2, hb.UNet_Plus)
    model2.load_state_dict(make_plus_state(c["in_ch"], c["n_cls"], c["seed"]))
    model2 = model2.to(DEV)
    ema_model = hb.UNet_Plus(c["in_ch"], c["n_cls"], precision=precision)
    ema_model.load_state_dict(make_plus_state(c["in_ch"], c["n_cls"], c["seed"] + 9))
    ema_model = ema_model.to(DEV)
    for p in ema_model.parameters():
        p.requires_grad = False
    x, _, y = make_batch(c["n"], 0, c["in_ch"], c["n_cls"], c["h"], c["w"], c["seed"] + 7)
    x, y = x.to(DEV), y.to(DEV)
    model2.set_dropout_masks(make_masks(c["n"], c["h"], c["w"], c["seed"] + 11))
    ema_model.set_dropout_masks(make_masks(c["n"], c["h"], c["w"], c["seed"] + 12))
    torch.backends.cudnn.allow_tf32 = False            # the necks' 1x1 convs are torch/cuDNN ops: keep them fp32 for the 1e-5 bar
    dense_loss = hb.Dense_Loss(batch_size=c["n"], device=torch.device(DEV))
    dice_loss = hb.DiceLoss(c["n_cls"])
    criterion = torch.nn.CrossEntropyLoss(ignore_index=255)
    outputs2, h1, h2 = model2(x)                                           # main.py:155-157, literally
    outputs_soft2 = torch.softmax(outputs2, dim=1)
    with torch.no_grad():
        ema_output, ema_h1, ema_h2 = ema_model(x)
    loss2 = 0.5 * (criterion(outputs2, y) + dice_loss(outputs_soft2, y.unsqueeze(1)))
    loss_constrivate = dense_loss(h1, ema_h1) + dense_loss(h2, ema_h2)
    loss = loss2 + c["weight"] * loss_constrivate
    loss.backward()
    tol = 1e-5 if f32 else 3e-2
    check_summary(outputs2, g["logits"], rtol=tol, what="logits")
    for a, b in zip(list(h1) + list(h2) + list(ema_h1) + list(ema_h2), g["h1"] + g["h2"] + g["ema_h1"] + g["ema_h2"]):
        assert rel_l2(a, b) < (1e-4 if f32 else 5e-2)
    assert abs(loss2.item() - g["sup"]) / g["sup"] < (1e-5 if f32 else 1e-3)
    assert abs(loss_constrivate.item() - g["contrast"]) / g["contrast"] < (1e-4 if f32 else 2e-2)
    grads = dict((k, p.grad) for k, p in model2.named_parameters())
    assert list(grads) == list(g["grads"]) and all(v is not None for v in grads.values())
    if f32:
        # conditioning: the reference's own fp32 gradients sit up to 3e-3 (rel-l2) from the fp64 truth on the up1 block
        # of this fixture, so each tensor is held to 5e-4 plus three times the fp32-vs-fp64 distance of the oracle
        o32, o64 = _oracle_plus_grads(c, torch.float32), _oracle_plus_grads(c, torch.float64)
        for k, gr in grads.items():
            if k.endswith(".bias") and g["grads"][k]["abs_sum"] < 1e-4:      # conv bias ahead of train-mode BN: analytically zero
                assert gr.abs().max().item() < 1e-4, k
                continue
            rt = 5e-4 + 3 * rel_l2(o32[k], o64[k])
            check_summary(gr, g["grads"][k], rtol=rt, atol=1e-6, what=k)
            assert rel_l2(gr, o64[k]) < rt, (k, rel_l2(gr, o64[k]), rt)
    else:      # bf16: whole-gradient direction (per-tensor comparison of tiny bias gradients is noise-dominated)
        import math
        dot = sum((gr.double().flatten()[::g["grads"][k].get("stride", 1)].cpu() * (g["grads"][k].get("full", g["grads"][k].get("sample")).double())).sum().item()
                  for k, gr in grads.items())
        na = math.sqrt(sum((gr.double().flatten()[::g["grads"][k].get("stride", 1)] ** 2).sum().item() for k, gr in grads.items()))
        nb = math.sqrt(sum((g["grads"][k].get("full", g["grads"][k].get("sample")).double() ** 2).sum().item() for k in grads))
        print("bf16 UNet_Plus whole-gradient cosine vs reference: %.4f" % (dot / (na * nb)))
        assert dot / (na * nb) > 0.9, dot / (na * nb)      # (plain bf16 U-Net backward at this size: per-tensor rel-l2 up to 0.7)
    # the encoder gradient must contain the bottleneck path: without the high neck's gradient it differs
    model2.eval()
    with torch.no_grad():
        val = model2.val(x)
    check_summary(val, g["val_logits"], rtol=tol, what="val logits")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_hpfg_main_step_vs_reference_golden(precision):
    """main.py:128-207 (the HPFG iteration: three UNet_Plus networks, CutMix batch, supervised + Dice-on-mixed-pseudo-labels
    + Mean-Teacher MSE + two Dense_Loss terms, two SGD steps, backbone EMA and teacher EMA).  The SAME transcription of the
    caller code (tests/golden/common.py:hpfg_main_step) produced the fixture with the reference's objects on CPU and runs
    here with hpfg_b200's drop-ins: only the imports differ."""
    import copy
    import types
    from tests.golden.common import make_plus_state, hpfg_main_step, make_hpfg_batch
    g = load_golden("hpfg_step_acdc.pt")
    c = g["cfg"]
    f32 = precision == "fp32"
    torch.backends.cudnn.allow_tf32 = False
    in_ch, n_cls, n_l, n_u, h, w, seed = c["in_ch"], c["n_cls"], c["n_l"], c["n_u"], c["h"], c["w"], c["seed"]
    args = types.SimpleNamespace(num_classes=n_cls, batch_size=n_l, unlabel_batch_size=n_u, consistency=0.1,
                                 consistency_rampup=200.0, ema_decay=0.99)
    before1, before2 = make_plus_state(in_ch, n_cls, seed), make_plus_state(in_ch, n_cls, seed + 20)
    model1 = hb.UNet_Plus(in_ch, n_cls, precision=precision)
    model1.load_state_dict(before1)
    model1 = model1.to(DEV)
    model2 = hb.UNet_Plus(in_ch, n_cls, precision=precision)
    model2.load_state_dict(before2)
    model2 = model2.to(DEV)
    ema_model = copy.deepcopy(model2)
    for name, param in ema_model.named_parameters():
        param.requires_grad = False
    optimizer1 = torch.optim.SGD(model1.parameters(), lr=0.01, momentum=0.9, weight_decay=0.0005)
    optimizer2 = torch.optim.SGD(model2.parameters(), lr=0.01, momentum=0.9, weight_decay=0.0005)
    lam = lambda e: (1.0 - (e - 1) / 30000) ** 0.9                         # Medical_LR (utils/scheduler/medical_lr.py:13-17)
    sch1 = torch.optim.lr_scheduler.LambdaLR(optimizer1, lam)
    sch2 = torch.optim.lr_scheduler.LambdaLR(optimizer2, lam)
    model1.train(), model2.train()
    model1.set_dropout_masks(make_masks(n_l + n_u, h, w, seed + 31))
    model2.set_dropout_masks(make_masks(n_l + n_u, h, w, seed + 32))
    ema_model.set_dropout_masks(make_masks(n_l + n_u, h, w, seed + 33))
    ns = types.SimpleNamespace(DiceLoss=hb.DiceLoss, Dense_Loss=hb.Dense_Loss, update_ema_variables=hb.update_ema_variables,
                               linear_rampup=hb.linear_rampup)
    r = hpfg_main_step(ns, model1, model2, ema_model, optimizer1, optimizer2, sch1, sch2,
                       make_hpfg_batch(n_l, n_u, in_ch, n_cls, h, w, seed + 40), c["cur_itrs"], args, torch.device(DEV))
    sc = g["scalars"]
    for k, tol32, tol16 in (("loss", 1e-5, 2e-3), ("loss_sup", 1e-5, 2e-3), ("contrast", 1e-4, 3e-2), ("pseudo", 1e-5, 5e-3),
                            ("cons2", 1e-4, 1e-1)):
        assert abs(r[k] - sc[k]) / abs(sc[k]) < (tol32 if f32 else tol16), (k, r[k], sc[k])
    tol = 1e-5 if f32 else 3e-2
    check_summary(r["outputs1"], g["outputs1"], rtol=tol, what="outputs1")
    check_summary(r["outputs2"], g["outputs2"], rtol=tol, what="outputs2")
    check_summary(r["ema_output"], g["ema_output"], rtol=tol, what="ema_output")
    assert model1._is_flat() and model2._is_flat() and ema_model._is_flat()
    if not f32:
        return
    for nm, m in (("model1", model1), ("model2", model2), ("ema_model", ema_model)):
        sd = m.state_dict()
        for k, summ in g["after"][nm].items():
            check_summary(sd[k], summ, rtol=1e-4 if "running_" in k else 2e-5, atol=1e-6, what=nm + "." + k)
    # the updates themselves (after - before), where the optimiser step and both EMA passes show: model1 moved by its SGD
    # step, the teacher moved 1 % of the way towards the updated model2 (whose backbone moved 1 % towards model1)
    for nm, m, before in (("model1", model1, before1), ("ema_model", ema_model, before2)):
        sd = m.state_dict()
        for k in ("encoder.down4.maxpool_conv.1.conv_conv.4.weight", "decoder.up4.conv.conv_conv.0.weight",
                  "decoder.out_conv.weight", "dense_projection_high.mlp_conv.2.weight", "dense_projection_head.mlp.0.weight"):
            summ = g["after"][nm][k]
            ref_after = summ["full"] if "full" in summ else summ["sample"]
            b = before[k].flatten()
            got = sd[k].detach().cpu().flatten()
            if "full" not in summ:
                b, got = b[::summ["stride"]], got[::summ["stride"]]
            d_ref, d_got = ref_after.double() - b.double(), got.double() - b.double()
            # (2e-7 * |w|: fp32 rounding of the stored weights, which is all that is left of the teacher's 1 % step on
            # tensors whose gradient is tiny)
            assert (d_got - d_ref).norm() <= 2e-2 * d_ref.norm() + 2e-7 * b.double().norm(), \
                (nm, k, float((d_got - d_ref).norm() / d_ref.norm()))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_hpfg_step_driver_vs_reference_golden(precision):
    """``HPFGStep`` (the packaged driver of main.py:128-207: autograd through the three UNet_Plus networks, fused flat SGD for
    the U-Net tensors + per-tensor SGD for the necks, flat backbone / teacher EMA passes) against the same reference fixture
    as the transcription test above."""
    import copy
    from tests.golden.common import make_plus_state, make_hpfg_batch
    g = load_golden("hpfg_step_acdc.pt")
    c = g["cfg"]
    f32 = precision == "fp32"
    torch.backends.cudnn.allow_tf32 = False
    in_ch, n_cls, n_l, n_u, h, w, seed = c["in_ch"], c["n_cls"], c["n_l"], c["n_u"], c["h"], c["w"], c["seed"]
    before1, before2 = make_plus_state(in_ch, n_cls, seed), make_plus_state(in_ch, n_cls, seed + 20)
    model1 = hb.UNet_Plus(in_ch, n_cls, precision=precision)
    model1.load_state_dict(before1)
    model1 = model1.to(DEV)
    model2 = hb.UNet_Plus(in_ch, n_cls, precision=precision)
    model2.load_state_dict(before2)
    model2 = model2.to(DEV)
    ema_model = copy.deepcopy(model2)
    step = hb.HPFGStep(model1, model2, ema_model, weight_decay=0.0005)
    model1.set_dropout_masks(make_masks(n_l + n_u, h, w, seed + 31))
    model2.set_dropout_masks(make_masks(n_l + n_u, h, w, seed + 32))
    ema_model.set_dropout_masks(make_masks(n_l + n_u, h, w, seed + 33))
    step.cur_itrs = c["cur_itrs"] - 1
    batch = [t.to(DEV) for t in make_hpfg_batch(n_l, n_u, in_ch, n_cls, h, w, seed + 40)]
    loss = step.step(*batch, lr=0.01 * (1.0 + 1.0 / 30000) ** 0.9)          # the fixture's fresh Medical_LR scheduler
    sc = g["scalars"]
    got = dict(loss=loss.item(), loss_sup=step.last["loss_sup"].item(), contrast=step.last["contrast"].item(),
               pseudo=step.last["pseudo"].item())
    for k, tol32, tol16 in (("loss", 1e-5, 2e-3), ("loss_sup", 1e-5, 2e-3), ("contrast", 1e-4, 3e-2), ("pseudo", 1e-5, 5e-3)):
        assert abs(got[k] - sc[k]) / abs(sc[k]) < (tol32 if f32 else tol16), (k, got[k], sc[k])
    tol = 1e-5 if f32 else 3e-2
    check_summary(step.last["outputs1"], g["outputs1"], rtol=tol, what="outputs1")
    check_summary(step.last["outputs2"], g["outputs2"], rtol=tol, what="outputs2")
    assert model1._is_flat() and model2._is_flat() and ema_model._is_flat()
    if f32:
        for nm, m in (("model1", model1), ("model2", model2), ("ema_model", ema_model)):
            sd = m.state_dict()
            for k, summ in g["after"][nm].items():
                check_summary(sd[k], summ, rtol=1e-4 if "running_" in k else 2e-5, atol=1e-6, what=nm + "." + k)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_s4cv_step_driver_vs_oracle(precision):
    """``S4CVStep`` (2022_08_CVPR_S4CVNet_ACDC.py:108-167) against the oracle's restatement of the iteration: before and
    after the Mean-Teacher terms switch on (mt_start), with dropout masks and the teacher's input noise supplied."""
    import oracle
    from tests.golden.common import make_state, make_batch
    in_ch, n_cls, n_l, n_u, h, w = 1, 4, 2, 4, 32, 48
    f32 = precision == "fp32"
    st1, st2 = make_state(in_ch, n_cls, 131), make_state(in_ch, n_cls, 132)
    m1, m2 = hb.UNet(in_ch, n_cls, precision=precision), hb.UNet(in_ch, n_cls, precision=precision)
    m1.load_state_dict(st1)
    m2.load_state_dict(st2)
    m1, m2 = m1.to(DEV), m2.to(DEV)
    import copy
    te = copy.deepcopy(m2)
    o1, o2 = {k: v.clone() for k, v in st1.items()}, {k: v.clone() for k, v in st2.items()}
    ot = {k: v.clone() for k, v in st2.items()}
    step = hb.S4CVStep(m1, m2, te, mt_start=2)
    opt1, opt2 = oracle.SGDState(), oracle.SGDState()
    gen = torch.Generator().manual_seed(9)
    for it in (1, 2, 3):
        x_l, x_u, y = make_batch(n_l, n_u, in_ch, n_cls, h, w, 140 + it)
        noise = torch.clamp(torch.randn(x_u.shape, generator=gen) * 0.1, -0.2, 0.2)
        k1, k2, kt = make_masks(n_l + n_u, h, w, 150 + it), make_masks(n_l + n_u, h, w, 160 + it), make_masks(n_u, h, w, 170 + it)
        m1.set_dropout_masks(k1)
        m2.set_dropout_masks(k2)
        te.set_dropout_masks(kt)
        loss = step.step(torch.cat([x_l, x_u]).to(DEV), y.to(DEV), noise.to(DEV))
        r = oracle.s4cv_step(o1, o2, ot, opt1, opt2, x_l, x_u, y, it, noise, mt_start=2, masks1=k1, masks2=k2, teacher_masks=kt)
        assert abs(loss.item() - r["loss"]) / r["loss"] < (2e-5 if f32 else 2e-2), (it, loss.item(), r["loss"])
        if f32:
            assert rel_l2(step.last["logits1"], r["logits1"]) < 1e-5 and rel_l2(step.last["teacher_logits"], r["teacher_logits"]) < 1e-5
            for m, o in ((m1, o1), (m2, o2), (te, ot)):
                sd = m.state_dict()
                for k in ("decoder.out_conv.weight", "encoder.in_conv.conv_conv.0.weight", "encoder.down4.maxpool_conv.1.conv_conv.5.running_var"):
                    assert torch.allclose(sd[k].cpu(), o[k], rtol=1e-4, atol=5e-6), (it, k)
