"""CPU: the oracle restatement against the golden vectors produced by the REAL reference
(tests/golden/make_golden.py).  This is what pins the oracle on machines without /root/reference."""
import math

import pytest
import torch

import oracle
from tests.golden.common import make_state, make_masks, make_batch
from tests.helpers import load_golden, check_summary, rel_l2


@pytest.mark.parametrize("tag", ["acdc_masks", "acdc_nodrop", "isic_masks"])
def test_unet_forward_backward(tag):
    g = load_golden("unet_%s.pt" % tag)
    c = g["cfg"]
    st = make_state(c["in_ch"], c["n_cls"], c["seed"])
    x, _, y = make_batch(c["n"], 0, c["in_ch"], c["n_cls"], c["h"], c["w"], c["seed"] + 7)
    masks = make_masks(c["n"], c["h"], c["w"], c["seed"] + 11) if c["use_masks"] else {}
    names = [n for n, _ in oracle.unet_param_spec(c["in_ch"], c["n_cls"])]
    leaves = {n: st[n].clone().requires_grad_(True) for n in names}
    view = dict(st)
    view.update(leaves)
    logits = oracle.unet_forward(view, x, True, masks)
    assert torch.allclose(logits, g["logits"], rtol=0, atol=1e-5)
    loss = oracle.med_sup_loss(logits, y, c["n_cls"])
    assert abs(loss.item() - g["loss"]) < 1e-6
    grads = torch.autograd.grad(loss, [leaves[n] for n in names])
    for n, gr in zip(names, grads):
        check_summary(gr, g["grads"][n], rtol=1e-4, atol=1e-7, what=n)
    for k, v in g["buffers"].items():
        assert torch.allclose(view[k].float(), v.float(), rtol=1e-5, atol=1e-6), k
    out_eval = oracle.unet_forward(view, x, False)
    assert torch.allclose(out_eval, g["logits_eval"], rtol=0, atol=1e-5)


@pytest.mark.parametrize("tag", ["c4", "c2"])
def test_losses(tag):
    g = load_golden("losses.pt")[tag]
    n_l, n_u, C, H, W = g["shape"]
    s = g["student"].clone().requires_grad_(True)
    t, y, y255 = g["teacher"], g["y"], g["y255"]
    for nm, yy in (("sup", y), ("sup255", y255)):
        l = oracle.med_sup_loss(s[:n_l], yy, C)
        (gr,) = torch.autograd.grad(l, s)
        assert abs(l.item() - g[nm]) < 1e-6
        assert rel_l2(gr, g[nm + "_grad"]) < 1e-6
    l = oracle.dice_loss(s[:n_l], y.unsqueeze(1), C, weight=g["dice_weights"], softmax=True)
    (gr,) = torch.autograd.grad(l, s)
    assert abs(l.item() - g["dice_w"]) < 1e-6 and rel_l2(gr, g["dice_w_grad"]) < 1e-6
    assert abs(oracle.dice_loss(torch.softmax(s, 1)[:n_l], y.unsqueeze(1), C).item() - g["dice"]) < 1e-6
    mt = g["mt"]
    sup = oracle.med_sup_loss(s[:n_l], y, C)
    cons = oracle.mt_consistency(s[n_l:], t[n_l:])
    l = sup + mt["w"] * cons
    (gr,) = torch.autograd.grad(l, s)
    assert abs(l.item() - mt["loss"]) < 1e-6 and abs(cons.item() - mt["cons"]) < 1e-8
    assert rel_l2(gr, mt["grad"]) < 1e-6
    cps = g["cps"]
    s2 = cps["logits2"].clone().requires_grad_(True)
    lsup, lsemi, pl1, pl2 = oracle.cps_losses(s, s2, y, n_l, C)
    l = lsup + cps["w"] * lsemi
    g1, g2 = torch.autograd.grad(l, [s, s2])
    assert torch.equal(pl1, cps["pl1"]) and torch.equal(pl2, cps["pl2"])
    assert abs(l.item() - cps["loss"]) < 2e-6
    assert rel_l2(g1, cps["grad1"]) < 1e-6 and rel_l2(g2, cps["grad2"]) < 1e-6
    u = g["uamt"]
    sup_u = 0.5 * (oracle.dice_loss(torch.softmax(s, 1)[:n_l], y.unsqueeze(1), C) + oracle.ce_loss(s[:n_l], y))
    cons_u, unc, mask = oracle.uamt_consistency(s[n_l:], t[n_l:], u["mc_logits"], u["T"], u["threshold"])
    l = sup_u + u["w"] * cons_u
    (gr,) = torch.autograd.grad(l, s)
    assert abs(l.item() - u["loss"]) < 1e-6 and mask.sum().item() == u["mask_sum"]
    assert torch.allclose(unc, u["uncertainty"], atol=1e-6) and rel_l2(gr, u["grad"]) < 1e-6


def test_schedules_and_ema():
    g = load_golden("schedules.pt")
    for it, w in g["rampup"]:
        assert oracle.consistency_weight(it) == pytest.approx(w, rel=1e-12)
    for c, L, v in g["sigmoid"]:
        assert oracle.sigmoid_rampup(c, L) == pytest.approx(v, rel=1e-12)
    for i, lr in enumerate(g["medical_lr_first5"]):
        assert oracle.medical_lr(i) == pytest.approx(lr, rel=1e-12)
    names = ["w", "b"]
    for step, outs in g["ema_out"].items():
        stu = dict(zip(names, [q.clone() for q in g["ema_in"]["student"]]))
        tea = dict(zip(names, [q.clone() for q in g["ema_in"]["teacher"]]))
        oracle.update_ema(stu, tea, 0.99, step, names)
        for n, o in zip(names, outs):
            assert torch.equal(tea[n], o)


@pytest.mark.parametrize("tag", ["acdc", "isic"])
def test_mt_steps(tag):
    g = load_golden("mt_steps_%s.pt" % tag)
    c = g["cfg"]
    student = make_state(c["in_ch"], c["n_cls"], c["seed"])
    teacher = {k: v.clone() for k, v in student.items()}
    opt = oracle.SGDState()
    names = [n for n, _ in oracle.unet_param_spec(c["in_ch"], c["n_cls"])]
    for it, rec in enumerate(g["steps"], start=1):
        x_l, x_u, y = make_batch(c["n_l"], c["n_u"], c["in_ch"], c["n_cls"], c["h"], c["w"], c["seed"] + 100 * it)
        n = c["n_l"] + c["n_u"]
        r = oracle.mt_step(student, teacher, opt, x_l, x_u, y, it,
                           student_masks=make_masks(n, c["h"], c["w"], c["seed"] + 100 * it + 1),
                           teacher_masks=make_masks(n, c["h"], c["w"], c["seed"] + 100 * it + 2))
        assert r["loss"] == pytest.approx(rec["loss"], abs=2e-6)
        assert r["loss_cons"] == pytest.approx(rec["cons"], rel=1e-4)
        assert r["w"] == pytest.approx(rec["w"], rel=1e-12) and r["lr"] == pytest.approx(rec["lr"], rel=1e-12)
        check_summary(r["logits"], rec["logits"], rtol=1e-5, what="logits")
        check_summary(r["teacher_logits"], rec["teacher_logits"], rtol=1e-5, what="teacher logits")
        assert torch.allclose(student["decoder.out_conv.weight"], rec["student_out_conv"], atol=1e-6)
        assert torch.allclose(teacher["decoder.out_conv.weight"], rec["teacher_out_conv"], atol=1e-6)
        assert torch.allclose(student["encoder.in_conv.conv_conv.0.weight"], rec["student_in_conv"], atol=1e-6)
        assert torch.allclose(teacher["encoder.in_conv.conv_conv.1.running_mean"], rec["teacher_rm"], atol=1e-6)
        assert torch.allclose(student["decoder.up4.conv.conv_conv.5.running_var"], rec["student_rv"], atol=1e-6)
        ssum = sum(student[k].double().sum().item() for k in names)
        tsum = sum(teacher[k].double().sum().item() for k in names)
        assert math.isclose(ssum, rec["student_sum"], abs_tol=1e-3) and math.isclose(tsum, rec["teacher_sum"], abs_tol=1e-3)


# ---- SURVEY 8f.3 / 8f.4 rows: ICT-MedSeg, S4CVNet, inference ----------------------------------------------------
@pytest.mark.parametrize("tag", ["c4", "c2"])
def test_f4_losses(tag):
    g = load_golden("f4_losses.pt")[tag]
    n_l, n_m, C, H, W = g["shape"]
    ict = g["ict"]
    s = ict["student"].clone().requires_grad_(True)
    sup, cons = oracle.ict_losses(s, ict["teacher"], ict["mix"], ict["y"], n_l, C)
    l = sup + ict["w"] * cons
    (gr,) = torch.autograd.grad(l, s)
    assert abs(l.item() - ict["loss"]) < 1e-6 and abs(cons.item() - ict["cons"]) < 1e-8
    assert rel_l2(gr, ict["grad"]) < 1e-6
    s4 = g["s4cv"]
    for branch in ("early", "late"):
        b = s4[branch]
        o1, o2 = s4["logits1"].clone().requires_grad_(True), s4["logits2"].clone().requires_grad_(True)
        t = s4["teacher"] if b["cur_itrs"] >= 1000 else None
        l, lsup, lsemi, pl1, pl2 = oracle.s4cv_losses(o1, o2, t, s4["y"], n_l, C, b["cps_weight"], b["mt_weight"])
        g1, g2 = torch.autograd.grad(l, [o1, o2])
        assert torch.equal(pl1, b["pl1"]) and torch.equal(pl2, b["pl2"])
        assert abs(l.item() - b["loss"]) < 2e-6 and abs(lsemi.item() - b["semi"]) < 2e-6
        assert rel_l2(g1, b["grad1"]) < 1e-6 and rel_l2(g2, b["grad2"]) < 1e-6


def test_ict_steps():
    g = load_golden("ict_steps_acdc.pt")
    c = g["cfg"]
    student = make_state(c["in_ch"], c["n_cls"], c["seed"])
    teacher = make_state(c["in_ch"], c["n_cls"], c["seed"] + 7)
    opt = oracle.SGDState()
    n_m = c["n_u"] // 2
    for i, rec in enumerate(g["steps"]):
        it = i + 1
        x_l, x_u, y = make_batch(c["n_l"], c["n_u"], c["in_ch"], c["n_cls"], c["h"], c["w"], c["seed"] + 100 * it)
        ms = make_masks(c["n_l"] + n_m, c["h"], c["w"], c["seed"] + 100 * it + 1)
        mt = make_masks(n_m, c["h"], c["w"], c["seed"] + 100 * it + 2)
        lam = torch.rand(n_m, 1, 1, 1, generator=torch.Generator().manual_seed(c["seed"] + 100 * it + 3))
        r = oracle.ict_step(student, teacher, opt, x_l, x_u, y, it, lam, student_masks=ms, teacher_masks=[mt, mt])
        assert r["loss"] == pytest.approx(rec["loss"], abs=2e-6)
        assert r["loss_cons"] == pytest.approx(rec["cons"], rel=1e-4)
        assert r["lr"] == pytest.approx(rec["lr"], rel=1e-12) and r["w"] == pytest.approx(rec["w"], rel=1e-12)
        check_summary(r["logits"], rec["logits"], rtol=1e-5, atol=1e-6, what="logits")
        check_summary(r["teacher_logits"], rec["teacher_logits"], rtol=1e-5, atol=1e-6, what="teacher logits")
        assert torch.allclose(student["decoder.out_conv.weight"], rec["student_out_conv"], atol=1e-6)
        assert torch.allclose(teacher["decoder.out_conv.weight"], rec["teacher_out_conv"], atol=1e-6)
        assert torch.allclose(teacher["encoder.in_conv.conv_conv.1.running_mean"], rec["teacher_rm"], atol=1e-6)


def test_predict_labels():
    from tests.golden.common import make_predict_case
    g = load_golden("predict_acdc.pt")
    c = g["cfg"]
    st, vol = make_predict_case(c["in_ch"], c["n_cls"], c["n"], c["h"], c["w"], c["seed"])
    st.update(g["buffers"])
    soft = torch.softmax(oracle.unet_forward(st, vol.unsqueeze(1), False), dim=1)     # one batch == slice by slice in eval
    labels = torch.argmax(soft, dim=1)
    sure = g["margin"].float() > 1e-3
    assert torch.equal(labels[sure], g["labels"].long()[sure])
    assert (labels == g["labels"].long()).float().mean().item() > 0.999


def test_unet_plus_and_dense_loss():
    """SURVEY 8f.2: UNet_Plus + Dense_Loss restatement vs the reference-generated fixture (main.py:151-170 usage)."""
    from tests.golden.common import make_plus_state
    g = load_golden("unet_plus_acdc.pt")
    c = g["cfg"]
    st = make_plus_state(c["in_ch"], c["n_cls"], c["seed"])
    te = make_plus_state(c["in_ch"], c["n_cls"], c["seed"] + 9)
    x, _, y = make_batch(c["n"], 0, c["in_ch"], c["n_cls"], c["h"], c["w"], c["seed"] + 7)
    names = [n for n, _ in oracle.unet_param_spec(c["in_ch"], c["n_cls"])] + [n for n, _ in oracle.unet_plus_neck_spec(c["n_cls"])]
    assert names == list(g["grads"].keys())
    leaves = {n: st[n].clone().requires_grad_(True) for n in names}
    view = dict(st)
    view.update(leaves)
    out, h1, h2 = oracle.unet_plus_forward(view, x, True, make_masks(c["n"], c["h"], c["w"], c["seed"] + 11))
    with torch.no_grad():
        _, e1, e2 = oracle.unet_plus_forward(te, x, True, make_masks(c["n"], c["h"], c["w"], c["seed"] + 12))
    check_summary(out, g["logits"], rtol=1e-5, atol=1e-6, what="logits")
    for a, b in zip(h1 + h2 + e1 + e2, g["h1"] + g["h2"] + g["ema_h1"] + g["ema_h2"]):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-5)
    sup = oracle.med_sup_loss(out, y, c["n_cls"])
    con = oracle.dense_loss(h1, e1) + oracle.dense_loss(h2, e2)
    loss = sup + c["weight"] * con
    assert abs(sup.item() - g["sup"]) < 1e-6 and abs(con.item() - g["contrast"]) / g["contrast"] < 1e-5
    assert abs(loss.item() - g["loss"]) / g["loss"] < 1e-5
    grads = torch.autograd.grad(loss, [leaves[n] for n in names])
    for n, gr in zip(names, grads):
        if n.endswith("conv_conv.0.bias") or n.endswith("conv_conv.4.bias"):
            # conv biases ahead of train-mode BatchNorm have an analytically zero gradient: both sides hold rounding noise,
            # which changes with the number of CPU threads, so it is bounded on an absolute scale
            assert g["grads"][n]["abs_sum"] < 1e-5 * g["grads"][n]["numel"], n
            assert gr.abs().max().item() < 1e-5, n
            continue
        check_summary(gr, g["grads"][n], rtol=2e-4, atol=1e-6, what=n)
    check_summary(oracle.unet_forward(view, x, False), g["val_logits"], rtol=1e-5, atol=1e-6, what="val logits")
