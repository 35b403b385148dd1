"""CPU: the oracle against what the REAL reference produced.

The first two tests are self-contained: they rebuild the reference's initial state and inputs from its seed and compare the
oracle with values the reference modules themselves printed (tests/golden/reference_mt_acdc.json, SURVEY.md Appendix B) and
with the parameter / buffer names recorded in the reference-generated fixtures.  The last two re-run the reference's code and
need a checkout of it (HPFG_REF=<path>); they skip without one."""
import json
import math
import os
from collections import OrderedDict

import pytest
import torch

import oracle
from oracle.ref_loader import find_reference, load_reference
from tests.helpers import GOLDEN, load_golden

needs_reference = pytest.mark.skipif(find_reference() is None, reason="no reference checkout (set HPFG_REF)")


def _reference_values():
    with open(os.path.join(GOLDEN, "reference_mt_acdc.json")) as f:
        return json.load(f)


def _reference_init_state(in_ch, n_cls):
    """The state `UNet(in_ch, n_cls)` of model/unet.py starts from under the current torch seed: its nn.Conv2d modules are
    built in parameter order and each draws weight then bias from torch's global RNG; BatchNorm starts at weight 1, bias 0."""
    st = OrderedDict()
    for name, shape in oracle.unet_param_spec(in_ch, n_cls):
        if len(shape) == 4:
            conv = torch.nn.Conv2d(shape[1], shape[0], shape[2])
            st[name], st[name[:-len("weight")] + "bias"] = conv.weight.detach(), conv.bias.detach()
        elif name not in st:
            st[name] = torch.ones(shape) if name.endswith("weight") else torch.zeros(shape)
    for name, shape, dt in oracle.unet_buffer_spec(in_ch, n_cls):
        st[name] = torch.ones(shape, dtype=dt) if name.endswith("running_var") else torch.zeros(shape, dtype=dt)
    return st


def _reference_case():
    """Seeded state and batch of the stored reference run, checked against the sums the reference printed."""
    ref = _reference_values()
    torch.manual_seed(ref["seed"])
    st = _reference_init_state(ref["in_channels"], ref["num_classes"])
    n_l, n_u, hw = ref["n_labeled"], ref["n_unlabeled"], ref["hw"]
    x_l, x_u = torch.rand(n_l, ref["in_channels"], hw, hw), torch.rand(n_u, ref["in_channels"], hw, hw)
    y = torch.randint(0, ref["num_classes"], (n_l, hw, hw))
    names = [n for n, _ in oracle.unet_param_spec(ref["in_channels"], ref["num_classes"])]
    assert sum(st[n].double().sum().item() for n in names) == pytest.approx(ref["param_sum_init"], abs=1e-5)
    assert sum(st[n].double().abs().sum().item() for n in names) == pytest.approx(ref["param_abs_sum_init"], abs=1e-5)
    assert x_l.double().sum().item() == pytest.approx(ref["x_l_sum"], abs=1e-3)
    assert x_u.double().sum().item() == pytest.approx(ref["x_u_sum"], abs=1e-3)
    assert y.sum().item() == ref["y_sum"]
    return ref, st, names, x_l, x_u, y


def test_names_shapes_and_rng_dropout_forward():
    """Parameter and buffer names / sizes in the reference's order (recorded in the reference-generated fixtures), and the
    student forward with dropout drawn from torch's RNG as nn.Dropout draws it: its supervised loss is the reference's."""
    for tag, (in_ch, n_cls) in (("acdc_masks", (1, 4)), ("isic_masks", (3, 2))):
        g = load_golden("unet_%s.pt" % tag)
        spec = oracle.unet_param_spec(in_ch, n_cls)
        assert [n for n, _ in spec] == list(g["grads"])
        assert [math.prod(s) for _, s in spec] == [g["grads"][n]["numel"] for n in g["grads"]]
        bufs = oracle.unet_buffer_spec(in_ch, n_cls)
        assert [(n, tuple(s)) for n, s, _ in bufs] == [(k, tuple(v.shape)) for k, v in g["buffers"].items()]
    ref, st, _, x_l, x_u, y = _reference_case()
    with torch.no_grad():
        out = oracle.unet_forward(st, torch.cat([x_l, x_u]), True)
    sup = oracle.med_sup_loss(out[:x_l.shape[0]], y, ref["num_classes"])
    assert sup.item() == pytest.approx(ref["steps"][0]["sup"], abs=1e-6)


def test_full_size_mt_step_matches_reference_objects():
    """Three literal MT steps at the benchmark shape (12+12, 1x224x224) with torch-RNG dropout against the reference's values."""
    ref, student, names, x_l, x_u, y = _reference_case()
    teacher = {k: v.clone() for k, v in student.items()}
    opt = oracle.SGDState()
    for rec in ref["steps"]:
        r = oracle.mt_step(student, teacher, opt, x_l, x_u, y, rec["it"])
        assert r["lr"] == pytest.approx(rec["lr"], abs=1e-10)
        assert r["loss"] == pytest.approx(rec["loss"], abs=1e-6)
        assert r["loss_sup"] == pytest.approx(rec["sup"], abs=1e-6)
        assert r["loss_cons"] == pytest.approx(rec["cons"], rel=1e-5)
        if "w" in rec:
            assert r["w"] == pytest.approx(rec["w"], rel=1e-6)
        assert sum(student[n].double().sum().item() for n in names) == pytest.approx(rec["student_param_sum"], abs=1e-4)
        assert sum(teacher[n].double().sum().item() for n in names) == pytest.approx(rec["ema_param_sum"], abs=1e-4)


def _same(a, b, path=""):
    if isinstance(a, dict):
        assert isinstance(b, dict) and list(a.keys()) == list(b.keys()), path
        for k in a:
            _same(a[k], b[k], path + "/" + str(k))
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, path + "[%d]" % i)
    elif torch.is_tensor(a):
        assert torch.is_tensor(b) and a.dtype == b.dtype and a.shape == b.shape, path
        assert torch.allclose(a.double(), b.double(), rtol=1e-5, atol=1e-7), path
    elif isinstance(a, float):
        assert a == pytest.approx(b, rel=1e-5, abs=1e-8), path
    else:
        assert a == b, path


@needs_reference
def test_committed_8f_fixtures_are_what_the_reference_produces(tmp_path, monkeypatch):
    """Re-run tests/golden/make_golden.py's SURVEY-8f generators against the REAL reference modules (UNet_Plus, Dense_Loss,
    DiceLoss, Medical_LR, update_ema_variables ...) and compare with the committed fixtures the GPU tests use."""
    import importlib.util
    import os
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    monkeypatch.setattr(sys, "argv", ["make_golden.py"])
    spec = importlib.util.spec_from_file_location("_make_golden_check", os.path.join(here, "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    monkeypatch.setattr(mg, "HERE", str(tmp_path))
    mg.golden_f4_losses()
    mg.golden_ict_steps("acdc", 1, 4, 2, 4, 32, 32, 606)
    mg.golden_predict(1, 4, 5, 32, 48, 707)
    mg.golden_unet_plus(1, 4, 3, 64, 64, 808)
    mg.golden_hpfg_step(1, 4, 2, 4, 64, 64, 909)
    for name in ("f4_losses.pt", "ict_steps_acdc.pt", "predict_acdc.pt", "unet_plus_acdc.pt", "hpfg_step_acdc.pt"):
        new = torch.load(os.path.join(str(tmp_path), name), weights_only=False)
        old = torch.load(os.path.join(here, "golden", name), weights_only=False)
        _same(old, new, name)


@needs_reference
def test_oracle_necks_and_dense_loss_match_reference_objects():
    """The oracle's projection_conv / dense_loss restatements (what the GPU tests of csrc/neck.cu compare against) give the
    same numbers as the reference modules (model/unet.py:120-152, utils/loss/dense_loss.py) on CPU, values and gradients."""
    import hpfg_b200 as hb
    ref = load_reference()
    from oracle.ref_loader import _load
    import os
    unet = _load("_hpfg_ref_unet_necks", os.path.join(ref.root, "model", "unet.py"))
    torch.manual_seed(3)
    for in_dim, hid, shape in ((256, 2048, (2, 256, 14, 14)), (4, 1024, (2, 4, 64, 64))):
        r = unet.projection_conv(in_dim, hid_dim=hid)
        m = hb.projection_conv(in_dim, hid_dim=hid)
        assert [k for k, _ in m.named_parameters()] == [k for k, _ in r.named_parameters()]
        assert [tuple(p.shape) for p in m._param_list()] == [tuple(p.shape) for p in r.parameters()]   # the kernel's params[8] order
        m.load_state_dict(r.state_dict())
        st = {"neck." + k: v for k, v in r.state_dict().items()}
        f = torch.randn(shape)
        (a1, a2), (b1, b2) = r(f), oracle.projection_conv(st, "neck", f)
        assert torch.equal(a1, b1) and torch.equal(a2, b2)
    for bs in (3, 8):
        x = (torch.randn(bs, 128, requires_grad=True), torch.randn(bs, 128, 16, requires_grad=True))
        y = (torch.randn(bs, 128), torch.randn(bs, 128, 16))
        la = ref.Dense_Loss(batch_size=bs, device=torch.device("cpu"))(x, y)
        lo = oracle.dense_loss(x, y)
        assert la.item() == pytest.approx(lo.item(), rel=1e-6)
        for ga, gb in zip(torch.autograd.grad(la, x), torch.autograd.grad(lo, x)):
            assert torch.allclose(ga, gb, rtol=1e-5, atol=1e-8)
