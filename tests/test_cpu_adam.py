"""CPU: the Adam / AdamW option of the step drivers -- argument checking, the host-side per-step scalars, and the
torch.optim.Adam / AdamW checkpoint layout (the kernel itself: tests/test_gpu_adam.py)."""
import copy

import pytest
import torch

import hpfg_b200 as hb
from hpfg_b200.optim import OptState

KINDS = ("mt", "cps", "uamt", "ict", "s4cv", "hpfg")
# per driver kind: the attribute holding each trained network's (exp_avg, exp_avg_sq) and its number of parameters
OPTS = {"mt": [("mom", 82)], "cps": [("b1", 82), ("b2", 82)], "uamt": [("mom", 82)], "ict": [("mom", 82)],
        "s4cv": [("b1", 82), ("b2", 82)], "hpfg": [("b1", 98), ("b2", 98)]}


def _driver(kind, **kw):
    torch.manual_seed(5)
    if kind == "hpfg":
        m1, m2 = hb.UNet_Plus(1, 4), hb.UNet_Plus(1, 4)
        nets = (m1, m2, copy.deepcopy(m2))
    else:
        a, b = hb.UNet(1, 4), hb.UNet(1, 4)
        nets = (a, b, copy.deepcopy(b)) if kind == "s4cv" else (a, b) if kind == "cps" else (a, copy.deepcopy(a))
    cls = dict(mt=hb.MeanTeacherStep, cps=hb.CPSStep, uamt=hb.UAMTStep, ict=hb.ICTStep, s4cv=hb.S4CVStep, hpfg=hb.HPFGStep)[kind]
    return cls(*nets, **kw), nets


@pytest.mark.parametrize("kind", KINDS)
def test_every_driver_accepts_adam_and_rejects_unknown_optimizers(kind):
    for name in ("adam", "adamw"):
        st, nets = _driver(kind, optimizer=name)
        assert st.optimizer == name
        for attr, _ in OPTS[kind]:
            m, v = getattr(st, attr)
            assert m.shape == v.shape == nets[0].flat_params.shape and not m.any() and not v.any()
    st, _ = _driver(kind)
    assert st.optimizer == "sgd" and isinstance(st.b1 if kind in ("cps", "s4cv", "hpfg") else st.mom, torch.Tensor)
    for bad in ("Adam", "rmsprop", None):
        with pytest.raises(ValueError):
            _driver(kind, optimizer=bad)


@pytest.mark.parametrize("name", ["adam", "adamw"])
def test_device_block_adam_groups_match_torch_python_formulas(name):
    """The Adam group of the device block is torch's double-precision scalars (adam.py, non-capturable foreach branch)
    rounded once to fp32; graph replays and eager launches read the same values."""
    lr0, wd, betas = 0.01, 1e-2, (0.9, 0.999)
    st, _ = _driver("cps", optimizer=name, lr=lr0, weight_decay=wd, betas=betas)
    for t in (1, 2, 3, 10, 150, 4000, 29999):
        st.cur_itrs = t
        for _, _, s in st._trained:
            s.step = t
        lr = hb.medical_lr(t, lr0, 30000)
        bc1, bc2 = 1 - betas[0] ** t, 1 - betas[1] ** t
        want = [(lr / bc1) * -1, bc2 ** 0.5, 1 - lr * wd if name == "adamw" else 1.0]
        assert st._opt.scalars(t, lr) == want
        block = torch.tensor(st._dyn_scalars(), dtype=torch.float32)
        assert block.numel() == 4 + 2 * 5
        for k in range(2):
            assert torch.equal(block[4 + 5 * k:4 + 5 * k + 3], torch.tensor(want, dtype=torch.float32))
    uamt, _ = _driver("uamt", optimizer=name)
    uamt.cur_itrs, uamt._trained[0][2].step = 3, 3
    block = uamt._dyn_scalars(0.99, 0.5)
    assert len(block) == 10 and block[4] == 0.5 and block[-2:] == block[1:3]       # [..., thr | step_size, bc2, decay, alpha, 1-alpha]


def _fill_state(st, kind):
    st.cur_itrs = 7
    for _, _, s in st._trained:
        s.step = 7
    for attr, _ in OPTS[kind]:
        m, v = getattr(st, attr)
        m.uniform_(-1, 1)
        v.uniform_(0, 1)
    if kind == "hpfg":
        for j, p in enumerate(st._neck_params(st.m2)):
            st._neck_states[id(p)] = OptState([torch.randn_like(p), torch.rand_like(p)], 3 + j)


@pytest.mark.parametrize("name", ["adam", "adamw"])
@pytest.mark.parametrize("kind", KINDS)
def test_adam_state_checkpoint_layout_and_roundtrip(kind, name):
    wd = 1e-4
    st, nets = _driver(kind, optimizer=name, weight_decay=wd)
    assert all(opt["state"] == {} for opt in st.state_dict()["optimizers"])       # no state before the first step
    _fill_state(st, kind)
    sd = st.state_dict()
    cls = torch.optim.AdamW if name == "adamw" else torch.optim.Adam
    ref_group = cls(nets[0].parameters(), lr=0.01, weight_decay=wd).state_dict()["param_groups"][0]
    assert len(sd["optimizers"]) == len(OPTS[kind])
    for k, (opt, (attr, n_params)) in enumerate(zip(sd["optimizers"], OPTS[kind])):
        group = opt["param_groups"][0]
        assert {a: b for a, b in group.items() if a not in ("params", "lr")} == \
            {a: b for a, b in ref_group.items() if a not in ("params", "lr")}
        assert group["lr"] == 0.00999819998199868 and group["params"] == list(range(n_params))
        n_state = 98 if kind == "hpfg" and attr == "b2" else 82      # model1's necks never get a gradient: no state
        assert sorted(opt["state"]) == list(range(n_state))
        for i in range(82):
            assert list(opt["state"][i]) == ["step", "exp_avg", "exp_avg_sq"]
            assert opt["state"][i]["step"].dtype == torch.float32 and float(opt["state"][i]["step"]) == 7.0
        m, v = getattr(st, attr)
        assert torch.equal(torch.cat([opt["state"][i]["exp_avg"].reshape(-1) for i in range(82)]), m)
        assert torch.equal(torch.cat([opt["state"][i]["exp_avg_sq"].reshape(-1) for i in range(82)]), v)
        # the entry is a torch.optim.Adam / AdamW state dict of the network's parameters, and comes back unchanged
        net = (nets[0], nets[1])[k]
        ref = cls(net.parameters(), lr=0.01, weight_decay=wd)
        ref.load_state_dict(copy.deepcopy(opt))
        back = ref.state_dict()
        assert sorted(back["state"]) == sorted(opt["state"])
        for i, s in opt["state"].items():
            assert all(torch.equal(back["state"][i][key], s[key]) for key in s)
        assert back["param_groups"][0] == group
    if kind == "hpfg":
        for j in range(16):
            assert float(sd["optimizers"][1]["state"][82 + j]["step"]) == 3 + j          # per-tensor step counts
    st2, nets2 = _driver(kind, optimizer=name, weight_decay=wd)
    st2.load_state_dict(sd)
    assert st2.cur_itrs == 7 and [s.step for _, _, s in st2._trained] == [7] * len(OPTS[kind])
    sd2 = st2.state_dict()
    for o, o2 in zip(sd["optimizers"], sd2["optimizers"]):
        assert o2["param_groups"] == o["param_groups"] and sorted(o2["state"]) == sorted(o["state"])
        for i in o["state"]:
            assert all(torch.equal(o2["state"][i][key], o["state"][i][key]) for key in o["state"][i])
    if kind == "hpfg":
        assert not any(id(q) in st2._neck_states for q in st2._neck_params(nets2[0]))
        assert [st2._neck_states[id(q)].step for q in st2._neck_params(nets2[1])] == [3 + j for j in range(16)]


@pytest.mark.parametrize("kind", ["mt", "hpfg"])
def test_adam_state_checkpoint_mismatches_raise(kind):
    st, _ = _driver(kind, optimizer="adamw")
    _fill_state(st, kind)
    sd = st.state_dict()
    bad = copy.deepcopy(sd)
    bad["optimizers"][0]["state"][5]["step"] = torch.tensor(6.0)          # one U-Net tensor one step behind
    with pytest.raises(ValueError, match="step count"):
        _driver(kind, optimizer="adamw")[0].load_state_dict(bad)
    bad = copy.deepcopy(sd)
    del bad["optimizers"][0]["state"][5]                                    # one U-Net tensor without state
    with pytest.raises(ValueError, match="step count"):
        _driver(kind, optimizer="adamw")[0].load_state_dict(bad)
    with pytest.raises(ValueError, match="Adam"):
        _driver(kind)[0].load_state_dict(sd)                                # Adam checkpoint -> SGD driver
    sgd, _ = _driver(kind)
    sgd.cur_itrs = 3
    for fresh in (sgd.state_dict(), _driver(kind)[0].state_dict()):         # with and without momentum state
        with pytest.raises(ValueError, match="SGD"):
            _driver(kind, optimizer="adam")[0].load_state_dict(fresh)


def _fill_any(st, kind, step):
    """State as after ``step`` iterations, for either optimiser kind: random buffers, step counts, Philox offsets."""
    st.cur_itrs = step
    for i, m in enumerate(st._networks):
        m._philox_offset = 8 * (step + i)
    for _, _, s in st._trained:
        s.step = step
        for b in s.bufs:
            b.uniform_(0, 1)
    if kind == "hpfg":
        for p in st._neck_params(st.m2):
            st._neck_states[id(p)] = OptState([torch.rand_like(p) for _ in st._opt.KEYS], step)


def _snapshot(st):
    states = [s for _, _, s in st._trained] + list(st._neck_states.values())
    return ((st.cur_itrs, [m._philox_offset for m in st._networks], sorted(st._neck_states), [s.step for s in states]),
            [b.clone() for s in states for b in s.bufs])


@pytest.mark.parametrize("name", ["sgd", "adamw"])
@pytest.mark.parametrize("kind", ["mt", "hpfg"])
def test_rejected_load_changes_nothing(kind, name):
    """load_state_dict checks the whole checkpoint before it changes anything: a checkpoint of the other optimiser kind, or
    one whose last network's U-Net tensors carry different Adam step counts, leaves cur_itrs, the Philox offsets, every
    optimiser buffer and every step count as they were."""
    st, _ = _driver(kind, optimizer=name)
    _fill_any(st, kind, 7)
    other, _ = _driver(kind, optimizer="adamw" if name == "sgd" else "sgd")
    _fill_any(other, kind, 9)
    bad = [(other.state_dict(), "Adam" if name == "sgd" else "SGD")]
    if name == "adamw":
        same, _ = _driver(kind, optimizer=name)
        _fill_any(same, kind, 9)
        sd = same.state_dict()
        sd["optimizers"][-1]["state"][5]["step"] = torch.tensor(6.0)
        bad.append((sd, "step count"))
    before = _snapshot(st)
    for sd, match in bad:
        with pytest.raises(ValueError, match=match):
            st.load_state_dict(sd)
        after = _snapshot(st)
        assert after[0] == before[0] and len(after[1]) == len(before[1])
        assert all(torch.equal(a, b) for a, b in zip(after[1], before[1]))
