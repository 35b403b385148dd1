"""CPU: the C-ABI library loads and exports every declared symbol, layout queries agree with the oracle's
parameter spec, the nn.Module mirrors the reference's state_dict, and the no-fallback rule holds."""
import copy
import ctypes
import os
import re

import pytest
import torch

import oracle
import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from hpfg_b200.optim import OptState

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "hpfg_b200.h")).read()
    declared = set(re.findall(r"\b(hpfg_[a-z0-9_]+)\s*\(", header))
    assert declared == set(L.SIGNATURES), declared ^ set(L.SIGNATURES)
    lib = L.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.hpfg_version() >= 100


@pytest.mark.parametrize("in_ch,n_cls", [(1, 4), (3, 2)])
def test_layout_queries_match_oracle_spec(in_ch, n_cls):
    lib = L.lib()
    offs, sizes, tot = (ctypes.c_int64 * 82)(), (ctypes.c_int64 * 82)(), ctypes.c_int64()
    L.check(lib.hpfg_unet_param_layout(in_ch, n_cls, offs, sizes, ctypes.byref(tot)))
    spec = oracle.unet_param_spec(in_ch, n_cls)
    exp_sizes = [int(torch.Size(s).numel()) for _, s in spec]
    assert list(sizes) == exp_sizes and tot.value == sum(exp_sizes)
    assert list(offs) == [sum(exp_sizes[:i]) for i in range(82)]
    boffs, bch, btot = (ctypes.c_int64 * 18)(), (ctypes.c_int64 * 18)(), ctypes.c_int64()
    L.check(lib.hpfg_unet_bn_layout(in_ch, n_cls, boffs, bch, ctypes.byref(btot)))
    chans = [s[0] for n, s, _ in oracle.unet_buffer_spec(in_ch, n_cls) if n.endswith("running_mean")]
    assert list(bch) == chans and btot.value == 2 * sum(chans)


def test_module_mirrors_reference_state_dict_and_survives_copies():
    torch.manual_seed(3)
    m = hb.build_model(type("A", (), dict(model="unet", in_channels=3, num_classes=2))())
    assert isinstance(m, hb.UNet) and isinstance(m, torch.nn.Module)
    assert [(n, tuple(p.shape)) for n, p in m.named_parameters()] == oracle.unet_param_spec(3, 2)
    bufs = [n for n, _ in m.named_buffers()]
    assert bufs == [n for n, _, _ in oracle.unet_buffer_spec(3, 2)]
    assert len(m.state_dict()) == 136
    assert m._is_flat()
    m2 = copy.deepcopy(m)
    assert m2._is_flat() and m2.flat_params.data_ptr() != m.flat_params.data_ptr()
    assert torch.equal(m2.flat_params, m.flat_params)
    for _, p in m2.named_parameters():
        p.requires_grad = False                      # what the MT trainer does to the teacher (:56-57)
    m.load_state_dict(copy.deepcopy(m.state_dict()))
    assert m._is_flat()
    opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
    assert len(opt.param_groups[0]["params"]) == 82
    with pytest.raises(NotImplementedError):
        hb.build_model(type("A", (), dict(model="swinunet", in_channels=1, num_classes=4))())


def test_no_cpu_fallback():
    m = hb.UNet(1, 4)
    with pytest.raises(L.HpfgError):
        m(torch.zeros(1, 1, 32, 32))
    with pytest.raises(L.HpfgError):
        hb.Med_Sup_Loss(4)(torch.zeros(1, 4, 16, 16, requires_grad=True), torch.zeros(1, 16, 16, dtype=torch.long))
    with pytest.raises(L.HpfgError):
        hb.update_ema_variables(m, copy.deepcopy(m), 0.99, 1)
    with pytest.raises(AssertionError):
        hb.DiceLoss(4)(torch.zeros(1, 4, 16, 16), torch.zeros(1, 1, 8, 8))
    # argument validation happens before any device work
    assert L.lib().hpfg_ema_update(None, None, 4, 0.5, None) == 1
    assert b"null" in L.lib().hpfg_last_error()


def test_host_schedules_match_oracle():
    for it in (1, 2, 3, 149, 150, 4000, 30000):
        assert hb.medical_lr(it, 0.01, 30000) == pytest.approx(oracle.medical_lr(it - 1), rel=1e-14)
    a = type("A", (), dict(consistency=0.1, consistency_rampup=200.0))()
    for it in (1, 150, 1500, 40000):
        assert hb.get_current_consistency_weight(it // 150, a) == pytest.approx(oracle.consistency_weight(it), rel=1e-14)


def test_python_constants_match_the_header():
    header = open(os.path.join(ROOT, "include", "hpfg_b200.h")).read()
    defs = dict(re.findall(r"#define\s+(HPFG_[A-Z0-9_]+)\s+(\d+)", header))
    for name in ("SUP", "MT", "CPS", "UAMT", "ICT", "S4CV"):
        assert int(defs["HPFG_LOSS_" + name]) == getattr(L, "LOSS_" + name), name
    assert int(defs["HPFG_PREC_FP32"]) == L.PREC_FP32 and int(defs["HPFG_PREC_BF16"]) == L.PREC_BF16
    assert int(defs["HPFG_NUM_BN"]) == L.NUM_BN and int(defs["HPFG_NUM_DROPOUT"]) == L.NUM_DROPOUT


def test_unet_plus_mirrors_reference_structure():
    """UNet_Plus (model/unet.py:178-206): 82 flat U-Net parameters + 16 neck parameters in the reference's order; the
    necks stay ordinary torch parameters, deepcopy / load_state_dict keep the flat views intact."""
    torch.manual_seed(4)
    m = hb.build_model(type("A", (), dict(model="unet_plus", in_channels=1, num_classes=4))())
    assert isinstance(m, hb.UNet_Plus)
    names = [n for n, _ in m.named_parameters()]
    spec = oracle.unet_param_spec(1, 4) + oracle.unet_plus_neck_spec(4)
    assert [(n, tuple(p.shape)) for n, p in m.named_parameters()] == spec and len(names) == 98
    assert m._is_flat() and len(m._flat_params_list) == 82
    m2 = copy.deepcopy(m)
    assert m2._is_flat() and m2.dense_projection_high.mlp[0].weight.data_ptr() != m.dense_projection_high.mlp[0].weight.data_ptr()
    m2.load_state_dict(m.state_dict())
    assert m2._is_flat() and all(torch.equal(a, b) for a, b in zip(m.parameters(), m2.parameters()))
    with pytest.raises(L.HpfgError):
        m(torch.zeros(1, 1, 32, 32))                      # CPU tensor: no fallback
    with pytest.raises(NotImplementedError):
        hb.build_model(type("A", (), dict(model="swinunet_plus", in_channels=1, num_classes=4))())


def test_graph_replay_policy_host_logic():
    """Which steps replay a CUDA graph is pure host logic: never the first iteration; under data parallelism only when asked
    to capture the NCCL bucket all-reduces with the step (a refused capture falls back to eager launches at run time)."""
    a, b = hb.UNet(1, 4), hb.UNet(1, 4)
    mt, cps, ict = hb.MeanTeacherStep(a, copy.deepcopy(a)), hb.CPSStep(a, b), hb.ICTStep(a, b)
    uamt = hb.UAMTStep(a, copy.deepcopy(a))
    for st in (mt, cps, uamt, ict):
        assert not st._use_graph()
        st.enable_graph(True)
        st.cur_itrs = 1
        assert not st._use_graph()
        st.cur_itrs = 2
        assert st._use_graph()
        st.world = 2
        assert not st._use_graph()                       # data parallel stays eager unless asked
        st.enable_graph(True, data_parallel=True)
    assert mt._use_graph() and cps._use_graph() and uamt._use_graph() and ict._use_graph()
    mt.enable_graph(False)
    assert not mt._use_graph()
    assert mt._dyn_scalars(0.99)[0] == pytest.approx(hb.medical_lr(2, 0.01, 30000))
    s4cv = hb.S4CVStep(a, b, copy.deepcopy(b))           # eager launches only
    s4cv.enable_graph(True, data_parallel=True)
    for it in (1, 2, 3):
        s4cv.cur_itrs = it
        assert not s4cv._use_graph()


def _step_driver(kind):
    torch.manual_seed(5)
    if kind == "hpfg":
        m1, m2 = hb.UNet_Plus(1, 4), hb.UNet_Plus(1, 4)
        nets = (m1, m2, copy.deepcopy(m2))
    else:
        a, b = hb.UNet(1, 4), hb.UNet(1, 4)
        nets = (a, b, copy.deepcopy(b)) if kind == "s4cv" else (a, b) if kind == "cps" else (a, copy.deepcopy(a))
    cls = dict(mt=hb.MeanTeacherStep, cps=hb.CPSStep, uamt=hb.UAMTStep, ict=hb.ICTStep, s4cv=hb.S4CVStep, hpfg=hb.HPFGStep)[kind]
    return cls(*nets), nets


# Checkpoint layout of each driver: the networks whose Philox offsets it saves (constructor positions, in order) and, per
# optimizer entry, the momentum buffer attribute and the number of parameters of its network.
CHECKPOINT_LAYOUT = {
    "mt": ([0, 1], [("mom", 82)]),
    "cps": ([0, 1], [("b1", 82), ("b2", 82)]),
    "uamt": ([0, 1], [("mom", 82)]),
    "ict": ([0, 1], [("mom", 82)]),
    "s4cv": ([0, 1, 2], [("b1", 82), ("b2", 82)]),
    "hpfg": ([0, 1, 2], [("b1", 98), ("b2", 98)]),
}


@pytest.mark.parametrize("kind", sorted(CHECKPOINT_LAYOUT))
def test_step_driver_sgd_checkpoint_layout_and_roundtrip(kind):
    """state_dict() of every step driver: Philox offsets of its networks in a fixed order, one torch.optim.SGD-style entry per
    trained network (lr of the next iteration, per-parameter momentum in parameters() order), and it round-trips."""
    philox_of, opts = CHECKPOINT_LAYOUT[kind]
    st, nets = _step_driver(kind)
    assert all(opt["state"] == {} for opt in st.state_dict()["optimizers"])       # no momentum before the first step
    for i, m in enumerate(nets):
        m._philox_offset = 8 * (i + 1)
    st.cur_itrs = 7
    for name, _ in opts:
        getattr(st, name).uniform_(-1, 1)
    if kind == "hpfg":
        for p in st._neck_params(nets[1]):
            st._neck_states[id(p)] = OptState([torch.randn_like(p)], 7)
    sd = st.state_dict()
    assert sd["cur_itrs"] == 7 and sd["philox"] == [8 * (i + 1) for i in philox_of]
    assert len(sd["optimizers"]) == len(opts)
    for opt, (name, n_params) in zip(sd["optimizers"], opts):
        assert opt["param_groups"] == [{"lr": 0.00999819998199868, "momentum": 0.9, "weight_decay": 1e-4,
                                        "params": list(range(n_params))}]
        assert sorted(opt["state"]) == list(range(98 if kind == "hpfg" and name == "b2" else 82))
        flat = torch.cat([opt["state"][i]["momentum_buffer"].reshape(-1) for i in range(82)])
        assert torch.equal(flat, getattr(st, name))
    st2, nets2 = _step_driver(kind)
    st2.load_state_dict(sd)
    assert [m._philox_offset for m in nets2] == [8 * (i + 1) if i in philox_of else 0 for i in range(len(nets2))]
    sd2 = st2.state_dict()
    assert sd2["cur_itrs"] == 7 and sd2["philox"] == sd["philox"]
    for o, o2 in zip(sd["optimizers"], sd2["optimizers"]):
        assert o2["param_groups"] == o["param_groups"] and sorted(o2["state"]) == sorted(o["state"])
        assert all(torch.equal(o2["state"][i]["momentum_buffer"], o["state"][i]["momentum_buffer"]) for i in o["state"])


def test_necks_and_dense_loss_have_no_cpu_path():
    """The projection necks and Dense_Loss run on the library's kernels (csrc/neck.cu): the modules keep the reference's
    parameter names / shapes, and CPU tensors raise instead of falling back to torch (parity with the oracle: GPU tests)."""
    torch.manual_seed(8)
    m = hb.UNet_Plus(1, 4)
    assert [(n, tuple(p.shape)) for n, p in m.named_parameters()][82:] == oracle.unet_plus_neck_spec(4)
    with pytest.raises(L.HpfgError):
        m.dense_projection_high(torch.randn(3, 256, 4, 4))
    with pytest.raises(L.HpfgError):
        hb.projection_conv(4, hid_dim=8, s=0)(torch.randn(1, 4, 8, 8))
    x = (torch.randn(3, 128), torch.randn(3, 128, 16))
    y = (torch.randn(3, 128), torch.randn(3, 128, 16))
    with pytest.raises(L.HpfgError):
        hb.Dense_Loss(batch_size=3)(x, y)
    with pytest.raises(RuntimeError):
        hb.Dense_Loss(batch_size=5)(x, y)                  # the reference's mask is built for the constructor's batch size


def test_hpfg_step_checkpoint_carries_neck_state():
    """HPFGStep.state_dict(): torch.optim.SGD layout over all 98 parameters of each UNet_Plus -- the flat U-Net momentum at
    indices 0..81, the neck tensors' buffers at 82..97 (only for tensors that have seen a gradient) -- and it round-trips."""
    torch.manual_seed(9)
    m1, m2 = hb.UNet_Plus(1, 4), hb.UNet_Plus(1, 4)
    st = hb.HPFGStep(m1, m2, copy.deepcopy(m2))
    st.cur_itrs = 7
    st.b1.uniform_(-1, 1)
    st.b2.uniform_(-1, 1)
    necks2 = st._neck_params(m2)
    assert len(necks2) == 16 and [tuple(p.shape) for p in necks2] == [s for _, s in oracle.unet_plus_neck_spec(4)]
    for p in necks2:
        st._neck_states[id(p)] = OptState([torch.randn_like(p)], 7)
    sd = st.state_dict()
    assert sd["cur_itrs"] == 7 and len(sd["optimizers"]) == 2
    o1, o2 = sd["optimizers"]
    assert o1["param_groups"][0]["params"] == list(range(98)) and sorted(o1["state"]) == list(range(82))      # model1's necks: no state
    assert sorted(o2["state"]) == list(range(98))
    ref = torch.optim.SGD(m2.parameters(), lr=0.01, momentum=0.9)
    ref.load_state_dict({"state": o2["state"], "param_groups": [dict(ref.state_dict()["param_groups"][0], **o2["param_groups"][0])]})
    n1, n2 = hb.UNet_Plus(1, 4), hb.UNet_Plus(1, 4)
    st2 = hb.HPFGStep(n1, n2, copy.deepcopy(n2))
    st2.load_state_dict(sd)
    assert st2.cur_itrs == 7 and torch.equal(st2.b1, st.b1) and torch.equal(st2.b2, st.b2)
    for p, q in zip(necks2, st2._neck_params(n2)):
        assert torch.equal(st2._neck_states[id(q)].bufs[0], st._neck_states[id(p)].bufs[0])
    assert not any(id(q) in st2._neck_states for q in st2._neck_params(n1))


def test_oracle_is_test_infrastructure_only():
    """oracle/ may be imported by tests/, __graft_entry__.smoke() and bench.py's CPU legs only: nothing under hpfg_b200/
    (Python or CUDA) refers to it, and importing the package does not pull it in."""
    import re
    import subprocess
    import sys
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "hpfg_b200")
    pat = re.compile(r"^\s*(import|from)\s+oracle\b|oracle/", re.M)
    for root, _, files in os.walk(pkg):
        if "build" in root.split(os.sep):
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                assert not pat.search(open(os.path.join(root, f)).read()), os.path.join(root, f)
    code = "import sys, hpfg_b200; assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules), 'oracle imported'"
    assert subprocess.run([sys.executable, "-c", code], cwd=os.path.dirname(pkg)).returncode == 0
