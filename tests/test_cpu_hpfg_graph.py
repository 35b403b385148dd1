"""CPU: the host side of HPFGStep's graph replay and of the CutMix loss mode -- the C constant, the batch-size check, the
replay policy and the device block of per-iteration scalars (the kernels and the replay itself: tests/test_gpu_hpfg_graph.py)."""
import copy
import os
import re

import pytest
import torch

import hpfg_b200 as hb
from hpfg_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _driver(**kw):
    torch.manual_seed(5)
    m1, m2 = hb.UNet_Plus(1, 4), hb.UNet_Plus(1, 4)
    return hb.HPFGStep(m1, m2, copy.deepcopy(m2), **kw), (m1, m2)


def test_cutmix_mode_constant_matches_header():
    text = open(os.path.join(ROOT, "include", "hpfg_b200.h")).read()
    assert int(re.search(r"#define HPFG_LOSS_CUTMIX (\d+)", text).group(1)) == L.LOSS_CUTMIX == 6


def test_unlabeled_batch_must_be_a_multiple_of_the_second_labeled_draw():
    import ctypes
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)           # (rejected before any device access)
    assert L.lib().hpfg_cutmix_loss(p, p, p, p, p, 2, 6, 4, 4, 8, 8, 1.0, None, None, 0.5, 0.5, p, p, None, p, None) == 1
    assert b"multiple of n_l1" in L.lib().hpfg_last_error()
    with pytest.raises(ValueError):
        hb.losses.check_cutmix_batch(6, 4)
    hb.losses.check_cutmix_batch(6, 3)
    st, _ = _driver()
    x = torch.zeros(2, 1, 32, 32)
    y = torch.zeros(2, 32, 32, dtype=torch.int64)
    with pytest.raises(ValueError):          # raised before anything changes
        st.step(x, y, torch.zeros(4, 1, 32, 32), torch.zeros(4, 32, 32, dtype=torch.int64), torch.zeros(6, 1, 32, 32),
                torch.zeros(6, 1, 32, 32))
    assert st.cur_itrs == 0


def _neck_states(st, m2, step):
    for p in st._neck_params(m2):
        st._neck_states[id(p)] = st._opt.new_state(p.data)
        st._neck_states[id(p)].step = step


def _set_steps(st, step):
    for _, _, s in st._trained:
        s.step = step


def test_hpfg_step_replays_only_after_its_first_update():
    st, (m1, m2) = _driver()
    assert not st._use_graph()
    st.enable_graph(True)
    st.cur_itrs = 147                 # a hand-set iteration count: the first step() still launches eagerly
    _set_steps(st, 1)
    _neck_states(st, m2, 1)
    assert not st._use_graph()
    st._stepped = True
    assert not st._use_graph()        # every state is at its first update (SGD initialises its momentum then)
    _set_steps(st, 2)
    assert not st._use_graph()        # the neck states too
    _neck_states(st, m2, 2)
    assert st._use_graph()
    del st._neck_states[id(st._neck_params(m2)[5])]
    assert not st._use_graph()        # a neck tensor without state
    _neck_states(st, m2, 2)
    st._stepped = False
    assert not st._use_graph()        # a fresh driver's first step (e.g. after load_state_dict) is eager
    st._stepped = True
    st.world = 2
    assert not st._use_graph()        # data parallel stays eager unless asked
    st.enable_graph(True, data_parallel=True)
    assert st._use_graph()
    st.exact_global = True
    assert not st._use_graph()
    st.exact_global = False
    st.enable_graph(False)
    assert not st._use_graph()


@pytest.mark.parametrize("name", ["adam", "adamw"])
def test_hpfg_device_block_has_a_group_per_neck_state(name):
    st, (m1, m2) = _driver(optimizer=name, consistency_rampup=2.0, mt_start=150)
    st.cur_itrs = 300
    _set_steps(st, 300)
    necks = st._neck_params(m2)
    for j, p in enumerate(necks):
        st._neck_states[id(p)] = st._opt.new_state(p.data)
        st._neck_states[id(p)].step = 2 + j
    w = st._consistency_weight()
    assert w == pytest.approx(0.1)
    block = st._dyn_scalars(st.ema_decay, st._mt_weight(), 7.0 * w, 0.5 * w)
    lr = hb.medical_lr(300, 0.01, 30000)
    alpha = min(1 - 1 / 301, 0.99)
    assert block[:4] == [lr, alpha, float(1.0 - torch.tensor(alpha, dtype=torch.float32)), w]
    assert block[4:7] == [w, 7.0 * w, 0.5 * w]
    assert len(block) == 7 + 5 * (2 + 16)
    states = [s for _, _, s in st._trained] + [st._neck_states[id(p)] for p in necks]
    assert [s.dv_offset for s in states] == [7 + 5 * k for k in range(18)]
    for s in states:
        assert block[s.dv_offset:s.dv_offset + 5] == st._opt.scalars(s.step, lr) + block[1:3]
    st.cur_itrs = 149
    assert st._mt_weight() == 0.0     # model2's Mean-Teacher term is off before mt_start


def test_other_drivers_device_block_is_unchanged_by_neck_groups():
    a, b = hb.UNet(1, 4), hb.UNet(1, 4)
    cps = hb.CPSStep(a, b, optimizer="adam")
    cps.cur_itrs = 3
    _set_steps(cps, 3)
    assert len(cps._dyn_scalars()) == 4 + 2 * 5 and not cps._neck_states
