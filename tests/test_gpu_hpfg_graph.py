"""GPU (B200): the CutMix loss mode, the CutMix input mix, the scaled contrastive gradient and the device-block EMA against
torch, and HPFGStep's graph replay against its eager launches, bit for bit."""
import copy
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp
import torch.nn.functional as F

import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from tests.golden.common import make_hpfg_batch
from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ---------------------------------------------------------------------------------------------------------------- kernels
def _dice64(p, target, n_cls):
    """DiceLoss (utils/loss/diceloss.py:155-191) in fp64: class c <=> target == c (the reference's one-hot on a float map)."""
    loss = 0.0
    for c in range(n_cls):
        t = (target == c).double()
        inter, y, z = (p[:, c] * t).sum(), (t * t).sum(), (p[:, c] * p[:, c]).sum()
        loss = loss + 1 - (2 * inter + 1e-5) / (z + y + 1e-5)
    return loss / n_cls


def _reference(s, t, y, y1, m, n_l, pw):
    """main.py:125-134,143 transcribed: fp32 pseudo-labels exactly as main.py forms them, the loss in fp64."""
    n_u, n_cls = s.shape[0] - n_l, s.shape[1]
    y1r = y1.repeat(n_u // y1.shape[0], 1, 1)
    mm = m.reshape(n_u, *s.shape[2:]).float()
    pseudo = y1r * (1.0 - mm) + torch.argmax(torch.softmax(t, dim=1), dim=1) * mm          # float32, main.py:132-133
    s64 = s.double().requires_grad_(True)
    p = torch.softmax(s64, dim=1)
    sup = 0.5 * F.cross_entropy(s64[:n_l], y, ignore_index=255) + 0.5 * _dice64(p[:n_l], y, n_cls)
    pd = _dice64(p[n_l:], pseudo, n_cls)
    loss = sup + pw * pd
    loss.backward()
    labels = torch.full_like(y1r, 255)
    for c in range(n_cls):
        labels[pseudo == c] = c
    return loss.item(), sup.item(), pd.item(), s64.grad, labels


def _inputs(n_cls, n_l, n_u, n_l1, h, w, seed, fractional):
    g = torch.Generator().manual_seed(seed)
    s = torch.randn(n_l + n_u, n_cls, h, w, generator=g) * 2
    # teacher logits with a margin between classes, so that torch's softmax and the kernel's pick the same maximum
    t = torch.randint(-6, 7, (n_u, n_cls, h, w), generator=g).float() + torch.arange(n_cls).view(1, -1, 1, 1) * 0.05
    y = torch.randint(0, n_cls, (n_l, h, w), generator=g)
    y1 = torch.randint(0, n_cls, (n_l1, h, w), generator=g)
    y[:, :3] = 255
    y1[:, :, :5] = 255
    if fractional:
        m = torch.randint(0, 5, (n_u, 1, h, w), generator=g).float() / 4
    else:
        m = (torch.rand(n_u, 1, h, w, generator=g) > 0.5).float()
    return [x.to(DEV) for x in (s, t, y, y1, m)]


@pytest.mark.parametrize("n_cls,fractional", [(c, False) for c in range(2, 9)] + [(3, True), (4, True), (8, True)])
def test_cutmix_loss_mode_matches_main_py(n_cls, fractional):
    n_l, n_u, n_l1, h, w, pw = 2, 6, 2, 32, 48, 0.35
    s, t, y, y1, m = _inputs(n_cls, n_l, n_u, n_l1, h, w, 40 + n_cls, fractional)
    r = hb.cutmix_loss_raw(s, t, y, y1, m, n_l, pseudo_weight=pw, want_pseudo=True)
    loss, sup, pd, grad, labels = _reference(s, t, y, y1, m, n_l, pw)
    sc = r["scalars"].cpu()
    assert abs(sc[0].item() - loss) <= 1e-5 * abs(loss), (sc[0].item(), loss)
    assert abs(sc[1].item() - sup) <= 1e-5 * abs(sup)
    assert abs(sc[2].item() - pd) <= 1e-5 * abs(pd)
    assert sc[6].item() == 0 and sc[7].item() == 0
    assert rel_l2(r["dstudent"], grad) < 1e-5
    assert torch.equal(r["pseudo"], labels)
    if not fractional:       # 0/1 masks: the torch.where form over argmax_labels
        want = torch.where(m.squeeze(1) > 0.5, hb.argmax_labels(t), y1.repeat(n_u // n_l1, 1, 1))
        assert torch.equal(r["pseudo"], want)
    # a weight read from device memory gives the same bits as the same weight by value
    rd = hb.cutmix_loss_raw(s, t, y, y1, m, n_l, pseudo_weight=0.0,
                            pseudo_weight_dev=torch.tensor([pw], device=DEV, dtype=torch.float32))
    assert torch.equal(rd["scalars"], r["scalars"]) and torch.equal(rd["dstudent"], r["dstudent"])


def test_cutmix_pseudo_labels_are_argmax_labels_on_any_logits():
    """Random logits (near-ties included): the kernel's argmax is hpfg_argmax_labels' argmax."""
    n_l, n_u, h, w = 1, 4, 32, 32
    g = torch.Generator().manual_seed(3)
    s = torch.randn(n_l + n_u, 4, h, w, generator=g).to(DEV)
    t = torch.randn(n_u, 4, h, w, generator=g).to(DEV)
    y = torch.randint(0, 4, (n_l, h, w), generator=g).to(DEV)
    y1 = torch.randint(0, 4, (1, h, w), generator=g).to(DEV)
    m = torch.ones(n_u, 1, h, w, device=DEV)
    r = hb.cutmix_loss_raw(s, t, y, y1, m, n_l, pseudo_weight=1.0, want_pseudo=True)
    assert torch.equal(r["pseudo"], hb.argmax_labels(t))


def test_cutmix_loss_autograd_wrapper_and_batch_check():
    n_l, n_u = 2, 4
    s, t, y, y1, m = _inputs(4, n_l, n_u, 2, 32, 32, 7, False)
    s = s.clone().requires_grad_(True)
    loss = hb.cutmix_pseudo_loss(s, t, y, y1, m, 0.7)
    loss.backward()
    r = hb.cutmix_loss_raw(s.detach(), t, y, y1, m, n_l, pseudo_weight=0.7)
    assert torch.equal(loss.detach(), r["scalars"][0]) and torch.equal(s.grad, r["dstudent"])
    with pytest.raises(ValueError):
        hb.cutmix_loss_raw(s.detach(), t, y, y1[:1].repeat(3, 1, 1), m, n_l, pseudo_weight=0.7)
    with pytest.raises(ValueError):
        hb.cutmix_mix_inputs(torch.rand(3, 1, 32, 32, device=DEV), torch.rand(4, 1, 32, 32, device=DEV), m)


@pytest.mark.parametrize("ch", [1, 3])
def test_cutmix_mix_is_bit_identical_to_torch(ch):
    g = torch.Generator().manual_seed(ch)
    a = torch.rand(2, ch, 40, 36, generator=g).to(DEV)
    b = torch.rand(6, ch, 40, 36, generator=g).to(DEV)
    for m in ((torch.rand(6, 1, 40, 36, generator=g) > 0.5).float(), torch.rand(6, 1, 40, 36, generator=g)):
        m = m.to(DEV)
        want = a.repeat(3, 1, 1, 1) * (1.0 - m) + b * m                # main.py:139,145
        assert torch.equal(hb.cutmix_mix_inputs(a, b, m), want)


@pytest.mark.parametrize("positions", [1, 16])
def test_scaled_contrastive_gradient_is_scale_times_unscaled(positions):
    g = torch.Generator().manual_seed(positions)
    batch, dim = 12, 128
    a = torch.randn(batch, dim, positions, generator=g).to(DEV)
    b = torch.randn(batch, dim, positions, generator=g).to(DEV)
    lib = L.lib()
    ws = torch.empty(lib.hpfg_dense_contrastive_workspace_floats(batch, dim, positions), device=DEV)
    loss0, loss1, loss2 = (torch.empty(1, device=DEV) for _ in range(3))
    d0, d1, d2 = (torch.empty_like(a) for _ in range(3))
    st = L.stream_ptr(a.device)
    L.check(lib.hpfg_dense_contrastive(L.ptr(a), L.ptr(b), batch, dim, positions, 0.7, L.ptr(loss0), L.ptr(d0), L.ptr(ws), st))
    scale = 0.5 * 0.037
    L.check(lib.hpfg_dense_contrastive_scaled(L.ptr(a), L.ptr(b), batch, dim, positions, 0.7, scale, None, L.ptr(loss1),
                                              L.ptr(d1), L.ptr(ws), st))
    dev_scale = torch.tensor([scale], device=DEV, dtype=torch.float32)
    L.check(lib.hpfg_dense_contrastive_scaled(L.ptr(a), L.ptr(b), batch, dim, positions, 0.7, 0.0, L.ptr(dev_scale),
                                              L.ptr(loss2), L.ptr(d2), L.ptr(ws), st))
    assert torch.equal(loss1, loss0) and torch.equal(loss2, loss0)
    assert torch.equal(d1, scale * d0) and torch.equal(d2, d1)


def test_ema_update_dv_is_bit_identical_to_by_value():
    g = torch.Generator().manual_seed(2)
    p = torch.randn(1000003, generator=g).to(DEV)
    e = torch.randn(1000003, generator=g).to(DEV)
    alpha = min(1 - 1 / 152, 0.99)
    e1, e2 = e.clone(), e.clone()
    hb.ema_update_flat(e1, p, alpha)
    a32 = torch.tensor(alpha, dtype=torch.float32)
    block = torch.tensor([float(a32), float(1.0 - a32)], device=DEV)
    L.check(L.lib().hpfg_ema_update_dv(L.ptr(e2), L.ptr(p), e2.numel(), L.ptr(block), L.stream_ptr(e2.device)))
    assert torch.equal(e1, e2)


# ---------------------------------------------------------------------------------------------- replay against eager
N_L, N_U, HW = 2, 4, 64


def _nets(seed=23):
    torch.manual_seed(seed)
    m1 = hb.UNet_Plus(1, 4, precision="bf16").to(DEV)
    m2 = hb.UNet_Plus(1, 4, precision="bf16").to(DEV)
    return m1, m2, copy.deepcopy(m2)


def _driver(nets, optimizer, graph):
    step = hb.HPFGStep(*nets, optimizer=optimizer, total_itrs=300, mt_start=150, consistency_rampup=2)
    step.cur_itrs = 147                     # w: 0 for 148, 149, 0.05 from 150 on, where model2's Mean-Teacher term starts
    step.enable_graph(graph)
    return step


def _batches(k):
    return [[t.to(DEV) for t in make_hpfg_batch(N_L, N_U, 1, 4, HW, HW, 300 + 7 * i)] for i in range(k)]


def _snapshot(nets, step):
    state = [{k: v.detach().clone() for k, v in m.state_dict().items()} for m in nets]
    return state, copy.deepcopy(step.state_dict())


def _last(step):
    return [step.last[k].item() for k in ("loss", "loss_sup", "contrast", "pseudo", "cons2")] + [step.last["lr"], step.last["w"]]


def _assert_same(a, b):
    (sa, da), (sb, db) = a, b
    for ma, mb in zip(sa, sb):
        for k in ma:
            assert torch.equal(ma[k], mb[k]), k
    assert da["cur_itrs"] == db["cur_itrs"] and da["philox"] == db["philox"]
    for oa, ob in zip(da["optimizers"], db["optimizers"]):
        assert sorted(oa["state"]) == sorted(ob["state"]) and oa["param_groups"] == ob["param_groups"]
        for i in oa["state"]:
            for k in oa["state"][i]:
                assert torch.equal(oa["state"][i][k], ob["state"][i][k]), (i, k)


def _run(optimizer, graph, steps=6):
    nets = _nets()
    step = _driver(nets, optimizer, graph)
    losses, lasts, counts = [], [], []
    for b in _batches(steps):
        counts.append(L.lib().hpfg_launch_count())
        losses.append(step.step(*b).item())
        lasts.append(_last(step))
    torch.cuda.synchronize()
    return losses, lasts, counts, _snapshot(nets, step), step, nets


@pytest.mark.parametrize("optimizer", ["sgd", "adamw"])
def test_hpfg_graph_replay_matches_eager(optimizer):
    l0, s0, _, snap0, _, _ = _run(optimizer, False)
    l1, s1, counts, snap1, step, nets = _run(optimizer, True)
    assert l0 == l1, (l0, l1)
    assert s0 == s1
    assert s1[0][-1] == 0.0 and s1[-1][-1] == 0.05       # w moved from 0 to 0.05 inside the run
    _assert_same(snap0, snap1)
    assert step.kernels_per_replay > 0
    assert counts[3] == counts[4] == counts[5]          # replayed steps launch nothing through the library
    m1, m2, _ = nets
    assert all(p.grad is not None for p in m2.parameters())
    assert all(p.grad is None for p in step._neck_params(m1))
    assert all(p.grad is not None for p in m1._flat_params_list)


def _run_async(graph, steps=24):
    nets = _nets(29)
    step = _driver(nets, "sgd", graph)
    batches = _batches(3)
    spin = torch.empty(64 << 20, device=DEV)
    torch.cuda.synchronize()
    losses = torch.zeros(steps, device=DEV)
    for _ in range(6):
        spin.add_(1.0)                              # queue device work first so the enqueue loop really runs ahead
    for i in range(steps):
        losses[i:i + 1].copy_(step.step(*batches[i % 3]).reshape(1))
    torch.cuda.synchronize()
    return losses.cpu(), _snapshot(nets, step)


def test_hpfg_graph_replay_matches_eager_without_per_step_sync():
    l0, s0 = _run_async(False)
    l1, s1 = _run_async(True)
    assert torch.equal(l0, l1), (l0, l1)
    _assert_same(s0, s1)


def test_hpfg_resume_under_replay_is_bit_exact():
    batches = _batches(6)
    nets = _nets()
    step = _driver(nets, "sgd", True)
    ref = [step.step(*b).item() for b in batches]
    want = _snapshot(nets, step)
    nets = _nets()
    step = _driver(nets, "sgd", True)
    got = [step.step(*b).item() for b in batches[:3]]
    ck = copy.deepcopy({"nets": [m.state_dict() for m in nets], "step": step.state_dict()})
    nets2 = _nets(99)
    torch.manual_seed(23)           # the dropout Philox seed is the generator's: a resumed run keeps the run's seed
    for m, sd in zip(nets2, ck["nets"]):
        m.load_state_dict(sd)
    step2 = hb.HPFGStep(*nets2, total_itrs=300, mt_start=150, consistency_rampup=2)
    step2.load_state_dict(ck["step"])
    step2.enable_graph(True)
    got += [step2.step(*b).item() for b in batches[3:]]
    torch.cuda.synchronize()
    assert got == ref, (got, ref)
    assert step2.kernels_per_replay > 0
    _assert_same(want, _snapshot(nets2, step2))


def _run_assign(graph):
    nets = _nets(31)
    step = _driver(nets, "sgd", graph)
    batches = _batches(6)
    losses, graphs = [], []
    for i, b in enumerate(batches):
        if i == 3:
            sd = {k: v.detach().clone() for k, v in nets[1].state_dict().items()}
            nets[1].load_state_dict(sd, assign=True)
        losses.append(step.step(*b).item())
        graphs.append(getattr(step, "_ggraph", None))
    torch.cuda.synchronize()
    return losses, graphs, _snapshot(nets, step)


def test_hpfg_load_state_dict_assign_captures_again():
    l0, _, s0 = _run_assign(False)
    l1, graphs, s1 = _run_assign(True)
    assert l0 == l1, (l0, l1)
    _assert_same(s0, s1)
    assert graphs[2] is not None and graphs[5] is not None and graphs[5] is not graphs[2]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, graph, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.manual_seed(23 + rank)             # different replicas: the driver broadcasts rank 0's
    nets = [hb.UNet_Plus(1, 4, precision="bf16").to(dev) for _ in range(2)]
    nets.append(copy.deepcopy(nets[1]))
    step = hb.HPFGStep(*nets, total_itrs=300, mt_start=150, consistency_rampup=2)
    step.cur_itrs = 147
    step.enable_graph(graph, data_parallel=True)
    losses = []
    for i in range(5):
        x_l, y, x_l1, y1, x_u, m = make_hpfg_batch(2 * world, 4 * world, 1, 4, HW, HW, 500 + i)
        sl, su = slice(2 * rank, 2 * rank + 2), slice(4 * rank, 4 * rank + 4)
        losses.append(step.step(x_l[sl].to(dev), y[sl].to(dev), x_l1[sl].to(dev), y1[sl].to(dev), x_u[su].to(dev),
                                m[su].to(dev)).item())
    torch.cuda.synchronize()
    digest = torch.cat([p.detach().reshape(-1) for m in nets for p in m.parameters()]).cpu()
    q.put((rank, losses, digest, step.kernels_per_replay))
    dist.barrier()
    dist.destroy_process_group()


def _dp_run(graph):
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, graph, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return res


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_hpfg_two_rank_replay_matches_eager():
    eager, graph = _dp_run(False), _dp_run(True)
    assert torch.equal(graph[0][2], graph[1][2])        # replicas stay identical
    assert graph[0][3] > 0
    for e, g in zip(eager, graph):
        assert e[1] == g[1] and torch.equal(e[2], g[2])
