"""GPU: the fused Adam / AdamW(+EMA) pass against torch.optim's foreach implementation, and the step drivers with
optimizer="adam"/"adamw": trajectory against the drop-in autograd loop, graph replay against eager launches, bit-exact
resume, data-parallel replicas."""
import copy
import os
import re
import socket

import pytest
import torch
import torch.multiprocessing as mp

import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from tests.golden.common import make_state, make_masks, make_batch, make_plus_state, make_hpfg_batch
from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BETAS, EPS = (0.9, 0.999), 1e-8
# conv biases ahead of a train-mode BatchNorm: analytically zero gradient, so both gradient paths hold rounding noise there
PRE_BN_BIAS = re.compile(r"conv_conv\.[04]\.bias$")


@pytest.mark.parametrize("ema", [False, True])
@pytest.mark.parametrize("grad_scale", [1.0, 0.5])
@pytest.mark.parametrize("wd", [0.0, 1e-2])
@pytest.mark.parametrize("name", ["adam", "adamw"])
def test_adam_kernel_matches_torch_foreach(name, wd, grad_scale, ema):
    """20 steps over the 82 parameter views of a UNet with random gradients and a moving lr, against
    torch.optim.Adam/AdamW(foreach=True) and the reference's update_ema_variables loop."""
    torch.manual_seed(21)
    model = hb.UNet(1, 4).to(DEV)
    p = model.flat_params.detach()
    n = p.numel()
    m, v, e = torch.zeros_like(p), torch.zeros_like(p), p.clone()
    ref_p = [q.detach().clone() for q in model.parameters()]
    ref_e = [q.clone() for q in ref_p]
    cls = torch.optim.AdamW if name == "adamw" else torch.optim.Adam
    opt = cls(ref_p, lr=1e-3, betas=BETAS, eps=EPS, weight_decay=wd, foreach=True)
    st = L.stream_ptr(torch.device(DEV))
    for t in range(1, 21):
        lr = hb.medical_lr(t, 1e-3, 40)
        g = torch.randn(n, device=DEV) * (10.0 ** (t % 5 - 3))
        for grp in opt.param_groups:
            grp["lr"] = lr
        for q, (o, k, shape) in zip(ref_p, model._layout):
            q.grad = (g[o:o + k] * grad_scale).view(shape)
        opt.step()
        alpha = min(1 - 1 / (t + 1), 0.99)
        if ema:
            for qe, q in zip(ref_e, ref_p):
                qe.mul_(alpha).add_(q, alpha=1 - alpha)
        step_size = (lr / (1 - BETAS[0] ** t)) * -1
        bc2_sqrt = (1 - BETAS[1] ** t) ** 0.5
        decay = 1 - lr * wd if name == "adamw" else 1.0
        L.check(L.lib().hpfg_adam(L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), L.ptr(e) if ema else None, n, 1 - BETAS[0], BETAS[1],
                                  1 - BETAS[1], EPS, wd, int(name == "adamw"), grad_scale, step_size, bc2_sqrt, decay, alpha,
                                  st), "hpfg_adam")
    torch.cuda.synchronize()
    cat = lambda ts: torch.cat([q.reshape(-1) for q in ts])
    want = dict(param=cat(ref_p), exp_avg=cat(opt.state[q]["exp_avg"] for q in ref_p),
                exp_avg_sq=cat(opt.state[q]["exp_avg_sq"] for q in ref_p))
    got = dict(param=p, exp_avg=m, exp_avg_sq=v)
    if ema:
        want["ema"], got["ema"] = cat(ref_e), e
    for k in want:
        assert torch.allclose(got[k], want[k], rtol=1e-6, atol=1e-7), (k, (got[k] - want[k]).abs().max().item())
    print("hpfg_adam %s wd=%g scale=%g ema=%s bit-identical to torch foreach: %s"
          % (name, wd, grad_scale, ema, {k: torch.equal(got[k], want[k]) for k in want}))


def test_mean_teacher_adamw_trajectory_matches_autograd_loop():
    """5 fp32 steps of MeanTeacherStep(optimizer="adamw") with fixed dropout masks against the drop-in loop (autograd,
    Med_Sup_Loss, inline consistency, torch.optim.AdamW(foreach=True), update_ema_variables).  Every step starts the loop
    from the driver's networks and its optimiser state, loaded through the torch.optim.AdamW layout of state_dict().  Then
    the loss and the gradient agree with autograd's; torch.optim.AdamW fed the driver's gradient gives the driver's
    parameters and moments bit for bit, and update_ema_variables its teacher; and the loop's own AdamW step agrees with the
    driver's wherever the gradient is above rounding noise.  (Adam's first steps move every element by about lr*sign(g), so
    an element whose gradient is rounding noise -- the conv biases ahead of train-mode BatchNorm, whose gradient is
    analytically zero, and single weights -- moves by up to +-lr on either side whatever the implementation, and a
    free-running comparison drifts apart from there: profiles/adam_trajectory_noise.txt.)"""
    in_ch, n_cls, n_l, n_u, h, w, seed = 1, 4, 2, 2, 64, 64, 41
    n, lr0, wd = n_l + n_u, 1e-3, 1e-2
    st = make_state(in_ch, n_cls, seed)

    def net():
        m = hb.UNet(in_ch, n_cls, precision="fp32")
        m.load_state_dict(st)
        return m.to(DEV)
    s1, s2 = net(), net()
    t1, t2 = copy.deepcopy(s1), copy.deepcopy(s2)
    step = hb.MeanTeacherStep(s1, t1, optimizer="adamw", lr=lr0, weight_decay=wd, total_itrs=100)
    for p in t2.parameters():
        p.requires_grad = False
    s2.train()
    t2.train()
    med_loss = hb.Med_Sup_Loss(n_cls)
    args = type("A", (), dict(consistency=0.1, consistency_rampup=200.0))()
    layout = s1._layout
    cat = lambda ts: torch.cat([t.detach().reshape(-1) for t in ts])
    pre_bn = torch.cat([torch.full((k,), bool(PRE_BN_BIAS.search(name)), device=DEV)
                        for (name, _), (_, k, _) in zip(s1.named_parameters(), layout)])

    def adamw(params, sd):
        opt = torch.optim.AdamW(params, lr=lr0, betas=BETAS, eps=EPS, weight_decay=wd, foreach=True)
        if sd["state"]:
            opt.load_state_dict(copy.deepcopy(sd))
        for grp in opt.param_groups:
            grp["lr"] = sd["param_groups"][0]["lr"]           # Medical_LR of the coming iteration
        return opt
    for it in range(1, 6):
        x_l, x_u, y = make_batch(n_l, n_u, in_ch, n_cls, h, w, seed + 100 * it)
        x, y = torch.cat([x_l, x_u]).to(DEV).float(), y.to(DEV).long()
        # the loop starts from the driver's state
        s2.load_state_dict(s1.state_dict())
        t2.load_state_dict(t1.state_dict())
        sd = step.state_dict()["optimizers"][0]
        assert sd["param_groups"][0]["lr"] == hb.medical_lr(it, lr0, 100)
        opt = adamw(s2.parameters(), sd)
        p0, e0 = s1.flat_params.detach().clone(), t1.flat_params.detach().clone()
        for s, t in ((s1, t1), (s2, t2)):
            s.set_dropout_masks(make_masks(n, h, w, seed + 100 * it + 1))
            t.set_dropout_masks(make_masks(n, h, w, seed + 100 * it + 2))
        loss_drv = step.step(x, y).item()
        out = s2(x)
        with torch.no_grad():
            ema_soft = torch.softmax(t2(x), dim=1)
        loss = med_loss(out[:n_l], y) + hb.get_current_consistency_weight(it // 150, args) * \
            torch.mean((torch.softmax(out, dim=1)[n_l:] - ema_soft[n_l:]) ** 2)
        opt.zero_grad()
        loss.backward()
        g_ref = cat(p.grad for p in s2.parameters())
        opt.step()
        hb.update_ema_variables(s2, t2, 0.99, it)
        torch.cuda.synchronize()
        assert abs(loss_drv - loss.item()) <= 1e-5 * abs(loss.item()), (it, loss_drv, loss.item())
        g_drv = step.grads.clone()
        assert rel_l2(g_drv, g_ref) <= 1e-5, (it, rel_l2(g_drv, g_ref))
        # the optimiser side alone: torch.optim.AdamW and update_ema_variables on the driver's own gradient
        views = [torch.nn.Parameter(p0[o:o + k].view(shape).clone()) for o, k, shape in layout]
        for v, (o, k, shape) in zip(views, layout):
            v.grad = g_drv[o:o + k].view(shape).clone()
        replay = adamw(views, sd)
        replay.step()
        assert torch.equal(cat(views), s1.flat_params.detach()), it
        exp_avg, exp_avg_sq = step.mom
        assert torch.equal(cat(replay.state[v]["exp_avg"] for v in views), exp_avg), it
        assert torch.equal(cat(replay.state[v]["exp_avg_sq"] for v in views), exp_avg_sq), it
        alpha = min(1 - 1 / (it + 1), 0.99)
        e_ref = e0.mul_(alpha).add_(cat(views), alpha=1 - alpha)
        assert torch.allclose(t1.flat_params.detach(), e_ref, rtol=1e-6, atol=1e-7), it
        # the loop's own step, except where the gradient is rounding noise: the conv biases ahead of train-mode BatchNorm
        # (analytically zero gradient) and the elements whose two computed gradients disagree in sign
        p_drv, p_ref = s1.flat_params.detach(), s2.flat_params.detach()
        resolved = (torch.sign(g_drv) == torch.sign(g_ref)) & ~pre_bn
        assert int((~resolved & ~pre_bn).sum()) <= 1e-3 * int((~pre_bn).sum()), (it, int((~resolved & ~pre_bn).sum()))
        assert rel_l2(p_drv[resolved], p_ref[resolved]) <= 1e-5, (it, rel_l2(p_drv[resolved], p_ref[resolved]))


def _run_graph(kind, graph, steps=5):
    torch.manual_seed(13)
    a = hb.UNet(1, 4, precision="bf16").to(DEV)
    b = copy.deepcopy(a) if kind in ("mt", "uamt", "ict") else hb.UNet(1, 4, precision="bf16").to(DEV)
    kw = dict(optimizer="adamw", total_itrs=40, consistency_rampup=0.2, weight_decay=1e-2)     # lr, alpha and w move every step
    step = dict(mt=lambda: hb.MeanTeacherStep(a, b, **kw), cps=lambda: hb.CPSStep(a, b, **kw),
                uamt=lambda: hb.UAMTStep(a, b, T=4, **kw), ict=lambda: hb.ICTStep(a, b, **kw))[kind]()
    step.enable_graph(graph)
    g = torch.Generator().manual_seed(6)
    losses = []
    for _ in range(steps):
        x = torch.rand(6, 1, 64, 64, generator=g).to(DEV)
        y = torch.randint(0, 4, (2, 64, 64), generator=g).to(DEV)
        if kind == "uamt":
            noise = torch.clamp(torch.randn(4, 1, 64, 64, generator=g) * 0.1, -0.2, 0.2).to(DEV)
            mc_noise = torch.clamp(torch.randn(2, 8, 1, 64, 64, generator=g) * 0.1, -0.2, 0.2).to(DEV)
            loss = step.step(x, y, noise, mc_noise)
        elif kind == "ict":
            loss = step.step(x, y, torch.rand(2, generator=g))
        else:
            loss = step.step(x, y)
        losses.append(loss.item())
    torch.cuda.synchronize()
    assert (step.kernels_per_replay > 0) == bool(graph)
    return losses, a.flat_params.detach().clone(), b.flat_params.detach().clone(), step.state_dict()


@pytest.mark.parametrize("kind", ["mt", "cps", "uamt", "ict"])
def test_adamw_graph_replay_matches_eager(kind):
    l0, a0, b0, sd0 = _run_graph(kind, False)
    l1, a1, b1, sd1 = _run_graph(kind, True)
    assert l0 == l1, (l0, l1)
    assert torch.equal(a0, a1) and torch.equal(b0, b1)
    for o0, o1 in zip(sd0["optimizers"], sd1["optimizers"]):
        for i in o0["state"]:
            assert all(torch.equal(o0["state"][i][k], o1["state"][i][k]) for k in o0["state"][i])


def _mt_fresh():
    torch.manual_seed(19)
    s = hb.UNet(1, 4, precision="bf16").to(DEV)
    return s, copy.deepcopy(s)


def test_mean_teacher_adamw_resume_is_bit_exact():
    g = torch.Generator().manual_seed(8)
    batches = [(torch.rand(6, 1, 64, 64, generator=g).to(DEV), torch.randint(0, 4, (2, 64, 64), generator=g).to(DEV))
               for _ in range(5)]
    s, t = _mt_fresh()
    step = hb.MeanTeacherStep(s, t, optimizer="adamw", total_itrs=40)
    ref = [step.step(*b).item() for b in batches]
    want = (s.flat_params.clone(), t.flat_params.clone())
    s, t = _mt_fresh()
    step = hb.MeanTeacherStep(s, t, optimizer="adamw", total_itrs=40)
    got = [step.step(*b).item() for b in batches[:3]]
    ck = copy.deepcopy({"model": s.state_dict(), "ema": t.state_dict(), "step": step.state_dict()})
    s2, t2 = _mt_fresh()
    s2.load_state_dict(ck["model"])
    t2.load_state_dict(ck["ema"])
    step2 = hb.MeanTeacherStep(s2, t2, optimizer="adamw", total_itrs=40)
    step2.load_state_dict(ck["step"])
    got += [step2.step(*b).item() for b in batches[3:]]
    assert got == ref, (got, ref)
    assert torch.equal(s2.flat_params, want[0]) and torch.equal(t2.flat_params, want[1])


def test_hpfg_step_adamw_resume_is_bit_exact():
    in_ch, n_cls, n_l, n_u, h, w, seed = 1, 4, 2, 2, 64, 64, 51
    batches = [[t.to(DEV) for t in make_hpfg_batch(n_l, n_u, in_ch, n_cls, h, w, seed + 10 * i)] for i in range(5)]

    def fresh():
        nets = []
        for k in range(2):
            m = hb.UNet_Plus(in_ch, n_cls, precision="fp32")
            m.load_state_dict(make_plus_state(in_ch, n_cls, seed + k))
            nets.append(m.to(DEV))
        nets.append(copy.deepcopy(nets[1]))
        for m in nets:
            m.set_dropout_enabled(False)
        return nets, hb.HPFGStep(*nets, optimizer="adamw", total_itrs=40, mt_start=2)

    def digest(nets):
        return torch.cat([p.detach().reshape(-1) for m in nets for p in m.parameters()])
    nets, step = fresh()
    ref = [step.step(*b).item() for b in batches]
    want = digest(nets)
    nets, step = fresh()
    got = [step.step(*b).item() for b in batches[:3]]
    sd = step.state_dict()
    assert sorted(sd["optimizers"][0]["state"]) == list(range(82))          # model1's necks never get a gradient
    assert sorted(sd["optimizers"][1]["state"]) == list(range(98))
    ck = copy.deepcopy({"nets": [m.state_dict() for m in nets], "step": sd})
    nets2, step2 = fresh()
    for m, msd in zip(nets2, ck["nets"]):
        m.load_state_dict(msd)
    step2.load_state_dict(ck["step"])
    got += [step2.step(*b).item() for b in batches[3:]]
    assert got == ref, (got, ref)
    assert torch.equal(digest(nets2), want)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    student = hb.UNet(1, 4, precision="fp32")
    student.load_state_dict(make_state(1, 4, 3))
    student.to(dev)
    teacher = copy.deepcopy(student)
    step = hb.MeanTeacherStep(student, teacher, optimizer="adamw")
    for it in (1, 2, 3):
        x_l, x_u, y = make_batch(2, 2, 1, 4, 32, 32, 10 + it)
        xl, xu, yy = hb.shard_batch(x_l, x_u, y, rank, world)
        step.step(torch.cat([xl, xu]).to(dev), yy.to(dev))
    torch.cuda.synchronize()
    q.put((rank, student.flat_params.cpu(), teacher.flat_params.cpu()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_adamw_replicas_stay_identical():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert torch.equal(res[0][1], res[1][1]) and torch.equal(res[0][2], res[1][2])
