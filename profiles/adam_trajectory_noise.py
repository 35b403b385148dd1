"""Where the fused Mean-Teacher AdamW trajectory and the drop-in autograd loop (torch.optim.AdamW) part ways, fp32 plans,
fixed dropout masks, 64x64, 2+2 images.  Per step: the two gradients (rel-L2), the driver's own gradient replayed through
torch.optim.AdamW(foreach=True) from the driver's parameters (the optimiser arithmetic alone), and the elements whose
parameters differ after one step, against the size of their gradient and whether the two gradients disagree in sign
(Adam's first step moves every element by ~lr*sign(g), so a noise-level gradient of opposite sign gives a 2*lr gap).
python profiles/adam_trajectory_noise.py"""
import copy
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import hpfg_b200 as hb
from tests.golden.common import make_state, make_masks, make_batch

DEV = "cuda:0"
in_ch, n_cls, n_l, n_u, h, w, seed = 1, 4, 2, 2, 64, 64, 41
n = n_l + n_u
print("card: %s" % torch.cuda.get_device_name(0))
st = make_state(in_ch, n_cls, seed)


def net():
    m = hb.UNet(in_ch, n_cls, precision="fp32")
    m.load_state_dict(st)
    return m.to(DEV)


s1, s2 = net(), net()
t1, t2 = copy.deepcopy(s1), copy.deepcopy(s2)
step = hb.MeanTeacherStep(s1, t1, optimizer="adamw", lr=1e-3, weight_decay=1e-2, total_itrs=100)
opt = torch.optim.AdamW(s2.parameters(), lr=1e-3, weight_decay=1e-2, foreach=True)
for p in t2.parameters():
    p.requires_grad = False
s2.train()
t2.train()
med_loss = hb.Med_Sup_Loss(n_cls)
args = type("A", (), dict(consistency=0.1, consistency_rampup=200.0))()
names = [k for k, _ in s1.named_parameters()]
layout = s1._layout


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


for it in range(1, 6):
    x_l, x_u, y = make_batch(n_l, n_u, in_ch, n_cls, h, w, seed + 100 * it)
    x, y = torch.cat([x_l, x_u]).to(DEV).float(), y.to(DEV).long()
    for s, t in ((s1, t1), (s2, t2)):
        s.set_dropout_masks(make_masks(n, h, w, seed + 100 * it + 1))
        t.set_dropout_masks(make_masks(n, h, w, seed + 100 * it + 2))
    p_before = s1.flat_params.detach().clone()
    opt_before = copy.deepcopy(step.state_dict()["optimizers"][0])
    step.step(x, y)
    g_drv = step.grads.clone()
    out = s2(x)
    with torch.no_grad():
        ema_soft = torch.softmax(t2(x), dim=1)
    loss = med_loss(out[:n_l], y) + hb.get_current_consistency_weight(it // 150, args) * \
        torch.mean((torch.softmax(out, dim=1)[n_l:] - ema_soft[n_l:]) ** 2)
    for grp in opt.param_groups:
        grp["lr"] = hb.medical_lr(it, 1e-3, 100)
    opt.zero_grad()
    loss.backward()
    g_ref = torch.cat([p.grad.reshape(-1) for p in s2.parameters()])
    p_ref_before = s2.flat_params.detach().clone()
    opt.step()
    hb.update_ema_variables(s2, t2, 0.99, it)
    torch.cuda.synchronize()
    # the driver's own gradient through torch.optim.AdamW, from the driver's parameters and optimiser state
    views = [torch.nn.Parameter(p_before[o:o + k].view(s).clone()) for o, k, s in layout]
    replay = torch.optim.AdamW(views, lr=hb.medical_lr(it, 1e-3, 100), weight_decay=1e-2, foreach=True)
    if opt_before["state"]:
        replay.load_state_dict({"state": opt_before["state"], "param_groups": [dict(replay.state_dict()["param_groups"][0],
                                                                                     params=list(range(82)))]})
        for grp in replay.param_groups:
            grp["lr"] = hb.medical_lr(it, 1e-3, 100)
    for v, (o, k, s) in zip(views, layout):
        v.grad = g_drv[o:o + k].view(s).clone()
    replay.step()
    p_replay = torch.cat([v.detach().reshape(-1) for v in views])
    p_drv, p_ref = s1.flat_params.detach(), s2.flat_params.detach()
    print("step %d: grad rel-L2 driver vs autograd %.3e | params before the step rel-L2 %.3e | driver params == torch AdamW on "
          "the driver's gradient: %s | params after rel-L2 %.3e"
          % (it, rel(g_drv, g_ref), rel(p_before, p_ref_before), torch.equal(p_replay, p_drv), rel(p_drv, p_ref)))
    if it == 1:
        diff = (p_drv - p_ref).abs() > 1e-6
        flip = torch.sign(g_drv) != torch.sign(g_ref)
        scale = torch.cat([g_ref[o:o + k].pow(2).mean().sqrt().expand(k) for o, k, _ in layout])
        r = (g_ref.abs() / scale)
        print("  step 1: %d of %d elements differ by > 1e-6 (max %.3e = %.2f lr); %d of them have gradients of opposite sign, "
              "and all differing elements have |g| / rms(g of their tensor) <= %.3e (median %.3e; median over all elements %.3e)"
              % (int(diff.sum()), diff.numel(), (p_drv - p_ref).abs().max().item(), (p_drv - p_ref).abs().max().item() / 1e-3,
                 int((diff & flip).sum()), r[diff].max().item(), r[diff].median().item(), r.median().item()))
        worst = sorted(((int(diff[o:o + k].sum()), names[i]) for i, (o, k, _) in enumerate(layout)), reverse=True)[:6]
        print("  step 1: tensors with the most differing elements: %s" % worst)
