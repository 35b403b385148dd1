"""Device time of the phases of one eager Mean-Teacher step (CUDA events on the main stream; the teacher forward and
the weight gradients overlap on side streams as in production): python profiles/phase_times.py"""
import copy, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import hpfg_b200 as hb
from hpfg_b200 import _lib as L
from hpfg_b200.losses import ssl_loss_raw

dev = torch.device("cuda:0")
torch.manual_seed(0)
student = hb.UNet(1, 4, precision="bf16").to(dev)
teacher = copy.deepcopy(student)
step = hb.MeanTeacherStep(student, teacher)
x = torch.rand(32, 1, 224, 224, device=dev)
y = torch.randint(0, 4, (8, 224, 224), device=dev)
for _ in range(5):
    step.step(x, y)
torch.cuda.synchronize()
names = ["student fwd alone", "teacher fwd alone", "both fwd (2 streams)", "loss", "backward (dgrad chain + wgrad stream)", "sgd+ema"]
acc = [0.0] * len(names)
ev = lambda: torch.cuda.Event(enable_timing=True)
n_l, shape = 8, (32, 4, 224, 224)
reps = 10
for _ in range(reps):
    main, side = torch.cuda.current_stream(), step._side_stream(dev)
    e = [ev() for _ in range(8)]
    e[0].record()
    plan, out = step._forward(student, x, True, step._persistent("s_out", shape, dev), None)
    e[1].record()
    _, t_out = step._forward(teacher, x, False, step._persistent("t_out", shape, dev), None)
    e[2].record()
    side.wait_stream(main)
    with torch.cuda.stream(side):
        _, t_out = step._forward(teacher, x, False, step._persistent("t_out", shape, dev), None)
    plan, out = step._forward(student, x, True, step._persistent("s_out", shape, dev), None)
    main.wait_stream(side)
    if os.environ.get("PHASE_SYNC"):
        torch.cuda.synchronize()
    e[3].record()
    r = ssl_loss_raw(L.LOSS_MT, out, t_out[n_l:], y, n_l, cons_weight=0.01)
    if os.environ.get("PHASE_SYNC"):
        torch.cuda.synchronize()
    e[4].record()
    step._backward(student, plan, r["dstudent"], step.grads)
    e[5].record()
    step._next_iteration()
    step._opt_step(step._trained[0], None, teacher)
    e[6].record()
    torch.cuda.synchronize()
    for i in range(6):
        acc[i] += e[i].elapsed_time(e[i + 1])
for n, a in zip(names, acc):
    print("%-42s %7.3f ms" % (n, a / reps))
