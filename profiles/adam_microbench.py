"""The fused Adam / AdamW(+EMA) pass (hpfg_adam: 28 B/param, 36 B/param with the EMA) on the real flat buffer
(1 813 764 parameters: L2-resident between calls, launch-latency dominated) and on a x64 replicated buffer (a pure HBM
stream), against torch.optim.AdamW(fused=True) and (foreach=True) followed by the reference's per-tensor EMA loop on the
same buffers, and the Mean-Teacher step under graph replay with "sgd" against "adamw".  CUDA events over 50 calls after
warm-up.  Also reports which fp32 contraction of torch's foreach lerp_ and add(alpha=) (the two Adam operations ATen leaves
to the compiler) the installed torch computes:  python profiles/adam_microbench.py"""
import copy
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import hpfg_b200 as hb
from hpfg_b200 import _lib as L

dev = torch.device("cuda:0")
lib = L.lib()
st = L.stream_ptr(dev)
N = 1813764


def timed(fn, iters=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3      # us


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print("card: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(dev), smi[0] if smi else "n/a"))

# ---- contraction probe: torch's foreach lerp_ (weight < 0.5) and add(alpha=) against fma / unfused fp32 emulations
g = torch.Generator().manual_seed(0)
a, b = torch.randn(1 << 20, generator=g), torch.randn(1 << 20, generator=g) * 1e-3
w, alpha = float(torch.tensor(1 - 0.9, dtype=torch.float32)), float(torch.tensor(1e-2, dtype=torch.float32))
ga, gb = [a.to(dev)], [b.to(dev)]
torch._foreach_lerp_(ga, gb, 1 - 0.9)
add = torch._foreach_add(gb, [a.to(dev)], alpha=1e-2)
a64, b64 = a.double().numpy(), b.double().numpy()
f32 = lambda x: np.asarray(x, dtype=np.float32)
d = f32(b64 - a64).astype(np.float64)
emul = {"lerp": (f32(a64 + w * d), f32(a64 + f32(w * d).astype(np.float64)), ga[0].cpu().numpy()),
        "add(alpha)": (f32(b64 + alpha * a64), f32(b64 + f32(alpha * a64).astype(np.float64)), add[0].cpu().numpy())}
for op, (fused, unfused, got) in emul.items():
    print("torch foreach %-10s equals the fma form on %.6f of elements, the unfused form on %.6f"
          % (op, np.mean(fused == got), np.mean(unfused == got)))

# ---- the optimiser passes
PEAK = 7700.0
for rep in (1, 64):
    n = N * rep
    p, gr, m, v, e = (torch.randn(n, device=dev) for _ in range(5))
    v.abs_()
    args = (1 - 0.9, 0.999, 1 - 0.999, 1e-8, 1e-2, 1, 1.0, -1e-3, 0.5, 1 - 1e-5)
    t_adam = timed(lambda: L.check(lib.hpfg_adam(L.ptr(p), L.ptr(gr), L.ptr(m), L.ptr(v), None, n, *args, 0.0, st)))
    t_adam_ema = timed(lambda: L.check(lib.hpfg_adam(L.ptr(p), L.ptr(gr), L.ptr(m), L.ptr(v), L.ptr(e), n, *args, 0.99, st)))
    t_sgd_ema = timed(lambda: L.check(lib.hpfg_sgd_momentum_ema(L.ptr(p), L.ptr(gr), L.ptr(m), L.ptr(e), n, 0.01, 0.9, 1e-4, 1.0,
                                                                0, 0.99, st)))
    rows = [("hpfg_adam", t_adam, 28), ("hpfg_adam + EMA", t_adam_ema, 36), ("hpfg_sgd_momentum_ema", t_sgd_ema, 28)]
    # torch on the same bytes: the 82 parameter views (replicated rep times), gradients set once
    model = hb.UNet(1, 4).to(dev)
    views = [(o, k, s) for o, k, s in model._layout]
    params, emas = [], []
    for r in range(rep):
        for o, k, s in views:
            params.append(torch.nn.Parameter(p[r * N + o:r * N + o + k].view(s)))
            params[-1].grad = gr[r * N + o:r * N + o + k].view(s)
            emas.append(e[r * N + o:r * N + o + k].view(s))

    def ema_loop():
        with torch.no_grad():
            for qe, q in zip(emas, params):
                qe.mul_(0.99).add_(q, alpha=1 - 0.99)
    for kind in ("fused", "foreach"):
        opt = torch.optim.AdamW(params, lr=1e-3, weight_decay=1e-2, **{kind: True})
        t_opt = timed(opt.step)
        t_loop = timed(ema_loop)
        rows.append(("torch AdamW(%s=True)" % kind, t_opt, 28))
        rows.append(("  + EMA loop", t_opt + t_loop, 36))
        del opt
    for name, t, bpp in rows:
        gbs = n * bpp / t / 1e3
        print("%-24s x%-2d %9d params  %9.2f us per call  %7.0f GB/s algorithmic = %5.1f %% of %.0f" % (name, rep, n, t, gbs, 100 * gbs / PEAK, PEAK))
    del p, gr, m, v, e, params, emas, model
    torch.cuda.empty_cache()

# ---- Mean-Teacher step under graph replay: SGD vs AdamW (bf16 plans, 12 x 1 x 256 x 256 batch, 6 labeled)
gen = torch.Generator().manual_seed(1)
x = torch.rand(12, 1, 256, 256, generator=gen).to(dev)
y = torch.randint(0, 4, (6, 256, 256), generator=gen).to(dev)
for rnd in range(2):
    for opt_name in ("sgd", "adamw"):
        torch.manual_seed(3)
        s = hb.UNet(1, 4, precision="bf16").to(dev)
        step = hb.MeanTeacherStep(s, copy.deepcopy(s), optimizer=opt_name)
        step.enable_graph(True)
        for _ in range(5):
            step.step(x, y)
        t = timed(lambda: step.step(x, y), iters=100)
        print("round %d  MeanTeacherStep(optimizer=%-6r) graph replay: %8.1f us per step" % (rnd, opt_name, t))
