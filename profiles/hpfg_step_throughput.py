"""Throughput of main.py's HPFG iteration (HPFGStep: three UNet_Plus networks, CutMix batch, necks + Dense_Loss) at the ACDC
shape, 8 labeled + 24 unlabeled 224x224 per step, bf16 U-Nets, 1 GPU, inputs resident:  python profiles/hpfg_step_throughput.py

Two drivers built from the same seed run the same batches: one launches eagerly, the other replays its step as one CUDA graph.
They alternate in blocks of steps, so both see the same machine state, and after every block their losses must be bit-identical;
at the end so must every parameter, BatchNorm buffer and optimiser buffer."""
import copy, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import hpfg_b200 as hb
from hpfg_b200 import _lib as L

dev = torch.device("cuda:0")
n_l, n_u, H, W = 8, 24, 224, 224
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except Exception as exc:          # the card name still comes from torch
    smi = "power limit not read (%s)" % exc
print("device: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(dev), smi))


def driver(graph):
    torch.manual_seed(0)
    m1, m2 = hb.UNet_Plus(1, 4).to(dev), hb.UNet_Plus(1, 4).to(dev)
    nets = (m1, m2, copy.deepcopy(m2))
    step = hb.HPFGStep(*nets, weight_decay=0.0005)
    step.cur_itrs = 1500                      # Mean-Teacher term on (main.py:137-142)
    step.enable_graph(graph)
    return step, nets


g = torch.Generator().manual_seed(3)
label_img, img_unlabel = torch.rand(n_l, 1, H, W, generator=g).to(dev), torch.rand(n_u, 1, H, W, generator=g).to(dev)
label_img1 = torch.rand(n_l, 1, H, W, generator=g).to(dev)
y, y1 = torch.randint(0, 4, (n_l, H, W), generator=g).to(dev), torch.randint(0, 4, (n_l, H, W), generator=g).to(dev)
mask = torch.zeros(n_u, 1, H, W)
mask[:, :, 40:150, 60:180] = 1.0
mask = mask.to(dev)
runs = {"eager": driver(False), "replay": driver(True)}
losses = {k: [] for k in runs}


def block(name, steps):
    step = runs[name][0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0 = L.lib().hpfg_launch_count()
    out = torch.empty(steps, device=dev)
    e0.record()
    for i in range(steps):
        out[i:i + 1].copy_(step.step(label_img, y, label_img1, y1, img_unlabel, mask).reshape(1))
    e1.record()
    torch.cuda.synchronize()
    losses[name] += out.tolist()
    return e0.elapsed_time(e1) / steps, (L.lib().hpfg_launch_count() - k0) / steps


for name in runs:                             # warm-up: plans, first updates, the capture
    block(name, 3)
times = {k: [] for k in runs}
launches = {}
rounds, steps = 6, 10
for r in range(rounds):
    for name in (("eager", "replay") if r % 2 == 0 else ("replay", "eager")):
        ms, launches[name] = block(name, steps)
        times[name].append(ms)
assert losses["eager"] == losses["replay"], "eager and replayed losses differ"
(s_e, nets_e), (s_r, nets_r) = runs["eager"], runs["replay"]
for a, b in zip(nets_e, nets_r):
    sa, sb = a.state_dict(), b.state_dict()
    assert all(torch.equal(sa[k], sb[k]) for k in sa), "eager and replayed parameters / buffers differ"
for oa, ob in zip(s_e.state_dict()["optimizers"], s_r.state_dict()["optimizers"]):
    assert all(torch.equal(oa["state"][i][k], ob["state"][i][k]) for i in oa["state"] for k in oa["state"][i])
print("eager vs replay: %d steps each, losses, parameters, BatchNorm buffers and optimiser state bit-identical"
      % len(losses["eager"]))
for name in runs:
    t = sorted(times[name])
    med = t[len(t) // 2]
    print("HPFGStep 8+24 @224 bf16 %-6s: %.3f ms/step median of %d blocks of %d (min %.3f, max %.3f)  %.0f images/s  "
          "(%.0f library launches per step on the host)"
          % (name, med, rounds, steps, t[0], t[-1], (n_l + n_u) / med * 1e3, launches[name]))
print("kernels per replay: %d   last loss %.5f  contrast %.5f"
      % (s_r.kernels_per_replay, losses["replay"][-1], s_r.last["contrast"].item()))
