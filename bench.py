#!/usr/bin/env python
"""bench.py -- throughput of the HPFG semi-supervised U-Net training step on B200.

    python bench.py --gpus N --steps K --warmup W                      # this repo's sm_100a path, BASELINE config 2 (Mean-Teacher 8+24)
    python bench.py --config {mt_acdc,mt_cfg1,mt_isic,cps,uamt} ...    # the other BASELINE.json configurations
    python bench.py --impl reference --gpus N --steps K --warmup W     # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                             # also write what the last timed step computed, DIR/<name>.npy

A "step" is one training iteration of the configured trainer over one synthetic batch of 224x224 slices:
  mt_*  2017_03_NIPS_Mean-Teacher_ACDC.py:89-113      student forward+backward, teacher forward, fused SSL loss, SGD, EMA
  cps   2021_06_CVPR_CPS_ACDC.py:90-120               two students forward+backward, cross pseudo supervision, two SGD steps
  uamt  2019_07_MICCAI_Uncertainty_Aware_ACDC.py:120-170   student forward+backward, 1 + T/2 noisy teacher forwards (T=8), masked MSE, SGD, EMA
Prints ONE JSON line (rank 0).  N>1 is launched by torchrun, one rank per GPU, data parallel, weak scaling (the configured
per-GPU batch on every rank, rank-distinct data, bucketed NCCL gradient all-reduce overlapped with backward)."""
import argparse
import copy
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W = 224, 224
F_FWD = 4516642816.0                 # conv FLOPs per image, forward (SURVEY 8d; identical for 1ch/4cls and 3ch/2cls)
CONFIGS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on (config/mean_teacher_unet_30k_224x224_ACDC.yaml:13-14)
    "mt_acdc": dict(kind="mt", in_ch=1, n_cls=4, n_l=8, n_u=24,
                    workload="mean_teacher_unet_30k_224x224_ACDC (UNet 1ch/4cls, 8 labeled + 24 unlabeled 224x224 per GPU per step)"),
    # configs[0]: the reference's own CPU-runnable case
    "mt_cfg1": dict(kind="mt", in_ch=1, n_cls=4, n_l=12, n_u=12,
                    workload="Mean-Teacher step, UNet 1ch/4cls, 12 labeled + 12 unlabeled 224x224 per GPU per step"),
    # configs[4]: ISIC shape, 24 images per GPU (global 192 on 8 GPUs)
    "mt_isic": dict(kind="mt", in_ch=3, n_cls=2, n_l=12, n_u=12,
                    workload="Mean-Teacher step, ISIC-shape UNet 3ch/2cls, 12 labeled + 12 unlabeled 224x224 per GPU per step (global 192 on 8 GPUs)"),
    # configs[2]: CPS (config/cps_unet_30k_224x224_ACDC.yaml:13-14)
    "cps": dict(kind="cps", in_ch=1, n_cls=4, n_l=8, n_u=24,
                workload="CPS cross pseudo supervision, two UNets 1ch/4cls, 8 labeled + 24 unlabeled 224x224 per GPU per step"),
    # configs[3]: UAMT, T = 8 stochastic teacher forwards
    "uamt": dict(kind="uamt", in_ch=1, n_cls=4, n_l=12, n_u=12, T=8,
                 workload="UAMT uncertainty-aware Mean-Teacher, T=8, UNet 1ch/4cls, 12 labeled + 12 unlabeled 224x224 per GPU per step"),
}
METRICS = {"mt": "UNet SSL train images/sec @224x224 (Mean-Teacher step)", "cps": "UNet SSL train images/sec @224x224 (CPS step)",
           "uamt": "UNet SSL train images/sec @224x224 (UAMT step, T=8)"}
# dram__bytes_read.sum + dram__bytes_write.sum from ncu (see the named profile); None until measured for the current kernels
TOP_KERNEL_DRAM_BYTES = 58.16e6      # one launch of the 3x3 16->16 @224 fprop (profiles/r01_ncu_prof_fprop16_final_raw.txt)
LOSS_DRAM_BYTES = 49748736 + 5297408      # dram read + write of the one-launch Mean-Teacher loss kernel (profiles/r02b_loss_mt_one_ncu.txt)
CONV_FAMILY_DRAM_BYTES = 1712.0e6    # all 68 tc_conv_kernel launches of one mt_acdc step (25 MB per launch on average)
CONV_FAMILY_DRAM_SOURCE = ("ncu dram__bytes_read.sum + dram__bytes_write.sum over the 68 tc_conv_kernel launches of one steady-state step, "
                           "profiles/r02b_launch_summary.txt (whole step: 5.65 GB of DRAM traffic)")


def flops_per_step(c):
    """Algorithmic conv FLOPs of one step (SURVEY 8d): forward F_FWD per image; backward 2*F_FWD - f_in0."""
    f_in0 = 2.0 * 9 * H * W * c["in_ch"] * 16
    n = c["n_l"] + c["n_u"]
    if c["kind"] == "mt":
        return n * (4 * F_FWD - f_in0)                        # student fwd+bwd, teacher fwd on the whole batch
    if c["kind"] == "cps":
        return n * 2 * (3 * F_FWD - f_in0)
    return n * (3 * F_FWD - f_in0) + c["n_u"] * F_FWD + c["T"] * c["n_u"] * F_FWD      # uamt: + teacher on n_u + T/2 forwards of 2*n_u


def tc_conv_flops_per_step(c):
    """FLOPs of the launches timed under the tensor-core conv category: EVERY forward conv (in_conv.0 padded to 16 channels
    and out_conv included -- both run on the tensor-core kernel) of all forwards + every data gradient (all convs but in_conv.0)."""
    f_in0 = 2.0 * 9 * H * W * c["in_ch"] * 16
    n = c["n_l"] + c["n_u"]
    if c["kind"] == "mt":
        return n * (2 * F_FWD + (F_FWD - f_in0))
    if c["kind"] == "cps":
        return n * 2 * (F_FWD + (F_FWD - f_in0))
    return n * (F_FWD + (F_FWD - f_in0)) + (c["n_u"] + c["T"] * c["n_u"]) * F_FWD


def config_block(c, world):
    """Identical in both arms (the driver compares them)."""
    n = c["n_l"] + c["n_u"]
    return {"workload": c["workload"], "global_batch": n * world, "parallelism": "dp%d" % world,
            "l2": "per-step working set (~2 GB of activations per network) exceeds the 126 MB L2"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


def _hbm_roofline(kernel, algo_bytes, cat, pk, note, traffic=None, traffic_source=None):
    """Achieved algorithmic GB/s of one kernel category of the serialized profiling pass (CUDA events in the library)."""
    if cat["ms_per_step"] <= 0:
        return None
    gbs = algo_bytes / (cat["ms_per_step"] * 1e-3) / 1e9
    return {"kernel": kernel, "bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
            "us_per_step": cat["ms_per_step"] * 1e3, "algorithmic_bytes": algo_bytes, "traffic": traffic,
            "traffic_source": traffic_source, "note": note}


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE = 2 << 20                # elements kept of a larger output: the same seeded positions in every run


def dump_outputs(out_dir, step):
    """Write what the step driver handed back after its last call, one DIR/<name>.npy per array (float32, float64 kept): the
    tensors of step.last (loss scalars, logits) and the flat parameters and BatchNorm running statistics of every network it
    updates.  An array of more than DUMP_SAMPLE elements is reduced to DUMP_SAMPLE positions drawn by a fixed seed, so two
    builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    arrays = {k: v for k, v in step.last.items() if torch.is_tensor(v)}
    for attr in ("model", "ema_model", "m1", "m2"):
        m = getattr(step, attr, None)
        if m is not None:
            arrays[attr + ".flat_params"], arrays[attr + ".bn_running"] = m.flat_params, m.bn_running
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach().flatten().cpu()
        t = t if t.dtype == torch.float64 else t.float()
        if t.numel() > DUMP_SAMPLE:
            t = t[torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values]
        total += t.numel() * t.element_size()
        assert total <= DUMP_MAX_BYTES, "outputs exceed %d bytes" % DUMP_MAX_BYTES
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())
    return sorted(arrays)


def synthetic_batch(c, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(c["n_l"] + c["n_u"], c["in_ch"], H, W, generator=g)
    y = torch.randint(0, c["n_cls"], (c["n_l"], H, W), generator=g)
    return x, y


# ------------------------------------------------------------------------------------------------ CPU legs
def _find_real_reference():
    """The reference's own files, if a copy travelled to this machine ($HPFG_REF or baseline/_ref); None on the GPU box."""
    for p in (os.environ.get("HPFG_REF"), os.path.join(ROOT, "baseline", "_ref")):
        if p and os.path.isfile(os.path.join(p, "model", "unet.py")):
            return p
    return None


def cpu_reference_steps(c, steps, warmup):
    """The reference's CPU path (config `cuda: False`) for one step of config c, torch CPU fp32 on all host threads.
    kind 'reference': the reference's own UNet / Med_Sup_Loss / update_ema_variables / Medical_LR objects loaded by file
    path (Mean-Teacher only); kind 'port': oracle/ (the restatement pinned to them by tests/test_oracle_vs_reference.py)."""
    import torch
    import oracle
    torch.set_num_threads(os.cpu_count())
    torch.manual_seed(1337)
    n_l, n_u, in_ch, n_cls = c["n_l"], c["n_u"], c["in_ch"], c["n_cls"]
    g = torch.Generator().manual_seed(1337)
    x_l = torch.rand(n_l, in_ch, H, W, generator=g)
    x_u = torch.rand(n_u, in_ch, H, W, generator=g)
    y = torch.randint(0, n_cls, (n_l, H, W), generator=g)
    ref_root = _find_real_reference() if c["kind"] == "mt" else None
    if ref_root is not None:
        os.environ["HPFG_REF"] = ref_root
        from oracle.ref_loader import load_reference
        ref = load_reference()
        model = ref.UNet(in_channels=in_ch, num_classes=n_cls)
        ema_model = copy.deepcopy(model)
        for p in ema_model.parameters():
            p.requires_grad = False
        optimizer = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4)
        sched = ref.Medical_LR(optimizer=optimizer, base_lr=0.01, max_iterations=30000)
        med_loss = ref.Med_Sup_Loss(n_cls)
        args = type("A", (), dict(consistency=0.1, consistency_rampup=200.0))()
        model.train()
        ema_model.train()
        x = torch.cat([x_l, x_u])

        def one(it):                                     # 2017_03_NIPS_Mean-Teacher_ACDC.py:94-113
            output = model(x)
            output_soft = torch.softmax(output, dim=1)
            with torch.no_grad():
                ema_soft = torch.softmax(ema_model(x), dim=1)
            loss = med_loss(output[:n_l], y) + ref.get_current_consistency_weight(it // 150, args) * \
                torch.mean((output_soft[n_l:] - ema_soft[n_l:]) ** 2)
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            sched.step()
            ref.update_ema_variables(model, ema_model, 0.99, it)
            return loss.item()
        kind = "reference"
    else:
        st = oracle.init_unet_state(in_ch, n_cls)
        opt = oracle.SGDState()
        if c["kind"] == "mt":
            te = {k: v.clone() for k, v in st.items()}
            one = lambda it: oracle.mt_step(st, te, opt, x_l, x_u, y, it)          # noqa: E731
        elif c["kind"] == "cps":
            st2, opt2 = oracle.init_unet_state(in_ch, n_cls), oracle.SGDState()
            one = lambda it: oracle.cps_step(st, st2, opt, opt2, x_l, x_u, y, it)  # noqa: E731
        else:
            te = oracle.init_unet_state(in_ch, n_cls)
            T = c["T"]

            def one(it):
                noise = torch.clamp(torch.randn(x_u.shape) * 0.1, -0.2, 0.2)
                mc = torch.clamp(torch.randn((T // 2, 2 * n_u) + tuple(x_u.shape[1:])) * 0.1, -0.2, 0.2)
                return oracle.uamt_step(st, te, opt, x_l, x_u, y, it, noise, mc)
        kind = "port"
    it = 0
    for _ in range(warmup):
        it += 1
        one(it)
    t0 = time.perf_counter()
    for _ in range(steps):
        it += 1
        one(it)
    dt = time.perf_counter() - t0
    return (n_l + n_u) * steps / dt, dt / steps, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    # every step is the full configured batch (BatchNorm / Dice see the real batch): ~1.7 s of host work per Mean-Teacher step
    # on 16 cores
    steps, warmup = args.steps, args.warmup
    ips, sec, kind = cpu_reference_steps(c, steps, warmup)
    cores = os.cpu_count()
    line = {"impl": "reference", "metric": METRICS[c["kind"]], "value": ips, "unit": "images/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_block(c, args.gpus),
            "note": "the reference's CPU path (config cuda: False) on the host cores of this box, one process, all threads",
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": kind,
                             "sample": "the configured %d+%d images per step, %d timed steps after %d warm-up (%.2f s per step), torch fp32"
                                       % (c["n_l"], c["n_u"], steps, warmup, sec)},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ torch-eager incumbent
def incumbent_torch_eager(c, dev, steps=6, warm=3):
    """SURVEY 8d "second baseline": the reference's module graph (the same Conv2d / BatchNorm2d / LeakyReLU / Dropout /
    MaxPool2d / Upsample modules, wired as model/unet.py:12-117) and its Mean-Teacher step body in plain torch eager on this
    GPU with cudnn.benchmark = True (2017_03...:44), fp32 and autocast(bf16) + channels_last.  Reported, not the product."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import incumbent_baseline as ib
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    out = {}
    try:
        for amp in (False, True):
            ms, _ = ib.run(dev, steps, warm, amp, n_l=c["n_l"], n_u=c["n_u"], in_ch=c["in_ch"], n_cls=c["n_cls"])
            out["autocast_bf16_channels_last" if amp else "fp32"] = {"ms_per_step": ms, "images_per_s": (c["n_l"] + c["n_u"]) / ms * 1e3}
    finally:
        torch.backends.cudnn.benchmark = old
    out["note"] = "torch %s eager, cudnn.benchmark=True, same module graph and step body as the reference trainer" % torch.__version__
    return out


# ------------------------------------------------------------------------------------------------ GPU arm
def make_step(c, dev, graph_on, world):
    import torch
    import hpfg_b200 as hb
    torch.manual_seed(1337)                              # identical replicas on every rank
    a = hb.UNet(c["in_ch"], c["n_cls"], precision="bf16").to(dev)
    if c["kind"] == "cps":
        b = hb.UNet(c["in_ch"], c["n_cls"], precision="bf16").to(dev)
        step = hb.CPSStep(a, b)
    elif c["kind"] == "uamt":
        b = hb.UNet(c["in_ch"], c["n_cls"], precision="bf16").to(dev)      # a separately built teacher (2019_07...:55)
        step = hb.UAMTStep(a, b, T=c["T"])
    else:
        b = copy.deepcopy(a)
        step = hb.MeanTeacherStep(a, b)
    step.enable_graph(graph_on, data_parallel=world > 1)
    return step, a, b


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from hpfg_b200 import _lib as L

    c = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.lib()
    graph_on = not args.eager
    n_img = c["n_l"] + c["n_u"]

    x_cpu, y_cpu = synthetic_batch(c, 1337 + rank)          # rank-distinct data, weak scaling
    x_pin, y_pin = x_cpu.pin_memory(), y_cpu.pin_memory()
    x_dev, y_dev = x_pin.to(dev), y_pin.to(dev)
    loss_pin = torch.empty(1, dtype=torch.float32).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- data-parallel parity check (N > 1): the graph-replayed step with the NCCL all-reduces captured inside against the
    # same step launched eagerly, and replica consistency across ranks -- so the scaling record carries DP parity
    dp_check = None
    if world > 1:
        sa, ma, ea = make_step(c, dev, graph_on, world)
        sb, mb, eb = make_step(c, dev, False, world)
        dl = []
        extra = []
        if c["kind"] == "uamt":      # UAMT draws its input noise from the torch generator: the same draws for both replica sets
            gen = torch.Generator(device=dev).manual_seed(4242 + rank)
            n_u = c["n_u"]
            for _ in range(4):
                extra.append((torch.clamp(torch.randn((n_u, c["in_ch"], H, W), device=dev, generator=gen) * 0.1, -0.2, 0.2),
                              torch.clamp(torch.randn((c["T"] // 2, 2 * n_u, c["in_ch"], H, W), device=dev, generator=gen) * 0.1, -0.2, 0.2)))
        for k in range(4):
            la = sa.step(x_dev, y_dev, *(extra[k] if extra else ()))
            lb = sb.step(x_dev, y_dev, *(extra[k] if extra else ()))
            dl.append(abs(la.item() - lb.item()))
        barrier()

        def digest(t):
            return torch.stack([t.double().sum(), t.double().abs().sum(), (t.double() * (torch.arange(t.numel(), device=dev, dtype=torch.float64) % 7)).sum()])
        dg = torch.cat([digest(ma.flat_params), digest(ea.flat_params), digest(ma.bn_running if c["kind"] == "cps" else sa.mom)])
        allg = [torch.empty_like(dg) for _ in range(world)]
        dist.all_gather(allg, dg)
        same = all(torch.equal(allg[0][:6], g[:6]) for g in allg)         # parameters of both networks identical on every rank
        dp_check = {"steps": 4, "graph_vs_eager_max_abs_loss_diff": max(dl),
                    "graph_vs_eager_max_abs_param_diff": (ma.flat_params - mb.flat_params).abs().max().item(),
                    "replicas_identical_across_ranks": bool(same), "loss_step4": la.item(),
                    "note": "4 iterations on this rank's batch with two fresh replica sets: whole-step CUDA-graph replay incl. the "
                            "captured NCCL bucket all-reduces vs eager launches; parameter digests all-gathered and compared"}
        del sa, sb, ma, mb, ea, eb
        torch.cuda.empty_cache()

    step, student, other = make_step(c, dev, graph_on, world)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    def resident_step():
        return step.step(x_dev, y_dev)

    # End-to-end leg: every step's inputs start in pinned HOST memory and the step's loss is read back to the host and
    # waited for (the reference trainers call loss.item() every iteration).  The copy of step k+1's batch is enqueued
    # on a copy stream while step k computes (what a prefetching data loader does); all K copies and K loss
    # read-backs happen inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [(torch.empty_like(x_dev), torch.empty_like(y_dev)) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"k": 0, "primed": False}

    def enqueue_copy(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])            # the step that last read this slot has finished
            bufs[slot][0].copy_(x_pin, non_blocking=True)
            bufs[slot][1].copy_(y_pin, non_blocking=True)
            copied[slot].record(copy_stream)

    def e2e_step():
        k = state["k"]
        slot = k & 1
        if not state["primed"]:                               # first step of a timed run: its copy is not hidden
            enqueue_copy(slot)
            state["primed"] = True
        main = torch.cuda.current_stream()
        main.wait_event(copied[slot])
        loss = step.step(bufs[slot][0], bufs[slot][1])
        consumed[slot].record(main)
        enqueue_copy(slot ^ 1)                                # prefetch the next step's batch while this step computes
        loss_pin.copy_(loss.reshape(1), non_blocking=True)
        main.synchronize()                                    # the host consumes the loss every step
        state["k"] = k + 1

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        resident_step()
    launches0 = lib.hpfg_launch_count() + step.replayed_kernels
    ms = timed(resident_step, args.steps)
    launches = lib.hpfg_launch_count() + step.replayed_kernels - launches0      # host launches + kernel nodes replayed
    dumped = dump_outputs(args.dump_outputs, step) if args.dump_outputs and rank == 0 else None
    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    state["primed"] = False
    ms_e2e = timed(e2e_step, args.steps)
    if sampler:
        sampler.stop_flag = True
    images = n_img * world
    value = images * args.steps / (ms * 1e-3)
    e2e_value = images * args.steps / (ms_e2e * 1e-3)
    final_loss = step.last["scalars"][0].item()

    # ---- per-category device time (separate, untimed pass): roofline of the dominant kernel family
    prof_steps = 3
    step.enable_graph(False)
    step.serialize = True                                # no side streams: per-category times must not overlap
    resident_step()
    lib.hpfg_profile_begin()
    for _ in range(prof_steps):
        resident_step()
    cat_ms = (ctypes.c_double * 8)()
    cat_calls = (ctypes.c_int64 * 8)()
    lib.hpfg_profile_end(cat_ms, cat_calls)
    step.serialize = False

    def layer_us(op, cin, cout, ks, res, iters=20):
        ms_l = ctypes.c_float()
        L.check(lib.hpfg_conv_tc_bench(op, n_img, res, res, cin, cout, ks, iters, ctypes.byref(ms_l), L.stream_ptr(dev)), "hpfg_conv_tc_bench")
        return ms_l.value * 1e3
    names = ["conv_tcgen05", "conv_cuda_core", "wgrad_cuda_core", "bn_pool_upsample_glue", "ssl_loss", "sgd_ema", "weight_pack", "wgrad_tcgen05"]
    prof = {names[i]: {"ms_per_step": cat_ms[i] / prof_steps, "calls_per_step": cat_calls[i] / prof_steps} for i in range(8)}
    pk = peaks()

    if rank == 0:
        n_params = student.flat_params.numel()
        tc_flops = tc_conv_flops_per_step(c)
        tc_ms = prof["conv_tcgen05"]["ms_per_step"]
        achieved = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
        step_flops = flops_per_step(c)
        whole = value / images * step_flops / 1e12         # per-GPU TFLOP/s over the whole step (BASELINE.md's formula)
        main_cfg = world == 1 and not args.quick
        cpu = cpu_reference_steps(c, 5 if c["kind"] == "mt" else 3, 1) if world == 1 and not args.no_cpu else None
        # the single most expensive kernel instance: the 3x3 16->16 conv at 224x224; bound by HBM / shared-memory operand
        # bandwidth, not by the tensor pipe (DESIGN.md section 3): algorithmic bytes = bf16 in + out once
        top_bytes = n_img * H * W * (16 + 16) * 2.0
        top_us = layer_us(0, 16, 16, 3, H) if main_cfg else None
        layers = []
        if main_cfg:
            for cin, cout, ks, res in [(16, 16, 3, 224), (32, 16, 3, 224), (32, 32, 3, 112), (64, 64, 3, 56), (128, 64, 3, 56), (128, 128, 3, 28),
                                       (256, 128, 3, 28), (256, 256, 3, 14)]:
                px = n_img * res * res
                t3 = [layer_us(op, cin, cout, ks, res) for op in (0, 1, 2)]
                fl = 2.0 * px * cin * cout * ks * ks
                layers.append({"layer": "%dx%d conv %d->%d @%d" % (ks, ks, cin, cout, res), "fprop_us": t3[0], "dgrad_us": t3[1], "wgrad_us": t3[2],
                               "fprop_hbm_frac": px * (cin + cout) * 2.0 / (t3[0] * 1e-6) / 1e9 / pk["hbm"],
                               "fprop_tensor_frac": fl / (t3[0] * 1e-6) / 1e12 / pk["tf_burst"],
                               "dgrad_tensor_frac": fl / (t3[1] * 1e-6) / 1e12 / pk["tf_burst"],
                               "wgrad_tensor_frac": fl / (t3[2] * 1e-6) / 1e12 / pk["tf_burst"]})
        # SURVEY 8d: the 7.26 MB flat buffers are launch-latency dominated (and L2-resident), so the optimiser passes are also timed
        # as a pure HBM stream on x64 replicated buffers (464 MB per array): the bandwidth the same kernels reach once size is out of the way
        stream_x64 = None
        if world == 1 and c["kind"] == "mt":
            try:
                rep_n = n_params * 64
                bufs64 = [torch.randn(rep_n, device=dev) for _ in range(4)]
                p64, g64, m64, e64 = [ctypes.c_void_p(t.data_ptr()) for t in bufs64]
                sp = L.stream_ptr(dev)
                calls = {"ema_kernel (update_ema_variables, 12 B per parameter)": (12.0, lambda: lib.hpfg_ema_update(e64, p64, rep_n, 0.99, sp)),
                         "sgd_kernel<EMA> (SGD momentum + weight decay + EMA, 28 B per parameter)": (
                             28.0, lambda: lib.hpfg_sgd_momentum_ema(p64, g64, m64, e64, rep_n, 0.01, 0.9, 1e-4, 1.0, 0, 0.99, sp))}
                stream_x64 = []
                for name, (bpp, fn) in calls.items():
                    for _ in range(3):
                        L.check(fn(), name)
                    torch.cuda.synchronize()
                    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    ev0.record()
                    for _ in range(10):
                        L.check(fn(), name)
                    ev1.record()
                    torch.cuda.synchronize()
                    us = ev0.elapsed_time(ev1) / 10 * 1e3
                    gbs = rep_n * bpp / (us * 1e-6) / 1e9
                    stream_x64.append({"kernel": name, "bound": "hbm", "params": rep_n, "us_per_call": us, "achieved": gbs, "peak": pk["hbm"],
                                       "unit": "GB/s", "frac": gbs / pk["hbm"]})
                del bufs64
                torch.cuda.empty_cache()
            except Exception as exc:                     # a reported extra; never fails the bench line
                stream_x64 = {"error": str(exc)[:200]}
        cfg = config_block(c, world)
        line = {"metric": METRICS[c["kind"]], "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": cfg,
                "run": {"config_name": args.config, "launch": "cuda-graph replay" if graph_on else "eager (PDL)", "final_loss": final_loss},
                "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": x_pin.numel() * 4 + y_pin.numel() * 8, "d2h_bytes_per_step": 4},
                "gpu_launches": int(launches),
                "conv_tensor_fraction_of_step": {"achieved_tflops_whole_step": whole, "frac_of_burst_peak": whole / pk["tf_burst"],
                                                 "note": "images/s/GPU x algorithmic conv FLOPs per image (SURVEY 8d) over the WHOLE step time"},
                "roofline": {"kernel": "tc_conv_kernel (tcgen05 implicit-GEMM conv family: every fprop incl. in_conv.0 and the logits conv, dgrad, 1x1)",
                             "bound": "tensor", "achieved": achieved, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": achieved / pk["tf_burst"],
                             "traffic": CONV_FAMILY_DRAM_BYTES if args.config == "mt_acdc" else None,
                             "traffic_source": CONV_FAMILY_DRAM_SOURCE if args.config == "mt_acdc" else None,
                             "peak_source": pk["src"] + ", burst bf16", "launches_per_step": prof["conv_tcgen05"]["calls_per_step"],
                             "us_per_step": tc_ms * 1e3, "algorithmic_flops_per_step": tc_flops,
                             "note": "ALL tensor-core conv launches of a step (serialized profiling pass, CUDA events in the library) "
                                     "over the algorithmic FLOPs of exactly those launches (SURVEY 8d)"},
                "roofline_top_kernel": None if top_us is None else {
                    "kernel": "tc_conv_kernel<3,16,16,RES,MT=4,XF=1> (3x3 16->16 @224, fused BN+LeakyReLU loader, BN-stat epilogue)",
                    "bound": "hbm", "achieved": top_bytes / (top_us * 1e-6) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                    "frac": top_bytes / (top_us * 1e-6) / 1e9 / pk["hbm"], "us_per_launch": top_us,
                    "traffic": TOP_KERNEL_DRAM_BYTES, "traffic_source": "ncu --set full, profiles/r01_ncu_prof_fprop16_final_raw.txt (dram read+write per launch; the 51 MB output mostly stays in the 126 MB L2)"},
                "roofline_sgd_ema": _hbm_roofline(
                    "sgd_kernel (SGD momentum + weight decay (+ EMA teacher), one pass per network over the flat buffers)",
                    (28.0 if c["kind"] != "cps" else 2 * 20.0) * n_params, prof["sgd_ema"], pk,
                    "28 B per parameter with EMA: read p, g, m, ema; write p, m, ema (20 B without)"),
                "roofline_optimiser_x64_stream": stream_x64,
                "layer_table": layers,
                "kernel_time_per_step": prof,
                "clocks": sampler.summary() if sampler else None}
        if c["kind"] == "mt":
            line["roofline_loss"] = _hbm_roofline(
                "loss_mt_one_kernel (fused SSL loss value + dlogits in ONE launch per step: labeled Dice/CE sums | unlabeled consistency "
                "gradient | grid barrier | labeled gradient)",
                (n_img * c["n_cls"] * H * W * 4.0 * 2 + c["n_u"] * c["n_cls"] * H * W * 4.0 + c["n_l"] * H * W * 8.0),
                prof["ssl_loss"], pk, "SURVEY 8d: student logits read + teacher logits read + int64 labels read + dlogits written, each once",
                traffic=LOSS_DRAM_BYTES if args.config == "mt_acdc" else None,
                traffic_source="ncu --set full, profiles/r02b_loss_mt_one_ncu.txt (dram read+write of the launch, L2 flushed before the call: the dlogits mostly stay in L2)")
        if dp_check is not None:
            line["dp_check"] = dp_check
        if dumped is not None:
            line["outputs_dumped"] = {"dir": args.dump_outputs, "names": dumped}
        if cpu is not None:
            line["cpu_baseline"] = {"value": cpu[0], "unit": "images/s", "cores": os.cpu_count(), "kind": cpu[2],
                                    "sample": "the configured %d+%d images per step, %d timed steps after 1 warm-up (%.2f s per step), torch fp32, all host threads"
                                              % (c["n_l"], c["n_u"], 5 if c["kind"] == "mt" else 3, cpu[1])}
        if main_cfg and c["kind"] == "mt" and not args.no_incumbent:
            try:
                line["incumbent_torch_eager"] = incumbent_torch_eager(c, dev)
            except Exception as exc:                     # a reported extra; never fails the bench line
                line["incumbent_torch_eager"] = {"error": str(exc)[:200]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="mt_acdc", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-incumbent", action="store_true", help="skip the torch-eager incumbent leg")
    ap.add_argument("--quick", action="store_true", help="skip the per-layer table and the incumbent leg")
    ap.add_argument("--eager", action="store_true", help="launch every kernel from the host each step instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this repository's GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
