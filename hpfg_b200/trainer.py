"""Fused training steps for the three north-star trainers, built from the C-ABI calls only:

* ``MeanTeacherStep``  -- 2017_03_NIPS_Mean-Teacher_ACDC.py:89-113
* ``CPSStep``          -- 2021_06_CVPR_CPS_ACDC.py:90-120
* ``UAMTStep``         -- 2019_07_MICCAI_Uncertainty_Aware_ACDC.py:120-170
* ``ICTStep``          -- 2022_02_ISBI_ICT-MedSeg_ACDC.py:96-140 (SURVEY 8f.4)
* ``S4CVStep``         -- 2022_08_CVPR_S4CVNet_ACDC.py:108-167 (SURVEY 8f.4)
* ``HPFGStep``         -- main.py:128-207, the HPFG iteration itself (SURVEY 8f.2)

Each ``step()`` enqueues: student forward (activations kept in the plan), teacher/peer forward(s), ONE fused
loss launch pair (value + dlogits), backward into a persistent flat gradient buffer, (data parallel: NCCL
all-reduce of the gradient buckets on a side stream, overlapped with the rest of backward), and ONE fused
SGD-momentum or Adam / AdamW (+EMA) pass over the flat parameter buffers.  Nothing synchronises the host; the returned loss is
a device scalar.  Host-side schedules (Medical_LR, consistency ramp-up, EMA alpha) are python floats exactly as
in the reference (utils/scheduler/medical_lr.py:13-17, utils/utils.py:67-86)."""
import contextlib
import ctypes
import math

import torch

from . import _lib as L
from .optim import SGD, Adam
from .losses import ssl_loss_raw, ict_loss_raw, ict_mix_inputs, s4cv_loss_raw, cutmix_loss_raw, cutmix_mix_inputs, check_cutmix_batch
from .unet import FT_CHNS
from .utils import sigmoid_rampup, linear_rampup


def medical_lr(cur_itrs, base_lr, max_iterations):
    """Learning rate used at iteration ``cur_itrs`` (1-based) by Medical_LR constructed with last_epoch=-1."""
    return base_lr * (1.0 - (cur_itrs - 2) / max_iterations) ** 0.9


def gradient_buckets(in_channels, num_classes):
    """[(offset, count)] of the flat-gradient buckets in the order backward completes them (tail of the
    parameter list first: out_conv/up4/up3 | up2/up1 | down4/down3 | in_conv..down2: the last bucket, whose all-reduce cannot
    overlap backward, is the smallest)."""
    import ctypes
    offs, cnts = (ctypes.c_int64 * 4)(), (ctypes.c_int64 * 4)()
    L.check(L.lib().hpfg_unet_bucket_layout(in_channels, num_classes, offs, cnts), "hpfg_unet_bucket_layout")
    return [(int(o), int(c)) for o, c in zip(offs, cnts)]


def allreduce_flat_buckets(flat_grad, buckets, group=None, before_bucket=None, stream=None):
    """Sum-all-reduce ``flat_grad`` bucket by bucket (async), returning the work handles.  ``before_bucket(i)`` is
    called before bucket i is enqueued (the CUDA path makes the comm stream wait for that bucket's event there).
    Works for CPU tensors + gloo (host-logic tests) and CUDA tensors + NCCL alike."""
    import torch.distributed as dist
    works = []
    for i, (off, cnt) in enumerate(buckets):
        if before_bucket is not None:
            before_bucket(i)
        ctx = torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()
        with ctx:
            works.append(dist.all_reduce(flat_grad[off:off + cnt], group=group, async_op=True))
    return works


def allreduce_tensor_list(tensors, group=None):
    """Sum-all-reduce a list of (small) tensors as ONE flat buffer and scatter the sums back in place: the neck gradients of a
    UNet_Plus (16 tensors) travel as one collective instead of 16.  CPU + gloo and CUDA + NCCL alike."""
    import torch.distributed as dist
    tensors = [t for t in tensors if t is not None]
    if not tensors:
        return
    flat = torch.cat([t.reshape(-1) for t in tensors])
    dist.all_reduce(flat, group=group)
    off = 0
    for t in tensors:
        t.copy_(flat[off:off + t.numel()].view_as(t))
        off += t.numel()


def shard_batch(x_l, x_u, y, rank, world):
    """Data-parallel split that keeps the labeled:unlabeled ratio per rank (both sub-batches are split, because the
    supervised and consistency terms normalise over their own pixels)."""
    n_l, n_u = x_l.shape[0], x_u.shape[0]
    assert n_l % world == 0 and n_u % world == 0, "labeled and unlabeled batch sizes must divide by the world size"
    a, b = n_l // world, n_u // world
    return x_l[rank * a:(rank + 1) * a], x_u[rank * b:(rank + 1) * b], y[rank * a:(rank + 1) * a]


def _input_noise(shape, like):
    """Clamped Gaussian perturbation of a teacher's input (2019_07...:130,141; 2022_08...:111), ONE draw of ``shape``."""
    return torch.clamp(torch.randn(shape, device=like.device, dtype=like.dtype) * 0.1, -0.2, 0.2)


class _StepBase:
    serialize = False             # profiling: every network on the calling stream, so per-category kernel times do not overlap

    OPTIMIZERS = {"sgd": SGD, "adam": Adam, "adamw": Adam}

    def __init__(self, *, lr=0.01, momentum=0.9, weight_decay=1e-4, total_itrs=30000, consistency=0.1,
                 consistency_rampup=200.0, process_group=None, exact_global=False, optimizer="sgd", betas=(0.9, 0.999),
                 eps=1e-8):
        """optimizer: "sgd" (torch.optim.SGD with ``momentum``), "adam" (torch.optim.Adam: L2 weight decay) or "adamw"
        (torch.optim.AdamW: decoupled weight decay) with ``betas`` / ``eps``, as the reference's optimiser factory builds
        them (utils/__init__.py:13-49); ``weight_decay`` applies to all three."""
        if optimizer not in self.OPTIMIZERS:
            raise ValueError("optimizer must be one of %s, got %r" % (", ".join(self.OPTIMIZERS), optimizer))
        self.base_lr, self.momentum, self.weight_decay = lr, momentum, weight_decay
        self.optimizer = optimizer
        self.total_itrs, self.consistency, self.consistency_rampup = total_itrs, consistency, consistency_rampup
        self.cur_itrs = 0
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self._comm = None
        self.last = {}
        # Data parallel semantics (SURVEY 8e): default = what wrapping the reference in DDP gives (BatchNorm / Dice / CE /
        # consistency means over each rank's shard, gradients averaged).  exact_global=True = the single-GPU reference on the
        # CONCATENATED batch: BatchNorm statistics (forward and backward) and the loss sums are all-reduced over the ranks
        # through the library's hook, parameter gradients are summed.  Eager launches only (one small all-reduce per BatchNorm).
        self.exact_global = bool(exact_global) and self.world > 1
        self._grad_scale = 1.0 if self.exact_global else 1.0 / self.world
        if self.exact_global:
            L.install_allreduce_hook(self.pg)
        self._opt = self.OPTIMIZERS[optimizer](optimizer, lr, momentum, weight_decay, betas, eps, self._grad_scale)
        self._neck_states = {}      # id(parameter) -> OptState of the parameters outside the flat buffers (_neck_params)

    def _setup(self, trained, networks, train=None, grads=True):
        """Construction shared by the drivers.  trained: the networks this driver optimises, in checkpoint order, each given a
        flat optimiser state and (unless autograd produces its gradients, grads=False) a flat gradient buffer; networks: every
        network of the step, in the order of the checkpointed Philox offsets; train: the networks put in train() mode (default:
        the trained ones).  Returns [(gradient buffer, optimiser buffers)] in the order of ``trained``: the momentum buffer
        (SGD) or the pair (exp_avg, exp_avg_sq) (Adam / AdamW)."""
        self.in_channels, self.num_classes = trained[0].in_channels, trained[0].num_classes
        for m in trained if train is None else train:
            m.train()
        for m in networks:
            m.ensure_flat()
        self._trained = [(m, torch.zeros_like(m.flat_params) if grads else None, self._opt.new_state(m.flat_params))
                         for m in trained]
        self._networks = list(networks)
        self._check_buffers()
        self._broadcast_from_rank0()
        return [(g, s.bufs[0] if len(s.bufs) == 1 else s.bufs) for _, g, s in self._trained]

    # ------------------------------------------------------------------ CUDA-graph replay of the whole step
    _graph_enabled = False
    _graph_dp = False
    kernels_per_replay = 0
    replayed_kernels = 0          # kernels executed through graph replays (the library's own counter sees host launches only)

    def enable_graph(self, enabled=True, data_parallel=False):
        """From the second iteration on, replay the step as ONE captured CUDA graph (all forwards on their streams, the
        fused loss, backward with its side-stream weight gradients, fused SGD(+EMA)).  The scalars that change per
        iteration -- learning rate, EMA alpha, consistency weight, UAMT threshold, dropout Philox offsets -- live in a
        small device block that is refreshed before every replay (the `_dv` entry points read them at run time).
        data_parallel=True also captures the bucketed NCCL all-reduces of a multi-process run (HPFGStep: the all-reduces of
        its flat and neck gradients); by default a data-parallel step stays eager, and so does the exact-global mode.
        HPFGStep captures once every optimiser state, flat and neck, has taken its first update (see its _use_graph).
        S4CVStep always launches eagerly."""
        self._graph_enabled = bool(enabled)
        self._graph_dp = bool(data_parallel)      # also capture the NCCL bucket all-reduces (torch >= 2.x captures NCCL work)
        if not enabled:
            self._ggraph = None
            self._gsig = None

    def _next_iteration(self):
        """Start of every step(): the iteration counter, the step counts of the flat optimiser states (every U-Net tensor
        gets a gradient every iteration; advanced on the host, so that graph replays see them move), and the buffer check."""
        self.cur_itrs += 1
        for _, _, state in self._trained:
            state.step += 1
        self._check_buffers()

    def _use_graph(self):
        dp_ok = self.world == 1 or self._graph_dp
        return self._graph_enabled and self.cur_itrs >= 2 and dp_ok and not self.exact_global

    @contextlib.contextmanager
    def _global_sums(self):
        """Loss sums over the batch of all ranks while a fused loss call is enqueued (exact-global mode; no-op otherwise)."""
        if not self.exact_global:
            yield
            return
        L.check(L.lib().hpfg_ssl_loss_set_global_sums(1), "hpfg_ssl_loss_set_global_sums")
        try:
            yield
        finally:
            L.check(L.lib().hpfg_ssl_loss_set_global_sums(0), "hpfg_ssl_loss_set_global_sums")

    def _global_consistency_value(self, scalars, w):
        """Mean-Teacher / ICT in exact-global mode: the kernel's consistency value is this rank's share of the global mean."""
        if self.exact_global:
            torch.distributed.all_reduce(scalars[2:3], group=self.pg)
            scalars[0:1].copy_(scalars[1:2] + w * scalars[2:3])

    def _graph_replay(self, inputs, dyn_f, fwd_models, body):
        """Generic capture-once / replay driver (all step drivers).
        inputs: tensors copied into static buffers before each replay; dyn_f: python floats for the device block
        (fp32); fwd_models: the network of each forward in the order the body enqueues them -> one Philox-offset slot each
        (the offsets advance exactly as eager launches advance them); body(static_inputs, dv) enqueues the step with
        dv = (device block, Philox-offset slots) and returns its output dict (static tensors).

        The per-iteration scalars travel through a RING of pinned host slots: an async H2D copy reads pinned memory when
        the stream reaches it, not at enqueue time, so a slot is only rewritten after the event recorded behind its copy
        has completed (the host may run up to `_RING` replays ahead of the device without syncing).
        The captured graph bakes in raw pointers (flat parameters, BN buffers, plan workspaces, gradient / momentum
        buffers): they are part of the signature, and a change (`.to()`, `load_state_dict(assign=True)`, ...) drops the
        graph and captures again."""
        dev = inputs[0].device
        models = []
        for m in fwd_models:
            if not any(m is q for q in models):
                models.append(m)
        for m in models:
            m.ensure_flat(quick=True)
        ptrs = tuple((m.flat_params.data_ptr(), m.bn_running.data_ptr(), m.bn_counters.data_ptr(), id(m._plans)) for m in models)
        ptrs += tuple(t.data_ptr() for _, g, s in self._trained for t in (g,) + s.bufs if t is not None)
        ptrs += self._graph_ptrs()
        # (the dropout seed is a by-value launch argument: a re-seeded generator needs a new capture)
        ptrs += (torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()].initial_seed(),)
        sig = tuple((tuple(t.shape), t.dtype) for t in inputs) + (len(dyn_f), len(fwd_models), ptrs)
        if getattr(self, "_gsig", None) != sig:
            self._gin = [torch.empty_like(t) for t in inputs]
            self._gf = torch.zeros(len(dyn_f), device=dev, dtype=torch.float32)
            self._go = torch.zeros(len(fwd_models), device=dev, dtype=torch.int64)
            self._ring = [(torch.zeros(len(dyn_f), dtype=torch.float32).pin_memory(),
                           torch.zeros(len(fwd_models), dtype=torch.int64).pin_memory(), torch.cuda.Event())
                          for _ in range(self._RING)]
            self._ring_used = [False] * self._RING
            self._ring_pos = 0
            self._ggraph, self._gsig = None, sig
        k = self._ring_pos
        self._ring_pos = (k + 1) % self._RING
        f_host, o_host, ev = self._ring[k]
        if self._ring_used[k]:
            ev.synchronize()               # only blocks when the host is a whole ring ahead of the device
        for i, v in enumerate(dyn_f):
            f_host[i] = v
        for i, m in enumerate(fwd_models):
            o_host[i] = m._philox_offset
            if m.training:
                m._philox_offset += 8
        self._gf.copy_(f_host, non_blocking=True)
        self._go.copy_(o_host, non_blocking=True)
        ev.record()
        self._ring_used[k] = True
        for s, t in zip(self._gin, inputs):
            s.copy_(t, non_blocking=True)
        if self._ggraph is None:
            g = torch.cuda.CUDAGraph()
            n0 = L.lib().hpfg_launch_count()
            try:
                with torch.cuda.graph(g):
                    self._gout = self._body_on_device_block(body, fwd_models)
            except Exception as exc:        # capture not possible here (e.g. a collective that refuses capture): stay eager
                import warnings
                warnings.warn("hpfg_b200: CUDA-graph capture of the step failed (%s); falling back to eager launches" % exc)
                self._graph_enabled, self._ggraph = False, None
                torch.cuda.synchronize()
                return self._body_on_device_block(body, fwd_models)
            self._ggraph = g
            self.kernels_per_replay = int(L.lib().hpfg_launch_count() - n0)   # kernel nodes of the captured step
        self._ggraph.replay()
        self.replayed_kernels += self.kernels_per_replay
        return self._gout

    _RING = 8

    def _graph_ptrs(self):
        """Further raw pointers a captured step bakes in (part of the graph signature); none beyond the networks' and the
        flat optimiser buffers for the drivers without tensors outside the flat buffers."""
        return ()

    def _body_on_device_block(self, body, fwd_models):
        """Enqueue body with every per-iteration scalar read from the device block; _forward takes the Philox slots of
        ``fwd_models`` in call order."""
        self._slots, self._slot = fwd_models, 0
        out = body(self._gin, (self._gf, self._go))
        assert self._slot == len(fwd_models), "the step ran %d forwards for %d Philox slots" % (self._slot, len(fwd_models))
        return out

    # ------------------------------------------------------------------ checkpoint / resume (2017_03...:126-133)
    def state_dict(self):
        """{cur_itrs, philox offsets, optimizer}: `optimizer` holds one torch.optim state dict per trained network, its
        per-parameter state in model.parameters() order (the flat buffer's tensors, then the ones outside it) so that a
        reference checkpoint's optimizer state and this driver's flat buffers interchange: state[i] = {momentum_buffer}
        (torch.optim.SGD) or {step, exp_avg, exp_avg_sq} (torch.optim.Adam / AdamW).  SGD state appears from the first
        iteration on, Adam state once it has taken a step; tensors that never received a gradient have none, as in torch."""
        out = {"cur_itrs": self.cur_itrs, "philox": [m._philox_offset for m in self._networks], "optimizers": []}
        lr = medical_lr(self.cur_itrs + 1, self.base_lr, self.total_itrs)
        for model, _, state in self._trained:
            entries = {i: self._opt.entry(state.step, [b[o:o + n].view(shape) for b in state.bufs])
                       for i, (o, n, shape) in enumerate(model._layout)} if self._opt.has_state(state, self.cur_itrs) else {}
            necks = self._neck_params(model)
            for j, p in enumerate(necks):
                s = self._neck_states.get(id(p))
                if s is not None and self._opt.has_state(s, self.cur_itrs):
                    entries[len(model._layout) + j] = self._opt.entry(s.step, s.bufs)
            out["optimizers"].append({"state": entries,
                                      "param_groups": [self._opt.param_group(lr, len(model._layout) + len(necks))]})
        return out

    def load_state_dict(self, sd):
        """Everything is checked before anything changes: a checkpoint of the other optimiser kind, or one whose U-Net tensors
        carry different Adam step counts, raises and leaves the driver as it was."""
        cur_itrs, opts = int(sd["cur_itrs"]), sd.get("optimizers", [])
        for opt in opts:
            self._opt.check_kind(opt)
        steps = [self._opt.checkpoint_step([opt["state"].get(i) for i in range(len(model._layout))], k, cur_itrs)
                 for k, ((model, _, _), opt) in enumerate(zip(self._trained, opts))]
        self.cur_itrs = cur_itrs
        for m, off in zip(self._networks, sd.get("philox", [])):
            m._philox_offset = int(off)
        self._neck_states = {}
        for k, ((model, _, state), opt, step) in enumerate(zip(self._trained, opts, steps)):
            state.step = step
            for b in state.bufs:
                b.zero_()
            for i, (o, n, _) in enumerate(model._layout):
                self._opt.load_entry(opt["state"].get(i), [b[o:o + n] for b in state.bufs])
            for j, p in enumerate(self._neck_params(model)):
                st = opt["state"].get(len(model._layout) + j)
                if st is not None and all(st.get(key) is not None for key in self._opt.KEYS):
                    s = self._neck_states[id(p)] = self._opt.new_state(p.data)
                    s.step = self._opt.checkpoint_step([st], k, cur_itrs)
                    self._opt.load_entry(st, s.bufs)

    def _check_buffers(self):
        """The flat gradient / optimiser buffers must match the (possibly re-flattened or moved) parameter buffer."""
        for model, g, state in self._trained:
            flat = model.flat_params
            for what, buf in zip(("gradient",) + self._opt.KEYS, (g,) + state.bufs):
                if buf is not None and (buf.device != flat.device or buf.numel() != flat.numel()):
                    raise L.HpfgError("step driver buffer %s (%s, %d) no longer matches the model's flat parameters (%s, %d): "
                                      "build the step driver after moving the model"
                                      % (what, buf.device, buf.numel(), flat.device, flat.numel()))
            if flat.is_cuda and flat.device.index != torch.cuda.current_device():
                raise L.HpfgError("the model lives on %s but the current CUDA device is %d: call torch.cuda.set_device first "
                                  "(the library launches on the current device)" % (flat.device, torch.cuda.current_device()))

    def _broadcast_from_rank0(self):
        """Data parallel: every rank starts from rank 0's parameters / BN buffers (what DDP does at construction), the
        tensors outside the flat buffers included."""
        if self.world <= 1:
            return
        import torch.distributed as dist
        for m in self._networks:
            m.ensure_flat()
            for t in (m.flat_params, m.bn_running, m.bn_counters, *(p.data for p in self._neck_params(m))):
                dist.broadcast(t, src=dist.get_global_rank(self.pg, 0) if self.pg is not None else 0, group=self.pg)

    @staticmethod
    def _neck_params(model):
        """The parameters of ``model`` outside its flat buffer, in parameters() order (a UNet_Plus: its 16 projection-neck
        tensors after the 82 U-Net tensors; a UNet: none).  Each gets an optimiser state when it first has a gradient."""
        core = {id(q) for q in model._flat_params_list}
        return [p for p in model.parameters() if id(p) not in core]

    # Two forwards enqueued on two streams share the machine: half of the SMs each (hpfg_unet_plan_set_forward_ctas).  Only the
    # drivers whose two streams carry about the same forward work do this (Mean-Teacher, CPS, ICT); with unbalanced streams
    # (UAMT: one student forward next to five teacher forwards; S4CVNet) the longer stream would finish on half a machine.
    SHARED_FORWARD_CTAS = 74
    share_forward = True
    sync_bn_exact_global = True     # exact-global mode: the plans' BatchNorm statistics are all-reduced (SyncBN)

    def _set_forward_share(self, plan, shared):
        if self.exact_global and self.sync_bn_exact_global and not getattr(plan, "sync_bn", False):
            L.check(L.lib().hpfg_unet_plan_set_sync_bn(plan.handle, 1), "hpfg_unet_plan_set_sync_bn")
            plan.sync_bn = True
        want = self.SHARED_FORWARD_CTAS if shared else 0
        if getattr(plan, "fwd_ctas", 0) != want:
            L.check(L.lib().hpfg_unet_plan_set_forward_ctas(plan.handle, want), "hpfg_unet_plan_set_forward_ctas")
            plan.fwd_ctas = want

    def _lr(self):
        return medical_lr(self.cur_itrs, self.base_lr, self.total_itrs)

    def _dyn_scalars(self, ema_decay=None, *extra):
        """The device block: [lr, ema_alpha, 1 - ema_alpha (fp32 subtraction, as the by-value entry point), consistency
        weight, *extra (UAMT: its threshold)], then the optimiser's group of each trained network in the order of ``_trained``
        and of each state of a tensor outside the flat buffers (HPFGStep's neck tensors; SGD: none; Adam / AdamW: [step_size,
        bc2_sqrt, decay_factor, ema_alpha, 1 - ema_alpha]), whose offset its state records."""
        alpha = min(1 - 1 / (self.cur_itrs + 1), ema_decay) if ema_decay is not None else 0.0
        one_minus = float(1.0 - torch.tensor(alpha, dtype=torch.float32))
        lr = self._lr()
        out = [lr, alpha, one_minus, self._consistency_weight(), *extra]
        for state in [s for _, _, s in self._trained] + list(self._neck_states.values()):
            state.dv_offset = len(out)
            out += self._opt.device_group(state.step, lr, alpha, one_minus)
        return out

    @staticmethod
    def _dv_scalar(dv, i):
        """Entry i of the device block during capture, None for eager launches."""
        return None if dv is None else dv[0][i:i + 1]

    def _side_stream(self, device):
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(device=device)
        return self._side

    def _fork(self, device):
        """(main, side): the calling stream and the stream the other network(s) run on (the same one when ``serialize`` is
        set), the side stream ordered after everything enqueued so far."""
        main = torch.cuda.current_stream(device)
        side = main if self.serialize else self._side_stream(device)
        side.wait_stream(main)
        return main, side

    def _consistency_weight(self):
        return self.consistency * sigmoid_rampup(self.cur_itrs // 150, self.consistency_rampup)

    def _forward(self, model, x, save, out, dv):
        """One network forward into ``out`` (activations kept in the plan when ``save``).  Eager launches (dv None) use the
        model's Philox offset; during capture the offset is read from the next slot of the device block."""
        if dv is None:
            model.ensure_flat(quick=True)          # (captures: _graph_replay has checked every network)
            offset_dev = None
        else:
            assert self._slots[self._slot] is model, "forward %d does not run the network of its Philox slot" % self._slot
            offset_dev = dv[1][self._slot:self._slot + 1]
            self._slot += 1
        plan = model._acquire_plan(x, need_grad=save)
        self._set_forward_share(plan, self.share_forward and not self.serialize)
        return plan, model._run_forward(plan, x, save=save, out=out, offset_dev=offset_dev)

    def _persistent(self, name, shape, device):
        """Step-persistent fp32 buffer (no per-step allocation: tensors that cross streams would otherwise need
        record_stream, which defeats the caching allocator when the host runs ahead of the device)."""
        buf = self.__dict__.setdefault("_bufs", {}).get(name)
        if buf is None or tuple(buf.shape) != tuple(shape) or buf.device != device:
            buf = torch.empty(shape, device=device, dtype=torch.float32)
            self._bufs[name] = buf
        return buf

    def _backward(self, model, plan, dlogits, grads):
        L.check(L.lib().hpfg_unet_backward(plan.handle, L.ptr(model.flat_params), L.ptr(dlogits), L.ptr(grads), 0,
                                           L.stream_ptr(grads.device)), "hpfg_unet_backward")
        if self.world > 1:
            self._allreduce_buckets(plan, grads)

    def _allreduce_buckets(self, plan, grads):
        """Bucketed gradient all-reduce overlapped with the tail of backward: the comm stream waits on the
        per-bucket events the plan recorded, NCCL runs there, the compute stream joins before the SGD pass."""
        import ctypes
        if self._comm is None:
            self._comm = torch.cuda.Stream(device=grads.device)
            self._buckets = gradient_buckets(self.in_channels, self.num_classes)
        lib = L.lib()
        comm = ctypes.c_void_p(self._comm.cuda_stream)
        works = allreduce_flat_buckets(
            grads, self._buckets, self.pg, stream=self._comm,
            before_bucket=lambda b: L.check(lib.hpfg_unet_bucket_wait(plan.handle, b, comm), "hpfg_unet_bucket_wait"))
        for w in works:
            w.wait()            # stream-level wait on the compute stream, not a host sync

    def _opt_step(self, trained, dv, ema_model=None):
        """The optimiser step of one ``_trained`` entry (network, gradient buffer, optimiser state) over its flat buffers, with
        the EMA of the network into ``ema_model`` in the same pass if given.  Eager launches take this iteration's scalars by
        value; captures read them from the device block."""
        model, grads, state = trained
        alpha = min(1 - 1 / (self.cur_itrs + 1), self.ema_decay) if ema_model is not None else 0.0      # utils/utils.py:84
        self._opt.launch(model.flat_params, grads, state, None if ema_model is None else ema_model.flat_params, self._lr(),
                         alpha, None if dv is None else dv[0], L.stream_ptr(grads.device))


class MeanTeacherStep(_StepBase):
    def __init__(self, model, ema_model, *, ema_decay=0.99, **kw):
        super().__init__(**kw)
        self.model, self.ema_model, self.ema_decay = model, ema_model, ema_decay
        # the teacher runs in train() mode (2017_03...:70)
        [(self.grads, self.mom)] = self._setup([model], [model, ema_model], train=[model, ema_model])

    def step(self, x, labels):
        """x: [n_l+n_u, C, H, W] fp32 CUDA (labeled slices first); labels: [n_l, H, W] int64 CUDA."""
        self._next_iteration()
        ins = [x, labels]
        out = (self._graph_replay(ins, self._dyn_scalars(self.ema_decay), [self.ema_model, self.model], self._body)
               if self._use_graph() else self._body(ins, None))
        self.last = dict(out, lr=self._lr(), w=self._consistency_weight())
        return out["scalars"][0]

    def _body(self, ins, dv):
        x, labels = ins
        n_l, dev = labels.shape[0], x.device
        shape = (x.shape[0], self.num_classes, x.shape[2], x.shape[3])
        # the teacher forward is independent of the student forward: it runs on a side stream so that each network's
        # small / dependent kernels fill the other's bubbles (the teacher sees the whole batch, 2017_03...:100)
        main, side = self._fork(dev)
        with torch.cuda.stream(side):
            _, t_out = self._forward(self.ema_model, x, False, self._persistent("t_out", shape, dev), dv)
        plan, out = self._forward(self.model, x, True, self._persistent("s_out", shape, dev), dv)
        main.wait_stream(side)
        w = self._consistency_weight()
        with self._global_sums():
            r = ssl_loss_raw(L.LOSS_MT, out, t_out[n_l:], labels, n_l, cons_weight=w, cons_weight_dev=self._dv_scalar(dv, 3))
        self._global_consistency_value(r["scalars"], w)
        self._backward(self.model, plan, r["dstudent"], self.grads)
        self._opt_step(self._trained[0], dv, self.ema_model)
        return dict(scalars=r["scalars"], logits=out, teacher_logits=t_out)


class CPSStep(_StepBase):
    def __init__(self, model1, model2, **kw):
        super().__init__(**kw)
        self.m1, self.m2 = model1, model2
        (self.g1, self.b1), (self.g2, self.b2) = self._setup([model1, model2], [model1, model2])

    def step(self, x, labels):
        self._next_iteration()
        ins = [x, labels]
        out = (self._graph_replay(ins, self._dyn_scalars(), [self.m2, self.m1], self._body)
               if self._use_graph() else self._body(ins, None))
        self.last = dict(out, lr=self._lr(), w=self._consistency_weight())
        return out["scalars"][0]

    def _body(self, ins, dv):
        x, labels = ins
        n_l, dev = labels.shape[0], x.device
        shape = (x.shape[0], self.num_classes, x.shape[2], x.shape[3])
        # the two networks are independent except for the loss: network 2 runs on a side stream (forward, then backward + SGD)
        main, side = self._fork(dev)
        with torch.cuda.stream(side):
            p2, o2 = self._forward(self.m2, x, True, self._persistent("o2", shape, dev), dv)
        p1, o1 = self._forward(self.m1, x, True, self._persistent("o1", shape, dev), dv)
        main.wait_stream(side)
        w = self._consistency_weight()
        with self._global_sums():
            r = ssl_loss_raw(L.LOSS_CPS, o1, o2, labels, n_l, cons_weight=w, cons_weight_dev=self._dv_scalar(dv, 3),
                             want_pseudo=False)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            self._backward(self.m2, p2, r["dother"], self.g2)
            self._opt_step(self._trained[1], dv)
        self._backward(self.m1, p1, r["dstudent"], self.g1)
        self._opt_step(self._trained[0], dv)
        main.wait_stream(side)
        return dict(scalars=r["scalars"], logits1=o1, logits2=o2)


class UAMTStep(_StepBase):
    share_forward = False

    def __init__(self, model, ema_model, *, ema_decay=0.99, T=8, **kw):
        super().__init__(**kw)
        self.model, self.ema_model, self.ema_decay, self.T = model, ema_model, ema_decay, T
        [(self.grads, self.mom)] = self._setup([model], [model, ema_model], train=[model, ema_model])

    def _threshold(self):
        """Entropy threshold of the certainty mask (2019_07...:150)."""
        return (0.75 + 0.25 * sigmoid_rampup(self.cur_itrs, self.total_itrs)) * math.log(2)

    def step(self, x, labels, noise=None, mc_noise=None, teacher_masks=None):
        """noise [n_u,...] / mc_noise [T//2, 2*n_u, ...]: the clamped perturbations; each drawn here (one draw) if None.
        teacher_masks (parity harness only, eager launches): 1 + T//2 dropout keep-mask sets, one per teacher forward in call
        order (the consistency forward on n_u slices, then the T//2 Monte-Carlo forwards on 2*n_u slices) -- every
        stochastic teacher pass draws its own masks, as nn.Dropout does in the reference (2019_07...:134-143)."""
        self._next_iteration()
        x_u = x[labels.shape[0]:]
        if noise is None:
            noise = _input_noise(x_u.shape, x_u)
        if mc_noise is None:
            mc_noise = _input_noise((self.T // 2, 2 * x_u.shape[0]) + tuple(x_u.shape[1:]), x_u)
        self._teacher_masks = None
        if teacher_masks is not None:
            assert len(teacher_masks) == 1 + self.T // 2, "one mask set per teacher forward"
            self._teacher_masks = []       # uploaded on the calling stream before the fork; kept alive until the next step
            for ms in teacher_masks:
                self.ema_model.set_dropout_masks(ms)
                self._teacher_masks.append(self.ema_model._dropout_masks)
        ins = [x, labels, noise, mc_noise.contiguous()]
        thr = self._threshold()
        if teacher_masks is None and self._use_graph():
            out = self._graph_replay(ins, self._dyn_scalars(self.ema_decay, thr),
                                     [self.ema_model] * (1 + self.T // 2) + [self.model], self._body)
        else:
            out = self._body(ins, None)
        self.last = dict(out, lr=self._lr(), w=self._consistency_weight(), threshold=thr)
        return out["scalars"][0]

    def _body(self, ins, dv):
        x, labels, noise, mc_noise = ins
        n_l, dev = labels.shape[0], x.device
        x_u = x[n_l:]
        n_u = x_u.shape[0]
        xr = x_u.repeat(2, 1, 1, 1)
        x_t = (x_u + noise).contiguous()
        x_mc = [(xr + mc_noise[i]).contiguous() for i in range(self.T // 2)]
        ncls, hh, ww = self.num_classes, x.shape[2], x.shape[3]
        mc = self._persistent("mc", (self.T * n_u, ncls, hh, ww), dev)
        # the five teacher forwards are independent of the student forward: side stream
        main, side = self._fork(dev)
        with torch.cuda.stream(side):
            t_out = self._persistent("t_out", (n_u, ncls, hh, ww), dev)
            outs = [t_out] + [mc[2 * n_u * i:2 * n_u * (i + 1)] for i in range(self.T // 2)]
            for i, (xi, oi) in enumerate(zip([x_t] + x_mc, outs)):
                if self._teacher_masks is not None:
                    self.ema_model._dropout_masks = self._teacher_masks[i]
                self._forward(self.ema_model, xi, False, oi, dv)
        plan, out = self._forward(self.model, x, True, self._persistent("s_out", (x.shape[0], ncls, hh, ww), dev), dv)
        main.wait_stream(side)
        w = self._consistency_weight()
        with self._global_sums():
            r = ssl_loss_raw(L.LOSS_UAMT, out, t_out, labels, n_l, cons_weight=w, mc_logits=mc, mc_passes=self.T,
                             uamt_threshold=self._threshold(), cons_weight_dev=self._dv_scalar(dv, 3),
                             uamt_threshold_dev=self._dv_scalar(dv, 4))
        self._backward(self.model, plan, r["dstudent"], self.grads)
        self._opt_step(self._trained[0], dv, self.ema_model)
        return dict(scalars=r["scalars"], logits=out, teacher_logits=t_out, mc_logits=mc)


class ICTStep(_StepBase):
    """Interpolation consistency training (2022_02_ISBI_ICT-MedSeg_ACDC.py:96-140): the student sees the labeled slices
    and a per-sample mix of the two halves of the unlabeled batch; the EMA teacher sees the two un-mixed halves (two
    forwards, as in the reference, so each has its own BatchNorm batch statistics) and the consistency target is the same
    mix of its two softmaxes."""

    def __init__(self, model, ema_model, *, ema_decay=0.99, ict_alpha=0.2, **kw):
        super().__init__(**kw)
        self.model, self.ema_model, self.ema_decay, self.ict_alpha = model, ema_model, ema_decay, ict_alpha
        [(self.grads, self.mom)] = self._setup([model], [model, ema_model])

    def draw_mix_factors(self, n_mixed):
        """np.random.beta(alpha, alpha, size=(n_u//2,1,1,1)) (2022_02...:112-113): host RNG, as in the reference."""
        import numpy as np
        return torch.tensor(np.random.beta(self.ict_alpha, self.ict_alpha, size=(n_mixed,)), dtype=torch.float)

    def step(self, x, labels, mix_factors=None):
        """x: [n_l+n_u, C, H, W] (labeled first, n_u even); mix_factors: [n_u//2] floats (drawn here if None)."""
        self._next_iteration()
        n_u = x.shape[0] - labels.shape[0]
        assert n_u % 2 == 0, "ICT needs an even unlabeled batch"
        if mix_factors is None:
            mix_factors = self.draw_mix_factors(n_u // 2)
        lam = mix_factors.reshape(-1).to(device=x.device, dtype=torch.float32, non_blocking=True).contiguous()
        ins = [x, labels, lam]
        out = (self._graph_replay(ins, self._dyn_scalars(self.ema_decay), [self.ema_model, self.ema_model, self.model], self._body)
               if self._use_graph() else self._body(ins, None))
        self.last = dict(out, lr=self._lr(), w=self._consistency_weight(), mix_factors=lam)
        return out["scalars"][0]

    def _body(self, ins, dv):
        x, labels, lam = ins
        n_l, dev = labels.shape[0], x.device
        n_m = (x.shape[0] - n_l) // 2
        ux0, ux1 = x[n_l:n_l + n_m], x[n_l + n_m:]
        ncls, hh, ww = self.num_classes, x.shape[2], x.shape[3]
        main, side = self._fork(dev)
        t_out = self._persistent("t_out", (2 * n_m, ncls, hh, ww), dev)
        with torch.cuda.stream(side):            # the two teacher forwards are independent of the student forward
            self._forward(self.ema_model, ux0, False, t_out[:n_m], dv)
            self._forward(self.ema_model, ux1, False, t_out[n_m:], dv)
        x_in = self._persistent("x_in", (n_l + n_m,) + tuple(x.shape[1:]), dev)
        x_in[:n_l].copy_(x[:n_l])
        L.check(L.lib().hpfg_ict_mix(L.ptr(ux0), L.ptr(ux1), L.ptr(lam), n_m, ux0[0].numel(), L.ptr(x_in[n_l:]),
                                     L.stream_ptr(dev)), "hpfg_ict_mix")
        plan, out = self._forward(self.model, x_in, True, self._persistent("s_out", (n_l + n_m, ncls, hh, ww), dev), dv)
        main.wait_stream(side)
        w = self._consistency_weight()
        with self._global_sums():
            r = ict_loss_raw(out, t_out, lam, labels, n_l, cons_weight=w, cons_weight_dev=self._dv_scalar(dv, 3))
        self._global_consistency_value(r["scalars"], w)
        self._backward(self.model, plan, r["dstudent"], self.grads)
        self._opt_step(self._trained[0], dv, self.ema_model)
        return dict(scalars=r["scalars"], logits=out, teacher_logits=t_out)


class S4CVStep(_StepBase):
    """S4CVNet (2022_08_CVPR_S4CVNet_ACDC.py:108-167): two student networks trained with cross pseudo supervision (Dice only,
    weight 7w) plus, from iteration ``mt_start`` on, Mean-Teacher MSE of both students against the EMA teacher of student 2,
    which sees the noise-perturbed unlabeled slices.  w = consistency * linear_rampup(cur_itrs // 150, rampup) (:148-149).
    One fused loss call (``hpfg_s4cv_loss``) produces the value and both logit gradients.  Eager launches only."""
    share_forward = False

    def __init__(self, model1, model2, ema_model, *, ema_decay=0.99, mt_start=1000, **kw):
        super().__init__(**kw)
        self.m1, self.m2, self.ema_model, self.ema_decay, self.mt_start = model1, model2, ema_model, ema_decay, mt_start
        (self.g1, self.b1), (self.g2, self.b2) = self._setup([model1, model2], [model1, model2, ema_model])

    def _use_graph(self):
        return False

    def _consistency_weight(self):
        return self.consistency * linear_rampup(self.cur_itrs // 150, self.consistency_rampup)

    def step(self, x, labels, noise=None):
        """x: [n_l+n_u, C, H, W] (labeled first); labels: [n_l, H, W]; noise [n_u, ...]: drawn here if None."""
        self._next_iteration()
        n_l, dev = labels.shape[0], x.device
        x_u = x[n_l:]
        if noise is None:
            noise = _input_noise(x_u.shape, x_u)
        x_t = (x_u + noise).contiguous()
        ncls, hh, ww = self.num_classes, x.shape[2], x.shape[3]
        shape = (x.shape[0], ncls, hh, ww)
        main, side = self._fork(dev)
        with torch.cuda.stream(side):               # student 2 and its teacher on the side stream, student 1 on the main stream
            p2, o2 = self._forward(self.m2, x, True, self._persistent("o2", shape, dev), None)
            _, t_out = self._forward(self.ema_model, x_t, False, self._persistent("t_out", (x_u.shape[0], ncls, hh, ww), dev), None)
        p1, o1 = self._forward(self.m1, x, True, self._persistent("o1", shape, dev), None)
        main.wait_stream(side)
        w = self._consistency_weight()
        mt_on = self.cur_itrs >= self.mt_start
        with self._global_sums():
            r = s4cv_loss_raw(o1, o2, t_out if mt_on else None, labels, n_l, cps_weight=7.0 * w, mt_weight=w)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            self._backward(self.m2, p2, r["dother"], self.g2)
            self._opt_step(self._trained[1], None, self.ema_model)      # student 2 + EMA into its teacher, one pass
        self._backward(self.m1, p1, r["dstudent"], self.g1)
        self._opt_step(self._trained[0], None)
        main.wait_stream(side)
        self.last = dict(scalars=r["scalars"], lr=self._lr(), w=w, logits1=o1, logits2=o2, teacher_logits=t_out)
        return r["scalars"][0]


class HPFGStep(_StepBase):
    """The HPFG iteration of main.py:128-207 on three ``UNet_Plus`` networks: model1 sees the CutMix batch, model2 and the EMA
    teacher the plain batch.  One step body (``_body``) runs eagerly or is captured and replayed as one CUDA graph
    (``enable_graph``): the CutMix input mix (``hpfg_cutmix_mix``); the three U-Net forwards; the projection necks of model2
    and of the teacher (model1's neck outputs are dropped by main.py:148, so they do not run); model2's supervised + Mean-Teacher
    terms as the MT mode of the fused loss kernels, model1's supervised + pseudo-label Dice as the CUTMIX mode, the four
    ``Dense_Loss`` terms with their gradients scaled by 0.5*w; the neck backwards (the head neck's input gradient joins model2's
    logits gradient, the high neck's the bottleneck); both U-Net backwards into flat gradient buffers; the optimiser over both
    flat buffers and each of model2's 16 neck tensors; the backbone EMA model2 <- model1 (main.py:68-76) and the teacher EMA
    (utils/utils.py:82-86) over the flat buffer and the neck tensors.  No autograd runs.

    After a step, ``p.grad`` of every parameter of model1 and model2 holds that step's gradient as a view into the driver's
    buffers (model1's neck tensors: None).  The exact-global data-parallel mode is not implemented by this step: with
    ``exact_global=True`` gradients are summed over the ranks and nothing else changes.

    step(label_img, target_label, label_img1, target_label1, img_unlabel, cutmix_mask): the tensors main.py:128-143 draws
    (label_img1 / target_label1: the second labeled draw, n_l1 images, never repeated: unlabeled image u reads u % n_l1 as
    main.py:139-140's repeat does; cutmix_mask [n_u,1,H,W] from BoxMaskGenerator)."""
    share_forward = False           # (the step runs on one stream: each forward has the whole machine)
    sync_bn_exact_global = False

    def __init__(self, model1, model2, ema_model, *, ema_decay=0.99, mt_start=1000, temperature=0.7, **kw):
        super().__init__(**kw)
        self.m1, self.m2, self.ema_model, self.ema_decay, self.mt_start = model1, model2, ema_model, ema_decay, mt_start
        (self.g1, self.b1), (self.g2, self.b2) = self._setup([model1, model2], [model1, model2, ema_model])
        for p in ema_model.parameters():
            p.requires_grad = False
        self.temperature = temperature
        self._step_lr = None
        self._stepped = False           # this driver has run a step (plans, neck states and buffers exist)

    def _consistency_weight(self):
        return self.consistency * linear_rampup(self.cur_itrs // 150, self.consistency_rampup)

    def _mt_weight(self):
        """Weight of model2's Mean-Teacher term: w from mt_start on, 0 before (main.py:137-142)."""
        return self._consistency_weight() if self.cur_itrs >= self.mt_start else 0.0

    def _lr(self):
        return medical_lr(self.cur_itrs, self.base_lr, self.total_itrs) if self._step_lr is None else self._step_lr

    def _use_graph(self):
        """Replay once this driver has run a step and every optimiser state, flat and neck, has taken its first update: the SGD
        launch bakes in whether it initialises the momentum buffer, and the neck states are created at their first gradient."""
        states = [s for _, _, s in self._trained] + [self._neck_states.get(id(p)) for p in self._neck_params(self.m2)]
        return (self._graph_enabled and self._stepped and (self.world == 1 or self._graph_dp) and not self.exact_global
                and all(s is not None and s.step >= 2 for s in states))

    def _graph_ptrs(self):
        necks2 = self._neck_params(self.m2)
        ptrs = tuple(p.data_ptr() for p in necks2 + self._neck_params(self.ema_model))
        ptrs += tuple(b.data_ptr() for p in necks2 for b in self._neck_states[id(p)].bufs)
        return ptrs + tuple(t.data_ptr() for t in self._bufs.values())      # neck gradients, neck / loss scratch, batches

    def step(self, label_img, target_label, label_img1, target_label1, img_unlabel, cutmix_mask, lr=None):
        """lr: override of the Medical_LR value of this iteration (resuming with a fresh scheduler; parity harness).
        cutmix_mask: the box masks of BoxMaskGenerator (main.py:141-143).  Returns the loss (device scalar)."""
        check_cutmix_batch(img_unlabel.shape[0], label_img1.shape[0])
        self._next_iteration()
        necks2 = self._neck_params(self.m2)
        for p in necks2:        # torch.optim: a tensor's state appears at its first gradient, and it counts its own steps
            s = self._neck_states.get(id(p))
            if s is None:
                s = self._neck_states[id(p)] = self._opt.new_state(p.data)
                self.__dict__.setdefault("_neck_owners", {})[id(p)] = p     # (keeps the id of a replaced tensor from being reused)
            s.step += 1
        self._step_lr = lr
        w = self._consistency_weight()
        ins = [label_img, target_label, label_img1, target_label1, img_unlabel, cutmix_mask]
        if self._use_graph():
            out = self._graph_replay(ins, self._dyn_scalars(self.ema_decay, self._mt_weight(), 7.0 * w, 0.5 * w),
                                     [self.m1, self.m2, self.ema_model], self._body)
        else:
            out = self._body(ins, None)
        self._stepped = True
        self._publish_grads(necks2)
        self.last = dict(out, lr=self._lr(), w=w)
        return out["loss"]

    def _publish_grads(self, necks2):
        """p.grad of model1 / model2: views into the flat gradient buffers and model2's neck gradient buffers."""
        views = self.__dict__.setdefault("_grad_views", {})
        for model, g, _ in self._trained:
            for p, (o, n, shape) in zip(model._flat_params_list, model._layout):
                v = views.get(id(p), (None, None))[1]
                if v is None:
                    v = g[o:o + n].view(shape)
                    views[id(p)] = (p, v)
                if p.grad is not v:
                    p.grad = v
        for p in self._neck_params(self.m1):
            p.grad = None
        for j, p in enumerate(necks2):
            g = self._bufs["neck_grad%d" % j]
            if p.grad is not g:
                p.grad = g

    def _neck_forward(self, neck, x, key):
        """projection_conv.forward of ``neck`` on x into step-persistent buffers: (pooled, hidden, out_global, out_dense)."""
        n, c, h, w = x.shape
        s, hid, dim = neck.is_s, neck.mlp[0].out_features, neck.mlp[2].out_features
        rows, dev = n * (1 + s * s), x.device
        bufs = (self._persistent(key + ".pooled", (rows, c), dev), self._persistent(key + ".hidden", (rows, hid), dev),
                self._persistent(key + ".global", (n, dim), dev), self._persistent(key + ".dense", (n, dim, s * s), dev))
        params = (ctypes.c_void_p * 8)(*[p.data_ptr() for p in neck._param_list()])
        L.check(L.lib().hpfg_neck_forward(L.ptr(x), n, c, h, w, s, hid, dim, params, *[L.ptr(b) for b in bufs],
                                          L.stream_ptr(dev)), "hpfg_neck_forward")
        return bufs

    def _neck_backward(self, neck, x, key, fwd, d_global, d_dense, grads, dx):
        n, c, h, w = x.shape
        s, hid, dim = neck.is_s, neck.mlp[0].out_features, neck.mlp[2].out_features
        scratch = self._persistent(key + ".scratch", (n * s * s * dim + n * (1 + s * s) * (hid + c),), x.device)
        params = (ctypes.c_void_p * 8)(*[p.data_ptr() for p in neck._param_list()])
        L.check(L.lib().hpfg_neck_backward(L.ptr(d_global), L.ptr(d_dense), n, c, h, w, s, hid, dim, params, L.ptr(fwd[0]),
                                           L.ptr(fwd[1]), (ctypes.c_void_p * 8)(*[g.data_ptr() for g in grads]), L.ptr(dx),
                                           L.ptr(scratch), L.stream_ptr(x.device)), "hpfg_neck_backward")

    def _ema(self, ema, param, alpha, dv):
        """ema <- alpha*ema + (1 - alpha)*param; captures read {alpha, 1 - alpha} from the device block."""
        if dv is None:
            L.check(L.lib().hpfg_ema_update(L.ptr(ema), L.ptr(param), ema.numel(), float(alpha), L.stream_ptr(ema.device)),
                    "hpfg_ema_update")
        else:
            L.check(L.lib().hpfg_ema_update_dv(L.ptr(ema), L.ptr(param), ema.numel(), L.ptr(dv[0][1:3]),
                                               L.stream_ptr(ema.device)), "hpfg_ema_update_dv")

    def _body(self, ins, dv):
        label_img, target_label, label_img1, target_label1, img_unlabel, cutmix_mask = ins
        m1, m2, ema = self.m1, self.m2, self.ema_model
        n_l, n_u = label_img.shape[0], img_unlabel.shape[0]
        n, dev = n_l + n_u, label_img.device
        img_shape, hh, ww = tuple(label_img.shape[1:]), label_img.shape[2], label_img.shape[3]
        lib = L.lib()
        # main.py:137-150: model1 sees cat(label_img, CutMix(label_img1, img_unlabel)), model2 and the teacher cat(label_img, img_unlabel)
        batch_mix = self._persistent("batch_mix", (n,) + img_shape, dev)
        volume = self._persistent("volume", (n,) + img_shape, dev)
        batch_mix[:n_l].copy_(label_img)
        cutmix_mix_inputs(label_img1, img_unlabel, cutmix_mask, out=batch_mix[n_l:])
        volume[:n_l].copy_(label_img)
        volume[n_l:].copy_(img_unlabel)
        shape = (n, self.num_classes, hh, ww)
        p1, o1 = self._forward(m1, batch_mix, True, self._persistent("o1", shape, dev), dv)
        p2, o2 = self._forward(m2, volume, True, self._persistent("o2", shape, dev), dv)
        pt, t_out = self._forward(ema, volume, False, self._persistent("t_out", shape, dev), dv)
        feat_shape = (n, FT_CHNS[-1], hh // 16, ww // 16)
        feats = []
        for plan, key in ((p2, "feat2"), (pt, "feat_t")):     # feature[-1] (model/unet.py:199-201)
            f = self._persistent(key, feat_shape, dev)
            L.check(lib.hpfg_unet_bottleneck(plan.handle, L.ptr(f), L.stream_ptr(dev)), "hpfg_unet_bottleneck")
            feats.append(f)
        necks = [(m2.dense_projection_high, ema.dense_projection_high, feats[0], feats[1], "high"),
                 (m2.dense_projection_head, ema.dense_projection_head, o2, t_out, "head")]
        fwd2 = [self._neck_forward(nk, x, key + "2") for nk, _, x, _, key in necks]
        fwd_t = [self._neck_forward(nk, x, key + "_t") for _, nk, _, x, key in necks]
        # main.py:144,166: w * (Dense_Loss(h1, ema_h1) + Dense_Loss(h2, ema_h2)), Dense_Loss = 0.5 * (global term + dense term):
        # four contrastive calls, each writing 0.5*w * its gradient wrt model2's neck output
        w = self._consistency_weight()
        contrast = self._persistent("contrast", (4,), dev)
        ws = self._persistent("contrast_ws", (lib.hpfg_dense_contrastive_workspace_floats(n, fwd2[0][3].shape[1],
                                                                                          fwd2[0][3].shape[2]),), dev)
        d_out = []
        for k, (a, b) in enumerate((a, b) for f2, ft in zip(fwd2, fwd_t) for a, b in ((f2[2], ft[2]), (f2[3], ft[3]))):
            d = self._persistent("d_contrast%d" % k, tuple(a.shape), dev)
            L.check(lib.hpfg_dense_contrastive_scaled(L.ptr(a), L.ptr(b), n, a.shape[1], a[0, 0].numel(), float(self.temperature),
                                                      float(0.5 * w), L.ptr(self._dv_scalar(dv, 6)), L.ptr(contrast[k:k + 1]),
                                                      L.ptr(d), L.ptr(ws), L.stream_ptr(dev)), "hpfg_dense_contrastive_scaled")
            d_out.append(d)
        # model2 (main.py:127,142,144): supervised + Mean-Teacher MSE from mt_start on; model1 (:125,131-134,143): supervised + 7w *
        # Dice against the teacher's argmax pasted into the second labeled draw's labels
        r2 = ssl_loss_raw(L.LOSS_MT, o2, t_out[n_l:], target_label, n_l, cons_weight=self._mt_weight(),
                          cons_weight_dev=self._dv_scalar(dv, 4))
        r1 = cutmix_loss_raw(o1, t_out[n_l:], target_label, target_label1, cutmix_mask, n_l, pseudo_weight=7.0 * w,
                             pseudo_weight_dev=self._dv_scalar(dv, 5))
        # neck backwards: the high neck's input gradient enters model2 at the bottleneck, the head neck's at the logits
        necks2 = self._neck_params(m2)
        ngrads = [self._persistent("neck_grad%d" % j, tuple(p.shape), dev) for j, p in enumerate(necks2)]
        dfeat = self._persistent("dfeat", feat_shape, dev)
        dx_head = self._persistent("dx_head", shape, dev)
        for i, ((nk, _, x, _, key), dx) in enumerate(zip(necks, (dfeat, dx_head))):
            self._neck_backward(nk, x, key + "2", fwd2[i], d_out[2 * i], d_out[2 * i + 1], ngrads[8 * i:8 * i + 8], dx)
        dl2 = r2["dstudent"]
        dl2.add_(dx_head)
        L.check(lib.hpfg_unet_backward(p1.handle, L.ptr(m1.flat_params), L.ptr(r1["dstudent"]), L.ptr(self.g1), 0,
                                       L.stream_ptr(dev)), "hpfg_unet_backward")
        L.check(lib.hpfg_unet_backward_ex(p2.handle, L.ptr(m2.flat_params), L.ptr(dl2), L.ptr(dfeat), L.ptr(self.g2), 0,
                                          L.stream_ptr(dev)), "hpfg_unet_backward_ex")
        if self.world > 1:      # data parallel (main.py itself is single-process): gradients summed here, scaled in the optimiser
            import torch.distributed as dist
            dist.all_reduce(self.g1, group=self.pg)
            dist.all_reduce(self.g2, group=self.pg)
            allreduce_tensor_list(ngrads, group=self.pg)
        self._opt_step(self._trained[0], dv)
        self._opt_step(self._trained[1], dv)
        block = None if dv is None else dv[0]
        for p, g in zip(necks2, ngrads):
            self._opt.launch(p.data, g, self._neck_states[id(p)], None, self._lr(), 0.0, block, L.stream_ptr(dev))
        alpha = min(1 - 1 / (self.cur_itrs + 1), self.ema_decay)
        self._ema(m2.flat_params, m1.flat_params, alpha, dv)        # update_ema_variables_backbone: encoder + decoder = the flat buffer
        self._ema(ema.flat_params, m2.flat_params, alpha, dv)
        for e, p in zip(self._neck_params(ema), necks2):
            self._ema(e.data, p.data, alpha, dv)
        lc = 0.5 * (contrast[0] + contrast[1]) + 0.5 * (contrast[2] + contrast[3])
        loss = r1["scalars"][0] + r2["scalars"][0] + (w if dv is None else dv[0][3]) * lc
        return dict(loss=loss, loss_sup=r1["scalars"][1] + r2["scalars"][1], contrast=lc, pseudo=r1["scalars"][2],
                    cons2=r2["scalars"][2], outputs1=o1, outputs2=o2, ema_output=t_out)
