"""The optimiser side of the step drivers: torch.optim.SGD (momentum) or Adam / AdamW as the fused passes of csrc/optim.cu,
over a network's flat parameter buffer or one tensor outside it.  A driver makes one optimiser (``SGD`` or ``Adam``); it
owns all that depends on the kind: hyperparameters, per-step host scalars and their device-block group, the entry point
it launches and torch.optim's per-parameter checkpoint entries.  ``OptState`` is the state of one parameter set."""
import torch

from . import _lib as L


class OptState:
    """Optimiser state of one parameter set: its buffers (in the order of the optimiser's KEYS) and its step count."""

    def __init__(self, bufs, step=0):
        self.bufs, self.step = tuple(bufs), step
        self.dv_offset = 0              # where its group starts in the device block of a captured step


class _Optimizer:
    KEYS = ()               # the tensors of torch.optim's per-parameter state, in the order of OptState.bufs

    def __init__(self, kind, weight_decay, grad_scale):
        self.kind, self.weight_decay, self.grad_scale = kind, weight_decay, grad_scale

    def new_state(self, like):
        return OptState([torch.zeros_like(like) for _ in self.KEYS])

    def load_entry(self, st, tensors):
        """Copy checkpoint entry ``st`` (None: no state) into ``tensors``, one parameter's slices of a state's buffers."""
        for k, t in zip(self.KEYS, tensors):
            if st is not None and st.get(k) is not None:
                t.copy_(st[k].reshape(t.shape))

    def check_kind(self, opt):
        """A checkpoint of the other optimiser kind (SGD momentum vs Adam moments) cannot be resumed by this driver."""
        groups, states = opt.get("param_groups", []), opt.get("state", {}).values()
        adam = any("betas" in g for g in groups) or any("exp_avg" in st for st in states)
        sgd = any("momentum_buffer" in st for st in states) or any("momentum" in g and "betas" not in g for g in groups)
        if (adam and "exp_avg" not in self.KEYS) or (sgd and "momentum_buffer" not in self.KEYS):
            raise ValueError("the checkpoint holds %s optimiser state but this step driver uses optimizer=%r"
                             % ("Adam" if adam else "SGD", self.kind))


class SGD(_Optimizer):
    """torch.optim.SGD with momentum: the first update of a state (step 1) initialises its momentum buffer."""
    KEYS = ("momentum_buffer",)
    _ENTRY = {(True, True): "hpfg_sgd_momentum", (False, True): "hpfg_sgd_momentum_ema",    # (no EMA, scalars by value)
              (True, False): "hpfg_sgd_momentum_dv", (False, False): "hpfg_sgd_momentum_ema_dv"}

    def __init__(self, kind, lr, momentum, weight_decay, betas, eps, grad_scale):
        super().__init__(kind, weight_decay, grad_scale)
        self.momentum = momentum

    def param_group(self, lr, n_params):
        return {"lr": lr, "momentum": self.momentum, "weight_decay": self.weight_decay, "params": list(range(n_params))}

    def device_group(self, step, lr, alpha, one_minus):
        return []               # the SGD pass reads [lr, alpha, 1 - alpha] at the head of the block

    @staticmethod
    def has_state(state, cur_itrs):         # checkpoints hold momentum from the driver's first iteration on
        return cur_itrs > 0

    @staticmethod
    def entry(step, tensors):
        return {"momentum_buffer": tensors[0].clone()}

    @staticmethod
    def checkpoint_step(entries, k, cur_itrs):
        """SGD checkpoints carry no step count: a loaded state continues from the driver's iteration (a checkpoint holds
        momentum only from its first iteration on, so a loaded buffer is not initialised again)."""
        return cur_itrs

    def launch(self, param, grad, state, ema, lr, alpha, block, stream):
        """hpfg_sgd_momentum{,_ema}{,_dv}: the EMA of ``param`` into ``ema`` in the same pass if given; ``block``: the device
        block of a captured step (None: ``lr`` and ``alpha`` by value)."""
        name = self._ENTRY[ema is None, block is None]
        bufs = (L.ptr(param), L.ptr(grad), L.ptr(state.bufs[0])) + (() if ema is None else (L.ptr(ema),))
        hyper = (self.momentum, self.weight_decay, self.grad_scale, int(state.step == 1))
        if block is None:
            args = (lr,) + hyper + (() if ema is None else (alpha,))
        else:
            args = hyper + (L.ptr(block),)
        L.check(getattr(L.lib(), name)(*bufs, param.numel(), *args, stream), name)


class Adam(_Optimizer):
    """torch.optim.Adam (L2 weight decay) or AdamW (decoupled), bias-corrected by the state's own step count."""
    KEYS = ("exp_avg", "exp_avg_sq")

    def __init__(self, kind, lr, momentum, weight_decay, betas, eps, grad_scale):
        super().__init__(kind, weight_decay, grad_scale)
        decoupled = kind == "adamw"
        self.betas, self.eps, self.decoupled = (float(betas[0]), float(betas[1])), float(eps), decoupled
        cls = torch.optim.AdamW if decoupled else torch.optim.Adam
        # the param_group keys and values the installed torch emits for these hyperparameters (checkpoint layout)
        group = cls([torch.zeros(1, requires_grad=True)], lr=lr, betas=self.betas, eps=self.eps,
                    weight_decay=weight_decay).state_dict()["param_groups"][0]
        self.group = {k: v for k, v in group.items() if k != "params"}
        # the launch arguments that do not change (the 1 - beta complements in double, rounded to fp32 by the call)
        self._fixed = (1 - self.betas[0], self.betas[1], 1 - self.betas[1], self.eps, weight_decay, int(decoupled), grad_scale)

    def param_group(self, lr, n_params):
        return dict(self.group, lr=lr, params=list(range(n_params)))

    def scalars(self, step, lr):
        """[step_size, bc2_sqrt, decay_factor] of Adam step ``step``, in double as torch.optim.adam._multi_tensor_adam
        computes them (bias corrections from the float step count) before they are cast to fp32."""
        beta1, beta2 = self.betas
        bias_correction1 = 1 - beta1 ** float(step)
        bias_correction2 = 1 - beta2 ** float(step)
        decay = 1 - lr * self.weight_decay if self.decoupled else 1.0
        return [(lr / bias_correction1) * -1, bias_correction2 ** 0.5, decay]

    def device_group(self, step, lr, alpha, one_minus):
        return self.scalars(step, lr) + [alpha, one_minus]

    @staticmethod
    def has_state(state, cur_itrs):         # checkpoints hold a state once it has taken a step, as torch.optim.Adam's
        return state.step > 0

    @staticmethod
    def entry(step, tensors):
        return {"step": torch.tensor(float(step), dtype=torch.float32), "exp_avg": tensors[0].clone(),
                "exp_avg_sq": tensors[1].clone()}

    @staticmethod
    def checkpoint_step(entries, k, cur_itrs):
        """The one step count of the per-parameter entries of a flat buffer (0: no state yet)."""
        steps = {float(st["step"]) for st in entries if st is not None}
        if len(steps) > 1 or (steps and any(st is None for st in entries)):
            raise ValueError("the %d U-Net tensors of optimizer entry %d carry different Adam step counts (%s): one flat "
                             "buffer keeps one step count" % (len(entries), k, sorted(steps)))
        return int(steps.pop()) if steps else 0

    def launch(self, param, grad, state, ema, lr, alpha, block, stream):
        """hpfg_adam(_dv): the EMA of ``param`` into ``ema`` in the same pass if given; ``block``: the device block of a
        captured step, this state's group at ``state.dv_offset`` (None: the scalars by value)."""
        exp_avg, exp_avg_sq = state.bufs
        common = (L.ptr(param), L.ptr(grad), L.ptr(exp_avg), L.ptr(exp_avg_sq), L.ptr(ema), param.numel()) + self._fixed
        if block is None:
            L.check(L.lib().hpfg_adam(*common, *self.scalars(state.step, lr), alpha, stream), "hpfg_adam")
        else:
            L.check(L.lib().hpfg_adam_dv(*common, L.ptr(block[state.dv_offset:]), stream), "hpfg_adam_dv")
