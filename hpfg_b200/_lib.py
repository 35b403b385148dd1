"""ctypes binding of libhpfg_b200.so (the C ABI declared in include/hpfg_b200.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HPFG_B200_LIB") or os.path.join(_HERE, "libhpfg_b200.so")   # override: A/B builds under profiles/

c_i64p = ctypes.POINTER(ctypes.c_int64)
c_vp = ctypes.c_void_p
c_int = ctypes.c_int
c_f = ctypes.c_float
c_i64 = ctypes.c_int64
c_u64 = ctypes.c_uint64

# every symbol include/hpfg_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "hpfg_last_error": (ctypes.c_char_p, []),
    "hpfg_version": (c_int, []),
    "hpfg_launch_count": (c_i64, []),
    "hpfg_profile_begin": (c_int, []),
    "hpfg_profile_end": (c_int, [ctypes.POINTER(ctypes.c_double), c_i64p]),
    "hpfg_unet_param_layout": (c_int, [c_int, c_int, c_i64p, c_i64p, c_i64p]),
    "hpfg_unet_bn_layout": (c_int, [c_int, c_int, c_i64p, c_i64p, c_i64p]),
    "hpfg_unet_plan_create": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_vp)]),
    "hpfg_unet_plan_destroy": (c_int, [c_vp]),
    "hpfg_unet_plan_workspace_bytes": (c_i64, [c_vp]),
    "hpfg_unet_plan_set_bwd_fusion": (c_int, [c_vp, c_int]),
    "hpfg_unet_plan_set_forward_ctas": (c_int, [c_vp, c_int]),
    "hpfg_unet_plan_set_sync_bn": (c_int, [c_vp, c_int]),
    "hpfg_ssl_loss_set_global_sums": (c_int, [c_int]),
    "hpfg_set_allreduce_hook": (c_int, [c_vp, c_vp, c_int]),
    "hpfg_unet_forward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_u64, c_u64,
                                  ctypes.POINTER(c_vp), c_vp]),
    "hpfg_unet_forward_dv": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_u64, c_vp,
                                     ctypes.POINTER(c_vp), c_vp]),
    "hpfg_unet_backward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_vp]),
    "hpfg_unet_bottleneck": (c_int, [c_vp, c_vp, c_vp]),
    "hpfg_unet_backward_ex": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp]),
    "hpfg_unet_num_buckets": (c_int, [c_vp]),
    "hpfg_unet_bucket_range": (c_int, [c_vp, c_int, c_i64p, c_i64p]),
    "hpfg_unet_bucket_wait": (c_int, [c_vp, c_int, c_vp]),
    "hpfg_unet_bucket_layout": (c_int, [c_int, c_int, c_i64p, c_i64p]),
    "hpfg_unet_debug_tap": (c_int, [c_vp, ctypes.c_char_p, c_vp, c_i64, c_vp]),
    "hpfg_conv_tc_debug": (c_int, [c_int] * 7 + [c_vp] * 8),
    "hpfg_conv_tc_bench": (c_int, [c_int] * 8 + [ctypes.POINTER(c_f), c_vp]),
    "hpfg_wgrad_tc_debug": (c_int, [c_int] * 6 + [c_vp] * 7),
    "hpfg_dgrad_tc_fused_debug": (c_int, [c_int] * 6 + [c_vp] * 10 + [c_f] + [c_vp] * 3),
    "hpfg_wgrad_tc_fused_debug": (c_int, [c_int] * 6 + [c_vp] * 11),
    "hpfg_glue_debug": (c_int, [c_int] * 5 + [c_vp] * 8 + [c_f] + [c_vp] * 3),
    "hpfg_ssl_loss_workspace_bytes": (c_i64, [c_int] * 6),
    "hpfg_ssl_loss": (c_int, [c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_f,
                              ctypes.POINTER(c_f), c_f, c_f, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "hpfg_ssl_loss_dv": (c_int, [c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_f, c_vp,
                                 ctypes.POINTER(c_f), c_f, c_f, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "hpfg_ict_loss": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_vp, ctypes.POINTER(c_f),
                              c_f, c_f, c_vp, c_vp, c_vp, c_vp]),
    "hpfg_ict_mix": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_vp]),
    "hpfg_cutmix_loss": (c_int, [c_vp] * 5 + [c_int] * 6 + [c_f, c_vp, ctypes.POINTER(c_f), c_f, c_f] + [c_vp] * 5),
    "hpfg_cutmix_mix": (c_int, [c_vp] * 3 + [c_int] * 5 + [c_vp, c_vp]),
    "hpfg_s4cv_loss": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_f, c_vp,
                               ctypes.POINTER(c_f), c_f, c_f, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "hpfg_softmax_mse": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "hpfg_argmax_labels": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "hpfg_dice_loss": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_f), c_vp, c_vp, c_vp,
                               c_vp]),
    "hpfg_neck_forward": (c_int, [c_vp] + [c_int] * 7 + [ctypes.POINTER(c_vp)] + [c_vp] * 5),
    "hpfg_neck_backward": (c_int, [c_vp, c_vp] + [c_int] * 7 + [ctypes.POINTER(c_vp), c_vp, c_vp, ctypes.POINTER(c_vp), c_vp, c_vp,
                                                               c_vp]),
    "hpfg_dense_contrastive_workspace_floats": (c_i64, [c_int, c_int, c_int]),
    "hpfg_dense_contrastive": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_f, c_vp, c_vp, c_vp, c_vp]),
    "hpfg_dense_contrastive_scaled": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_f, c_f, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "hpfg_ema_update": (c_int, [c_vp, c_vp, c_i64, c_f, c_vp]),
    "hpfg_ema_update_dv": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "hpfg_sgd_momentum": (c_int, [c_vp, c_vp, c_vp, c_i64, c_f, c_f, c_f, c_f, c_int, c_vp]),
    "hpfg_sgd_momentum_ema": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f, c_f, c_f, c_f, c_int, c_f, c_vp]),
    "hpfg_sgd_momentum_ema_dv": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f, c_f, c_f, c_int, c_vp, c_vp]),
    "hpfg_sgd_momentum_dv": (c_int, [c_vp, c_vp, c_vp, c_i64, c_f, c_f, c_f, c_int, c_vp, c_vp]),
    "hpfg_adam": (c_int, [c_vp] * 5 + [c_i64] + [c_f] * 5 + [c_int] + [c_f] * 5 + [c_vp]),
    "hpfg_adam_dv": (c_int, [c_vp] * 5 + [c_i64] + [c_f] * 5 + [c_int, c_f, c_vp, c_vp]),
}

PREC_FP32, PREC_BF16 = 0, 1
LOSS_SUP, LOSS_MT, LOSS_CPS, LOSS_UAMT, LOSS_ICT, LOSS_S4CV, LOSS_CUTMIX = 0, 1, 2, 3, 4, 5, 6
NUM_BN, NUM_DROPOUT, NUM_PARAMS = 18, 5, 82

_lib = None


class HpfgError(RuntimeError):
    pass


def lib():
    """The loaded library (loads on first use; raises if libhpfg_b200.so has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise HpfgError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU / PyTorch fallback)" % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().hpfg_last_error()
        raise HpfgError("%s failed (code %d): %s" % (what or "hpfg call", rc, msg.decode() if msg else "?"))


def ptr(t):
    """Device/host pointer of a tensor (None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, what):
    if not t.is_cuda:
        raise HpfgError("%s must be a CUDA tensor: hpfg_b200 has no CPU path (got device %s)" % (what, t.device))


# ---- exact-global data-parallel mode: the library's sum-all-reduce hook, served by torch.distributed -------------------------
ALLREDUCE_FN = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_void_p)
_hook_keepalive = {}


class _DevBuf:
    """Zero-copy view of a raw device pointer for torch.as_tensor (CUDA array interface)."""

    def __init__(self, ptr, count, is_double):
        self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": "<f8" if is_double else "<f4", "data": (int(ptr), False),
                                         "version": 2}


def install_allreduce_hook(group=None):
    """Register torch.distributed's all_reduce(SUM) over ``group`` as the library's hook (hpfg_set_allreduce_hook)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)

    def _hook(ctx, ptr, count, is_double, stream):
        # Exact-global mode is a verification mode (one small collective per BatchNorm, eager launches): every collective is
        # host-synchronised on both sides.  Stream-ordered hand-over between the library's programmatically-launched kernels
        # and ProcessGroupNCCL's internal stream was measured unreliable on the legacy default stream (profiles/README.md).
        dev = torch.cuda.current_device()
        t = torch.as_tensor(_DevBuf(ptr, count, is_double), device=torch.device("cuda", dev))
        torch.cuda.synchronize(dev)
        dist.all_reduce(t, group=group)
        torch.cuda.synchronize(dev)
    cb = ALLREDUCE_FN(_hook)
    _hook_keepalive["cb"] = cb
    check(lib().hpfg_set_allreduce_hook(ctypes.cast(cb, ctypes.c_void_p), None, world), "hpfg_set_allreduce_hook")
    return world
