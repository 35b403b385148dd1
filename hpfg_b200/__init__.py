"""hpfg_b200 -- B200-native (sm_100a) implementation of HPFG's semi-supervised U-Net training hot path,
behind the reference's own Python API:

    build_model(args)                      model/builder.py:14-62 ('unet' branch)
    UNet(in_channels, num_classes)         model/unet.py:155-175
    UNet_Plus(in_channels, num_classes)    model/unet.py:178-206 (main.py's HPFG networks)
    Med_Sup_Loss, DiceLoss, softmax_mse_loss   utils/loss/medloss.py, utils/loss/diceloss.py
    update_ema_variables, get_current_consistency_weight, sigmoid_rampup   utils/utils.py:67-86

plus fused whole-step drivers (MeanTeacherStep / CPSStep / UAMTStep / ICTStep / S4CVStep) and the HPFG iteration driver (HPFGStep), the ICT-MedSeg / S4CVNet / HPFG CutMix step losses and the
batched inference path of val.py:268-281 (predict_volume).  All compute goes through
libhpfg_b200.so (include/hpfg_b200.h); there is no CPU or PyTorch fallback."""
from .builder import build_model
from .unet import UNet, UNet_Plus, projection_conv, predict_volume
from .losses import (Med_Sup_Loss, DiceLoss, softmax_mse_loss, mean_teacher_loss, cps_loss, uamt_loss, ssl_loss_raw,
                     ict_loss, ict_loss_raw, ict_mix_inputs, s4cvnet_loss, s4cv_loss_raw, cutmix_loss_raw, cutmix_pseudo_loss,
                     cutmix_mix_inputs, argmax_labels, Dense_Loss)
from .utils import (update_ema_variables, get_current_consistency_weight, sigmoid_rampup, linear_rampup,
                    ema_update_flat)
from .trainer import (MeanTeacherStep, CPSStep, UAMTStep, ICTStep, S4CVStep, HPFGStep, medical_lr, gradient_buckets, allreduce_flat_buckets,
                      allreduce_tensor_list, shard_batch)

__all__ = ["build_model", "UNet", "UNet_Plus", "projection_conv", "Dense_Loss", "Med_Sup_Loss", "DiceLoss", "softmax_mse_loss", "mean_teacher_loss", "cps_loss",
           "uamt_loss", "ssl_loss_raw", "update_ema_variables", "get_current_consistency_weight", "sigmoid_rampup",
           "linear_rampup", "ema_update_flat", "MeanTeacherStep", "CPSStep", "UAMTStep", "ICTStep", "S4CVStep", "HPFGStep", "ict_loss", "ict_loss_raw",
           "ict_mix_inputs", "s4cvnet_loss", "s4cv_loss_raw", "cutmix_loss_raw", "cutmix_pseudo_loss", "cutmix_mix_inputs", "argmax_labels", "predict_volume", "medical_lr", "gradient_buckets", "allreduce_flat_buckets", "allreduce_tensor_list", "shard_batch"]
