"""CPU oracle for the HPFG semi-supervised U-Net hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``hpfg_b200/`` may import this package; only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs do, and
there only as the checker / the timed CPU baseline, never as the product path.

The oracle is a plain PyTorch fp32 *restatement* of the reference algorithm (the reference itself is
pure PyTorch; every function cites the reference file:line it follows).  It is pinned two ways:

* ``tests/test_oracle_vs_reference.py`` runs it against values the real reference modules printed
  (``tests/golden/reference_mt_acdc.json``), and against the modules themselves, loaded by file path from
  a checkout named by ``$HPFG_REF``, where one is given;
* ``tests/golden/*.pt`` hold input/output vectors produced by the real reference
  (``tests/golden/make_golden.py``), which travel to the GPU box.
"""
from .unet_ref import (unet_param_spec, unet_buffer_spec, init_unet_state, unet_forward,
                       ENC_DROPOUT, FT_CHNS, unet_plus_forward, unet_plus_neck_spec, projection_conv)
from .losses_ref import (dice_loss, med_sup_loss, softmax_mse, mt_consistency, cps_losses,
                         uamt_consistency, ce_loss, ict_losses, s4cv_losses, dense_loss, dense_contrastive)
from .steps_ref import (update_ema, sigmoid_rampup, consistency_weight, medical_lr, SGDState,
                        sgd_step, mt_step, cps_step, uamt_step, ema_alpha, ict_step, s4cv_step, linear_rampup)
