"""Load the REAL reference hot-path modules by file path (never `import model` / `import utils`: those
pull timm/easydict/medpy which are not installed).  Only available where a checkout of the reference is named by
$HPFG_REF; everywhere else the tests rely on tests/golden/ instead."""
import importlib.util
import os
import sys
import types


def find_reference():
    p = os.environ.get("HPFG_REF")
    return p if p and os.path.isfile(os.path.join(p, "model", "unet.py")) else None


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_reference():
    """Returns a namespace with UNet, Med_Sup_Loss, DiceLoss, softmax_mse_loss, update_ema_variables,
    get_current_consistency_weight, sigmoid_rampup, Medical_LR -- the reference's own objects."""
    root = find_reference()
    if root is None:
        raise FileNotFoundError("reference checkout not found (set HPFG_REF)")
    if "easydict" not in sys.modules:                       # utils/utils.py:3 imports it at module top
        stub = types.ModuleType("easydict")

        class EasyDict(dict):
            __getattr__ = dict.__getitem__
            __setattr__ = dict.__setitem__
        stub.EasyDict = EasyDict
        sys.modules["easydict"] = stub
    ns = types.SimpleNamespace(root=root)
    unet = _load("_hpfg_ref_unet", os.path.join(root, "model", "unet.py"))
    medloss = _load("_hpfg_ref_medloss", os.path.join(root, "utils", "loss", "medloss.py"))
    diceloss = _load("_hpfg_ref_diceloss", os.path.join(root, "utils", "loss", "diceloss.py"))
    utils = _load("_hpfg_ref_utils", os.path.join(root, "utils", "utils.py"))
    mlr = _load("_hpfg_ref_medical_lr", os.path.join(root, "utils", "scheduler", "medical_lr.py"))
    ns.UNet = unet.UNet
    ns.UNet_Plus = unet.UNet_Plus
    ns.Med_Sup_Loss = medloss.Med_Sup_Loss
    ns.DiceLoss = diceloss.DiceLoss
    ns.Dense_Loss = _load("_hpfg_ref_dense_loss", os.path.join(root, "utils", "loss", "dense_loss.py")).Dense_Loss
    ns.softmax_mse_loss = diceloss.softmax_mse_loss
    ns.update_ema_variables = utils.update_ema_variables
    ns.get_current_consistency_weight = utils.get_current_consistency_weight
    ns.sigmoid_rampup = utils.sigmoid_rampup
    ns.linear_rampup = utils.linear_rampup
    ns.Medical_LR = mlr.Medical_LR
    return ns
