"""Seconds per validation pass of val.py's test_single_volume over a synthetic ACDC-shaped test split, on one GPU:
    python profiles/val_throughput.py [--precision fp32|bf16] [--rounds 3]      (profiles/val_throughput.txt: both precisions)

The split: 20 volumes of 6..18 slices at the in-plane sizes of ACDC's test volumes (256x216, 232x256, 154x224, 224x224),
images of smooth random intensities, labels of smooth random blobs of 4 classes; a fixed seeded U-Net (the library's, eval mode)
at the 224x224 patch size.  Two paths run in the same process and alternate pass by pass:

  reference  val.py as written: the network at batch 1 on the GPU, scipy.ndimage.zoom(order=0) on the host, and medpy's dc /
             hd95 as restated in oracle/val_ref.py (scipy binary_erosion, distance_transform_edt, numpy.percentile) on the host;
  device     hpfg_b200.test_single_volume: one copy of each volume in, zoom / network / zoom back / metrics on the GPU, one read of
             the integer result block.

Both passes' metric lists must be identical.  The card name and power limit are read at the start of the run."""
import argparse, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import hpfg_b200 as hb
from hpfg_b200.validation import volume_metrics_raw
from oracle import val_ref
from tests.golden.common import make_predict_case
from tests.val_cases import blobs

ap = argparse.ArgumentParser()
ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"])
ap.add_argument("--rounds", type=int, default=3)
args = ap.parse_args()

dev = torch.device("cuda:0")
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except Exception as exc:          # the card name still comes from torch
    smi = "power limit not read (%s)" % exc
lines = ["device: %s | nvidia-smi: %s | host cores: %d" % (torch.cuda.get_device_name(dev), smi, os.cpu_count())]

PATCH = (224, 224)
SIZES = [(256, 216), (232, 256), (154, 224), (224, 224)]
rng = np.random.default_rng(0)
split = []
for k in range(20):
    s = int(rng.integers(6, 19))
    h, w = SIZES[k % len(SIZES)]
    g = torch.Generator().manual_seed(100 + k)
    coarse = torch.rand(s, 1, 4, 6, generator=g)
    image = torch.nn.functional.interpolate(coarse, size=(h, w), mode="bilinear", align_corners=True)[:, 0]
    image = (image + 0.05 * torch.rand(s, h, w, generator=g)).contiguous()
    split.append((image[None], torch.from_numpy(blobs((s, h, w), 4, 200 + k))[None]))   # [1,S,H,W] as the loader yields them
voxels = sum(int(lab.numel()) for _, lab in split)
lines.append("split: %d volumes, %d slices, %d voxels; patch %dx%d; %s U-Net" % (len(split), sum(int(i.shape[1]) for i, _ in split),
                                                                               voxels, PATCH[0], PATCH[1], args.precision))

st, _ = make_predict_case(1, 4, 1, 8, 8, 5)
net = hb.UNet(1, 4, precision=args.precision)
net.load_state_dict(st)
net.to(dev).eval()


def reference_pass():
    out = []
    for image, label in split:
        def predict_slice(sl):                    # val.py:273-276: batch 1 on the GPU, labels back to the host
            with torch.no_grad():
                x = torch.from_numpy(sl).unsqueeze(0).unsqueeze(0).float().to(dev)
                return torch.argmax(torch.softmax(net(x), dim=1), dim=1).squeeze(0).cpu().numpy()
        out.append(val_ref.test_single_volume(image[0].numpy(), label[0].numpy(), predict_slice, 4, PATCH)[0])
    return out


def device_pass():
    return [hb.test_single_volume(image, label, net, 4, patch_size=list(PATCH)) for image, label in split]


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def as_floats(ms):
    return [[(float(a), float(b)) for a, b in m] for m in ms]


timed(device_pass)                                # warm-up: plans, modules
times = {"reference": [], "device": []}
identical = True
for _ in range(args.rounds):
    tr, rr = timed(reference_pass)
    td, rd = timed(device_pass)
    times["reference"].append(tr)
    times["device"].append(td)
    identical &= as_floats(rr) == as_floats(rd)
for name, ts in times.items():
    med = float(np.median(ts))
    lines.append("%-9s: %.4f s per validation pass (median of %d; min %.4f, max %.4f)  %.2f ms per volume"
                 % (name, med, len(ts), min(ts), max(ts), 1e3 * med / len(split)))
preds = [hb.predict_single_volume(image, net, list(PATCH)) for image, _ in split]
labels = [lab[0].to(dev) for _, lab in split]
parts = {"network": [], "metrics": []}
for _ in range(args.rounds):                      # where the device pass spends its time
    parts["network"].append(timed(lambda: [hb.predict_single_volume(image, net, list(PATCH)) for image, _ in split])[0])
    parts["metrics"].append(timed(lambda: [volume_metrics_raw(p, l, 4) for p, l in zip(preds, labels)])[0])
lines.append("device pass parts: zoom + network + argmax + zoom back %.4f s, metrics kernels (inputs resident) %.4f s"
             % (np.median(parts["network"]), np.median(parts["metrics"])))
ratio = np.median(times["reference"]) / np.median(times["device"])
lines.append("speed-up of the device path: %.1fx" % ratio)
lines.append("metric lists of the two paths identical in every pass: %s" % ("yes" if identical else "NO"))
lines.append("first volumes' (dice, hd95): %s" % as_floats(rd)[:2])
print("\n".join(lines))
sys.exit(0 if identical else 1)
