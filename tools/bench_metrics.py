"""Per-window cost of test.py's metrics: bin_b200.metrics.image_metrics on the GPU vs the host implementations.

One test.py window scores four 1280x720x3 uint8 pairs (test.py:404-458: two deblurred frames, one interpolated frame,
the blurry input).  Device time: CUDA events around >= 200 calls of image_metrics on those 4 pairs, after a warm-up,
for each SSIM kind; "hot" reuses one window (its 22 MB stay in the 126 MB L2), "cold" cycles through 8 windows
(177 MB).  Host time: one pair through fp64 CPU formulations of the same metrics, times 4:
  util_cv2      utils/util.py:211-252 calculate_ssim as the reference computes it (cv2.filter2D, 11x11 Gaussian,
                whole-image SSIM three times for 3-channel input)
  skimage_scipy skimage 0.14 compare_ssim(multichannel=True) through scipy uniform_filter (oracle/metrics_oracle.py)
  psnr_numpy    utils/util.py:201-208 calculate_psnr
With BIN_REFERENCE_ROOT pointing at a reference checkout, the unmodified util.calculate_ssim / calculate_psnr are
timed as well.  Prints the card name and power limit with the numbers.  The host leg is the slow part: the cv2
formulation alone can take minutes on a shared host.

    python tools/bench_metrics.py [--iters 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bin_b200.metrics import image_metrics          # noqa: E402
from oracle import metrics_oracle as MO             # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def device_ms(A, B, kind, iters):
    n = len(A)
    for i in range(10):
        image_metrics(A[i % n], B[i % n], kind)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        image_metrics(A[i % n], B[i % n], kind)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def cv2_util_ssim(a, b):
    """utils/util.py:211-231 ssim, with cv2.filter2D as the reference calls it."""
    import cv2
    a, b = a.astype(np.float64), b.astype(np.float64)
    k = cv2.getGaussianKernel(11, 1.5)
    win = np.outer(k, k.transpose())
    f = lambda t: cv2.filter2D(t, -1, win)[5:-5, 5:-5]
    mu1, mu2 = f(a), f(b)
    s1, s2, s12 = f(a * a) - mu1 ** 2, f(b * b) - mu2 ** 2, f(a * b) - mu1 * mu2
    return (((2 * mu1 * mu2 + MO.C1) * (2 * s12 + MO.C2)) / ((mu1 ** 2 + mu2 ** 2 + MO.C1) * (s1 + s2 + MO.C2))).mean()


def host_ms(fn, a, b, reps=1):
    t = time.perf_counter()
    for _ in range(reps):
        fn(a, b)
    return (time.perf_counter() - t) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_metrics: no CUDA device")
    windows = []
    for w in range(8):
        pairs = [MO.make_pair(1000 + 4 * w + k, (720, 1280, 3)) for k in range(4)]
        windows.append((torch.stack([torch.from_numpy(a) for a, _ in pairs]).cuda(),
                        torch.stack([torch.from_numpy(b) for _, b in pairs]).cuda()))
    A = [a for a, _ in windows]
    B = [b for _, b in windows]
    out = {"card": card(), "pairs_per_window": 4, "shape": [720, 1280, 3], "iters": args.iters, "device_ms_per_window": {}}
    for kind in ("skimage", "util"):
        out["device_ms_per_window"][kind] = {"hot": device_ms(A[:1], B[:1], kind, args.iters),
                                             "cold": device_ms(A, B, kind, args.iters)}
    a, b = MO.make_pair(1000, (720, 1280, 3))
    per_pair = {
        "util_cv2_calculate_ssim": host_ms(lambda x, y: [cv2_util_ssim(x, y) for _ in range(3)], a, b),
        "skimage_scipy_compare_ssim": host_ms(MO.ssim_box7_scipy, a, b),
        "psnr_numpy": host_ms(MO.psnr_util, a, b, reps=5),
    }
    ref = os.environ.get("BIN_REFERENCE_ROOT")
    if ref and os.path.isfile(os.path.join(ref, "utils", "util.py")):
        sys.path.insert(0, ref)
        import utils.util as util
        per_pair["reference_util_calculate_ssim"] = host_ms(util.calculate_ssim, a, b)
        per_pair["reference_util_calculate_psnr"] = host_ms(util.calculate_psnr, a, b, reps=5)
    out["host_ms_per_window"] = {k: 4 * v for k, v in per_pair.items()}
    out["host_threads"] = torch.get_num_threads()
    out["host_cpus"] = os.cpu_count()
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
