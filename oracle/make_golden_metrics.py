"""Generate tests/golden/metrics.npz by EXECUTING THE UNMODIFIED REFERENCE utils/util.py (laomao0/BIN):

    python oracle/make_golden_metrics.py /path/to/BIN

Needs what util.py imports (cv2, torch, torchvision, yaml).  For every case it records util.calculate_psnr,
util.calculate_ssim and util.ssim (the function calculate_ssim averages; util.py:211-252):

  rand_<shape>   seeded pairs from oracle.metrics_oracle.make_pair at 11x11x3, 12x13 (2-D), 37x53x3, 64x96x3,
                 127x255x3; pixels stored as <name>_a / <name>_b
  identical      one image against itself (PSNR inf, SSIM 1)
  constant       two different constant images
  black_white    all-0 against all-255
  hd             one 720x1280x3 pair; only its seed is stored (<name>_seed), make_pair(seed, shape) rebuilds it
tests/test_metrics_cpu.py checks oracle.metrics_oracle against these values; tests/test_gpu_metrics.py checks the
kernels against them.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
if len(sys.argv) != 2 or not os.path.isfile(os.path.join(sys.argv[1], "utils", "util.py")):
    raise SystemExit(__doc__)
sys.path.insert(0, os.path.abspath(sys.argv[1]))

import utils.util as util                         # noqa: E402  (the reference itself)
from oracle.metrics_oracle import make_pair       # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "metrics.npz")
HD_SEED, HD_SHAPE = 720, (720, 1280, 3)


def main():
    cases = {}
    for i, shape in enumerate([(11, 11, 3), (12, 13), (37, 53, 3), (64, 96, 3), (127, 255, 3)]):
        cases["rand_" + "x".join(map(str, shape))] = make_pair(100 + i, shape)
    rng = np.random.default_rng(7)
    img = rng.integers(0, 256, size=(16, 24, 3), dtype=np.uint8)
    cases["identical"] = (img, img.copy())
    cases["constant"] = (np.full((16, 24, 3), 100, np.uint8), np.full((16, 24, 3), 37, np.uint8))
    cases["black_white"] = (np.zeros((16, 24, 3), np.uint8), np.full((16, 24, 3), 255, np.uint8))
    out = {"names": np.array(sorted(cases) + ["hd"])}
    for name, (a, b) in cases.items():
        out[name + "_a"], out[name + "_b"] = a, b
    cases["hd"] = make_pair(HD_SEED, HD_SHAPE)
    out["hd_seed"] = np.array(HD_SEED)
    out["hd_shape"] = np.array(HD_SHAPE)
    for name, (a, b) in cases.items():
        out[name + "_calculate_psnr"] = np.float64(util.calculate_psnr(a, b))
        out[name + "_calculate_ssim"] = np.float64(util.calculate_ssim(a, b))
        out[name + "_ssim"] = np.float64(util.ssim(a, b))
        print(f"{name:16s} psnr {out[name + '_calculate_psnr']:.12f}  ssim {out[name + '_calculate_ssim']:.15f}")
    np.savez_compressed(OUT, **out)
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
