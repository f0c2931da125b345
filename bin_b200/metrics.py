"""Image-quality metrics of the evaluation loop on the GPU: PSNR, SSIM and mean absolute error of uint8 images.

`image_metrics(a, b, kind)` computes them for a batch of image pairs on the device, with no host synchronisation.
`kind` picks one of the two SSIM definitions the reference uses:

  "skimage"  skimage 0.14-0.16 `compare_ssim(X, Y, multichannel=True)` with its defaults, which is what test.py:33-35
             reports (7x7 uniform window, sample covariance);
  "util"     utils/util.py:211-252 `calculate_ssim`, which is what bin_model.compute_current_psnr_ssim
             (bin_model.py:564-589) reports (11x11 Gaussian window, sigma 1.5).

The module also provides drop-ins with the reference's signatures that take numpy uint8 HWC images and return Python
floats: `compare_psnr` / `compare_ssim` for `skimage.measure` (so `sys.modules["skimage.measure"] = bin_b200.metrics`
lets test.py run unchanged) and `calculate_psnr` / `calculate_ssim` for `utils.util`.  They implement exactly the
configuration the reference calls; any other keyword value or a non-uint8 image raises instead of computing something
else.  Every computation runs in libbin_b200.so (csrc/metrics.cu); there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Tuple

import numpy as np
import torch

from ._lib import BIN_MAX_METRIC_PAIRS, SSIM_BOX7, SSIM_GAUSS11, BinB200Error, check, lib

KINDS = {"skimage": SSIM_BOX7, "util": SSIM_GAUSS11}
WINDOW = {SSIM_BOX7: 7, SSIM_GAUSS11: 11}


def _as_nhwc(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.dim() == 2:
        return t.unsqueeze(0).unsqueeze(-1)
    if t.dim() == 3:
        return t.unsqueeze(0)
    if t.dim() == 4:
        return t
    raise BinB200Error(f"{name}: expected shape (h, w), (h, w, c) or (n, h, w, c), got {tuple(t.shape)}")


def _metrics(a: torch.Tensor, b: torch.Tensor, kind: int) -> torch.Tensor:
    """(n, 3) float64 device tensor of {mse, mae, ssim} per pair."""
    for t, name in ((a, "a"), (b, "b")):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise BinB200Error(f"image_metrics: {name} must be a CUDA tensor (bin_b200 has no CPU path)")
        if t.dtype != torch.uint8:
            raise BinB200Error(f"image_metrics: {name} must be uint8, got {t.dtype}")
    if a.shape != b.shape:
        raise BinB200Error(f"image_metrics: shapes differ: {tuple(a.shape)} vs {tuple(b.shape)}")
    if a.device != b.device:
        raise BinB200Error("image_metrics: a and b are on different devices")
    a, b = _as_nhwc(a, "a").contiguous(), _as_nhwc(b, "b").contiguous()
    n, h, w, c = a.shape
    if c not in (1, 3):
        raise BinB200Error(f"image_metrics: channels must be 1 or 3, got {c}")
    K = WINDOW[kind]
    if h < K or w < K:
        raise BinB200Error(f"image_metrics: {h}x{w} image is smaller than the {K}x{K} SSIM window")
    res = torch.empty((n, 3), dtype=torch.float64, device=a.device)
    if n == 0:
        return res
    L = lib()
    with torch.cuda.device(a.device):
        stream = torch.cuda.current_stream().cuda_stream
        for k0 in range(0, n, BIN_MAX_METRIC_PAIRS):
            m = min(BIN_MAX_METRIC_PAIRS, n - k0)
            ws_bytes = L.bin_image_metrics_workspace_bytes(m, h, w, c, kind)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=a.device)        # caching allocator, stream-ordered
            ap = (C.c_void_p * m)(*[a[k].data_ptr() for k in range(k0, k0 + m)])
            bp = (C.c_void_p * m)(*[b[k].data_ptr() for k in range(k0, k0 + m)])
            check(L.bin_image_metrics_u8(ap, bp, m, h, w, c, kind, res[k0].data_ptr(), ws.data_ptr(), ws_bytes, stream))
    return res


def image_metrics(a: torch.Tensor, b: torch.Tensor, kind: str = "skimage") -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """PSNR, SSIM and mean absolute error of uint8 CUDA images a vs b, shape (h, w), (h, w, c) or (n, h, w, c) with
    c = 1 or 3.  Returns float64 tensors on the inputs' device, of shape () for one image and (n,) for a batch:
    psnr = 10 log10(255^2 / mse) (inf for identical images), ssim of the given kind, mae = mean |a - b| (test.py's
    "interpolation error", test.py:431-435).  Runs on the device's current stream without synchronising."""
    if kind not in KINDS:
        raise BinB200Error(f"image_metrics: kind must be one of {sorted(KINDS)}, got {kind!r}")
    res = _metrics(a, b, KINDS[kind])
    if isinstance(a, torch.Tensor) and a.dim() < 4:
        res = res[0]
    mse, mae, ssim = res.unbind(-1)
    psnr = 10.0 * torch.log10((255.0 * 255.0) / mse)
    return psnr, ssim, mae


# ---------------------------------------------------------------------------------------------- reference drop-ins
def _check_image(x, name: str) -> np.ndarray:
    if not isinstance(x, np.ndarray):
        raise BinB200Error(f"{name}: expected a numpy array, got {type(x).__name__}")
    if x.dtype != np.uint8:
        raise BinB200Error(f"{name}: only uint8 images are implemented, got {x.dtype}")
    return x


def _check_pair(x, y) -> None:
    _check_image(x, "first image")
    _check_image(y, "second image")
    if x.shape != y.shape:
        raise BinB200Error(f"input images must have the same dimensions: {x.shape} vs {y.shape}")
    if x.ndim not in (2, 3) or (x.ndim == 3 and x.shape[2] not in (1, 3)):
        raise BinB200Error(f"expected an (h, w), (h, w, 1) or (h, w, 3) image, got shape {x.shape}")


def _host_metrics(x: np.ndarray, y: np.ndarray, kind: int) -> Tuple[float, float, float]:
    """(mse, mae, ssim) of one validated numpy pair, computed on the current CUDA device."""
    dev = torch.device("cuda", torch.cuda.current_device())
    a = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(y)).to(dev)
    mse, mae, ssim = _metrics(a, b, kind)[0].tolist()
    return mse, mae, ssim


def _no_extra(fn: str, kwargs) -> None:
    if kwargs:
        raise BinB200Error(f"{fn}: keyword(s) {sorted(kwargs)} are not implemented")


def compare_psnr(im_true, im_test, data_range=None, **kwargs) -> float:
    """skimage.measure.compare_psnr (0.14-0.16) for uint8 images of at least 7x7 pixels: 10 log10(255^2 / mse), inf
    when mse is 0."""
    _no_extra("compare_psnr", kwargs)
    if data_range not in (None, 255):
        raise BinB200Error("compare_psnr: only the uint8 data range 255 is implemented")
    _check_pair(im_true, im_test)
    mse = _host_metrics(im_true, im_test, SSIM_BOX7)[0]
    return float("inf") if mse == 0 else float(10 * np.log10((255 ** 2) / mse))


def compare_ssim(X, Y, win_size=None, gradient=False, data_range=None, multichannel=False, gaussian_weights=False,
                 full=False, **kwargs) -> float:
    """skimage.measure.compare_ssim (0.14-0.16) with its default 7x7 uniform window and sample covariance, for uint8
    images: (h, w, c) with multichannel=True (c = 1 or 3, mean of the per-channel SSIMs), or (h, w) with
    multichannel=False."""
    _no_extra("compare_ssim", kwargs)
    if win_size not in (None, 7) or gradient or data_range not in (None, 255) or gaussian_weights or full:
        raise BinB200Error("compare_ssim: only the default configuration (7x7 uniform window, data range 255, no "
                           "gradient / full map) is implemented")
    _check_pair(X, Y)
    if X.ndim == 3 and not multichannel:
        raise BinB200Error("compare_ssim: a 3-D image needs multichannel=True (volumetric SSIM is not implemented)")
    if X.ndim == 2 and multichannel:
        raise BinB200Error("compare_ssim: multichannel=True expects an (h, w, c) image")
    return _host_metrics(X, Y, SSIM_BOX7)[2]


def calculate_psnr(img1, img2) -> float:
    """utils/util.py:201-208 for uint8 images of at least 7x7 pixels: 20 log10(255 / sqrt(mse)), inf when mse is 0."""
    _check_pair(img1, img2)
    mse = _host_metrics(img1, img2, SSIM_BOX7)[0]
    return float("inf") if mse == 0 else 20 * math.log10(255.0 / math.sqrt(mse))


def calculate_ssim(img1, img2) -> float:
    """utils/util.py:234-252 for uint8 (h, w), (h, w, 1) or (h, w, 3) images (11x11 Gaussian window, sigma 1.5)."""
    _check_pair(img1, img2)
    return _host_metrics(img1, img2, SSIM_GAUSS11)[2]
