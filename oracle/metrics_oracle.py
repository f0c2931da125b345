"""fp64 numpy restatement of the evaluation metrics -- TEST INFRASTRUCTURE ONLY (like the rest of oracle/).

What bin_b200.metrics computes on the GPU, restated on the CPU so that tests can check it without the reference:

  psnr_util     utils/util.py:201-208   20 log10(255 / sqrt(mse)), inf for mse 0
  psnr_skimage  skimage 0.14 compare_psnr: 10 log10(data_range^2 / mse), data_range 255 for uint8
  mae           test.py:431-435         mean |rec - gt| ("interpolation error")
  ssim_util     utils/util.py:211-231 ssim (= calculate_ssim, :234-252, for 1- and 3-channel input)
  ssim_box7     skimage 0.14 compare_ssim(X, Y, multichannel=True) with its defaults, from exact integer window sums
  ssim_box7_scipy  the same through scipy.ndimage.uniform_filter, as skimage computes it

skimage 0.14-0.16 compare_ssim defaults (skimage/measure/_structural_similarity.py): win_size 7, K1 0.01, K2 0.03,
use_sample_covariance True (cov_norm = NP / (NP - 1), NP = 49), data_range = dtype range (255 for uint8),
filter = uniform_filter(size=7), mean over crop(S, (win_size - 1) // 2); with multichannel=True the result is the
mean over channels of the per-channel values.

Both SSIMs are valid-region filters: the reference crops exactly the map entries whose window leaves the image.
"""
from __future__ import annotations

import math

import numpy as np

C1 = (0.01 * 255) ** 2          # util.py:212, skimage (K1 * R) ** 2
C2 = (0.03 * 255) ** 2          # util.py:213


def make_pair(seed: int, shape, noise: int = 24):
    """Seeded uint8 pair: a uniform, b = clip(a + uniform integer noise in [-noise, noise])."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, size=shape, dtype=np.uint8)
    d = rng.integers(-noise, noise + 1, size=shape)
    b = np.clip(a.astype(np.int64) + d, 0, 255).astype(np.uint8)
    return a, b


def mse(a: np.ndarray, b: np.ndarray) -> float:
    return float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))          # util.py:203-205


def mae(a: np.ndarray, b: np.ndarray) -> float:
    return float(np.mean(np.abs(a.astype(np.float64) - b.astype(np.float64))))        # test.py:431-435


def psnr_util(a, b) -> float:
    m = mse(a, b)
    return float("inf") if m == 0 else 20 * math.log10(255.0 / math.sqrt(m))           # util.py:206-208


def psnr_skimage(a, b) -> float:
    m = mse(a, b)
    return float("inf") if m == 0 else float(10 * np.log10((255 ** 2) / m))


def gaussian_kernel_11() -> np.ndarray:
    """cv2.getGaussianKernel(11, 1.5) in double: exp(-x^2 / (2 sigma^2)), then times 1 / sum."""
    x = np.arange(11, dtype=np.float64) - 5.0
    t = np.exp((-0.5 / (1.5 * 1.5)) * x * x)
    return t * (1.0 / t.sum())


def _valid_sep(img: np.ndarray, k: np.ndarray) -> np.ndarray:
    """Valid-region separable correlation of a 2-D float64 image with the outer product k k^T."""
    K = k.size
    h, w = img.shape
    rows = sum(k[j] * img[:, j:w - K + 1 + j] for j in range(K))
    return sum(k[j] * rows[j:h - K + 1 + j, :] for j in range(K))


def _ssim_util_2d(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """util.py:211-229 ssim_map of one channel, valid region."""
    g = gaussian_kernel_11()
    x = x.astype(np.float64)
    y = y.astype(np.float64)
    mu1, mu2 = _valid_sep(x, g), _valid_sep(y, g)
    mu1_sq, mu2_sq, mu1_mu2 = mu1 ** 2, mu2 ** 2, mu1 * mu2
    s1 = _valid_sep(x * x, g) - mu1_sq
    s2 = _valid_sep(y * y, g) - mu2_sq
    s12 = _valid_sep(x * y, g) - mu1_mu2
    return ((2 * mu1_mu2 + C1) * (2 * s12 + C2)) / ((mu1_sq + mu2_sq + C1) * (s1 + s2 + C2))


def ssim_util(a: np.ndarray, b: np.ndarray) -> float:
    """utils.util.calculate_ssim: mean over every element of the valid (h-10, w-10, c) map."""
    if a.ndim == 2:
        return float(_ssim_util_2d(a, b).mean())
    return float(np.stack([_ssim_util_2d(a[..., ch], b[..., ch]) for ch in range(a.shape[2])], -1).mean())


def _box_sums(img: np.ndarray, K: int) -> np.ndarray:
    """Exact int64 KxK valid-region window sums."""
    c = np.zeros((img.shape[0] + 1, img.shape[1] + 1), dtype=np.int64)
    c[1:, 1:] = img.astype(np.int64).cumsum(0).cumsum(1)
    return c[K:, K:] - c[:-K, K:] - c[K:, :-K] + c[:-K, :-K]


def _ssim_box7_2d(x: np.ndarray, y: np.ndarray) -> float:
    """skimage compare_ssim of one channel from integer window sums: with ux = Sx/N and vx = (N Sxx - Sx^2)/(N(N-1))
    the factors 1/N^2 and 1/(N(N-1)) of skimage's A1 A2 / (B1 B2) cancel."""
    N = 49
    x = x.astype(np.int64)
    y = y.astype(np.int64)
    sx, sy = _box_sums(x, 7), _box_sums(y, 7)
    sxx, syy, sxy = _box_sums(x * x, 7), _box_sums(y * y, 7), _box_sums(x * y, 7)
    nx, ny, nxy = N * sxx - sx * sx, N * syy - sy * sy, N * sxy - sx * sy
    a1 = (2 * sx * sy).astype(np.float64) + (N * N) * C1
    a2 = (2 * nxy).astype(np.float64) + (N * (N - 1)) * C2
    b1 = (sx * sx + sy * sy).astype(np.float64) + (N * N) * C1
    b2 = (nx + ny).astype(np.float64) + (N * (N - 1)) * C2
    return float(((a1 * a2) / (b1 * b2)).mean())


def _ssim_box7_scipy_2d(x: np.ndarray, y: np.ndarray) -> float:
    """skimage 0.14 compare_ssim body for one channel (uniform_filter, cov_norm 49/48, crop 3)."""
    from scipy.ndimage import uniform_filter
    X, Y = x.astype(np.float64), y.astype(np.float64)
    f = lambda t: uniform_filter(t, size=7)
    ux, uy = f(X), f(Y)
    uxx, uyy, uxy = f(X * X), f(Y * Y), f(X * Y)
    cov_norm = 49.0 / 48.0
    vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
    A1, A2, B1, B2 = 2 * ux * uy + C1, 2 * vxy + C2, ux ** 2 + uy ** 2 + C1, vx + vy + C2
    S = (A1 * A2) / (B1 * B2)
    return float(S[3:-3, 3:-3].mean())


def _per_channel_mean(fn, a, b) -> float:
    if a.ndim == 2:
        return fn(a, b)
    return float(np.mean([fn(a[..., ch], b[..., ch]) for ch in range(a.shape[2])]))


def ssim_box7(a: np.ndarray, b: np.ndarray) -> float:
    return _per_channel_mean(_ssim_box7_2d, a, b)


def ssim_box7_scipy(a: np.ndarray, b: np.ndarray) -> float:
    return _per_channel_mean(_ssim_box7_scipy_2d, a, b)
