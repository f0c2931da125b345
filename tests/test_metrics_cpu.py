"""CPU checks of the evaluation-metric layer: the fp64 oracle against the reference's own util.py values
(tests/golden/metrics.npz), the two BOX7 formulations against each other, the workspace query, and the drop-ins'
argument checks (which must fire before any device is touched)."""
import math
import os

import numpy as np
import pytest

from oracle import metrics_oracle as MO


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "metrics.npz"))


def golden_pair(g, name):
    if name == "hd":
        return MO.make_pair(int(g["hd_seed"]), tuple(int(v) for v in g["hd_shape"]))
    return g[name + "_a"], g[name + "_b"]


def small_names(g):
    return [str(n) for n in g["names"] if str(n) != "hd"]


def _close(x, y, tol):
    if math.isinf(y):
        return x == y
    return abs(x - y) <= tol


def test_oracle_matches_reference_util(golden):
    for name in small_names(golden) + ["hd"]:
        a, b = golden_pair(golden, name)
        assert _close(MO.psnr_util(a, b), float(golden[name + "_calculate_psnr"]), 1e-10), name
        s = MO.ssim_util(a, b)
        assert abs(s - float(golden[name + "_calculate_ssim"])) <= 1e-12, (name, s)
        assert abs(s - float(golden[name + "_ssim"])) <= 1e-12, (name, s)
        assert _close(MO.psnr_skimage(a, b), float(golden[name + "_calculate_psnr"]), 1e-10), name


def test_box7_integer_and_scipy_formulations_agree(golden):
    for name in small_names(golden) + ["hd"]:
        a, b = golden_pair(golden, name)
        if min(a.shape[:2]) < 7:
            continue
        x, y = MO.ssim_box7(a, b), MO.ssim_box7_scipy(a, b)
        assert abs(x - y) <= 1e-12, (name, x, y)
    a, b = MO.make_pair(5, (7, 7, 1))           # the minimum size: a 1x1 map
    assert abs(MO.ssim_box7(a, b) - MO.ssim_box7_scipy(a, b)) <= 1e-12


def test_golden_edge_values(golden):
    assert float(golden["identical_calculate_psnr"]) == math.inf
    assert float(golden["identical_calculate_ssim"]) == 1.0
    a, b = golden_pair(golden, "black_white")
    assert float(golden["black_white_calculate_psnr"]) == 0.0
    assert MO.mae(a, b) == 255.0


def test_skimage_if_installed(golden):
    skm = pytest.importorskip("skimage.metrics")
    for name in ("rand_37x53x3", "rand_127x255x3", "constant"):
        a, b = golden_pair(golden, name)
        ref = skm.structural_similarity(a, b, channel_axis=-1)
        assert abs(MO.ssim_box7(a, b) - ref) <= 1e-12, name


def test_workspace_query_is_pure_and_grows():
    from bin_b200 import _lib
    L = _lib.lib()
    q = L.bin_image_metrics_workspace_bytes
    for kind in (_lib.SSIM_BOX7, _lib.SSIM_GAUSS11):
        base = q(1, 64, 96, 3, kind)
        assert base > 0 and q(1, 64, 96, 3, kind) == base
        assert q(2, 64, 96, 3, kind) > base
        assert q(1, 720, 1280, 3, kind) > q(1, 64, 96, 3, kind)
        assert q(1, 64, 96, 1, kind) < base
        assert q(_lib.BIN_MAX_METRIC_PAIRS, 720, 1280, 3, kind) >= _lib.BIN_MAX_METRIC_PAIRS * q(1, 720, 1280, 3, kind)
    # arguments the launch would reject size to 0
    assert q(0, 64, 96, 3, 0) == 0 and q(_lib.BIN_MAX_METRIC_PAIRS + 1, 64, 96, 3, 0) == 0
    assert q(1, 6, 96, 3, 0) == 0 and q(1, 10, 96, 3, 1) == 0 and q(1, 64, 96, 2, 0) == 0 and q(1, 64, 96, 3, 2) == 0
    assert q(1, 7, 7, 1, 0) > 0 and q(1, 11, 11, 1, 1) > 0


def test_dropins_reject_before_touching_a_device(monkeypatch):
    from bin_b200 import BinB200Error, metrics
    import torch

    def no_device(*args, **kwargs):
        raise AssertionError("a rejected call reached the device")

    monkeypatch.setattr(metrics, "_host_metrics", no_device)
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    a = np.zeros((16, 16, 3), np.uint8)
    bad = [
        lambda: metrics.compare_ssim(a, a, multichannel=True, win_size=11),
        lambda: metrics.compare_ssim(a, a, multichannel=True, gaussian_weights=True),
        lambda: metrics.compare_ssim(a, a, multichannel=True, data_range=1.0),
        lambda: metrics.compare_ssim(a, a, multichannel=True, full=True),
        lambda: metrics.compare_ssim(a, a, multichannel=True, gradient=True),
        lambda: metrics.compare_ssim(a, a, multichannel=True, use_sample_covariance=False),
        lambda: metrics.compare_ssim(a, a),                                      # 3-D without multichannel
        lambda: metrics.compare_ssim(a[..., 0], a[..., 0], multichannel=True),
        lambda: metrics.compare_ssim(a.astype(np.float64), a.astype(np.float64), multichannel=True),
        lambda: metrics.compare_ssim(a, a[:8], multichannel=True),
        lambda: metrics.compare_psnr(a, a, data_range=1.0),
        lambda: metrics.compare_psnr(a.astype(np.float32), a.astype(np.float32)),
        lambda: metrics.compare_psnr(a, a, dynamic_range=255),
        lambda: metrics.calculate_psnr(a.astype(np.uint16), a.astype(np.uint16)),
        lambda: metrics.calculate_ssim(a.astype(np.float64), a.astype(np.float64)),
        lambda: metrics.calculate_ssim(a, a[:, :8]),
        lambda: metrics.calculate_ssim(np.zeros((16, 16, 4), np.uint8), np.zeros((16, 16, 4), np.uint8)),
        lambda: metrics.calculate_ssim(torch.zeros((16, 16, 3), dtype=torch.uint8), a),
    ]
    for i, call in enumerate(bad):
        with pytest.raises(BinB200Error):
            call()


def test_image_metrics_rejects_cpu_tensors():
    import torch
    from bin_b200 import BinB200Error, metrics
    a = torch.zeros((16, 16, 3), dtype=torch.uint8)
    with pytest.raises(BinB200Error):
        metrics.image_metrics(a, a)
    with pytest.raises(BinB200Error):
        metrics.image_metrics(a, a, kind="matlab")
