"""GPU checks of bin_b200.metrics (csrc/metrics.cu): accuracy against the reference's own util.py values
(tests/golden/metrics.npz) and the fp64 oracle, edge cases, bit-exact determinism, argument errors, and the drop-ins
on the images test.py writes."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

TOL_SSIM = 1e-9
TOL_PSNR = 1e-9      # dB
TOL_MAE = 1e-12


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "metrics.npz"))


def golden_pair(g, name):
    if name == "hd":
        return MO.make_pair(int(g["hd_seed"]), tuple(int(v) for v in g["hd_shape"]))
    return g[name + "_a"], g[name + "_b"]


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def metrics(a, b, kind):
    from bin_b200.metrics import image_metrics
    return [t.item() for t in image_metrics(dev(a), dev(b), kind)]


def assert_psnr(x, want, what):
    if math.isinf(want):
        assert x == want, what
    else:
        assert abs(x - want) <= TOL_PSNR, (what, x, want)


def check_pair(a, b, what, util_ssim=None, util_psnr=None):
    """Both kinds of one pair against the oracle (and the reference's util values when given)."""
    for kind in ("skimage", "util"):
        if min(a.shape[:2]) < (7 if kind == "skimage" else 11):
            continue
        psnr, ssim, mae = metrics(a, b, kind)
        if kind == "util":
            want = MO.ssim_util(a, b) if util_ssim is None else util_ssim
        else:
            want = MO.ssim_box7(a, b)
        assert abs(ssim - want) <= TOL_SSIM, (what, kind, ssim, want)
        assert_psnr(psnr, MO.psnr_skimage(a, b) if util_psnr is None else util_psnr, (what, kind))
        assert abs(mae - MO.mae(a, b)) <= TOL_MAE, (what, kind, mae)


def test_golden_shapes_both_kinds_c1_and_c3(golden):
    for name in [str(n) for n in golden["names"]]:
        a, b = golden_pair(golden, name)
        check_pair(a, b, name, float(golden[name + "_calculate_ssim"]), float(golden[name + "_calculate_psnr"]))
        if a.ndim == 3:                                           # the same pixels as single-channel images
            check_pair(a[..., :1], b[..., :1], name + "[c=1]")
            check_pair(a[..., 1], b[..., 1], name + "[2-D]")


def test_minimum_and_odd_sizes():
    for i, shape in enumerate([(7, 7, 1), (7, 7, 3), (11, 11, 1), (11, 11, 3), (7, 300, 3), (300, 7, 1),
                               (11, 77, 3), (17, 65, 3), (33, 129, 1), (81, 193, 3), (12, 13)]):
        a, b = MO.make_pair(300 + i, shape, noise=60)
        check_pair(a, b, shape)


def test_seeded_720p_pairs_c1_and_c3():
    for seed in (1, 2):
        a, b = MO.make_pair(seed, (720, 1280, 3), noise=40)
        check_pair(a, b, ("720p", seed))
    check_pair(a[..., :1], b[..., :1], "720p c=1")


def test_edge_cases(golden):
    from bin_b200.metrics import image_metrics
    a, _ = golden_pair(golden, "identical")
    for kind in ("skimage", "util"):
        psnr, ssim, mae = image_metrics(dev(a), dev(a.copy()), kind)
        assert ssim.item() == 1.0 and psnr.item() == math.inf and mae.item() == 0.0, kind
        assert psnr.dtype == ssim.dtype == mae.dtype == torch.float64 and psnr.device.type == "cuda"
    for name in ("constant", "black_white"):
        a, b = golden_pair(golden, name)
        check_pair(a, b, name, float(golden[name + "_calculate_ssim"]), float(golden[name + "_calculate_psnr"]))
    a, b = golden_pair(golden, "black_white")
    psnr, ssim, mae = metrics(a, b, "skimage")
    assert psnr == 0.0 and mae == 255.0


def test_deterministic_across_calls_batches_and_streams():
    from bin_b200.metrics import image_metrics
    pairs = [MO.make_pair(500 + k, (97, 131, 3), noise=30) for k in range(70)]
    A = torch.stack([dev(a) for a, _ in pairs])
    B = torch.stack([dev(b) for _, b in pairs])
    for kind in ("skimage", "util"):
        full = torch.stack(image_metrics(A, B, kind))                      # 70 pairs: split 64 + 6
        assert full.shape == (3, 70)
        again = torch.stack(image_metrics(A, B, kind))
        assert torch.equal(full, again), kind
        four = torch.stack(image_metrics(A[:4], B[:4], kind))
        assert torch.equal(four, full[:, :4]), kind
        for k in (0, 3, 65, 69):
            one = torch.stack(image_metrics(A[k], B[k], kind))
            assert torch.equal(one, full[:, k]), (kind, k)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            side = torch.stack(image_metrics(A, B, kind))
        torch.cuda.current_stream().wait_stream(s)
        assert torch.equal(side, full), kind


def test_invalid_arguments_raise():
    from bin_b200 import BinB200Error, _lib
    from bin_b200.metrics import image_metrics
    a = torch.zeros((16, 16, 3), dtype=torch.uint8, device="cuda")
    bad = [
        lambda: image_metrics(a.cpu(), a.cpu()),
        lambda: image_metrics(a.float(), a.float()),
        lambda: image_metrics(a, a[:, :15]),
        lambda: image_metrics(a, a, kind="gauss"),
        lambda: image_metrics(a[..., :2], a[..., :2]),
        lambda: image_metrics(a[:6], a[:6], "skimage"),
        lambda: image_metrics(a[:, :10], a[:, :10], "util"),
        lambda: image_metrics(a[None, None], a[None, None]),
    ]
    for call in bad:
        with pytest.raises(BinB200Error):
            call()
    # the C ABI checks its own arguments
    L = _lib.lib()
    ws = torch.empty(L.bin_image_metrics_workspace_bytes(1, 16, 16, 3, 0), dtype=torch.uint8, device="cuda")
    res = torch.empty((2, 3), dtype=torch.float64, device="cuda")
    P = lambda *ts: (C.c_void_p * len(ts))(*[t.data_ptr() if t is not None else None for t in ts])
    s = torch.cuda.current_stream().cuda_stream
    call = lambda ap, bp, n, h, w, c, kind, r, wsp, nb: _lib.check(L.bin_image_metrics_u8(ap, bp, n, h, w, c, kind, r, wsp, nb, s))
    ok = (P(a), P(a), 1, 16, 16, 3, 0, res.data_ptr(), ws.data_ptr(), ws.numel())
    call(*ok)
    for i, v in [(0, None), (1, None), (7, None), (8, None), (0, P(None)), (2, 0), (2, _lib.BIN_MAX_METRIC_PAIRS + 1),
                 (5, 2), (5, 4), (3, 6), (4, 6), (6, 2), (6, -1), (9, ws.numel() - 1)]:
        args = list(ok)
        args[i] = v
        with pytest.raises(BinB200Error):
            call(*args)
    torch.cuda.synchronize()


def test_dropins_on_the_images_test_py_writes():
    """test.py:404-458 on one window driven through the caller harness: the skimage and util drop-ins on the three
    images test.py writes, against a GT image, equal the oracle's values."""
    from caller_harness import CallerModel, run_test_py_window
    from oracle import bin_oracle as O
    from bin_b200 import metrics as M, rdn
    sd = O.synth_state_dict(0)
    model = CallerModel(rdn.bin_stage4_lstm(), "cuda:0", device_ids=[0])
    model.load_state_dict_like_load_network({"InterpNet." + k: v for k, v in sd.items()})
    frames = [f[0] for f in O.synth_frames(6, 1, 96, 160, seed=11, smooth=True)]
    imgs, _, _ = run_test_py_window(model, frames)
    rng = np.random.default_rng(3)
    for img in imgs:
        assert img.shape == (96, 160, 3) and img.dtype == np.uint8
        rec_rgb = img[:, :, [2, 1, 0]]                                    # test.py:58-66 read_image_np: BGR -> RGB
        gt = np.clip(rec_rgb.astype(np.int64) + rng.integers(-9, 10, size=rec_rgb.shape), 0, 255).astype(np.uint8)
        assert_psnr(M.compare_psnr(rec_rgb, gt), MO.psnr_skimage(rec_rgb, gt), "compare_psnr")
        assert abs(M.compare_ssim(rec_rgb, gt, multichannel=True) - MO.ssim_box7(rec_rgb, gt)) <= TOL_SSIM
        assert_psnr(M.calculate_psnr(rec_rgb, gt), MO.psnr_util(rec_rgb, gt), "calculate_psnr")
        assert abs(M.calculate_ssim(rec_rgb, gt) - MO.ssim_util(rec_rgb, gt)) <= TOL_SSIM
        assert M.compare_psnr(gt, gt) == math.inf and M.compare_ssim(gt, gt, multichannel=True) == 1.0
        # test.py:431-435 interpolation error = mean |rec - gt|
        _, _, mae = M.image_metrics(dev(rec_rgb), dev(gt))
        assert abs(mae.item() - MO.mae(rec_rgb, gt)) <= TOL_MAE
