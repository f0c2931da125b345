"""Cost of one training batch: bin_b200.train_data.DeviceBINDataset.batch on the GPU vs the reference's host loader.

The store is built with DeviceBINDataset.from_sharp_frames from random 240-fps frames of 352x640 (two clips of
`--frames` frames each); it holds the blurry frames and 3/8 of the sharp ones, larger than the 126 MB L2, and every
call draws fresh windows, crops and flips.  For B = 8 x 256x256 and B = 2 x 128x256 (the yml) it reports:
  call_ms        CUDA events around >= 200 back-to-back batch() calls, after a warm-up (host draws + launch + kernel)
  host_us        the host's share of one call (perf_counter around the same loop, no synchronise inside)
  kernel_us      train_batch_u8_kernel alone, from torch.profiler over the same number of calls (a separate pass)
  hbm_frac       algorithmic bytes (3 read + 12 written per output pixel and slot) / kernel time / 7.7 TB/s
  ref_loader_ms  the reference's per-batch host work on one core: 17 x cv2.imread of a 640x352 PNG, float32 / 255 of
                 the whole frame, crop, fliplr, BGR->RGB + CHW, stack (BIN_dataset.py:63-183, data/util.py:73-95);
                 "not measured" without cv2
and, for B = 8 x 256x256, one training step (forward, fused L1 get_loss, backward, Adam) fed by batch() against one
fed by a batch built once, alternated.  Prints the card name and power limit with the numbers, one JSON document.

    python tools/bench_train_batch.py [--iters 200] [--frames 480] [--out FILE]
"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bin_b200.train_data import DeviceBINDataset  # noqa: E402

HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def time_calls(ds, B, iters, rng):
    n = len(ds)
    for _ in range(20):
        ds.batch([rng.randrange(n) for _ in range(B)], rng)
    torch.cuda.synchronize()
    idx = [[rng.randrange(n) for _ in range(B)] for _ in range(iters)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for i in idx:
        ds.batch(i, rng)
    t1 = time.perf_counter()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (t1 - t0) / iters * 1e6


def kernel_us(ds, B, iters, rng):
    from torch.profiler import ProfilerActivity, profile
    n = len(ds)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            ds.batch([rng.randrange(n) for _ in range(B)], rng)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if "train_batch_u8_kernel" in e.name]
    if len(ev) != iters:
        raise RuntimeError(f"profiler saw {len(ev)} train_batch_u8_kernel launches, expected {iters}")
    return sum(e.device_time for e in ev) / iters


def ref_loader_ms(B, h, w, reps=3):
    try:
        import cv2
    except ImportError:
        return "not measured (no cv2)"
    yy, xx = np.mgrid[0:352, 0:640]
    rng = np.random.default_rng(0)
    with tempfile.TemporaryDirectory() as d:
        paths = []
        for k in range(17):            # natural-looking content: smooth gradients + mild noise (PNG cost depends on it)
            img = np.stack([(yy * (1 + c) + xx * (k + 1) // 3 + 40 * np.sin(xx / (20 + k))) for c in range(3)], -1)
            img = (img + rng.normal(0, 3, img.shape)).astype(np.int64) % 256
            p = os.path.join(d, f"{k:05d}.png")
            cv2.imwrite(p, img.astype(np.uint8))
            paths.append(p)
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            samples = []
            for _b in range(B):
                y0, x0 = random.randrange(352 - h + 1), random.randrange(640 - w + 1)
                fr = []
                for p in paths:
                    img = cv2.imread(p, cv2.IMREAD_UNCHANGED).astype(np.float32) / 255.
                    fr.append(np.fliplr(img[y0:y0 + h, x0:x0 + w, :]))
                x = np.stack(fr)[:, :, :, [2, 1, 0]]
                samples.append(torch.from_numpy(np.ascontiguousarray(np.transpose(x, (0, 3, 1, 2)))).float())
            torch.stack(samples)
            t = (time.perf_counter() - t0) * 1e3
            best = t if best is None else min(best, t)
    return round(best, 1)


def train_step_ms(ds, B, steps=10, rounds=2):
    from bin_b200 import rdn
    from bin_b200.loss import pixel_loss
    from bin_b200.optim import Adam
    from oracle import bin_oracle as O
    net = rdn.bin_stage4_lstm()
    net.load_state_dict(O.synth_state_dict(0), strict=True)
    net = net.cuda().train()
    opt = Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.99))
    rng = random.Random(1)
    fixed = ds.batch(list(range(B)), rng)

    def step(d):
        L, E, I = d["LQs"], d["GTenh"], d["GTinp"]
        gts = [I[:, 0], I[:, 1], I[:, 2], I[:, 3], E[:, 1], E[:, 2], E[:, 3], I[:, 1], I[:, 2], E[:, 2], I[:, 4],
               E[:, 4], I[:, 3], E[:, 3]]                          # bin_model.get_info, 6 frames (:529-535)
        opt.zero_grad(set_to_none=True)
        outs = net(*[L[:, i] for i in range(6)])
        loss, _ = pixel_loss(outs, gts, "l1")
        loss.backward()
        opt.step()

    def timed(fresh):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step(ds.batch([rng.randrange(len(ds)) for _ in range(B)], rng) if fresh else fixed)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for _ in range(3):
        step(fixed)
        step(ds.batch(list(range(B)), rng))
    torch.cuda.synchronize()
    res = {"fed_by_batch": [], "prebuilt": []}
    for _ in range(rounds):
        res["fed_by_batch"].append(round(timed(True), 2))
        res["prebuilt"].append(round(timed(False), 2))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--frames", type=int, default=480)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_batch: needs a CUDA device")
    g = torch.Generator(device="cuda").manual_seed(0)
    clips = {f"clip{k}": torch.randint(0, 256, (a.frames, 352, 640, 3), dtype=torch.uint8, device="cuda", generator=g)
             for k in range(2)}
    res = {"card": card(), "frames_per_clip": a.frames, "iters": a.iters, "configs": []}
    for B, h, w in ((8, 256, 256), (2, 128, 256)):
        t0 = time.perf_counter()
        ds = DeviceBINDataset.from_sharp_frames(clips, LQ_size=(3, h, w), shuffle_rng=random.Random(0))
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
        rng = random.Random(B * h)
        call_ms, host_us = time_calls(ds, B, a.iters, rng)
        k_us = kernel_us(ds, B, a.iters, rng)
        nbytes = B * 17 * h * w * 15
        res["configs"].append({"B": B, "h": h, "w": w, "store_windows": len(ds), "store_MB": round(ds.nbytes / 1e6, 1),
                               "from_sharp_frames_s": round(build_s, 3),
                               "call_ms": round(call_ms, 4), "host_us": round(host_us, 1),
                               "kernel_us": round(k_us, 2), "algorithmic_MB": round(nbytes / 1e6, 2),
                               "achieved_TBps": round(nbytes / (k_us * 1e-6) / 1e12, 3),
                               "hbm_frac": round(nbytes / (k_us * 1e-6) / (HBM_TBPS * 1e12), 3),
                               "ref_loader_ms": ref_loader_ms(B, h, w)})
        if B == 8:
            res["train_step_ms_B8_256"] = train_step_ms(ds, 8)
        del ds
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
