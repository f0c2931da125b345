"""Training batches assembled on the GPU (DESIGN 5c rank 6): BINDataset + DataLoader of data/BIN_dataset.py.

The reference decodes 17 PNGs per sample on the host, converts each whole frame to float32 and only then crops, flips
and reverses (Adobe_BIN_loader, BIN_dataset.py:63-183).  `DeviceBINDataset` keeps the clips in HBM as uint8 instead,
and `batch()` builds the `{'LQs', 'GTenh', 'GTinp', 'key'}` batch that BINDataset + DataLoader would deliver in one
sm_100a launch (csrc/train_data.cu), bit-identical to the reference for the same Python `random` state.

Windows (BIN_dataset.py:186-288): in a clip whose blurry files are numbered from `first`, window w takes blurry files
first + 8(w+s) for s = 0..5 (LQs), the sharp files of the same numbers (GTenh) and sharp files first + 8(w+s) + 4 for
s = 0..4 (GTinp).  A store therefore keeps the blurry frames and only the sharp frames first + 4k.

CUDA only; there is no CPU path.  Samplers are not re-implemented: the reference's own sampler supplies `indices`.
"""
from __future__ import annotations

import os
import random as _random
from typing import Dict, Iterable, List, Mapping, NamedTuple, Sequence, Tuple

import torch

from ._lib import BinB200Error, TrainSample, check, lib

FRAME_H, FRAME_W = 352, 640        # BIN_dataset.py:132-133: the crop range is hard-coded, whatever the frame size
NUM_LQ, NUM_ENH, NUM_INP = 6, 6, 5
NUM_WIN_PER_BUNCH = 4              # BIN_dataset.py:204, num_win = n_blur - 4 - 1 (:224)
BLUR_FIRST, BLUR_STRIDE = 17, 8    # create_dataset_blur_N_frames_average.py:99-128: blurry w is file 17 + 8w


class Window(NamedTuple):
    """One training window: its key and the file numbers of its 6 blurry, 6 sharp and 5 interpolation frames."""
    key: str
    blur: Tuple[int, ...]
    enh: Tuple[int, ...]
    inp: Tuple[int, ...]


def windows_from_names(clip: str, blur_names: Iterable[str], list_names: Iterable[str]) -> List[Window]:
    """The windows _make_dataset_deep_long_ makes for one clip (BIN_dataset.py:212-281), in its order.

    blur_names: the file names in `{mode}_blur/{clip}/`; list_names: the lines of `{mode}_list/{clip}_im_list.txt`.
    Windows with a blurry name missing from the list are dropped (:272-277)."""
    blur_pics = sorted(blur_names)
    if not blur_pics:
        return []
    first = int(blur_pics[0][:-4])                                          # :231-232
    listed = set(list_names)
    out = []
    for w in range(len(blur_pics) - NUM_WIN_PER_BUNCH - 1):                # :224, :238
        base = first + 8 * w
        blur = tuple(base + 8 * s for s in range(NUM_LQ))                    # :242-250
        if all(f"{n:05d}.png" in listed for n in blur):
            inp = tuple(base + 8 * s + 4 for s in range(NUM_INP))            # :262-268
            out.append(Window(f"{clip}_{base:05d}", blur, blur, inp))       # sharp = blurry numbers (:253-259), key :270
    return out


def _check_lq_size(LQ_size) -> Tuple[int, int]:
    if len(LQ_size) != 3 or int(LQ_size[0]) != 3:
        raise BinB200Error(f"LQ_size must be (3, h, w), got {tuple(LQ_size)}")
    h, w = int(LQ_size[1]), int(LQ_size[2])
    if not (1 <= h <= FRAME_H and 1 <= w <= FRAME_W):
        raise BinB200Error(f"LQ_size {tuple(LQ_size)}: the crop must lie in the reference's 1..{FRAME_H} x 1..{FRAME_W} range")
    return h, w


def _check_frame(t, what: str) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise BinB200Error(f"{what}: frames must be CUDA tensors (bin_b200 has no CPU path)")
    if t.dtype != torch.uint8:
        raise BinB200Error(f"{what}: frames must be uint8, got {t.dtype}")
    if t.dim() < 3 or t.shape[-1] != 3:
        raise BinB200Error(f"{what}: frames must be (H, W, 3) BGR, got shape {tuple(t.shape)}")
    if t.shape[-3] < FRAME_H or t.shape[-2] < FRAME_W:
        raise BinB200Error(f"{what}: frames of {t.shape[-3]}x{t.shape[-2]} are smaller than the reference's "
                           f"{FRAME_H}x{FRAME_W} crop range")


class DeviceBINDataset:
    """HBM-resident training windows.  `clips`: one (windows, blurry, sharp) triple per clip, where `blurry` and `sharp`
    map file numbers to uint8 CUDA (H, W, 3) BGR frames and hold every number the windows reference.  The referenced frames
    of a clip are stacked into one tensor; all clips share one frame size and device.  `shuffle_rng`, when given, shuffles
    the window list once with `shuffle_rng.shuffle`, as _make_dataset_deep_long_ does (:283)."""

    def __init__(self, clips: Iterable[Tuple[Sequence[Window], Mapping[int, torch.Tensor], Mapping[int, torch.Tensor]]],
                 LQ_size=(3, 128, 256), shuffle_rng=None):
        self.h, self.w = _check_lq_size(LQ_size)
        self.LQ_size = (3, self.h, self.w)
        self._frames: List[torch.Tensor] = []
        entries: List[Tuple[Window, Tuple[int, ...]]] = []
        shape = device = None
        for windows, blurry, sharp in clips:
            rows: Dict[Tuple[str, int], int] = {}
            stack = []
            for kind, frames in (("blurry", blurry), ("sharp", sharp)):
                for n in sorted({n for win in windows for n in (win.blur if kind == "blurry" else win.enh + win.inp)}):
                    if n not in frames:
                        raise BinB200Error(f"{kind} frame {n} of a window is missing")
                    t = frames[n]
                    _check_frame(t, kind)
                    if t.dim() != 3:
                        raise BinB200Error(f"{kind} frame {n}: expected (H, W, 3), got {tuple(t.shape)}")
                    if shape is None:
                        shape, device = tuple(t.shape), t.device
                    if tuple(t.shape) != shape or t.device != device:
                        raise BinB200Error("all frames of a store must have one size and one device")
                    rows[(kind, n)] = len(stack)
                    stack.append(t)
            if not stack:
                continue
            store = torch.stack(stack)                         # one uint8 (n, H, W, 3) tensor per clip
            self._frames.append(store)
            step = store[0].numel()
            p0 = store.data_ptr()
            for win in windows:
                ptrs = ([p0 + step * rows[("blurry", n)] for n in win.blur] +
                        [p0 + step * rows[("sharp", n)] for n in win.enh + win.inp])
                entries.append((win, tuple(ptrs)))
        if not entries:
            raise BinB200Error("DeviceBINDataset: no window")
        if shuffle_rng is not None:
            shuffle_rng.shuffle(entries)
        self.windows: List[Window] = [e[0] for e in entries]
        self._ptrs: List[Tuple[int, ...]] = [e[1] for e in entries]
        self.H, self.W = shape[0], shape[1]
        self.device = device

    def __len__(self) -> int:
        return len(self.windows)

    @property
    def keys(self) -> List[str]:
        return [w.key for w in self.windows]

    @property
    def nbytes(self) -> int:
        """HBM held by the frames of the store."""
        return sum(t.numel() for t in self._frames)

    def batch(self, indices: Sequence[int], rng=_random) -> dict:
        """The collated batch of windows `indices`: per sample the four draws of Adobe_BIN_loader, in its order, from
        `rng` (the global `random` by default): randint(0, 1) natural order or reversed (:68), the row and column
        offsets choice(range(352 - h + 1)) and choice(range(640 - w + 1)) (:132-133), randint(0, 1) np.fliplr (:156).
        Returns {'LQs': (B,6,3,h,w), 'GTenh': (B,6,3,h,w), 'GTinp': (B,5,3,h,w), 'key': [...]}: fp32 views of
        slot-major storage on the store's device, so each `LQs[:, i]` is contiguous.  Runs on the device's current
        stream without synchronising."""
        indices = [int(i) for i in indices]
        B = len(indices)
        if B < 1:
            raise BinB200Error("batch: no index")
        n = len(self.windows)
        if any(i < -n or i >= n for i in indices):
            raise BinB200Error(f"batch: index out of range for {n} windows")
        h, w = self.h, self.w
        table = (TrainSample * B)()
        for b, i in enumerate(indices):
            p = self._ptrs[i]
            natural = rng.randint(0, 1)
            y0 = rng.choice(range(FRAME_H - h + 1))
            x0 = rng.choice(range(FRAME_W - w + 1))
            flip = rng.randint(0, 1)
            if not natural:                                  # :89-109 all three lists reversed
                p = p[NUM_LQ - 1::-1] + p[NUM_LQ + NUM_ENH - 1:NUM_LQ - 1:-1] + p[:NUM_LQ + NUM_ENH - 1:-1]
            table[b].src[:] = p
            table[b].y0, table[b].x0, table[b].flip = y0, x0, flip
        dev = self.device
        lqs = torch.empty((NUM_LQ, B, 3, h, w), dtype=torch.float32, device=dev)
        enh = torch.empty((NUM_ENH, B, 3, h, w), dtype=torch.float32, device=dev)
        inp = torch.empty((NUM_INP, B, 3, h, w), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().bin_train_batch_u8(table, B, self.H, self.W, h, w, lqs.data_ptr(), enh.data_ptr(), inp.data_ptr(),
                                           torch.cuda.current_stream().cuda_stream))
        return {"LQs": lqs.transpose(0, 1), "GTenh": enh.transpose(0, 1), "GTinp": inp.transpose(0, 1),
                "key": [self.windows[i].key for i in indices]}

    # ------------------------------------------------------------------------------------------------ constructors
    @classmethod
    def from_sharp_frames(cls, clips: Mapping[str, torch.Tensor], window_size: int = 11, LQ_size=(3, 128, 256),
                          shuffle_rng=None) -> "DeviceBINDataset":
        """Train straight from 240-fps frames: {clip: uint8 CUDA (T, H, W, 3) BGR}.  The blurry frames are synthesised
        with dataprep.blur_average (blurry w = file 17 + 8w, the blur script's naming); of the sharp frames only those
        a window references (files 17 + 4k; file n is frame n - 1) are kept."""
        from .dataprep import blur_average

        def each_clip():
            for clip, frames in clips.items():
                yield clip_triple(clip, frames)

        def clip_triple(clip, frames):
            _check_frame(frames, f"from_sharp_frames[{clip!r}]")
            if frames.dim() != 4:
                raise BinB200Error(f"from_sharp_frames[{clip!r}]: expected (T, H, W, 3), got {tuple(frames.shape)}")
            blurry = blur_average(frames, window_size)
            names = [f"{BLUR_FIRST + BLUR_STRIDE * k:05d}.png" for k in range(blurry.shape[0])]
            windows = windows_from_names(clip, names, names)
            blur_map = {BLUR_FIRST + BLUR_STRIDE * k: blurry[k] for k in range(blurry.shape[0])}
            sharp_map = {n: frames[n - 1] for win in windows for n in win.enh + win.inp}
            return windows, blur_map, sharp_map

        return cls(each_clip(), LQ_size, shuffle_rng)

    @classmethod
    def from_folders(cls, root: str, mode: str = "train", LQ_size=(3, 128, 256), shuffle_rng=None,
                     device=None) -> "DeviceBINDataset":
        """The dataset tree the reference reads (BIN_dataset.py:206-231): `{root}/{mode}_blur/{clip}/*.png`,
        `{root}/{mode}/{clip}/*.png` and `{root}/{mode}_list/{clip}_im_list.txt`, clips in os.listdir order.  Each PNG a
        window needs is decoded once (cv2.IMREAD_UNCHANGED, first 3 channels, as read_img does, data/util.py:73-95),
        uploaded, and the host copy dropped clip by clip."""
        import cv2
        import numpy as np
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        _check_lq_size(LQ_size)
        blur_dir, sharp_dir, list_dir = (os.path.join(root, d) for d in (mode + "_blur", mode, mode + "_list"))

        def load(path: str) -> torch.Tensor:
            img = cv2.imread(path, cv2.IMREAD_UNCHANGED)
            if img is None:
                raise BinB200Error(f"from_folders: cannot read {path}")
            if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] < 3:
                raise BinB200Error(f"from_folders: {path} is not an 8-bit image with 3 or 4 channels")
            return torch.from_numpy(np.ascontiguousarray(img[:, :, :3])).to(dev)

        def each_clip():                       # one clip's frames at a time: the store stacks them before the next is read
            for clip in os.listdir(blur_dir):
                yield clip_triple(clip)

        def clip_triple(clip):
            with open(os.path.join(list_dir, clip + "_im_list.txt")) as fh:
                listed = fh.read().split("\n")
            windows = windows_from_names(clip, os.listdir(os.path.join(blur_dir, clip)), listed)
            blur_map = {n: load(os.path.join(blur_dir, clip, f"{n:05d}.png")) for n in sorted({n for w in windows for n in w.blur})}
            sharp_map = {n: load(os.path.join(sharp_dir, clip, f"{n:05d}.png"))
                         for n in sorted({n for w in windows for n in w.enh + w.inp})}
            return windows, blur_map, sharp_map

        return cls(each_clip(), LQ_size, shuffle_rng)
