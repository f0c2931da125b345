"""numpy restatement of the reference's training-sample pipeline (data/BIN_dataset.py): window enumeration, the four
random draws per sample, crop / flip / reversal and the float32 conversion.  Independent of bin_b200; tests compare
it with tests/golden/train_data.npz (written by the unmodified reference, oracle/make_golden_train_data.py) and
bin_b200.train_data with it.

Synthetic frames are defined by `pixel(number, y, x, c)`, a closed-form integer hash of the file number and the
position, so a test can rebuild any frame of the fixture's dataset without storing it."""
from __future__ import annotations

import functools
from typing import Callable, Dict, List, Sequence, Tuple

import numpy as np

FRAME_H, FRAME_W = 352, 640        # BIN_dataset.py:132-133


def pixel(number, y, x, c) -> np.ndarray:
    """uint8 value of channel c (BGR, as stored in the PNG) at (y, x) of file `number`; broadcasts like numpy."""
    h = (np.asarray(number, np.uint32) * np.uint32(0x9E3779B1) + np.asarray(y, np.uint32) * np.uint32(0x85EBCA77) +
         np.asarray(x, np.uint32) * np.uint32(0xC2B2AE3D) + np.asarray(c, np.uint32) * np.uint32(0x27D4EB2F))
    h = h ^ (h >> np.uint32(15))
    h = h * np.uint32(0x2C1B3C6D)
    h = h ^ (h >> np.uint32(12))
    return (h >> np.uint32(24)).astype(np.uint8)


@functools.lru_cache(maxsize=256)
def frame(number: int, salt: int = 0, H: int = FRAME_H, W: int = FRAME_W) -> np.ndarray:
    """uint8 (H, W, 3) BGR frame of file `number` (read-only; cached).  `salt` separates frames that share a number."""
    y, x, c = np.meshgrid(np.arange(H), np.arange(W), np.arange(3), indexing="ij")
    f = pixel(number + (salt << 20), y, x, c)
    f.flags.writeable = False
    return f


def synthetic_reader(clip_index: int, H: int = FRAME_H, W: int = FRAME_W) -> Callable[[int, bool], np.ndarray]:
    """read(number, blurry) of clip `clip_index` of a synthetic dataset: blurry and sharp files of one number differ."""
    return lambda number, blurry: frame(number, 2 * clip_index + 1 + int(blurry), H, W)


def windows(clip: str, blur_names: Sequence[str], list_names: Sequence[str]) -> List[Tuple[str, List[int], List[int], List[int]]]:
    """_make_dataset_deep_long_ for one clip (BIN_dataset.py:212-281): [(key, blurry, sharp, interp file numbers)]."""
    pics = sorted(blur_names)                                   # :221
    num_win = int(len(pics) - 4 - 1)                            # :204, :224
    listed = sorted(list_names)                                 # :228-229
    first = int(pics[0][:-4]) if pics else 0                    # :231-232
    blurry, sharp, interp = [0, 8, 16, 24, 32, 40], [0, 8, 16, 24, 32, 40], [4, 12, 20, 28, 36]   # :234-236
    out = []
    for _ in range(num_win):                                    # :238
        b = [first + i for i in blurry]
        if all(str(n).zfill(5) + ".png" in listed for n in b):  # :272-277
            out.append((clip + "_" + str(b[0]).zfill(5), b, [first + i for i in sharp], [first + i for i in interp]))
        blurry, sharp, interp = [i + 8 for i in blurry], [i + 8 for i in sharp], [i + 8 for i in interp]   # :279-281
    return out


def sample(win, read: Callable[[int, bool], np.ndarray], size: Tuple[int, int, int], rng) -> Tuple[np.ndarray, ...]:
    """Adobe_BIN_loader (:63-183) + the conversion of __getitem__ (:37-49) for one window.  read(number, blurry) returns
    the uint8 (H, W, 3) BGR frame of a file.  Returns float32 LQs (6,3,h,w), GTenh (6,3,h,w), GTinp (5,3,h,w)."""
    _, b, s, i = win
    if not rng.randint(0, 1):                                   # :68, :89-109
        b, s, i = b[::-1], s[::-1], i[::-1]
    h, w = size[1], size[2]
    y0 = rng.choice(range(FRAME_H - h + 1))                     # :132
    x0 = rng.choice(range(FRAME_W - w + 1))                     # :133
    flip = rng.randint(0, 1)                                    # :156

    def one(n, blurry):
        img = read(n, blurry).astype(np.float32) / 255.         # data/util.py:89
        img = img[y0:y0 + h, x0:x0 + w, :]                      # :135-153
        if flip:
            img = np.fliplr(img)                                # :158-177
        return np.ascontiguousarray(img[:, :, [2, 1, 0]].transpose(2, 0, 1))   # :42-49

    return (np.stack([one(n, True) for n in b]), np.stack([one(n, False) for n in s]),
            np.stack([one(n, False) for n in i]))


def batch(wins, readers, size, rng) -> Dict[str, np.ndarray]:
    """DataLoader collation of `sample` over wins (readers[k] reads the clip of wins[k]):
    {'LQs': (B,6,3,h,w), 'GTenh': ..., 'GTinp': ..., 'key': [...]}."""
    out = [sample(w, r, size, rng) for w, r in zip(wins, readers)]
    return {"LQs": np.stack([o[0] for o in out]), "GTenh": np.stack([o[1] for o in out]),
            "GTinp": np.stack([o[2] for o in out]), "key": [w[0] for w in wins]}
