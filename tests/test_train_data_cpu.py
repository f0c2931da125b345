"""CPU checks of the training-batch layer: window enumeration and the shuffled order against what the reference's own
BINDataset produced (tests/golden/train_data.npz), the numpy oracle against every recorded sample, the argument checks
of bin_b200.train_data and of the C entry (which must reject before any device work), and the ctypes mirror of
bin_train_sample_t."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest
import torch

from oracle import train_data_oracle as TO

SIZES = [(3, 16, 24), (3, 15, 23)]


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "train_data.npz"))


def clip_windows(g, fn):
    """fn(clip, blur_names, list_names) over the clips in the reference's listdir order."""
    out = []
    for clip in g["listdir"]:
        clip = str(clip)
        out += fn(clip, [str(n) for n in g[f"clip_{clip}_blur_names"]], [str(n) for n in g[f"clip_{clip}_list_names"]])
    return out


def reader_of(g, key):
    clips = [str(c) for c in g["clips"]]
    return TO.synthetic_reader(next(k for k, c in enumerate(clips) if key.startswith(c + "_")))


def test_windows_match_the_reference(golden):
    from bin_b200.train_data import windows_from_names
    wins = clip_windows(golden, windows_from_names)
    assert [w.key for w in wins] == [str(k) for k in golden["windows_key"]]
    assert [list(w.blur) for w in wins] == golden["windows_blur"].tolist()
    assert [list(w.enh) for w in wins] == golden["windows_enh"].tolist()
    assert [list(w.inp) for w in wins] == golden["windows_inp"].tolist()
    ow = clip_windows(golden, TO.windows)
    assert [(w.key, list(w.blur), list(w.enh), list(w.inp)) for w in wins] == ow
    # the list file drops exactly the window that needs the unlisted blurry file
    assert len(wins) == 6 and "IMG_0034_00049" not in [w.key for w in wins]


def test_shuffled_order_matches_the_reference(golden):
    from bin_b200.train_data import windows_from_names
    wins = clip_windows(golden, windows_from_names)
    random.seed(int(golden["seed"]))
    random.shuffle(wins)
    assert [w.key for w in wins] == [str(k) for k in golden["order_key"]]


@pytest.mark.parametrize("size", SIZES, ids=lambda s: f"{s[1]}x{s[2]}")
def test_oracle_reproduces_every_reference_sample(golden, size):
    tag = f"{size[1]}x{size[2]}"
    wins = clip_windows(golden, TO.windows)
    random.seed(int(golden["seed"]))
    random.shuffle(wins)
    picked = [wins[int(i)] for i in golden[tag + "_indices"]]
    out = TO.batch(picked, [reader_of(golden, w[0]) for w in picked], size, random)
    assert out["key"] == [str(k) for k in golden[tag + "_key"]]
    for k in ("LQs", "GTenh", "GTinp"):
        ref = golden[f"{tag}_{k}"].astype(np.float32) / np.float32(255)
        assert out[k].dtype == np.float32 and out[k].shape == ref.shape
        assert np.array_equal(out[k], ref), k


def test_fixture_covers_every_reversal_and_flip(golden):
    for size in SIZES:
        d = golden[f"{size[1]}x{size[2]}_draws"]
        assert {(int(a), int(f)) for a, _, _, f in d} == {(0, 0), (0, 1), (1, 0), (1, 1)}


def test_rejections_before_any_device_work():
    from bin_b200 import BinB200Error
    from bin_b200.train_data import DeviceBINDataset, windows_from_names
    names = [f"{17 + 8 * k:05d}.png" for k in range(7)]
    wins = windows_from_names("c", names, names)
    assert len(wins) == 2
    cpu = torch.zeros((352, 640, 3), dtype=torch.uint8)
    blur = {n: cpu for w in wins for n in w.blur}
    sharp = {n: cpu for w in wins for n in w.enh + w.inp}
    with pytest.raises(BinB200Error, match="CUDA"):
        DeviceBINDataset([(wins, blur, sharp)])
    with pytest.raises(BinB200Error, match="CUDA"):
        DeviceBINDataset.from_sharp_frames({"c": torch.zeros((80, 352, 640, 3), dtype=torch.uint8)})
    for bad in [(3, 0, 256), (3, 128, 0), (3, 353, 256), (3, 128, 641), (1, 128, 256), (3, 128)]:
        with pytest.raises(BinB200Error, match="LQ_size"):
            DeviceBINDataset([(wins, blur, sharp)], LQ_size=bad)
    with pytest.raises(BinB200Error, match="missing"):
        DeviceBINDataset([(wins, {}, sharp)])
    with pytest.raises(BinB200Error, match="no window"):
        DeviceBINDataset([([], {}, {})])
    assert windows_from_names("c", [], []) == []
    assert windows_from_names("c", names[:5], names[:5]) == []          # fewer than 6 blurry frames: no window


def _sample_table(B, ptr=1 << 20, y0=0, x0=0, flip=0):
    from bin_b200 import _lib
    t = (_lib.TrainSample * B)()
    for b in range(B):
        t[b].src[:] = [ptr] * _lib.BIN_TRAIN_FRAMES
        t[b].y0, t[b].x0, t[b].flip = y0, x0, flip
    return t


def test_c_entry_rejects_bad_arguments():
    """Every one of these returns BIN_ERR_ARG from the argument checks, before a launch."""
    from bin_b200 import _lib
    L = _lib.lib()
    out = C.c_void_p(1 << 21)
    ok = _sample_table(2)
    bad_null = _sample_table(2)
    bad_null[1].src[16] = None
    calls = [
        (None, 2, 352, 640, 16, 16, out, out, out),
        (ok, 2, 352, 640, 16, 16, None, out, out),
        (ok, 0, 352, 640, 16, 16, out, out, out),
        (ok, 2, 352, 640, 0, 16, out, out, out),
        (ok, 2, 352, 640, 16, 641, out, out, out),
        (ok, 2, 0, 640, 16, 16, out, out, out),
        (bad_null, 2, 352, 640, 16, 16, out, out, out),
        (_sample_table(2, y0=337), 2, 352, 640, 16, 16, out, out, out),
        (_sample_table(2, x0=-1), 2, 352, 640, 16, 16, out, out, out),
        (_sample_table(2, x0=625), 2, 352, 640, 16, 16, out, out, out),
        (_sample_table(2, flip=2), 2, 352, 640, 16, 16, out, out, out),
    ]
    for i, args in enumerate(calls):
        assert L.bin_train_batch_u8(*args, None) == 1, i
        assert L.bin_last_error().decode().startswith("train_batch"), i


def test_train_sample_struct_matches_the_header(tmp_path):
    from bin_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "probe.c"
    src.write_text("\n".join([
        '#include <stdio.h>', '#include <stddef.h>', '#include "bin_b200.h"', 'int main(void) {',
        '  printf("%zu %zu %zu %zu %zu %d %d\\n", sizeof(bin_train_sample_t), offsetof(bin_train_sample_t, src),',
        '         offsetof(bin_train_sample_t, y0), offsetof(bin_train_sample_t, x0), offsetof(bin_train_sample_t, flip),',
        '         BIN_TRAIN_FRAMES, BIN_MAX_TRAIN_SAMPLES);', '  return 0;', '}']))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    T = _lib.TrainSample
    assert got == [C.sizeof(T), T.src.offset, T.y0.offset, T.x0.offset, T.flip.offset, _lib.BIN_TRAIN_FRAMES,
                   _lib.BIN_MAX_TRAIN_SAMPLES]
