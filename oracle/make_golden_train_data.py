"""Generate tests/golden/train_data.npz by EXECUTING THE UNMODIFIED REFERENCE data/BIN_dataset.py (laomao0/BIN):

    python oracle/make_golden_train_data.py /path/to/BIN

Needs what BIN_dataset.py imports (cv2, torch, numpy).  Writes a temporary Adobe240-style tree of synthetic PNGs whose
pixels are oracle.train_data_oracle.frame (a closed-form hash, so tests rebuild them without storing them):

  GOPR0001_11_00  8 blurry files from 00017, every name listed            -> 3 windows
  IMG_0034        9 blurry files from 00025, 00089 missing from the list -> 3 of 4 windows

Clip k's file n is frame(n, 2k + 1) when sharp and frame(n, 2k + 2) when blurry (synthetic_reader).  Recorded:

  clips                    clip names in reader order (clip k reads with synthetic_reader(k))
  listdir                  os.listdir order of train_blur (the reference's clip order)
  clip_<name>_blur_names / _list_names   what the clip's folder and list file hold
  windows_key / _blur / _enh / _inp      _make_dataset_deep_long_ before its random.shuffle
  seed, order_key          the key order after random.seed(seed) + BINDataset(opt) (shuffled once)
  <h>x<w>_indices          the dataset indices sampled next, ds[i] in that order (DataLoader's sequential sampler)
  <h>x<w>_draws            per sample the loader's four draws (natural order, row, column, flip), recorded by wrapping
                           random.randint / random.choice
  <h>x<w>_LQs / _GTenh / _GTinp   ds[i] outputs as uint8 (every value is an exact u / 255)

The generator asserts that all four (reversed, flipped) combinations occur at each size.
"""
import os
import random
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
if len(sys.argv) != 2 or not os.path.isfile(os.path.join(sys.argv[1], "data", "BIN_dataset.py")):
    raise SystemExit(__doc__)
sys.path.insert(0, os.path.abspath(sys.argv[1]))

import cv2                                                   # noqa: E402
from data.BIN_dataset import BINDataset                     # noqa: E402  (the reference itself)
from oracle.train_data_oracle import synthetic_reader       # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "train_data.npz")
CLIPS = [("GOPR0001_11_00", 17, 8, None), ("IMG_0034", 25, 9, 25 + 8 * 8)]     # name, first, n_blur, unlisted
SEED = 2026
SIZES = [(3, 16, 24), (3, 15, 23)]
INDICES = [0, 1, 2, 3, 4, 5, 0, 1]


def write_tree(root):
    for k, (clip, first, nb, unlisted) in enumerate(CLIPS):
        read = synthetic_reader(k)
        for d in ("train_blur", "train", "train_list"):
            os.makedirs(os.path.join(root, d, clip) if d != "train_list" else os.path.join(root, d), exist_ok=True)
        names = []
        for j in range(nb):
            n = first + 8 * j
            cv2.imwrite(os.path.join(root, "train_blur", clip, f"{n:05d}.png"), read(n, True))
            if n != unlisted:
                names.append(f"{n:05d}.png")
        for j in range(2 * nb - 1):
            n = first + 4 * j
            cv2.imwrite(os.path.join(root, "train", clip, f"{n:05d}.png"), read(n, False))
        with open(os.path.join(root, "train_list", clip + "_im_list.txt"), "w") as fh:
            fh.write("\n".join(names))                       # create_dataset_blur_N_frames_average.py:145-148


def as_u8(x):
    x = np.asarray(x, np.float32)
    u = np.rint(x * 255).astype(np.uint8)
    assert np.array_equal(u.astype(np.float32) / np.float32(255), x), "a value is not an exact u / 255"
    return u


def nums(paths):
    return [int(os.path.basename(p)[:-4]) for p in paths]


def main():
    out = {"seed": np.array(SEED), "clips": np.array([c[0] for c in CLIPS])}
    with tempfile.TemporaryDirectory() as root:
        write_tree(root)
        out["listdir"] = np.array(os.listdir(os.path.join(root, "train_blur")))
        for clip, *_ in CLIPS:
            out[f"clip_{clip}_blur_names"] = np.array(os.listdir(os.path.join(root, "train_blur", clip)))
            with open(os.path.join(root, "train_list", clip + "_im_list.txt")) as fh:
                out[f"clip_{clip}_list_names"] = np.array(fh.read().split("\n"))

        shuffle = random.shuffle
        random.shuffle = lambda x: None                      # the window list before its one shuffle (:283)
        try:
            wins, _ = BINDataset._make_dataset_deep_long_(dir=root, sharp_index=(2, 3), mode="train")
        finally:
            random.shuffle = shuffle
        out["windows_key"] = np.array([w[3] for w in wins])
        for i, name in enumerate(("blur", "enh", "inp")):
            out["windows_" + name] = np.array([nums(w[i]) for w in wins])

        draws = []
        randint, choice = random.randint, random.choice

        def rec_randint(a, b):
            v = randint(a, b)
            draws.append(v)
            return v

        def rec_choice(seq):
            v = choice(seq)
            draws.append(v)
            return v

        for size in SIZES:
            tag = f"{size[1]}x{size[2]}"
            random.seed(SEED)
            ds = BINDataset({"dataroot_GT": root, "dataroot_LQ": root, "data_type": "img", "LQ_size": size,
                             "name": "train"})
            if size == SIZES[0]:
                out["order_key"] = np.array([w[3] for w in ds.all_paths])
            assert [w[3] for w in ds.all_paths] == list(out["order_key"])
            samples = []
            draws.clear()
            random.randint, random.choice = rec_randint, rec_choice
            try:
                for i in INDICES:
                    samples.append(ds[i])
            finally:
                random.randint, random.choice = randint, choice
            d = np.array(draws).reshape(len(INDICES), 4)
            combos = {(int(a), int(f)) for a, _, _, f in d}
            assert combos == {(0, 0), (0, 1), (1, 0), (1, 1)}, f"seed {SEED} misses a (natural, flip) combination: {combos}"
            out[tag + "_indices"] = np.array(INDICES)
            out[tag + "_draws"] = d
            for k in ("LQs", "GTenh", "GTinp"):
                out[f"{tag}_{k}"] = as_u8(np.stack([s[k].numpy() for s in samples]))
            out[tag + "_key"] = np.array([s["key"] for s in samples])
    np.savez_compressed(OUT, **out)
    print(OUT, os.path.getsize(OUT), "bytes;", len(out["windows_key"]), "windows, order", list(out["order_key"]))


if __name__ == "__main__":
    main()
