"""bin_b200.train_data on the GPU: batches bit-identical to what the reference's BINDataset delivered
(tests/golden/train_data.npz) and to the numpy oracle on other draws and sizes, the slot-major layout, both
constructors, argument errors, and a training forward + loss fed by a device batch."""
import os
import random

import numpy as np
import pytest
import torch

from oracle import train_data_oracle as TO

pytestmark = pytest.mark.gpu

FIX_SIZES = [(3, 16, 24), (3, 15, 23)]


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "train_data.npz"))


def clip_index(g, clip):
    return [str(c) for c in g["clips"]].index(clip)


def triples(g, order=None):
    """(windows, blurry, sharp) per clip of the fixture's dataset, in its listdir order (or `order`), frames rebuilt
    from the hash."""
    from bin_b200.train_data import windows_from_names
    out = []
    for clip in order or [str(c) for c in g["listdir"]]:
        wins = windows_from_names(clip, [str(n) for n in g[f"clip_{clip}_blur_names"]],
                                  [str(n) for n in g[f"clip_{clip}_list_names"]])
        read = TO.synthetic_reader(clip_index(g, clip))
        up = lambda n, b: torch.from_numpy(read(n, b).copy()).cuda()
        out.append((wins, {n: up(n, True) for w in wins for n in w.blur},
                    {n: up(n, False) for w in wins for n in w.enh + w.inp}))
    return out


def store(g, size, rng, order=None):
    from bin_b200.train_data import DeviceBINDataset
    return DeviceBINDataset(triples(g, order), LQ_size=size, shuffle_rng=rng)


def oracle_batch(g, ds, indices, size, rng):
    wins = [(w.key, list(w.blur), list(w.enh), list(w.inp)) for w in (ds.windows[i] for i in indices)]
    readers = [TO.synthetic_reader(clip_index(g, next(str(c) for c in g["clips"] if w[0].startswith(str(c) + "_"))))
               for w in wins]
    return TO.batch(wins, readers, size, rng)


def assert_same(dev, ref):
    assert dev["key"] == list(ref["key"])
    for k in ("LQs", "GTenh", "GTinp"):
        got = dev[k].cpu().numpy()
        assert got.dtype == np.float32 and got.shape == ref[k].shape, k
        assert np.array_equal(got, ref[k]), (k, np.argwhere(got != ref[k])[:5])


@pytest.mark.parametrize("size", FIX_SIZES, ids=lambda s: f"{s[1]}x{s[2]}")
def test_batch_is_bit_identical_to_the_reference(golden, size):
    tag = f"{size[1]}x{size[2]}"
    idx = [int(i) for i in golden[tag + "_indices"]]
    ref = {k: golden[f"{tag}_{k}"].astype(np.float32) / np.float32(255) for k in ("LQs", "GTenh", "GTinp")}
    ref["key"] = [str(k) for k in golden[tag + "_key"]]
    random.seed(int(golden["seed"]))
    ds = store(golden, size, random)
    assert ds.keys == [str(k) for k in golden["order_key"]]
    assert_same(ds.batch(idx), ref)                                    # one batch
    random.seed(int(golden["seed"]))
    ds = store(golden, size, random)
    parts = [ds.batch([i]) for i in idx]                               # B = 1 calls: independent of batch composition
    cat = {k: torch.cat([p[k] for p in parts]) for k in ("LQs", "GTenh", "GTinp")}
    cat["key"] = sum((p["key"] for p in parts), [])
    assert_same(cat, ref)


@pytest.mark.parametrize("size,B", [((3, 128, 256), 8), ((3, 256, 256), 3), ((3, 37, 61), 5), ((3, 1, 1), 2),
                                    ((3, 352, 640), 2), ((3, 64, 96), 64), ((3, 33, 50), 65)],
                         ids=["yml", "256sq", "odd", "1px", "full", "B64", "B65"])
def test_batch_matches_the_oracle(golden, size, B):
    seed = 1000 + B * size[1]
    ds = store(golden, size, random.Random(seed))
    pick = random.Random(seed + 1)
    idx = [pick.randrange(len(ds)) for _ in range(B)]
    dev = ds.batch(idx, rng=random.Random(seed + 2))
    assert_same(dev, oracle_batch(golden, ds, idx, size, random.Random(seed + 2)))


def test_slot_major_views_do_not_copy(golden):
    ds = store(golden, (3, 32, 48), None)
    out = ds.batch([0, 1, 2], rng=random.Random(3))
    assert out["LQs"].shape == (3, 6, 3, 32, 48) and out["GTenh"].shape == (3, 6, 3, 32, 48)
    assert out["GTinp"].shape == (3, 5, 3, 32, 48)
    for k, n in (("LQs", 6), ("GTenh", 6), ("GTinp", 5)):
        assert out[k].dtype == torch.float32 and out[k].device == ds.device
        for i in range(n):
            v = out[k][:, i, ...]                                      # feed_data's slicing (bin_model.py:156-178)
            assert v.is_contiguous() and v.contiguous().data_ptr() == v.data_ptr()


def test_store_is_unchanged_by_sampling(golden):
    ds = store(golden, (3, 352, 640), None)
    before = [t.clone() for t in ds._frames]
    for s in range(3):
        ds.batch(list(range(len(ds))), rng=random.Random(s))
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(before, ds._frames))


def test_from_sharp_frames_blurs_and_compacts():
    from bin_b200 import BinB200Error
    from bin_b200.dataprep import blur_average
    from bin_b200.train_data import DeviceBINDataset
    g = torch.Generator(device="cuda").manual_seed(11)
    frames = torch.randint(0, 256, (72, 352, 640, 3), dtype=torch.uint8, device="cuda", generator=g)
    ds = DeviceBINDataset.from_sharp_frames({"clipA": frames}, LQ_size=(3, 352, 640))
    blurry = blur_average(frames)
    assert blurry.shape[0] == 7                                         # floor(72 / 8) - 2 blurry frames -> 2 windows
    assert ds.keys == ["clipA_00017", "clipA_00025"]
    sharp = sorted({n for w in ds.windows for n in w.enh + w.inp})
    assert sharp == [17 + 4 * k for k in range(13)]
    assert ds.nbytes == (7 + 13) * 352 * 640 * 3
    fb, fs = blurry.cpu().numpy(), frames.cpu().numpy()
    read = lambda n, b: fb[(n - 17) // 8] if b else fs[n - 1]
    wins = [(w.key, list(w.blur), list(w.enh), list(w.inp)) for w in ds.windows]
    for s in range(4):                                                  # full frames, four different draws
        dev = ds.batch([0, 1], rng=random.Random(s))
        assert_same(dev, TO.batch(wins, [read, read], (3, 352, 640), random.Random(s)))
    for bad in (frames[:, :351], frames[:, :, :639], frames[..., :2], frames.float(), frames[0]):
        with pytest.raises(BinB200Error):
            DeviceBINDataset.from_sharp_frames({"c": bad})


def test_from_folders_equals_the_in_memory_store(golden, tmp_path):
    cv2 = pytest.importorskip("cv2")
    from bin_b200.train_data import DeviceBINDataset
    for clip in (str(c) for c in golden["clips"]):
        read = TO.synthetic_reader(clip_index(golden, clip))
        names = [str(n) for n in golden[f"clip_{clip}_blur_names"]]
        for d in ("train_blur", "train"):
            os.makedirs(tmp_path / d / clip)
        os.makedirs(tmp_path / "train_list", exist_ok=True)
        for name in names:
            n = int(name[:-4])
            cv2.imwrite(str(tmp_path / "train_blur" / clip / name), read(n, True))
            for m in (n, n + 4):
                cv2.imwrite(str(tmp_path / "train" / clip / f"{m:05d}.png"), read(m, False))
        (tmp_path / "train_list" / f"{clip}_im_list.txt").write_text(
            "\n".join(str(n) for n in golden[f"clip_{clip}_list_names"]))
    size = (3, 48, 80)
    a = DeviceBINDataset.from_folders(str(tmp_path), "train", LQ_size=size, shuffle_rng=random.Random(5))
    b = store(golden, size, random.Random(5), order=os.listdir(tmp_path / "train_blur"))
    assert a.keys == b.keys and a.nbytes == b.nbytes
    ra, rb = a.batch(range(len(a)), rng=random.Random(6)), b.batch(range(len(b)), rng=random.Random(6))
    assert ra["key"] == rb["key"]
    assert all(torch.equal(ra[k], rb[k]) for k in ("LQs", "GTenh", "GTinp"))


def test_c_entry_argument_errors_on_device(golden):
    from bin_b200 import _lib
    ds = store(golden, (3, 16, 16), None)
    out = torch.empty(6 * 16 * 16 * 3, device="cuda")
    t = (_lib.TrainSample * 1)()
    t[0].src[:] = ds._ptrs[0]
    t[0].y0, t[0].x0, t[0].flip = 0, 625, 0
    L = _lib.lib()
    p = out.data_ptr()
    assert L.bin_train_batch_u8(t, 1, ds.H, ds.W, 16, 16, p, p, p, None) == 1
    t[0].x0 = 624
    assert L.bin_train_batch_u8(t, 1, ds.H, ds.W, 16, 16, p, p, p, None) == 0          # the last valid column
    assert L.bin_train_batch_u8(t, 1, ds.H, ds.W, 17, 16, p, p, None, None) == 1
    from bin_b200 import BinB200Error
    with pytest.raises(BinB200Error):
        ds.batch([])
    with pytest.raises(BinB200Error):
        ds.batch([len(ds)])
    torch.cuda.synchronize()


def test_training_forward_and_loss_fed_by_a_device_batch(golden):
    """feed_data's slicing of a device batch through the network and the fused get_loss is bit-identical to the same
    batch built by the oracle on the host and uploaded (bin_model.py:147-202, get_info :529-535)."""
    from bin_b200 import rdn
    from bin_b200.loss import pixel_loss
    from oracle import bin_oracle as O
    size = (3, 64, 64)
    ds = store(golden, size, random.Random(8))
    idx = [0, 3]
    dev = ds.batch(idx, rng=random.Random(9))
    host = oracle_batch(golden, ds, idx, size, random.Random(9))
    net = rdn.bin_stage4_lstm()
    net.load_state_dict(O.synth_state_dict(0), strict=True)
    net = net.cuda().eval()

    def run(d):
        LQs, E, I = (torch.as_tensor(d[k]).cuda() for k in ("LQs", "GTenh", "GTinp"))
        B = [LQs[:, i, ...] for i in range(6)]
        I1, I3, I5, I7, I9, I11 = (E[:, i, ...] for i in range(6))
        I2, I4, I6, I8, I10 = (I[:, i, ...] for i in range(5))
        gts = [I2, I4, I6, I8, I3, I5, I7, I4, I6, I5, I10, I9, I8, I7]
        with torch.no_grad():
            outs = net(*B)
            loss, _ = pixel_loss(outs, gts, "l1")
        return outs, loss

    o1, l1 = run(dev)
    o2, l2 = run(host)
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(o1, o2))
    assert torch.equal(l1, l2) and torch.isfinite(l1)
