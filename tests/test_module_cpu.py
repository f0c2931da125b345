"""CPU-side checks of the drop-in boundary (SURVEY 8b): schema, strict load, loud failure
without CUDA, and that the C-ABI library exports every symbol the header declares."""
import os
import re

import pytest
import torch

from oracle import bin_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def net():
    from bin_b200 import rdn
    torch.manual_seed(0)
    return rdn.bin_stage4_lstm()


def test_state_dict_schema_matches_reference(net):
    sd_ref = O.synth_state_dict(0)            # key order + shapes were asserted against the reference in make_golden.py
    sd = net.state_dict()
    assert list(sd.keys()) == list(sd_ref.keys())
    for k in sd:
        assert tuple(sd[k].shape) == tuple(sd_ref[k].shape), k
    assert len(sd) == 1332
    uniq = list(net.parameters())
    assert len(uniq) == 540 and sum(p.numel() for p in uniq) == 11_441_668


def test_strict_load_and_aliasing(net):
    sd_ref = O.synth_state_dict(3)
    res = net.load_state_dict(sd_ref, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    m = net.model
    assert m.model1_2 is m.model1_1 and m.model1_4 is m.model1_1 and m.model2_3 is m.model2_1 and m.model3_2 is m.model3_1
    assert torch.equal(m.model1_3.SFENet1.weight, sd_ref["model.model1_1.SFENet1.weight"])


def test_prefix_stripping_like_base_model(net):
    """base_model.load_network strips 'module.' / 'InterpNet.' prefixes then loads strictly (base_model.py:89-103)."""
    sd_ref = O.synth_state_dict(1)
    wrapped = {"module." + k: v for k, v in sd_ref.items()}
    clean = {k[7:] if k.startswith("module.") else k: v for k, v in wrapped.items()}
    net.load_state_dict(clean, strict=True)


def test_cpu_forward_fails_loudly(net):
    from bin_b200 import BinB200Error
    fr = O.synth_frames(6, 1, 16, 16)
    with torch.no_grad(), pytest.raises(BinB200Error):
        net(*fr)


def test_grad_path_on_cpu_fails_loudly(net):
    """Training goes through the same CUDA library: a grad-enabled CPU call must raise, not fall back."""
    from bin_b200 import BinB200Error
    fr = O.synth_frames(6, 1, 16, 16)
    with pytest.raises(BinB200Error):
        net(*fr)


def test_library_exports_every_declared_symbol():
    import ctypes
    from bin_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "bin_b200.h")).read()
    declared = set(re.findall(r"\b(bin_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"bin_b200"}
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/bin_b200.h but not exported"
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    assert _lib.lib().bin_abi_version() == _lib.ABI_VERSION == int(re.search(r"#define BIN_ABI_VERSION (\d+)", hdr).group(1))
    # measurement tooling lives in libbin_b200_tools.so / csrc/tools_abi.h, never in the product library or its header
    assert not any(n.startswith(("bin_tools_", "bin_microbench", "bin_debug")) for n in declared)
    assert not hasattr(L, "bin_tools_microbench_mma") and not hasattr(L, "bin_microbench_mma")


def test_workspace_queries_are_pure():
    from bin_b200 import _lib
    L = _lib.lib()
    assert L.bin_backbone_packed_bytes(2) > 5_000_000 and L.bin_backbone_packed_bytes(4) == 0
    a = L.bin_window_workspace_bytes(1, 64, 64)
    assert 0 < a < L.bin_window_workspace_bytes(1, 128, 128)


def test_training_side_modules_refuse_cpu_tensors():
    """bin_b200.optim / bin_b200.dataprep have no CPU path: they must say so instead of computing something."""
    import torch
    from bin_b200 import BinB200Error
    from bin_b200.dataprep import blur_average, window_count
    from bin_b200.optim import Adam
    p = torch.nn.Parameter(torch.ones(4))
    p.grad = torch.ones(4)
    opt = Adam([p], lr=1e-3, betas=(0.9, 0.99), weight_decay=1e-4)
    assert opt.param_groups[0]["betas"] == (0.9, 0.99) and opt.param_groups[0]["weight_decay"] == 1e-4
    with pytest.raises(BinB200Error):
        opt.step()
    assert torch.all(p == 1)
    with pytest.raises(ValueError):
        Adam([p], lr=-1.0)
    with pytest.raises(BinB200Error):
        blur_average(torch.zeros((40, 4, 4, 3), dtype=torch.uint8))
    # create_dataset_blur_N_frames_average.py:104  window_total_num = floor(n_length / 8) - 2
    assert [window_count(n) for n in (24, 40, 47, 48, 240)] == [1, 3, 3, 4, 28]


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """sizeof / offsetof of every ABI struct as gcc sees include/bin_b200.h == the ctypes mirror in bin_b200/_lib.py
    (and the 5 x int64 rows bin_b200.optim uploads == bin_adam_tensor_t)."""
    import ctypes as C
    import subprocess
    from bin_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    probes = {"bin_act_t": (_lib.Act, ["ptr", "B", "planes", "H", "W"]),
              "bin_frames_t": (_lib.Frames, ["frame", "out", "ncalls", "nframes", "Bc"]),
              "bin_conv_args_t": (_lib.ConvArgs, [f[0] for f in _lib.ConvArgs._fields_]),
              "bin_net_t": (_lib.Net, ["blob", "lstm_w", "lstm_b"])}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "bin_b200.h"', 'int main(void) {']
    for cname, (_, fields) in probes.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for f in fields:
            lines.append(f'  printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));')
    lines += ['  printf("bin_adam_tensor_t %zu\\n", sizeof(bin_adam_tensor_t));',
              '  printf("bin_adam_tensor_t.n %zu\\n", offsetof(bin_adam_tensor_t, n));', '  return 0;', '}']
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, (ct, fields) in probes.items():
        assert int(got[cname]) == C.sizeof(ct), cname
        for f in fields:
            assert int(got[f"{cname}.{f}"]) == getattr(ct, f).offset, f"{cname}.{f}"
    assert int(got["bin_adam_tensor_t"]) == 5 * 8 and int(got["bin_adam_tensor_t.n"]) == 4 * 8


def test_weight_walk_matches_parameters_and_survives_replication(net):
    """nn.DataParallel replicas (bin_model.py:42) have EMPTY _parameters and carry their weights as plain attributes
    (torch/nn/parallel/replicate.py): the tensors handed to the C ABI must therefore be read from the conv modules, in
    the registration order bin_backbone_pack expects."""
    import torch
    for bb in (net.model.model1_1, net.model.model2_1, net.model.model3_1, net.model.model4_1):
        walked, regs = bb._conv_params(), list(bb.parameters())
        assert len(walked) == 132 and all(a is b for a, b in zip(walked, regs))
    allt = net._all_tensors()
    assert len(allt) == 540 and {id(t) for t in allt} == {id(p) for p in net.parameters()}
    # what replicate() does to one module tree, on CPU: copy every module, drop _parameters, set plain tensor attributes
    mods = list(net.modules())
    copies = {id(m): m._replicate_for_data_parallel() for m in mods}
    for m in mods:
        r = copies[id(m)]
        for key, child in m._modules.items():
            setattr(r, key, copies[id(child)])
        for key, p in m._parameters.items():
            setattr(r, key, p.detach() * 2.0)
    rep = copies[id(net)]
    assert len(list(rep.parameters())) == 0                       # the reason self.parameters() cannot be used
    rw = rep._all_tensors()
    assert len(rw) == 540 and all(torch.equal(a, b * 2.0) for a, b in zip(rw, allt))
    assert rep.model.model1_3 is rep.model.model1_1               # aliases stay aliases inside a replica


def test_bench_reference_arm_line_on_cpu():
    """`bench.py --impl reference` (the driver's reference arm) on a tiny window: one JSON line with the contract's keys,
    kind "reference" where the unmodified reference is mounted and "port" otherwise; a non-zero rank prints nothing."""
    import json
    import subprocess
    import sys
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--height", "48", "--width", "64",
           "--steps", "3", "--warmup", "1", "--gpus", "2"]
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().split("\n") if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "720p frame-windows/sec" and j["unit"] == "windows/s"
    assert j["higher_is_better"] is True and j["value"] > 0 and j["n_gpus"] == 2
    assert j["steps"] == 2 and j["requested_steps"] == 3            # bounded sample: at most two timed windows
    cb = j["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == j["value"] and cb["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    r1 = subprocess.run(cmd, env=dict(env, RANK="1", LOCAL_RANK="1"), capture_output=True, text=True, timeout=600)
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_bench_dump_outputs(tmp_path):
    """`bench.py --dump-outputs DIR` writes the 14 outputs of the last timed window as float32 .npy, computed from the
    fixed seeded inputs (checked against the oracle on those inputs); a step larger than the byte budget is written as
    the same seeded sample of every output, under the budget, identically from run to run."""
    import json
    import subprocess
    import sys
    import importlib.util
    import numpy as np
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--height", "48", "--width", "64",
           "--steps", "1", "--warmup", "0", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, env=dict(os.environ, RANK="0"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads([l for l in r.stdout.strip().split("\n") if l.startswith("{")][0])
    assert j["dump_outputs"]["files"] == 14 and j["dump_outputs"]["sampled_files"] == 0
    assert sorted(p.name for p in out.iterdir()) == [f"w0_out{k:02d}.npy" for k in range(14)]
    ref = O.window_forward(O.synth_frames(6, 1, 48, 64, seed=1234, smooth=True), O.synth_state_dict(0))
    for k, want in enumerate(ref):
        got = np.load(out / f"w0_out{k:02d}.npy")
        assert got.dtype == np.float32 and got.shape == tuple(want.shape)
        assert np.abs(got - want.numpy()).max() <= 1e-5, k

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = 3 * 40 * 50
    step = [[torch.arange(n, dtype=torch.float32).reshape(1, 3, 40, 50) + 10_000 * k for k in range(14)] for _ in range(2)]
    budget = 100_000
    a = bench.dump_outputs(str(tmp_path / "a"), step, budget=budget)
    b = bench.dump_outputs(str(tmp_path / "b"), step, budget=budget)
    assert a["files"] == b["files"] == 28 and a["sampled_files"] == 28 and a["bytes"] == b["bytes"] <= budget
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) == a["bytes"]
    idx = None
    for w in range(2):
        for k in range(14):
            x = np.load(tmp_path / "a" / f"w{w}_out{k:02d}.npy")
            assert np.array_equal(x, np.load(tmp_path / "b" / f"w{w}_out{k:02d}.npy"))
            assert x.dtype == np.float32 and x.shape == (a["elements_per_sampled_file"],)
            i = x - 10_000 * k                                  # the values are the sampled flat indices
            idx = i if idx is None else idx
            assert np.array_equal(i, idx)
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < n


def test_bench_clock_sampler_uses_only_samples_of_the_timed_region():
    """bench.py's ClockSampler: median / min SM clock and throttle reasons come from the samples that arrived between
    mark_begin and mark_end (the sampler itself starts before the warm-up); without nvidia-smi it says so."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class FakeProc:
        def terminate(self):
            pass
    s = bench.ClockSampler(0)
    s.proc = FakeProc()
    row = lambda mhz, cap: ["0", str(mhz), "1965", "700.0", "Not Active", "Not Active", "Not Active", cap]
    s.rows = [(10.0, row(1965, "Not Active")), (20.5, row(1500, "Active")), (21.0, row(1470, "Active")), (21.5, row(1530, "Active")),
              (40.0, row(600, "Not Active"))]
    s.t0, s.t1 = 20.0, 22.0
    r = s.stop()
    assert r["sm_mhz"] == 1500 and r["sm_min_mhz"] == 1470 and r["sm_max_mhz"] == 1965 and r["samples"] == 3
    assert r["reasons"] == ["sw_power_cap"]
    s2 = bench.ClockSampler(0)                        # nvidia-smi absent (this container)
    assert s2.stop()["reasons"] == ["nvidia-smi unavailable"]
    p = bench.peaks()
    assert p["bf16_tflops"] > 0 and p["hbm_gbs"] > 0 and p["source"] in ("measured", "fallback")
