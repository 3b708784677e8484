"""The JSON line bench.py prints is a contract with its readers: every required key must be there for the
HBM-bound (N=1) and the NVLink-bound (N>1) form, with traffic figures coming from the committed ncu table.
--dump-outputs writes a bounded, reproducible sample of what the timed path computed."""

import importlib
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    return importlib.import_module("bench")


INFO = {"num_rects": 1194, "num_tiles": 22665, "payload_bytes": 2008031232, "src_bytes": 2008031232,
        "remote_src_bytes": 528948224, "num_link_tiles": 143815, "link_bytes": 528948224, "grid": 444, "block": 288,
        "tile_bytes": 65536, "num_vector_rects": 1194, "link_tile_bytes": 4096, "link_stages": 6}
REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"]


def test_roofline_blocks_have_the_contract_keys_and_live_traffic():
    b = _bench()
    hbm = b.roofline_for(False, dict(INFO, remote_src_bytes=0), 4.7, 1)
    nvl = b.roofline_for(True, INFO, 0.81, 8)
    for r in (hbm, nvl):
        for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
            assert k in r
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert hbm["bound"] == "hbm" and nvl["bound"] == "nvlink"
    table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    assert sorted(table) == ["1", "2", "4", "8"]
    assert hbm["traffic"] == table["1"]["dram_bytes"] and nvl["traffic"] == table["8"]["dram_bytes"]
    assert nvl["nvlink_traffic"] == table["8"]["nvlrx_bytes"]
    # the capture of the shipped build moves exactly the algorithmic bytes over the link, and no more than them through DRAM
    assert table["8"]["nvlrx_user_bytes"] == INFO["remote_src_bytes"]
    algo_hbm_n1 = 2 * 16060522496
    assert 0.99 < table["1"]["dram_bytes"] / algo_hbm_n1 < 1.01
    assert nvl["frac_of_bidirectional_peak"] > nvl["frac"]  # the two-way link rate is the tighter bound
    assert nvl["hbm"]["algorithmic_bytes_per_launch_incl_serving_peers"] == 2 * INFO["payload_bytes"]


def test_base_line_carries_every_contract_key():
    b = _bench()
    ctx = types.SimpleNamespace(world=8, args=types.SimpleNamespace(steps=30, warmup=3, config="4"), numa={"bound": True})
    timed = {"clocks": {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": []}, "launches": 240}
    line = b.base_line(ctx, 18000.0, 0.85, "workload", {"state_dict_bytes": 16060522496}, timed,
                       b.roofline_for(True, INFO, 0.81, 8),
                       {"value": 414.0, "unit": "GB/s", "h2d_bytes_per_step": 16060522496, "d2h_bytes_per_step": 1}, None, 0.7)
    for k in REQUIRED:
        assert k in line, k
    assert line["config"]["workload"] == "workload" and "model" not in line["config"]
    assert line["higher_is_better"] is True and line["n_gpus"] == 8 and line["gpu_launches"] == 240
    json.dumps(line)  # serialisable


def test_dump_outputs_writes_whole_small_tensors_and_a_fixed_sample_of_large_ones(tmp_path):
    import numpy as np
    import torch

    b = _bench()
    big = torch.arange(3_000_000, dtype=torch.float32).reshape(1000, 3000)  # value == flat position
    norm = (torch.randn(4096, generator=torch.Generator().manual_seed(0))).to(torch.bfloat16)
    tensors = {"layers.0.w1.weight": big, "norm.weight": norm}
    budget = 64 << 10  # 8192 float32 elements per tensor
    b.dump_outputs(str(tmp_path / "a"), tensors, budget=budget)
    b.dump_outputs(str(tmp_path / "b"), tensors, budget=budget)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["layers.0.w1.weight.npy", "norm.weight.npy"]
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()  # same arguments, same sample
    whole = np.load(tmp_path / "a" / "norm.weight.npy")
    assert whole.dtype == np.float32 and np.array_equal(whole, norm.float().numpy())
    sample = np.load(tmp_path / "a" / "layers.0.w1.weight.npy")
    assert sample.dtype == np.float32 and sample.shape == (8192,)
    assert np.all(np.diff(sample) > 0) and sample[0] >= 0 and sample[-1] < big.numel()  # distinct sorted positions
    b.dump_outputs(str(tmp_path / "c"), dict(reversed(tensors.items())), budget=budget)
    for f in files:  # the sample follows the tensor's name, not its place in the dict
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "c" / f).read_bytes()
    b.dump_outputs(str(tmp_path / "r"), tensors, rank=1, world=2, budget=budget)
    assert sorted(os.listdir(tmp_path / "r")) == ["layers.0.w1.weight.rank1.npy", "norm.weight.rank1.npy"]
    assert np.load(tmp_path / "r" / "layers.0.w1.weight.rank1.npy").shape == (4096,)


def test_dump_outputs_of_the_headline_workload_stay_within_64_mb():
    import math

    b = _bench()
    layout = b.workloads.llama_layout(b.workloads.LLAMA3_8B)
    cap = b.DUMP_BYTES // 4 // len(layout)
    header = 128  # numpy .npy header of a version-1 file
    assert sum(min(math.prod(shape), cap) * 4 + header for shape, _ in layout.values()) <= 64 << 20


def test_cpu_reference_run_times_exactly_the_requested_steps(monkeypatch):
    """--steps K means K timed syncs however long they take: a clock that runs 100 s per reading would
    end any time budget after the first one."""
    b = _bench()
    clock = iter(range(0, 10**9, 100))
    monkeypatch.setattr(b.time, "perf_counter", lambda: float(next(clock)))
    for k in (1, 4):
        res = b.cpu_reference_run(2, steps=k, warmup=1, layers=1)
        assert res["steps"] == k and res["value"] > 0 and res["ms_min"] <= res["ms_per_step"] <= res["ms_max"]


def test_cpu_baseline_oracle_rebuilds_outside_a_read_only_tree(tmp_path, monkeypatch):
    """bench.py's CPU baseline loads the C oracle; a stale or missing copy in a tree it cannot write is
    rebuilt in a temporary directory instead of failing."""
    import numpy as np

    from oracle import c_oracle
    from torchstore_b200 import _native

    tree = tmp_path / "tree"
    monkeypatch.setattr(c_oracle, "LIB", str(tree / "_build" / "liboracle_copy_rects.so"))
    monkeypatch.setattr(c_oracle, "_writable_dir", lambda path: False)
    monkeypatch.setattr(c_oracle, "_lib", None)
    path = c_oracle.build()
    assert os.path.exists(path) and not path.startswith(str(tree)) and not tree.exists()
    src = np.arange(64, dtype=np.uint16)
    dst = np.zeros(64, dtype=np.uint16)
    rects = _native.make_rect_array(1)
    r = rects[0]
    r.src, r.dst, r.ndim = src.ctypes.data, dst.ctypes.data, 1
    for i in range(_native.TSB_MAX_DIMS):
        r.extent[i], r.src_stride[i], r.dst_stride[i] = 1, 0, 0
    r.extent[0], r.src_stride[0], r.dst_stride[0] = 64, 2, 2
    r.src_dtype = r.dst_dtype = _native.TSB_U16
    r.src_device = -1
    c_oracle.copy_rects(rects, 1)
    assert np.array_equal(dst, src)


def test_dump_outputs_is_refused_where_it_is_not_implemented(tmp_path):
    import subprocess

    for extra in (["--config", "2"], ["--impl", "reference"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path), *extra],
                             capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "--dump-outputs" in out.stderr
    assert not os.listdir(tmp_path)
