"""The JSON line bench.py prints (the driver's contract), checked on the lines recorded on B200s under profiles/ and —
on a GPU box — on a short live run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def check_line(d, reference=False):
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "circuit-timesteps/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None      # BASELINE.md publishes no number
    assert "workload" in d["config"] and "model" not in d["config"] and "l2" in d["config"]
    e = d["e2e"]
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(e) and e["value"] > 0
    if reference:
        assert d["impl"] == "reference" and d["gpu_launches"] == 0 and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
        c = d["cpu_baseline"]
        assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] == d["value"] and c["sample"]
        return
    assert d["gpu_launches"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    assert d["value"] > 1e9 and d["steps"] >= 1 and d["warmup"] >= 3
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0 < r["frac"] < 1.2
    cl = d["clocks"]
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(cl)
    assert not set(cl["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if d["n_gpus"] == 1:
        c = d["cpu_baseline"]
        assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]


@pytest.mark.parametrize("name", ["bench_r01_final_1m.json", "bench_r01_final_2gpu.json", "bench_r01_final_8gpu.json"])
def test_recorded_bench_lines_follow_the_contract(name):
    d = json.load(open(os.path.join(ROOT, "profiles", name)))
    check_line(d)


def test_recorded_reference_arm_line():
    check_line(json.load(open(os.path.join(ROOT, "profiles", "bench_r01_final_reference_arm.json"))), reference=True)


def load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    B = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(B)
    return B


def check_dump(out_dir, n):
    """--dump-outputs: float64 arrays only, 64 MB at most, the sampled instances' statistics / rows / status of rc and rlc."""
    files = sorted(os.listdir(out_dir))
    assert files == sorted(f"{deck}_{a}.npy" for deck in ("rc", "rlc") for a in ("stats", "rows", "status", "instance")), files
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in files) <= 64 << 20
    arr = {f[:-4]: np.load(os.path.join(out_dir, f)) for f in files}
    assert all(a.dtype == np.float64 for a in arr.values())
    k = min(n, 1 << 16)
    for deck, ncol in (("rc", 5), ("rlc", 7)):
        idx = arr[f"{deck}_instance"]
        assert idx.shape == (k,) and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < n
        assert arr[f"{deck}_stats"].shape == (4, ncol, k) and arr[f"{deck}_rows"].shape == (k,) and arr[f"{deck}_status"].shape == (k,)
    return arr


def test_dump_outputs_with_stand_in_batches(tmp_path):
    """dump_outputs on the CPU: batches whose results are known functions of the instance index, so the sample can be checked
    value for value; the same call twice gives the same files."""
    B = load_bench()

    class StandIn:
        def __init__(self, n, ncol):
            self.n, self.ncol = n, ncol

        def stats_all(self):
            return np.arange(4 * self.ncol * self.n, dtype=np.float64).reshape(4, self.ncol, self.n)

        def rows(self):
            return np.arange(self.n, dtype=np.int64) + 300

        def status(self):
            return (np.arange(self.n) % 3 == 0).astype(np.int32)

    n = 100_000
    decks = [dict(name="rc", b_res=StandIn(n, 5)), dict(name="rlc", b_res=StandIn(n, 7))]
    B.dump_outputs(str(tmp_path / "a"), decks, n)
    B.dump_outputs(str(tmp_path / "b"), decks, n)
    arr = check_dump(tmp_path / "a", n)
    for name, a in arr.items():
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{name}.npy")), name
    for d in decks:
        idx = arr[d["name"] + "_instance"].astype(np.int64)
        assert np.array_equal(arr[d["name"] + "_stats"], d["b_res"].stats_all()[:, :, idx])
        assert np.array_equal(arr[d["name"] + "_rows"], idx + 300) and np.array_equal(arr[d["name"] + "_status"], idx % 3 == 0)


def test_private_kernel_cache_leaves_the_prebuilt_cache_untouched(tmp_path, monkeypatch):
    """The kernel cache bench.py hands the library: every pre-built file readable through it, and a file the library writes
    (under a private name, then renamed into place) replaces the link, not the pre-built file."""
    B = load_bench()
    src = tmp_path / "kcache"
    src.mkdir()
    (src / "k.cubin").write_bytes(b"prebuilt")
    (src / "k.auto").write_text("3\n")
    monkeypatch.setenv("TSB_KCACHE", str(src))
    cache = B.private_kernel_cache()
    d = cache.name
    assert not d.startswith(ROOT) and sorted(os.listdir(d)) == ["k.auto", "k.cubin"]
    assert open(os.path.join(d, "k.cubin"), "rb").read() == b"prebuilt"
    with open(os.path.join(d, "k.auto.tmp1"), "w") as f:
        f.write("5\n")
    os.rename(os.path.join(d, "k.auto.tmp1"), os.path.join(d, "k.auto"))
    assert (src / "k.auto").read_text() == "3\n" and open(os.path.join(d, "k.auto")).read() == "5\n"
    cache.cleanup()
    assert not os.path.exists(d) and sorted(os.listdir(src)) == ["k.auto", "k.cubin"]


@pytest.mark.gpu
def test_live_bench_line(built, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--instances", "65536", "--no-cpu-baseline",
                        "--config-scale", "0.004", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    arr = check_dump(tmp_path / "out", 65536)
    for deck in ("rc", "rlc"):
        assert np.all(arr[f"{deck}_status"] == 0) and np.all(arr[f"{deck}_rows"] > 0) and np.isfinite(arr[f"{deck}_stats"]).all()
    d = json.loads(r.stdout.strip().splitlines()[-1])
    d["cpu_baseline"] = d["cpu_baseline"] or {"value": 1.0, "unit": "", "cores": 1, "kind": "port", "sample": "skipped"}
    check_line(d)
    # one entry per BASELINE.json config, every deck with a time, a throughput and a roofline fraction
    cfgs = d["configs"]
    assert len(cfgs) == 5 and not any("error" in c for c in cfgs), cfgs
    assert cfgs[0]["exact"] is True
    names = [[e["deck"] for e in c["decks"]] for c in cfgs[1:]]
    assert names == [["rc", "rlc"], ["diode2", "diode4", "diode1", "diode5", "diode3"], ["mosfet1", "bjt2", "bjt1", "bjt3"],
                     ["transformer3", "transformer1", "transformer2"]]
    for c in cfgs[1:]:
        for e in c["decks"]:
            assert e["ms_per_launch"] > 0 and e["circuit_timesteps_per_sec"] > 0 and 0 < e["frac"] < 1.2 and 0 < e["lane_util"] <= 1.0, e
    assert d["strong"]["scaling"] == "strong" and d["e2e"]["results_check"] is True and "excluded" in d["config"]
    # the larger-n entry: both ladders on the thread mapping and on the cooperative mapping, nothing failed
    ln = d["larger_n"]
    assert "error" not in ln and len(ln["workloads"]) == 2, ln
    for w in ln["workloads"]:
        assert [m["coop_parts"] for m in w["mappings"]] == [0, 2, 4] and all(m["failed"] == 0 and m["steps"] > 0 for m in w["mappings"]), w


def test_operator_lu_entry_with_a_stand_in_context(built):
    """bench.py's `operator_lu` entry (measure_lu_operator) end to end on the CPU: the synthetic systems, the pivot order of the
    nominal matrix (tsb_lu_order, host only), the call shape of tsb_lu_solve_batched_dev, the figures it derives — with a
    stand-in context that solves the systems with torch.linalg.solve where the real one launches csrc/lu_warp.cu."""
    import gc
    import time

    import torch
    B = load_bench()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import parity_util as PU

    class StandIn:
        def lu_solve_batched_dev(self, n, n_inst, a_ptr, b_ptr, x_ptr, st_ptr, order, strict=False):
            assert len(order[0]) == n and sorted(order[0]) == list(range(1, n + 1))
            ts = {t.data_ptr(): t for t in gc.get_objects() if isinstance(t, torch.Tensor)}
            A, b, x, st = ts[a_ptr], ts[b_ptr], ts[x_ptr], ts[st_ptr]
            assert A.shape == (n_inst, n, n) and A.is_contiguous()
            x.copy_(torch.linalg.solve(A, b.unsqueeze(-1)).squeeze(-1)); st.zero_()

    def timed(fn, reps=3, warm=1):
        out = []
        for _ in range(reps):
            t0 = time.time(); fn(); out.append((time.time() - t0) * 1e3)
        return out

    r = B.measure_lu_operator(PU.T, StandIn(), timed, "cpu", 36.6, budget_bytes=2e6)
    assert [o["n"] for o in r["orders"]] == [8, 16, 32]
    for o in r["orders"]:
        assert o["singular"] == 0 and o["max_backward_error"] < 1e-13 and o["systems"] > 100
        assert abs(o["tflops_dense_count"] - o["systems_per_sec"] * B.lu_dense_flops(o["n"]) / 1e12) < 1e-9 * o["tflops_dense_count"] + 1e-18
    assert B.lu_dense_flops(5) == 120 and B.lu_dense_flops(32) == 23376          # SURVEY a11: the reference's dense count
