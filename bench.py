#!/usr/bin/env python
"""bench.py — circuit-timesteps/sec of the batched FP64 transient hot path (BASELINE.json metric).

Headline workload (BASELINE.json configs[1]): rc.cir + rlc.cir linear transient, 2^20-instance R/L/C parameter
sweep per GPU (SURVEY.md §8(d): nominal * LogUniform[0.5, 2], PCG64 seed 1234), summary-statistics output
(min / max / sum / last per signal + row counts; full rlc waveforms for 2^20 instances would be ~640 GB).
One "step" = one pass of the hot path over that batch: one transient launch per deck.

  value     whole-job accepted transient steps / s with parameters already resident in HBM
  e2e       the same through the public API with HOST buffers: every step the parameter arrays are copied H2D from
            pinned memory and every instance's statistics / row count / status are read back into pinned memory
            (tsb_result_fetch_async: the read-back of one launch overlaps the next launch)
  roofline  the dominant launch (rlc transient): algorithmic FP64 flops / CUDA-event time vs the DFMA-chain peak
            measured in this run (MEASURED_PEAKS.json has no FP64 figure)
  configs   one entry per BASELINE.json config (rr plumbing; rc + rlc; diode1-5; bjt1-3 + mosfet1; transformer1-3
            with 2^24 instances split over the N GPUs): ms per launch, circuit-timesteps/s, executed solves, FP64
            roofline fraction of an executed-flop model, lane utilisation
  strong    transformer1.cir, 2^24 instances IN TOTAL over the N GPUs (strong scaling)
  operator_lu
            the operator-level batched LU (tsb_lu_solve_batched_dev): dense systems of order 8 / 16 / 32, systems/s, dense-count
            TFLOP/s against the same FP64 peak, backward error of a sample
  cpu_baseline / --impl reference
            the CPU restatement of the reference solver (oracle/, `kind: port` — the Go reference cannot be built
            here), one task per instance on all host threads, bounded sample.  The reference arm imports nothing of
            the product (front-end: oracle/netlist.py; draws: the workload module loaded by file path).

Launch: `python bench.py --gpus N --steps K --warmup W`; for N > 1 under torchrun (one rank per GPU, instances
sharded by rank, no collective on the data path; totals all-reduced at the end).

`--dump-outputs DIR` (e.g. bench_out/) writes what the last timed step returned for a fixed sample of instances, so that two
builds can be compared output for output (dump_outputs).  bench.py writes nothing into the tree it runs from: kernels it
compiles or tunes at run time go to a temporary directory (private_kernel_cache).
"""
from __future__ import annotations

import argparse
import importlib
import importlib.util
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DECKS = ("rc", "rlc")
DUMP_SAMPLE = 1 << 16       # instances per deck in --dump-outputs: at most (4 x 7 + 3) x 8 bytes each, under 33 MB for rc + rlc
DUMP_SEED = 2024


def load_workloads():
    """toy-spice_b200/workloads.py (decks = input data, sweep definitions) loaded BY FILE PATH: no import of the
    product package, no CUDA library in the process — what the reference arm needs."""
    spec = importlib.util.spec_from_file_location("tsb_workloads", os.path.join(ROOT, "toy-spice_b200", "workloads.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# --------------------------------------------------------------------------------------------
# Algorithmic FP64 work per Newton solve (SURVEY.md §8(d) / a11), stated in DESIGN.md §6.1.
def f_lu_dense(n: int) -> int:
    """Dense LU + triangular solves as the reference performs them (structure is dense n x n,
    SURVEY Q16): sum_k [1 + (n-k) + 2(n-k)^2] + n + 2n(n-1)."""
    return sum(1 + (n - k) + 2 * (n - k) ** 2 for k in range(1, n + 1)) + n + 2 * n * (n - 1)


# per device kind: stamp arithmetic incl. the transcendental functions at ~40 flop per exp / log / pow and ~20 per
# sqrt (SURVEY §8(d): "nonlinear add ~40-60 flops per exp/pow"): R 5, C 8, L 9, V 5 (+ sin), I 2, D 15 + 1 exp,
# Q 60 + 2 exp + 1 pow, M 60 + 2 sqrt (Level 1), K 12 per pair, core L 9
STAMP_FLOPS = {0: 5, 1: 8, 2: 9, 3: 5, 4: 2, 5: 55, 6: 180, 7: 100, 8: 12, 9: 9}


def flops_per_solve(devs, n) -> dict:
    stamp = sum(STAMP_FLOPS[d["kind"]] for d in devs)
    conv = 5 * n
    return dict(n=n, lu=f_lu_dense(n), stamp=stamp, conv=conv, total=f_lu_dense(n) + stamp + conv)


def executed_flops(deck: str, strict: int = 0):
    """FP64 flops per EXECUTED solve as ncu counted them (2*DFMA + DMUL + DADD, thread level; tests/gpu_flops.py ->
    profiles/executed_flops.json), or None.  The generated kernels skip structural zeros, condense the invariant pivots and
    hoist invariant stamps, so this is well below the dense-algorithm model above — `frac` is reported on THIS figure."""
    try:
        e = json.load(open(os.path.join(ROOT, "profiles", "executed_flops.json")))["decks"].get(deck + (":strict" if strict else ""))
        return float(e["flops_per_executed_solve"]) if e else None
    except Exception:
        return None


def lu_dense_flops(n: int) -> int:
    """Factor + solve of one dense system of order n as the reference's sparse module does it (SURVEY a11)."""
    return sum(1 + (n - k) + 2 * (n - k) ** 2 for k in range(1, n + 1)) + n + 2 * n * (n - 1)


def measure_lu_operator(T, ctx, timed_launches, dev_name: str, fp64_peak, budget_bytes: float = 1e9, orders=(8, 16, 32)) -> dict:
    """Operator-level entry (tsb_lu_solve_batched_dev, csrc/lu_warp.cu: the drop-in for the reference's matrix operator): batches
    of dense systems of one order sharing the pivot order of a nominal matrix, device pointers, fast build.  Synthetic systems: a
    diagonally dominant conductance-like nominal matrix, every entry of every instance scaled by LogUniform[0.5, 2]."""
    import torch
    out = {"kernel": "tsb_k_lu_warp (2 - 3 rows per lane, cp.async staging; fast build)", "orders": []}
    for n in orders:
        rng = np.random.default_rng(1234 + n)
        base = rng.uniform(-1e-3, 0.0, (n, n)) * (rng.random((n, n)) < 0.35)
        base = base + base.T
        np.fill_diagonal(base, 0.0)
        np.fill_diagonal(base, -base.sum(axis=1) + 1e-4)
        order = T.lu_order(base)
        n_inst = int(min(1 << 22, budget_bytes // (n * n * 8)))
        gen = torch.Generator(device=dev_name); gen.manual_seed(99 + n)
        scale = torch.exp(torch.empty((n_inst, n, n), dtype=torch.float64, device=dev_name).uniform_(float(np.log(0.5)), float(np.log(2.0)), generator=gen))
        dA = (torch.from_numpy(base).to(dev_name)[None] * scale).contiguous()
        del scale
        db = torch.empty((n_inst, n), dtype=torch.float64, device=dev_name).normal_(generator=gen)
        dx = torch.empty_like(db)
        dst = torch.empty(n_inst, dtype=torch.int32, device=dev_name)
        ms = min(timed_launches(lambda: ctx.lu_solve_batched_dev(n, n_inst, dA.data_ptr(), db.data_ptr(), dx.data_ptr(), dst.data_ptr(), order, strict=False), reps=3))
        # normwise backward error of the first 256 systems (the check travels with the number)
        k = min(256, n_inst)
        A, b, x = dA[:k].cpu().numpy(), db[:k].cpu().numpy(), dx[:k].cpu().numpy()
        den = np.abs(A).sum(axis=2).max(axis=1) * np.abs(x).max(axis=1) + np.abs(b).max(axis=1)
        berr = float((np.abs(np.einsum("qij,qj->qi", A, x) - b).max(axis=1) / den).max())
        tf = n_inst * lu_dense_flops(n) / (ms * 1e-3) / 1e12
        out["orders"].append({"n": n, "systems": n_inst, "ms_per_launch": ms, "systems_per_sec": n_inst / (ms * 1e-3), "tflops_dense_count": tf,
                              "frac_fp64": tf / fp64_peak if fp64_peak else None,
                              "algorithmic_gbs": n_inst * ((n * n + 2 * n) * 8 + 4) / (ms * 1e-3) / 1e9,
                              "singular": int(dst.sum().item()), "max_backward_error": berr})
        del dA, db, dx, dst
        torch.cuda.empty_cache() if dev_name.startswith("cuda") else None
    return out


def flop_fields(deck: str, strict: int, executed_solves: int, ms: float, model_flops: int, fp64_peak, n_gpus: int = 1) -> dict:
    """tflops / frac of one launch.  Top level: ALGORITHMIC flops as SURVEY §8(d) defines them (dense n x n LU as the reference
    factors it + stamps + convergence test, per executed solve) — the contract's roofline numerator; a value above 1 means
    the kernel does less arithmetic than the algorithm's count (structural zeros skipped, invariant pivots condensed), like
    DRAM traffic below the algorithmic bytes.  `executed`: the FP64 flops the kernel really issues (ncu opcode counts)."""
    sec = ms * 1e-3
    mt = executed_solves * model_flops / sec / 1e12
    out = {"flops_per_solve": model_flops, "tflops": mt, "frac": mt / (fp64_peak * n_gpus) if fp64_peak else None}
    fe = executed_flops(deck, strict)
    et = executed_solves * fe / sec / 1e12 if fe else None
    out["executed"] = {"flops_per_solve": fe, "tflops": et, "frac": et / (fp64_peak * n_gpus) if (fe and fp64_peak) else None,
                       "source": "ncu opcode counts, 2*DFMA + DMUL + DADD (profiles/executed_flops.json)" if fe else "no capture for this deck"}
    return out


def ncu_json(key: str):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(key)
    except Exception:
        return None


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
        sm, smax, reasons = [], 0.0, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ts, line in self.rows:
            if ts < t0 - 0.1 or ts > t1 + 0.3:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); smax = max(smax, float(f[2]))
                for nm, val in zip(names, f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def private_kernel_cache() -> tempfile.TemporaryDirectory:
    """A temporary kernel-cache directory holding a link to every file of the pre-built cache (build() ->
    toy-spice_b200/_kcache, or $TSB_KCACHE).  The library reads the pre-built cubins through the links and puts what it
    compiles or tunes at run time (NVRTC cubins, launch-bounds choices) there, each file renamed into place over any link
    of that name, so the tree bench.py runs from is only read and may be read-only.  Removed when the process exits."""
    src = os.path.abspath(os.environ.get("TSB_KCACHE") or os.path.join(ROOT, "toy-spice_b200", "_kcache"))
    tmp = tempfile.TemporaryDirectory(prefix="tsb_kcache_")
    if os.path.isdir(src):
        for f in os.listdir(src):
            os.symlink(os.path.join(src, f), os.path.join(tmp.name, f))
    return tmp


def dump_outputs(out_dir: str, decks, n: int) -> None:
    """--dump-outputs: what the last run of every deck's batch returned to its caller -- statistics [4: min, max, sum, last]
    [result column][instance], stored rows and status per instance -- for a fixed sample of instances (DUMP_SAMPLE drawn
    with DUMP_SEED, ascending), as float64 arrays in out_dir/<deck>_{stats,rows,status}.npy; <deck>_instance.npy holds the
    sampled instance indices."""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, min(n, DUMP_SAMPLE), replace=False))
    for d in decks:
        b = d["b_res"]
        arrays = {"stats": b.stats_all()[:, :, idx], "rows": b.rows()[idx], "status": b.status()[idx], "instance": idx}
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, f"{d['name']}_{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


# --------------------------------------------------------------------------------------------
def cpu_sample(O, W, target_seconds: float, threads: int):
    """Time the CPU oracle on a bounded sample of the SAME workload (same decks, same draws).  Device table from the
    oracle's own front-end (oracle/netlist.py): nothing of the product is imported here."""
    per_deck = {}
    total_steps, total_time = 0, 0.0
    desc = []
    for name in DECKS:
        oc = O.OracleCircuit(W.BUNDLED[name])
        devs = [dict(kind=r.kind, name=r.name, p=list(r.p)) for r in oc.plan.devices]
        probe_n = max(threads, 8)
        ov = W.sweep_draws(devs, probe_n, W.sweep_seed(name))
        t0 = time.time()
        oc.run(probe_n, overrides=ov, threads=threads, want_wave=False, want_stats=True)
        rate = probe_n / max(time.time() - t0, 1e-6)
        n = int(min(1 << 16, max(probe_n, rate * target_seconds / len(DECKS))))
        ov = W.sweep_draws(devs, n, W.sweep_seed(name))
        t0 = time.time()
        res = oc.run(n, overrides=ov, threads=threads, want_wave=False, want_stats=True)
        dt = time.time() - t0
        steps = int(res["counters"][:, 0].sum())
        per_deck[name] = dict(instances=n, seconds=dt, steps=steps)
        # weight decks as in the full workload (equal instance counts): time per instance
        total_steps += steps / n
        total_time += dt / n
        desc.append(f"{name}: {n} instances in {dt:.2f}s")
    return total_steps / total_time, "; ".join(desc), per_deck


def headline_config(n, world, strict_fp):
    return {"workload": f"rc.cir + rlc.cir transient, {n}-instance R/L/C sweep per GPU (LogUniform[0.5,2], PCG64 seed 1234), "
                        "summary-statistics output", "instances_per_deck_per_gpu": n,
            "parallelism": f"instances sharded over {world} GPU(s), no collective", "l2": "flushed between timed iterations (256 MB write)",
            "strict_fp": strict_fp,
            "excluded": "one-time set-up outside the timed region: plan + batch creation (netlist front-end, symbolic pass), loading the "
                        "pre-built cubins (NVRTC on a cache miss), the launch-bounds timing pass of a batch's first run, the shared-time-grid "
                        "pilot of a batch's first run (later runs with unchanged analysis arguments reuse its table), pinned-buffer allocation"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Go solver cannot be
    built in this image (no Go toolchain, un-vendored sparse module), so this is the C++ restatement
    (oracle/, kind 'port') on all host threads, one task per instance, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    W = load_workloads()
    from oracle import oracle as O
    threads = host_threads()
    for _ in range(args.warmup):
        cpu_sample(O, W, 1.0, threads)
    vals, t_all, sample = [], 0.0, ""
    for _ in range(args.steps):
        t0 = time.time()
        v, sample, _ = cpu_sample(O, W, max(2.0, 20.0 / max(1, args.steps)), threads)
        t_all += time.time() - t0
        vals.append(v)
    value = float(np.mean(vals))
    cfg = headline_config(args.instances, args.gpus, args.strict_fp)
    cfg["l2"] = "n/a (CPU)"
    cfg["reference_arm"] = "bounded CPU sample of the same decks and draws, per-instance rate"
    line = {
        "metric": "circuit-timesteps/sec (batched FP64 transient)", "value": value, "unit": "circuit-timesteps/s",
        "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_all / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": "circuit-timesteps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "circuit-timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--instances", type=int, default=1 << 20, help="instances per deck per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-BASELINE-config entries and the strong-scaling entry")
    ap.add_argument("--config-scale", type=float, default=1.0, help="scale the instance counts of the `configs` / `strong` entries")
    ap.add_argument("--strict-fp", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step (sampled instances) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the results of the GPU path: not with --impl reference")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    T = importlib.import_module("toy-spice_b200")
    W = importlib.import_module("toy-spice_b200.workloads")
    S = importlib.import_module("toy-spice_b200.sharding")
    ctx = T.Context(local)
    kcache = private_kernel_cache()
    ctx.set_cache_dir(kcache.name)
    stream = torch.cuda.Stream(device=local)
    ctx.set_stream(stream.cuda_stream)
    opts = T.default_opts(strict_fp=args.strict_fp)
    n = args.instances
    dev_name = f"cuda:{local}"

    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype).pin_memory().numpy()

    # ---- workload: decks, per-rank parameter draws (rank r owns its own instance range) ---------
    decks = []
    h2d_bytes = 0
    for name in DECKS:
        ckt = T.Circuit.from_netlist(T.BUNDLED[name], ctx)
        card = ckt.analysis_card()
        ov = W.sweep_draws(ckt.devices(), n, W.sweep_seed(name) + 7919 * rank)
        host = {k: torch.from_numpy(v).pin_memory() for k, v in ov.items()}
        dev = {k: v.to(dev_name, non_blocking=True) for k, v in host.items()}
        b_res = ckt.batch(n)       # parameters resident in HBM (borrowed torch tensors)
        for (d, p), v in dev.items():
            b_res.set_param(d, p, v)
        ncol = len(ckt.columns(T.AN_TRAN))
        # end-to-end: two batches per deck, used alternately, so that the read-back of step i overlaps step i + 1
        e2e = []
        for _ in range(2):
            b = ckt.batch(n)
            for (d, p), v in host.items():
                b.set_param(d, p, v.numpy(), zero_copy=True)
            e2e.append(dict(batch=b, stats=pinned((4, ncol, n), torch.float64), rows=pinned((n,), torch.int64), status=pinned((n,), torch.int32)))
        h2d_bytes += sum(v.numel() * 8 for v in host.values())
        decks.append(dict(name=name, ckt=ckt, card=card, host=host, dev=dev, b_res=b_res, e2e=e2e,
                          flops=flops_per_solve(ckt.devices(), ckt.n), ncol=ncol))
    torch.cuda.synchronize()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev_name)   # 256 MB > 126 MB L2

    def launch_deck(d, batch, out=None):
        c = d["card"]
        batch.run_tran(c["tstart"], c["tstop"], c["tstep"], c["tmax"], c["uic"], out=T.OUT_STATS if out is None else out, opts=opts)

    def step_resident():
        for d in decks:
            launch_deck(d, d["b_res"])

    d2h_bytes = sum(n * (4 * d["ncol"] * 8 + 8 + 4) for d in decks)

    def step_e2e(i):
        """Host buffers in, host buffers out: parameters H2D from pinned memory (DMA on the context's upload stream: beside the
        other batch's running launch), launch, and the read-back of every instance's statistics / rows / status queued behind
        the launch on the copy stream."""
        for d in decks:
            e = d["e2e"][i & 1]
            b = e["batch"]
            b.sync()                                   # THIS batch's step i - 2 and its read-back are complete (results consumed by the host here)
            for (dv, p), v in d["host"].items():
                b.set_param(dv, p, v.numpy(), zero_copy=True)
            launch_deck(d, b)
            b.fetch_async(e["stats"], e["rows"], e["status"])

    def e2e_drain():
        for d in decks:
            for e in d["e2e"]:
                e["batch"].sync()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- FP64 roof of this GPU -----------------------------------------------------------------
    fp64_peak = ctx.measure_fp64_peak()

    # ---- warm-up (also loads / compiles the specialised kernels) --------------------------------
    step_resident()             # priming pass (not one of the W warm-up steps): loads the kernels, runs the launch-bounds autotuner, the pilot
    for _ in range(max(args.warmup, 3 if args.warmup > 0 else 0)):
        step_resident()
    torch.cuda.synchronize()

    # ---- timed: resident parameters (value), per-step CUDA events on the launch stream ----------
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    barrier()
    launches0 = ctx.launch_count
    t_wall0 = time.time()
    ms_steps, ms_dom = [], []
    for _ in range(args.steps):
        flush.zero_()                       # L2 flush between timed iterations (not timed)
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(len(decks) + 1)]
        with torch.cuda.stream(stream):
            e[0].record(stream)
            for i, d in enumerate(decks):
                launch_deck(d, d["b_res"])
                e[i + 1].record(stream)
        stream.synchronize()
        ms_steps.append(e[0].elapsed_time(e[-1]))
        ms_dom.append(e[len(decks) - 1].elapsed_time(e[len(decks)]))      # last deck = rlc = dominant launch
    barrier()
    t_wall1 = time.time()
    launches = ctx.launch_count - launches0
    clocks = sampler.stop(t_wall0, t_wall1)

    totals = {d["name"]: d["b_res"].totals() for d in decks}
    acc_local = int(sum(t[0] for t in totals.values()))
    solves_local = int(sum(t[2] + t[3] for t in totals.values()))     # as the reference counts them
    exec_local = int(sum(t[4] for t in totals.values()))              # factor+solve passes actually executed
    t_local = sum(ms_steps) * 1e-3
    t_job, (acc_job, solves_job, exec_job) = S.reduce_job(t_local, [acc_local, solves_local, exec_local], device=dev_name)
    value = acc_job * args.steps / t_job if t_job > 0 else 0.0
    if args.dump_outputs:
        dump_outputs(os.path.join(args.dump_outputs, f"rank{rank}") if world > 1 else args.dump_outputs, decks, n)

    # ---- timed: end to end through the public API with host buffers -----------------------------
    step_e2e(0); step_e2e(1)
    e2e_drain()
    barrier()
    t0 = time.time()
    for i in range(args.steps):
        step_e2e(i)
    e2e_drain()
    torch.cuda.synchronize()
    t_e2e_local = time.time() - t0
    te = torch.tensor([t_e2e_local], dtype=torch.float64, device=dev_name)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = acc_job * args.steps / float(te[0])
    bad_status = int(sum((e["status"] != 0).sum() for d in decks for e in d["e2e"][:1]))
    # the read-back really is this step's result: the e2e statistics equal the resident run's (same draws)
    e2e_ok = all(np.array_equal(d["e2e"][0]["rows"], d["b_res"].rows()) for d in decks)

    # ---- roofline of the dominant launch (rlc transient) -----------------------------------------
    dom = decks[-1]
    dom_tot = totals[dom["name"]]
    dom_solves = int(dom_tot[4])          # EXECUTED factor+solve passes (the redundant linear re-solve is not run, not counted)
    dom_ms = float(np.mean(ms_dom))
    dom_ff = flop_fields(dom["name"], args.strict_fp, dom_solves, dom_ms, dom["flops"]["total"], fp64_peak)
    ncu_dom = ncu_json(f"ncu:{dom['name']}:{n}:stats") or {}
    # Issue-rate view of the same launch: the kernel's arithmetic is ~1/4 of its instructions (statistics, step control,
    # state rotation, table look-ups are the rest), so the scheduler — 4 warp instructions per clock and SM — is the binding
    # unit, not the FP64 pipe.  warp instructions per executed solve from the ncu capture x executed solves / time / peak.
    wi = ncu_dom.get("warp_instructions_per_executed_solve")
    issue_peak = 148 * 4 * (clocks.get("sm_mhz") or 1965.0) * 1e6
    issue = {"warp_instructions_per_executed_solve": wi, "achieved_per_s": dom_solves / 32 * wi / (dom_ms * 1e-3) if wi else None,
             "peak_per_s": issue_peak, "frac": (dom_solves / 32 * wi / (dom_ms * 1e-3)) / issue_peak if wi else None,
             "peak_source": "148 SMs x 4 schedulers x 1 warp instruction per clock x the SM clock sampled in this run"}
    roofline = {
        "bound": "fp64", "kernel": "tsb_optran (rlc.cir)", "achieved": dom_ff["tflops"], "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": dom_ff["frac"], "traffic": ncu_json(f"{dom['name']}:{n}:stats"),
        "peak_source": "DFMA-chain microbenchmark measured in this run (tsb_ctx_measure_fp64_peak); MEASURED_PEAKS.json has no FP64 figure",
        # `achieved` / `frac`: ALGORITHMIC flops — SURVEY §8(d)'s per-solve figure F_LU(n, dense as the reference factors it) +
        # F_stamp + F_conv x the factor+solve passes this kernel EXECUTES — over the measured FP64 peak (the same accounting
        # as round 1's 0.404).  `executed`: the FP64 arithmetic the kernel really issues per solve (ncu opcode counts): the
        # generated code skips structural zeros and, since round 2, eliminates the run-invariant pivots once per instance,
        # so it issues ~1/3 of the algorithmic count.  Neither figure counts the reference's second solve per step or its
        # LTE-rejected solves (proved redundant, not run): those are in `reference_algorithm`.
        "flops_per_solve": dom["flops"], "executed": dom_ff["executed"],
        "executed_solves_per_launch": dom_solves, "ms_per_launch": dom_ms,
        "reference_algorithm": {"solves_per_launch": int(dom_tot[2]), "flops_per_launch": int(dom_tot[2]) * dom["flops"]["total"],
                                "frac": (int(dom_tot[2]) * dom["flops"]["total"] / (dom_ms * 1e-3) / 1e12) / fp64_peak if fp64_peak else None},
        "issue": issue, "ncu": ncu_dom,
        "algorithmic_hbm_bytes_per_launch": n * (8 * 3 + 4 * dom["ncol"] * 8 + 8 + 4 + 6 * 8),
    }

    def timed_launches(fn, reps=3, warm=1):
        ms = []
        for i in range(warm + reps):
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); fn(); e1.record(stream)
            stream.synchronize()
            if i >= warm:
                ms.append(e0.elapsed_time(e1))
        return ms

    # ---- the HBM-bound regime of the same kernel: rc.cir with every stored row materialised --------------
    # (SURVEY §8(d)(i): 8*O bytes per stored row; not part of `value`, reported beside the FP64 roofline)
    roofline_hbm = None
    try:
        rc = decks[0]
        c = rc["card"]
        bw = rc["ckt"].batch(n)
        for (d, p), v in rc["dev"].items():
            bw.set_param(d, p, v)
        ms_w = timed_launches(lambda: bw.run_tran(c["tstart"], c["tstop"], c["tstep"], c["tmax"], c["uic"], out=T.OUT_WAVE, cap_rows=320, opts=opts))
        rows_total = int(bw.totals()[0])                    # rc stores every accepted step (305 rows per instance)
        alg_bytes = rows_total * rc["ncol"] * 8 + n * (2 * 8 + 8 + 4 + 8 * 8)
        hp, src = hbm_peak()
        ach = alg_bytes / (min(ms_w) * 1e-3) / 1e9
        roofline_hbm = {"bound": "hbm", "kernel": "tsb_optran (rc.cir, TSB_OUT_WAVE)", "achieved": ach, "peak": hp,
                        "unit": "GB/s", "frac": ach / hp, "traffic": ncu_json(f"rc:{n}:wave"), "peak_source": src,
                        "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": min(ms_w),
                        "circuit_timesteps_per_sec": rows_total / (min(ms_w) * 1e-3)}
        del bw
    except Exception as ex:       # the FP64-bound headline must not depend on this extra measurement
        roofline_hbm = {"error": str(ex)[:200]}

    # ---- the operator-level device-stamp kernel (HBM-write-bound: (n^2 + n) * 8 bytes per instance) -----------------
    roofline_stamp = None
    try:
        ns = 1 << 22
        rl = decks[-1]
        nn = rl["ckt"].n
        ovs = W.sweep_draws(rl["ckt"].devices(), ns, 99)
        bs = rl["ckt"].batch(ns)
        keep = []
        for (d, p), v in ovs.items():
            t = torch.from_numpy(v).to(dev_name); keep.append(t)
            bs.set_param(d, p, t)
        dA = torch.empty((ns, nn, nn), dtype=torch.float64, device=dev_name)
        dB = torch.empty((ns, nn), dtype=torch.float64, device=dev_name)
        ms_s = timed_launches(lambda: bs.stamp_dev(T.AN_TRAN, 1e-4, 1e-6, 0.0, dA.data_ptr(), dB.data_ptr(), opts=opts), reps=4)
        sbytes = ns * ((nn * nn + nn) * 8 + len(ovs) * 8)
        hp, hsrc = hbm_peak()
        ach_s = sbytes / (min(ms_s) * 1e-3) / 1e9
        roofline_stamp = {"bound": "hbm", "kernel": "tsb_stamp_staged (rlc.cir transient stamps, operator level)", "achieved": ach_s, "peak": hp,
                          "unit": "GB/s", "frac": ach_s / hp, "traffic": None, "peak_source": hsrc, "algorithmic_bytes_per_launch": sbytes,
                          "ms_per_launch": min(ms_s), "instances": ns}
        del bs, dA, dB, keep
    except Exception as ex:
        roofline_stamp = {"error": str(ex)[:200]}

    # ---- one entry per BASELINE.json config ------------------------------------------------------------------------
    def lane_util(cnt_exec):
        """Share of the lane-iterations of a warp-synchronous run that do work: sum of the executed solves over 32 x the
        slowest lane of every warp (from per-instance totals: an upper bound, waits inside a step are not visible)."""
        m = len(cnt_exec) // 32 * 32
        if m == 0:
            return None
        w = cnt_exec[:m].reshape(-1, 32)
        den = float(32 * w.max(axis=1).sum())
        return float(w.sum()) / den if den > 0 else None

    def measure_deck(name, n_inst, text=None, analysis=None, tran=None, seed=None, reps=2, strict=None):
        text = T.BUNDLED[name] if text is None else text
        ckt = T.Circuit.from_netlist(text, ctx)
        card = ckt.analysis_card()
        if tran:
            card = dict(card, **tran, analysis=T.AN_TRAN)
        an = card["analysis"] if analysis is None else analysis
        lo, hi = S.shard_range(n_inst, rank, world) if seed == "global" else (0, n_inst)
        ov = W.sweep_draws(ckt.devices(), n_inst, W.sweep_seed(name) + (0 if seed == "global" else 7919 * rank))
        b = ckt.batch(hi - lo)
        keep = []
        for (d, p), v in ov.items():
            t = torch.from_numpy(np.ascontiguousarray(v[lo:hi])).to(dev_name); keep.append(t)
            b.set_param(d, p, t)
        del ov
        o = T.default_opts(strict_fp=args.strict_fp if strict is None else strict)
        if an == T.AN_TRAN:
            run = lambda: b.run_tran(card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"], out=T.OUT_STATS, opts=o)
        elif an == T.AN_OP:
            run = lambda: b.run_op(o)
        else:
            run = lambda: b.run_dc(card["dc_src_dev"], card["dc_start"], card["dc_stop"], card["dc_inc"], out=T.OUT_STATS, opts=o)
        ms = min(timed_launches(run, reps=reps))
        tot = b.totals()
        nl = ckt_has_nonlinear(ckt)
        cnt = b.counters() if (nl or an != T.AN_TRAN) else None               # per-instance counters only where they are looked at
        st = b.status()
        fl = flops_per_solve(ckt.devices(), ckt.n)
        steps = int(tot[0]) if an == T.AN_TRAN else int(cnt[7].sum())        # accepted steps / stored sweep points / 1 per OP
        ent = {"deck": name, "analysis": {T.AN_OP: "op", T.AN_TRAN: "tran", T.AN_DC: "dc"}[an], "instances": hi - lo, "n": ckt.n,
               "ms_per_launch": ms, "steps": steps, "circuit_timesteps_per_sec": steps / (ms * 1e-3), "executed_solves": int(tot[4]),
               **flop_fields(name, args.strict_fp if strict is None else strict, int(tot[4]), ms, fl["total"], fp64_peak),
               "lane_util": lane_util(cnt[6]) if nl else 1.0,
               "status_counts": {int(k): int(v) for k, v in zip(*np.unique(st, return_counts=True))},
               "nan_instances": int(np.isnan(b.stats_all()[3]).any(axis=0).sum()) if (an != T.AN_OP and hi - lo <= (1 << 22)) else None}
        del b, keep
        return ent

    def ckt_has_nonlinear(ckt):
        return any(d["kind"] in (T.api.K_D, T.api.K_Q, T.api.K_M) for d in ckt.devices())

    configs, strong = None, None
    if not args.no_configs:
        sc = args.config_scale
        n20, n22, n24 = max(1024, int((1 << 20) * sc)), max(1024, int((1 << 22) * sc)), max(1024 * world, int((1 << 24) * sc))
        tran150 = dict(tstart=0.0, tstop=150e-6, tstep=1e-6, tmax=0.0, uic=False)
        configs = []
        try:
            # [0] rr.cir operating point, batch = 1: plumbing (exact known answer)
            ckt = T.Circuit.from_netlist(T.BUNDLED["rr"], ctx)
            op = T.NewOP(); op.Setup(ckt); op.Execute(); r = op.GetResults()
            configs.append({"config": "configs[0] rr.cir DC operating point, batch=1", "V(2)": float(r["V(2)"][0]), "I(Vin)": float(r["I(Vin)"][0]),
                            "exact": bool(r["V(1)"][0] == 5.0 and r["V(2)"][0] == 2.5)})
            # [1] the headline decks
            configs.append({"config": "configs[1] rc.cir + rlc.cir linear transient, R/L/C sweep",
                            "decks": [{"deck": d["name"], "analysis": "tran", "instances": n, "n": d["ckt"].n,
                                       "ms_per_launch": float(np.mean([ms_steps[i] - ms_dom[i] for i in range(len(ms_dom))])) if d is decks[0] else dom_ms,
                                       "steps": int(totals[d["name"]][0]), "executed_solves": int(totals[d["name"]][4]),
                                       "model_flops": d["flops"]["total"], "lane_util": 1.0} for d in decks]})
            for e in configs[-1]["decks"]:
                e["circuit_timesteps_per_sec"] = e["steps"] / (e["ms_per_launch"] * 1e-3)
                e.update(flop_fields(e["deck"], args.strict_fp, e["executed_solves"], e["ms_per_launch"], e.pop("model_flops"), fp64_peak))
            # [2] diode1-5: Monte Carlo over Is / n
            configs.append({"config": "configs[2] diode1-5.cir, Monte Carlo over Is / n (Newton with per-instance convergence masks)",
                            "decks": [measure_deck(nm, n20) for nm in ("diode2", "diode4", "diode1", "diode5", "diode3")]})
            # [3] bjt1-3 + mosfet1: device-parameter sweep (bjt1 / bjt3 with the supplied .tran 1u 150u, SURVEY §8(d)(4))
            configs.append({"config": "configs[3] bjt1-3.cir + mosfet1.cir nonlinear transient, device-parameter sweep",
                            "decks": [measure_deck("mosfet1", n22), measure_deck("bjt2", n22), measure_deck("bjt1", n22, tran=tran150),
                                      measure_deck("bjt3", n22, tran=tran150)]})
            # [4] transformer1-3: coupled inductors, 2^24 instances over the N GPUs (each rank its contiguous shard of ONE global draw)
            configs.append({"config": f"configs[4] transformer1-3.cir coupled-inductor transient, {n24} instances over {world} GPU(s)",
                            "decks": [measure_deck(nm, n24, seed="global", reps=1) for nm in ("transformer3", "transformer1", "transformer2")]})
        except Exception as ex:
            configs.append({"error": repr(ex)[:300]})
        # multi-GPU: per-deck time = max over ranks, work = sum over ranks
        if world > 1:
            for cfg in configs:
                for e in cfg.get("decks", []):
                    t = torch.tensor([e["ms_per_launch"]], dtype=torch.float64, device=dev_name)
                    w = torch.tensor([float(e["steps"]), float(e["executed_solves"]), float(e["instances"])], dtype=torch.float64, device=dev_name)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(w, op=dist.ReduceOp.SUM)
                    e["ms_per_launch"], e["steps"], e["executed_solves"], e["instances"] = float(t[0]), int(w[0]), int(w[1]), int(w[2])
                    e["circuit_timesteps_per_sec"] = e["steps"] / (e["ms_per_launch"] * 1e-3)
                    e.update(flop_fields(e["deck"], args.strict_fp, e["executed_solves"], e["ms_per_launch"], e["flops_per_solve"], fp64_peak, world))
        t1 = [e for cfg in configs for e in cfg.get("decks", []) if e.get("deck") == "transformer1"]
        if t1:
            e = t1[0]
            strong = {"workload": f"transformer1.cir transient, {e['instances']} instances in total over {world} GPU(s) (strong scaling: "
                                  "contiguous shards of one global draw, seed 4567)", "n_gpus": world, "ms": e["ms_per_launch"],
                      "circuit_timesteps_per_sec": e["circuit_timesteps_per_sec"], "scaling": "strong"}

    # ---- larger n (SURVEY §8(f)4): a 24-section RC ladder (26 unknowns, 51 result columns), one thread per circuit against the
    # cooperative mapping (one instance per 2 threads in different warps, tsb_opts.coop_parts; the default picks it) ----------
    larger_n = None
    if not args.no_configs:
        try:
            nl = max(1024, int((1 << 18) * args.config_scale))
            larger_n = {"default": "coop_parts = -1 picks 2 parts for circuits of >= 16 unknowns without BJTs / mutual couplings (fast build)", "workloads": []}
            for title, ltext in (("RC ladder, 24 sections (n = 26 unknowns, 51 result columns)", W.rc_ladder(24)),
                                 ("diode-clamped RC ladder, 24 sections (n = 26, 14 diodes: Newton loops)", W.diode_rc_ladder(24))):
                lckt = T.Circuit.from_netlist(ltext, ctx)
                lcard = lckt.analysis_card()
                lov = W.sweep_draws(lckt.devices(), nl, 5 + 7919 * rank)
                ldev = {k: torch.from_numpy(v).to(dev_name) for k, v in lov.items()}
                ent = {"workload": f"{title}, {nl} instances per GPU, transient, statistics output", "mappings": []}
                for parts, label in ((0, "one thread per circuit"), (2, "cooperative, 2 threads per circuit"), (4, "cooperative, 4 threads per circuit")):
                    lb = lckt.batch(nl)
                    for (d, p), v in ldev.items():
                        lb.set_param(d, p, v)
                    lo = T.default_opts(strict_fp=0, coop_parts=parts)
                    ms = min(timed_launches(lambda: lb.run_tran(lcard["tstart"], lcard["tstop"], lcard["tstep"], lcard["tmax"], lcard["uic"],
                                                                out=T.OUT_STATS, opts=lo), reps=2))
                    tot = lb.totals()
                    ent["mappings"].append({"mapping": label, "coop_parts": parts, "ms_per_launch": ms, "steps": int(tot[0]),
                                            "circuit_timesteps_per_sec": int(tot[0]) / (ms * 1e-3), "failed": int((lb.status() != 0).sum())})
                    del lb
                base = ent["mappings"][0]["ms_per_launch"]
                for e in ent["mappings"]:
                    e["speedup_vs_thread_mapping"] = base / e["ms_per_launch"]
                larger_n["workloads"].append(ent)
                del ldev
        except Exception as ex:
            larger_n = {"error": repr(ex)[:300]}

    # ---- operator level: the batched LU behind tsb_lu_solve_batched (drop-in for the reference's matrix operator) -----------------
    operator_lu = None
    if not args.no_configs:
        try:
            operator_lu = measure_lu_operator(T, ctx, timed_launches, dev_name, fp64_peak, budget_bytes=1e9 * min(1.0, args.config_scale))
        except Exception as ex:
            operator_lu = {"error": repr(ex)[:300]}

    # ---- CPU baseline on this box's host cores (rank 0, N = 1 only) ------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        threads = host_threads()
        v, sample, _ = cpu_sample(O, W, 16.0, threads)
        cpu = {"value": v, "unit": "circuit-timesteps/s", "cores": threads, "kind": "port", "sample": sample}

    if rank == 0:
        line = {
            "metric": "circuit-timesteps/sec (batched FP64 transient)", "value": value, "unit": "circuit-timesteps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_job / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": headline_config(n, world, args.strict_fp),
            "accepted_steps_per_step": acc_job, "newton_solves_per_step": solves_job,
            "newton_solves_per_sec": solves_job * args.steps / t_job if t_job > 0 else 0.0,
            "executed_solves_per_step": exec_job,
            "e2e": {"value": e2e_value, "unit": "circuit-timesteps/s", "h2d_bytes_per_step": h2d_bytes * world, "d2h_bytes_per_step": d2h_bytes * world,
                    "pipelined": "two batches per deck: the read-back of step i (tsb_result_fetch_async) and the parameter upload of step i+1 overlap the launches", "results_check": bool(e2e_ok)},
            "gpu_launches": int(launches), "failed_instances": bad_status,
            "clocks": clocks, "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_hbm_stamp": roofline_stamp,
            "configs": configs, "strong": strong, "larger_n": larger_n, "operator_lu": operator_lu, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
