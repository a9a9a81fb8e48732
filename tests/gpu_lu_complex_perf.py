"""Development driver (not a pytest file): throughput of the complex batched LU (tsb_lu_solve_batched_complex_dev,
csrc/lu_warp.cu: tsb_k_clu_warp) next to the real one (tsb_lu_solve_batched_dev) on the same systems (imaginary parts
added) and the same number of systems, both builds, device pointers, CUDA events, with the card's name and power limit.
Real and complex runs alternate.  Usage: python tests/gpu_lu_complex_perf.py [bytes_of_complex_A, default 2e9] [n,n,...,
default 8,16,24,32]"""
import subprocess
import sys

import numpy as np
import torch

import parity_util as PU
from gpu_lu_perf import f_lu_dense
from test_lu_operator import mna_like

T = PU.T


def f_clu_dense(n):
    """Dense complex flop count: per step a Smith reciprocal (6 flops + the one division, counted as 7), the U row scaled
    (6 per complex multiply), the trailing update (8 per complex multiply-subtract); forward substitution n multiplies by
    the reciprocal pivot and n (n - 1) / 2 multiply-subtracts, back substitution n (n - 1) / 2 multiply-subtracts."""
    return sum(7 + 6 * (n - k) + 8 * (n - k) ** 2 for k in range(1, n + 1)) + 6 * n + 8 * n * (n - 1)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def main():
    budget = float(sys.argv[1]) if len(sys.argv) > 1 else 2e9
    ns = tuple(int(v) for v in sys.argv[2].split(",")) if len(sys.argv) > 2 else (8, 16, 24, 32)
    ctx = T.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    peak = ctx.measure_fp64_peak()
    print(f"card: {card()}")
    print(f"fp64 peak (tsb_ctx_measure_fp64_peak) {peak:.1f} TFLOP/s")
    for n in ns:
        n_inst = int(min(1 << 24, budget // (n * n * 16)))           # complex A of `budget` bytes; the real run: the same systems
        base, A1, b1 = mna_like(n, 4096, n)
        rng = np.random.default_rng(n)
        Ai = 1e-3 * rng.uniform(-1.0, 1.0, A1.shape) * (A1 != 0)
        order = T.lu_order(base)
        reps = (n_inst + 4095) // 4096
        dA = torch.from_numpy(A1).cuda().repeat(reps, 1, 1)[:n_inst].contiguous()
        db = torch.from_numpy(b1).cuda().repeat(reps, 1)[:n_inst].contiguous()
        dAc = torch.complex(torch.from_numpy(A1), torch.from_numpy(Ai)).cuda().repeat(reps, 1, 1)[:n_inst].contiguous()
        dbc = torch.from_numpy(b1 + 0.5j * b1).cuda().repeat(reps, 1)[:n_inst].contiguous()
        dx, dxc = torch.empty_like(db), torch.empty_like(dbc)
        dst = torch.empty(n_inst, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        runs = {}
        for it in range(5):                                           # real and complex alternate; the first round warms up
            for strict in (0, 1):
                for kind in ("real", "complex"):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    if kind == "real":
                        ctx.lu_solve_batched_dev(n, n_inst, dA.data_ptr(), db.data_ptr(), dx.data_ptr(), dst.data_ptr(), order,
                                                 strict=bool(strict))
                    else:
                        ctx.lu_solve_batched_complex_dev(n, n_inst, dAc.data_ptr(), dbc.data_ptr(), dxc.data_ptr(), dst.data_ptr(),
                                                         order, strict=bool(strict))
                    e1.record(stream)
                    stream.synchronize()
                    assert int(dst.sum()) == 0
                    if it:
                        runs.setdefault((strict, kind), []).append(e0.elapsed_time(e1))
        for strict in (0, 1):
            for kind in ("real", "complex"):
                ms = runs[(strict, kind)]
                t = min(ms) * 1e-3
                w, f = (8, f_lu_dense(n)) if kind == "real" else (16, f_clu_dense(n))
                byts = n_inst * ((n * n + 2 * n) * w + 4)
                print(f"n={n:2d} {kind:7s} strict={strict} inst={n_inst:9d}  {min(ms):8.3f} ms (max {max(ms):8.3f})  "
                      f"{n_inst / t:.3e} systems/s  {byts / t / 1e9:7.1f} GB/s  {n_inst * f / t / 1e12:6.2f} TFLOP/s "
                      f"({100 * n_inst * f / t / 1e12 / peak:4.1f} % of fp64 peak; dense count {f})", flush=True)
        del dA, db, dx, dAc, dbc, dxc, dst
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
