"""Development driver (not a pytest file) for `compute-sanitizer --tool memcheck`, beside gpu_memcheck_driver.py: one small
run of the complex operator-level LU (tsb_k_clu_warp) at each lane width and in both builds, on batches that are not a
multiple of the systems per block, so that out-of-bounds accesses and misaligned shared-memory traffic surface."""
import numpy as np

import parity_util as PU
from test_lu_operator import mna_like

T = PU.T


def main():
    ctx = T.Context(0)
    for n in (1, 5, 8, 9, 16, 17, 32):                  # 4 x 2, 8 x 2 and 32 x 1 lanes x rows
        base, A, b = mna_like(n, 333, n)
        order = T.lu_order(base)
        for strict in (False, True):
            x, st = ctx.lu_solve_batched_complex(A + 1e-4j * A, b + 0.5j * b, order, strict=strict)
            assert np.all(st == 0) and np.all(np.isfinite(x))
    print("complex lu ok", flush=True)


if __name__ == "__main__":
    main()
