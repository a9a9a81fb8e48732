"""Operator-level drop-in (tsb_lu_order / tsb_lu_solve_batched, csrc/lu_warp.cu): the reference's matrix operator
(pkg/matrix/circuit.go:126-150 Solve = sparse Factor + Solve on the dense structure SetupElements leaves) over a batch,
one circuit per warp.  Checker: the oracle's Sparse 1.3 restatement (orc_lu_batch)."""
import numpy as np
import pytest

import parity_util as PU

T, O = PU.T, PU.O


def mna_like(n, n_inst, seed, zero_diag_rows=2):
    """Synthetic MNA-shaped systems: a diagonally dominant conductance block plus `zero_diag_rows` voltage-source
    style rows / columns (+-1 off the diagonal, 0 on it) so the order cannot be the identity."""
    rng = np.random.default_rng(seed)
    base = rng.uniform(-1e-3, 0.0, (n, n)) * (rng.random((n, n)) < 0.35)
    base = base + base.T
    np.fill_diagonal(base, 0.0)
    np.fill_diagonal(base, -base.sum(axis=1) + 1e-4)
    k = min(zero_diag_rows, n // 3)
    for q in range(k):
        r, c = n - 1 - q, q
        base[r, :] = 0.0; base[:, r] = 0.0
        base[r, c] = 1.0; base[c, r] = 1.0
    scale = np.exp(rng.uniform(np.log(0.5), np.log(2.0), (n_inst, n, n)))
    A = base[None] * scale
    if k:
        for q in range(k):
            r, c = n - 1 - q, q
            A[:, r, c] = 1.0; A[:, c, r] = 1.0
    b = rng.normal(size=(n_inst, n))
    b[:, : max(1, n // 4)] = 0.0          # structural zeros in the right-hand side (spSolve skips them)
    return base, A, b


@pytest.mark.parametrize("n", [3, 8, 13, 32])
def test_symbolic_pass_on_a_dense_matrix_matches_the_oracle(built, n):
    base, A, b = mna_like(n, 1, 100 + n)
    pr, pc = T.lu_order(base)
    _, _, (opr, opc) = O.lu_batch(base, A, b)
    assert sorted(pr) == list(range(1, n + 1)) and sorted(pc) == list(range(1, n + 1))
    assert np.array_equal(pr, opr) and np.array_equal(pc, opc)


def test_order_rejects_singular_and_oversize(built):
    with pytest.raises(T.TsbError):
        T.lu_order(np.zeros((4, 4)))
    with pytest.raises(T.TsbError):
        T.lu_order(np.eye(33))


def test_every_built_mapping_keeps_the_matrix_in_registers(built):
    """The rows a lane owns are C arrays indexed by the (compile-time) elimination step; if the optimiser loses that, the
    whole matrix goes to local memory (R x N x 8 bytes of stack: it happened to the 3- and 4-row mappings under
    `#pragma unroll`, hence static_for).  Checked on the kernels in the built library: a few spilled registers at most."""
    import os
    import re
    import subprocess
    lib = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "toy-spice_b200", "libtspice_b200.so")
    out = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout
    found = re.findall(r"tsb_k_lu_warpILi(\d+)ELi(\d+)ELb([01])ELb([01])ELb([01])\S*:\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    assert len(found) >= 18, len(found)              # 9 lane x row mappings x {strict, fast} at least
    for w, r, strict, bcast, asyn, reg, stack in found:
        matrix_bytes = int(w) * int(r) * int(r) * 8
        assert int(stack) <= 160 and int(stack) < max(matrix_bytes, 161), (w, r, strict, bcast, asyn, reg, stack)
        assert int(reg) <= 170, (w, r, strict, bcast, asyn, reg)     # three 128-thread blocks per SM for the widest mappings


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 5, 8, 10, 16, 21, 32])
def test_strict_build_is_bit_identical_to_sparse13(ctx, n):
    n_inst = 257                                   # not a multiple of the systems-per-block of any lane width
    base, A, b = mna_like(n, n_inst, 7 * n)
    order = T.lu_order(base)
    x, st = ctx.lu_solve_batched(A, b, order, strict=True)
    xo, sto, _ = O.lu_batch(base, A, b)
    assert np.array_equal(st, sto) and np.all(st == 0)
    assert np.array_equal(x, xo), float(np.max(np.abs(x - xo)))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5, 16, 32])
def test_fast_build_within_tolerance_and_zero_pivot_is_data(ctx, n):
    n_inst = 1000
    base, A, b = mna_like(n, n_inst, 11 * n)
    A[17] = 0.0                                    # a singular instance: status 1, never a call failure
    order = T.lu_order(base)
    x, st = ctx.lu_solve_batched(A, b, order, strict=False)
    xo, sto, _ = O.lu_batch(base, A, b)
    assert np.array_equal(st, sto) and st[17] == 1 and st.sum() == 1
    ok = st == 0
    # the fast build re-associates the elimination (multipliers instead of a scaled pivot row), so it is held to the
    # normwise backward error of a stable LU, and to the 1e-9 contract against the oracle where the system is
    # well-conditioned enough for that to be meaningful (forward error <= cond * backward error)
    Aok, xok, bok = A[ok], x[ok], b[ok]
    res = np.einsum("qij,qj->qi", Aok, xok) - bok
    den = np.abs(Aok).sum(axis=2).max(axis=1) * np.abs(xok).max(axis=1) + np.abs(bok).max(axis=1)
    berr = np.abs(res).max(axis=1) / den
    # the frozen (nominal) pivot order costs some instances a few digits in BOTH implementations: compare with the
    # backward error of the oracle's own solution
    berr_o = np.abs(np.einsum("qij,qj->qi", Aok, xo[ok]) - bok).max(axis=1) / den
    assert berr.max() <= 8 * berr_o.max() + 1e-15 and np.median(berr) <= 8 * np.median(berr_o) + 1e-16, \
        (float(berr.max()), float(berr_o.max()), float(np.median(berr)), float(np.median(berr_o)))
    cond = np.linalg.cond(Aok[:64])
    ferr = np.abs(xok[:64] - xo[ok][:64]).max(axis=1) / np.abs(xo[ok][:64]).max(axis=1)
    assert np.all(ferr <= 1e-15 * cond + 1e-13), (float(ferr.max()), float(cond.max()))
    well = cond < 1e5
    assert np.all(ferr[well] <= 1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["1,0,0", "1,0,1", "2,0,0", "2,0,1", "3,0,0", "3,0,1", "4,0,1"])
def test_every_mapping_variant_gives_the_same_answers(ctx, variant, monkeypatch):
    """$TSB_LU_VARIANT = "rows per lane, shared-memory broadcast, asynchronous staging" forces a mapping other than the
    measured default (csrc/lu_warp.cu: launch_lu_warp): the strict build stays bit-identical to Sparse 1.3 whatever the
    mapping, the fast build stays within the backward error of the oracle's own solution."""
    monkeypatch.setenv("TSB_LU_VARIANT", variant)
    for n in (3, 8, 11, 16, 23, 32):
        n_inst = 261
        base, A, b = mna_like(n, n_inst, 13 * n + 1)
        order = T.lu_order(base)
        xo, sto, _ = O.lu_batch(base, A, b)
        x, st = ctx.lu_solve_batched(A, b, order, strict=True)
        assert np.array_equal(st, sto) and np.array_equal(x, xo), (variant, n, float(np.max(np.abs(x - xo))))
        xf, stf = ctx.lu_solve_batched(A, b, order, strict=False)
        assert np.array_equal(stf, sto)
        den = np.abs(A).sum(axis=2).max(axis=1) * np.abs(xf).max(axis=1) + np.abs(b).max(axis=1)
        berr = (np.abs(np.einsum("qij,qj->qi", A, xf) - b).max(axis=1) / den).max()
        berr_o = (np.abs(np.einsum("qij,qj->qi", A, xo) - b).max(axis=1) / den).max()
        assert berr <= 8 * berr_o + 1e-15, (variant, n, float(berr), float(berr_o))


@pytest.mark.gpu
@pytest.mark.parametrize("n,strict", [(8, False), (12, False), (12, True), (32, False)])
def test_every_pass_of_the_grid_stride_loop_computes_alike(ctx, n, strict):
    """More systems than one pass of the resident grid holds (the next system of a lane group is copied into the staging
    tile while the current one is eliminated): copies of the same system give the same bits in every pass, the last,
    ragged one included."""
    reps, m = (300 if n <= 16 else 90), 509        # a pass holds 2 368 blocks x 32 systems (4 lanes each) or x 8 (16 lanes)
    base, A, b = mna_like(n, m, 3 * n)
    order = T.lu_order(base)
    x, st = ctx.lu_solve_batched(np.tile(A, (reps, 1, 1))[: reps * m - 7], np.tile(b, (reps, 1))[: reps * m - 7], order, strict=strict)
    assert np.all(st == 0)
    x0 = x[:m]
    for r in range(1, reps):
        seg = x[r * m:(r + 1) * m]
        assert np.array_equal(seg, x0[: len(seg)]), (r, n)


@pytest.mark.gpu
def test_device_pointer_entry_and_permutation_equivariance(ctx):
    import torch
    n, n_inst = 16, 1 << 16
    base, A, b = mna_like(n, n_inst, 5)
    order = T.lu_order(base)
    dA, db = torch.from_numpy(A).cuda(), torch.from_numpy(b).cuda()
    dx = torch.empty_like(db); dst = torch.empty(n_inst, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.lu_solve_batched_dev(n, n_inst, dA.data_ptr(), db.data_ptr(), dx.data_ptr(), dst.data_ptr(), order, strict=True)
    import importlib
    importlib.import_module("toy-spice_b200")   # noqa
    torch.cuda.synchronize()
    x1 = dx.cpu().numpy()
    perm = np.random.default_rng(1).permutation(n_inst)
    x2, st2 = ctx.lu_solve_batched(A[perm], b[perm], order, strict=True)
    assert np.array_equal(x2, x1[perm]) and np.all(st2 == 0) and int(dst.sum()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rr", "rc", "rlc", "transformer1", "transformer2"])
def test_two_kernel_newton_iteration_equals_the_fused_kernel(ctx, name):
    """Operator-level pipeline: device-stamp kernel (tsb_batch_stamp_dev) -> warp-per-circuit LU (strict, the plan's own
    pivot order) reproduces, bit for bit, the operating point the fused thread-per-circuit analysis kernel computes
    for a linear circuit (its Newton loop solves exactly this system)."""
    import torch
    text = T.BUNDLED[name]
    n_inst = 1000
    ckt = T.Circuit.from_netlist(text, ctx)
    n = ckt.n
    ov = PU.draws(name, ckt, n_inst)
    b = ckt.batch(n_inst)
    for (d, p), v in ov.items():
        b.set_param(d, p, v)
    strict = T.default_opts(strict_fp=1)
    dA = torch.full((n_inst, n, n), float("nan"), dtype=torch.float64, device="cuda")
    db = torch.full((n_inst, n), float("nan"), dtype=torch.float64, device="cuda")
    dx = torch.empty_like(db); dst = torch.empty(n_inst, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    b.stamp_dev(T.AN_OP, 0.0, 0.0, 0.0, dA.data_ptr(), db.data_ptr(), opts=strict)
    st = ckt.structure()
    ctx.lu_solve_batched_dev(n, n_inst, dA.data_ptr(), db.data_ptr(), dx.data_ptr(), dst.data_ptr(), (st["pivot_row"], st["pivot_col"]), strict=True)
    b.sync()
    torch.cuda.synchronize()
    assert not torch.isnan(dA).any() and not torch.isnan(db).any() and int(dst.sum()) == 0
    b.run_op(strict)
    b.sync()
    x_fused = b.wave_all()[0].T                            # OP row: [n columns = x[1..n]][n_inst] -> [n_inst, n]
    assert np.array_equal(dx.cpu().numpy(), x_fused), name


@pytest.mark.gpu
def test_stamp_kernel_transient_companion_models(ctx):
    """rc.cir in transient mode at (t, dt): G + C/dt and the source value, written by the stamp kernel — bit for bit the
    reference's system (tests/stamp_ref.py, whose CPU test holds it to the hand-written companion matrix)."""
    import torch
    import stamp_ref as R
    n_inst = 257
    ckt = T.Circuit.from_netlist(T.BUNDLED["rc"], ctx)
    ov = PU.draws("rc", ckt, n_inst)
    b = ckt.batch(n_inst)
    for (d, p), v in ov.items():
        b.set_param(d, p, v)
    dA = torch.zeros((n_inst, 3, 3), dtype=torch.float64, device="cuda"); db = torch.zeros((n_inst, 3), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    t, dt = 1.25e-4, 2e-7
    b.stamp_dev(T.AN_TRAN, t, dt, 0.0, dA.data_ptr(), db.data_ptr(), opts=T.default_opts(strict_fp=1))
    b.sync(); torch.cuda.synchronize()
    A, rhs = dA.cpu().numpy(), db.cpu().numpy()
    ref = R.stamp_batch(R.Deck(T.BUNDLED["rc"]), ov, range(n_inst), R.TRAN, t, dt, 0.0)
    assert np.array_equal(A.view(np.int64), ref.A.view(np.int64))
    assert np.array_equal(rhs.view(np.int64), ref.b.view(np.int64))
