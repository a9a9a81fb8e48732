"""Batched LU operator (tsb_lu_solve_batched[_dev], csrc/lu_warp.cu) at the edges: every order n = 1..32 under every lane x
row mapping, caller-chosen pivot orders, exact references, zero / infinite / NaN pivots and entries, batch sizes at the
group and resident-pass edges, 8-byte aligned device pointers, which kernel the dispatcher launches, and the refusals.

References:
* exact-integer systems (`exact_systems`): A = P^T (L U) Q^T with small integer L, U (diagonal of U a power of two) and
  integer x.  Every operation of both builds is exact on them (scaled U rows, multipliers, reciprocals of powers of two),
  so x must come back exactly whatever the order, the mapping or the build.  No oracle needed: they check the row and
  column scatter of staging, elimination and write-back for any pivot order and at batch sizes no oracle run could cover.
* the oracle's Sparse 1.3 restatement (orc_lu_batch) for the strict build, bit for bit, signed zeros included.
* a correctly rounded residual (`residual_exact`: Dekker products summed with math.fsum) for the fast build, held to the
  normwise backward-error bound of LU in the frozen order, gamma(3n + 4) * growth, with the growth factor
  || |L||U| || / ||A|| of that elimination computed here.

What is not specified and therefore not tested: x of a status-1 system (zero pivot).  The oracle writes 0 there; the
kernel leaves whatever the elimination produced (Inf / NaN from the reciprocal of the zero pivot).
"""
import ctypes as C
import math
import re
from fractions import Fraction

import numpy as np
import pytest

import parity_util as PU
from test_lu_operator import mna_like

T, O = PU.T, PU.O
U_RND = 2.0 ** -53

# (W, R): lanes per system x rows per lane; the forced rows per lane that reaches the mapping, an order n it serves (several
# with identity padding up to W R), and whether the strict build has it (4 rows per lane above n = 8: fast build only).
MAPPINGS = [((8, 1), 1, 7, True), ((16, 1), 1, 16, True), ((32, 1), 1, 29, True), ((4, 2), 2, 8, True), ((8, 2), 2, 13, True),
            ((16, 2), 2, 32, True), ((4, 3), 3, 11, True), ((8, 3), 3, 24, True), ((2, 4), 4, 6, True), ((4, 4), 4, 16, False)]
MAPPING_CASES = [pytest.param(wr, r, n, strict, id=f"{wr[0]}x{wr[1]}-{'strict' if strict else 'fast'}")
                 for wr, r, n, has_strict in MAPPINGS for strict in (True, False) if has_strict or not strict]
VARIANTS = [f"{r},0,{a}" for r in (1, 2, 3, 4) for a in (0, 1)]     # $TSB_LU_VARIANT: rows per lane, no broadcast, staging


# ---- generators -----------------------------------------------------------------------------------------------------
def exact_systems(n, n_inst, seed, order=None, zero_step=None):
    """Exact-integer systems in a pivot order: L unit lower triangular with off-diagonal entries in {-1, 0, 1}; U upper
    triangular, diagonal in {+-1, +-2, +-4}, off-diagonal integers in [-2, 2] at ~30 % fill; x integers in [-8, 8];
    A[prow[i], pcol[j]] = (L U)[i, j], b = A x (exact in int64).  `order` = (prow, pcol) 1-based as tsb_lu_order returns it
    (random permutations if None).  zero_step = k: U_kk = 0, i.e. an exact zero pivot at step k of that order (a scalar for
    every system, or an array of one step per system).  Returns A, b, x (float64) and the 1-based order."""
    rng = np.random.default_rng(seed)
    if order is None:
        prow, pcol = rng.permutation(n), rng.permutation(n)
    else:
        prow, pcol = np.asarray(order[0]) - 1, np.asarray(order[1]) - 1
    L = np.tril(rng.integers(-1, 2, (n_inst, n, n)), -1) + np.eye(n, dtype=np.int64)
    U = np.triu(rng.integers(-2, 3, (n_inst, n, n)) * (rng.random((n_inst, n, n)) < 0.3), 1)
    U[:, np.arange(n), np.arange(n)] = rng.choice([-4, -2, -1, 1, 2, 4], (n_inst, n))
    if zero_step is not None:
        U[np.arange(n_inst), np.broadcast_to(zero_step, (n_inst,)), np.broadcast_to(zero_step, (n_inst,))] = 0
    x = rng.integers(-8, 9, (n_inst, n))
    A = np.empty((n_inst, n, n), dtype=np.int64)
    A[:, prow[:, None], pcol[None, :]] = L @ U
    b = np.einsum("qij,qj->qi", A, x)
    return A.astype(np.float64), b.astype(np.float64), x.astype(np.float64), (prow + 1, pcol + 1)


def graded_mna(n, n_inst, seed):
    """MNA-like systems with strongly graded entries: a connected conductance network (a chain plus random branches, and
    branches to ground) with conductances log-uniform in 1e-12 .. 1e3 S, and up to two voltage sources (+-1 incidence rows
    and columns, zero diagonal).  Every instance scales each conductance by a factor in [0.5, 2] (one circuit, swept).
    Returns the nominal matrix, A and b."""
    rng = np.random.default_rng(seed)
    n_src = min(2, n // 3)
    nodes = n - n_src
    branches = [(i, i + 1) for i in range(nodes - 1)]
    branches += [tuple(sorted(rng.choice(nodes, 2, replace=False))) for _ in range(nodes // 2)] if nodes > 1 else []
    branches += [(i, -1) for i in rng.choice(nodes, max(1, nodes // 4), replace=False)]     # to ground
    g_nom = 10.0 ** (rng.permutation(np.linspace(-12.0, 3.0, len(branches))) + rng.uniform(-0.5, 0.5, len(branches)))
    g_nom = np.clip(g_nom, 1e-12, 1e3)

    def stamp(g):
        A = np.zeros(g.shape[:1] + (n, n))
        for (i, j), gq in zip(branches, g.T):
            A[:, i, i] += gq
            if j >= 0:
                A[:, j, j] += gq
                A[:, i, j] -= gq
                A[:, j, i] -= gq
        for q in range(n_src):              # source q between node 2q + 1 (or q) and ground / node 0
            v, a = nodes + q, min(2 * q + 1, nodes - 1)
            A[:, v, a] = A[:, a, v] = 1.0
            if q == 1 and a != 0:
                A[:, v, 0] = A[:, 0, v] = -1.0
        return A

    base = stamp(g_nom[None])[0]
    A = stamp(g_nom[None] * np.exp(rng.uniform(np.log(0.5), np.log(2.0), (n_inst, len(branches)))))
    b = rng.normal(size=(n_inst, n)) * np.exp(rng.uniform(np.log(1e-6), np.log(1e2), (n_inst, n)))
    return base, A, b


# ---- CPU references -------------------------------------------------------------------------------------------------
def sparse13_solve(A, b, order):
    """Sparse 1.3's arithmetic in a frozen pivot order, float64, batched (the strict build's operation order): U rows scaled
    by the reciprocal pivot, L unscaled, zero right-hand-side entries skipped in the forward substitution, back
    substitution row by row with ascending columns; entries loaded as AddElement onto +0 loads them (-0.0 -> +0.0).
    Returns x and the largest magnitude of any intermediate."""
    prow, pcol = np.asarray(order[0]) - 1, np.asarray(order[1]) - 1
    n = len(prow)
    P = A[:, prow][:, :, pcol] + 0.0
    c = b[:, prow].copy()
    big = max(np.abs(P).max(initial=0.0), np.abs(c).max(initial=0.0))
    with np.errstate(all="ignore"):
        for k in range(n):
            P[:, k, k] = 1.0 / P[:, k, k]
            P[:, k, k + 1:] *= P[:, k, k, None]
            P[:, k + 1:, k + 1:] = P[:, k + 1:, k + 1:] - P[:, k + 1:, k, None] * P[:, None, k, k + 1:]
            big = max(big, np.abs(P[:, k:, k + 1:]).max(initial=0.0))
        for k in range(n):
            nz = c[:, k] != 0.0
            c[:, k] = np.where(nz, c[:, k] * P[:, k, k], c[:, k])
            c[:, k + 1:] = np.where(nz[:, None], c[:, k + 1:] - c[:, k, None] * P[:, k + 1:, k], c[:, k + 1:])
            big = max(big, np.abs(c).max())
        for i in range(n - 2, -1, -1):
            for j in range(i + 1, n):
                c[:, i] = c[:, i] - P[:, i, j] * c[:, j]
            big = max(big, np.abs(c[:, i]).max())
    x = np.empty_like(c)
    x[:, pcol] = c
    return x, big


def frozen_lu(A, order):
    """Doolittle LU of P A Q in the given order (no pivoting), float64, batched: L unit lower (multipliers), U unscaled."""
    prow, pcol = np.asarray(order[0]) - 1, np.asarray(order[1]) - 1
    n = len(prow)
    P = A[:, prow][:, :, pcol].copy()
    Lm = np.zeros_like(P)
    Lm[:, np.arange(n), np.arange(n)] = 1.0
    for k in range(n):
        m = P[:, k + 1:, k] * (1.0 / P[:, k, k, None])
        Lm[:, k + 1:, k] = m
        P[:, k + 1:, k:] -= m[:, :, None] * P[:, None, k, k:]
    return Lm, np.triu(P)


def abs_lu(A, order):
    """|L||U| of the frozen-order elimination, in EXTERNAL row / column numbering (so that |L||U| |x| lines up with A x)."""
    prow, pcol = np.asarray(order[0]) - 1, np.asarray(order[1]) - 1
    Lm, Um = frozen_lu(A, order)
    out = np.empty_like(A)
    out[:, prow[:, None], pcol[None, :]] = np.abs(Lm) @ np.abs(Um)
    return out


def growth(A, order):
    """|| |L||U| ||_inf / ||A||_inf of the frozen-order elimination, per system."""
    return abs_lu(A, order).sum(axis=2).max(axis=1) / np.abs(A).sum(axis=2).max(axis=1)


def _split(a):
    c = 134217729.0 * a                    # Veltkamp: 2^27 + 1
    hi = c - (c - a)
    return hi, a - hi


def residual_exact(A, x, b):
    """b - A x, correctly rounded per component: every product a_ij x_j as an exact pair p + e (Dekker), all summed with
    math.fsum.  (Products must stay inside ~2^-969 .. 2^996 in magnitude for the pairs to be exact.)"""
    p = A * x[:, None, :]
    ah, al = _split(A)
    xh, xl = _split(np.broadcast_to(x[:, None, :], A.shape))
    e = ((ah * xh - p) + ah * xl + al * xh) + al * xl
    terms = np.concatenate([b[:, :, None], -p, -e], axis=2).reshape(-1, 2 * A.shape[2] + 1)
    return np.array([math.fsum(t) for t in terms.tolist()]).reshape(b.shape)


def gamma(m):
    return m * U_RND / (1.0 - m * U_RND)


def fast_backward_error_bound(A, order):
    """Backward-error bound of the fast build's solve.  LU in a fixed order with the standard rounding model gives
    (A + dA) x = b with |dA| <= gamma(3n) |L||U| (Higham, Accuracy and Stability of Numerical Algorithms, Thm. 9.4); the fast
    build takes reciprocal pivots (seed + cubic step, within 2 u) and multiplies by them, for the multipliers and in the
    back substitution, which adds at most 4 more roundings: gamma(3n + 4).  Returns (gamma(3n + 4) |L||U| for the
    componentwise bound |b - A x| <= gamma(3n + 4) |L||U| |x|, and the normwise bound
    ||b - A x||_inf / (||A||_inf ||x||_inf) <= gamma(3n + 4) * growth per system)."""
    g = gamma(3 * A.shape[1] + 4)
    lu = abs_lu(A, order)
    return g * lu, g * lu.sum(axis=2).max(axis=1) / np.abs(A).sum(axis=2).max(axis=1)


def expected_mapping(n, strict, rows=None):
    """(W, R) that launch_lu_warp runs for order n; rows = the rows per lane $TSB_LU_VARIANT forces (None: the default)."""
    if rows is None:
        return (4, 2) if n <= 8 else (4, 3) if n <= 12 else (8, 2) if n <= 16 else (8, 3) if n <= 24 else (16, 2)
    if rows == 3:
        return (4, 3) if n <= 12 else (8, 3) if n <= 24 else (16, 2)
    if rows == 4 and (n <= 8 or (n <= 16 and not strict)):
        return (2, 4) if n <= 8 else (4, 4)
    if rows == 4:
        rows = 2                           # 4 rows per lane do not fit the registers there: 2 rows per lane
    w = {1: (8, 16, 32), 2: (4, 8, 16)}[rows][0 if n <= 8 else 1 if n <= 16 else 2]
    return (w, rows)


def bits(v):
    return np.ascontiguousarray(v, dtype=np.float64).view(np.int64)


# ---- CPU tests ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", range(1, 33))
def test_exact_systems_solve_exactly_in_sparse13_order(n):
    """The generator's promise, checked in float64 with Sparse 1.3's operation order and with the multiplier form of the
    fast build: x comes back exactly in a random order, every intermediate is small (no rounding anywhere)."""
    A, b, x, order = exact_systems(n, 50, 1000 + n)
    assert np.array_equal(np.einsum("qij,qj->qi", A, x), b)
    xs, big = sparse13_solve(A, b, order)
    assert np.array_equal(xs, x) and big <= 2.0 ** 12, (n, big)
    Lm, Um = frozen_lu(A, order)
    prow, pcol = order[0] - 1, order[1] - 1
    assert np.all(Lm == np.round(Lm)) and np.all(Um == np.round(Um)) and np.abs(Um).max() <= 2.0 ** 12
    assert np.array_equal(Lm @ Um, A[:, prow][:, :, pcol])


@pytest.mark.parametrize("n", [1, 2, 5, 9, 16, 25, 32])
def test_sparse13_restatement_matches_the_oracle(built, n):
    """sparse13_solve is the oracle's Sparse 1.3 bit for bit in the oracle's own frozen order, signed zeros included, also
    with infinite pivots (mna_like has -0.0 entries: the oracle loads them as +0.0, which decides the sign of the zero
    that an infinite pivot leaves in x)."""
    base, A, b = mna_like(n, 40, 500 + n)
    assert n < 3 or np.signbit(A[A == 0]).any()
    xo, sto, opo = O.lu_batch(base, A, b)
    xs, _ = sparse13_solve(A, b, opo)
    assert np.all(sto == 0) and np.array_equal(bits(xs), bits(xo))
    ks = np.arange(len(A)) % n
    A[np.arange(len(A)), opo[0][ks] - 1, opo[1][ks] - 1] = np.inf
    xo, sto, _ = O.lu_batch(base, A, b)
    xs, _ = sparse13_solve(A, b, opo)
    ok = sto == 0
    assert np.array_equal(bits(xs[ok]), bits(xo[ok]))


def test_residual_helper_is_correctly_rounded():
    """residual_exact against exact rational arithmetic, on residuals that cancel to the last bits (b = fl(A x)) and on
    entries spread over 30 orders of magnitude."""
    rng = np.random.default_rng(3)
    n, q = 12, 30
    A = rng.normal(size=(q, n, n)) * np.exp(rng.uniform(-35, 35, (q, n, n)))
    x = rng.normal(size=(q, n)) * np.exp(rng.uniform(-10, 10, (q, n)))
    b = np.einsum("qij,qj->qi", A, x)
    b[::2] = rng.normal(size=b[::2].shape)
    r = residual_exact(A, x, b)
    for s in range(q):
        for i in range(n):
            exact = Fraction(b[s, i]) - sum(Fraction(A[s, i, j]) * Fraction(x[s, j]) for j in range(n))
            assert r[s, i] == float(exact), (s, i, r[s, i], float(exact))


@pytest.mark.parametrize("n", [1, 2, 3, 8, 13, 24, 32])
def test_oracle_reports_the_constructed_zero_pivots(built, n):
    """The singular systems of the GPU zero-pivot test: an exact zero at step k of the oracle's frozen order.  The oracle
    (Sparse 1.3 re-factorisation in that order) reports status 1 on exactly those, 0 on the regular ones."""
    base, _, _ = mna_like(n, 1, 40 + n)
    order = T.lu_order(base)
    steps = np.array([0, n // 2, n - 1, 0, n // 2, n - 1])
    As, bs, _, _ = exact_systems(n, len(steps), 7 * n, order=order, zero_step=steps)
    Ar, br, _, _ = exact_systems(n, 4, 7 * n + 1, order=order)
    _, st, opo = O.lu_batch(base, np.concatenate([As, Ar]), np.concatenate([bs, br]))
    assert np.array_equal(opo[0], order[0]) and np.array_equal(opo[1], order[1])
    assert st.tolist() == [1] * len(steps) + [0] * 4


def test_graded_systems_are_graded_and_regular(built):
    for n in (12, 20, 32):
        base, A, b = graded_mna(n, 8, n)
        nz = np.abs(base[base != 0])
        assert nz.max() / nz.min() > 1e10
        order = T.lu_order(base)
        assert np.all(np.isfinite(growth(A, order)))


def test_expected_mapping_table():
    """The default column of DESIGN §5.2b's table, and the ten mappings the forced variants reach."""
    assert [expected_mapping(n, s) for s in (True, False) for n in (1, 8, 9, 12, 13, 16, 17, 24, 25, 32)] == 2 * [
        (4, 2), (4, 2), (4, 3), (4, 3), (8, 2), (8, 2), (8, 3), (8, 3), (16, 2), (16, 2)]
    reached = {expected_mapping(n, s, r) for n in range(1, 33) for s in (True, False) for r in (1, 2, 3, 4)}
    assert reached == {wr for wr, _, _, _ in MAPPINGS}
    for wr, r, n, has_strict in MAPPINGS:
        assert expected_mapping(n, False, r) == wr and (expected_mapping(n, True, r) == wr) == has_strict


# ---- GPU tests ------------------------------------------------------------------------------------------------------
@pytest.fixture
def variant(monkeypatch):
    """Sets $TSB_LU_VARIANT for the calls of one test (read by the library at every call); None restores the default."""
    def set_(v):
        if v is None:
            monkeypatch.delenv("TSB_LU_VARIANT", raising=False)
        else:
            monkeypatch.setenv("TSB_LU_VARIANT", v)
    set_(None)
    return set_


def pass_size(ctx, wr):
    """Systems of one pass of the resident grid: SMs x 16 blocks x 128 / W systems per block."""
    return ctx.sm_count * 16 * (128 // wr[0])


def tiled_exact(n, n_inst, seed, order, pool=509):
    """n_inst exact systems in `order`: `pool` distinct ones repeated (large batches without large generation cost)."""
    A, b, x, _ = exact_systems(n, pool, seed, order=order)
    idx = np.arange(n_inst) % pool
    return A[idx], b[idx], x[idx]


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
@pytest.mark.parametrize("var", VARIANTS)
def test_exact_systems_in_a_random_order_every_n_and_mapping(ctx, variant, var, strict):
    """Caller-chosen random pivot orders, every n = 1..32 under every forced mapping and staging: x exact in both builds."""
    variant(var)
    for n in range(1, 33):
        A, b, x, order = exact_systems(n, 131, 17 * n + 3)
        xk, st = ctx.lu_solve_batched(A, b, order, strict=strict)
        assert np.all(st == 0), (var, n)
        assert np.array_equal(xk, x), (var, n, int(np.sum(xk != x)), np.argwhere(xk != x)[:3].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("var", VARIANTS)
def test_strict_build_bit_identical_to_sparse13_every_n_and_mapping(ctx, variant, var):
    """The strict build against the oracle for every n = 1..32 under every forced mapping and staging, in the order of
    tsb_lu_order: the same bits, signs of zeros included (np.array_equal alone takes -0.0 == 0.0)."""
    variant(var)
    for n in range(1, 33):
        base, A, b = mna_like(n, 67, 29 * n + 5)
        order = T.lu_order(base)
        xo, sto, _ = O.lu_batch(base, A, b)
        x, st = ctx.lu_solve_batched(A, b, order, strict=True)
        assert np.array_equal(st, sto) and np.all(st == 0), (var, n)
        assert np.array_equal(x, xo) and np.array_equal(np.signbit(x), np.signbit(xo)), (var, n, float(np.max(np.abs(x - xo))))


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
def test_power_of_two_scaling_is_equivariant(ctx, variant, strict):
    """(D1 A D2, D1 b) with diagonal D1, D2 of powers of two (2^-200 .. 2^200) gives D2^-1 x bit for bit: every rounding
    commutes with an exact scaling inside the normal range.  That holds for the IEEE arithmetic of the strict build and
    for the fast build too, whose reciprocal seed depends on the significand alone (scaled pivots give scaled seeds)."""
    rng = np.random.default_rng(23)
    for n in range(1, 33):
        base, A, b = mna_like(n, 129, 31 * n)
        order = T.lu_order(base)
        e1 = rng.integers(-200, 201, (len(A), n))
        e2 = rng.integers(-200, 201, (len(A), n))
        As = np.ldexp(np.ldexp(A, e1[:, :, None]), e2[:, None, :])
        bs = np.ldexp(b, e1)
        x, st = ctx.lu_solve_batched(A, b, order, strict=strict)
        xs, sts = ctx.lu_solve_batched(As, bs, order, strict=strict)
        assert np.all(st == 0) and np.all(sts == 0)
        assert np.array_equal(bits(xs), bits(np.ldexp(x, -e2))), (n, strict)


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["mna_like", "graded"])
def test_fast_build_backward_error_within_the_lu_bound(ctx, variant, family):
    """Fast build: the correctly rounded residual is within the backward-error bounds of LU in the frozen order
    (fast_backward_error_bound), componentwise |b - A x| <= gamma(3n + 4) |L||U| |x| and normwise
    ||b - A x||_inf <= gamma(3n + 4) * growth * ||A||_inf ||x||_inf, per system.  (The frozen order costs mna_like systems
    a growth factor up to ~1e6; the componentwise bound is the sharp one there.)"""
    for n in (2, 4, 7, 8, 12, 16, 20, 24, 32):
        base, A, b = (mna_like(n, 300, 41 * n) if family == "mna_like" else graded_mna(n, 300, 43 * n))
        order = T.lu_order(base)
        x, st = ctx.lu_solve_batched(A, b, order, strict=False)
        assert np.all(st == 0) and np.all(np.isfinite(x)), n
        r = np.abs(residual_exact(A, x, b))
        comp, norm = fast_backward_error_bound(A, order)
        cbound = np.einsum("qij,qj->qi", comp, np.abs(x))
        worst = np.unravel_index(np.argmax(r - cbound), r.shape)
        assert np.all(r <= cbound), (family, n, worst, float(r[worst]), float(cbound[worst]))
        berr = r.max(axis=1) / (np.abs(A).sum(axis=2).max(axis=1) * np.abs(x).max(axis=1))
        worst = int(np.argmax(berr / norm))
        assert np.all(berr <= norm), (family, n, worst, float(berr[worst]), float(norm[worst]))


@pytest.mark.gpu
@pytest.mark.parametrize("wr,rows,n,strict", MAPPING_CASES)
def test_zero_pivots_are_isolated_in_their_lane_group(ctx, variant, wr, rows, n, strict):
    """Singular systems (an exact zero pivot at some step of the order) at every group slot of a warp and at the first and
    last instance of a resident pass, over more than one pass: status 1 on exactly those, and every other system has the
    same bits as in a run where the singular ones are replaced by regular ones (the per-group `ok` flag, and the tile of
    the next system that is staged while a singular one is eliminated).  x of a singular system is unspecified."""
    variant(f"{rows},0,1")
    groups = 128 // wr[0]
    per_warp = 32 // wr[0]
    ps = pass_size(ctx, wr)
    n_inst = ps + 2 * groups + 3
    rng = np.random.default_rng(n)
    order = (rng.permutation(n) + 1, rng.permutation(n) + 1)
    A, b, x = tiled_exact(n, n_inst, 61 * n, order)
    sing = sorted({g * (per_warp + 1) for g in range(per_warp)} | {ps - 1, ps, n_inst - 1})
    As, bs, _, _ = exact_systems(n, len(sing), 67 * n, order=order, zero_step=rng.integers(0, n, len(sing)))
    A2, b2 = A.copy(), b.copy()
    A2[sing], b2[sing] = As, bs
    x1, st1 = ctx.lu_solve_batched(A, b, order, strict=strict)
    x2, st2 = ctx.lu_solve_batched(A2, b2, order, strict=strict)
    assert np.all(st1 == 0) and np.array_equal(x1, x)
    expect = np.zeros(n_inst, dtype=np.int32)
    expect[sing] = 1
    assert np.array_equal(st2, expect), np.flatnonzero(st2 != expect)[:8].tolist()
    keep = expect == 0
    assert np.array_equal(bits(x2[keep]), bits(x1[keep]))


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
@pytest.mark.parametrize("var", [None, "1,0,1", "2,0,0", "3,0,0", "4,0,1"])
def test_infinite_pivot_gives_zero_for_its_column(ctx, variant, var, strict):
    """+Inf on the internal diagonal at step k of the frozen order (k varies over the batch): the reciprocal pivot is 0,
    x[pcol[k]] = 0 and everything else finite, as Sparse 1.3 computes it (strict build: its bits).  On diagonally dominant
    systems the status is 0; on MNA-like ones an infinite pivot can leave a later pivot exactly 0 (a voltage-source row
    whose only coupling went through row k): status 1 there, as in the oracle."""
    variant(var)
    for n in (1, 2, 5, 8, 11, 16, 21, 32):
        for zero_diag_rows in (0, 2):
            base, A, b = mna_like(n, 97, 37 * n, zero_diag_rows=zero_diag_rows)
            order = T.lu_order(base)
            ks = np.arange(len(A)) % n
            A[np.arange(len(A)), order[0][ks] - 1, order[1][ks] - 1] = np.inf
            xo, sto, _ = O.lu_batch(base, A, b)
            x, st = ctx.lu_solve_batched(A, b, order, strict=strict)
            ok = sto == 0
            assert ok.sum() >= len(A) // 2 and (zero_diag_rows or ok.all()), (n, zero_diag_rows, int(ok.sum()))
            assert np.all(np.isfinite(xo[ok])) and np.all(xo[ok, order[1][ks[ok]] - 1] == 0.0)
            assert np.array_equal(st, sto), (var, n, zero_diag_rows)
            if strict:
                assert np.array_equal(bits(x[ok]), bits(xo[ok])), (var, n, zero_diag_rows)
            else:
                bad = ~np.isfinite(x[ok])
                assert not bad.any(), (var, n, zero_diag_rows, int(bad.sum()), np.flatnonzero(bad.any(axis=1))[:5].tolist())
                assert np.all(x[ok, order[1][ks[ok]] - 1] == 0.0), (var, n, zero_diag_rows)


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
def test_nan_entries_and_infinite_right_hand_sides(ctx, variant, strict):
    """NaN at a random entry of A (every third system) and +-Inf at a random entry of b (every third, shifted by one):
    status as the oracle's; the strict build has the oracle's bits (NaN where the oracle has NaN, the same values
    elsewhere); the fast build is non-finite at least where the oracle is.  Not exactly there: it does not skip zero
    right-hand-side entries in the forward substitution as spSolve does, so NaN x 0 spreads further."""
    rng = np.random.default_rng(5)
    for n in (1, 3, 8, 12, 17, 32):
        base, A, b = mna_like(n, 150, 47 * n)
        order = T.lu_order(base)
        qa, qb = np.arange(0, len(A), 3), np.arange(1, len(A), 3)
        A[qa, rng.integers(0, n, len(qa)), rng.integers(0, n, len(qa))] = np.nan
        b[qb, rng.integers(0, n, len(qb))] = np.where(rng.random(len(qb)) < 0.5, np.inf, -np.inf)
        xo, sto, _ = O.lu_batch(base, A, b)
        x, st = ctx.lu_solve_batched(A, b, order, strict=strict)
        assert np.array_equal(st, sto), n
        if strict:
            assert np.array_equal(np.isnan(x), np.isnan(xo)), n
            assert np.array_equal(x, xo, equal_nan=True), n
        else:
            assert np.all(~np.isfinite(x) | np.isfinite(xo)), n


@pytest.mark.gpu
@pytest.mark.parametrize("wr,rows,n,strict", MAPPING_CASES)
def test_batch_sizes_at_the_group_and_pass_edges(ctx, variant, wr, rows, n, strict):
    """n_inst = 1, one block's systems -+ 1, exactly one resident pass and one more, with both stagings: exact x."""
    groups = 128 // wr[0]
    ps = pass_size(ctx, wr)
    rng = np.random.default_rng(100 + n)
    order = (rng.permutation(n) + 1, rng.permutation(n) + 1)
    A, b, x = tiled_exact(n, ps + 1, 71 * n, order)
    for staging in (0, 1):
        variant(f"{rows},0,{staging}")
        for m in (1, groups - 1, groups + 1, ps, ps + 1):
            xk, st = ctx.lu_solve_batched(A[:m], b[:m], order, strict=strict)
            assert np.all(st == 0) and np.array_equal(xk, x[:m]), (staging, m, int(np.sum(xk != x[:m])))


@pytest.mark.gpu
@pytest.mark.parametrize("wr,rows,n,strict", MAPPING_CASES)
def test_device_pointers_aligned_to_8_bytes_only(ctx, variant, wr, rows, n, strict):
    """lu_solve_batched_dev on buffers that start one element into their allocation (A, b, x 8-byte but not 16-byte
    aligned, status 4-byte): the same bits and status as from aligned buffers."""
    import torch
    variant(f"{rows},0,1")
    n_inst = 3 * (128 // wr[0]) + 5
    base, A, b = mna_like(n, n_inst, 53 * n)
    order = T.lu_order(base)
    out = []
    for off in (0, 1):
        fa = torch.zeros(n_inst * n * n + 2, dtype=torch.float64, device="cuda")
        fb = torch.zeros(n_inst * n + 2, dtype=torch.float64, device="cuda")
        fx = torch.full((n_inst * n + 2,), float("nan"), dtype=torch.float64, device="cuda")
        fs = torch.full((n_inst + 2,), -1, dtype=torch.int32, device="cuda")
        dA, db = fa[off:off + n_inst * n * n], fb[off:off + n_inst * n]
        dx, ds = fx[off:off + n_inst * n], fs[off:off + n_inst]
        dA.copy_(torch.from_numpy(A.reshape(-1)))
        db.copy_(torch.from_numpy(b.reshape(-1)))
        assert [p.data_ptr() % 16 for p in (dA, db, dx)] == [8 * off] * 3
        ctx.lu_solve_batched_dev(n, n_inst, dA.data_ptr(), db.data_ptr(), dx.data_ptr(), ds.data_ptr(), order, strict=strict)
        torch.cuda.synchronize()
        assert torch.isnan(fx[:off]).all() and torch.isnan(fx[off + n_inst * n:]).all() and int(fs[off + n_inst:][0]) == -1
        out.append((dx.cpu().numpy().reshape(n_inst, n), ds.cpu().numpy()))
    (x0, s0), (x1, s1) = out
    assert np.all(s0 == 0) and np.array_equal(s1, s0) and np.array_equal(bits(x1), bits(x0))


_KNAME = [re.compile(r"tsb_k_lu_warp<(\d+), ?(\d+), ?(true|false), ?(true|false), ?(true|false)>"),
          re.compile(r"tsb_k_lu_warpILi(\d+)ELi(\d+)ELb([01])ELb([01])ELb([01])E")]


def launched_lu_kernels(calls):
    """Runs `calls` under torch.profiler (CUDA activities) and returns, in launch order, (W, R, STRICT, BCAST, ASYNC) of every
    tsb_k_lu_warp kernel that ran."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.zeros(1, device="cuda")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for f in calls:
            f()
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if "tsb_k_lu_warp" in e.name), key=lambda e: e.time_range.start)
    assert evs, ("torch.profiler recorded no tsb_k_lu_warp kernel (CUDA activity tracing unavailable?): the dispatch "
                 "cannot be checked")
    out = []
    for e in evs:
        m = _KNAME[0].search(e.name) or _KNAME[1].search(e.name)
        assert m, e.name
        w, r, s, bc, a = m.groups()
        out.append((int(w), int(r), *(v in ("true", "1") for v in (s, bc, a))))
    return out


def _dispatch_calls(ctx, variant, cases):
    def call(n, strict, var):
        def f():
            variant(var)
            A, b, _, order = exact_systems(n, 1, n)
            x, st = ctx.lu_solve_batched(A, b, order, strict=strict)
            assert st[0] == 0
        return f
    return [call(n, s, v) for n, s, v in cases]


@pytest.mark.gpu
def test_default_dispatch_follows_the_design_table(ctx, variant):
    """n <= 8: 4 lanes x 2 rows, <= 12: 4 x 3, <= 16: 8 x 2, <= 24: 8 x 3, <= 32: 16 x 2; asynchronous staging, shuffles,
    in both builds (DESIGN §5.2b, launch_lu_warp)."""
    cases = [(n, s, None) for s in (True, False) for n in range(1, 33)]
    got = launched_lu_kernels(_dispatch_calls(ctx, variant, cases))
    want = [(*expected_mapping(n, s), s, False, True) for n, s, _ in cases]
    assert len(got) == len(want)
    bad = [(c, g, w) for c, g, w in zip(cases, got, want) if g != w]
    assert not bad, bad[:6]
    table = {(1, 8): (4, 2), (9, 12): (4, 3), (13, 16): (8, 2), (17, 24): (8, 3), (25, 32): (16, 2)}
    assert all(g[:2] == table[next(k for k in table if k[0] <= c[0] <= k[1])] for c, g in zip(cases, got))


@pytest.mark.gpu
def test_forced_variants_and_their_fallbacks(ctx, variant):
    """$TSB_LU_VARIANT = "R,0,A" runs R rows per lane with the staging A where those rows fit the register file, and falls
    back to 2 rows per lane where they do not (4 rows: above n = 16, and above n = 8 in the strict build; 3 rows: above
    n = 24)."""
    cases = [(n, s, f"{r},0,{a}") for r in (1, 2, 3, 4) for a in (0, 1) for s in (True, False) for n in range(1, 33)]
    got = launched_lu_kernels(_dispatch_calls(ctx, variant, cases))
    want = [(*expected_mapping(n, s, int(v[0])), s, False, v.endswith("1")) for n, s, v in cases]
    assert len(got) == len(want)
    bad = [(c, g, w) for c, g, w in zip(cases, got, want) if g != w]
    assert not bad, bad[:6]
    assert got[cases.index((9, True, "4,0,1"))][:2] == (8, 2) and got[cases.index((17, True, "4,0,1"))][:2] == (16, 2)
    assert got[cases.index((9, False, "4,0,1"))][:2] == (4, 4) and got[cases.index((25, False, "3,0,0"))][:2] == (16, 2)


def _raw_solve(ctx, n, prow, pcol, n_inst, A=None, b=None):
    """tsb_lu_solve_batched through the C ABI, returning the raw code; x / status prefilled with sentinels to see writes."""
    L = T.lib()
    nn = max(n, 1)
    A = np.ones((max(n_inst, 1), nn, nn)) if A is None else A
    b = np.ones((max(n_inst, 1), nn)) if b is None else b
    x = np.full(b.shape, -7.0)
    st = np.full(max(n_inst, 1), -7, dtype=np.int32)
    pr = np.ascontiguousarray(prow, dtype=np.int32)
    pc = np.ascontiguousarray(pcol, dtype=np.int32)
    ip, dp = C.POINTER(C.c_int), C.POINTER(C.c_double)
    rc = L.tsb_lu_solve_batched(ctx.h, n, pr.ctypes.data_as(ip), pc.ctypes.data_as(ip), A.ctypes.data_as(dp),
                                b.ctypes.data_as(dp), x.ctypes.data_as(dp), st.ctypes.data_as(C.POINTER(C.c_int32)), n_inst, 1)
    return rc, x, st


@pytest.mark.gpu
def test_refusals_return_their_codes_before_any_launch(ctx):
    """tsb_lu_solve_batched refuses, without launching or writing x / status: an order that is not a permutation, an index
    out of 1..n (TSB_E_INVALID); n = 0 or 33 (TSB_E_INVALID); n_inst = 0 is a successful no-op."""
    TSB_OK, TSB_E_INVALID = 0, -1
    ident = np.arange(1, 6)
    before = ctx.launch_count
    for prow, pcol in (([1, 1, 3, 4, 5], ident), (ident, [2, 3, 4, 5, 5]), ([0, 2, 3, 4, 5], ident), (ident, [1, 2, 3, 4, 6]),
                       ([1, 2, 3, 4, -1], ident)):
        rc, x, st = _raw_solve(ctx, 5, prow, pcol, 3)
        assert rc == TSB_E_INVALID and np.all(x == -7.0) and np.all(st == -7), (prow, pcol, rc)
    for n in (0, 33):
        rc, x, st = _raw_solve(ctx, n, np.arange(1, n + 1), np.arange(1, n + 1), 2)
        assert rc == TSB_E_INVALID and np.all(x == -7.0) and np.all(st == -7), (n, rc)
    rc, x, st = _raw_solve(ctx, 5, ident, ident, 0)
    assert rc == TSB_OK and np.all(x == -7.0) and np.all(st == -7)
    assert ctx.launch_count == before
    rc, x, st = _raw_solve(ctx, 5, ident, ident, 1, A=np.eye(5)[None] * 2.0)      # and the library still works
    assert rc == TSB_OK and np.array_equal(x, np.full((1, 5), 0.5)) and st[0] == 0 and ctx.launch_count == before + 1
