"""Batched complex LU operator (tsb_lu_solve_batched_complex[_dev], csrc/lu_warp.cu: tsb_k_clu_warp): the reference's
FactorComplex + SolveComplex (pkg/matrix/circuit.go:130, 140) over a batch, in a pivot order frozen on the real matrix.

References:
* exact Gaussian-integer systems (`exact_complex_systems`): L unit lower triangular with entries in {0, +-1, +-i}, U with
  pivots in {+-1, +-2, +-4, +-i, +-2i, +-4i} and sparse Gaussian-integer entries, x Gaussian integers.  Smith's reciprocal
  of these pivots is exact and so is every product with it, so x must come back exactly in any order, mapping or build.
* the oracle's Sparse 1.3 complex path (Sparse13::factor_complex / solve_complex, driven by tests/cpp/lu_complex_oracle.cpp
  with the AC analysis' call sequence) for the strict build, bit for bit, signs of zeros included; `sparse13_solve_complex`
  restates it in NumPy for any caller order.
* a correctly rounded complex residual (residual_exact on the real embedding [[Ar, -Ai], [Ai, Ar]]) for the fast build,
  held to a backward-error bound derived from complex rounding (fast_complex_bound).
* tsb_run_ac end to end: the linear AC decks assembled here with pin_numpy.ac_sweep's stamps and solved by the operator.

What is not specified and therefore not tested: x of a status-1 system (zero pivot).
"""
import ctypes as C
import math
import os
import re
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import parity_util as PU
from ac_decks import AC_DECKS, ac_draws
from oracle import pin_numpy as P
from test_lu_operator import mna_like
from test_lu_operator_edges import bits, gamma, graded_mna, pass_size, residual_exact, variant  # noqa: F401 (fixture)

T, O = PU.T, PU.O
ROOT = PU.ROOT

# (W, R) built for the complex kernel: the forced rows per lane that reaches it and an order n it serves
CMAPPINGS = [((4, 2), 2, 8), ((8, 2), 2, 13), ((32, 1), 1, 29)]
CMAPPING_CASES = [pytest.param(wr, r, n, strict, id=f"{wr[0]}x{wr[1]}-{'strict' if strict else 'fast'}")
                  for wr, r, n in CMAPPINGS for strict in (True, False)]
CVARIANTS = [f"{r},0,{a}" for r in (1, 2) for a in (0, 1)]       # $TSB_LU_VARIANT: every built mapping, both stagings


# ---- the complex oracle (Sparse 1.3 restatement of oracle/sparse13.hpp, compiled here) -------------------------------
_OLIB = {}


def oracle_lib():
    if "L" not in _OLIB:
        import tempfile
        d = tempfile.mkdtemp(prefix="tsb_lucx_")
        so = os.path.join(d, "liblucx.so")
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-shared",
               "-I", os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests", "cpp", "lu_complex_oracle.cpp"), "-o", so]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        L = C.CDLL(so)
        dp = C.POINTER(C.c_double)
        L.orc_lu_batch_complex.argtypes = [C.c_int, dp, C.c_int64, dp, dp, dp, C.POINTER(C.c_int32), C.POINTER(C.c_int),
                                           C.POINTER(C.c_int)]
        _OLIB["L"] = L
    return _OLIB["L"]


def lu_batch_complex(A_nominal, A, b):
    """Sparse 1.3's complex path on a batch, order frozen by factor() on the REAL nominal matrix (orc_lu_batch_complex).
    Returns x [n_inst, n] complex128, status [n_inst], (pivot_row, pivot_col) 1-based."""
    n = A_nominal.shape[0]
    An = np.ascontiguousarray(A_nominal, dtype=np.float64)
    A = np.ascontiguousarray(A, dtype=np.complex128)
    b = np.ascontiguousarray(b, dtype=np.complex128)
    x = np.zeros(b.shape, dtype=np.complex128)
    st = np.zeros(len(b), dtype=np.int32)
    pr, pc = (C.c_int * n)(), (C.c_int * n)()
    dp = C.POINTER(C.c_double)
    rc = oracle_lib().orc_lu_batch_complex(n, An.ctypes.data_as(dp), len(b), A.ctypes.data_as(dp), b.ctypes.data_as(dp),
                                           x.ctypes.data_as(dp), st.ctypes.data_as(C.POINTER(C.c_int32)), pr, pc)
    if rc != 0:
        raise RuntimeError("oracle: nominal matrix is singular")
    return x, st, (np.array(pr[:]), np.array(pc[:]))


def cbits(z):
    z = np.ascontiguousarray(z, dtype=np.complex128)
    return z.view(np.float64).view(np.int64)


def make_complex(re, im):
    """re + i im without arithmetic (1j * im would turn signed zeros and infinities into other values)."""
    z = np.empty(np.broadcast(re, im).shape, dtype=np.complex128)
    z.real, z.imag = re, im
    return z


# ---- generators -----------------------------------------------------------------------------------------------------
GAUSS_UNITS = np.array([0, 1, -1, 1j, -1j])
PIVOTS = np.array([1, -1, 2, -2, 4, -4, 1j, -1j, 2j, -2j, 4j, -4j])


def exact_complex_systems(n, n_inst, seed, order=None, zero_step=None):
    """Gaussian-integer systems in a pivot order: L unit lower triangular with entries in {0, +-1, +-i}, U upper triangular
    with pivots in {+-1, +-2, +-4, +-i, +-2i, +-4i} and entries a + bi, a, b in [-2, 2], at ~30 % fill; x a + bi with a, b in
    [-8, 8]; A[prow[i], pcol[j]] = (L U)[i, j], b = A x (exact: small integers in float64).  zero_step = k: U_kk = 0 (a
    scalar, or one step per system).  Returns A, b, x (complex128) and the 1-based order."""
    rng = np.random.default_rng(seed)
    if order is None:
        prow, pcol = rng.permutation(n), rng.permutation(n)
    else:
        prow, pcol = np.asarray(order[0]) - 1, np.asarray(order[1]) - 1
    L = np.tril(rng.choice(GAUSS_UNITS, (n_inst, n, n)), -1) + np.eye(n)
    fill = rng.random((n_inst, n, n)) < 0.3
    U = np.triu((rng.integers(-2, 3, (n_inst, n, n)) + 1j * rng.integers(-2, 3, (n_inst, n, n))) * fill, 1)
    U[:, np.arange(n), np.arange(n)] = rng.choice(PIVOTS, (n_inst, n))
    if zero_step is not None:
        ks = np.broadcast_to(zero_step, (n_inst,))
        U[np.arange(n_inst), ks, ks] = 0
    x = rng.integers(-8, 9, (n_inst, n)) + 1j * rng.integers(-8, 9, (n_inst, n))
    A = np.empty((n_inst, n, n), dtype=np.complex128)
    A[:, prow[:, None], pcol[None, :]] = L @ U
    b = np.einsum("qij,qj->qi", A, x)
    return A + 0.0, b + 0.0, x.astype(np.complex128), (prow + 1, pcol + 1)


def mna_gc(n, n_inst, seed, freq):
    """MNA-like G + j omega C systems: G from mna_like (its nominal matrix freezes the order), C a capacitance network
    (branches and caps to ground, 1 pF .. 10 nF, scaled per instance by 0.5 .. 2) on the node rows only: the voltage-source
    rows and columns stay real.  freq: one frequency per instance (Hz).  Returns the real nominal G, A and b (complex)."""
    base, G, br = mna_like(n, n_inst, seed)
    rng = np.random.default_rng(seed + 1)
    k = min(2, n // 3)
    nodes = np.setdiff1d(np.arange(n), [n - 1 - q for q in range(k)])
    Cn = np.zeros((n, n))
    for _ in range(max(1, len(nodes))):
        i, j = rng.choice(nodes, 2) if len(nodes) > 1 else (nodes[0], nodes[0])
        c = 10.0 ** rng.uniform(-12, -8)
        Cn[i, i] += c
        if i != j:
            Cn[j, j] += c
            Cn[i, j] -= c
            Cn[j, i] -= c
    Cq = Cn[None] * np.exp(rng.uniform(np.log(0.5), np.log(2.0), (n_inst, n, n)))
    Cq = (Cq + np.transpose(Cq, (0, 2, 1))) / 2
    omega = 2 * np.pi * np.broadcast_to(np.asarray(freq, dtype=np.float64), (n_inst,))
    A = make_complex(G, omega[:, None, None] * Cq)
    b = make_complex(br, rng.normal(size=br.shape) * (rng.random(br.shape) < 0.5))
    return base, A, b


def freqs(n_inst, seed):
    """Log-uniform frequencies 1 Hz .. 1 GHz, both ends included."""
    f = 10.0 ** np.random.default_rng(seed).uniform(0.0, 9.0, n_inst)
    f[0], f[-1] = 1.0, 1e9
    return f


# ---- CPU references -------------------------------------------------------------------------------------------------
def crecip(re, im):
    """CMPLX_RECIPROCAL (Smith), Sparse 1.3's branch predicates: a NaN takes the else branch."""
    with np.errstate(all="ignore"):
        first = ((re >= im) & (re > -im)) | ((re < im) & (re <= -im))
        r1 = im / re
        t1 = 1.0 / (re + r1 * im)
        r2 = re / im
        t2 = -1.0 / (im + r2 * re)
        return np.where(first, t1, -r2 * t2), np.where(first, -r1 * t1, t2)


def sparse13_solve_complex(A, b, order):
    """Sparse 1.3's complex arithmetic in a frozen pivot order, float64 real and imaginary parts, batched: reciprocal pivots
    by Smith's form, U rows scaled by them (CMPLX_MULT), trailing rows dest - (m e) (CMPLX_MULT_SUBT_ASSIGN), forward
    substitution skipped where both parts of the entry are zero, back substitution row by row with ascending columns;
    entries of A loaded onto +0 (-0.0 -> +0.0).  Returns x (complex128) and the largest magnitude of any intermediate part."""
    prow, pcol = np.asarray(order[0]) - 1, np.asarray(order[1]) - 1
    n = len(prow)
    Pr = A.real[:, prow][:, :, pcol] + 0.0
    Pi = A.imag[:, prow][:, :, pcol] + 0.0
    cr, ci = b.real[:, prow].copy(), b.imag[:, prow].copy()
    big = max(np.abs(Pr).max(initial=0.0), np.abs(Pi).max(initial=0.0))
    with np.errstate(all="ignore"):
        for k in range(n):
            pr, pi = crecip(Pr[:, k, k], Pi[:, k, k])
            Pr[:, k, k], Pi[:, k, k] = pr, pi
            dr, di = Pr[:, k, k + 1:], Pi[:, k, k + 1:]
            ur, ui = dr * pr[:, None] - di * pi[:, None], dr * pi[:, None] + di * pr[:, None]
            Pr[:, k, k + 1:], Pi[:, k, k + 1:] = ur, ui
            er, ei = Pr[:, k + 1:, k, None], Pi[:, k + 1:, k, None]
            Pr[:, k + 1:, k + 1:] = Pr[:, k + 1:, k + 1:] - (ur[:, None, :] * er - ui[:, None, :] * ei)
            Pi[:, k + 1:, k + 1:] = Pi[:, k + 1:, k + 1:] - (ur[:, None, :] * ei + ui[:, None, :] * er)
            big = max(big, np.abs(Pr[:, k:, k + 1:]).max(initial=0.0), np.abs(Pi[:, k:, k + 1:]).max(initial=0.0))
        for k in range(n):
            nz = (cr[:, k] != 0.0) | (ci[:, k] != 0.0)
            tr, ti = cr[:, k], ci[:, k]
            mr, mi = tr * Pr[:, k, k] - ti * Pi[:, k, k], tr * Pi[:, k, k] + ti * Pr[:, k, k]
            cr[:, k], ci[:, k] = np.where(nz, mr, tr), np.where(nz, mi, ti)
            er, ei = Pr[:, k + 1:, k], Pi[:, k + 1:, k]
            m2r, m2i = mr[:, None], mi[:, None]
            cr[:, k + 1:] = np.where(nz[:, None], cr[:, k + 1:] - (m2r * er - m2i * ei), cr[:, k + 1:])
            ci[:, k + 1:] = np.where(nz[:, None], ci[:, k + 1:] - (m2r * ei + m2i * er), ci[:, k + 1:])
            big = max(big, np.abs(cr).max(), np.abs(ci).max())
        for i in range(n - 2, -1, -1):
            tr, ti = cr[:, i], ci[:, i]
            for j in range(i + 1, n):
                er, ei = Pr[:, i, j], Pi[:, i, j]
                tr, ti = tr - (er * cr[:, j] - ei * ci[:, j]), ti - (er * ci[:, j] + ei * cr[:, j])
            cr[:, i], ci[:, i] = tr, ti
            big = max(big, np.abs(tr).max(), np.abs(ti).max())
    xr, xi = np.empty_like(cr), np.empty_like(ci)
    xr[:, pcol], xi[:, pcol] = cr, ci
    return make_complex(xr, xi), big


def embed(A):
    """The 2n real embedding [[Ar, -Ai], [Ai, Ar]] of complex A (x = [xr; xi], b = [br; bi])."""
    return np.concatenate([np.concatenate([A.real, -A.imag], axis=2), np.concatenate([A.imag, A.real], axis=2)], axis=1)


def residual_complex(A, x, b):
    """b - A x of complex systems, each part correctly rounded (residual_exact on the real embedding)."""
    n = A.shape[1]
    r = residual_exact(embed(A), np.concatenate([x.real, x.imag], axis=1), np.concatenate([b.real, b.imag], axis=1))
    return make_complex(r[:, :n], r[:, n:])


def abs_lu_complex(A, order):
    """|L||U| (moduli) of the frozen-order complex Doolittle elimination, in external row / column numbering."""
    prow, pcol = np.asarray(order[0]) - 1, np.asarray(order[1]) - 1
    n = len(prow)
    Pm = A[:, prow][:, :, pcol].copy()
    Lm = np.zeros_like(Pm)
    Lm[:, np.arange(n), np.arange(n)] = 1.0
    for k in range(n):
        m = Pm[:, k + 1:, k] / Pm[:, k, k, None]
        Lm[:, k + 1:, k] = m
        Pm[:, k + 1:, k:] -= m[:, :, None] * Pm[:, None, k, k:]
    out = np.empty(A.shape)
    out[:, prow[:, None], pcol[None, :]] = np.abs(Lm) @ np.abs(np.triu(Pm))
    return out


def fast_complex_bound(n):
    """Componentwise backward-error constant c of the fast build: |b - A x| <= c |L||U| |x| (moduli).

    Model (Higham, Accuracy and Stability of Numerical Algorithms, §3.6): a real operation rounds with |delta| <= u.  In the
    fast build every part of dest - m e is two DFMA, fma(-mr, er, fma(mi, ei, dr)): a part of an entry that receives k
    updates is a recursive sum of 2k + 1 real terms with 2k roundings, so its error is within gamma(2k) times the sum of the
    magnitudes of those terms, and |mr er| + |mi ei| <= |m| |e| (Cauchy-Schwarz): per part gamma(2k) (|d| + sum |m| |e|),
    for the complex modulus sqrt(2) gamma(2k) (Higham's sqrt(2) gamma_2 for one complex multiply, accumulated).  The
    reciprocal pivot (Smith's form: r = b * rcp(a) with rcp within 2u, d = fma(r, b, a), t = rcp(d), -r t) is within
    gamma(10) of 1/p in each part, and multiplying by it (the multipliers, the back substitution's x_j = y_j / u_jj) adds a
    complex multiply, sqrt(2) gamma(2) <= gamma(3): gamma(13) per division.  Factor, forward and back substitution each
    contribute one such inner product of at most n - 1 terms plus one division, as in the real case (Higham Thm. 9.4: gamma(3n)
    for the three together): c = sqrt(2) gamma(3 (2n + 13))."""
    return math.sqrt(2.0) * gamma(3 * (2 * n + 13))


# ---- CPU tests ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 5, 8, 13, 16, 24, 32])
def test_exact_complex_systems_solve_exactly(n):
    """The generator's promise: x comes back exactly in a random order through the Sparse 1.3 restatement, and every
    intermediate stays small (nothing is rounded)."""
    A, b, x, order = exact_complex_systems(n, 40, 2000 + n)
    assert np.array_equal(np.einsum("qij,qj->qi", A, x), b)
    xs, big = sparse13_solve_complex(A, b, order)
    assert np.array_equal(xs, x) and big <= 2.0 ** 20, (n, big)


def test_smith_reciprocal_of_the_generator_pivots_is_exact():
    re, im = crecip(PIVOTS.real.copy(), PIVOTS.imag.copy())
    assert np.array_equal(make_complex(re, im), 1.0 / PIVOTS)


@pytest.mark.parametrize("n", [1, 2, 5, 9, 16, 25, 32])
def test_complex_restatement_matches_the_oracle(built, n):
    """sparse13_solve_complex is the oracle's factor_complex / solve_complex bit for bit in the oracle's own order (frozen on
    the real nominal matrix), signed zeros included, on G + j omega C systems from 1 Hz to 1 GHz; also with infinite pivots,
    NaN entries and infinite right-hand sides (NaN at the same places)."""
    base, A, b = mna_gc(n, 60, 600 + n, freqs(60, n))
    xo, sto, opo = lu_batch_complex(base, A, b)
    assert np.array_equal(opo[0], T.lu_order(base)[0]) and np.array_equal(opo[1], T.lu_order(base)[1])
    xs, _ = sparse13_solve_complex(A, b, opo)
    assert np.all(sto == 0) and np.array_equal(cbits(xs), cbits(xo))
    rng = np.random.default_rng(n)
    ks = np.arange(len(A)) % n
    A2 = A.copy()
    A2[np.arange(len(A)), opo[0][ks] - 1, opo[1][ks] - 1] = make_complex(np.inf, A.imag[np.arange(len(A)), opo[0][ks] - 1, opo[1][ks] - 1])
    A2[::5, rng.integers(0, n), rng.integers(0, n)] = make_complex(np.nan, 0.0)
    b2 = b.copy()
    b2[1::4, rng.integers(0, n)] = make_complex(0.0, -np.inf)
    xo, sto, _ = lu_batch_complex(base, A2, b2)
    xs, _ = sparse13_solve_complex(A2, b2, opo)
    ok = sto == 0
    assert ok.sum() > 0
    assert np.array_equal(np.isnan(xs.view(np.float64))[ok], np.isnan(xo.view(np.float64))[ok])
    assert np.array_equal(xs[ok], xo[ok], equal_nan=True)


def test_complex_residual_is_correctly_rounded():
    """residual_complex against exact rational arithmetic, on residuals that cancel to the last bits and on parts spread
    over 30 orders of magnitude."""
    rng = np.random.default_rng(4)
    n, q = 7, 12
    A = make_complex(rng.normal(size=(q, n, n)) * np.exp(rng.uniform(-30, 30, (q, n, n))),
                     rng.normal(size=(q, n, n)) * np.exp(rng.uniform(-30, 30, (q, n, n))))
    x = make_complex(rng.normal(size=(q, n)) * np.exp(rng.uniform(-8, 8, (q, n))), rng.normal(size=(q, n)))
    b = np.einsum("qij,qj->qi", A, x)
    b[::2] = make_complex(rng.normal(size=(q // 2, n)), rng.normal(size=(q // 2, n)))
    r = residual_complex(A, x, b)
    F = Fraction
    for s in range(q):
        for i in range(n):
            er = F(b[s, i].real) - sum(F(A[s, i, j].real) * F(x[s, j].real) - F(A[s, i, j].imag) * F(x[s, j].imag) for j in range(n))
            ei = F(b[s, i].imag) - sum(F(A[s, i, j].real) * F(x[s, j].imag) + F(A[s, i, j].imag) * F(x[s, j].real) for j in range(n))
            assert r[s, i].real == float(er) and r[s, i].imag == float(ei), (s, i)


@pytest.mark.parametrize("n", [1, 2, 3, 8, 13, 24, 32])
def test_oracle_reports_the_constructed_complex_zero_pivots(built, n):
    """Exact zero pivots (both parts 0) at step k of the order frozen on the real nominal matrix: status 1 on exactly those."""
    base, _, _ = mna_like(n, 1, 40 + n)
    order = T.lu_order(base)
    steps = np.array([0, n // 2, n - 1, 0, n // 2, n - 1])
    As, bs, _, _ = exact_complex_systems(n, len(steps), 9 * n, order=order, zero_step=steps)
    Ar, br, _, _ = exact_complex_systems(n, 4, 9 * n + 1, order=order)
    _, st, opo = lu_batch_complex(base, np.concatenate([As, Ar]), np.concatenate([bs, br]))
    assert np.array_equal(opo[0], order[0]) and np.array_equal(opo[1], order[1])
    assert st.tolist() == [1] * len(steps) + [0] * 4


def test_every_built_complex_mapping_keeps_the_matrix_in_registers(built):
    """Every tsb_k_clu_warp instantiation in the built library keeps its rows in registers: a few spilled bytes at most
    (2 R N x 8 bytes of stack if the register arrays were lost), and at most 170 registers (three 128-thread blocks per SM)."""
    lib = os.path.join(ROOT, "toy-spice_b200", "libtspice_b200.so")
    out = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout
    found = re.findall(r"tsb_k_clu_warpILi(\d+)ELi(\d+)ELb([01])ELb([01])\S*:\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    assert sorted({(int(w), int(r), s, a) for w, r, s, a, _, _ in found}) == sorted(
        {(w, r, s, a) for (w, r), _, _ in CMAPPINGS for s in "01" for a in "01"}), found
    for w, r, strict, asyn, reg, stack in found:
        assert int(stack) <= 160, (w, r, strict, asyn, reg, stack)
        assert int(reg) <= 170, (w, r, strict, asyn, reg)


def ac_system(devices, n, f, params):
    """The AC system of a linear deck at frequency f for every instance, with pin_numpy.ac_sweep's stamps (resistor g,
    capacitor and inductor j omega X between the nodes, voltage-source incidence and phasor, current-source phasor).
    params: {(device name, parameter): per-instance values}.  Returns A [n_inst, n, n], b [n_inst, n] (0-based = MNA - 1)."""
    n_inst = len(next(iter(params.values())))
    A = np.zeros((n_inst, n + 1, n + 1), dtype=complex)
    rhs = np.zeros((n_inst, n + 1), dtype=complex)
    omega = 2 * math.pi * f

    def p_of(d, k):
        return np.asarray(params.get((d["name"], k), np.full(n_inst, d["p"][k])), dtype=np.float64)

    def two_terminal(n1, n2, y):
        if n1:
            A[:, n1, n1] += y
        if n2:
            A[:, n2, n2] += y
        if n1 and n2:
            A[:, n1, n2] -= y
            A[:, n2, n1] -= y

    def phasor(d):
        mag, ph = p_of(d, 1), p_of(d, 2)
        return mag * np.array([complex(math.cos(v * math.pi / 180.0), math.sin(v * math.pi / 180.0)) for v in ph])

    for d in devices:
        k, nd = d["kind"], d["nodes"]
        if k == T.api.K_R:
            two_terminal(nd[0], nd[1], 1.0 / p_of(d, 0))
        elif k in (T.api.K_C, T.api.K_L):
            two_terminal(nd[0], nd[1], 1j * omega * p_of(d, 0))
        elif k == T.api.K_V:
            br = d["branch"]
            if nd[0]:
                A[:, br, nd[0]] += 1
                A[:, nd[0], br] += 1
            if nd[1]:
                A[:, br, nd[1]] -= 1
                A[:, nd[1], br] -= 1
            if (not d["ip"] or d["ip"][0] == 0) and len(d["p"]) >= 3:
                rhs[:, br] += phasor(d)
        elif k == T.api.K_I:
            if (not d["ip"] or d["ip"][0] == 0) and len(d["p"]) >= 3:
                cur = phasor(d)
                if nd[0]:
                    rhs[:, nd[0]] += cur
                if nd[1]:
                    rhs[:, nd[1]] -= cur
        else:
            raise ValueError("linear R / C / V / I decks only")
    return A[:, 1:, 1:], rhs[:, 1:]


def ac_rows(x, devices, n_nodes):
    """[mag, phase_deg] per node voltage, then per V-source current, as tsb_run_ac's columns 1..."""
    idx = list(range(n_nodes)) + [d["branch"] - 1 for d in devices if d["kind"] == T.api.K_V]
    z = x[..., idx]
    out = np.empty(z.shape[:-1] + (2 * len(idx),))
    out[..., 0::2] = np.abs(z)
    out[..., 1::2] = np.degrees(np.arctan2(z.imag, z.real))
    return out


def _deck(name):
    ckt = T.Circuit.from_netlist(AC_DECKS[name])
    devs = ckt.devices()
    n = ckt.n
    n_nodes = n - len({d["branch"] for d in devs if d["kind"] == T.api.K_V})
    return ckt, devs, n, n_nodes


@pytest.mark.parametrize("name", sorted(AC_DECKS))
def test_ac_assembly_has_the_stamps_of_the_numpy_pin(built, name):
    """ac_system solved with numpy.linalg.solve reproduces pin_numpy.ac_sweep's rows (the same stamps, the same read-out),
    one instance at the deck's nominal values."""
    _, devs, n, n_nodes = _deck(name)
    oc = O.OracleCircuit(AC_DECKS[name])
    a = oc.netlist.ac
    rows, fail = P.ac_sweep(oc.plan, a["sweep"], a["points"], a["fstart"], a["fstop"])
    assert fail is None and oc.plan.n_nodes == n_nodes
    nominal = {(d["name"], k): np.array([v]) for d in devs for k, v in enumerate(d["p"])}
    for row in rows:
        A, b = ac_system(devs, n, row[0], nominal)
        x = np.linalg.solve(A[0], b[0])
        assert np.allclose(ac_rows(x, devs, n_nodes), row[1:], rtol=1e-13, atol=1e-15), (name, row[0])


# ---- GPU tests ------------------------------------------------------------------------------------------------------
def expected_cmapping(n, rows=None):
    """(W, R) launch_clu_warp runs for order n; rows = the rows per lane $TSB_LU_VARIANT forces (None: the default)."""
    if rows == 1:
        return (32, 1)
    return (4, 2) if n <= 8 else (8, 2) if n <= 16 else (32, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
@pytest.mark.parametrize("var", CVARIANTS)
def test_exact_complex_systems_every_n_and_mapping(ctx, variant, var, strict):
    """Caller-chosen random pivot orders, every n = 1..32 under every built mapping and staging: x exact in both builds."""
    variant(var)
    for n in range(1, 33):
        A, b, x, order = exact_complex_systems(n, 131, 19 * n + 3)
        xk, st = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
        assert np.all(st == 0), (var, n)
        assert np.array_equal(xk, x), (var, n, int(np.sum(xk != x)), np.argwhere(xk != x)[:3].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("var", CVARIANTS)
def test_strict_build_bit_identical_to_sparse13_complex(ctx, variant, var):
    """The strict build against the oracle's factor_complex / solve_complex, every n = 1..32 under every built mapping and
    staging, G + j omega C systems over 1 Hz .. 1 GHz in the order tsb_lu_order picks on G: the same bits, signs of zeros
    included."""
    variant(var)
    for n in range(1, 33):
        base, A, b = mna_gc(n, 67, 29 * n + 7, freqs(67, n))
        order = T.lu_order(base)
        xo, sto, _ = lu_batch_complex(base, A, b)
        x, st = ctx.lu_solve_batched_complex(A, b, order, strict=True)
        assert np.array_equal(st, sto) and np.all(st == 0), (var, n)
        assert np.array_equal(cbits(x), cbits(xo)), (var, n, float(np.max(np.abs(x - xo))))


def graded_complex(n, n_inst, seed):
    """graded_mna systems (conductances over 15 decades) with every entry given a random phase: strongly graded complex
    matrices whose order is frozen on the real graded nominal matrix."""
    base, A, b = graded_mna(n, n_inst, seed)
    ph = np.random.default_rng(seed + 7).uniform(-np.pi, np.pi, A.shape)
    return base, A * np.exp(1j * ph), b * np.exp(1j * ph[:, :, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["mna_gc", "graded"])
def test_fast_build_within_the_derived_complex_bound(ctx, variant, family):
    """Fast build: the correctly rounded complex residual is within the bound of fast_complex_bound, componentwise per
    system: |b - A x|_i <= c (|L||U| |x|)_i, with |.| the complex modulus (of a correctly rounded pair: the modulus itself is
    taken in float64, hence the factor 1 + 4u)."""
    for n in (2, 4, 7, 8, 12, 16, 20, 24, 32):
        if family == "mna_gc":
            base, A, b = mna_gc(n, 300, 41 * n, freqs(300, 41 * n))
        else:
            base, A, b = graded_complex(n, 300, 43 * n)
        order = T.lu_order(base)
        x, st = ctx.lu_solve_batched_complex(A, b, order, strict=False)
        assert np.all(st == 0) and np.all(np.isfinite(x)), n
        r = np.abs(residual_complex(A, x, b))
        bound = fast_complex_bound(n) * (1 + 4 * 2.0 ** -53) * np.einsum("qij,qj->qi", abs_lu_complex(A, order), np.abs(x))
        worst = np.unravel_index(np.argmax(r / np.maximum(bound, 1e-300)), r.shape)
        assert np.all(r <= bound), (family, n, worst, float(r[worst]), float(bound[worst]))


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
def test_power_of_two_scaling_is_equivariant(ctx, strict):
    """(D1 A D2, D1 b), D1, D2 diagonal powers of two (2^-200 .. 2^200), gives D2^-1 x bit for bit in both builds (the fast
    reciprocal's seed depends on the significand alone)."""
    rng = np.random.default_rng(29)
    for n in range(1, 33):
        base, A, b = mna_gc(n, 129, 31 * n, freqs(129, 31 * n))
        order = T.lu_order(base)
        e1 = rng.integers(-200, 201, (len(A), n))
        e2 = rng.integers(-200, 201, (len(A), n))
        sc = lambda z, e: make_complex(np.ldexp(z.real, e), np.ldexp(z.imag, e))   # noqa: E731
        As = sc(sc(A, e1[:, :, None]), e2[:, None, :])
        bs = sc(b, e1)
        x, st = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
        xs, sts = ctx.lu_solve_batched_complex(As, bs, order, strict=strict)
        assert np.all(st == 0) and np.all(sts == 0)
        assert np.array_equal(cbits(xs), cbits(sc(x, -e2))), (n, strict)


@pytest.mark.gpu
def test_real_systems_give_the_real_operators_result(ctx, variant):
    """Imaginary parts all zero: the complex strict build equals the real operator's strict build (==: signs of zeros may
    differ, the reciprocal of a real pivot has a signed-zero imaginary part), and x.imag == 0 — under every built mapping."""
    for var in CVARIANTS:
        variant(var)
        for n in range(1, 33):
            base, A, b = mna_like(n, 65, 13 * n + 1)
            order = T.lu_order(base)
            xr, str_ = ctx.lu_solve_batched(A, b, order, strict=True)
            xc, stc = ctx.lu_solve_batched_complex(A.astype(np.complex128), b.astype(np.complex128), order, strict=True)
            assert np.array_equal(stc, str_) and np.all(stc == 0), (var, n)
            assert np.all(xc.real == xr) and np.all(xc.imag == 0.0), (var, n)


@pytest.mark.gpu
@pytest.mark.parametrize("wr,rows,n,strict", CMAPPING_CASES)
def test_zero_pivots_are_isolated_in_their_lane_group(ctx, variant, wr, rows, n, strict):
    """Singular systems (both parts of a pivot exactly 0) at every group slot of a warp and at the first and last instance
    of a resident pass, over more than one pass: status 1 on exactly those; every other system has the bits of a run in
    which the singular ones are replaced by regular ones."""
    variant(f"{rows},0,1")
    groups = 128 // wr[0]
    per_warp = 32 // wr[0]
    ps = pass_size(ctx, wr)
    n_inst = ps + 2 * groups + 3
    rng = np.random.default_rng(n)
    order = (rng.permutation(n) + 1, rng.permutation(n) + 1)
    A0, b0, x0, _ = exact_complex_systems(n, 509, 61 * n, order=order)
    idx = np.arange(n_inst) % 509
    A, b, x = A0[idx], b0[idx], x0[idx]
    sing = sorted({g * (per_warp + 1) for g in range(per_warp)} | {ps - 1, ps, n_inst - 1})
    As, bs, _, _ = exact_complex_systems(n, len(sing), 67 * n, order=order, zero_step=rng.integers(0, n, len(sing)))
    A2, b2 = A.copy(), b.copy()
    A2[sing], b2[sing] = As, bs
    x1, st1 = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
    x2, st2 = ctx.lu_solve_batched_complex(A2, b2, order, strict=strict)
    assert np.all(st1 == 0) and np.array_equal(x1, x)
    expect = np.zeros(n_inst, dtype=np.int32)
    expect[sing] = 1
    assert np.array_equal(st2, expect), np.flatnonzero(st2 != expect)[:8].tolist()
    keep = expect == 0
    assert np.array_equal(cbits(x2[keep]), cbits(x1[keep]))


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
@pytest.mark.parametrize("var", [None, "1,0,1", "2,0,0"])
def test_infinite_pivot_gives_zero_for_its_column(ctx, variant, var, strict):
    """A pivot with an infinite real part and a finite imaginary part at step k of the frozen order (k varies over the
    batch): its reciprocal is 0, x[pcol[k]] = 0 and everything else finite, as Sparse 1.3 computes it (strict: its bits).
    An infinite pivot can leave a later pivot exactly 0 (a source row whose only coupling went through row k): status 1
    there, as in the oracle."""
    variant(var)
    for n in (1, 2, 5, 8, 11, 16, 21, 32):
        base, A, b = mna_gc(n, 97, 37 * n, freqs(97, 37 * n))
        order = T.lu_order(base)
        ks = np.arange(len(A)) % n
        q, r, c = np.arange(len(A)), order[0][ks] - 1, order[1][ks] - 1
        A[q, r, c] = make_complex(np.inf, A.imag[q, r, c])
        xo, sto, _ = lu_batch_complex(base, A, b)
        x, st = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
        ok = sto == 0
        assert ok.sum() >= len(A) // 2, (n, int(ok.sum()))
        assert np.all(np.isfinite(xo[ok])) and np.all(xo[ok, order[1][ks[ok]] - 1] == 0.0)
        assert np.array_equal(st, sto), (var, n)
        if strict:
            assert np.array_equal(cbits(x[ok]), cbits(xo[ok])), (var, n)
        else:
            assert np.all(np.isfinite(x[ok])), (var, n)
            assert np.all(x[ok, order[1][ks[ok]] - 1] == 0.0), (var, n)


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
def test_nan_entries_and_infinite_right_hand_sides(ctx, strict):
    """NaN in one part of a random entry of A (every third system), +-Inf in one part of a random entry of b (every third,
    shifted by one): status as the oracle's; the strict build has the oracle's bits (NaN at the same places); the fast
    build is non-finite at least where the oracle is."""
    rng = np.random.default_rng(6)
    for n in (1, 3, 8, 12, 17, 32):
        base, A, b = mna_gc(n, 150, 47 * n, freqs(150, 47 * n))
        order = T.lu_order(base)
        qa, qb = np.arange(0, len(A), 3), np.arange(1, len(A), 3)
        ia, ja = rng.integers(0, n, len(qa)), rng.integers(0, n, len(qa))
        part = rng.random(len(qa)) < 0.5
        A[qa, ia, ja] = np.where(part, make_complex(np.nan, A.imag[qa, ia, ja]), make_complex(A.real[qa, ia, ja], np.nan))
        ib = rng.integers(0, n, len(qb))
        inf = np.where(rng.random(len(qb)) < 0.5, np.inf, -np.inf)
        b[qb, ib] = np.where(rng.random(len(qb)) < 0.5, make_complex(inf, b.imag[qb, ib]), make_complex(b.real[qb, ib], inf))
        xo, sto, _ = lu_batch_complex(base, A, b)
        x, st = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
        assert np.array_equal(st, sto), n
        xf, xof = x.view(np.float64), xo.view(np.float64)
        if strict:
            assert np.array_equal(np.isnan(xf), np.isnan(xof)), n
            assert np.array_equal(xf, xof, equal_nan=True), n
        else:
            assert np.all(~np.isfinite(xf) | np.isfinite(xof)), n


@pytest.mark.gpu
@pytest.mark.parametrize("wr,rows,n,strict", CMAPPING_CASES)
def test_batch_sizes_at_the_group_and_pass_edges(ctx, variant, wr, rows, n, strict):
    """n_inst = 1, one block's systems -+ 1, exactly one resident pass and one more, with both stagings: exact x."""
    groups = 128 // wr[0]
    ps = pass_size(ctx, wr)
    rng = np.random.default_rng(200 + n)
    order = (rng.permutation(n) + 1, rng.permutation(n) + 1)
    A0, b0, x0, _ = exact_complex_systems(n, 509, 71 * n, order=order)
    idx = np.arange(ps + 1) % 509
    A, b, x = A0[idx], b0[idx], x0[idx]
    for staging in (0, 1):
        variant(f"{rows},0,{staging}")
        for m in (1, groups - 1, groups + 1, ps, ps + 1):
            xk, st = ctx.lu_solve_batched_complex(A[:m], b[:m], order, strict=strict)
            assert np.all(st == 0) and np.array_equal(xk, x[:m]), (staging, m, int(np.sum(xk != x[:m])))


@pytest.mark.gpu
@pytest.mark.parametrize("wr,rows,n,strict", CMAPPING_CASES)
def test_device_pointers_aligned_to_8_bytes_only(ctx, variant, wr, rows, n, strict):
    """lu_solve_batched_complex_dev on interleaved data that starts one double into its allocation (A, b, x 8-byte but not
    16-byte aligned, status 4-byte): the same bits and status as from complex128 tensors, and those equal the host entry's."""
    import torch
    variant(f"{rows},0,1")
    n_inst = 3 * (128 // wr[0]) + 5
    base, A, b = mna_gc(n, n_inst, 53 * n, freqs(n_inst, 53 * n))
    order = T.lu_order(base)
    xh, sh = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
    # complex128 tensors (16-byte aligned)
    tA, tb = torch.from_numpy(A).cuda(), torch.from_numpy(b).cuda()
    tx = torch.full((n_inst, n), complex(float("nan"), float("nan")), dtype=torch.complex128, device="cuda")
    ts = torch.full((n_inst,), -1, dtype=torch.int32, device="cuda")
    ctx.lu_solve_batched_complex_dev(n, n_inst, tA.data_ptr(), tb.data_ptr(), tx.data_ptr(), ts.data_ptr(), order, strict=strict)
    torch.cuda.synchronize()
    assert np.array_equal(ts.cpu().numpy(), sh) and np.array_equal(cbits(tx.cpu().numpy()), cbits(xh))
    # float64 buffers one element in
    fa = torch.zeros(2 * n_inst * n * n + 2, dtype=torch.float64, device="cuda")
    fb = torch.zeros(2 * n_inst * n + 2, dtype=torch.float64, device="cuda")
    fx = torch.full((2 * n_inst * n + 2,), float("nan"), dtype=torch.float64, device="cuda")
    fs = torch.full((n_inst + 2,), -1, dtype=torch.int32, device="cuda")
    dA, db, dx, ds = fa[1:1 + 2 * n_inst * n * n], fb[1:1 + 2 * n_inst * n], fx[1:1 + 2 * n_inst * n], fs[1:1 + n_inst]
    dA.copy_(torch.from_numpy(A.view(np.float64).reshape(-1)))
    db.copy_(torch.from_numpy(b.view(np.float64).reshape(-1)))
    assert [p.data_ptr() % 16 for p in (dA, db, dx)] == [8] * 3
    ctx.lu_solve_batched_complex_dev(n, n_inst, dA.data_ptr(), db.data_ptr(), dx.data_ptr(), ds.data_ptr(), order, strict=strict)
    torch.cuda.synchronize()
    assert torch.isnan(fx[:1]).all() and torch.isnan(fx[1 + 2 * n_inst * n:]).all() and int(fs[1 + n_inst]) == -1
    x1 = dx.cpu().numpy().view(np.complex128).reshape(n_inst, n)
    assert np.all(sh == 0) and np.array_equal(ds.cpu().numpy(), sh) and np.array_equal(cbits(x1), cbits(xh))


_CKNAME = [re.compile(r"tsb_k_clu_warp<(\d+), ?(\d+), ?(true|false), ?(true|false)>"),
           re.compile(r"tsb_k_clu_warpILi(\d+)ELi(\d+)ELb([01])ELb([01])E")]


def launched_clu_kernels(calls):
    """Runs `calls` under torch.profiler (CUDA activities) and returns (W, R, STRICT, ASYNC) of every tsb_k_clu_warp kernel
    that ran, in launch order."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.zeros(1, device="cuda")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for f in calls:
            f()
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if "tsb_k_clu_warp" in e.name), key=lambda e: e.time_range.start)
    assert evs, "torch.profiler recorded no tsb_k_clu_warp kernel: the dispatch cannot be checked"
    out = []
    for e in evs:
        m = _CKNAME[0].search(e.name) or _CKNAME[1].search(e.name)
        assert m, e.name
        w, r, s, a = m.groups()
        out.append((int(w), int(r), s in ("true", "1"), a in ("true", "1")))
    return out


@pytest.mark.gpu
def test_dispatch_follows_the_design_table(ctx, variant):
    """Default: n <= 8: 4 lanes x 2 rows, <= 16: 8 x 2, <= 32: 32 x 1, asynchronous staging; forced "R,0,A": R = 1 runs
    32 x 1 at every n, R = 2 and 3 the default mapping, R = 4 falls back to it, A the staging — in both builds."""
    cases = [(n, s, v) for v in (None, "1,0,0", "1,0,1", "2,0,0", "3,0,1", "4,0,0") for s in (True, False) for n in range(1, 33)]

    def call(n, strict, var):
        def f():
            variant(var)
            A, b, _, order = exact_complex_systems(n, 1, n)
            _, st = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
            assert st[0] == 0
        return f
    got = launched_clu_kernels([call(*c) for c in cases])
    want = [(*expected_cmapping(n, int(v[0]) if v else None), s, v is None or v.endswith("1")) for n, s, v in cases]
    assert len(got) == len(want)
    bad = [(c, g, w) for c, g, w in zip(cases, got, want) if g != w]
    assert not bad, bad[:6]


def _raw_solve(ctx, n, prow, pcol, n_inst, A=None, b=None):
    """tsb_lu_solve_batched_complex through the C ABI, returning the raw code; x / status prefilled with sentinels."""
    L = T.lib()
    nn = max(n, 1)
    A = np.ones((max(n_inst, 1), nn, nn), dtype=np.complex128) if A is None else A
    b = np.ones((max(n_inst, 1), nn), dtype=np.complex128) if b is None else b
    x = np.full(b.shape, -7.0 - 7.0j)
    st = np.full(max(n_inst, 1), -7, dtype=np.int32)
    pr = np.ascontiguousarray(prow, dtype=np.int32)
    pc = np.ascontiguousarray(pcol, dtype=np.int32)
    ip, dp = C.POINTER(C.c_int), C.POINTER(C.c_double)
    rc = L.tsb_lu_solve_batched_complex(ctx.h, n, pr.ctypes.data_as(ip), pc.ctypes.data_as(ip), A.ctypes.data_as(dp),
                                        b.ctypes.data_as(dp), x.ctypes.data_as(dp), st.ctypes.data_as(C.POINTER(C.c_int32)),
                                        n_inst, 1)
    return rc, x, st


@pytest.mark.gpu
def test_refusals_return_their_codes_before_any_launch(ctx):
    """The real operator's refusals, nothing launched or written: an order that is not a permutation or has an index outside
    1..n (TSB_E_INVALID), n = 0 or 33 (TSB_E_INVALID; the _dev entry: TSB_E_UNSUPPORTED), n_inst = 0 a successful no-op."""
    TSB_OK, TSB_E_INVALID, TSB_E_UNSUPPORTED = 0, -1, -5
    ident = np.arange(1, 6)
    before = ctx.launch_count
    for prow, pcol in (([1, 1, 3, 4, 5], ident), (ident, [2, 3, 4, 5, 5]), ([0, 2, 3, 4, 5], ident), (ident, [1, 2, 3, 4, 6]),
                       ([1, 2, 3, 4, -1], ident)):
        rc, x, st = _raw_solve(ctx, 5, prow, pcol, 3)
        assert rc == TSB_E_INVALID and np.all(x == -7.0 - 7.0j) and np.all(st == -7), (prow, pcol, rc)
    for n in (0, 33):
        rc, x, st = _raw_solve(ctx, n, np.arange(1, n + 1), np.arange(1, n + 1), 2)
        assert rc == TSB_E_INVALID and np.all(x == -7.0 - 7.0j) and np.all(st == -7), (n, rc)
        ar = np.arange(1, n + 1, dtype=np.int32)
        ip = C.POINTER(C.c_int)
        rc = T.lib().tsb_lu_solve_batched_complex_dev(ctx.h, n, ar.ctypes.data_as(ip), ar.ctypes.data_as(ip), 8, 8, 8, 8, 2, 1)
        assert rc == TSB_E_UNSUPPORTED, (n, rc)
    rc, x, st = _raw_solve(ctx, 5, ident, ident, 0)
    assert rc == TSB_OK and np.all(x == -7.0 - 7.0j) and np.all(st == -7)
    assert ctx.launch_count == before
    rc, x, st = _raw_solve(ctx, 5, ident, ident, 1, A=np.eye(5)[None] * 2j)        # and the library still works
    assert rc == TSB_OK and np.array_equal(x, np.full((1, 5), -0.5j)) and st[0] == 0 and ctx.launch_count == before + 1


def _phase_close(got, ref, atol):
    d = np.abs((got - ref + 180.0) % 360.0 - 180.0)
    return d <= 1e-9 * np.abs(ref) + atol


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
@pytest.mark.parametrize("name", sorted(AC_DECKS))
def test_end_to_end_against_tsb_run_ac(ctx, name, strict):
    """The linear AC decks, 48 instances of ac_draws: the systems assembled with pin_numpy.ac_sweep's stamps at the
    frequencies of tsb_run_ac's rows, solved by the complex operator in the plan's own order (tsb_plan_structure), agree
    with tsb_run_ac's magnitudes and phases within test_ac's tolerance (1e-9 relative, 1e-12 absolute), in both builds.
    Phases are compared modulo 360 degrees; where the value is exactly 0 on both sides (the DC source's branch of
    ac_two_v) the phase is atan2 of signed zeros, a convention rather than a result, and only the magnitude is compared."""
    n_inst = 48
    ckt, devs, n, n_nodes = _deck(name)
    ov = ac_draws(devs, n_inst)
    c = T.Circuit.from_netlist(AC_DECKS[name], ctx)
    bt = c.batch(n_inst)
    for (d, p), v in ov.items():
        bt.set_param(d, p, v)
    a = O.OracleCircuit(AC_DECKS[name]).netlist.ac
    bt.run_ac(a["sweep"], a["points"], a["fstart"], a["fstop"], out=T.OUT_WAVE, opts=T.default_opts(strict_fp=int(strict)))
    bt.sync()
    assert np.all(bt.status() == 0)
    wg = np.transpose(bt.wave_all(), (2, 0, 1))[:, :a["points"]]              # [inst][row][FREQ, mag, phase, ...]
    st = c.structure()
    order = (np.array(st["pivot_row"]), np.array(st["pivot_col"]))
    fs = wg[0, :, 0]
    assert np.all(wg[:, :, 0] == fs[None])
    As, bs = zip(*(ac_system(devs, n, f, ov) for f in fs))
    A, b = np.concatenate(As), np.concatenate(bs)                             # [freq][inst] flattened
    x, stx = ctx.lu_solve_batched_complex(A, b, order, strict=strict)
    assert np.all(stx == 0)
    got = ac_rows(x, devs, n_nodes).reshape(len(fs), n_inst, -1).transpose(1, 0, 2)
    ref = wg[:, :, 1:]
    mag, rmag = got[..., 0::2], ref[..., 0::2]
    assert np.allclose(mag, rmag, rtol=1e-9, atol=1e-12), (name, float(np.max(np.abs(mag - rmag))))
    live = (mag != 0) | (rmag != 0)
    ph_ok = _phase_close(got[..., 1::2], ref[..., 1::2], 1e-12)
    assert np.all(ph_ok | ~live), (name, int(np.sum(~ph_ok & live)))
