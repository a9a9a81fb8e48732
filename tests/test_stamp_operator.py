"""Device-stamp kernel (tsb_batch_stamp_dev -> generated tsb_stamp_staged / tsb_stamp) against the independent reference of
tests/stamp_ref.py: the dense system the reference holds after mat.Clear(); ckt.Stamp(status); mat.LoadGmin(gmin) on a
freshly set-up circuit.

CPU: the reference itself (hand-written rc companion system, linear operating points through numpy.linalg.solve, PULSE /
PWL values at their edges) and the generated stamp code compiled for the host (strict), bit for bit, on every bundled and
extra deck, seeded random decks and an n = 28 ladder, OP and transient, at source edge times and gmin on both sides of
the capacitor's 1e-12 floor.

GPU: both store paths at every block-size step, every word written and nothing else, a second trip of the grid-stride
loop, the strict build bit for bit, the fast build within a derived bound, processing order / device / uniform
parameters, refusals.  Every comparison of stamped values is on bits (signed zeros count)."""
import math

import numpy as np
import pytest

import parity_util as PU
import random_decks as RD
import stamp_host_emul as SH
import stamp_ref as R
from oracle import pin_numpy as P
from extra_decks import EXTRA

T, O = PU.T, PU.O
U = 2.0 ** -53                       # unit roundoff of binary64
GMINS = (0.0, 1e-13, 1e-12, 1e-9)    # LoadGmin off / on; the capacitor's OP conductance is max(Gmin, 1e-12)
N_INST = 19                          # instances per deck in the deck sweeps (draws of workloads.py)


def _deck_text(d):
    return d[0] if isinstance(d, tuple) else d


DECKS = dict(T.BUNDLED)
DECKS.update({name: text for name, (text, _) in EXTRA.items()})
DECKS.update({f"random{s}": _deck_text(RD.random_deck(s)) for s in (3, 8, 21)})
DECKS.update({f"random_active{s}": _deck_text(RD.random_active_deck(s)) for s in (1, 4, 6, 11)})
DECKS["rc_ladder26"] = RD.rc_ladder(26)                  # n = 28: the first order the runtime stamps with the direct kernel


def params_of(name, text, n):
    return PU.draws(name, T.Circuit.from_netlist(text), n)


def cases_of(deck):
    """(mode, time, dt, gmin): OP and transient at t = 0, a time between edges and up to four source edge times, two
    steps, every gmin."""
    ts = R.source_times(deck)
    times = [0.0, 1.25e-4] + [ts[k] for k in np.linspace(0, len(ts) - 1, min(4, len(ts))).astype(int)] if ts else [0.0, 1.25e-4]
    out = []
    for t in times:
        for g in GMINS:
            out.append((R.OP, t, 0.0, g))
            for dt in (2e-7, 1e-5):
                out.append((R.TRAN, t, dt, g))
    return out


def same_bits(x, y):
    """Equal as binary64 words; NaN against NaN counts as equal whatever the payload."""
    x, y = np.ascontiguousarray(x, dtype=np.float64), np.ascontiguousarray(y, dtype=np.float64)
    return bool(np.all((x.view(np.int64) == y.view(np.int64)) | (np.isnan(x) & np.isnan(y))))


def same_words(x, y):
    """Equal as binary64 words, NaN payloads included: for two outputs of the same device."""
    return np.array_equal(np.ascontiguousarray(x).view(np.int64), np.ascontiguousarray(y).view(np.int64))


def first_diff(x, y):
    bad = np.argwhere(~((x.view(np.int64) == y.view(np.int64)) | (np.isnan(x) & np.isnan(y))))
    if not len(bad):
        return None
    i = tuple(bad[0])
    return i, float(x[i]), float(y[i]), len(bad)


# ------------------------------------------------------------------------------------------------------ the reference
def test_rc_reference_is_the_companion_system(built):
    """rc.cir at (t, dt) in transient mode: G + C/dt on the capacitor's node, the source's incidence and its value
    5 sin(2 pi 1000 t) (Go's sine), and a fresh capacitor's charge1 = 0 on the right-hand side."""
    text = T.BUNDLED["rc"]
    deck = R.Deck(text)
    params = params_of("rc", text, 5)
    t, dt = 1.25e-4, 2e-7
    A, b, S, Sb = R.stamp_batch(deck, params, range(5), R.TRAN, t, dt, 0.0)[:4]
    g = 1.0 / params[("r1", 0)]
    geq = params[("c1", 0)] / dt
    ref = np.zeros((5, 3, 3))
    ref[:, 0, 0] = g; ref[:, 0, 1] = -g; ref[:, 1, 0] = -g; ref[:, 1, 1] = g + geq; ref[:, 2, 0] = 1.0; ref[:, 0, 2] = 1.0
    assert same_bits(A, ref)
    assert same_bits(b[:, :2], np.zeros((5, 2)))
    assert np.all(b[:, 2] == 0.0 + 5.0 * O.go_sin(2.0 * math.pi * 1000.0 * t + 0.0 * math.pi / 180.0))
    assert same_bits(S, np.abs(ref)) and same_bits(Sb, np.abs(b))


LINEAR = ["rr", "rc", "rl", "rlc", "idc", "ipulse", "ipwl", "isin", "vpulse", "vpwl", "transformer1", "transformer2", "transformer3"]


@pytest.mark.parametrize("name", LINEAR)
def test_reference_op_system_solves_to_the_oracle_operating_point(built, name):
    """For a linear deck the operating point is one solve of the OP system (gmin = 0, time 0): numpy.linalg.solve of the
    reference's A, b equals the oracle's operating point within the conditioning of A (kappa * eps)."""
    text = T.BUNDLED[name]
    deck = R.Deck(text)
    params = params_of(name, text, 6)
    A, b = R.stamp_batch(deck, params, range(6), R.OP, 0.0, 0.0, 0.0)[:2]
    x = np.linalg.solve(A, b[..., None])[..., 0]
    res = O.OracleCircuit(text).run(6, overrides=params, analysis=0)
    xo = res["wave"][:, 0, : deck.n]
    assert np.all(res["status"] == 0)
    kappa = np.linalg.cond(A)
    err = np.abs(x - xo).max(axis=1)
    assert np.all(err <= 8 * kappa * 2 * U * np.abs(xo).max(axis=1)), (name, err, kappa)


def test_source_values_at_edges_equal_a_hand_table(built):
    """PULSE(0 5 2ms 0.5ms 0.5ms 5ms 10ms) and PWL(0 0 2m 0 2.5m 3.3m 5m 3.3m 5.5m 0 10m 0): the value the stamp puts on the
    right-hand side at the delay, the ends of rise and flat top, the end of the fall, one and two periods later, and at
    every PWL breakpoint.  Rows: (time, value); every product here is exact or the hand table says how it rounds."""
    vp = R.Deck(T.BUNDLED["vpulse"])
    pulse = [(0.0, 0.0), (2e-3, 0.0), (2.25e-3, 0.0 + (5.0 - 0.0) * (2.25e-3 - 2e-3) / 0.5e-3), (2.5e-3, 5.0), (7.5e-3, 5.0),
             (7.75e-3, 5.0 - (5.0 - 0.0) * ((7.75e-3 - 2e-3) - 5.5e-3) / 0.5e-3), (8e-3, 0.0), (11e-3, 0.0), (12e-3, 0.0),
             (12.5e-3, 5.0), (22e-3, 0.0)]
    for t, v in pulse:
        b = R.stamp(vp, {}, R.TRAN, t, 1e-5, 0.0).b
        assert same_bits(b[-1], v), (t, b[-1], v)
    ip = R.Deck(T.BUNDLED["ipwl"])
    pwl = [(0.0, 0.0), (2e-3, 0.0), (2.5e-3, 3.3e-3), (3e-3, 3.3e-3), (5e-3, 3.3e-3), (5.5e-3, 0.0), (10e-3, 0.0), (20e-3, 0.0),
           (2.25e-3, 0.0 + ((3.3e-3 - 0.0) / (2.5e-3 - 2e-3)) * (2.25e-3 - 2e-3))]
    for t, v in pwl:
        b = R.stamp(ip, {}, R.OP, t, 0.0, 0.0).b
        assert same_bits(b[0], 0.0 + v), (t, b[0], v)     # isource.go: AddRHS(n1, +I) onto a cleared 0.0


def test_pin_go_math_equals_the_oracle(built):
    """The pin's restatements of Go's math.Sin and math.Pow (oracle/pin_numpy.py: go_sin, go_pow, written from sin.go and
    pow.go) equal the oracle's (orc_go_sin, orc_go_pow) bit for bit: fractional, integer and +-0.5 exponents, special
    values, sines up to and past many periods."""
    rng = np.random.default_rng(5)
    L = O.lib()
    xs = [float(x) for x in np.concatenate([rng.uniform(0.01, 40.0, 200), 10.0 ** rng.uniform(-8, 8, 50), -rng.uniform(0.1, 9, 20)])]
    nan, inf = float("nan"), float("inf")
    for x in xs + [0.0, -0.0, 1.0, -1.0, inf, -inf, nan]:
        for y in (0.5, -0.5, 1.0, 2.0, -2.0, 3.0, -7.0, 0.1, 0.15, 0.33, -0.75, 2.4, 3.9, 0.0, inf, -inf):
            g, o = P.go_pow(x, y), L.orc_go_pow(x, y)
            assert R.bits(g) == R.bits(o) or (g != g and o != o), (x, y, g, o)
    for t in list(rng.uniform(-40.0, 40.0, 500)) + [k * math.pi / 4 for k in range(-40, 41)] + [0.0, -0.0, 1e6 + 0.5, -3e8]:
        assert R.bits(P.go_sin(float(t))) == R.bits(O.go_sin(float(t))), t


# ------------------------------------------------------------------------------------ the generated code on the host
@pytest.mark.parametrize("name", sorted(DECKS))
def test_host_compiled_stamp_kernel_equals_the_reference(built, tmp_path_factory, name):
    """tsb_stamp of the generated source, compiled for the host (strict arithmetic, glibc exp / log), against the reference
    on the same draws: every case of cases_of, every entry, bit for bit."""
    text = DECKS[name]
    deck = R.Deck(text)
    params = params_of(name, text, N_INST)
    cases = cases_of(deck)
    out = SH.run(text, params, cases, str(tmp_path_factory.mktemp("stamp")))
    assert out[0][0].shape[1] == deck.n
    for (A, b), case in zip(out, cases):
        Ar, br = R.stamp_batch(deck, params, range(N_INST), *case)[:2]
        assert same_bits(A, Ar), (name, case, first_diff(A, Ar))
        assert same_bits(b, br), (name, case, first_diff(b, br))


# -------------------------------------------------------------------------------------------------------------- GPU
SENTINEL = 0x7FF8DEADBEEFCAFE       # a quiet NaN with a recognisable payload
GUARD = 64


class GpuStamper:
    """One batch of a deck on the GPU; every call fills A and b with SENTINEL, leaves a GUARD-word tail after each, stamps,
    and checks that every in-range word was written and no tail word was."""

    def __init__(self, ctx, text, params, n_inst=None, order=None, dev_params=False, uniform=None):
        import torch
        self.torch = torch
        self.ctx = ctx
        self.ckt = T.Circuit.from_netlist(text, ctx)
        self.n = self.ckt.n
        self.n_inst = n_inst if n_inst is not None else len(next(iter(params.values())))
        self.b = self.ckt.batch(self.n_inst)
        self._keep = []
        for (d, p), v in params.items():
            v = np.ascontiguousarray(v[: self.n_inst], dtype=np.float64)
            if dev_params:
                t = torch.from_numpy(v).cuda()
                self._keep.append(t)
                self.b.set_param(d, p, t)
            else:
                self.b.set_param(d, p, v)
        for (d, p), v in (uniform or {}).items():
            self.b.set_param(d, p, float(v))
        if order is not None:
            self.b.set_order(order)
        na, nb = self.n_inst * self.n * self.n, self.n_inst * self.n
        self.dA = torch.empty(na + GUARD, dtype=torch.int64, device="cuda")
        self.dB = torch.empty(nb + GUARD, dtype=torch.int64, device="cuda")

    def __call__(self, mode, time, dt, gmin, strict=True):
        torch = self.torch
        self.dA.fill_(SENTINEL)
        self.dB.fill_(SENTINEL)
        torch.cuda.synchronize()
        self.b.stamp_dev(mode, time, dt, gmin, self.dA.data_ptr(), self.dB.data_ptr(), opts=T.default_opts(strict_fp=1 if strict else 0))
        self.b.sync()
        torch.cuda.synchronize()
        na, nb = self.n_inst * self.n * self.n, self.n_inst * self.n
        A, B = self.dA.cpu().numpy(), self.dB.cpu().numpy()
        assert np.all(A[na:] == SENTINEL) and np.all(B[nb:] == SENTINEL), "a word past the end of A or b was written"
        unwritten = int(np.count_nonzero(A[:na] == SENTINEL)) + int(np.count_nonzero(B[:nb] == SENTINEL))
        assert unwritten == 0, f"{unwritten} words of A / b not written"
        return A[:na].view(np.float64).reshape(self.n_inst, self.n, self.n), B[:nb].view(np.float64).reshape(self.n_inst, self.n)


_DEVICE_REFS = {}


def device_reference(name):
    """(deck, params, cases, results, table) of DECKS[name] with the device's exp / log, computed once per session (the
    strict and the fast test share it)."""
    if name not in _DEVICE_REFS:
        text = DECKS[name]
        deck = R.Deck(text)
        params = params_of(name, text, N_INST)
        cases = cases_of(deck)
        refs, table = device_gomath_reference(deck, params, range(N_INST), cases)
        _DEVICE_REFS[name] = (deck, params, cases, refs, table)
    return _DEVICE_REFS[name]


def device_gomath_reference(deck, params, idx, cases):
    """Reference results of `cases` with the CUDA math library's exp / log (evaluated by torch on the device) in place of
    the host's: iterated until every argument the stamps reach has its device value (an argument can depend on an earlier
    result: the BJT's vbe = Nf Vt log(1e-3 / Ies) feeds exp(vbe / (Nf Vt))).  Returns (results per case, table)."""
    import torch
    table = {}
    while True:
        lm = R.Libm(table)
        refs = [R.stamp_batch(deck, params, idx, *c, libm=lm) for c in cases]
        missing = {}
        for nm, x in lm.calls:
            if (nm, R.bits(x)) not in table:
                missing[(nm, R.bits(x))] = x
        if not missing:
            return refs, table
        for nm in ("exp", "log"):
            keys = [k for k in missing if k[0] == nm]
            if keys:
                y = getattr(torch, nm)(torch.tensor([missing[k] for k in keys], dtype=torch.float64, device="cuda")).cpu().numpy()
                table.update(zip(keys, (float(v) for v in y)))


def assert_libm_within_one_ulp(table):
    """The only arithmetic the device may do differently from the reference's host: CUDA's exp and log are documented
    within 1 ulp of the exact value (CUDA C++ Programming Guide, double-precision functions), glibc's are correctly
    rounded on these arguments; two such values of one argument are at most 1 ulp apart."""
    for (nm, xb), v in table.items():
        x = struct_float(xb)
        h = R.host_exp(x) if nm == "exp" else math.log(x)
        if math.isfinite(h):
            assert abs(R.bits(v) - R.bits(h)) <= 1, (nm, x, v, h)
        else:
            assert v == h, (nm, x, v, h)


def struct_float(b):
    return float(np.array([b], dtype=np.int64).view(np.float64)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(DECKS))
def test_strict_build_equals_the_reference_bit_for_bit(ctx, tmp_path_factory, name):
    """Strict build, every case of cases_of (PULSE edges, PWL breakpoints, k * per, SIN quarter periods; OP and transient;
    gmin 0, 1e-13, 1e-12, 1e-9).

    Bit for bit against the reference evaluated with the device's own exp / log.  Derivation of why nothing looser is
    needed: the strict build performs exactly the reference's IEEE operations (no contraction, correctly rounded
    quotients and square roots, Go's sine and pow restated operation for operation), so the only values that can differ
    are the results of exp and log at arguments where they are not exact (the BJT's initial operating point and its
    junction exponentials, Level 2 mobility degradation through Go's Pow = Exp(yf Log x) * x^yi).  Those results are
    taken from the CUDA math library itself, checked to lie within its documented 1 ulp of glibc's, and every later
    operation of the device's stamp is then reproduced exactly by the reference — the documented ulp error propagated
    through the stamp, with nothing left for a tolerance to absorb.

    Also: the GPU equals the host-compiled stamp code bit for bit wherever the two math libraries agree (every deck whose
    table is empty or identical), and on the others each equals the reference evaluated with its own library."""
    text = DECKS[name]
    deck, params, cases, refs, table = device_reference(name)
    assert_libm_within_one_ulp(table)
    g = GpuStamper(ctx, text, params)
    host = SH.run(text, params, cases, str(tmp_path_factory.mktemp("stamp")))
    libm_agrees = all(v == (R.host_exp(struct_float(xb)) if nm == "exp" else math.log(struct_float(xb))) for (nm, xb), v in table.items())
    for case, (Ar, br, *_), (Ah, bh) in zip(cases, refs, host):
        A, b = g(*case)
        assert same_bits(A, Ar), (name, case, first_diff(A, Ar))
        assert same_bits(b, br), (name, case, first_diff(b, br))
        if libm_agrees:
            assert same_bits(A, Ah) and same_bits(b, bh), (name, case)


def _ill_conditioned_under_fast(text):
    """A BJT, or a MOSFET of Level 2 / 3 (see test_fast_build_within_its_derived_bound)."""
    return any(r.kind == P.K_Q or (r.kind == P.K_M and int(r.ip[0]) in (2, 3)) for r in O.OracleCircuit(text).plan.devices)


FAST_DECKS = sorted(n for n, text in DECKS.items() if not _ill_conditioned_under_fast(text))


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAST_DECKS)
def test_fast_build_within_its_derived_bound(ctx, name):
    """Fast build: |A_fast - A_ref| <= c * u * S + 2 u * P componentwise (S = sum of |contributions| into the entry, P = sum
    of |products| that feed a cancelling add inside a contribution: stamp_ref._products), b likewise, u = 2^-53, with c
    derived from the fast build's liberties (DESIGN 5.3):

      * a quotient x / y becomes x * r with r the hardware-seeded reciprocal after its correction step (x / dt: r = 1/dt
        formed once per call; x / y in the models: tsb_qrcp) — r is within 1 ulp (2u relative) of 1/y, the product adds
        one rounding (u): within 3u of the exact quotient, so within 4u of the strict build's correctly rounded one;
      * a contribution passes at most two such quotients in series on these decks (the diode's geq = Tt * (Is / nVt) / dt,
        a Meyer capacitance / dt): 8u;
      * FMA contraction drops the rounding of a product feeding an add: at most u * |product| per contracted pair.  Where
        all terms of the add have one sign the product is at most the contribution: the diode's Is / nVt + 1e-12 and
        gd + Tt gd / dt, the factors 1 + lambda vds, the Meyer capacitances cgate / 2 + cgso, the sine polynomial (whose
        terms are small corrections to z; the Cody-Waite products y * PI4A, y * PI4B are exact) — at most 4u per
        contribution on these decks.  Where the add can cancel — p0 + p1 sin of a SIN source, a + slope (t - t1) of a PWL
        source, the Level 1 MOSFET's ieq and linear-region gds — the dropped roundings are bounded by u * P, and the
        change they make to the rounding of the add by u * P again: 2u * P.  The other contributions of the included
        devices (R, C, L, K, core L, DC and PULSE sources) have no product feeding an add: 1 / (R * 1), C * 1 / dt,
        L / dt, M / dt, L0 / dt with L0 = mu0 N^2 A / len, and the PULSE ramp (v2 - v1) t / rise is a quotient;
      * hoisted quotients are the same operation on the same operands: no change;
      * both builds add the m contributions of an entry in the same order; each of the m - 1 partial sums is rounded from
        operands that differ by the above, which adds at most 2u * S per addition.

    Hence c = 12 + 2 (m - 1), m counted per entry by the reference.  Decks left out (_ill_conditioned_under_fast: every
    deck, bundled, extra or random, that has one of these devices, and no other): a BJT (a 4u change of the exponent's
    argument Vbe / (Nf Vt) ~ 25 is amplified 25-fold by exp) and a Level 2 / 3 MOSFET (conductances are 1e-6 forward
    differences of the drain current, which amplify its last bit a million-fold): there the liberties are not small
    against S, and those decks are held to the strict build only."""
    text = DECKS[name]
    deck, params, cases, refs, _ = device_reference(name)
    g = GpuStamper(ctx, text, params)
    worst = 0.0
    for case, r in zip(cases, refs):
        A, b = g(*case, strict=False)
        for got, want, S, m, Pp in ((A, r.A, r.S, r.m, r.P), (b, r.b, r.Sb, r.mb, r.Pb)):
            c = 12 + 2 * np.maximum(m - 1, 0)
            err = np.abs(got - want)
            bound = c * U * S + 2 * U * Pp
            ok = err <= bound
            assert np.all(ok), (name, case, np.argwhere(~ok)[0].tolist(), float(err[~ok][0]), float(bound[~ok][0]))
            with np.errstate(all="ignore"):
                worst = max(worst, float(np.where(S > 0, err / (U * S), 0.0).max()))
    print(f"{name}: worst |A_fast - A_ref| / (u S) = {worst:.2f}")


# block-size steps of the staged kernel: threads = largest multiple of 32 <= 128 with threads * ((n*n + n) | 1) doubles in
# 200 KB; below 32 the runtime stamps with the direct kernel
def _staged_threads(n):
    return min((200 * 1024 // (((n * n + n) | 1) * 8)) // 32 * 32, 128)


def launched_stamp_kernels(call, tmp_path):
    """Runs `call` under torch.profiler (CUDA activities) and returns (kernel, grid x, block x) of every tsb_stamp /
    tsb_stamp_staged launch it made, from the exported trace: what the runtime really chose.  `call` runs once before
    (kernel compilation and module loading stay outside the profiled window).  `call` makes one launch; CUDA activity
    tracing has been seen to miss a short kernel right after a session starts, so a session whose trace holds no stamp
    kernel record is repeated, up to three sessions."""
    import json
    import torch
    from torch.profiler import ProfilerActivity, profile
    call()
    for attempt in range(3):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        path = str(tmp_path / f"stamp_trace{attempt}.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            evs = [e for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel" and e.get("name") in ("tsb_stamp", "tsb_stamp_staged")]
        if evs:
            return [(e["name"], int(e["args"]["grid"][0]), int(e["args"]["block"][0])) for e in evs]
    raise AssertionError("torch.profiler recorded no stamp kernel in three sessions: the launch cannot be checked")


LADDERS = {13: RD.rc_ladder(11), 14: RD.rlc_ladder(4), 16: RD.rc_ladder(14), 20: RD.rlc_ladder(6), 27: RD.rc_ladder(25),
           28: RD.rc_ladder(26), 34: RD.rc_ladder(32)}


def test_block_size_steps_of_the_ladders(built):
    """The ladders below sit at the steps of the staged kernel's block size, and 28 / 34 on the direct kernel."""
    want = {13: 128, 14: 96, 16: 64, 20: 32, 27: 32, 28: 0, 34: 0}
    for n, text in LADDERS.items():
        assert T.Circuit.from_netlist(text).n == n
        assert _staged_threads(n) == want[n], (n, _staged_threads(n))


@pytest.mark.gpu
@pytest.mark.parametrize("n", sorted(LADDERS))
def test_staged_and_direct_kernels_write_the_same_bits(ctx, monkeypatch, tmp_path, n):
    """TSB_STAMP_DIRECT=1 forces the direct kernel (tsb_stamp); without it the runtime picks the staged one where it fits
    (n <= 27).  Same inputs, same bits, in both builds, on a batch that ends in a partial block; and the strict output
    against the reference on the first and the last block's instances.  n = 28 / 34 have the direct kernel only: there the
    strict build against the reference is the test.  Which kernel ran, with how many threads per block, is read back from
    torch.profiler."""
    text = LADDERS[n]
    deck = R.Deck(text)
    n_inst = 3 * max(_staged_threads(n), 32) + 5
    params = params_of(f"ladder{n}", text, n_inst)
    g = GpuStamper(ctx, text, params)
    threads = _staged_threads(n)
    staged_launch = ("tsb_stamp_staged", -(-n_inst // threads), threads) if threads >= 32 else ("tsb_stamp", -(-n_inst // 128), 128)
    monkeypatch.delenv("TSB_STAMP_DIRECT", raising=False)
    launches = launched_stamp_kernels(lambda: g(R.OP, 0.0, 0.0, 0.0), tmp_path)
    assert launches == [staged_launch], launches
    monkeypatch.setenv("TSB_STAMP_DIRECT", "1")
    launches = launched_stamp_kernels(lambda: g(R.OP, 0.0, 0.0, 0.0), tmp_path)
    assert launches == [("tsb_stamp", -(-n_inst // 128), 128)], launches
    for case in [(R.TRAN, 2.5e-4, 2e-7, 0.0), (R.OP, 0.0, 0.0, 1e-9)]:
        builds = (True, False) if _staged_threads(n) >= 32 else (True,)
        monkeypatch.delenv("TSB_STAMP_DIRECT", raising=False)
        staged = [g(*case, strict=s) for s in builds]
        monkeypatch.setenv("TSB_STAMP_DIRECT", "1")
        direct = [g(*case, strict=s) for s in builds]
        monkeypatch.delenv("TSB_STAMP_DIRECT")
        for (As, bs), (Ad, bd) in zip(staged, direct):
            assert same_words(As, Ad) and same_words(bs, bd), (n, case, first_diff(As, Ad))
        idx = list(range(8)) + list(range(n_inst - 8, n_inst))
        Ar, br = R.stamp_batch(deck, params, idx, *case)[:2]
        As, bs = staged[0]
        assert same_bits(As[idx], Ar) and same_bits(bs[idx], br), (n, case, first_diff(As[idx], Ar))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 20])
def test_every_word_written_at_batch_edges_and_a_second_grid_stride_trip(ctx, tmp_path, n):
    """Batch sizes 1, 31, 32, 33, block - 1, block, block + 1 and sms * 32 * block + 33 (the grid is capped at sms * 32
    blocks, so the last size makes the loop take a second trip, which ends in a partial block).  Every in-range word is
    written and no word past the end (GpuStamper); the reference agrees on every instance of the small batches and on a
    sample of the large one taken from the first trip, around the trip boundary and from the last partial block.  The
    launch of the large batch is read back from torch.profiler: the staged kernel, `block` threads, sms * 32 blocks."""
    text = T.BUNDLED["rc"] if n == 3 else LADDERS[20]
    deck = R.Deck(text)
    block = _staged_threads(n)
    resident = ctx.sm_count * 32 * block
    big = resident + 33
    params = params_of(f"edges{n}", text, big)
    case = (R.TRAN, 1.25e-4, 2e-7, 1e-12)
    for size in sorted({1, 31, 32, 33, block - 1, block, block + 1}):
        A, b = GpuStamper(ctx, text, params, n_inst=size)(*case)
        Ar, br = R.stamp_batch(deck, params, range(size), *case)[:2]
        assert same_bits(A, Ar) and same_bits(b, br), (n, size, first_diff(A, Ar))
    g = GpuStamper(ctx, text, params, n_inst=big)
    out = []
    launches = launched_stamp_kernels(lambda: out.append(g(*case)), tmp_path)
    assert launches == [("tsb_stamp_staged", ctx.sm_count * 32, block)], launches
    A, b = out[0]
    sample = sorted(set(list(range(40)) + list(range(resident - 40, big)) + list(range(resident // 2, resident // 2 + 8))))
    Ar, br = R.stamp_batch(deck, params, sample, *case)[:2]
    assert same_bits(A[sample], Ar) and same_bits(b[sample], br), (n, first_diff(A[sample], Ar))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rlc", "diode4", "mosfet1", "transformer2", "bjt2"])
def test_order_device_and_uniform_parameters_give_the_same_bits(ctx, name):
    """A processing order (Batch.set_order) leaves the output bit-identical and in caller order; parameters handed over as
    CUDA tensors (tsb_batch_set_param_dev) give the bits of host arrays; a parameter set uniform
    (tsb_batch_set_param_uniform: a specialised kernel reads it as a constant) gives the bits of a varying array holding
    the same value."""
    text = T.BUNDLED[name]
    n_inst = 301
    params = params_of(name, text, n_inst)
    case = (R.TRAN, 3e-6, 1e-7, 1e-12)
    for strict in (True, False):
        A0, b0 = GpuStamper(ctx, text, params)(*case, strict=strict)
        perm = np.random.default_rng(3).permutation(n_inst)
        A1, b1 = GpuStamper(ctx, text, params, order=perm)(*case, strict=strict)
        assert same_words(A1, A0) and same_words(b1, b0), (name, strict, "order")
        A2, b2 = GpuStamper(ctx, text, params, dev_params=True)(*case, strict=strict)
        assert same_words(A2, A0) and same_words(b2, b0), (name, strict, "device parameters")
        key = next(iter(params))
        val = float(params[key][7])
        varying = dict(params)
        varying[key] = np.full(n_inst, val)
        rest = {k: v for k, v in params.items() if k != key}
        A3, b3 = GpuStamper(ctx, text, varying)(*case, strict=strict)
        A4, b4 = GpuStamper(ctx, text, rest, n_inst=n_inst, uniform={key: val})(*case, strict=strict)
        assert same_words(A4, A3) and same_words(b4, b3), (name, strict, "uniform")


@pytest.mark.gpu
def test_refusals_launch_nothing(ctx):
    """TSB_E_INVALID before any launch: a mode other than OP / transient, a null A or b, and a transient stamp with a step
    that is not > 0 (0, negative, NaN) — the fast build would stamp C/dt as 0 there (it multiplies by 1/dt, which the
    kernel only forms for dt > 0), the strict build as +-Inf or a negative conductance.  An OP stamp ignores dt."""
    import torch
    text = T.BUNDLED["rc"]
    params = params_of("rc", text, 40)
    ckt = T.Circuit.from_netlist(text, ctx)
    b = ckt.batch(40)
    for (d, p), v in params.items():
        b.set_param(d, p, v)
    dA = torch.zeros(40 * 9, dtype=torch.float64, device="cuda")
    dB = torch.zeros(40 * 3, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    bad = [(2, 0.0, 1e-6, dA.data_ptr(), dB.data_ptr()), (-1, 0.0, 1e-6, dA.data_ptr(), dB.data_ptr()),
           (R.OP, 0.0, 0.0, 0, dB.data_ptr()), (R.OP, 0.0, 0.0, dA.data_ptr(), 0)]
    bad += [(R.TRAN, 1e-4, dt, dA.data_ptr(), dB.data_ptr()) for dt in (0.0, -1e-6, float("nan"))]
    for strict in (0, 1):
        for mode, t, dt, pa, pb in bad:
            before = ctx.launch_count
            with pytest.raises(T.TsbError):
                b.stamp_dev(mode, t, dt, 0.0, pa, pb, opts=T.default_opts(strict_fp=strict))
            assert ctx.launch_count == before, (mode, dt, strict)
        before = ctx.launch_count
        b.stamp_dev(R.OP, 0.0, 0.0, 0.0, dA.data_ptr(), dB.data_ptr(), opts=T.default_opts(strict_fp=strict))
        b.sync()
        assert ctx.launch_count == before + 1
