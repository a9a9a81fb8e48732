"""Fourier analysis on the device (TSB_OUT_FOUR, the SPICE .four card; include/tspice_b200.h).

* CPU: the restatement (tests/four_ref.py) on series whose coefficients have closed forms (dyadic polylines sampled at and
  between grid points, a cosine and a sine sampled on the grid), grid points on a row and several in one segment, windows
  outside the rows, NaN samples, t_end = +inf, G = 2H + 1, and a scalar loop as an independent restatement; the table's
  validation; the kernel source with and without a table; the analytic pin of the isin deck on the oracle's rows.
* CPU, device source on the host (tests/four_host_emul.py over tests/host_emul.py, strict configuration): the sink's
  Fourier code is bit for bit the restatement applied to the same run's rows (rc, rlc, isin, diode2).
* GPU: bit identity with the restatement on the run's own rows for every bundled deck driven by a sine, in both builds;
  everything that must not move a bit (processing order, lane refill, shared time grid, waveform capacity, statistics,
  measurements, grid output, a job over two contexts, the auto mapping); agreement with the oracle's rows; refusals."""
import math
import re
import tempfile

import numpy as np
import pytest

import four_ref as F
import meas_ref as R
import parity_util as PU
from random_decks import rc_ladder

T = PU.T
INF = math.inf
NAN = math.nan


def Fo(column=1, freq=1.0, n_harm=1, n_grid=4, t_end=INF):
    return T.four(column, freq, n_harm=n_harm, n_grid=n_grid, t_end=t_end)


def _scalar(x, y, f, tstop):
    """Independent restatement: plain Python floats (IEEE doubles, one rounding per operation), one sample at a time."""
    Tp = 1.0 / f.freq
    e = tstop if f.t_end == INF else f.t_end
    s, dt, G = e - Tp, Tp / f.n_grid, f.n_grid
    ys = []
    for k in range(G):
        tk = s + float(k) * dt
        j = next((r for r in range(len(x)) if x[r] >= tk), None)
        if j is None or (j == 0 and x[0] != tk):
            return [NAN] * (1 + 2 * f.n_harm)
        ys.append(y[j] if x[j] == tk else y[j - 1] + ((tk - x[j - 1]) / (x[j] - x[j - 1])) * (y[j] - y[j - 1]))
    out = [0.0]
    for v in ys:
        out[0] = out[0] + v
    out[0] = out[0] / G
    for h in range(1, f.n_harm + 1):
        ca = sb = 0.0
        for k, v in enumerate(ys):
            ca = ca + v * math.cos(2.0 * math.pi * ((h * k) % G) / G)
            sb = sb + v * math.sin(2.0 * math.pi * ((h * k) % G) / G)
        out += [(2.0 * ca) / G, (2.0 * sb) / G]
    return out


# ---- restatement ------------------------------------------------------------------------------------------------------
def test_twiddles_g4():
    """libm's cos(pi / 2) and sin(pi) are 6.1e-17 and 1.2e-16, not 0: the closed forms below hold to that size."""
    c, s = F.twiddles(4)
    assert c[0] == 1.0 and c[2] == -1.0 and s[1] == 1.0 and s[3] == -1.0 and s[0] == 0.0
    assert max(abs(c[1]), abs(c[3]), abs(s[2])) < 2e-16


def test_polyline_at_and_between_grid_points():
    """Period 1 ending at 4: tau = 3, 3.25, 3.5, 3.75.  Rows every 0.5 of a dyadic polyline: tau = 3 and 3.5 are rows,
    3.25 and 3.75 are interpolated, and every sample is exact."""
    x = np.arange(0, 9) * 0.5
    y = np.array([0.0, 1.0, -2.0, 3.0, 0.5, -1.5, 4.0, 2.0, 1.0])
    f = Fo(t_end=4.0)
    yk = F.samples(x, y, F.grid(f, 4.0))
    assert list(F.grid(f, 4.0)) == [3.0, 3.25, 3.5, 3.75]
    assert list(yk) == [4.0, 3.0, 2.0, 1.5]
    got = F.fourier(x, y, f, 4.0)
    assert got[0] == (4.0 + 3.0 + 2.0 + 1.5) / 4                # a0: the sum of dyadic samples is exact
    assert abs(got[1] - (4.0 - 2.0) / 2) < 1e-15                # A_1 = (y0 - y2) / 2
    assert abs(got[2] - (3.0 - 1.5) / 2) < 1e-15                # B_1 = (y1 - y3) / 2
    assert R.same_bits(got, _scalar(list(x), list(y), f, 4.0))


def test_several_grid_points_in_one_segment():
    x, y = [0.0, 2.0, 4.0], [1.0, 5.0, 9.0]                     # y = 2x + 1: the samples are exact
    f = Fo(t_end=4.0)
    assert list(F.samples(x, y, F.grid(f, 4.0))) == [7.0, 7.5, 8.0, 8.5]
    got = F.fourier(x, y, f, 4.0)
    assert got[0] == 7.75 and abs(got[1] + 0.5) < 1e-15 and abs(got[2] + 0.5) < 1e-15
    assert R.same_bits(got, _scalar(x, y, f, 4.0))


@pytest.mark.parametrize("h0, G", [(1, 8), (3, 8), (2, 5), (4, 16)])
def test_cosine_and_sine_on_the_grid(h0, G):
    """y = 0.75 + 1.5 cos(2 pi h0 (t - s)) - 0.5 sin(2 pi h0 (t - s)) sampled exactly at the grid times (and one row after):
    a0 = 0.75, A_h0 = 1.5, B_h0 = -0.5, every other harmonic 0, to rounding."""
    H = min(G // 2 - (G % 2 == 0), 4) if G > 2 else 1
    H = max(1, min(H, (G - 1) // 2))
    f = Fo(n_harm=H, n_grid=G, t_end=2.0)
    tau = F.grid(f, 2.0)
    x = np.concatenate([tau, [2.0]])
    ph = 2 * np.pi * h0 * (x - 1.0)
    y = 0.75 + 1.5 * np.cos(ph) - 0.5 * np.sin(ph)
    got = F.fourier(x, y, f, 2.0)
    want = np.zeros(1 + 2 * H)
    want[0] = 0.75
    if h0 <= H:
        want[2 * h0 - 1], want[2 * h0] = 1.5, -0.5
    assert np.max(np.abs(got - want)) < 1e-14, (got, want)
    assert R.same_bits(got, _scalar(list(x), list(y), f, 2.0))


def test_window_outside_the_rows_and_nan_samples():
    x, y = list(np.arange(0, 9) * 0.5), [0.0, 1.0, -2.0, 3.0, 0.5, -1.5, 4.0, 2.0, 1.0]
    f = Fo(t_end=4.0)
    assert np.isnan(F.fourier(x[7:], y[7:], f, 4.0)).all()                  # starts at 3.5 > tau_0 = 3
    assert np.isnan(F.fourier(x[:8], y[:8], f, 4.0)).all()                  # ends at 3.5 < tau_3 = 3.75
    assert not np.isnan(F.fourier(x[6:], y[6:], f, 4.0)).any()              # starts at tau_0 exactly
    assert np.isnan(F.fourier(x, y, Fo(t_end=4.5), 4.0)).all()              # tau_3 = 4.25 > x_last = 4
    yn = list(y)
    yn[7] = NAN                                                             # row 3.5 is a sample
    assert np.isnan(F.fourier(x, yn, f, 4.0)).all()
    yn = list(y)
    yn[1] = NAN                                                             # before the window: no effect
    assert R.same_bits(F.fourier(x, yn, f, 4.0), F.fourier(x, y, f, 4.0))
    assert np.isnan(F.fourier([], [], f, 4.0)).all()


def test_t_end_inf_is_tstop_and_smallest_grid():
    x = list(np.arange(0, 9) * 0.5)
    y = [0.0, 1.0, -2.0, 3.0, 0.5, -1.5, 4.0, 2.0, 1.0]
    assert R.same_bits(F.fourier(x, y, Fo(t_end=INF), 4.0), F.fourier(x, y, Fo(t_end=4.0), 4.0))
    f = Fo(n_harm=2, n_grid=5, t_end=4.0)                                   # G = 2H + 1
    got = F.fourier(x, y, f, 4.0)
    assert got.shape == (5,) and np.isfinite(got).all()
    assert R.same_bits(got, _scalar(x, y, f, 4.0))


def test_restatement_matches_scalar_loop_on_random_rows():
    rng = np.random.default_rng(3)
    x = np.cumsum(rng.uniform(1e-6, 3e-5, 400))
    y = np.sin(2 * np.pi * 1e3 * x) + 0.1 * rng.standard_normal(400)
    f = T.four(1, 1e3, n_harm=5, n_grid=37, t_end=x[-1] * 0.9)
    assert R.same_bits(F.fourier(x, y, f, x[-1]), _scalar(list(x), list(y), f, x[-1]))


# ---- validation and kernel source (host-only plans) -------------------------------------------------------------------
def _host_batch(deck="rc"):
    return T.Circuit.from_netlist(T.BUNDLED[deck]).batch(2)


@pytest.mark.parametrize("bad", [
    dict(column=0), dict(n_harm=0), dict(n_harm=33), dict(n_harm=4, n_grid=8), dict(n_grid=65537), dict(freq=0.0),
    dict(freq=-1e3), dict(freq=INF), dict(freq=NAN), dict(t_end=NAN), dict(t_end=-INF),
])
def test_set_fourier_refuses(bad, built):
    kw = dict(column=1, freq=1e3, n_harm=9, n_grid=200, t_end=INF)
    kw.update(bad)
    b = _host_batch()
    b.set_fourier([T.four(2, 1e3, n_harm=3)])
    b.kernel_variant(four=True)
    before = b.kernel_source(T.default_opts(min_blocks=2))
    with pytest.raises(T.TsbError):
        b.set_fourier([T.Four(kw["column"], kw["n_harm"], kw["n_grid"], kw["freq"], kw["t_end"])])
    assert b.kernel_source(T.default_opts(min_blocks=2)) == before       # no change of state on refusal


def test_set_fourier_limits(built):
    b = _host_batch()
    b.set_fourier([T.four(1, 1e3)] * 8)
    with pytest.raises(T.TsbError):
        b.set_fourier([T.four(1, 1e3)] * 9)
    b.set_fourier([T.four(1, 1e3, n_harm=32, n_grid=65), T.four(1, 1e3, n_harm=1, n_grid=65536, t_end=1e-3)])
    b.set_fourier([])


def _strip_four(src):
    """The source without the Fourier table's defines and `#if TSB_FOUR` blocks."""
    out, depth = [], 0
    for line in src.split("\n"):
        if depth == 0 and (line.startswith("#if TSB_FOUR") or line.startswith("#define TSB_FOUR")):
            depth = 1 if line.startswith("#if") else 0
            continue
        if depth:
            depth += line.startswith("#if") - line.startswith("#endif")
            continue
        out.append(line)
    return "\n".join(out)


@pytest.mark.parametrize("meas", [False, True], ids=["plain", "with_meas"])
def test_kernel_source_with_and_without_table(meas, built):
    """Without a Fourier table the kernels are generated from the text they had before the feature (no TSB_FOUR line at
    all); with one, the source is that text plus the table's defines and the `#if TSB_FOUR` blocks."""
    for deck in ("rc", "rlc", "diode2"):
        b = _host_batch(deck)
        opts = T.default_opts(strict_fp=1, min_blocks=2)
        if meas:
            b.set_measures([T.meas(T.MEAS_MAX, 1), T.meas(T.MEAS_RMS, 2)])
        b.kernel_variant(meas=meas)
        plain, key0 = b.kernel_source(opts), b.kernel_key(opts)
        assert "TSB_FOUR" not in plain
        b.set_fourier([T.four(2, 1e3), T.four(1, 500.0, n_harm=3, n_grid=64, t_end=2e-3)])
        assert b.kernel_source(opts) == plain                   # a table alone selects nothing
        b.kernel_variant(meas=meas, four=True)
        src, key = b.kernel_source(opts), b.kernel_key(opts)
        assert "#define TSB_FOUR 2\n#define TSB_FOUR_SPEC {2, 9}, {1, 3}\n" in src and key != key0
        assert _strip_four(src) == plain
        b.set_fourier([T.four(2, 2e3, n_grid=100), T.four(1, 50.0, n_harm=3, n_grid=640, t_end=INF)])
        assert b.kernel_key(opts) == key                        # frequency, grid and window are run-time arguments
        b.set_fourier([T.four(2, 1e3, n_harm=8), T.four(1, 500.0, n_harm=3)])
        assert b.kernel_key(opts) != key


def test_fourier_summary():
    A1, B1, A2, B2 = 0.0, 2.0, 0.3, 0.4
    coeffs = np.array([[0.5], [A1], [B1], [A2], [B2]])
    s = T.fourier_summary(coeffs, [T.four(1, 1e3, n_harm=2)])[0]
    assert s["a0"][0] == 0.5 and s["M"][:, 0].tolist() == [2.0, 0.5]
    assert s["phase_deg"][0, 0] == 0.0 and abs(s["phase_deg"][1, 0] - math.degrees(math.atan2(0.3, 0.4))) < 1e-12
    assert abs(s["thd"][0] - 0.25) < 1e-15


# ---- analytic pin on the oracle's rows --------------------------------------------------------------------------------
def isin_pin(x, c, amp=2.0):
    """isin: a 2 mA, 1 kHz sine into 1 kOhm, window = the last period [2 ms, 3 ms], H = 9, G = 200; c are the coefficients
    of V(n1) (amp = 2 V) or of I(R1) (amp = 2 mA, whatever R1 is).

    The reference evaluates a source at the start of the step and stores the solution at its end (SURVEY Q2), so row r
    holds 2 sin(2 pi f x_{r-1}).  Where the rows are equally spaced (h) that is the sine z(t) = 2 sin(2 pi f (t - h))
    sampled at the rows: a phase shift, not a change of amplitude (amp = 2 V here; the bound scales with amp).  The one segment that is not (the last step, clamped to
    tstop) moves its row off z by at most 2 (2 pi f) |h_r - h| (z is Lipschitz).  The samples y_k interpolate the rows
    linearly, so |y_k - z(tau_k)| <= emax = h^2 / 8 max|z''| + 2 (2 pi f) max_r |h_r - h|, max|z''| = 2 (2 pi f)^2.
    Parseval on the G-point grid, sum e_k^2 = G a0(e)^2 + G / 2 sum_h (A_h(e)^2 + B_h(e)^2) + ..., gives |a0(e)| <= emax
    and sqrt(A_h(e)^2 + B_h(e)^2) <= sqrt(2) emax.  So |a0| <= emax, |M_1 - 2| <= sqrt(2) emax and M_h <= sqrt(2) emax
    for h >= 2 (rounding in the sums, ~1e-15, is far below)."""
    w = x[(x >= 2e-3 - 1e-4) & (x <= 3e-3)]
    hs = np.diff(w)
    h = hs.max()
    w2 = 2 * math.pi * 1e3
    emax = amp / 2 * (h ** 2 / 8 * 2 * w2 ** 2 + 2 * w2 * np.max(h - hs))
    assert emax < 0.075 * amp                                          # a bound that still says something about M_1 = 2
    s = T.fourier_summary(c[:, None], [T.four(1, 1e3)])[0]
    assert abs(s["a0"][0]) <= emax
    assert abs(s["M"][0, 0] - amp) <= math.sqrt(2) * emax
    assert (s["M"][1:, 0] <= math.sqrt(2) * emax).all()
    return s


def test_isin_pin_on_oracle_rows(built):
    _, res = PU.run_oracle(T.BUNDLED["isin"], 1, {})
    n = int(res["n_rows"][0])
    x, y = res["wave"][0, :n, 0], res["wave"][0, :n, 1]
    assert np.allclose(y[1:], 2 * np.sin(2 * np.pi * 1e3 * x[:-1]), rtol=1e-12, atol=1e-15)    # the one-step source lag
    s = isin_pin(x, F.fourier(x, y, T.four(1, 1e3), 3e-3))
    assert abs(s["phase_deg"][0, 0] + 36.0) < 1.0              # the lag of one 0.1 ms step: -36 degrees


# ---- device source on the host ----------------------------------------------------------------------------------------
def tables(ncol, tstop):
    """Two entries on different columns with different H, G and windows: the last period of 1 kHz at tstop, and 2 kHz
    (H = 3, G = 64) over a window ending at 0.8 tstop."""
    return [T.four(ncol - 1, 1e3), T.four(1, 2e3, n_harm=3, n_grid=64, t_end=0.8 * tstop)]


@pytest.mark.parametrize("deck", ["rc", "rlc", "isin", "diode2"])
def test_device_source_on_host_matches_restatement(deck, built):
    import four_host_emul as FH
    text = T.BUNDLED[deck]
    n = 6
    ckt0 = T.Circuit.from_netlist(text)
    card = ckt0.analysis_card()
    table = tables(len(ckt0.columns(T.AN_TRAN)), card["tstop"])
    ov = PU.draws(deck, ckt0, n)
    with tempfile.TemporaryDirectory() as tmp:
        _, hb, _ = FH.run(text, n, ov, tmp, table, card["tstop"])
        ref = F.fourier_batch(hb.wave_all(), hb.rows(), table, card["tstop"])
        assert R.same_bits(hb.four, ref)
        assert np.isfinite(hb.four).all(), hb.four


# ---- GPU --------------------------------------------------------------------------------------------------------------
SINE_DECKS = ["rc", "rl", "rlc", "isin", "diode2", "transformer1", "transformer2", "transformer3"]
N_GPU = 256


def _gpu_batch(ctx, deck, n=N_GPU, text=None):
    text = text or T.BUNDLED[deck]
    ckt = T.Circuit.from_netlist(text, ctx)
    b = ckt.batch(n)
    for (dev, par), vals in PU.draws(deck, T.Circuit.from_netlist(text), n).items():
        b.set_param(dev, par, vals)
    card = ckt.analysis_card()
    return ckt, b, card, tables(len(ckt.columns(T.AN_TRAN)), card["tstop"])


def _tran(b, card, out, opts, cap=1 << 15):
    b.run_tran(card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"], out, cap, opts)
    b.sync()


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [1, 0], ids=["strict", "fast"])
@pytest.mark.parametrize("deck", SINE_DECKS)
def test_gpu_matches_restatement(ctx, deck, strict):
    ckt, b, card, table = _gpu_batch(ctx, deck)
    b.set_fourier(table)
    _tran(b, card, T.OUT_WAVE | T.OUT_FOUR, T.default_opts(strict_fp=strict, min_blocks=2))
    assert (b.rows() < (1 << 15)).all()
    got = b.fourier()
    ref = F.fourier_batch(b.wave_all(), b.rows(), table, card["tstop"])
    assert R.same_bits(got, ref), np.argwhere(~((got == ref) | (np.isnan(got) & np.isnan(ref))))[:10]
    ok = b.status() == 0
    assert np.isfinite(got[:, ok]).all()
    if deck == "isin":
        isin_pin(b.wave_all()[:int(b.rows()[0]), 0, 0], got[:19, 0], amp=2e-3)     # entry 0 is I(R1)


def _four_run(ctx, deck, strict, out=T.OUT_STATS | T.OUT_FOUR, setup=None, cap=1 << 15, opts_kw=None):
    ckt, b, card, table = _gpu_batch(ctx, deck)
    if setup:
        setup(b)
    b.set_fourier(table)
    _tran(b, card, out, T.default_opts(strict_fp=strict, min_blocks=2, **(opts_kw or {})), cap)
    return b


INVARIANCE = [
    ("order", "diode2", dict(setup=lambda b: b.set_order(np.random.default_rng(5).permutation(b.n_inst)))),
    ("lane_refill", "diode2", dict(opts_kw=dict(lane_refill=1))),
    ("share_time_grid_on", "rlc", dict(opts_kw=dict(share_time_grid=1))),
    ("share_time_grid_off", "rlc", dict(opts_kw=dict(share_time_grid=0))),
    ("small_wave_cap", "rc", dict(out=T.OUT_WAVE | T.OUT_FOUR, cap=40)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [1, 0], ids=["strict", "fast"])
@pytest.mark.parametrize("what, deck, kw", INVARIANCE, ids=[c[0] for c in INVARIANCE])
def test_gpu_fourier_does_not_depend_on_the_mapping(ctx, what, deck, kw, strict):
    plain = _four_run(ctx, deck, strict)
    other = _four_run(ctx, deck, strict, **kw)
    assert R.same_bits(plain.fourier(), other.fourier())
    if what == "small_wave_cap":
        assert (other.rows() > 40).all() and (other.status() == T.api.ST_OVERFLOW).all()


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [1, 0], ids=["strict", "fast"])
def test_gpu_other_outputs_unchanged(ctx, strict):
    """Adding OUT_FOUR leaves statistics, measurements and grid output bit for bit as they are without it."""
    opts = T.default_opts(strict_fp=strict, min_blocks=2)
    for deck in ("rlc", "diode2"):
        ckt, b, card, table = _gpu_batch(ctx, deck)
        b.set_measures([T.meas(T.MEAS_MAX, 1), T.meas(T.MEAS_RMS, 2), T.meas(T.MEAS_AT, 1, 0.5 * card["tstop"])])
        b.set_fourier(table)
        _tran(b, card, T.OUT_STATS | T.OUT_MEAS, opts)
        stats, meas = b.stats_all(), b.measures()
        _tran(b, card, T.OUT_STATS | T.OUT_MEAS | T.OUT_FOUR, opts)
        assert R.same_bits(b.stats_all(), stats) and R.same_bits(b.measures(), meas), deck
        four = b.fourier()
        _tran(b, card, T.OUT_GRID | T.OUT_STATS, opts)
        grid, gstats = b.wave_all(), b.stats_all()
        _tran(b, card, T.OUT_GRID | T.OUT_FOUR, opts)
        assert R.same_bits(b.wave_all(), grid) and R.same_bits(b.stats_all(), gstats), deck
        assert R.same_bits(b.fourier(), four), deck


@pytest.mark.gpu
def test_gpu_agrees_with_oracle_rows(ctx):
    """The restatement on the oracle's rows against the GPU's coefficients.  Rows agree to |d| <= 1e-9 |ref| + 1e-12 at
    the same times (the parity contract); a sample interpolates two rows with weights in [0, 1], so it moves by at most
    the larger row error, and |twiddle| <= 1 gives |d coefficient| <= 2 max_k |d y_k| <= 2 max_r (1e-9 |y_r| + 1e-12)."""
    for deck in ("rc", "rlc", "diode2"):
        n = 8
        ckt, b, card, table = _gpu_batch(ctx, deck, n)
        b.set_fourier(table)
        _tran(b, card, T.OUT_STATS | T.OUT_FOUR, T.default_opts(strict_fp=1, min_blocks=2))
        got = b.fourier()
        _, res = PU.run_oracle(T.BUNDLED[deck], n, PU.draws(deck, T.Circuit.from_netlist(T.BUNDLED[deck]), n))
        for i in range(n):
            r = int(res["n_rows"][i])
            w = res["wave"][i, :r]
            o = 0
            for f in table:
                ref = F.fourier(w[:, 0], w[:, f.column], f, card["tstop"])
                tol = 2 * (1e-9 * np.max(np.abs(w[:, f.column])) + 1e-12)
                assert np.all(np.abs(got[o:o + len(ref), i] - ref) <= tol), (deck, i, got[o:o + len(ref), i] - ref, tol)
                o += len(ref)


@pytest.mark.gpu
def test_gpu_job_over_two_contexts(ctx):
    deck, n = "diode2", 300
    text = T.BUNDLED[deck]
    ckt, b, card, table = _gpu_batch(ctx, deck, n)
    b.set_fourier(table)
    opts = T.default_opts(strict_fp=1, min_blocks=2)
    _tran(b, card, T.OUT_STATS | T.OUT_FOUR, opts)
    job = T.Job([0, 0], text, n)
    for (dev, par), vals in PU.draws(deck, T.Circuit.from_netlist(text), n).items():
        job.set_param(dev, par, vals)
    job.set_fourier(table)
    job.run_tran(card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"], T.OUT_STATS | T.OUT_FOUR, 0, opts)
    job.sync()
    assert R.same_bits(job.fourier(), b.fourier())


@pytest.mark.gpu
def test_gpu_refusals(ctx):
    ckt = T.Circuit.from_netlist(T.BUNDLED["rc"], ctx)
    card = ckt.analysis_card()
    b = ckt.batch(64)
    tran = (card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"])
    L = T.lib()

    def code(fn):
        n0 = ctx.launch_count
        rc = fn()
        assert ctx.launch_count == n0
        return rc

    assert code(lambda: L.tsb_run_tran(b.h, *tran, T.OUT_FOUR, 0, None)) == -1                 # no table
    b.set_fourier([T.four(5, 1e3)])                                                             # rc has 5 columns: 0..4
    assert code(lambda: L.tsb_run_tran(b.h, *tran, T.OUT_FOUR, 0, None)) == -1
    b.set_fourier([T.four(2, 1e3)])
    o = T.default_opts(coop_parts=2)
    assert code(lambda: L.tsb_run_tran(b.h, *tran, T.OUT_FOUR, 0, T.api.C.byref(o))) == -5
    v = [d["name"].lower() for d in ckt.devices()].index("vin")
    assert code(lambda: L.tsb_run_dc(b.h, v, 0.0, 1.0, 0.5, T.OUT_STATS | T.OUT_FOUR, None)) == -5
    assert code(lambda: L.tsb_run_dc2(b.h, v, 0.0, 1.0, 0.5, v, 0.0, 1.0, 0.5, T.OUT_STATS | T.OUT_FOUR, None)) == -5
    assert code(lambda: L.tsb_run_ac(b.h, 0, 7, 1.0, 1e6, T.OUT_STATS | T.OUT_FOUR, None)) == -5
    # results after a run without the flag, and after a new table
    b.run_tran(*tran, out=T.OUT_STATS)
    b.sync()
    with pytest.raises(T.TsbError):
        b.fourier()
    b.run_tran(*tran, out=T.OUT_WAVE | T.OUT_FOUR, cap_rows=1 << 12)
    b.sync()
    assert R.same_bits(b.fourier(), F.fourier_batch(b.wave_all(), b.rows(), [T.four(2, 1e3)], card["tstop"]))
    b.set_fourier([T.four(2, 1e3)])
    with pytest.raises(T.TsbError):
        b.fourier()


@pytest.mark.gpu
def test_gpu_auto_mapping_takes_thread_per_circuit(ctx):
    """rc_ladder(16) would take the cooperative mapping by default; with OUT_FOUR the auto mapping is thread-per-circuit,
    bit for bit what coop_parts = 0 gives."""
    text = rc_ladder(16)
    ckt = T.Circuit.from_netlist(text, ctx)
    card = ckt.analysis_card()
    ncol = len(ckt.columns(T.AN_TRAN))
    tran = (card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"])
    table = [T.four(ncol - 1, 1e3), T.four(1, 1e3, n_harm=4, n_grid=50)]
    res = []
    for parts in (-1, 0):
        b = ckt.batch(512)
        b.set_fourier(table)
        b.run_tran(*tran, out=T.OUT_WAVE | T.OUT_FOUR, cap_rows=1 << 14, opts=T.default_opts(coop_parts=parts))
        b.sync()
        res.append(b.fourier())
        assert R.same_bits(res[-1], F.fourier_batch(b.wave_all(), b.rows(), table, card["tstop"]))
    assert R.same_bits(res[0], res[1])
