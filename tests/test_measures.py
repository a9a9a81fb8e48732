"""Measurements on the device (TSB_OUT_MEAS: WHEN, AT, MAX, MIN, AVG, INTEG, RMS; include/tspice_b200.h).

* CPU: the restatement (tests/meas_ref.py) on hand-built series whose results are exact (dyadic values), crossings exactly
  at samples, both edges at one level, count = -1 and past the last crossing, NaN samples, windows partly outside the data,
  zero-width windows; the table's validation; the kernel source with and without a table.
* CPU, device source on the host (tests/meas_host_emul.py over tests/host_emul.py, strict configuration): the measurement code of the sink is bit for bit
  the restatement applied to the same run's rows (rc, rlc, diode2 transients; the diode3 DC sweep).
* GPU: bit identity with the restatement on the run's own rows for every bundled transient deck, diode3 and the AC decks,
  in both builds; everything that must not change a bit (processing order, lane refill, shared time grid, a waveform
  capacity below the row count, grid output, statistics, a job over two contexts); the -3 dB point of a low pass; refusals."""
import math
import tempfile

import numpy as np
import pytest

import meas_ref as R
import parity_util as PU
from ac_decks import AC_DECKS
from random_decks import rc_ladder

T = PU.T
INF = math.inf
NAN = math.nan


def M(kind, column=1, level=0.0, **kw):
    return T.meas(kind, column, level, **kw)


def _eq(got, want):
    """Exact equality of (value, abscissa), NaN == NaN."""
    return R.same_bits(np.array(got), np.array(want, dtype=np.float64))


# ---- restatement, hand-built series ----------------------------------------------------------------------------------
X = [0.0, 1.0, 2.0, 3.0, 4.0]
TRI = [0.0, 2.0, 4.0, 2.0, 0.0]


@pytest.mark.parametrize("m, want", [
    (M(R.MEAS_WHEN, level=1.0), (1.0, 0.5)),
    (M(R.MEAS_WHEN, level=1.0, count=2), (1.0, 3.5)),
    (M(R.MEAS_WHEN, level=1.0, count=-1), (1.0, 3.5)),
    (M(R.MEAS_WHEN, level=1.0, count=3), (NAN, NAN)),                       # past the last crossing
    (M(R.MEAS_WHEN, level=1.0, edge=R.EDGE_RISE, count=2), (NAN, NAN)),
    (M(R.MEAS_WHEN, level=1.0, edge=R.EDGE_FALL), (1.0, 3.5)),              # rise and fall at the same level
    (M(R.MEAS_WHEN, level=2.0), (2.0, 1.0)),                                # exactly at a sample: counted once per side
    (M(R.MEAS_WHEN, level=2.0, count=-1), (2.0, 3.0)),
    (M(R.MEAS_WHEN, level=2.0, count=3), (NAN, NAN)),
    (M(R.MEAS_WHEN, level=4.0), (4.0, 2.0)),                                # touching the peak rises, never falls
    (M(R.MEAS_WHEN, level=4.0, edge=R.EDGE_FALL), (NAN, NAN)),
    (M(R.MEAS_WHEN, level=1.0, from_=1.0, to=3.5), (1.0, 3.5)),             # window on the crossing's abscissa, inclusive
    (M(R.MEAS_WHEN, level=1.0, from_=0.75, to=3.25), (NAN, NAN)),
    (M(R.MEAS_AT, level=2.5), (3.0, 2.5)),
    (M(R.MEAS_AT, level=3.0), (2.0, 3.0)),
    (M(R.MEAS_AT, level=0.0), (0.0, 0.0)),
    (M(R.MEAS_AT, level=-1.0), (NAN, -1.0)),
    (M(R.MEAS_AT, level=4.5), (NAN, 4.5)),
    (M(R.MEAS_MAX), (4.0, 2.0)),
    (M(R.MEAS_MIN), (0.0, 0.0)),                                            # a tie goes to the first row
    (M(R.MEAS_MIN, from_=1.0, to=4.0), (0.0, 4.0)),
    (M(R.MEAS_MAX, from_=2.5, to=2.75), (NAN, NAN)),                        # no row in the window
    (M(R.MEAS_INTEG), (8.0, NAN)),
    (M(R.MEAS_AVG), (2.0, NAN)),
    (M(R.MEAS_RMS), (math.sqrt(6.0), NAN)),
    (M(R.MEAS_INTEG, from_=0.5, to=3.5), (7.5, NAN)),                       # clipped segments, interpolated ends
    (M(R.MEAS_AVG, from_=0.5, to=3.5), (2.5, NAN)),
    (M(R.MEAS_INTEG, from_=-1.0), (NAN, NAN)),                              # window partly outside the data
    (M(R.MEAS_AVG, to=5.0), (NAN, NAN)),
    (M(R.MEAS_INTEG, from_=2.0, to=2.0), (0.0, NAN)),                       # zero width
    (M(R.MEAS_AVG, from_=2.0, to=2.0), (NAN, NAN)),
    (M(R.MEAS_RMS, from_=1.5, to=1.5), (NAN, NAN)),
    (M(R.MEAS_INTEG, from_=1.0, to=INF), (7.0, NAN)),
])
def test_restatement_triangle(m, want):
    assert _eq(R.measure(X, TRI, TRI, m), want), (R.measure(X, TRI, TRI, m), want)


def test_restatement_nan_samples_and_trigger_column():
    y = [0.0, 2.0, NAN, 2.0, 0.0]
    assert _eq(R.measure(X, y, y, M(R.MEAS_MAX)), (2.0, 1.0))              # NaN ignored, tie -> first row
    assert _eq(R.measure(X, y, y, M(R.MEAS_MIN, from_=0.5, to=3.0)), (2.0, 1.0))
    assert _eq(R.measure(X, y, y, M(R.MEAS_WHEN, level=1.0, count=-1)), (1.0, 3.5))
    assert _eq(R.measure(X, y, y, M(R.MEAS_WHEN, level=1.0, count=2)), (1.0, 3.5))   # segments next to the NaN never cross
    assert _eq(R.measure(X, y, y, M(R.MEAS_INTEG)), (NAN, NAN))
    # value of one column where ANOTHER crosses: y at t = 1
    t = [-2.0, -1.0, 0.0, 1.0, 2.0]
    assert _eq(R.measure(X, TRI, t, M(R.MEAS_WHEN, level=1.0)), (2.0, 3.0))
    assert _eq(R.measure(X, TRI, t, M(R.MEAS_WHEN, level=0.5, edge=R.EDGE_FALL)), (NAN, NAN))


def test_restatement_piecewise_linear_exact():
    """A piecewise-linear series with dyadic breakpoints and values, sampled at every breakpoint and at dyadic points in
    between: every operation is exact, so every result equals its closed form."""
    xs = np.arange(0, 65) / 8.0                                 # 0 .. 8 step 1/8
    y = np.interp(xs, [0, 2, 4, 6, 8], [-1.0, 3.0, 3.0, -5.0, 1.0])
    assert _eq(R.measure(xs, y, y, M(R.MEAS_WHEN, level=1.0)), (1.0, 1.0))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_WHEN, level=1.0, edge=R.EDGE_FALL)), (1.0, 4.5))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_WHEN, level=-2.0, edge=R.EDGE_RISE)), (-2.0, 7.0))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_AT, level=5.0)), (-1.0, 5.0))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_MAX)), (3.0, 2.0))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_MIN)), (-5.0, 6.0))
    # integral of the polyline: 2 (0..2) + 6 (2..4) - 2 (4..6) - 4 (6..8) = 2
    assert _eq(R.measure(xs, y, y, M(R.MEAS_INTEG)), (2.0, NAN))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_AVG)), (0.25, NAN))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_INTEG, from_=2.0, to=4.0)), (6.0, NAN))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_AVG, from_=2.0, to=4.0)), (3.0, NAN))
    assert _eq(R.measure(xs, y, y, M(R.MEAS_RMS, from_=2.0, to=4.0)), (3.0, NAN))


def test_restatement_short_series():
    assert _eq(R.measure([], [], [], M(R.MEAS_INTEG)), (NAN, NAN))
    assert _eq(R.measure([], [], [], M(R.MEAS_MAX)), (NAN, NAN))
    assert _eq(R.measure([1.0], [3.0], [3.0], M(R.MEAS_AVG)), (NAN, NAN))     # one row: zero width
    assert _eq(R.measure([1.0], [3.0], [3.0], M(R.MEAS_INTEG)), (0.0, NAN))
    assert _eq(R.measure([1.0], [3.0], [3.0], M(R.MEAS_AT, level=1.0)), (3.0, 1.0))
    assert _eq(R.measure([1.0], [3.0], [3.0], M(R.MEAS_WHEN, level=3.0)), (NAN, NAN))


# ---- table validation and kernel source (host-only plans) -----------------------------------------------------------
def _host_batch(deck="rc"):
    return T.Circuit.from_netlist(T.BUNDLED[deck]).batch(2)


@pytest.mark.parametrize("bad", [
    dict(kind=7), dict(kind=-1), dict(column=0), dict(trig_column=0), dict(edge=3), dict(count=0), dict(count=-2),
    dict(level=NAN), dict(from_=NAN), dict(to=NAN), dict(from_=2.0, to=1.0),
])
def test_set_measures_refuses(bad, built):
    kw = dict(kind=R.MEAS_WHEN, column=1, level=0.5)
    kw.update(bad)
    m = T.Meas(kw["kind"], kw["column"], kw.get("trig_column", 1), kw.get("edge", 0), kw.get("count", 1), kw["level"],
               kw.get("from_", -INF), kw.get("to", INF))
    with pytest.raises(T.TsbError):
        _host_batch().set_measures([m])


def test_set_measures_limits(built):
    b = _host_batch()
    b.set_measures([M(R.MEAS_MAX)] * 16)
    with pytest.raises(T.TsbError):
        b.set_measures([M(R.MEAS_MAX)] * 17)
    b.set_measures([])
    # outside WHEN, count / edge / trig_column are not looked at (and not part of the kernel)
    b.set_measures([T.Meas(R.MEAS_MAX, 1, 0, 9, 0, NAN, -INF, INF)])


def test_kernel_source_with_and_without_table(built):
    b = _host_batch()
    opts = T.default_opts(strict_fp=1, min_blocks=2)
    plain = b.kernel_source(opts)
    b.set_measures([M(R.MEAS_WHEN, 2, 0.5), M(R.MEAS_RMS, 3)])
    assert b.kernel_source(opts) == plain                       # a table alone selects nothing
    b.kernel_variant(meas=True)
    src = b.kernel_source(opts)
    assert "#define TSB_MEAS 2\n#define TSB_MEAS_SPEC {0, 2, 2}, {6, 3, 3}\n" in src and "#define TSB_MEAS_SPEC" not in plain
    key = b.kernel_key(opts)
    b.set_measures([M(R.MEAS_WHEN, 2, 0.75, from_=1e-3), M(R.MEAS_RMS, 3, to=2e-3)])
    assert b.kernel_key(opts) == key                            # levels and windows are run-time arguments
    b.set_measures([M(R.MEAS_WHEN, 1, 0.5), M(R.MEAS_RMS, 3)])
    assert b.kernel_key(opts) != key


# ---- a table that uses every kind, derived from a run's own rows ----------------------------------------------------
def every_kind(ncol, wave, rows):
    """Levels and windows from instance 0's rows: both signal levels at mid-range, windows over the middle of the series."""
    r = int(min(rows[0], wave.shape[0]))
    s = wave[:r, :, 0]
    c1, c2, cl = 1, min(2, ncol - 1), ncol - 1
    x0, xl = float(s[0, 0]), float(s[-1, 0])
    xa, xb, xm = x0 + 0.2 * (xl - x0), x0 + 0.8 * (xl - x0), x0 + 0.37 * (xl - x0)
    mid = lambda c: float(0.5 * (np.nanmin(s[:, c]) + np.nanmax(s[:, c]))) if np.isfinite(s[:, c]).any() else 0.0
    return [
        M(R.MEAS_WHEN, c1, mid(c1)),
        M(R.MEAS_WHEN, c1, mid(c2), trig_column=c2, edge=R.EDGE_RISE, count=-1),
        M(R.MEAS_WHEN, c2, mid(c2), edge=R.EDGE_FALL, count=2, from_=xa, to=xb),
        M(R.MEAS_AT, c2, xm),
        M(R.MEAS_AT, c1, x0),
        M(R.MEAS_MAX, c1, from_=xa, to=xb),
        M(R.MEAS_MIN, cl),
        M(R.MEAS_AVG, c1),
        M(R.MEAS_INTEG, c2, from_=xa, to=xb),
        M(R.MEAS_RMS, cl, from_=xa),
        M(R.MEAS_AVG, cl, from_=xm, to=xm),
    ]


# ---- device source on the host ----------------------------------------------------------------------------------------
HOST_CASES = [("rc", {}), ("rlc", {}), ("diode2", {}), ("diode3", {})]


@pytest.mark.parametrize("deck, kw", HOST_CASES, ids=[c[0] for c in HOST_CASES])
def test_device_source_on_host_matches_restatement(deck, kw, built):
    import meas_host_emul as MH
    text = T.BUNDLED[deck]
    n = 6
    ov = PU.draws(deck, T.Circuit.from_netlist(text), n)
    ckt0 = T.Circuit.from_netlist(text)
    ncol = len(ckt0.columns(ckt0.analysis_card()["analysis"]))
    with tempfile.TemporaryDirectory() as tmp:
        # pass 1 with provisional levels, pass 2 with levels from pass 1's rows: the same kernel (levels are run-time)
        table = every_kind(ncol, np.zeros((2, ncol, 1)) + np.arange(2.0)[:, None, None], [2])
        _, hb, _ = MH.run(text, n, ov, tmp, table, **kw)
        table = every_kind(ncol, hb.wave_all(), hb.rows())
        _, hb, _ = MH.run(text, n, ov, tmp, table, **kw)
        ref = R.measure_batch(hb.wave_all(), hb.rows(), table)
        assert R.same_bits(hb.meas, ref)
        assert np.isfinite(hb.meas[0, 0]).all(), hb.meas[0, 0]      # the mid-range crossing exists in every instance
        if deck == "diode3":
            # WHEN V(2) = level on the DC transfer curve: the input threshold, between two sweep points of the curve
            th = hb.meas[1, 0]
            assert ((th >= -1.0) & (th <= 3.0)).all()


# ---- GPU --------------------------------------------------------------------------------------------------------------
TRAN_DECKS = sorted(n for n in T.BUNDLED if T.Circuit.from_netlist(T.BUNDLED[n]).analysis_card()["analysis"] == T.AN_TRAN)
N_GPU = 256


def _batch(ctx, text, n, deck):
    ckt = T.Circuit.from_netlist(text, ctx)
    b = ckt.batch(n)
    for (dev, par), vals in PU.draws(deck, T.Circuit.from_netlist(text), n).items():
        b.set_param(dev, par, vals)
    return ckt, b


def _run(b, card, an, out, opts, cap=0, ac=None):
    if an == T.AN_TRAN:
        b.run_tran(card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"], out, cap or 1 << 15, opts)
    elif an == T.AN_DC:
        b.run_dc(card["dc_src_dev"], card["dc_start"], card["dc_stop"], card["dc_inc"], out, opts)
    else:
        b.run_ac(*ac, out=out, opts=opts)
    b.sync()


def _gpu_case(ctx, deck, strict, n=N_GPU):
    """(batch, card, analysis, ac args, table): rows of a plain run give the table's levels."""
    if deck in AC_DECKS:
        text = AC_DECKS[deck]
    else:
        text = T.BUNDLED[deck]
    ckt, b = _batch(ctx, text, n, deck if deck in T.BUNDLED else "rc")
    card = ckt.analysis_card()
    an = card["analysis"]
    ac = (card["ac_sweep"], card["ac_points"], card["ac_fstart"], card["ac_fstop"]) if an == T.AN_AC else None
    opts = T.default_opts(strict_fp=strict, min_blocks=2)        # one kernel per table (no launch-bounds search)
    _run(b, card, an, T.OUT_WAVE, opts, ac=ac)
    table = every_kind(len(ckt.columns(an)), b.wave_all(), b.rows())
    return b, card, an, ac, table, opts


GPU_DECKS = TRAN_DECKS + ["diode3"] + sorted(AC_DECKS)


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [1, 0], ids=["strict", "fast"])
@pytest.mark.parametrize("deck", GPU_DECKS)
def test_gpu_matches_restatement(ctx, deck, strict):
    b, card, an, ac, table, opts = _gpu_case(ctx, deck, strict)
    b.set_measures(table)
    _run(b, card, an, T.OUT_WAVE | T.OUT_MEAS, opts, ac=ac)
    got = b.measures()
    ref = R.measure_batch(b.wave_all(), b.rows(), table)
    assert R.same_bits(got, ref), np.argwhere(~((got == ref) | (np.isnan(got) & np.isnan(ref))))[:10]
    if deck == "bjt2":
        assert np.isnan(got[0]).any()                            # lanes with NaN samples / no crossing


def _meas_run(ctx, deck, strict, out=T.OUT_STATS | T.OUT_MEAS, setup=None, cap=0, opts_kw=None, n=N_GPU):
    b, card, an, ac, table, _ = _gpu_case(ctx, deck, strict, n)
    opts = T.default_opts(strict_fp=strict, min_blocks=2, **(opts_kw or {}))
    if setup:
        setup(b)
    b.set_measures(table)
    _run(b, card, an, out, opts, cap=cap, ac=ac)
    return b, table


INVARIANCE = [
    ("order", "diode2", dict(setup=lambda b: b.set_order(np.random.default_rng(5).permutation(b.n_inst)))),
    ("lane_refill", "diode2", dict(opts_kw=dict(lane_refill=1))),
    ("share_time_grid", "rlc", dict(opts_kw=dict(share_time_grid=1))),
    ("small_wave_cap", "rc", dict(out=T.OUT_WAVE | T.OUT_MEAS, cap=40)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [1, 0], ids=["strict", "fast"])
@pytest.mark.parametrize("what, deck, kw", INVARIANCE, ids=[c[0] for c in INVARIANCE])
def test_gpu_measures_do_not_depend_on_the_mapping(ctx, what, deck, kw, strict):
    plain, _ = _meas_run(ctx, deck, strict)
    other, _ = _meas_run(ctx, deck, strict, **kw)
    assert R.same_bits(plain.measures(), other.measures())
    if what == "small_wave_cap":
        assert (other.rows() > 40).all() and (other.status() == T.api.ST_OVERFLOW).all()


@pytest.mark.gpu
@pytest.mark.parametrize("strict", [1, 0], ids=["strict", "fast"])
def test_gpu_grid_and_statistics_unchanged(ctx, strict):
    b, card, an, ac, table, opts = _gpu_case(ctx, "rlc", strict)
    _run(b, card, an, T.OUT_GRID | T.OUT_STATS, opts)
    grid, stats = b.wave_all(), b.stats_all()
    b.set_measures(table)
    _run(b, card, an, T.OUT_GRID | T.OUT_MEAS, opts)
    assert R.same_bits(b.wave_all(), grid) and R.same_bits(b.stats_all(), stats)
    with_grid = b.measures()
    _run(b, card, an, T.OUT_STATS | T.OUT_MEAS, opts)
    assert R.same_bits(b.stats_all(), stats) and R.same_bits(b.measures(), with_grid)
    for deck in ("diode2", "diode3", "ac_ladder"):
        b, card, an, ac, table, opts = _gpu_case(ctx, deck, strict)
        _run(b, card, an, T.OUT_STATS, opts, ac=ac)
        stats = b.stats_all()
        b.set_measures(table)
        _run(b, card, an, T.OUT_STATS | T.OUT_MEAS, opts, ac=ac)
        assert R.same_bits(b.stats_all(), stats), deck


@pytest.mark.gpu
def test_gpu_job_over_two_contexts(ctx):
    text, n = T.BUNDLED["diode2"], 300
    b, card, an, _, table, opts = _gpu_case(ctx, "diode2", 1, n)
    b.set_measures(table)
    _run(b, card, an, T.OUT_STATS | T.OUT_MEAS, opts)
    job = T.Job([0, 0], text, n)
    for (dev, par), vals in PU.draws("diode2", T.Circuit.from_netlist(text), n).items():
        job.set_param(dev, par, vals)
    job.set_measures(table)
    job.run_tran(card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"], T.OUT_STATS | T.OUT_MEAS, 0, opts)
    job.sync()
    assert R.same_bits(job.measures(), b.measures())


@pytest.mark.gpu
def test_gpu_lowpass_minus_3db(ctx):
    """WHEN on V(2)_MAG = 1/sqrt(2) of ac_lowpass (R = 1k, C = 1u): the corner 1/(2 pi R C) = 159.15 Hz, to within the
    error of linear interpolation between the sweep's points (DEC 31 -> neighbouring points 7.7 % apart)."""
    text = AC_DECKS["ac_lowpass"]
    ckt = T.Circuit.from_netlist(text, ctx)
    cols = ckt.columns(T.AN_AC)
    b = ckt.batch(4)
    b.set_measures([M(R.MEAS_WHEN, cols.index("V(2)_MAG"), 1 / math.sqrt(2), edge=R.EDGE_FALL),
                    M(R.MEAS_WHEN, cols.index("V(2)_PHASE"), -45.0)])
    b.run_ac("DEC", 31, 1.0, 1e6, out=T.OUT_MEAS)
    b.sync()
    got = b.measures()
    fc = 1 / (2 * math.pi * 1e3 * 1e-6)
    assert np.all(np.abs(got[1] / fc - 1) < 0.01), got[1]
    assert np.all(np.abs(got[0, 0] - 1 / math.sqrt(2)) < 1e-12)


@pytest.mark.gpu
def test_gpu_refusals(ctx):
    text = T.BUNDLED["rc"]
    ckt = T.Circuit.from_netlist(text, ctx)
    card = ckt.analysis_card()
    b = ckt.batch(64)
    tran = (card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"])
    L = T.lib()

    def code(fn):
        n0 = ctx.launch_count
        rc = fn()
        assert ctx.launch_count == n0
        return rc

    assert code(lambda: L.tsb_run_tran(b.h, *tran, T.OUT_MEAS, 0, None)) == -1                 # no table
    b.set_measures([M(R.MEAS_MAX, 5)])                                                          # rc has 5 columns: 0..4
    assert code(lambda: L.tsb_run_tran(b.h, *tran, T.OUT_MEAS, 0, None)) == -1
    b.set_measures([M(R.MEAS_WHEN, 1, 0.5, trig_column=7)])
    assert code(lambda: L.tsb_run_tran(b.h, *tran, T.OUT_MEAS, 0, None)) == -1
    b.set_measures([M(R.MEAS_MAX, 2)])
    o = T.default_opts(coop_parts=2)
    assert code(lambda: L.tsb_run_tran(b.h, *tran, T.OUT_MEAS, 0, T.api.C.byref(o))) == -5
    d = T.Circuit.from_netlist(T.BUNDLED["diode3"], ctx)
    db = d.batch(32)
    db.set_measures([M(R.MEAS_MAX, 2)])
    assert code(lambda: L.tsb_run_dc2(db.h, 0, 0.0, 1.0, 0.5, 0, 0.0, 1.0, 0.5, T.OUT_MEAS, None)) in (-5, -1)
    # AC columns: the table is checked against the analysis that runs
    ac = T.Circuit.from_netlist(AC_DECKS["ac_lowpass"], ctx)
    ab = ac.batch(8)
    ab.set_measures([M(R.MEAS_MAX, len(ac.columns(T.AN_AC)))])
    assert code(lambda: L.tsb_run_ac(ab.h, 0, 7, 1.0, 1e6, T.OUT_MEAS, None)) == -1
    # results after a run without measurements
    b.set_measures([M(R.MEAS_MAX, 2)])
    b.run_tran(*tran, out=T.OUT_STATS)
    b.sync()
    with pytest.raises(T.TsbError):
        b.measures()
    b.run_tran(*tran, out=T.OUT_WAVE | T.OUT_MEAS, cap_rows=1 << 12)
    b.sync()
    assert R.same_bits(b.measures(), R.measure_batch(b.wave_all(), b.rows(), [M(R.MEAS_MAX, 2)]))


@pytest.mark.gpu
def test_gpu_nested_dc_refused(ctx):
    text = """nested
V1 1 0 DC 1
V2 2 0 DC 1
R1 1 2 1k
R2 2 0 1k
.dc V1 0 1 0.5 V2 0 1 0.5
"""
    ckt = T.Circuit.from_netlist(text, ctx)
    b = ckt.batch(32)
    b.set_measures([M(R.MEAS_MAX, 2)])
    n0 = ctx.launch_count
    assert T.lib().tsb_run_dc2(b.h, 0, 0.0, 1.0, 0.5, 1, 0.0, 1.0, 0.5, T.OUT_MEAS, None) == -5
    assert ctx.launch_count == n0


@pytest.mark.gpu
def test_gpu_auto_mapping_takes_thread_per_circuit(ctx):
    """rc_ladder(16) would take the cooperative mapping by default; with OUT_MEAS the auto mapping is thread-per-circuit,
    bit for bit what coop_parts = 0 gives."""
    text = rc_ladder(16)
    ckt = T.Circuit.from_netlist(text, ctx)
    card = ckt.analysis_card()
    ncol = len(ckt.columns(T.AN_TRAN))
    tran = (card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"])
    res = []
    for parts in (-1, 0):
        b = ckt.batch(512)
        b.set_measures([M(R.MEAS_MAX, ncol - 1), M(R.MEAS_RMS, 2), M(R.MEAS_AT, 1, 0.5 * card["tstop"])])
        b.run_tran(*tran, out=T.OUT_WAVE | T.OUT_MEAS, cap_rows=1 << 14, opts=T.default_opts(coop_parts=parts))
        b.sync()
        res.append(b.measures())
        assert R.same_bits(res[-1], R.measure_batch(b.wave_all(), b.rows(), [M(R.MEAS_MAX, ncol - 1), M(R.MEAS_RMS, 2),
                                                                                M(R.MEAS_AT, 1, 0.5 * card["tstop"])]))
    assert R.same_bits(res[0], res[1])
