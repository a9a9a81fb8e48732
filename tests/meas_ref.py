"""Restatement of the measurement definitions (include/tspice_b200.h, TSB_OUT_MEAS) on one instance's stored series.

Operation for operation what the header defines, in float64 numpy arithmetic: every elementwise operation is one IEEE
operation rounded to nearest (numpy never contracts a multiply and an add), and the trapezoid sums are accumulated in
row order from 0.0 (np.add.accumulate is sequential), so a result of the device is expected BIT FOR BIT.

A measurement is a `toy-spice_b200.Meas` (or anything with the same attributes: kind, column, trig_column, edge, count,
level, from_, to)."""
import numpy as np

MEAS_WHEN, MEAS_AT, MEAS_MAX, MEAS_MIN, MEAS_AVG, MEAS_INTEG, MEAS_RMS = range(7)
EDGE_CROSS, EDGE_RISE, EDGE_FALL = range(3)
NAN = float("nan")


def _interp(x0, y0, x1, y1, L):
    """AT's value at L on the segment (x0, y0) - (x1, y1): y1 where L == x1, else y0 + ((L - x0) / (x1 - x0)) (y1 - y0)."""
    v = y0 + ((L - x0) / (x1 - x0)) * (y1 - y0)
    return np.where(L == x1, y1, v)


def measure(x, y, t, m):
    """(value, abscissa) of measurement `m` on the series x (column 0), y (m.column), t (m.trig_column): 1-D float64
    arrays of the stored rows."""
    x, y, t = (np.asarray(v, dtype=np.float64) for v in (x, y, t))
    fr, to = np.float64(m.from_), np.float64(m.to)
    n = len(x)
    with np.errstate(all="ignore"):
        if m.kind == MEAS_WHEN:
            if n < 2:
                return NAN, NAN
            L = np.float64(m.level)
            t0, t1, x0, x1, y0, y1 = t[:-1], t[1:], x[:-1], x[1:], y[:-1], y[1:]
            rise = (t0 < L) & (L <= t1)
            fall = (t0 > L) & (L >= t1)
            sel = (rise & (m.edge != EDGE_FALL)) | (fall & (m.edge != EDGE_RISE))
            f = (L - t0) / (t1 - t0)
            xs = x0 + f * (x1 - x0)
            ok = np.flatnonzero(sel & (xs >= fr) & (xs <= to))
            if m.count < 0:
                if ok.size == 0:
                    return NAN, NAN
                k = ok[-1]
            else:
                if ok.size < m.count:
                    return NAN, NAN
                k = ok[m.count - 1]
            return float(y0[k] + f[k] * (y1[k] - y0[k])), float(xs[k])
        if m.kind == MEAS_AT:
            L = np.float64(m.level)
            hit = np.flatnonzero(x >= L)
            if hit.size == 0:
                return NAN, float(L)
            j = hit[0]
            if j == 0:
                return (float(y[0]) if x[0] == L else NAN), float(L)
            return float(_interp(x[j - 1], y[j - 1], x[j], y[j], L)), float(L)
        if m.kind in (MEAS_MAX, MEAS_MIN):
            idx = np.flatnonzero((x >= fr) & (x <= to) & ~np.isnan(y))
            if idx.size == 0:
                return NAN, NAN
            v = y[idx]
            e = v.max() if m.kind == MEAS_MAX else v.min()
            k = idx[np.flatnonzero(v == e)[0]]           # a tie goes to the first row
            return float(y[k]), float(x[k])
        # INTEG / AVG / RMS
        if n == 0:
            return NAN, NAN
        a = x[0] if fr == -np.inf else fr
        b = x[-1] if to == np.inf else to
        if a < x[0] or b > x[-1] or a > b:
            return NAN, NAN
        x0, x1, y0, y1 = x[:-1], x[1:], y[:-1], y[1:]
        lo = np.where(x0 > fr, x0, fr)
        hi = np.where(x1 < to, x1, to)
        sel = lo < hi
        x0, x1, y0, y1, lo, hi = (v[sel] for v in (x0, x1, y0, y1, lo, hi))
        ylo = np.where(lo == x0, y0, _interp(x0, y0, x1, y1, lo))
        yhi = _interp(x0, y0, x1, y1, hi)
        h = ylo * ylo + yhi * yhi if m.kind == MEAS_RMS else ylo + yhi
        terms = ((hi - lo) * h) * 0.5
        s = np.add.accumulate(np.concatenate([[0.0], terms]))[-1]
        if m.kind == MEAS_INTEG:
            return float(s), NAN
        q = s / (b - a)
        return (float(q) if m.kind == MEAS_AVG else float(np.sqrt(q))), NAN


def measure_batch(wave, rows, measures):
    """Restatement applied to a whole run's rows: wave [cap_rows][n_columns][n_inst] (Batch.wave_all), rows [n_inst]
    -> [2][n_meas][n_inst] in the layout of Batch.measures()."""
    wave = np.asarray(wave)
    n = wave.shape[2]
    out = np.empty((2, len(measures), n))
    for i in range(n):
        r = min(int(rows[i]), wave.shape[0])
        s = wave[:r, :, i]
        for k, m in enumerate(measures):
            out[:, k, i] = measure(s[:, 0], s[:, m.column], s[:, m.trig_column], m)
    return out


def same_bits(a, b):
    """Bit identity with every NaN taken as equal to every NaN (positions must agree)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64))
