"""Restatement of the Fourier definition (include/tspice_b200.h, TSB_OUT_FOUR) on one instance's stored series.

Operation for operation what the header defines, in float64 numpy arithmetic: every elementwise operation is one IEEE
operation rounded to nearest (numpy never contracts a multiply and an add), the sums are accumulated over ascending k
from 0.0 (np.add.accumulate is sequential), and the twiddles come from the C library's cos and sin (Python's math module),
as the library computes them.  So a result of the device is expected BIT FOR BIT.

An entry is a `toy-spice_b200.Four` (or anything with the attributes column, n_harm, n_grid, freq, t_end)."""
import math

import numpy as np

from meas_ref import _interp, same_bits  # noqa: F401  (same_bits: re-exported for the tests)

NAN = float("nan")


def twiddles(G):
    """c[j] = cos(2.0 pi j / G), s[j] = sin(2.0 pi j / G), evaluated left to right with libm."""
    c = np.array([math.cos(2.0 * math.pi * j / G) for j in range(G)])
    s = np.array([math.sin(2.0 * math.pi * j / G) for j in range(G)])
    return c, s


def window(f, tstop):
    """(s, dt): the window start s = e - 1/f and the grid spacing (1/f) / G, e = t_end or tstop for t_end = +inf."""
    T = 1.0 / f.freq
    e = tstop if f.t_end == math.inf else f.t_end
    return e - T, T / f.n_grid


def grid(f, tstop):
    """tau_k = s + k dt, k = 0 .. G-1: a product and a sum, each rounded."""
    s, dt = window(f, tstop)
    return np.float64(s) + np.arange(f.n_grid, dtype=np.float64) * np.float64(dt)


def samples(x, y, tau):
    """y at every tau as AT defines it; None when tau_0 < x_0 or tau_{G-1} > x_last (every coefficient is then NaN)."""
    x, y, tau = (np.asarray(v, dtype=np.float64) for v in (x, y, tau))
    if x.size == 0:
        return None
    j = np.searchsorted(x, tau, side="left")            # the first row with x >= tau
    if j[-1] >= x.size or (j[0] == 0 and x[0] != tau[0]):
        return None
    on = x[j] == tau
    jm = np.maximum(j - 1, 0)
    with np.errstate(all="ignore"):
        v = _interp(x[jm], y[jm], x[j], y[j], tau)
    return np.where(on, y[j], v)


def _sum(terms):
    return np.add.accumulate(np.concatenate([[0.0], terms]))[-1]


def fourier(x, y, f, tstop):
    """[a0, A_1, B_1, ..., A_H, B_H] of entry f on the series x (column 0), y (f.column): 1-D float64 rows."""
    H, G = f.n_harm, f.n_grid
    yk = samples(x, y, grid(f, tstop))
    if yk is None:
        return np.full(1 + 2 * H, NAN)
    c, s = twiddles(G)
    k = np.arange(G)
    out = np.empty(1 + 2 * H)
    with np.errstate(all="ignore"):
        out[0] = _sum(yk) / G
        for h in range(1, H + 1):
            idx = (h * k) % G
            out[2 * h - 1] = (2.0 * _sum(yk * c[idx])) / G
            out[2 * h] = (2.0 * _sum(yk * s[idx])) / G
    return out


def fourier_batch(wave, rows, table, tstop):
    """Restatement applied to a whole run's rows: wave [cap_rows][n_columns][n_inst] (Batch.wave_all), rows [n_inst]
    -> [sum (1 + 2H)][n_inst] in the layout of Batch.fourier()."""
    wave = np.asarray(wave)
    n = wave.shape[2]
    out = np.empty((sum(1 + 2 * f.n_harm for f in table), n))
    for i in range(n):
        r = min(int(rows[i]), wave.shape[0])
        s = wave[:r, :, i]
        o = 0
        for f in table:
            out[o:o + 1 + 2 * f.n_harm, i] = fourier(s[:, 0], s[:, f.column], f, tstop)
            o += 1 + 2 * f.n_harm
    return out
