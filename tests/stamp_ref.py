"""Test infrastructure: the reference of the device-stamp kernel (tsb_batch_stamp_dev).

What the kernel writes for one instance is the matrix the reference holds after

    SetupDevices (the set-up stamp, circuit.go:154-156);  mat.Clear();  ckt.Stamp(status);  mat.LoadGmin(gmin)

with status = {Mode, Time, TimeStep = dt, Temp = 300.15, Gmin}.  `stamp` computes it with the independent NumPy
restatement of the device layer (oracle/pin_numpy.py: plain Python floats, a dense 1-based matrix that accumulates onto a
cleared 0.0) and adds gmin onto the pivot positions of the plan's frozen order (LoadGmin, SURVEY Q17).  Alongside every
entry it accumulates the sum of |contribution| (S, Sb), the scale a re-associated or contracted build is held to.

The pin computes sine and power as Go does (pin_numpy.go_sin, go_pow) and takes exp and log from Python's `math`.  While
`stamp` runs, the pin's `math` is `Libm`: the host's libm by default, or a table of exp / log values computed elsewhere
(the CUDA math library's, so the GPU's strict build can be held to the reference bit for bit; `Libm.calls` lists the
arguments a table has to cover)."""
import collections
import math
import struct

import numpy as np

import parity_util as PU
from oracle import pin_numpy as P

O, T = PU.O, PU.T
OP, TRAN = P.OP_MODE, P.TRAN_MODE


def bits(x):
    return struct.unpack("<q", struct.pack("<d", float(x)))[0]


def host_exp(x):
    try:
        return math.exp(x)
    except OverflowError:
        return math.inf


class Libm:
    """Stands in for the `math` module inside oracle/pin_numpy.py while `stamp` runs (see the module docstring)."""

    def __init__(self, table=None):
        self.table = table              # {(name, bits(x)): value}; None or a missing key: the host's libm
        self.calls = []                 # (name, x) of every exp / log evaluated

    def __getattr__(self, name):
        return getattr(math, name)

    def _lib(self, name, x, host):
        x = float(x)
        self.calls.append((name, x))
        if self.table is not None:
            v = self.table.get((name, bits(x)))
            if v is not None:
                return v
        return host(x)

    def exp(self, x):
        return self._lib("exp", x, host_exp)

    def log(self, x):
        return self._lib("log", x, math.log)


class AbsMatrix(P.Matrix):
    """pin_numpy.Matrix that also accumulates |v| of every contribution (S for A, Sb for b) and counts them (m, mb)."""

    def __init__(self, n):
        super().__init__(n)
        self.S = np.zeros((n + 1, n + 1))
        self.Sb = np.zeros(n + 1)
        self.m = np.zeros((n + 1, n + 1), dtype=np.int64)
        self.mb = np.zeros(n + 1, dtype=np.int64)

    def AddElement(self, i, j, v):
        self.A[i, j] += v
        self.S[i, j] += abs(v)
        self.m[i, j] += 1

    def AddRHS(self, i, v):
        self.rhs[i] += v
        self.Sb[i] += abs(v)
        self.mb[i] += 1


class Deck:
    """What `stamp` needs of a netlist, parsed once: the oracle front-end's plan (device table) and the product's frozen
    pivot order (Circuit.structure(): 1-based MNA indices)."""

    def __init__(self, text):
        self.text = text
        self.plan = O.OracleCircuit(text).plan
        st = T.Circuit.from_netlist(text).structure()
        self.pivots = list(zip(st["pivot_row"], st["pivot_col"]))
        self.n = self.plan.n_nodes + self.plan.n_branches


Stamped = collections.namedtuple("Stamped", "A b S Sb m mb P Pb")


def _products(c, m, t):
    """Sum of |a * b| over the products that feed an add INSIDE one contribution, where the add can cancel (so that a
    contraction into an FMA is not bounded by u * |contribution|), for the device kinds the fast-build bound covers: a SIN
    source's p1 * sin(arg) + p0, a PWL source's a + slope * (t - t1), and the Level 1 MOSFET's ieq = -id + gds vds + gm vgs
    + gmbs vbs and linear-region gds = beta (vgst - vds)(1 + lambda vds) + beta lambda (vgst vds - vds^2 / 2)."""
    PA, PB = np.zeros_like(m.S), np.zeros_like(m.Sb)
    for d in c.devices:
        if isinstance(d, P.Source) and d.stype in (1, 3):
            p = d.p
            if d.stype == 1:
                v = abs(p[1] * P.go_sin(2.0 * P.PI * p[2] * t + p[3] * P.PI / 180.0))
            else:
                ts, vs = p[0::2], p[1::2]
                v = 0.0
                if ts[0] < t < ts[-1]:
                    i = next(i for i in range(1, len(ts)) if t <= ts[i])
                    v = abs((vs[i] - vs[i - 1]) / (ts[i] - ts[i - 1]) * (t - ts[i - 1]))
            rows = [d.b] if isinstance(d, P.VSource) else [k for k in d.Nodes[:2] if k]
            for r in rows:
                PB[r] += v
        elif isinstance(d, P.Mosfet) and d.Level == 1:
            nd, ng, ns, nb = d.Nodes
            Pieq = abs(d.gds * d.vds) + abs(d.gm * d.vgs) + abs(d.gmbs * d.vbs)
            for r in (nd, ns):
                if r:
                    PB[r] += Pieq
            if d.region == P.LINEAR:
                sg = -1.0 if d.pmos else 1.0
                vgs, vds, vbs = d.vgs * sg, d.vds * sg, d.vbs * sg
                vgst = vgs - d.vth(vbs)
                beta = d.KP * d.W / d.L
                Pg = abs(beta * (vgst - vds) * (1.0 + d.LAMBDA * vds)) + abs(beta * d.LAMBDA) * (abs(vgst * vds) + 0.5 * vds * vds)
                for i, j in ((nd, nd), (nd, ns), (ns, ns), (ns, nd)):
                    if i and j:
                        PA[i, j] += Pg
    return PA[1:, 1:], PB[1:]


def stamp(deck, overrides, mode, time, dt, gmin, libm=None):
    """One instance: Stamped(A [n][n], b [n], S [n][n], Sb [n], m [n][n], mb [n], P [n][n], Pb [n]) in the kernel's 0-based
    layout (m, mb: number of contributions per entry; P, Pb: see _products).  `overrides` maps (device name, parameter index) to this instance's value."""
    if isinstance(deck, str):
        deck = Deck(deck)
    saved = P.math
    P.math = libm if libm is not None else Libm()
    try:
        with np.errstate(all="ignore"):
            c = P.Circuit(deck.plan, overrides)
            m = AbsMatrix(c.n)
            c.M = m
            c.Stamp(P.Status(time, dt, mode, 300.15, gmin))
            if gmin != 0.0:
                for r, k in deck.pivots:
                    m.AddElement(r, k, gmin)
    finally:
        P.math = saved
    return Stamped(m.A[1:, 1:].copy(), m.rhs[1:].copy(), m.S[1:, 1:].copy(), m.Sb[1:].copy(), m.m[1:, 1:].copy(), m.mb[1:].copy(),
                   *_products(c, m, time))


def stamp_batch(deck, params, idx, mode, time, dt, gmin, libm=None):
    """`stamp` of instances `idx` of a batch whose per-instance parameters are `params` {(device, param): array}:
    the fields of Stamped stacked over the instances."""
    if isinstance(deck, str):
        deck = Deck(deck)
    out = [stamp(deck, {key: float(v[i]) for key, v in params.items()}, mode, time, dt, gmin, libm) for i in idx]
    return Stamped(*(np.stack([o[j] for o in out]) for j in range(len(Stamped._fields))))


def source_times(deck, count=3):
    """Times at which the deck's sources sit on an edge: PULSE delay, end of rise, start and end of fall, and the same
    plus k * per for `count` periods; every PWL breakpoint; SIN quarter periods and period multiples.  Sorted, unique."""
    if isinstance(deck, str):
        deck = Deck(deck)
    ts = set()
    for r in deck.plan.devices:
        if r.kind not in (P.K_V, P.K_I) or not r.ip:
            continue
        p = list(r.p)
        if r.ip[0] == 1:
            f = p[2]
            if f > 0:
                ts.update(k / (4.0 * f) for k in range(1, 4 * count + 1))
        elif r.ip[0] == 2:
            v1, v2, delay, rise, fall, pw, per = p
            edges = [delay, delay + rise, delay + rise + pw, delay + rise + pw + fall]
            ts.update(edges)
            if per > 0:
                ts.update(delay + k * per for k in range(1, count + 1))
                ts.update(delay + k * per + rise for k in range(1, count + 1))
                ts.update(delay + k * per + (rise + pw) for k in range(1, count + 1))
        elif r.ip[0] == 3:
            ts.update(p[0::2])
    return sorted(t for t in ts if t >= 0.0)
