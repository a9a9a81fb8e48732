"""ORACLE PIN — TEST INFRASTRUCTURE ONLY.  Not part of the shipped product path.

pin_numpy.py — a SECOND, independent restatement of the reference's device and analysis layers, written from the Go
sources (pkg/device/*.go, pkg/analysis/{op,tran,dc,anlysis}.go, pkg/circuit/circuit.go) and NOT from oracle/engine.hpp:
plain Python floats (IEEE doubles), a dense NumPy matrix, numpy.linalg.solve.  Its purpose is to catch transcription
slips that the C++ oracle and the CUDA device code could share (both were restated by the same hand): tests/test_oracle.py
holds the C++ oracle to this restatement at 1e-9 relative on every device kind, with identical step / row / solve counts.

What it deliberately does NOT restate: the sparse LU (LAPACK's partial pivoting solves the same systems; the pivot
order only matters at kappa*eps), the netlist front-end (the device table comes from oracle/netlist.py, which is pinned
separately against the product's C++ front-end), and LoadGmin with a non-zero gmin (Gmin stepping adds to the pivot
positions of the factorisation, matrix/circuit.go:107-114 — decks that reach that fallback are outside this pin).

Only tests/ may import this module.
"""
from __future__ import annotations

import math
from decimal import Decimal

import numpy as np

K_R, K_C, K_L, K_V, K_I, K_D, K_Q, K_M, K_K, K_LCORE = range(10)
OP_MODE, TRAN_MODE = 0, 1
CHARGE, BOLTZMANN, KELVIN = 1.6021918e-19, 1.3806226e-23, 273.15            # internal/consts/consts.go:4-6
# Go evaluates constant expressions exactly and rounds once: 4*math.Pi*1e-7 (magnetic.go:11) and 4.0e-7*math.Pi (:240)
MU0 = float(Decimal("3.14159265358979323846264338327950288419716939937510582097494459") * 4 * Decimal("1e-7"))
PI = math.pi


class SingularMatrix(Exception):
    pass


class Status:
    """device.CircuitStatus (device.go:85-97): the fields any device reads."""

    def __init__(self, time=0.0, dt=0.0, mode=OP_MODE, temp=0.0, gmin=0.0):
        self.Time, self.TimeStep, self.Mode, self.Temp, self.Gmin = time, dt, mode, temp, gmin


class Matrix:
    """matrix.CircuitMatrix (matrix/circuit.go): 1-based accumulate, Solve, Solution with [0] = 0."""

    def __init__(self, n):
        self.n = n
        self.A = np.zeros((n + 1, n + 1))
        self.rhs = np.zeros(n + 1)
        self.solution = np.zeros(n + 1)
        self.n_solves = 0

    def Clear(self):
        self.A[:] = 0.0
        self.rhs[:] = 0.0

    def AddElement(self, i, j, v):
        self.A[i, j] += v

    def AddRHS(self, i, v):
        self.rhs[i] += v

    def Solve(self):
        self.n_solves += 1
        A = self.A[1:, 1:]
        with np.errstate(all="ignore"):
            if not np.all(np.isfinite(A)) or not np.all(np.isfinite(self.rhs[1:])):
                x = np.full(self.n, np.nan)                   # Inf / NaN flow through the reference's LU too
            else:
                try:
                    x = np.linalg.solve(A, self.rhs[1:])
                except np.linalg.LinAlgError:
                    raise SingularMatrix()
        self.solution = np.concatenate([[0.0], x])


# ------------------------------------------------------------------------------------------- Go's math where it is not libm's
_SIN = (1.58962301576546568060e-10, -2.50507477628578072866e-8, 2.75573136213857245213e-6, -1.98412698295895385996e-4,
        8.33333333332211858878e-3, -1.66666666666666307295e-1)
_COS = (-1.13585365213876817300e-11, 2.08757008419747316778e-9, -2.75573141792967388112e-7, 2.48015872888517045348e-5,
        -1.38888888888730564116e-3, 4.16666666666665929218e-2)


def go_sin(x):
    """math.Sin (Go src/math/sin.go; pure Go on amd64): Cody-Waite reduction by pi/4 in three parts and the Cephes
    polynomials.  It differs from libm's sine in the last bit.  |x| >= 2^29 (Payne-Hanek in Go) is not restated: libm."""
    if x == 0 or x != x:
        return x
    if math.isinf(x):
        return math.nan
    sign = x < 0
    x = abs(x)
    if x >= 536870912.0:
        return -math.sin(x) if sign else math.sin(x)
    j = int(x * 1.2732395447351626861510701069801148)         # 4/Pi, a Go constant: rounded once
    y = float(j)
    if j & 1:
        j += 1
        y += 1.0
    j &= 7
    z = ((x - y * 7.85398125648498535156e-1) - y * 3.77489470793079817668e-8) - y * 2.69515142907905952645e-15
    if j > 3:
        sign = not sign
        j -= 4
    zz = z * z
    if j == 1 or j == 2:
        c = _COS
        y = 1.0 - 0.5 * zz + zz * zz * ((((((c[0] * zz) + c[1]) * zz + c[2]) * zz + c[3]) * zz + c[4]) * zz + c[5])
    else:
        c = _SIN
        y = z + z * zz * ((((((c[0] * zz) + c[1]) * zz + c[2]) * zz + c[3]) * zz + c[4]) * zz + c[5])
    return -y if sign else y


def _is_odd_int(y):
    return abs(y) < 2.0 ** 53 and y == math.floor(y) and int(y) % 2 == 1


def go_pow(x, y):
    """math.Pow (Go src/math/pow.go): the special cases, Sqrt for y = +-0.5, otherwise Exp(yf * Log(x)) for the fractional
    part of |y| (yf in (-0.5, 0.5]) times the integer power by repeated squaring of the Frexp mantissa, one Ldexp at the
    end — a few ulp from the correctly rounded power that libm's pow returns."""
    if y == 0 or x == 1:
        return 1.0
    if y == 1:
        return x
    if x != x or y != y:
        return math.nan
    if x == 0:
        if y < 0:
            return -math.inf if math.copysign(1.0, x) < 0 and _is_odd_int(y) else math.inf
        return x if math.copysign(1.0, x) < 0 and _is_odd_int(y) else 0.0
    if math.isinf(y):
        if x == -1:
            return 1.0
        return 0.0 if (abs(x) < 1) == (y > 0) else math.inf
    if math.isinf(x):
        if x < 0:
            return go_pow(1 / x, -y)
        return 0.0 if y < 0 else math.inf
    if y == 0.5:
        return math.sqrt(x) if x >= 0 else math.nan
    if y == -0.5:
        return 1 / math.sqrt(x) if x > 0 else math.nan
    yf, yi = math.modf(abs(y))
    if yf != 0 and x < 0:
        return math.nan
    if yi >= 2.0 ** 63:
        if x == -1:
            return 1.0
        return 0.0 if (abs(x) < 1) == (y > 0) else math.inf
    a1, ae = 1.0, 0
    if yf != 0:
        if yf > 0.5:
            yf -= 1
            yi += 1
        a1 = math.exp(yf * math.log(x))
    x1, xe = math.frexp(x)
    i = int(yi)
    while i != 0:
        if xe < -(1 << 12) or (1 << 12) < xe:
            ae += xe
            break
        if i & 1:
            a1 *= x1
            ae += xe
        x1 *= x1
        xe <<= 1
        if x1 < 0.5:
            x1 += x1
            xe -= 1
        i >>= 1
    if y < 0:
        a1 = math.copysign(math.inf, a1) if a1 == 0 else 1 / a1
        ae = -ae
    try:
        return math.ldexp(a1, ae)
    except OverflowError:
        return math.copysign(math.inf, a1)


def _v(voltages, node):
    return voltages[node] if node != 0 else 0.0


# ------------------------------------------------------------------------------------------- devices
class Resistor:                                                     # resistor.go
    typ, nonlinear, time_dependent = "R", False, False

    def __init__(self, row):
        self.name, self.Nodes, self.Value = row.name, list(row.nodes), row.p[0]

    def Stamp(self, m, st):                                         # :32-75
        n1, n2 = self.Nodes
        dt = st.Temp - 300.15
        g = 1.0 / (self.Value * (1.0 + 0.0 * dt + 0.0 * dt * dt))   # :77-81, Tc1 = Tc2 = 0
        if n1 != 0:
            m.AddElement(n1, n1, g)
            if n2 != 0:
                m.AddElement(n1, n2, -g)
        if n2 != 0:
            if n1 != 0:
                m.AddElement(n2, n1, -g)
            m.AddElement(n2, n2, g)


class Capacitor:                                                    # capacitor.go
    typ, nonlinear, time_dependent = "C", False, True

    def __init__(self, row):
        self.name, self.Nodes, self.Value = row.name, list(row.nodes), row.p[0]
        self.Voltage0 = self.Voltage1 = self.charge0 = self.charge1 = 0.0

    def Stamp(self, m, st):                                         # :43-109
        n1, n2 = self.Nodes
        if st.Mode == OP_MODE:
            g = st.Gmin if st.Gmin >= 1e-12 else 1e-12
            ceq = None
        else:
            g = self.Value / st.TimeStep
            ceq = self.charge1 / st.TimeStep
        if n1 != 0:
            m.AddElement(n1, n1, g)
            if n2 != 0:
                m.AddElement(n1, n2, -g)
            if ceq is not None:
                m.AddRHS(n1, ceq)
        if n2 != 0:
            m.AddElement(n2, n2, g)
            if n1 != 0:
                m.AddElement(n2, n1, -g)
            if ceq is not None:
                m.AddRHS(n2, -ceq)

    def SetTimeStep(self, dt, st):
        st.TimeStep = dt

    def LoadState(self, v, st):                                     # :111-124 (only sets the unused current0)
        pass

    def UpdateState(self, v, st):                                   # :155-171
        vd = _v(v, self.Nodes[0]) - _v(v, self.Nodes[1])
        self.charge1 = self.charge0
        self.charge0 = self.Value * vd
        self.Voltage1 = self.Voltage0
        self.Voltage0 = vd

    def CalculateLTE(self, st):                                     # :173-178
        return abs(self.Value * self.Voltage0 - self.Value * self.Voltage1) / (2.0 * st.TimeStep)


def _bdf1(dt):                                                      # util/integrator.go:33-48, order 1
    return 1.0 / (1.0 * dt)


class Inductor:                                                     # inductor.go
    typ, nonlinear, time_dependent = "L", False, True

    def __init__(self, row):
        self.name, self.Nodes, self.Value, self.b = row.name, list(row.nodes), row.p[0], row.branch
        self.Current0 = self.Current1 = self.Voltage0 = self.Voltage1 = 0.0

    def Stamp(self, m, st):                                         # :58-76
        n1, n2, b = self.Nodes[0], self.Nodes[1], self.b
        if n1 != 0:
            m.AddElement(n1, b, -1)
            m.AddElement(b, n1, -1)
        if n2 != 0:
            m.AddElement(n2, b, 1)
            m.AddElement(b, n2, 1)
        dt = st.TimeStep
        if dt <= 0:
            dt = 1e-9
        c0 = _bdf1(dt)
        m.AddElement(b, b, -c0 * self.Value)
        m.AddRHS(b, c0 * self.Value * self.Current1)

    def SetTimeStep(self, dt, st):
        st.TimeStep = dt

    def LoadState(self, v, st):                                     # :81-95
        vd = _v(v, self.Nodes[0]) - _v(v, self.Nodes[1])
        self.Current0 = self.Current1 + (vd * st.TimeStep) / self.Value

    def UpdateState(self, v, st):                                   # :97-114
        self.Voltage1 = self.Voltage0
        self.Voltage0 = _v(v, self.Nodes[0]) - _v(v, self.Nodes[1])
        self.Current1 = self.Current0
        self.Current0 = self.Voltage0 / (self.Value / 1e-9)

    def CalculateLTE(self, st):                                     # :116-121
        return max(abs(self.Current0 - self.Current1) / (2.0 * st.TimeStep), abs(self.Voltage0 - self.Voltage1) / (2.0 * st.TimeStep))

    def GetValue(self):
        return self.Value

    def GetCurrent(self):
        return self.Current0


class Source:
    """vsource.go / isource.go waveforms.  p layout per source type (include/tspice_b200.h)."""

    def __init__(self, row):
        self.name, self.Nodes, self.b = row.name, list(row.nodes), row.branch
        self.stype = row.ip[0] if row.ip else 0
        self.p = list(row.p)

    def value(self, t):                                             # vsource.go:113-127
        p = self.p
        if self.stype == 0:
            return p[0]
        if self.stype == 1:
            return p[0] + p[1] * go_sin(2.0 * PI * p[2] * t + p[3] * PI / 180.0)
        if self.stype == 2:                                         # :179-209
            v1, v2, delay, rise, fall, pw, per = p
            if t < delay:
                return v1
            t = t - delay
            if per > 0:
                t = math.fmod(t, per)
            if t < rise:
                return v2 if rise == 0 else v1 + (v2 - v1) * t / rise
            if t < rise + pw:
                return v2
            fs = rise + pw
            if t < fs + fall:
                return v1 if fall == 0 else v2 - (v2 - v1) * (t - fs) / fall
            return v1
        times, vals = p[0::2], p[1::2]                              # :211-231
        if t <= times[0]:
            return vals[0]
        if t >= times[-1]:
            return vals[-1]
        for i in range(1, len(times)):
            if t <= times[i]:
                slope = (vals[i] - vals[i - 1]) / (times[i] - times[i - 1])
                return vals[i - 1] + slope * (t - times[i - 1])
        return vals[-1]

    def SetValue(self, v):                                          # :241-244 — reaches dcValue only
        if self.stype in (0, 1):
            self.p[0] = v

    def GetValue(self):
        # BaseDevice.Value: the DC value / SIN offset / PULSE v1 / first PWL value given at construction (vsource.go:36-96)
        return self.p[1] if self.stype == 3 else self.p[0]


class VSource(Source):
    typ, nonlinear, time_dependent = "V", False, False

    def Stamp(self, m, st):                                         # vsource.go:131-152
        n1, n2, b = self.Nodes[0], self.Nodes[1], self.b
        if n1 != 0:
            m.AddElement(b, n1, 1)
            m.AddElement(n1, b, 1)
        if n2 != 0:
            m.AddElement(b, n2, -1)
            m.AddElement(n2, b, -1)
        m.AddRHS(b, self.value(st.Time))


class ISource(Source):
    typ, nonlinear, time_dependent = "I", False, False

    def Stamp(self, m, st):                                         # isource.go:130-147
        n1, n2 = self.Nodes[0], self.Nodes[1]
        cur = self.value(st.Time)
        if n1 != 0:
            m.AddRHS(n1, cur)
        if n2 != 0:
            m.AddRHS(n2, -cur)


def _vt(temp):                                                      # diode.go:78-84, bjt.go:122-127
    if temp <= 0:
        temp = 300.15
    return BOLTZMANN * temp / CHARGE


class Diode:                                                        # diode.go
    typ, nonlinear, time_dependent = "D", True, False               # no LoadState method -> not TimeDependent (SURVEY Q11)

    def __init__(self, row):
        self.name, self.Nodes = row.name, list(row.nodes)
        self.Is, self.N, self.Tt = row.p[:3]
        self.Eg, self.Xti, self.Gmin = 1.11, 3.0, 1e-12
        self.vd = 0.0
        self.prevCharge = 0.0

    def adjIs(self, temp):                                          # :108-117
        vt = _vt(temp)
        ratio = temp / (KELVIN + 27)
        egfact = -self.Eg / (2 * vt) * (temp / (KELVIN + 27) - 1.0)
        return self.Is * go_pow(ratio, self.Xti / self.N) * math.exp(egfact)

    def Stamp(self, m, st):                                         # :184-227
        nvt = self.N * _vt(st.Temp)
        vd = self.vd
        if vd > -3.0 * nvt:                                         # :119-148
            arg = vd / nvt
            if arg > 40.0:
                arg = 40.0
            idc = self.adjIs(st.Temp) * (math.exp(arg) - 1.0)
            gd = (abs(idc) + self.adjIs(st.Temp)) / nvt + self.Gmin
        else:
            idc = -self.adjIs(st.Temp)
            gd = self.Gmin
        if st.Mode == TRAN_MODE:
            charge = self.Tt * idc
            if st.TimeStep > 0:
                cap = (charge - self.prevCharge) / st.TimeStep
                geq = self.Tt * gd / st.TimeStep
                gd += geq
                idc += cap
        n1, n2 = self.Nodes
        if n1 != 0:
            m.AddElement(n1, n1, gd)
            if n2 != 0:
                m.AddElement(n1, n2, -gd)
            m.AddRHS(n1, -(idc - gd * vd))
        if n2 != 0:
            if n1 != 0:
                m.AddElement(n2, n1, -gd)
            m.AddElement(n2, n2, gd)
            m.AddRHS(n2, (idc - gd * vd))

    def UpdateVoltages(self, v):                                    # :307-324
        self.vd = _v(v, self.Nodes[0]) - _v(v, self.Nodes[1])


def _exp(x):
    try:
        return math.exp(x)
    except OverflowError:
        return math.inf


class Bjt:                                                          # bjt.go
    typ, nonlinear, time_dependent = "Q", True, False

    def __init__(self, row):
        self.name, self.Nodes = row.name, list(row.nodes)
        (self.Ies, self.Ics, self.AlphaF, self.Ikf, self.Ikr, self.Vaf, self.Var, self.Nf, self.Nr) = row.p[:9]
        self.pnp = bool(row.ip and row.ip[0])
        self.vbe = self.vbc = self.vce = 0.0

    def Stamp(self, m, st):                                         # :315-374
        nc, nb, ne = self.Nodes
        vt = _vt(st.Temp)
        if self.vbe == 0 and self.vce == 0:                         # :110-120
            self.vbe = self.Nf * vt * math.log(1e-3 / self.Ies)
            self.vce = max(2.0, self.vbe + 1.0)
            self.vbc = self.vbe - self.vce
        with np.errstate(all="ignore"):
            f = np.float64
            vbe, vbc, vce = f(self.vbe), f(self.vbc), f(self.vce)
            expVbe = f(_exp(vbe / (self.Nf * vt)))                  # :214-255
            expVbc = f(_exp(vbc / (self.Nr * vt)))
            sign = -1.0 if self.pnp else 1.0
            iF0 = sign * self.Ies * (expVbe - 1)
            iR0 = sign * self.Ics * (expVbc - 1)
            iF = iF0 * (1 - vbc / self.Vaf) if self.Vaf > 0 else iF0
            iR = iR0 * (1 + vbe / self.Var) if self.Var > 0 else iR0
            qb = f(1.0) / (1 - vbc / self.Vaf) if self.Vaf > 0 else f(1.0)
            if self.Ikf > 0:
                iF = iF / (1 + abs(iF) / (self.Ikf * qb))
            if self.Ikr > 0:
                iR = iR / (1 + abs(iR) / (self.Ikr * qb))
            ie = sign * (iF - iR)
            ic = sign * ((self.AlphaF * iF - iR) / qb)
            ib = ie - ic
            dIes = self.Ies * expVbe / (self.Nf * vt)               # :257-281
            gm = self.AlphaF * dIes / qb
            gpi = abs(ib) / vt
            if self.Vaf != 0:
                gout = self.AlphaF * self.Ies * (expVbe - 1) * (1 / self.Vaf) * (f(1.0) / ((1 + vce / self.Vaf) * (1 + vce / self.Vaf)))
            else:
                gout = 1e-12
            if nc != 0:
                m.AddElement(nc, nc, gout)
                if nb != 0:
                    m.AddElement(nc, nb, -gout - gm)
                if ne != 0:
                    m.AddElement(nc, ne, gm)
                m.AddRHS(nc, -ic + gout * vce)
            if nb != 0:
                m.AddElement(nb, nb, gpi)
                if nc != 0:
                    m.AddElement(nb, nc, -gpi)
                m.AddRHS(nb, -ib + gpi * vbe)
            if ne != 0:
                m.AddElement(ne, ne, gpi + gm)
                if nb != 0:
                    m.AddElement(ne, nb, -gpi - gm)
                m.AddRHS(ne, -ie)

    def UpdateVoltages(self, v):                                    # :283-313
        vc, vb, ve = (_v(v, n) for n in self.Nodes)
        if self.pnp:
            self.vbe, self.vbc, self.vce = ve - vb, vc - vb, ve - vc
        else:
            self.vbe, self.vbc, self.vce = vb - ve, vb - vc, vc - ve


CUTOFF, LINEAR, SATURATION = 0, 1, 2
_MOS_KEYS = ("VTO KP GAMMA PHI LAMBDA W L TOX CGSO CGDO CGBO CBD CBS CJ CJSW AS AD PS PD MJ PB UO UCRIT UEXP VMAX THETA ETA "
             "KAPPA DELTA").split()


class Mosfet:                                                       # mosfet.go
    typ, nonlinear, time_dependent = "M", True, False

    def __init__(self, row):
        self.name, self.Nodes = row.name, list(row.nodes)
        for k, val in zip(_MOS_KEYS, row.p):
            setattr(self, k, val)
        self.Level, self.pmos = int(row.ip[0]), bool(row.ip[1])
        self.vgs = self.vds = self.vbs = self.vgd = self.vbd = 0.0
        self.gm = self.gds = self.gmbs = 0.0
        self.id, self.region = 0.0, CUTOFF

    def vth(self, vbs):                                             # :296-318
        if self.GAMMA > 0:
            v = self.VTO + self.GAMMA * (math.sqrt(max(0.0, self.PHI - vbs)) - math.sqrt(self.PHI))
            return -v if self.pmos else v
        return -self.VTO if self.pmos else self.VTO

    def currents(self, vgs, vds, vbs):                              # :321-355
        sign = 1.0
        if self.pmos:
            vgs, vds, vbs, sign = -vgs, -vds, -vbs, -1.0
        vth = self.vth(vbs)
        vgst = vgs - vth
        if vgst <= 0:
            return 0.0, CUTOFF
        if self.Level == 2:                                         # :378-420
            cox = (3.9 * 8.85e-14) / self.TOX
            eeff = vgst / (self.TOX * 100)
            ueff = self.UO
            if self.UCRIT > 0 and eeff > 0:
                ueff /= (1.0 + go_pow(eeff / self.UCRIT, self.UEXP))
            vdsat = vgst
            if self.VMAX > 0:
                ecrit = self.VMAX / ueff * 100
                vdsat = min(vgst, ecrit * self.L)
            beta = ueff * cox * self.W / (self.L * 100)
            if vds < vdsat:
                i, reg = beta * (vgst * vds - 0.5 * vds * vds) * (1.0 + self.LAMBDA * vds), LINEAR
            else:
                i, reg = 0.5 * beta * vdsat * vdsat * (1.0 + self.LAMBDA * vds), SATURATION
        elif self.Level == 3:                                       # :423-459
            ve = vgst / (1.0 + self.THETA * vgst) if self.THETA > 0 else vgst
            vdsat = ve / math.sqrt(1.0 + self.KAPPA * ve) if self.KAPPA > 0 else ve
            beta = self.KP * self.W / self.L
            if self.DELTA > 0:
                beta /= (1.0 + self.DELTA / self.W)
            if vds < vdsat:
                i, reg = beta * (ve * vds - 0.5 * vds * vds / (1.0 + self.KAPPA * ve)) * (1.0 + self.LAMBDA * vds), LINEAR
            else:
                i, reg = 0.5 * beta * vdsat * vdsat * (1.0 + self.LAMBDA * vds), SATURATION
        else:                                                       # :358-375
            beta = self.KP * self.W / self.L
            if vds < vgst:
                i, reg = beta * (vgst * vds - 0.5 * vds * vds) * (1.0 + self.LAMBDA * vds), LINEAR
            else:
                i, reg = 0.5 * beta * vgst * vgst * (1.0 + self.LAMBDA * vds), SATURATION
        return sign * i, reg

    def conductances(self):                                         # :462-537
        sign = -1.0 if self.pmos else 1.0
        vgs, vds, vbs = self.vgs * sign, self.vds * sign, self.vbs * sign
        vgst = vgs - self.vth(vbs)
        beta = self.KP * self.W / self.L
        gmin = 1e-12
        if self.region == CUTOFF:
            self.gm = self.gds = self.gmbs = gmin
            return
        if self.GAMMA > 0 and self.PHI > 0:
            self.gmbs = self.gm * self.GAMMA / (2.0 * math.sqrt(self.PHI - vbs)) if vbs < 0 else gmin
        else:
            self.gmbs = gmin
        if self.Level == 1:
            if self.region == LINEAR:
                self.gm = beta * vds * (1.0 + self.LAMBDA * vds)
                self.gds = beta * (vgst - vds) * (1.0 + self.LAMBDA * vds) + beta * self.LAMBDA * (vgst * vds - 0.5 * vds * vds)
            else:
                self.gm = beta * vgst * (1.0 + self.LAMBDA * vds)
                self.gds = 0.5 * beta * vgst * vgst * self.LAMBDA
        elif self.Level in (2, 3):
            delta = 1e-6
            id0 = self.id
            self.gm = max((self.currents(vgs + delta, vds, vbs)[0] - id0) / delta, gmin)
            self.gds = max((self.currents(vgs, vds + delta, vbs)[0] - id0) / delta, gmin)
            self.gmbs = max((self.currents(vgs, vds, vbs + delta)[0] - id0) / delta, gmin)
        self.gm *= sign
        self.gmbs *= sign

    def Stamp(self, m, st):                                         # :668-786
        nd, ng, ns, nb = self.Nodes
        if self.vgs == 0 and self.vds == 0 and self.vbs == 0:
            self.vgs, self.vds = (-0.7, -0.1) if self.pmos else (0.7, 0.1)
            self.vbs = 0.0
            self.vgd = self.vgs - self.vds
            self.vbd = self.vbs - self.vds
        self.id, self.region = self.currents(self.vgs, self.vds, self.vbs)
        self.conductances()
        # calculateCapacitances :540-594
        cgate = (3.9 * 8.85e-14 / self.TOX) * self.W * self.L
        cgso, cgdo, cgbo = self.CGSO * self.W, self.CGDO * self.W, self.CGBO * self.L
        if self.CBS == 0 and self.CJ > 0:
            self.CBS = self.CJ * self.AS + self.CJSW * self.PS
        if self.CBD == 0 and self.CJ > 0:
            self.CBD = self.CJ * self.AD + self.CJSW * self.PD
        if self.region == CUTOFF:
            cgb, cgs, cgd = 2.0 * cgate / 3.0, cgso, cgdo
        elif self.region == LINEAR:
            cgs, cgd, cgb = cgate / 2.0 + cgso, cgate / 2.0 + cgdo, cgbo
        else:
            cgs, cgd, cgb = 2.0 * cgate / 3.0 + cgso, cgdo, cgbo + cgate / 3.0
        gmin = st.Gmin
        ieq = -self.id + self.gds * self.vds + self.gm * self.vgs + self.gmbs * self.vbs
        if nd != 0:
            m.AddElement(nd, nd, self.gds + gmin)
            if ng != 0:
                m.AddElement(nd, ng, self.gm)
            if ns != 0:
                m.AddElement(nd, ns, -self.gds - self.gm - self.gmbs)
            if nb != 0:
                m.AddElement(nd, nb, self.gmbs)
            m.AddRHS(nd, ieq)
        if ns != 0:
            m.AddElement(ns, ns, self.gds + self.gm + self.gmbs + gmin)
            if nd != 0:
                m.AddElement(ns, nd, -self.gds)
            if ng != 0:
                m.AddElement(ns, ng, -self.gm)
            if nb != 0:
                m.AddElement(ns, nb, -self.gmbs)
            m.AddRHS(ns, self.id - self.gds * self.vds - self.gm * self.vgs - self.gmbs * self.vbs)
        if st.Mode == TRAN_MODE and st.TimeStep > 0:
            dt = st.TimeStep
            # calculateCharges :597-637; the prevQ* never advance (the device is not TimeDependent, SURVEY Q11)
            if self.region == CUTOFF:
                qgs, qgd = 0.0, 0.0
            else:
                qgs, qgd = cgs * self.vgs, cgd * self.vgd
            qgb = cgb * (self.vgs - self.vbs)
            cbs = self.CBS / go_pow(1.0 - self.vbs / self.PB, self.MJ) if self.vbs < 0 else self.CBS * (1.0 + self.MJ * self.vbs / self.PB)
            cbd = self.CBD / go_pow(1.0 - self.vbd / self.PB, self.MJ) if self.vbd < 0 else self.CBD * (1.0 + self.MJ * self.vbd / self.PB)
            qbs, qbd = cbs * self.vbs, cbd * self.vbd
            icgs, icgd, icgb, icbs, icbd = (qgs - 0.0) / dt, (qgd - 0.0) / dt, (qgb - 0.0) / dt, (qbs - 0.0) / dt, (qbd - 0.0) / dt
            if ng != 0:
                if nd != 0:
                    m.AddElement(ng, nd, cgd / dt); m.AddElement(nd, ng, cgd / dt)
                    m.AddRHS(ng, icgd); m.AddRHS(nd, -icgd)
                if ns != 0:
                    m.AddElement(ng, ns, cgs / dt); m.AddElement(ns, ng, cgs / dt)
                    m.AddRHS(ng, icgs); m.AddRHS(ns, -icgs)
                if nb != 0:
                    m.AddElement(ng, nb, cgb / dt); m.AddElement(nb, ng, cgb / dt)
                    m.AddRHS(ng, icgb); m.AddRHS(nb, -icgb)
                m.AddElement(ng, ng, (cgd + cgs + cgb) / dt)
            if nb != 0:
                if ns != 0:
                    m.AddElement(nb, ns, self.CBS / dt); m.AddElement(ns, nb, self.CBS / dt)
                    m.AddRHS(nb, icbs); m.AddRHS(ns, -icbs)
                if nd != 0:
                    m.AddElement(nb, nd, self.CBD / dt); m.AddElement(nd, nb, self.CBD / dt)
                    m.AddRHS(nb, icbd); m.AddRHS(nd, -icbd)
                m.AddElement(nb, nb, (self.CBD + self.CBS) / dt)

    def UpdateVoltages(self, v):                                    # :640-665 — voltages[0] is read for grounded terminals
        vd, vg, vs, vb = (v[n] for n in self.Nodes)
        t = -1.0 if self.pmos else 1.0
        self.vgs, self.vds, self.vbs = t * (vg - vs), t * (vd - vs), t * (vb - vs)
        self.vgd = self.vgs - self.vds
        self.vbd = self.vbs - self.vds


class MagneticInductor:                                             # magnetic.go (the reachable, air-core branch: SURVEY Q12)
    typ, nonlinear, time_dependent = "L", False, False              # has no TimeDependent method set -> state never advances

    def __init__(self, row):
        self.name, self.Nodes, self.b = row.name, list(row.nodes), row.branch
        self.turns, self.area, self.len = int(row.p[0]), row.p[1], row.p[2]
        self.current0 = self.current1 = 0.0

    def L0(self):
        return MU0 * float(self.turns * self.turns) * self.area / self.len

    def GetValue(self):                                             # :147-154 with Calculate(0) -> dMdH = 0 (:88-94)
        return MU0 * float(self.turns * self.turns) * self.area * (1 + 0.0) / self.len

    def GetCurrent(self):
        return self.current0

    def Stamp(self, m, st):                                         # :197-274
        n1, n2, b = self.Nodes[0], self.Nodes[1], self.b
        if n1 != 0:
            m.AddElement(n1, b, -1)
            m.AddElement(b, n1, -1)
        if n2 != 0:
            m.AddElement(n2, b, 1)
            m.AddElement(b, n2, 1)
        if st.Mode == OP_MODE:
            m.AddElement(b, b, 1e-3)
            self.current0 = self.current1 = 0.0
        else:
            dt = st.TimeStep if st.TimeStep > 0 else 1e-9
            assert st.Time < dt or abs(self.current0) < 1e-9        # current0 never advances: always the linear branch
            diag = _bdf1(dt) * self.L0()
            m.AddElement(b, b, -diag)
            m.AddRHS(b, diag * self.current1)


class Mutual:                                                       # mutual.go:57-120
    typ, nonlinear, time_dependent = "K", False, False

    def __init__(self, row, inductors):
        self.name, self.k, self.inductors = row.name, row.p[0], inductors

    def Stamp(self, m, st):
        if st.Mode != TRAN_MODE or st.TimeStep <= 0:
            return
        dt = st.TimeStep
        info = [(ind.b, ind.GetValue(), ind.GetCurrent()) for ind in self.inductors]
        for i in range(len(info)):
            for j in range(i + 1, len(info)):
                Mij = self.k * math.sqrt(info[i][1] * info[j][1])
                m.AddElement(info[i][0], info[j][0], -Mij / dt)
                m.AddElement(info[j][0], info[i][0], -Mij / dt)
                m.AddRHS(info[i][0], -Mij * info[j][2] / dt)
                m.AddRHS(info[j][0], -Mij * info[i][2] / dt)


_CTORS = {K_R: Resistor, K_C: Capacitor, K_L: Inductor, K_V: VSource, K_I: ISource, K_D: Diode, K_Q: Bjt, K_M: Mosfet,
          K_LCORE: MagneticInductor}


# ------------------------------------------------------------------------------------------- circuit
class Circuit:
    """circuit.go: devices in netlist order with the mutual couplings last (:83-152), the set-up stamp (:154-156)."""

    def __init__(self, plan, overrides=None):
        self.n_nodes, self.n_branches = plan.n_nodes, plan.n_branches
        self.n = self.n_nodes + self.n_branches
        rows = [type("Row", (), dict(kind=r.kind, name=r.name, nodes=list(r.nodes), branch=r.branch, p=list(r.p), ip=list(r.ip)))
                for r in plan.devices]
        for (dev, par), val in (overrides or {}).items():
            idx = dev if isinstance(dev, int) else [r.name for r in rows].index(dev)
            rows[idx].p[par] = float(val)
        by_index, self.devices = {}, []
        for k, r in enumerate(rows):
            if r.kind == K_K:
                continue
            d = _CTORS[r.kind](r)
            by_index[k] = d
            self.devices.append(d)
        for k, r in enumerate(rows):
            if r.kind == K_K:
                self.devices.append(Mutual(r, [by_index[i] for i in r.ip]))
        self.M = Matrix(self.n)
        self.Status = Status()
        for d in self.devices:                                      # initial stamp with CircuitStatus{Time: 0}
            d.Stamp(self.M, Status())
        self.r_order = [d for d in self.devices if d.typ == "R"]

    def Stamp(self, st):
        for d in self.devices:
            d.Stamp(self.M, st)

    def UpdateNonlinearVoltages(self, sol):
        for d in self.devices:
            if d.nonlinear:
                d.UpdateVoltages(sol)

    def SetTimeStep(self, dt):                                      # :178-190
        self.Status.TimeStep = dt
        for d in self.devices:
            if d.time_dependent:
                d.SetTimeStep(dt, self.Status)

    def LoadState(self):
        for d in self.devices:
            if d.time_dependent:
                d.LoadState(self.M.solution, self.Status)

    def Update(self):
        for d in self.devices:
            if d.time_dependent:
                d.UpdateState(self.M.solution, self.Status)

    def GetSolution(self):                                          # :242-273, in the column order of the batched engine
        s = self.M.solution
        out = [s[i] for i in range(1, self.n_nodes + 1)]
        out += [-s[i] for i in range(self.n_nodes + 1, self.n + 1)]
        out += [(_v(s, d.Nodes[0]) - _v(s, d.Nodes[1])) / d.Value for d in self.r_order]
        return out


# ------------------------------------------------------------------------------------------- analyses
MAXITER, ABSTOL, RELTOL, GMIN = 100, 1e-12, 1e-6, 1e-12             # anlysis.go:35-44


def _op_converged(sol, old):                                        # op.go:67-77 / tran.go:192-207
    for i in range(1, len(sol)):
        if abs(sol[i] - old[i]) > RELTOL * max(abs(sol[i]), abs(old[i])) + ABSTOL:
            return False
    return True


class OperatingPoint:                                               # op.go
    def __init__(self, ckt):
        self.c = ckt
        self.path = 0

    def doNRiter(self, gmin, initial):                              # :25-88
        c, m = self.c, self.c.M
        assert gmin == 0, "Gmin stepping is outside this pin (LoadGmin adds to the LU's pivot positions)"
        old = np.array(initial, dtype=float) if initial is not None else np.zeros(c.n + 1)
        c.Status = Status(0.0, 0.0, OP_MODE, 300.15, gmin)
        for it in range(MAXITER):
            m.Clear()
            c.UpdateNonlinearVoltages(old)
            c.Stamp(c.Status)
            try:
                m.Solve()
            except SingularMatrix:
                return False
            if it > 0 and _op_converged(m.solution, old):
                return True
            old = m.solution.copy()
        return False

    def calculateInitialEstimate(self):                             # :90-111
        c = self.c
        init = Matrix(c.n)
        for d in c.devices:
            if not d.nonlinear:
                d.Stamp(init, c.Status)
        c.M.n_solves += 1
        try:
            init.Solve()
        except SingularMatrix:
            return None
        return init.solution

    def Execute(self):                                              # :171-233 (direct path only)
        init = self.calculateInitialEstimate()
        if init is not None:
            self.c.UpdateNonlinearVoltages(init)
        if self.doNRiter(0, init):
            self.result = self.c.M.solution[1:].copy()              # storeResults: I(branch) = +x[b]
            return True
        raise NotImplementedError("operating point needs Gmin / source stepping: outside this pin")


def _fmt_time(v):                                                   # util/formatter.go:8-24
    a = abs(v)
    if a >= 1:
        return "%.3f s" % v
    if a >= 1e-3:
        return "%.3f ms" % (v * 1e3)
    if a >= 1e-6:
        return "%.3f us" % (v * 1e6)
    if a >= 1e-9:
        return "%.3f ns" % (v * 1e9)
    if a >= 1e-12:
        return "%.3f ps" % (v * 1e12)
    return "%.3e s" % v


class Transient:                                                    # tran.go
    def __init__(self, ckt, tstart, tstop, tstep, tmax, uic=False, max_accepted=None):
        if tstep > tstop / 300:                                     # :29-55
            tstep = tstop / 300
        self.c = ckt
        self.startTime, self.stopTime, self.timeStep, self.maxStep = tstart, tstop, tstep, (tmax if tmax != 0 else tstep)
        self.minStep = tstep / 50.0
        self.useUIC, self.trtol, self.time = uic, 7.0, 0.0
        self.rows, self.accepted, self.rejected = [], 0, 0
        self.max_accepted = max_accepted        # stop early (pin of the first part of a long run); None = the whole run
        self.failed_at = None

    def doNRiter(self):                                             # :157-216
        c, m = self.c, self.c.M
        st = Status(self.time, self.timeStep, TRAN_MODE, 300.15, 0.0)
        old = None
        for it in range(MAXITER):
            m.Clear()
            if it > 0:
                c.UpdateNonlinearVoltages(old)
            c.Stamp(st)
            try:
                m.Solve()
            except SingularMatrix:
                return False
            if it > 0 and _op_converged(m.solution, old):
                return True
            old = m.solution.copy()
        return False

    def run(self):                                                  # Setup :57-75 + Execute :77-155
        c = self.c
        if not self.useUIC:
            OperatingPoint(c).Execute()
        c.SetTimeStep(self.timeStep)
        if not self.useUIC:
            OperatingPoint(c).Execute()
        self.op_solves = c.M.n_solves
        self.timeStep = self.minStep
        while self.time < self.stopTime:
            if self.max_accepted is not None and self.accepted >= self.max_accepted:
                break
            nextTime = self.time + self.timeStep
            if nextTime > self.stopTime:
                nextTime = self.stopTime
                self.timeStep = nextTime - self.time
            c.Status = Status(self.time, self.timeStep, TRAN_MODE, 300.15, GMIN)
            if not self.doNRiter():
                if self.timeStep > self.minStep:
                    self.timeStep /= 2
                    self.rejected += 1
                    continue
                self.failed_at = self.time
                break
            lte = 0.0                                               # :239-250
            for d in c.devices:
                if d.time_dependent:
                    l = d.CalculateLTE(c.Status)
                    if l > lte:
                        lte = l
            if lte > self.trtol and self.timeStep > self.minStep:
                self.timeStep /= 2
                self.rejected += 1
                continue
            c.LoadState()
            c.Update()
            self.time = nextTime
            self.accepted += 1
            if self.time >= self.startTime:                         # StoreTimeResult, anlysis.go:61-85
                if not self.rows or (self.time != self.rows[-1][0] and _fmt_time(self.time) != _fmt_time(self.rows[-1][0])):
                    self.rows.append([self.time] + c.GetSolution())
            if self.time < self.stopTime and self.timeStep < self.maxStep:
                self.timeStep = min(self.timeStep * 2, self.maxStep) if lte < self.trtol / 100 else min(self.timeStep * 1.1, self.maxStep)
        self.tran_solves = c.M.n_solves - self.op_solves
        return np.array(self.rows)


class DCSweep:                                                      # dc.go
    def __init__(self, ckt, sources, starts, stops, incs):
        self.c = ckt
        self.src = [next(d for d in ckt.devices if d.name == s and d.typ == "V") for s in sources]
        self.sweeps = []
        for a, b, inc in zip(starts, stops, incs):                  # :36-42
            vals, v = [], a
            while v <= b:
                vals.append(v)
                v += inc
            self.sweeps.append(vals)
        self.rows, self.failed_at = [], None

    def doNRiter(self):                                             # :142-187 + CheckConvergence (anlysis.go:46-59, index 0 included)
        c, m = self.c, self.c.M
        st = Status(0.0, 0.0, OP_MODE, 300.15, 0.0)
        old = None
        for it in range(MAXITER):
            m.Clear()
            if it > 0:
                c.UpdateNonlinearVoltages(old)
            c.Stamp(st)
            try:
                m.Solve()
            except SingularMatrix:
                return False
            if it > 0:
                d = np.abs(m.solution - old)
                if not np.any((d > ABSTOL) & (d > RELTOL * np.abs(m.solution))):
                    return True
            old = m.solution.copy()
        return False

    def _point(self, head):
        c = self.c
        c.M.Clear()
        c.Stamp(Status(0.0, 0.0, OP_MODE, 300.15, GMIN))             # :113-125
        if not self.doNRiter():
            self.failed_at = head
            return False
        self.rows.append(list(head) + c.GetSolution())
        return True

    def run(self):
        if len(self.src) == 1:                                      # singleSweep :88-140
            for v in self.sweeps[0]:
                self.src[0].SetValue(v)
                if not self._point([v]):
                    break
        else:                                                       # nestedSweep :205-270
            done = False
            for v1 in self.sweeps[0]:
                self.src[0].SetValue(v1)
                for v2 in self.sweeps[1]:
                    self.src[1].SetValue(v2)
                    if not self._point([v1, v2]):
                        done = True
                        break
                if done:
                    break
        return np.array(self.rows)


# ------------------------------------------------------------------------------------------- AC analysis (ac.go)
def ac_frequencies(sweep, points, fstart, fstop):                   # ac.go:100-126
    if sweep == "DEC":
        a, b = math.log10(fstart), math.log10(fstop)
        return [10.0 ** (a + i * ((b - a) / (points - 1))) for i in range(points)]
    if sweep == "OCT":
        a, b = math.log2(fstart), math.log2(fstop)
        return [2.0 ** (a + i * ((b - a) / (points - 1))) for i in range(points)]
    return [fstart + i * ((fstop - fstart) / (points - 1)) for i in range(points)]


def ac_sweep(plan, sweep, points, fstart, fstop, overrides=None, refread=False):
    """ACAnalysis.Execute (ac.go:51-98) for a circuit without nonlinear devices, written from the device files' AC cases:
    per frequency a complex MNA system solved with numpy.linalg.solve.  What each device's Stamp does in Mode == ACAnalysis:
    resistor.go:43-54 (g), capacitor.go:48-66 (j*omega*C), inductor.go:43-57 (j*omega*L between the NODES, branch row left
    empty), vsource.go:155-177 / isource.go:149-165 (incidence, magnitude and phase), mutual.go:63-65 and magnetic.go:205-273
    (nothing).  Returns (rows, fail_freq): rows = [FREQ, mag, phase_deg per node voltage, then per V-source current];
    fail_freq = the frequency of the first singular system (the reference's "matrix solve error at f=..."), else None."""
    rows_in = [dict(kind=r.kind, name=r.name, nodes=list(r.nodes), branch=r.branch, p=list(r.p), ip=list(r.ip)) for r in plan.devices]
    for (dev, par), val in (overrides or {}).items():
        idx = dev if isinstance(dev, int) else [r["name"] for r in rows_in].index(dev)
        rows_in[idx]["p"][par] = float(val)
    n_nodes, n = plan.n_nodes, plan.n_nodes + plan.n_branches
    vsrc = [r for r in rows_in if r["kind"] == K_V]
    out, fail = [], None
    for f in ac_frequencies(sweep, points, fstart, fstop):
        omega = 2 * math.pi * f
        A = np.zeros((n + 1, n + 1), dtype=complex)
        rhs = np.zeros(n + 1, dtype=complex)

        def two_terminal(n1, n2, y):
            if n1:
                A[n1, n1] += y
            if n2:
                A[n2, n2] += y
            if n1 and n2:
                A[n1, n2] -= y
                A[n2, n1] -= y

        for r in rows_in:
            k, nd, p = r["kind"], r["nodes"], r["p"]
            if k == K_R:
                two_terminal(nd[0], nd[1], 1.0 / p[0])
            elif k == K_C:
                two_terminal(nd[0], nd[1], 1j * omega * p[0])
            elif k == K_L:
                two_terminal(nd[0], nd[1], 1j * omega * p[0])
            elif k == K_V:
                b = r["branch"]
                if nd[0]:
                    A[b, nd[0]] += 1
                    A[nd[0], b] += 1
                if nd[1]:
                    A[b, nd[1]] -= 1
                    A[nd[1], b] -= 1
                if (not r["ip"] or r["ip"][0] == 0) and len(p) >= 3:
                    rhs[b] += p[1] * complex(math.cos(p[2] * math.pi / 180.0), math.sin(p[2] * math.pi / 180.0))
            elif k == K_I:
                if (not r["ip"] or r["ip"][0] == 0) and len(p) >= 3:
                    cur = p[1] * complex(math.cos(p[2] * math.pi / 180.0), math.sin(p[2] * math.pi / 180.0))
                    if nd[0]:
                        rhs[nd[0]] += cur
                    if nd[1]:
                        rhs[nd[1]] -= cur
            elif k in (K_K, K_LCORE):
                pass
            else:
                raise ValueError("AC analysis of nonlinear circuits is outside this pin")
        M = A[1:, 1:]
        if np.linalg.matrix_rank(M) < n:                            # an empty branch row: exactly singular
            fail = f
            break
        x = np.concatenate([[0.0], np.linalg.solve(M, rhs[1:])])
        flat = np.zeros(3 * n + 4)
        flat[2:2 * n + 2:2] = x[1:].real
        flat[3:2 * n + 3:2] = x[1:].imag

        def get(i):
            return complex(flat[i], flat[i + n]) if refread else x[i]

        row = [f]
        for i in list(range(1, n_nodes + 1)) + [r["branch"] for r in vsrc]:
            z = get(i)
            row += [abs(z), math.degrees(math.atan2(z.imag, z.real))]
        out.append(row)
    return np.array(out), fail
