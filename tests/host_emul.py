"""Test infrastructure (never on the product path): the DEVICE source of a netlist's specialised kernels — models.cuh +
skeleton.cuh + the generated `struct Ckt` + the `__global__` entries, exactly the text NVRTC / nvcc compile for sm_100a
(`Batch.kernel_source`) — compiled for the HOST with g++ behind a shim of the CUDA built-ins and run one "thread" at a time
(a warp of one lane: every vote is the lane's own predicate; shared memory is a static array; threadIdx / blockIdx are
set per instance).  With `strict_fp = 1` and `-ffp-contract=off` this is the arithmetic of the strict GPU build, so whole
analyses (operating point incl. its Gmin / source-stepping fallbacks, transient, single and nested DC sweeps) can be held
against the oracle on a machine without a GPU: row counts, status, counters and values.

The shared time grid is emulated sequentially (the pilot instance runs to completion and publishes, then the readers run).
What it does NOT cover: anything that is a property of the parallel execution (warp votes across different lanes, lanes
refilling from the work counter, a reader overtaking the pilot, the cooperative mapping — which has its own host check) and
the fast build's device-only arithmetic (`__CUDA_ARCH__` branches of models.cuh: reciprocal seeds, table-driven exp) —
those are the GPU tests' job."""
import os
import re
import struct
import subprocess

import numpy as np

import parity_util as PU

T = PU.T

SHIM = r'''
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>
#include <algorithm>
using std::max;
using std::min;
#define __device__
#define __host__
#define __global__
#define __forceinline__ inline
#define __restrict__
#define __launch_bounds__(...)
#define __shared__
#define __constant__ static const
#define __grid_constant__
#define __builtin_assume(x) ((void)0)
struct double2 { double x, y; };
static inline double2 make_double2(double x, double y) { double2 r; r.x = x; r.y = y; return r; }
struct TsbDim3 { unsigned x, y, z; };
static TsbDim3 threadIdx = {0, 0, 0}, blockIdx = {0, 0, 0}, blockDim = {1, 1, 1}, gridDim = {1u << 30, 1, 1};
#define __any_sync(m, p) ((p) ? 1 : 0)
#define __all_sync(m, p) ((p) ? 1 : 0)
#define __ballot_sync(m, p) ((p) ? 1u : 0u)
#define __activemask() 1u
#define __syncthreads() ((void)0)
#define __syncwarp(...) ((void)0)
template <class P, class V> static inline void __stcs(P* p, V v) { *p = v; }
template <class P, class V> static inline void __stcg(P* p, V v) { *p = v; }
template <class P> static inline P __ldcs(const P* p) { return *p; }
template <class P> static inline P __ldcg(const P* p) { return *p; }
template <class P> static inline P __ldca(const P* p) { return *p; }
template <class P> static inline P __ldg(const P* p) { return *p; }
static inline long long __double_as_longlong(double d) { long long v; memcpy(&v, &d, 8); return v; }
static inline double __longlong_as_double(long long v) { double d; memcpy(&d, &v, 8); return d; }
static inline int __double2hiint(double d) { return (int)(__double_as_longlong(d) >> 32); }
static inline int __double2loint(double d) { return (int)(__double_as_longlong(d) & 0xffffffffLL); }
static inline double __hiloint2double(int hi, int lo) { return __longlong_as_double(((long long)hi << 32) | (unsigned)lo); }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
static inline double __ddiv_rn(double a, double b) { return a / b; }
static inline double __fma_rn(double a, double b, double c) { return fma(a, b, c); }
template <class A, class V> static inline A atomicAdd(A* p, V v) { A o = *p; *p = (A)(o + v); return o; }
double tsb_smem[1 << 17];
'''

MAIN = r'''
// ---- test driver: one kernel "thread" per instance, sequentially ---------------------------------------------------
static std::vector<char> slurp(const char* path) {
    FILE* f = fopen(path, "rb"); if (!f) { perror(path); exit(2); }
    fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
    std::vector<char> b(n); if (fread(b.data(), 1, n, f) != (size_t)n) exit(2); fclose(f); return b;
}
int main(int argc, char** argv) {
    std::vector<char> in = slurp(argv[1]);
    const long long* h = (const long long*)in.data();
    const long long n = h[0], nvar = h[1], npar = h[2], analysis = h[3], uic = h[4], max_iter = h[5], out_flags = h[6],
                    cap_rows = h[7], n_sweep = h[8], kernel = h[9], n_grid = h[10], refill_chain = h[11];
    const double* d = (const double*)(h + 16);
    TsbArgs a; memset(&a, 0, sizeof a);
    a.n_inst = n; a.n_run = n; a.analysis = (int)analysis; a.uic = (int)uic; a.max_iter = (int)max_iter;
    a.tstart = d[0]; a.tstop = d[1]; a.tstep = d[2]; a.maxstep = d[3]; a.minstep = d[4];
    a.abstol = d[5]; a.reltol = d[6]; a.trtol = d[7]; a.grid_dt = d[8]; a.n_grid = (int)n_grid;
    a.out_flags = (int)out_flags; a.cap_rows = cap_rows; a.skip_linear_resolve = TSB_SKIP_LINEAR_RESOLVE;
    const double* p = d + 9;
    a.U = p; for (long long k = 0; k < npar && k < TSB_UC_MAX; ++k) a.Uc[k] = p[k];
    p += npar;
    for (long long s = 0; s < nvar; ++s) { a.pv[s] = p; p += n; }
    a.sweep = p; p += n_sweep; a.sweep2 = p; p += n_sweep; a.n_sweep = (int)n_sweep;
    constexpr int NC = Ckt::NCOL_MAX + Ckt::DC_NESTED;          // the row stride of the kernels' result store
    std::vector<double> wave((size_t)(cap_rows + 1) * NC * n, 0.0), stats((size_t)4 * NC * n, 0.0), scratch((size_t)(Ckt::N + 2) * n, 0.0);
    std::vector<long long> rows(n, 0), counters((size_t)8 * n, 0);
    std::vector<int> status(n, -1);
    unsigned long long work = 0;
    a.wave = wave.data(); a.stats = stats.data(); a.scratch = scratch.data(); a.rows = rows.data(); a.counters = counters.data();
    a.status = status.data(); a.work_counter = &work; a.first_free = n;
    blockDim.x = TSB_BLOCK;
#if TSB_TGRID
    // shared time grid (runtime.cpp: launch_pilot): the pilot — instance 0, no outputs — publishes its attempts, then the readers run
    std::vector<double> tgrid((size_t)(1 << 16) * TsbTgLayout<Ckt::NSRC>::ND, 0.0);
    unsigned long long tgrid_pub = 0;
    a.tgrid = tgrid.data(); a.tgrid_pub = &tgrid_pub; a.tgrid_cap = 1 << 16; a.tgrid_role = 0;
    if (kernel == 0 && analysis == 1) {
        TsbArgs ap = a;
        ap.tgrid_role = 1; ap.n_run = 1; ap.out_flags = 0; ap.first_free = 1;
        blockIdx.x = 0; threadIdx.x = 0;
        tsb_optran(ap);
        fprintf(stderr, "tgrid entries published: %llu\n", tgrid_pub);
    }
#endif
    if (refill_chain) a.first_free = 1;          // lane refill: ONE lane starts on instance 0 and takes every further instance from the work counter
    for (long long i = 0; i < (refill_chain ? 1 : n); ++i) {
        blockIdx.x = (unsigned)(i / TSB_BLOCK); threadIdx.x = (unsigned)(i % TSB_BLOCK);
        if (kernel == 0) tsb_optran(a); else tsb_dc(a);
    }
    FILE* f = fopen(argv[2], "wb");
    long long dims[4] = {n, NC, cap_rows + 1, 0};
    fwrite(dims, 8, 4, f);
    fwrite(wave.data(), 8, wave.size(), f); fwrite(stats.data(), 8, stats.size(), f); fwrite(rows.data(), 8, n, f);
    fwrite(counters.data(), 8, counters.size(), f); fwrite(status.data(), 4, n, f);
    fclose(f);
    return 0;
}
'''


class HostBatch:
    """Results of a host run behind the accessors parity_util.compare_waves uses on a GPU batch."""

    def __init__(self, n, ncol, wave, stats, rows, counters, status):
        self.n_inst, self.ncol = n, ncol
        self._wave, self._stats, self._rows, self._counters, self._status = wave, stats, rows, counters, status

    def rows(self):
        return self._rows

    def status(self):
        return self._status

    def counters(self):
        return self._counters

    def wave_all(self):
        return self._wave[:, : self.ncol, :]

    def waveform(self, i):
        return self._wave[: int(self._rows[i]), : self.ncol, i]

    def stats_all(self):
        return self._stats[:, : self.ncol, :]


_BUILT = {}

# The five PTX one-liners of the shared time grid (acquire / release / relaxed accesses of the published count, a fence, a
# prefetch) have no host spelling; in the sequential emulation — the pilot runs to completion before the first reader — plain
# accesses are what they mean.
_ASM_HOST = [
    (r'asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");', "v = *p;"),
    (r'asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");', "*p = v;"),
    (r'asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");', "v = *p;"),
    (r'asm volatile("fence.acq_rel.gpu;" ::: "memory");', ""),
    (r'asm volatile("prefetch.global.L1 [%0];" ::"l"(p));', "(void)p;"),
]


def _flat_parameters(ckt):
    """The plan's flat parameter table (runtime.cpp: b->uniform = plan nominal) and the flat index of (device, param)."""
    nominal, index = [], {}
    for d in ckt.devices():
        for j, v in enumerate(d["p"]):
            index[(d["name"], j)] = len(nominal)
            nominal.append(float(v))
    return nominal, index


def build(text, overrides, tmpdir, strict=True, dc_src=-1, dc_src2=-1, opts_kw=None, grid=False, main=None):
    """g++-compile the kernel source of this netlist / set of per-instance parameters [/ swept source(s)]; returns (exe, info).
    `main`: a driver of the caller's own in place of MAIN."""
    ckt = T.Circuit.from_netlist(text)
    b = ckt.batch(2)
    if dc_src != -1:
        b.kernel_variant(dc_src, dc_src2)               # the DC kernels are specialised on the swept parameter(s)
    elif grid:
        b.kernel_variant(grid=True)                     # TSB_OUT_GRID is a specialisation too
    for (dev, par), vals in overrides.items():
        b.set_param(dev, par, np.resize(np.asarray(vals, dtype=np.float64), 2))      # (which parameters vary is what specialises the source)
    opts = T.default_opts(**{**dict(strict_fp=1 if strict else 0, min_blocks=1, block_size=32, share_time_grid=0, coop_parts=0), **(opts_kw or {})})
    src = b.kernel_source(opts)
    key = (src, strict, tmpdir, main)
    info = dict(ckt=ckt, opts=opts,
                slots=[(int(s), int(k)) for k, s in re.findall(r"P\[(\d+)\] = __ldcs\(a\.pv\[(\d+)\]", src)],
                ncol_max=int(re.search(r"NCOL_MAX = (\d+)", src).group(1)), n=int(re.search(r"static constexpr int N = (\d+)", src).group(1)))
    if key in _BUILT:
        return _BUILT[key], info
    tag = f"h{len(_BUILT)}"
    cpp = os.path.join(tmpdir, tag + ".cpp")
    exe = os.path.join(tmpdir, tag)
    with open(cpp, "w") as f:
        host_src = src.replace("extern __shared__ double tsb_smem[];", "")
        for ptx, c in _ASM_HOST:
            host_src = host_src.replace(ptx, c)
        f.write(SHIM + host_src + (MAIN if main is None else main))
    flags = ["-O1", "-std=c++17", "-ffp-contract=off", "-w"] + ([] if strict else ["-DTSB_FAST_DIV"])
    r = subprocess.run(["g++"] + flags + ["-o", exe, cpp], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    _BUILT[key] = exe
    return exe, info


def _sweep_points(start, stop, inc):
    """dc.go:36-42 as tsb_run_dc restates it: for v := start; v <= stop; v += inc."""
    out, v = [], float(start)
    while v <= stop:
        out.append(v)
        v += inc
    return out


def run(text, n, overrides, tmpdir, analysis=None, tran=None, dc=None, dc2=None, strict=True, cap_rows=None, opts_kw=None, grid_dt=None,
        refill_chain=False):
    """Whole analysis of `n` instances on the host-compiled device source.  dc = (source, start, stop, inc) overrides the
    deck's .dc card; dc2 = ((outer ...), (inner ...)) runs the nested sweep.  Returns (circuit, HostBatch, column names)."""
    probe = T.Circuit.from_netlist(text)
    pcard = probe.analysis_card()
    pkind = pcard["analysis"] if analysis is None else analysis
    dc_src = dc_src2 = -1
    if pkind == T.AN_DC:
        if dc2 is not None:
            dc_src, dc_src2 = dc2[0][0], dc2[1][0]
        elif dc is not None:
            dc_src = dc[0]
        else:
            dc_src = probe.devices()[pcard["dc_src_dev"]]["name"]
            dc = (dc_src, pcard["dc_start"], pcard["dc_stop"], pcard["dc_inc"])
    exe, info = build(text, overrides, tmpdir, strict, dc_src, dc_src2, opts_kw, grid=grid_dt is not None)
    ckt, opts = info["ckt"], info["opts"]
    card = ckt.analysis_card()
    if tran:
        card.update(tran)
    kind = card["analysis"] if analysis is None else analysis
    nominal, index = _flat_parameters(ckt)
    slot_of = dict(info["slots"])                       # kernel slot -> flat parameter index
    flat_to_key = {v: k for k, v in index.items()}
    names = {d["name"]: d for d in ckt.devices()}
    pv = []
    for s in range(len(slot_of)):
        dev, par = flat_to_key[slot_of[s]]
        vals = None
        for (dn, p), v in overrides.items():
            if (dn if isinstance(dn, str) else ckt.devices()[dn]["name"]) == dev and p == par:
                vals = v
        assert vals is not None, (dev, par)
        pv.append(np.ascontiguousarray(vals, dtype=np.float64)[:n])
    tstart = tstop = tstep = tmax = minstep = 0.0
    sweep = np.zeros(0)
    sweep2 = None
    kernel = 0
    n_grid, gdt, out_flags = 0, 0.0, T.OUT_WAVE | T.OUT_STATS
    if kind == T.AN_OP:
        ncol, rows_cap, an = len(ckt.columns(T.AN_OP)), 1, 0
    elif kind == T.AN_TRAN:
        tstart, tstop, tstep, tmax = card["tstart"], card["tstop"], card["tstep"], card["tmax"]
        if tstep > tstop / 300:                        # NewTransient (tran.go:29-55), as tsb_run_tran does it
            tstep = tstop / 300
        minstep = tstep / 50.0
        if tmax == 0:
            tmax = tstep
        ncol, an = len(ckt.columns(T.AN_TRAN)), 1
        rows_cap = cap_rows or 65536
        if grid_dt is not None:                        # tsb_run_tran: TSB_OUT_GRID (statistics carry the previous stored row)
            gdt = grid_dt if grid_dt > 0 else tstep
            n_grid = max(1, int(np.floor((tstop - tstart) / gdt * (1.0 + 1e-12) + 1e-9)))
            rows_cap, out_flags = n_grid, T.OUT_GRID | T.OUT_STATS
    else:
        kernel, an = 1, 3
        if dc2 is not None:                             # tsb_run_dc2: the nested loops flattened into one list of points
            s1, s2 = _sweep_points(*dc2[0][1:]), _sweep_points(*dc2[1][1:])
            sweep = np.array([v1 for v1 in s1 for _ in s2], dtype=np.float64)
            sweep2 = np.array([v2 for _ in s1 for v2 in s2], dtype=np.float64)
            ncol = len(ckt.columns(T.AN_DC)) + 1
        else:
            sweep = np.array(_sweep_points(*dc[1:]), dtype=np.float64)
            ncol = len(ckt.columns(T.AN_DC))
        rows_cap = len(sweep)
    hdr = np.zeros(16, dtype=np.int64)
    hdr[:12] = [n, len(pv), len(nominal), an, int(card.get("uic", False)), opts.max_iter, out_flags, rows_cap, len(sweep), kernel, n_grid,
                int(bool(refill_chain))]
    dbl = np.array([tstart, tstop, tstep, tmax, minstep, opts.abstol, opts.reltol, opts.trtol, gdt], dtype=np.float64)
    blob = hdr.tobytes() + dbl.tobytes() + np.asarray(nominal, dtype=np.float64).tobytes() + b"".join(v.tobytes() for v in pv) \
        + sweep.tobytes() + (sweep if sweep2 is None else sweep2).tobytes()
    fin, fout = os.path.join(tmpdir, "in.bin"), os.path.join(tmpdir, "out.bin")
    with open(fin, "wb") as f:
        f.write(blob)
    r = subprocess.run([exe, fin, fout], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stderr[-2000:])
    raw = open(fout, "rb").read()
    nn, nc, cap1, _ = struct.unpack("4q", raw[:32])
    off = 32
    wave = np.frombuffer(raw, dtype=np.float64, count=cap1 * nc * nn, offset=off).reshape(cap1, nc, nn); off += wave.nbytes
    stats = np.frombuffer(raw, dtype=np.float64, count=4 * nc * nn, offset=off).reshape(4, nc, nn); off += stats.nbytes
    rows = np.frombuffer(raw, dtype=np.int64, count=nn, offset=off); off += rows.nbytes
    counters = np.frombuffer(raw, dtype=np.int64, count=8 * nn, offset=off).reshape(8, nn); off += counters.nbytes
    status = np.frombuffer(raw, dtype=np.int32, count=nn, offset=off)
    hb = HostBatch(nn, ncol, wave, stats, rows, counters, status)
    m = re.search(r"tgrid entries published: (\d+)", r.stderr)
    hb.tgrid_entries = int(m.group(1)) if m else None     # shared time grid: what the pilot published (None: not a TSB_TGRID kernel)
    if n_grid:
        t = tstart + (np.arange(n_grid) + 1.0) * gdt    # Batch.grid_times: two roundings, the last point clamped to tstop
        hb.grid_times = np.where(t < tstop, t, tstop)
    return ckt, hb, ckt.columns(kind)
