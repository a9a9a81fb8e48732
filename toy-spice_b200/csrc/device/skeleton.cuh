// skeleton.cuh — per-thread analysis drivers of the batched engine (hand-written, generic).
//
// One GPU thread owns one circuit instance for the whole analysis: parameters, device state,
// solution vectors and the MNA matrix live in registers; nothing is exchanged between threads.
// The drivers are templated on a generated struct `Ckt` (codegen.cpp) that provides the
// netlist-specific straight-line code (stamps, LU in the frozen pivot order, state updates).
//
// Drivers in this file (each entered by WHOLE warps: lanes without an instance only take part in the votes):
//   tsb_run_optran_instance  operating point(s) as one loop around one Newton-iteration body (a small state machine:
//                            main loop, Gmin stepping, source stepping), then hands the transient to
//   tsb_tran_linear          circuits without nonlinear devices: one solve per step, LTE test before the solve,
//                            branch-free step body;
//   tsb_tran_nonlinear       circuits with nonlinear devices: time loop and Newton loop as two nested loops whose
//                            trip counts are decided by warp votes (per-lane convergence predicate; converged lanes
//                            wait for the slowest live lane, post-Newton work runs once per step for the warp);
//   tsb_run_dc_instance      DC sweep: warp-uniform sweep loop, vote-controlled Newton loop.
// With lane refill (TSB_LANE_REFILL) the state machine also runs the transient, free-running per lane.
// Compile-time A/B switches (TSB_X_*) keep every measured alternative buildable; profiles/r01_notes.md has the numbers.
//
// Reference behaviour reproduced (statement by statement; see SURVEY.md §3.6 for the quirks):
//   OperatingPoint.Execute / doNRiter / calculateInitialEstimate / performSourceStepping   op.go:25-233
//   Transient.Setup / Execute / doNRiter / calculateTruncError                            tran.go:57-250
//   DCSweep.singleSweep / doNRiter, BaseAnalysis.CheckConvergence / StoreTimeResult       dc.go:88-187, anlysis.go:46-85
#ifndef TSB_SKELETON_CUH
#define TSB_SKELETON_CUH

#define TSB_MAX_VARYING 128
#define TSB_UC_MAX 32

struct TsbArgs {
    long long n_inst;
    const double* pv[TSB_MAX_VARYING];   // per varying parameter: [n_inst] doubles (SoA, instance fastest)
    const double* U;           // [n_params]       uniform parameter values (+ PWL tables)
    int analysis;              // 0 OP, 1 TRAN, 3 DC
    int uic;
    double tstart, tstop, tstep, maxstep, minstep;   // after NewTransient's clamping (tran.go:29-37)
    int max_iter;
    double abstol, reltol, trtol;
    int out_flags;             // 1 wave, 2 stats
    long long cap_rows;
    double* wave;              // [cap_rows][ncol][n_inst]
    double* stats;             // [4][ncol][n_inst]
    long long* rows;           // [n_inst]
    int* status;               // [n_inst]
    long long* counters;       // [6][n_inst]
    double* scratch;           // [N+1][n_inst]  "currentSolution" of the OP fallbacks
    const double* sweep;       // [n_sweep] DC sweep values
    int n_sweep;
    int skip_linear_resolve;   // (compile-time TSB_SKIP_LINEAR_RESOLVE decides; kept for layout stability)
    unsigned long long* work_counter;   // lane refill: next unprocessed instance = first_free + atomicAdd(counter, 1)
    long long first_free;
    double grid_dt;            // TSB_OUT_GRID: grid row k is at tstart + (k+1)*grid_dt (the last one clamped to tstop)
    int n_grid;
    long long n_run;           // instances [0, n_run) are processed (n_inst stays the array stride); < n_inst only
                               // while the library times launch-bounds candidates on a sub-batch
    const long long* order;    // optional processing order (tsb_batch_set_order): slot s works on instance order[s]
    const double* sweep2;      // nested DC sweep (dc.go:205-270): value of the inner source at point k (sweep[] holds the outer one)
    // Shared time grid (TSB_TGRID kernels, see tsb_tran_linear): attempt k of the PILOT instance as
    // [time, dt | result-store key, source value 0 | further source values...]
    double* tgrid;                       // [tgrid_cap][TsbTgLayout::ND] doubles, or NULL (feature off for this launch)
    unsigned long long* tgrid_pub;       // number of entries published so far (release / acquire)
    int tgrid_cap;
    int tgrid_role;                      // 0: reader, 1: the pilot launch (one instance, publishes)
    // The first TSB_UC_MAX uniform parameter values BY VALUE: kernel parameters live in the constant bank, so a value
    // that is the same for every instance can be an instruction operand (or be re-read) instead of occupying a register
    // pair of every thread for the whole run.  U (global memory) keeps the full table (PWL points, parameters beyond).
    double Uc[TSB_UC_MAX];
    // Cooperative mapping (device/coop.cuh, kernels generated with TSB_COOP): the operating point runs thread-per-circuit in
    // tsb_optran, which then hands the device state and the solution over — [n_state + N + 1][n_inst] doubles — instead of
    // running the transient itself; tsb_coop_tran picks them up.  NULL: tsb_optran runs the whole analysis.
    double* coop_state;
    // TSB_OUT_MEAS (kernels generated with TSB_MEAS): the run-time half of the measurement table — kind, column and trigger
    // column are compile-time (tsb_meas_spec), so a new level or window reuses the kernel.  Appended: every field above
    // keeps its offset.
    double meas_level[16], meas_from[16], meas_to[16];
    int meas_count[16], meas_edge[16];
    double* meas_out;          // [2][n_meas][n_inst]: value, abscissa
#if TSB_FOUR
    // TSB_OUT_FOUR (kernels generated with TSB_FOUR): the run-time half of the Fourier table — column and number of
    // harmonics are compile-time (tsb_four_spec).  Appended after meas_out: every field above keeps its offset.  The host
    // always passes them; kernels without a table declare the struct without them and read its prefix.
    double four_s[8], four_dt[8];   // window start s and grid spacing T / G of entry e
    int four_g[8];                  // G
    int four_tw_off[8];             // entry e's twiddles: four_tw[off .. off + G) cosines, [off + G .. off + 2G) sines
    const double* four_tw;
    double* four_out;               // [sum (1 + 2H)][n_inst]: the sums while the run accumulates, the coefficients after it
#endif
};

// Slot -> instance.  With an order, lanes of a warp can be given instances that behave alike (similar Newton
// iteration counts) whatever their position in the caller's arrays; parameters and results stay where the caller put them.
__device__ __forceinline__ long long tsb_slot_instance(const TsbArgs& a, long long slot, bool valid) {
    return (TSB_ORDER && valid && a.order) ? a.order[slot] : slot;      // TSB_ORDER: kernels specialised for ordered batches
}

#define TSB_ST_OK 0
#define TSB_ST_OP_FAILED 1
#define TSB_ST_TRAN_FAILED 2
#define TSB_ST_DC_FAILED 3
#define TSB_ST_OVERFLOW 4
#define TSB_AN_OP 0
#define TSB_AN_TRAN 1
#define TSB_AN_DC 3
#define TSB_OUT_WAVE 1
#define TSB_OUT_STATS 2
#define TSB_OUT_GRID 4
#define TSB_OUT_AC_REFREAD 8
#define TSB_OUT_MEAS 16

#ifndef TSB_COOP
#define TSB_COOP 0
#endif
#ifndef TSB_X_STATS_PRED
#define TSB_X_STATS_PRED 1
#endif
#ifndef TSB_X_CONVSEL
#define TSB_X_CONVSEL 1
#endif
#ifndef TSB_X_LTE_OPAQUE
#define TSB_X_LTE_OPAQUE 1          // truncation-error predicates: keep the two compares of an inductor's terms apart (TSB_OPAQUE, models.cuh)
#endif
#ifndef TSB_X_UNROLL2
#define TSB_X_UNROLL2 0             // linear transient loop unrolled twice (loop-carried state without register moves): see r02_notes.md
#endif
#ifndef TSB_X_TGLOOK
#define TSB_X_TGLOOK 1              // shared time grid: one compare on the hot path of the look-up bookkeeping (tsb_tran_linear)
#endif
#ifndef TSB_X_CONV2TOL
#define TSB_X_CONV2TOL 1            // convergence test against two tolerances instead of the tolerance of a selected maximum
#endif
#ifndef TSB_X_NRSTATE
#define TSB_X_NRSTATE 1             // nonlinear transient: one integer state per lane in the Newton loop instead of three bools
#endif
#ifndef TSB_X_LTEFLAGS
#define TSB_X_LTEFLAGS 1            // linear loop: truncation-error DECISIONS from predicates instead of selecting the maximum
#endif
extern __shared__ double tsb_smem[];

// op.go:67-77 / tran.go:192-207: |new-old| <= reltol*max(|new|,|old|) + abstol for i = 1..n.
// Written as "no element exceeds" so that NaN passes, as in the reference (SURVEY Q4).
template <int N>
__device__ __forceinline__ bool tsb_converged(const double* x, const double* xo, double reltol, double abstol) {
    bool ok = true;
#pragma unroll
    for (int i = 1; i <= N; ++i) {
        const double diff = fabs(x[i] - xo[i]);
        const double ax = fabs(x[i]), ao = fabs(xo[i]);
#if TSB_X_CONV2TOL
        // diff > reltol * max(|new|, |old|) + abstol  <=>  diff exceeds BOTH reltol * |new| + abstol and reltol * |old| + abstol:
        // a rounded product by reltol > 0 and a rounded sum are monotone in the operand, so the larger of the two tolerances IS
        // the tolerance of the larger magnitude, bit for bit — two multiply-adds with |.| operand modifiers and two compares
        // instead of materialising the magnitudes and selecting their maximum (8 -> 5 instructions per unknown and trip).
        // NaN: diff is NaN whenever an operand is, both compares are false, the test passes as in the reference (SURVEY Q4).
        if ((diff > reltol * ax + abstol) & (diff > reltol * ao + abstol)) ok = false;
#else
        // math.Max(|new|, |old|) as a plain select: the two differ only when an operand is NaN — and then diff is NaN too, so
        // `diff > tol` is false whatever tol is (the library fmax costs ~10 instructions per element for its NaN handling)
        const double tol = reltol * (TSB_X_CONVSEL ? (ax > ao ? ax : ao) : fmax(ax, ao)) + abstol;
        if (diff > tol) ok = false;
#endif
    }
    return ok;
}
// anlysis.go:46-59 (DC sweep): |d| > abstol && |d| > reltol*|new| -> not converged.
template <int N>
__device__ __forceinline__ bool tsb_converged_dc(const double* x, const double* xo, double reltol, double abstol) {
    bool ok = true;
#pragma unroll
    for (int i = 1; i <= N; ++i) {
        double diff = fabs(x[i] - xo[i]);
        if (diff > abstol && diff > reltol * fabs(x[i])) ok = false;
    }
    return ok;
}

// Measurements (TSB_OUT_MEAS, the SPICE .meas family; definitions in include/tspice_b200.h).  Kernels generated for a
// measurement table define TSB_MEAS (its length) and TSB_MEAS_SPEC ({kind, column, trigger column} per entry): the sink
// walks the table at compile time, so every column index into the row — a register array — is a literal.  Every
// operation is individually rounded in both builds, so a result depends on the stored rows only.
#ifndef TSB_MEAS
#define TSB_MEAS 0
#endif
#define TSB_MEAS_WHEN 0
#define TSB_MEAS_AT 1
#define TSB_MEAS_MAX 2
#define TSB_MEAS_MIN 3
#define TSB_MEAS_AVG 4
#define TSB_MEAS_INTEG 5
#define TSB_MEAS_RMS 6
#define TSB_EDGE_RISE 1
#define TSB_EDGE_FALL 2
#if TSB_MEAS
struct TsbMeasSpec { int kind, col, tcol; };
__host__ __device__ constexpr TsbMeasSpec tsb_meas_spec(int i) {
    constexpr TsbMeasSpec t[TSB_MEAS] = {TSB_MEAS_SPEC};
    return t[i];
}
// The value at abscissa L of the segment (x0, y0) - (x1, y1) with x0 < L <= x1, as AT defines it.
__device__ __forceinline__ double tsb_meas_interp(double x0, double y0, double x1, double y1, double L) {
    if (L == x1) return y1;
    return __dadd_rn(y0, __dmul_rn(__ddiv_rn(__dsub_rn(L, x0), __dsub_rn(x1, x0)), __dsub_rn(y1, y0)));
}
#endif
#if TSB_FOUR
// Fourier analysis (TSB_OUT_FOUR, the SPICE .four card; definitions in include/tspice_b200.h).  Kernels generated for a
// Fourier table define TSB_FOUR (its length) and TSB_FOUR_SPEC ({column, harmonics} per entry).  Every line of it sits in
// an `#if TSB_FOUR` block, which the code generator leaves out of kernels without a table: their source stays the same.
#define TSB_OUT_FOUR 32
struct TsbFourSpec { int col, harm; };
__host__ __device__ constexpr TsbFourSpec tsb_four_spec(int i) {
    constexpr TsbFourSpec t[TSB_FOUR] = {TSB_FOUR_SPEC};
    return t[i];
}
// first output row of entry e: the entries before it take 1 + 2H rows each
__host__ __device__ constexpr int tsb_four_row(int e) { return e == 0 ? 0 : tsb_four_row(e - 1) + 1 + 2 * tsb_four_spec(e - 1).harm; }
#if !TSB_MEAS
// a sample y_k is the series' value at tau_k as AT defines it: the interpolation of the measurement code above
__device__ __forceinline__ double tsb_meas_interp(double x0, double y0, double x1, double y1, double L) {
    if (L == x1) return y1;
    return __dadd_rn(y0, __dmul_rn(__ddiv_rn(__dsub_rn(L, x0), __dsub_rn(x1, x0)), __dsub_rn(y1, y0)));
}
#endif
#endif

// Result sink of one instance: waveform rows to HBM (instance-fastest layout, so a warp whose
// lanes are at the same row index writes 256 contiguous bytes per column) and running
// min / max / sum / last per column in shared memory.
// Shared-memory layout: per column two double2 arrays of TSB_BLOCK entries, {min, max} and {sum, last}; a thread
// owns entry threadIdx.x of each, so a warp reads or writes 512 contiguous bytes per 128-bit access (conflict-free)
// and one stored row costs 4 shared-memory instructions per column instead of 7 scalar ones.  Column 0 (TIME /
// the sweep value) is monotone by construction: its extremes are the first and the last row — only {sum, last} updated.
template <int NCOL>
struct TsbSink {
    const TsbArgs& a;
    long long inst;
    long long n_rows;
    bool overflow;
    double2* sm;                // this thread's first pair; pairs are TSB_BLOCK double2 apart
    int grid_k;                 // TSB_OUT_GRID: next grid row to write
    __device__ __forceinline__ TsbSink(const TsbArgs& a_, long long inst_) : a(a_), inst(inst_), n_rows(0), overflow(false), grid_k(0) {
        sm = reinterpret_cast<double2*>(tsb_smem) + threadIdx.x;   // launched with blockDim.x == TSB_BLOCK: every offset below is an immediate
    }
    __device__ __forceinline__ void begin(long long inst_) {      // (re)start for one instance
        inst = inst_; n_rows = 0; overflow = false; grid_k = 0;
        if (a.out_flags & TSB_OUT_STATS) {
#pragma unroll
            for (int j = 0; j < NCOL; ++j) {
                sm[(2 * j) * TSB_BLOCK] = make_double2(__longlong_as_double(0x7ff0000000000000LL),     // +inf
                                                       __longlong_as_double(0xfff0000000000000LL));    // -inf
                sm[(2 * j + 1) * TSB_BLOCK] = make_double2(0.0, 0.0);
            }
        }
#if TSB_MEAS
        if (a.out_flags & TSB_OUT_MEAS) meas_begin();
#endif
#if TSB_FOUR
        if (a.out_flags & TSB_OUT_FOUR) four_begin();
#endif
    }
#if TSB_FOUR
    // Entry e keeps one double2 per thread after the statistics and measurement pairs: {tau_k, k} of the next grid point
    // k it waits for (tau = +inf once all G are taken).  A stored row costs one shared-memory load and one compare per
    // entry; the sums live in place in four_out (instance-fastest rows, so a warp that takes a grid point together
    // touches contiguous lines) and are read, updated and written at each of the G grid points.  Shared memory or
    // registers for the 2H + 1 sums would cost residency or spills in the step loop (measured: DESIGN.md §5.2a).
    __device__ __forceinline__ double2* four_slot(int e) const { return sm + (2 * NCOL + 2 * TSB_MEAS + e) * TSB_BLOCK; }
    template <int e = 0> __device__ __forceinline__ void four_begin() {
        if constexpr (e < TSB_FOUR) {
            if constexpr (tsb_four_spec(e).col < NCOL) four_slot(e)[0] = make_double2(__dadd_rn(a.four_s[e], __dmul_rn(0.0, a.four_dt[e])), 0.0);
            four_begin<e + 1>();
        }
    }
    // One stored row, before the statistics update (the previous row is in the `last` slots): every grid point in
    // (previous row, this row] is sampled and added into the sums.
    template <int e = 0> __device__ __forceinline__ void emit_four(const double* row) {
        if constexpr (e < TSB_FOUR) {
            constexpr TsbFourSpec sp = tsb_four_spec(e);
            if constexpr (sp.col < NCOL) {
                double2* slot = four_slot(e);
                const double x1 = row[0];
                if (x1 >= slot[0].x) four_take<e>(x1, row[sp.col], slot);
            }
            emit_four<e + 1>(row);
        }
    }
    template <int e> __device__ __forceinline__ void four_take(double x1, double y1, double2* slot) {
        constexpr TsbFourSpec sp = tsb_four_spec(e);
        const int G = a.four_g[e];
        const double s = a.four_s[e], dt = a.four_dt[e];
        const double* c = a.four_tw + a.four_tw_off[e];
        const double* sn = c + G;
        const double x0 = sm[1 * TSB_BLOCK].y, y0 = sm[(2 * sp.col + 1) * TSB_BLOCK].y;
        double* o = a.four_out + (long long)tsb_four_row(e) * a.n_inst + inst;
        int k = (int)slot[0].y;
        double tk = slot[0].x;
        while (x1 >= tk) {
            // no row before this one: tau_0 < x_0 is outside the series, a NaN sample turns every sum NaN
            const double y = n_rows > 0 ? tsb_meas_interp(x0, y0, x1, y1, tk) : (x1 == tk ? y1 : __longlong_as_double(0x7ff8000000000000LL));
            const bool first = k == 0;                 // the sums start at 0.0: nothing to read yet
            o[0] = __dadd_rn(first ? 0.0 : o[0], y);
            int j = 0;
#pragma unroll
            for (int h = 1; h <= sp.harm; ++h) {
                j += k; if (j >= G) j -= G;              // (h k) mod G
                double* oh = o + (long long)(2 * h - 1) * a.n_inst;
                oh[0] = __dadd_rn(first ? 0.0 : oh[0], __dmul_rn(y, __ldg(c + j)));
                oh[a.n_inst] = __dadd_rn(first ? 0.0 : oh[a.n_inst], __dmul_rn(y, __ldg(sn + j)));
            }
            ++k;
            tk = k < G ? __dadd_rn(s, __dmul_rn((double)k, dt)) : TSB_INF;
        }
        slot[0] = make_double2(tk, (double)k);
    }
    // coefficients from the sums; NaN for every row when a grid point was not reached (tau_{G-1} > x_last, no rows)
    template <int e = 0> __device__ __forceinline__ void four_finish() {
        if constexpr (e < TSB_FOUR) {
            constexpr TsbFourSpec sp = tsb_four_spec(e);
            if constexpr (sp.col < NCOL) {
                const int G = a.four_g[e];
                const bool all = (int)four_slot(e)[0].y == G;
                const double g = (double)G;
                double* o = a.four_out + (long long)tsb_four_row(e) * a.n_inst + inst;
                const double nan = __longlong_as_double(0x7ff8000000000000LL);
                o[0] = all ? __ddiv_rn(o[0], g) : nan;
#pragma unroll
                for (int r = 1; r <= 2 * sp.harm; ++r) {
                    double* orow = o + (long long)r * a.n_inst;
                    orow[0] = all ? __ddiv_rn(__dmul_rn(2.0, orow[0]), g) : nan;
                }
            }
            four_finish<e + 1>();
        }
    }
#endif
#if TSB_MEAS
    // Measurement m keeps two double2 per thread after the statistics pairs (same thread-interleaved layout):
    //   WHEN            {value, abscissa} of the crossing taken, {crossings counted, -}
    //   AT              {value, -}, {1 once the row at or past the level was seen, -}
    //   MAX / MIN       {extreme, its abscissa} (NaN: no row in the window yet)
    //   AVG/INTEG/RMS   {trapezoid sum of y (of y^2 for RMS) over the window, -}
    // Each step walks the table by template recursion (entry m, then m + 1): m is a literal in every instance.  Entries
    // whose columns this kernel's rows do not have belong to another analysis (the run checks the table against its own
    // columns) and compile to nothing here.
    __device__ __forceinline__ double2* meas_slot(int m) const { return sm + (2 * NCOL + 2 * m) * TSB_BLOCK; }
    template <int m = 0> __device__ __forceinline__ void meas_begin() {
        if constexpr (m < TSB_MEAS) {
            constexpr TsbMeasSpec s = tsb_meas_spec(m);
            if constexpr (s.col < NCOL && s.tcol < NCOL) {
                const double nan = __longlong_as_double(0x7ff8000000000000LL);
                double2* st = meas_slot(m);
                st[0] = s.kind >= TSB_MEAS_AVG ? make_double2(0.0, 0.0) : make_double2(nan, nan);
                st[TSB_BLOCK] = make_double2(0.0, 0.0);
            }
            meas_begin<m + 1>();
        }
    }
    // One stored row; runs before the statistics update, so the previous row (n_rows > 0) is still in the `last` slots.
    __device__ __forceinline__ void emit_meas(const double* row) { emit_meas_entry<0>(row, n_rows > 0, sm[1 * TSB_BLOCK].y, row[0]); }
    template <int m> __device__ __forceinline__ void emit_meas_entry(const double* row, bool prev, double x0, double x1) {
        if constexpr (m < TSB_MEAS) {
            constexpr TsbMeasSpec s = tsb_meas_spec(m);
            if constexpr (s.col < NCOL && s.tcol < NCOL) {
                double2* st = meas_slot(m);
                const double y1 = row[s.col];
                if constexpr (s.kind == TSB_MEAS_WHEN) {
                    if (prev) {
                        const double L = a.meas_level[m], t0 = sm[(2 * s.tcol + 1) * TSB_BLOCK].y, t1 = row[s.tcol];
                        const int edge = a.meas_edge[m];
                        const bool rise = (t0 < L) & (L <= t1), fall = (t0 > L) & (L >= t1);      // NaN: neither
                        if ((rise & (edge != TSB_EDGE_FALL)) | (fall & (edge != TSB_EDGE_RISE))) {
                            const double f = __ddiv_rn(__dsub_rn(L, t0), __dsub_rn(t1, t0));
                            const double xs = __dadd_rn(x0, __dmul_rn(f, __dsub_rn(x1, x0)));
                            const int count = a.meas_count[m];
                            const double seen = st[TSB_BLOCK].x;
                            if (xs >= a.meas_from[m] && xs <= a.meas_to[m] && (count < 0 || seen < (double)count)) {
                                st[TSB_BLOCK].x = seen + 1.0;
                                if (count < 0 || seen + 1.0 == (double)count) {
                                    const double y0 = sm[(2 * s.col + 1) * TSB_BLOCK].y;
                                    st[0] = make_double2(__dadd_rn(y0, __dmul_rn(f, __dsub_rn(y1, y0))), xs);
                                }
                            }
                        }
                    }
                } else if constexpr (s.kind == TSB_MEAS_AT) {
                    const double L = a.meas_level[m];
                    if (st[TSB_BLOCK].x == 0.0 && x1 >= L) {
                        st[TSB_BLOCK].x = 1.0;
                        if (prev) st[0].x = tsb_meas_interp(x0, sm[(2 * s.col + 1) * TSB_BLOCK].y, x1, y1, L);
                        else if (x1 == L) st[0].x = y1;                  // (x_0 > level: outside the series, stays NaN)
                    }
                } else if constexpr (s.kind == TSB_MEAS_MAX || s.kind == TSB_MEAS_MIN) {
                    if (x1 >= a.meas_from[m] && x1 <= a.meas_to[m]) {
                        const double e = st[0].x;
                        const bool better = s.kind == TSB_MEAS_MAX ? y1 > e : y1 < e;      // strict: a tie keeps the first row
                        if (better | ((e != e) & (y1 == y1))) st[0] = make_double2(y1, x1);
                    }
                } else {
                    if (prev) {
                        const double from = a.meas_from[m], to = a.meas_to[m];
                        const double lo = x0 > from ? x0 : from, hi = x1 < to ? x1 : to;      // the segment clipped to the window
                        if (lo < hi) {
                            const double y0 = sm[(2 * s.col + 1) * TSB_BLOCK].y;
                            const double ylo = lo == x0 ? y0 : tsb_meas_interp(x0, y0, x1, y1, lo);
                            const double yhi = tsb_meas_interp(x0, y0, x1, y1, hi);
                            const double w = __dsub_rn(hi, lo);
                            const double h = s.kind == TSB_MEAS_RMS ? __dadd_rn(__dmul_rn(ylo, ylo), __dmul_rn(yhi, yhi)) : __dadd_rn(ylo, yhi);
                            st[0].x = __dadd_rn(st[0].x, __dmul_rn(__dmul_rn(w, h), 0.5));
                        }
                    }
                }
            }
            emit_meas_entry<m + 1>(row, prev, x0, x1);
        }
    }
    // xf, xl: column 0 of the first and of the last stored row
    __device__ __forceinline__ void meas_finish() { meas_finish_entry<0>(sm[0].x, sm[1 * TSB_BLOCK].y); }
    template <int m> __device__ __forceinline__ void meas_finish_entry(double xf, double xl) {
        if constexpr (m < TSB_MEAS) {
            constexpr TsbMeasSpec s = tsb_meas_spec(m);
            const double nan = __longlong_as_double(0x7ff8000000000000LL);
            if constexpr (s.col < NCOL && s.tcol < NCOL) {
                const double2 st = meas_slot(m)[0];
                double v = st.x, xa = st.y;
                if constexpr (s.kind == TSB_MEAS_AT) xa = a.meas_level[m];
                if constexpr (s.kind >= TSB_MEAS_AVG) {
                    const double from = a.meas_from[m], to = a.meas_to[m];
                    const double lo = from == -TSB_INF ? xf : from, hi = to == TSB_INF ? xl : to;
                    xa = nan;
                    if (n_rows == 0 || lo < xf || hi > xl || lo > hi) v = nan;
                    else if (s.kind == TSB_MEAS_AVG) v = __ddiv_rn(v, __dsub_rn(hi, lo));
                    else if (s.kind == TSB_MEAS_RMS) v = __dsqrt_rn(__ddiv_rn(v, __dsub_rn(hi, lo)));
                }
                a.meas_out[(long long)m * a.n_inst + inst] = v;
                a.meas_out[(long long)(TSB_MEAS + m) * a.n_inst + inst] = xa;
            }
            meas_finish_entry<m + 1>(xf, xl);
        }
    }
#endif
    __device__ __forceinline__ double grid_time(int k) const {
        const double t = __dadd_rn(a.tstart, __dmul_rn((double)(k + 1), a.grid_dt));   // two roundings in every build (no FMA)
        return t < a.tstop ? t : a.tstop;
    }
    // TSB_OUT_GRID: every grid time in (previous stored row, this row] is written now, interpolated linearly between
    // the two rows (the previous one is the `last` slot of the statistics pairs; before the first row: constant).
    __device__ __forceinline__ void emit_grid(const double* row) {
        const double t1 = row[0];
        while (grid_k < a.n_grid) {
            const double tg = grid_time(grid_k);
            if (tg > t1) break;
            double w = 1.0;
            if (n_rows > 0) { const double t0 = sm[1 * TSB_BLOCK].y; w = (tg - t0) / (t1 - t0); }
            double* o = a.wave + ((long long)grid_k * NCOL) * a.n_inst + inst;
            __stcs(o, tg);
#pragma unroll
            for (int j = 1; j < NCOL; ++j) {
                const double v0 = n_rows > 0 ? sm[(2 * j + 1) * TSB_BLOCK].y : row[j];
                __stcs(o + j * a.n_inst, v0 + (row[j] - v0) * w);
            }
            ++grid_k;
        }
    }
    __device__ __forceinline__ void push(const double* row) {
        if (TSB_GRID && (a.out_flags & TSB_OUT_GRID)) emit_grid(row);      // TSB_GRID: kernels specialised for grid output
        if (a.out_flags & TSB_OUT_WAVE) {
            if (n_rows < a.cap_rows) {
                double* w = a.wave + (n_rows * NCOL) * a.n_inst + inst;
#pragma unroll
                for (int j = 0; j < NCOL; ++j) __stcs(w + j * a.n_inst, row[j]);     // streaming store: written once, never re-read
            } else overflow = true;
        }
#if TSB_MEAS
        if (a.out_flags & TSB_OUT_MEAS) emit_meas(row);      // TSB_OUT_MEAS implies TSB_OUT_STATS: reads the `last` slots first
#endif
#if TSB_FOUR
        if (a.out_flags & TSB_OUT_FOUR) emit_four(row);      // TSB_OUT_FOUR implies TSB_OUT_STATS: reads the `last` slots first
#endif
        if (a.out_flags & TSB_OUT_STATS) {
            if (n_rows == 0) sm[0] = make_double2(row[0], row[0]);     // column 0: the first row, kept in the {min, max} slot
            // running min / max that ignore NaN samples (the accumulators start at +-inf and can never become NaN
            // themselves), i.e. fmin / fmax semantics without their NaN fix-up code.  TSB_X_GROW = 1 tests all columns
            // first and updates under one seldom-taken branch; measured slower than the unconditional selects
            // (260 vs 277 ms, rlc 2^20), so it is off.
            bool grow = !TSB_X_GROW;
#pragma unroll
            for (int j = 1; TSB_X_GROW && j < NCOL; ++j) {
                const double2 mm = sm[(2 * j) * TSB_BLOCK];
                grow |= (row[j] < mm.x) | (row[j] > mm.y);
            }
            if (grow) {
#pragma unroll
                for (int j = 1; j < NCOL; ++j) {
                    const double v = row[j];
                    double2 mm = sm[(2 * j) * TSB_BLOCK];
                    if (TSB_X_STATS_PRED) {
                        // two predicated 8-byte stores instead of four selects and an unconditional 16-byte store: an extreme
                        // seldom moves, so most of them are predicated off (no shared-memory traffic at all)
                        double* slot = reinterpret_cast<double*>(&sm[(2 * j) * TSB_BLOCK]);
                        if (v < mm.x) slot[0] = v;
                        if (v > mm.y) slot[1] = v;
                    } else {
                        mm.x = v < mm.x ? v : mm.x;
                        mm.y = v > mm.y ? v : mm.y;
                        sm[(2 * j) * TSB_BLOCK] = mm;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < NCOL; ++j) {
                double2 sl = sm[(2 * j + 1) * TSB_BLOCK];
                sl.x += row[j];
                sl.y = row[j];
                sm[(2 * j + 1) * TSB_BLOCK] = sl;
            }
        }
        ++n_rows;
    }
    __device__ __forceinline__ void finish(bool ok = true) {
        if (TSB_GRID && (a.out_flags & TSB_OUT_GRID) && ok && n_rows > 0) {
            // grid times after the last stored row (it was dropped by StoreTimeResult's de-duplication): hold its values
            while (grid_k < a.n_grid) {
                double* o = a.wave + ((long long)grid_k * NCOL) * a.n_inst + inst;
                __stcs(o, grid_time(grid_k));
#pragma unroll
                for (int j = 1; j < NCOL; ++j) __stcs(o + j * a.n_inst, sm[(2 * j + 1) * TSB_BLOCK].y);
                ++grid_k;
            }
        }
#if TSB_MEAS
        if (a.out_flags & TSB_OUT_MEAS) meas_finish();
#endif
#if TSB_FOUR
        if (a.out_flags & TSB_OUT_FOUR) four_finish();
#endif
        if (a.out_flags & TSB_OUT_STATS) {
#pragma unroll
            for (int j = 0; j < NCOL; ++j) {
                double2 mm = sm[(2 * j) * TSB_BLOCK];
                const double2 sl = sm[(2 * j + 1) * TSB_BLOCK];
                if (j == 0 && n_rows > 0) {          // monotone in either direction: extremes are the first and the last row
                    const double f = mm.x, l = sl.y;
                    mm.x = f < l ? f : l; mm.y = f < l ? l : f;
                }
                a.stats[(long long)(0 * NCOL + j) * a.n_inst + inst] = mm.x;
                a.stats[(long long)(1 * NCOL + j) * a.n_inst + inst] = mm.y;
                a.stats[(long long)(2 * NCOL + j) * a.n_inst + inst] = sl.x;
                a.stats[(long long)(3 * NCOL + j) * a.n_inst + inst] = sl.y;
            }
        }
        a.rows[inst] = (TSB_GRID && (a.out_flags & TSB_OUT_GRID)) ? (long long)grid_k : n_rows;
    }
};

// ------------------------------------------------------------------------------------------------
// Shared time grid.  In a sweep over R / L / C ... values the SOURCES are the same in every instance, and as long as
// two instances have taken the same accept / reject decisions so far they are at the same (time, dt): everything that
// depends on those two numbers only — the clamped step, 1/dt, every source value (a 45-instruction math.Sin), the
// formatted-time key of StoreTimeResult — is the same in both, bit for bit.  One extra launch of the SAME kernel, the
// pilot (one instance, one warp, an SM to itself, so it advances ~2-3x faster per step than a warp that shares its
// scheduler with five others), publishes these values per attempt; every other thread looks attempt k up, checks that
// the entry's (time, dt) are its own bit for bit, and on a hit skips the computation.  A miss — entry not published
// yet, or this instance took another decision somewhere (its LTE differs) — runs the very instructions the pilot ran,
// so results do not depend on hits and misses (test_shared_time_grid_changes_no_bit).  Decisions (LTE, step growth,
// solve failures) always stay per instance.  Entries are immutable once published: the pilot stores the entry, then
// the count with release semantics; readers load the count with acquire semantics and entries below it through L2.
#ifndef TSB_TGRID
#define TSB_TGRID 0
#endif
#ifndef TSB_X_TG_EARLY
#define TSB_X_TG_EARLY 1            // issue the table loads at the top of the attempt (in flight during the LTE test and the
#endif                              // factorisation) instead of where their values are consumed
// entry = [time, dt | key, SV[0] | SV[1], SV[2] | ...]: 32 bytes for a circuit with one source
#define TSB_TG_HDR 3
#define TSB_TG_NO_KEY (-3.0)       // key slot of an attempt the pilot rejected before it needed sources and key
template <int NSRC> struct TsbTgLayout { static constexpr int ND = ((TSB_TG_HDR + NSRC + 1) / 2) * 2; };
__device__ __forceinline__ unsigned long long tsb_ld_acquire(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void tsb_st_release(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// A look at the published count is a relaxed load (no L1 invalidation — ld.acquire costs a CCTL.IVALL, which also evicts
// the block's spilled registers); only a look that FINDS new entries is followed by the acquire fence.
__device__ __forceinline__ unsigned long long tsb_ld_relaxed(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void tsb_fence_acquire() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void tsb_prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
#ifndef TSB_TG_PUBLISH_EVERY
#define TSB_TG_PUBLISH_EVERY 8      // the pilot releases the count every 8 entries (a release is a MEMBAR: ~1 us)
#endif
#ifndef TSB_TG_LOOK_EVERY
#define TSB_TG_LOOK_EVERY 16        // a reader that has caught up with the published count looks again every 16 attempts
#endif
#ifndef TSB_TG_CACHED
#define TSB_TG_CACHED 0             // 0: entries are read from L2 (ld.global.cg) — measured FASTER than through L1 (rlc, 2^20
#endif                              // instances: 219 vs 236 ms): the block's spilled registers live in L1 and table lines evict them
#ifndef TSB_TG_PREFETCH
#define TSB_TG_PREFETCH 0           // L1 prefetch one attempt ahead (only with TSB_TG_CACHED)
#endif
#if TSB_TG_CACHED
#define TSB_TG_LD(p) __ldca(p)
#else
#define TSB_TG_LD(p) __ldcg(p)
#endif

// ------------------------------------------------------------------------------------------------
// An accepted transient step (tran.go:137-151): LoadState, Update, advance time, StoreTimeResult with its
// formatted-time de-duplication (anlysis.go:61-85; `last_key` < 0 = nothing stored yet), step growth.
// HAVE_KEY: the caller already holds key(next_time) (tsb_tran_linear computes or looks it up with the step's other
// time-only quantities); otherwise it is computed here.
template <bool HAVE_KEY = false, bool HAVE_SMALL = false, class Ckt, class Sink>
__device__ __forceinline__ void tsb_accept_step(const TsbArgs& a, Ckt& c, Sink& sink, double& time, double& dt,
                                                double next_time, double lte, TsbTimeKeyer& keyer, double& last_key, double key_in = 0.0,
                                                bool lte_small = false) {
    c.load_state(dt);
    c.update_state();
    time = next_time;
    if (time >= a.tstart) {
        double key = HAVE_KEY ? key_in : keyer.key(time);             // equal times give equal keys, so one comparison covers both tests
        if (key != last_key) {
            double row[Ckt::NCOL_MAX];
            row[0] = time;
            c.signals(row + 1);
            sink.push(row);
            last_key = key;
        }
    }
    if (time < a.tstop && dt < a.maxstep) {
        // math.Min of two finite positive numbers (dt is never NaN): a plain select
        const double grown = (HAVE_SMALL ? lte_small : lte < a.trtol / 100) ? dt * 2 : dt * 1.1;
        dt = grown < a.maxstep ? grown : a.maxstep;
    }
}

// Transient loop of a circuit WITHOUT nonlinear devices when work whose result the reference discards is compiled
// away (tsb_opts.skip_linear_resolve): no Newton state machine, analysis mode fixed at compile time (mode selects,
// the LoadGmin branch and the dt > 0 guards fold away).  Same statements as tran.go:96-151 / 157-216 with
//   * iter = 0, 1 collapsed into one stamp+factor+solve (the second solve repeats identical bits);
//   * the truncation-error test hoisted ABOVE the solve: calculateTruncError (tran.go:239-250) reads only the device
//     state of the last ACCEPTED steps (CalculateLTE uses Voltage0/1, Current0/1, set by LoadState/UpdateState after
//     an accept), never the solution just computed, so a step the reference rejects for LTE is known to be rejected
//     before its solve — which the reference executes and throws away.  Not executed here; counted as the
//     reference counts it (2 solves; a lane whose matrix is singular exactly at such a step would count 1);
//   * the step body kept free of branches up to the accept (TSB_X_NB): reciprocal of dt, source evaluation,
//     factorisation and substitution form one basic block, so the independent chains (math.Sin polynomial, 1/dt,
//     pivot reciprocals) overlap instead of queueing behind each other's latency.
//   * everything that depends on (time, dt) only is computed at the top of the attempt — or looked up in the shared
//     time grid (above), when the batch has one.
template <class Ckt, class Sink>
__device__ __forceinline__ void tsb_tran_linear(const TsbArgs& a, Ckt& c, Sink& sink, long long& n_acc_out, long long& n_rej_out,
                                                long long& n_sol_tran_out, long long& n_exec_out, int& status, double& fail_at) {
    double time = 0.0, dt = a.minstep;
    double last_key = -1.0;
    TsbTimeKeyer keyer; keyer.reset();
    int n_acc = 0, n_rej = 0, n_bad = 0;   // accepted, rejected, failed solves; attempt number = n_acc + n_rej
    constexpr int ND = TsbTgLayout<Ckt::NSRC>::ND;
    const bool tg_pub = TSB_TGRID && a.tgrid != nullptr && a.tgrid_role == 1;
    // entries [0, tg_limit) are known to be published.  TSB_X_TGLOOK: tg_limit is 0 when this thread does not (or no longer)
    // read the table, and tg_next is the attempt at which the published count is looked at again — the first multiple of
    // TSB_TG_LOOK_EVERY at or above tg_limit, INT_MAX when off — so the hot path is two integer compares (k == tg_next,
    // k < tg_limit); the older form (tg_limit = -1 for "off", three tests and two reconvergence points) cost 12 instructions
    // per attempt.  Same look-ups at the same attempts either way.
    const bool tg_reader = TSB_TGRID && a.tgrid != nullptr && a.tgrid_role == 0;
    int tg_limit = TSB_X_TGLOOK ? 0 : (tg_reader ? 0 : -1);
    int tg_next = tg_reader ? 0 : 0x7fffffff;
#if TSB_X_UNROLL2
#pragma unroll 2
#endif
    while (time < a.tstop) {
        const int k = n_acc + n_rej;                       // attempt number: the table index
        const double t_tag = time, dt_tag = dt;
        bool look = false;
        if (TSB_TGRID && TSB_X_TGLOOK) {
            if (k == tg_next) {
                // caught up with what this thread knows to be published: look again every few attempts (a reader that
                // runs ahead of the pilot will not find anything new for a while)
                const unsigned long long pub = tsb_ld_relaxed(a.tgrid_pub);
                const int lim = pub < (unsigned long long)a.tgrid_cap ? (int)pub : a.tgrid_cap;
                if (lim > k) { tsb_fence_acquire(); tg_limit = lim; tg_next = (lim + TSB_TG_LOOK_EVERY - 1) & ~(TSB_TG_LOOK_EVERY - 1); }
                else tg_next = k + TSB_TG_LOOK_EVERY;
                if (k >= a.tgrid_cap) { tg_limit = 0; tg_next = 0x7fffffff; }
            }
            look = k < tg_limit;
        } else if (TSB_TGRID && tg_limit >= 0) {
            if (k >= tg_limit && (k & (TSB_TG_LOOK_EVERY - 1)) == 0) {
                const unsigned long long pub = tsb_ld_relaxed(a.tgrid_pub);
                const int lim = pub < (unsigned long long)a.tgrid_cap ? (int)pub : a.tgrid_cap;
                if (lim > k) { tsb_fence_acquire(); tg_limit = lim; }
                if (k >= a.tgrid_cap) tg_limit = -1;
            }
            look = k < tg_limit;
            if (TSB_TG_PREFETCH && look) tsb_prefetch_l1(a.tgrid + (long long)k * ND);      // consumed after the factorisation
        }
#if TSB_X_TGLOOK
        double2 e0, e1;            // only read under `look` (no zero-initialisation: four instructions per attempt)
#else
        double2 e0 = make_double2(0.0, 0.0), e1 = make_double2(0.0, 0.0);
#endif
        if (TSB_TGRID && TSB_X_TG_EARLY && look) {          // in flight during the LTE test and the factorisation
            const double2* e = reinterpret_cast<const double2*>(a.tgrid + (long long)k * ND);
            e0 = TSB_TG_LD(e); e1 = TSB_TG_LD(e + 1);
        }
        double next_time = time + dt;
        if (next_time > a.tstop) { next_time = a.tstop; dt = next_time - time; }
        __builtin_assume(dt > 0.0);               // time < tstop and dt only halves while > minstep: lets the dt > 0 guards fold
        const double rdt = tsb_rcp_dt(dt);        // the one division by the time step of this attempt
        // the two decisions the truncation error feeds (reject; how the step grows), NaN semantics of the reference's maximum kept
        double lte = 0.0;
        bool lte_gt, lte_small;
        if (TSB_X_LTEFLAGS) c.lte_flags(dt, rdt, a.trtol, a.trtol / 100, lte_gt, lte_small);
        else { lte = c.lte(dt, rdt); lte_gt = lte > a.trtol; lte_small = lte < a.trtol / 100; }
        if (lte_gt && dt > a.minstep) {
            if (tg_pub && k < a.tgrid_cap) {      // the pilot rejected this attempt before it needed sources or key
                double2* e = reinterpret_cast<double2*>(a.tgrid + (long long)k * ND);
                __stcg(e, make_double2(t_tag, dt_tag));
                __stcg(e + 1, make_double2(TSB_TG_NO_KEY, 0.0));
                if ((k & (TSB_TG_PUBLISH_EVERY - 1)) == TSB_TG_PUBLISH_EVERY - 1) tsb_st_release(a.tgrid_pub, (unsigned long long)k + 1);
            }
            dt /= 2; ++n_rej; continue;
        }
        double key = 0.0;
        // Between the factorisation and the substitution (assemble_solve's `mid` hook): the source values at the START
        // of the step (SURVEY Q2) and the result-store key of its end — taken from the table when the entry's (time, dt)
        // are this thread's own, else computed here, the one place they are computed (the pilot's values come from
        // here too).  Branch-free sine core, general routine only for an argument beyond its range.
        auto mid = [&]() {
            bool hit = false;
            if (TSB_TGRID && look) {
                const double2* e = reinterpret_cast<const double2*>(a.tgrid + (long long)k * ND);
                if (!TSB_X_TG_EARLY) { e0 = TSB_TG_LD(e); e1 = TSB_TG_LD(e + 1); }
                hit = ((__double_as_longlong(e0.x) ^ __double_as_longlong(t_tag)) | (__double_as_longlong(e0.y) ^ __double_as_longlong(dt_tag))) == 0;
                if (!hit) { tg_limit = TSB_X_TGLOOK ? 0 : -1; tg_next = 0x7fffffff; }      // this instance has left the pilot's grid: stop looking
                hit = hit && e1.x != TSB_TG_NO_KEY;
                if (hit) {
                    key = e1.x;
                    if (Ckt::SRC_UNIFORM) {
                        c.SV[0] = e1.y;
#pragma unroll
                        for (int j = 1; j < Ckt::NSRC; j += 2) {
                            const double2 sv = TSB_TG_LD(e + 2 + j / 2);
                            c.SV[j] = sv.x;
                            if (j + 1 < Ckt::NSRC) c.SV[j + 1] = sv.y;
                        }
                    }
                }
            }
            if (!hit || !Ckt::SRC_UNIFORM) { if (!c.eval_sources_nb(time)) c.eval_sources(time, 1.0); }
            if (!hit) key = next_time >= a.tstart ? keyer.key_any(next_time) : -2.0;
            if (tg_pub && k < a.tgrid_cap) {
                double2* e = reinterpret_cast<double2*>(a.tgrid + (long long)k * ND);
                __stcg(e, make_double2(t_tag, dt_tag));
                __stcg(e + 1, make_double2(key, c.SV[0]));
#pragma unroll
                for (int j = 1; j < Ckt::NSRC; j += 2) __stcg(e + 2 + j / 2, make_double2(c.SV[j], j + 1 < Ckt::NSRC ? c.SV[j + 1] : 0.0));
                if ((k & (TSB_TG_PUBLISH_EVERY - 1)) == TSB_TG_PUBLISH_EVERY - 1) tsb_st_release(a.tgrid_pub, (unsigned long long)k + 1);
            }
        };
        bool solved;
        if constexpr (Ckt::HAS_TF) solved = c.template assemble_solve_tf<false>(time, dt, rdt, mid);      // condensed elimination (fast build)
        else solved = c.template assemble_solve<TSB_MODE_TRAN, false>(TSB_MODE_TRAN, time, dt, rdt, 0.0, mid);
        if (!solved) {
            ++n_bad;
            if (dt > a.minstep) { dt /= 2; ++n_rej; continue; }
            status = TSB_ST_TRAN_FAILED; fail_at = time;
            break;
        }
        tsb_accept_step<true, true>(a, c, sink, time, dt, next_time, lte, keyer, last_key, key, lte_small);
        ++n_acc;
    }
    if (tg_pub) { const int k = n_acc + n_rej; tsb_st_release(a.tgrid_pub, (unsigned long long)(k < a.tgrid_cap ? k : a.tgrid_cap)); }
    n_acc_out += n_acc; n_rej_out += n_rej;
    const int failed = status == TSB_ST_TRAN_FAILED ? 1 : 0;
    // rejected attempts whose solve WAS executed: those rejected for a failing solve (n_bad - failed)
    n_exec_out += n_acc + (n_bad - failed) + failed;
    n_sol_tran_out += 2LL * (n_acc + n_rej) - n_bad + 2 * failed;      // the reference stops at a failing solve, else runs two
}

// ------------------------------------------------------------------------------------------------
// Transient loop of a circuit WITH nonlinear devices, warp-synchronous: the time loop and the Newton loop of
// tran.go:96-151 / 157-216 as two nested loops whose trip counts are decided by warp votes — every lane of the warp
// starts a step attempt together, iterates until the slowest live lane's Newton loop has returned (lanes that are
// through idle, a ballot per trip), then the whole warp does truncation error / accept / store together.  The
// analysis mode is a compile-time constant here (mode selects and the LoadGmin branch fold away), and there is no
// phase / continuation state machine in the hot loop.  `active` = this lane has an instance that reached the
// transient; every lane of the warp must call (the votes use the full mask).
#ifndef TSB_X_NLLOOP
#define TSB_X_NLLOOP 1
#endif
template <class Ckt, class Sink>
__device__ __forceinline__ void tsb_tran_nonlinear(const TsbArgs& a, Ckt& c, Sink& sink, bool active, long long& n_acc_out,
                                                   long long& n_rej_out, long long& n_sol_tran_out, long long& n_exec_out,
                                                   int& status, double& fail_at) {
    constexpr int N = Ckt::N;
    double time = 0.0, dt = a.minstep;                  // tran.go:93
    double last_key = -1.0;
    TsbTimeKeyer keyer; keyer.reset();
    int n_acc = 0, n_rej = 0, n_sol = 0;
    bool live = active && time < a.tstop;
    while (__any_sync(0xffffffffu, live)) {
        // ---- top of `for tr.time < tr.stopTime` (tran.go:96-111) ------------------------------------------
        double next_time = time + dt;
        if (next_time > a.tstop) { next_time = a.tstop; dt = next_time - time; }
        double rdt = 0.0;
        if (live) {
            // sources are evaluated at the START of the step (SURVEY Q2); branch-free sine core, general routine only
            // for an argument beyond its range
            if (!c.eval_sources_nb(time)) c.eval_sources(time, 1.0);
            rdt = tsb_rcp_dt(dt);                        // the one division by the time step of this attempt
        }
        // ---- doNRiter (tran.go:157-216) ---------------------------------------------------------------------
        int iter = 0;
#if TSB_X_NRSTATE
        // one integer per lane (0 iterating, 1 converged, 2 failed / not live): three bools carried across the loop were kept
        // byte-packed by the compiler — 9 PRMT and a dozen flag instructions per trip (r02_notes section 9)
        int nr = live ? 0 : 2;
        while (__any_sync(0xffffffffu, nr == 0)) {
            if (nr == 0) {
                if (iter > 0) c.update_nl(c.xo);
                bool solved;
                if constexpr (Ckt::HAS_TF) solved = c.template assemble_solve_tf<true>(time, dt, rdt, typename Ckt::TsbNoMid());   // condensed elimination
                else solved = c.template assemble_solve<TSB_MODE_TRAN>(TSB_MODE_TRAN, time, dt, rdt, 0.0);
                ++n_sol;
                if (!solved) nr = 2;
                else {
                    const bool cv = iter > 0 && tsb_converged<N>(c.x, c.xo, a.reltol, a.abstol);
                    if (cv) nr = 1;
                    else {
#pragma unroll
                        for (int i = 1; i <= N; ++i) c.xo[i] = c.x[i];
                        if (++iter >= a.max_iter) nr = 2;
                    }
                }
            }
        }
        const bool fail = nr == 2;
#else
        bool conv = false, fail = false, iterating = live;
        while (__any_sync(0xffffffffu, iterating)) {
            if (iterating) {
                if (iter > 0) c.update_nl(c.xo);
                bool solved;
                if constexpr (Ckt::HAS_TF) solved = c.template assemble_solve_tf<true>(time, dt, rdt, typename Ckt::TsbNoMid());   // condensed elimination
                else solved = c.template assemble_solve<TSB_MODE_TRAN>(TSB_MODE_TRAN, time, dt, rdt, 0.0);
                ++n_sol;
                if (!solved) fail = true;
                else {
                    if (iter > 0) conv = tsb_converged<N>(c.x, c.xo, a.reltol, a.abstol);
                    if (!conv) {
#pragma unroll
                        for (int i = 1; i <= N; ++i) c.xo[i] = c.x[i];
                        if (++iter >= a.max_iter) fail = true;
                    }
                }
                iterating = !(conv || fail);
            }
        }
#endif
        // ---- tran.go:113-151 ------------------------------------------------------------------------------------
        if (live) {
            if (fail) {
                if (dt > a.minstep) { dt /= 2; ++n_rej; }
                else { status = TSB_ST_TRAN_FAILED; fail_at = time; live = false; }
            } else {
                const double lte = c.lte(dt, rdt);
                if (lte > a.trtol && dt > a.minstep) { dt /= 2; ++n_rej; }
                else {
                    tsb_accept_step(a, c, sink, time, dt, next_time, lte, keyer, last_key);
                    ++n_acc;
                    live = time < a.tstop;
                }
            }
        }
    }
    n_acc_out += n_acc; n_rej_out += n_rej; n_sol_tran_out += n_sol; n_exec_out += n_sol;
}

// ------------------------------------------------------------------------------------------------
// Operating point + transient (analysis == TSB_AN_OP stops after the first operating point).
#ifndef TSB_X_WSYNC
#define TSB_X_WSYNC 1
#endif
template <class Ckt>
__device__ __forceinline__ void tsb_run_optran_instance(const TsbArgs& a, long long inst, bool valid) {
    constexpr int N = Ckt::N;
    constexpr bool LINEAR_LOOP = !Ckt::HAS_NL && (TSB_SKIP_LINEAR_RESOLVE != 0);
    // Lane refill (the "compaction of finished lanes" of the north star): lanes of a NONLINEAR circuit finish
    // at different trips (Newton counts differ, some lanes fail early).  Instead of idling until the slowest
    // lane of the warp is done, a finished lane writes its results, takes the next unprocessed instance from a
    // global counter and re-enters the SAME loop, so every trip keeps doing useful work in every lane.  Linear
    // circuits have identical step sequences in every lane of the bundled sweeps and keep the static mapping.
    // Compile-time option (tsb_opts.lane_refill -> TSB_LANE_REFILL): a de-synchronised warp executes the
    // phase-specific code (OP start, initial estimate, accept) once per distinct phase, so on sweeps whose lanes
    // all take similar trip counts refill LOSES 3-17 % (profiles/r01_notes.md) and is off by default.
    constexpr bool REFILL = Ckt::HAS_NL && (TSB_LANE_REFILL != 0);
    // Warp-synchronous Newton loops (nonlinear circuits).  Each trip of the loop below is one Newton iteration for every
    // lane, but the code that runs when a Newton loop RETURNS (truncation error, accept, result store, source
    // evaluation of the next step: ~2x the instructions of an iteration) is executed once per group of lanes that
    // return in the same trip.  Left alone, lanes drift apart and that code runs almost every trip for a handful of
    // lanes: the first profile of diode2 showed 15 of 32 threads active per instruction and 3 800 warp instructions
    // per accepted step.  With WSYNC a lane whose Newton loop has returned waits (one ballot per trip) until every
    // live lane of its warp has returned as well, then the whole warp runs the post-Newton code together: the trip
    // count becomes the per-step maximum over the warp, the expensive code runs once per step.
    constexpr bool WSYNC = Ckt::HAS_NL && !REFILL && (TSB_X_WSYNC != 0);
    constexpr bool NL_LOOP = WSYNC && (TSB_X_NLLOOP != 0);     // transient in tsb_tran_nonlinear, entered by the whole warp
    if (!WSYNC && !valid) return;
    Ckt c;
    TsbSink<Ckt::NCOL_MAX> sink(a, inst);   // NCOL_MAX = transient column count (>= OP column count)

    long long n_acc, n_rej, n_sol_tran, n_sol_op;   // as the reference would count them
    long long n_exec;                               // factor+solve passes actually executed
    int op_path, status;
    double fail_at;

    enum { PH_OP_START, PH_TRAN_BEGIN, PH_NR, PH_DONE };
    enum { C_MAIN, C_GMIN, C_GFINAL, C_SRC, C_SFINAL, C_TRAN };
    int phase, op_pass, cont, iter, mode, gstep;
    double gmin, sfac, status_dt;
    double time, dt, next_time, rdt;
    double last_key;
    TsbTimeKeyer keyer;
    bool linear_tran;                          // hand the transient over to tsb_tran_linear / tsb_tran_nonlinear

    auto begin_instance = [&]() {
        c.load(a, inst);
        c.init();
        if constexpr (Ckt::HAS_TF) c.prefactor();
        sink.begin(inst);
        n_acc = n_rej = n_sol_tran = n_sol_op = n_exec = 0;
        op_path = 0; status = TSB_ST_OK; fail_at = 0.0;
        phase = (a.analysis == TSB_AN_TRAN && a.uic) ? PH_TRAN_BEGIN : PH_OP_START;
        op_pass = 0; cont = C_MAIN; iter = 0; mode = TSB_MODE_OP; gstep = 0;
        gmin = 0.0; sfac = 0.0; status_dt = 0.0;
        time = 0.0; dt = a.minstep; next_time = 0.0; rdt = 0.0;
        last_key = -1.0; keyer.reset();
        linear_tran = false;
        if (phase == PH_TRAN_BEGIN && !(time < a.tstop)) phase = PH_DONE;
        if ((LINEAR_LOOP || NL_LOOP) && phase == PH_TRAN_BEGIN) { linear_tran = true; phase = PH_DONE; }
    };
    auto finish_instance = [&]() {
        if (sink.overflow && status == TSB_ST_OK) status = TSB_ST_OVERFLOW;
        if (a.analysis == TSB_AN_OP) a.rows[inst] = sink.n_rows; else sink.finish(status == TSB_ST_OK);
        a.status[inst] = status;
        a.counters[0 * a.n_inst + inst] = n_acc;
        a.counters[1 * a.n_inst + inst] = n_rej;
        a.counters[2 * a.n_inst + inst] = n_sol_tran;
        a.counters[3 * a.n_inst + inst] = n_sol_op;
        a.counters[4 * a.n_inst + inst] = op_path;
        a.counters[5 * a.n_inst + inst] = __double_as_longlong(fail_at);
        a.counters[6 * a.n_inst + inst] = n_exec;
        a.counters[7 * a.n_inst + inst] = sink.n_rows;
    };
    bool done = !valid;                 // lanes without an instance only take part in the ballots
    bool pend = false;                  // this lane's Newton loop has returned (conv / fail hold how)
    bool conv = false, fail = false;
    phase = PH_DONE;
    if (valid) begin_instance();

    for (;;) {
        if (!done && !pend && phase == PH_DONE) {
            if (!LINEAR_LOOP && !NL_LOOP) finish_instance();       // (else: transient + finish follow the loop, below)
            done = true;
            if (REFILL) {
                const long long slot = a.first_free + (long long)atomicAdd(a.work_counter, 1ULL);
                if (slot < a.n_run) { inst = tsb_slot_instance(a, slot, true); done = false; begin_instance(); }
            }
        } else if (!done && !pend) {
        if (phase == PH_OP_START) {
            // OperatingPoint.Execute(): linear-only initial estimate from a separate sparse matrix
            c.eval_sources(0.0, 1.0);
            bool ok = c.init_estimate(status_dt, c.xo);
            ++n_sol_op;
            if (!ok) {
#pragma unroll
                for (int i = 1; i <= N; ++i) c.xo[i] = 0.0;
            }
            gmin = 0.0; cont = C_MAIN; iter = 0; mode = TSB_MODE_OP; phase = PH_NR;
        } else if (!LINEAR_LOOP && !NL_LOOP && phase == PH_TRAN_BEGIN) {
            // top of the `for tr.time < tr.stopTime` loop (tran.go:96-111)
            next_time = time + dt;
            if (next_time > a.tstop) { next_time = a.tstop; dt = next_time - time; }
            c.eval_sources(time, 1.0);          // sources are evaluated at the START of the step (SURVEY Q2)
            rdt = tsb_rcp_dt(dt);               // the one division by the time step of this attempt
            iter = 0; mode = TSB_MODE_TRAN; gmin = 0.0; cont = C_TRAN; phase = PH_NR;
        }

        // ---------------- one Newton iteration (op.go:45-86, tran.go:172-213) -------------------
        if (Ckt::HAS_NL && (mode == TSB_MODE_OP || iter > 0)) c.update_nl(c.xo);
        const bool is_tran = mode == TSB_MODE_TRAN;
        bool solved;
        if constexpr (Ckt::HAS_TF && !(LINEAR_LOOP || NL_LOOP)) {
            // the transient runs in this state machine (lane refill, or the warp-synchronous loops switched off): its solves
            // must be the SAME arithmetic as tsb_tran_nonlinear's — the condensed elimination — or the result of an
            // instance would depend on the mapping that ran it
            if (is_tran) solved = c.template assemble_solve_tf<true>(time, dt, rdt, typename Ckt::TsbNoMid());
            else solved = c.template assemble_solve<-1>(mode, 0.0, 0.0, rdt, gmin);      // the very instantiation the other mappings' operating point runs
        } else solved = c.template assemble_solve<-1>(mode, is_tran ? time : 0.0, is_tran ? dt : 0.0, rdt, gmin);
        if (is_tran) ++n_sol_tran; else ++n_sol_op;
        ++n_exec;
        conv = false; fail = !solved;
        if (solved) {
            if (!Ckt::HAS_NL && TSB_SKIP_LINEAR_RESOLVE) {
                // A circuit without NonLinear devices re-stamps identical values in iteration 1, so the
                // reference's second solve returns the very same bits and its test |x - x| <= tol passes
                // (NaN / Inf included, SURVEY Q4).  Skip executing it; count it as the reference would.
                conv = true;
                if (is_tran) ++n_sol_tran; else ++n_sol_op;
            } else if (iter > 0) conv = tsb_converged<N>(c.x, c.xo, a.reltol, a.abstol);
            if (!conv) {
#pragma unroll
                for (int i = 1; i <= N; ++i) c.xo[i] = c.x[i];
                if (++iter >= a.max_iter) fail = true;
            }
        }
        pend = conv || fail;
        }
        if (WSYNC) {
            if (__all_sync(0xffffffffu, done)) break;
            if (!__all_sync(0xffffffffu, done || pend)) continue;      // somebody is still iterating: wait for them
            if (!pend) continue;                                       // (a finished lane)
        } else {
            if (done) break;
            if (!pend) continue;
        }
        pend = false;

        // ---------------- the Newton loop returned: decide what runs next -----------------------
        bool op_done = false, op_failed = false;
        switch (cont) {
        case C_MAIN:
            if (conv) { op_done = true; break; }
            // Gmin stepping (op.go:192-205): gmin = n*1e-3*10^10, 11 solves dividing by 10
            op_path = max(op_path, 1);
            gmin = ((double)N * 0.001) * 1e10;
            gstep = 0;
#pragma unroll
            for (int i = 1; i <= N; ++i) { a.scratch[(long long)i * a.n_inst + inst] = c.x[i]; c.xo[i] = c.x[i]; }
            iter = 0; cont = C_GMIN;
            break;
        case C_GMIN:
            if (conv) {
#pragma unroll
                for (int i = 1; i <= N; ++i) { a.scratch[(long long)i * a.n_inst + inst] = c.x[i]; c.xo[i] = c.x[i]; }
                gmin /= 10;
                if (++gstep <= 10) { iter = 0; break; }
            } else {
#pragma unroll
                for (int i = 1; i <= N; ++i) c.xo[i] = a.scratch[(long long)i * a.n_inst + inst];
            }
            gmin = 0.0; iter = 0; cont = C_GFINAL;
            break;
        case C_GFINAL:
            if (conv) { op_done = true; break; }
            // performSourceStepping (op.go:113-169): V-source DC values * 0.1 .. ~1.0
            op_path = max(op_path, 2);
            c.eval_sources(0.0, 0.1);
            {
                bool ok = c.init_estimate(0.0, c.xo);
                ++n_sol_op;
                if (!ok) {
#pragma unroll
                    for (int i = 1; i <= N; ++i) c.xo[i] = 0.0;
                }
            }
            sfac = 0.1; gmin = 0.0; iter = 0; cont = C_SRC;
            break;
        case C_SRC:
            if (!conv) { c.eval_sources(0.0, 1.0); op_failed = true; break; }
#pragma unroll
            for (int i = 1; i <= N; ++i) c.xo[i] = c.x[i];
            sfac += 0.1;
            if (sfac <= 1.0) { c.eval_sources(0.0, sfac); iter = 0; }
            else { c.eval_sources(0.0, 1.0); iter = 0; cont = C_SFINAL; }
            break;
        case C_SFINAL:
            if (conv) op_done = true; else op_failed = true;
            break;
        case C_TRAN:
            if (LINEAR_LOOP || NL_LOOP) break;    // these run their transient in tsb_tran_linear / tsb_tran_nonlinear
            if (fail) {
                // tran.go:113-120
                if (dt > a.minstep) { dt /= 2; ++n_rej; phase = PH_TRAN_BEGIN; }
                else { status = TSB_ST_TRAN_FAILED; fail_at = time; phase = PH_DONE; }
                break;
            }
            {
                double lte = c.lte(dt, rdt);                      // tran.go:122, 239-250
                if (lte > a.trtol && dt > a.minstep) { dt /= 2; ++n_rej; phase = PH_TRAN_BEGIN; break; }
                tsb_accept_step(a, c, sink, time, dt, next_time, lte, keyer, last_key);
                ++n_acc;
                phase = time < a.tstop ? PH_TRAN_BEGIN : PH_DONE;
            }
            break;
        }
        if (op_failed) { status = TSB_ST_OP_FAILED; phase = PH_DONE; }
        if (op_done) {
            if (a.analysis == TSB_AN_OP) {
                // storeResults (op.go:235-248): V(node) = x[i], I(dev) = x[branch] (not negated)
                double row[Ckt::NCOL_MAX];
#pragma unroll
                for (int i = 1; i <= N; ++i) row[i - 1] = c.x[i];
                // an OP row has N columns; the sink is dimensioned for the transient layout, so
                // write it directly
                if (a.out_flags & TSB_OUT_WAVE) {
#pragma unroll
                    for (int i = 0; i < N; ++i) a.wave[(long long)i * a.n_inst + inst] = row[i];
                }
                sink.n_rows = 1;
                phase = PH_DONE;
            } else if (op_pass == 0) {
                // Transient.Setup ran the first OP; SetTimeStep(tStep) leaks into the status the second
                // OP's initial estimate sees (SURVEY Q27); Transient.Execute then runs the OP again.
                op_pass = 1; status_dt = a.tstep; phase = PH_OP_START;
            } else {
                time = 0.0; dt = a.minstep;                        // tran.go:93
                phase = time < a.tstop ? PH_TRAN_BEGIN : PH_DONE;
                if (LINEAR_LOOP || NL_LOOP) { linear_tran = true; phase = PH_DONE; }
            }
        }
    }
    if (LINEAR_LOOP) {
#if TSB_COOP
        if (a.coop_state) {           // hand-over to the cooperative transient kernel (status != OK: it has nothing to run)
            if (linear_tran) c.dump_state(a.coop_state, a.n_inst, inst);
            finish_instance();
            return;
        }
#endif
        // the operating point(s) ran in the loop above; the transient of a linear circuit has its own loop, kept
        // outside so that its register allocation is not entangled with the Newton state machine
        if (linear_tran) tsb_tran_linear(a, c, sink, n_acc, n_rej, n_sol_tran, n_exec, status, fail_at);
        finish_instance();
    }
    if (NL_LOOP) {
#if TSB_COOP
        if (a.coop_state) {           // hand-over to the cooperative transient kernel, as for linear circuits above
            if (valid) {
                if (linear_tran) c.dump_state(a.coop_state, a.n_inst, inst);
                finish_instance();
            }
            return;
        }
#endif
        // every lane of the warp arrives here together (the loop above ends on a full-warp vote)
        tsb_tran_nonlinear(a, c, sink, valid && linear_tran, n_acc, n_rej, n_sol_tran, n_exec, status, fail_at);
        if (valid) finish_instance();
    }
}

// ------------------------------------------------------------------------------------------------
// DC sweep (dc.go:88-187): per sweep value one stamp whose solution is never used, then Newton with state continuation.
// The sweep values are the same for every instance, so the outer loop is warp-uniform; the Newton loop is
// vote-controlled like the transient one (lanes that have converged wait for the slowest live lane, then the whole
// warp stores the point together).  The discarded pass (dc.go:119-125: Stamp + LoadGmin + Solve before doNRiter)
// keeps only what has an effect — the side effects of Stamp() on device state; its factor + solve, whose result the
// first Newton iteration overwrites before anything reads it, are not executed.  `valid`: this lane has an instance
// (every lane of a warp must call: full-mask votes).
// Nested sweep (dc.go:205-288, Ckt::DC_NESTED): the host flattens `for val1 { for val2 {...} }` into one list of
// points (sweep[k], sweep2[k]) — SetValue on the outer source with an unchanged value is idempotent — and a stored row
// is [SWEEP1, SWEEP2, signals...] (StoreNestedResult).
template <class Ckt>
__device__ __forceinline__ void tsb_run_dc_instance(const TsbArgs& a, long long inst, bool valid) {
    constexpr int N = Ckt::N;
    constexpr int NC = Ckt::NCOL_MAX + Ckt::DC_NESTED;
    Ckt c;
    TsbSink<NC> sink(a, inst);
    if (valid) { c.load(a, inst); c.init(); sink.begin(inst); }
    int n_sol = 0, n_pts = 0;
    int status = TSB_ST_OK;
    double fail_at = 0.0;
    bool live = valid;
    for (int k = 0; k < a.n_sweep && __any_sync(0xffffffffu, live); ++k) {
        if (live) {
            c.set_dc(a.sweep[k]);
            if (Ckt::DC_NESTED) c.set_dc2(a.sweep2[k]);
            c.eval_sources(0.0, 1.0);
            (void)c.template assemble_solve<TSB_MODE_OP, true, false>(TSB_MODE_OP, 0.0, 0.0, 0.0, 1e-12);
            ++n_pts;
        }
        int iter = 0;
        int nr = live ? 0 : 2;                       // 0 iterating, 1 converged, 2 failed / not live (see tsb_tran_nonlinear)
        while (__any_sync(0xffffffffu, nr == 0)) {
            if (nr == 0) {
                if (Ckt::HAS_NL && iter > 0) c.update_nl(c.xo);
                const bool solved = c.template assemble_solve<TSB_MODE_OP>(TSB_MODE_OP, 0.0, 0.0, 0.0, 0.0);
                ++n_sol;
                if (!solved) nr = 2;
                else {
                    const bool cv = iter > 0 && tsb_converged_dc<N>(c.x, c.xo, a.reltol, a.abstol);
                    if (cv) nr = 1;
                    else {
#pragma unroll
                        for (int i = 1; i <= N; ++i) c.xo[i] = c.x[i];
                        if (++iter >= a.max_iter) nr = 2;
                    }
                }
            }
        }
        const bool fail = nr == 2;
        if (live) {
            if (fail) { status = TSB_ST_DC_FAILED; fail_at = a.sweep[k]; live = false; }
            else {
                double row[NC];
                row[0] = a.sweep[k];
                if (Ckt::DC_NESTED) row[1] = a.sweep2[k];
                c.signals(row + 1 + Ckt::DC_NESTED);
                sink.push(row);
            }
        }
    }
    if (!valid) return;
    if (sink.overflow && status == TSB_ST_OK) status = TSB_ST_OVERFLOW;
    sink.finish();
    a.status[inst] = status;
    a.counters[0 * a.n_inst + inst] = 0;
    a.counters[1 * a.n_inst + inst] = 0;
    a.counters[2 * a.n_inst + inst] = 0;
    a.counters[3 * a.n_inst + inst] = n_sol;
    a.counters[4 * a.n_inst + inst] = 0;
    a.counters[5 * a.n_inst + inst] = __double_as_longlong(fail_at);
    a.counters[6 * a.n_inst + inst] = n_sol;                  // factor + solve passes executed (the discarded pass solves nothing)
    a.counters[7 * a.n_inst + inst] = sink.n_rows;
}

// ------------------------------------------------------------------------------------------------
// AC analysis (ac.go:51-98): for every frequency of the sweep (the same list for every instance) one complex solve of
// the small-signal system; a row is [FREQ, |V(n)|, phase(V(n)) in degrees ..., |I(Vsrc)|, phase ...].  Linear circuits
// only (see plan.cpp: device_ac_entries).  A zero pivot is the reference's "matrix solve error at f=...": the instance
// keeps the rows stored so far and fails there.
#define TSB_ST_AC_FAILED 5
template <class Ckt>
__device__ __forceinline__ void tsb_run_ac_instance(const TsbArgs& a, long long inst) {
    if constexpr (Ckt::HAS_AC) {
        constexpr int N = Ckt::N;
        Ckt c;
        TsbSink<Ckt::NCOL_AC> sink(a, inst);
        c.load(a, inst);
        sink.begin(inst);
        int status = TSB_ST_OK, n_sol = 0;
        double fail_at = 0.0;
        for (int k = 0; k < a.n_sweep; ++k) {
            const double freq = a.sweep[k];
            const double omega = 6.283185307179586 * freq;           // 2 * math.Pi * status.Frequency
            double xr[N + 1], xi[N + 1];
            ++n_sol;
            if (!c.solve_ac(omega, xr, xi)) { status = TSB_ST_AC_FAILED; fail_at = freq; break; }
            double row[Ckt::NCOL_AC];
            row[0] = freq;
            c.signals_ac(xr, xi, (a.out_flags & TSB_OUT_AC_REFREAD) != 0, row + 1);
            sink.push(row);
        }
        if (sink.overflow && status == TSB_ST_OK) status = TSB_ST_OVERFLOW;
        sink.finish();
        a.status[inst] = status;
        for (int q = 0; q < 5; ++q) a.counters[q * a.n_inst + inst] = 0;
        a.counters[3 * a.n_inst + inst] = n_sol;
        a.counters[5 * a.n_inst + inst] = __double_as_longlong(fail_at);
        a.counters[6 * a.n_inst + inst] = n_sol;
        a.counters[7 * a.n_inst + inst] = sink.n_rows;
    }
}

#endif  // TSB_SKELETON_CUH
