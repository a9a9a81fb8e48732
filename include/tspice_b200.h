/* tspice_b200.h — C ABI of the B200-native batched circuit-simulation engine.
 *
 * Drop-in boundary for ONE hot path of edp1096/toy-spice: many independent instances of one
 * parsed netlist (parameter sweep / Monte Carlo) solved at once for operating point, DC sweep
 * and transient analysis.  Netlist parsing and MNA node numbering stay on the host (the
 * reference's own pkg/netlist + pkg/circuit); this library takes the already-numbered device
 * table and replaces, for the whole batch, what the reference does per circuit in
 *
 *   pkg/analysis/op.go:171-233    OperatingPoint.Execute  (+ doNRiter :25-88, initial
 *                                 estimate :90-111, Gmin stepping :192-214, source stepping :113-169)
 *   pkg/analysis/dc.go:88-187     DCSweep.singleSweep / doNRiter
 *   pkg/analysis/tran.go:57-250   Transient.Setup / Execute / doNRiter / calculateTruncError
 *   pkg/analysis/anlysis.go:46-85 CheckConvergence / StoreTimeResult
 *   pkg/circuit/circuit.go:165-313 Stamp / LoadState / Update / GetSolution / UpdateNonlinearVoltages
 *   pkg/device/<kind>.go          every Stamp / UpdateVoltages / LoadState / UpdateState / CalculateLTE
 *   pkg/matrix/circuit.go:57-166  Clear / AddElement / AddRHS / LoadGmin / Solve / Solution
 *   github.com/edp1096/sparse     Factor / Solve with the pivot order of the first factorization
 *
 * Conventions
 *   - every function returns TSB_OK (0) or a negative TSB_E_* code; tsb_last_error() gives text.
 *   - per-instance failures (no convergence, singular matrix, NaN) are DATA (status array),
 *     never a call failure.  No C++ exception crosses this boundary.
 *   - handles are opaque and owned by the library; every create has a destroy.  Plans keep their context alive and
 *     batches their plan, so the destroy calls may come in any order (garbage-collected hosts).
 *   - buffers passed in/out are caller-owned HOST memory unless the name says `_dev`.
 *   - indices: nodes and branches are 1-based MNA unknown numbers, 0 = ground
 *     (pkg/matrix/device.go:3-8); devices are numbered 0.. in tsb_plan_add_device call order,
 *     which must be netlist order (mutual couplings are stamped last, circuit.go:126-152).
 *   - one context drives one GPU (one process per GPU; shard instances across ranks).
 */
#ifndef TSPICE_B200_H
#define TSPICE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tsb_ctx tsb_ctx;
typedef struct tsb_plan tsb_plan;
typedef struct tsb_batch tsb_batch;
typedef struct tsb_job tsb_job;

enum {
    TSB_OK = 0,
    TSB_E_INVALID = -1,     /* bad argument / wrong state */
    TSB_E_PARSE = -2,       /* netlist front-end error (mirrors netlist.Parse errors) */
    TSB_E_CUDA = -3,        /* CUDA driver/runtime error, or no GPU / driver library */
    TSB_E_COMPILE = -4,     /* kernel specialisation failed (NVRTC) */
    TSB_E_UNSUPPORTED = -5, /* e.g. AC analysis, > 2 sweep sources */
    TSB_E_NOMEM = -6
};

/* Device kinds (pkg/netlist/parser.go:752-915 CreateDevice). */
enum {
    TSB_R = 0,     /* p: [R]                                              resistor.go  */
    TSB_C = 1,     /* p: [C]                                              capacitor.go */
    TSB_L = 2,     /* p: [L]                      branch required         inductor.go  */
    TSB_V = 3,     /* p: waveform (below), ip: [src type]  branch required vsource.go  */
    TSB_I = 4,     /* p: waveform (below), ip: [src type]                 isource.go   */
    TSB_D = 5,     /* p: [is, n, tt]                                      diode.go     */
    TSB_Q = 6,     /* p: [ies, ics, alphaf, ikf, ikr, vaf, var, nf, nr], ip: [pnp]   bjt.go */
    TSB_M = 7,     /* p: [vto,kp,gamma,phi,lambda,w,l,tox,cgso,cgdo,cgbo,cbd,cbs,cj,cjsw,as,ad,ps,pd,
                          mj,pb,uo,ucrit,uexp,vmax,theta,eta,kappa,delta], ip: [level, pmos]  mosfet.go */
    TSB_K = 8,     /* p: [k], ip: device indices of the coupled inductors  mutual.go   */
    TSB_LCORE = 9  /* p: [turns, area, len]       branch required         magnetic.go  */
};

/* Source waveforms (pkg/device/device.go:58-62).  p layout:
 *   DC    [value (, ac_mag, ac_phase_deg)]   SIN   [offset, amplitude, freq, phase_deg]
 *   PULSE [v1, v2, td, tr, tf, pw, per]   PWL [t0, v0, t1, v1, ...] (not sweepable) */
enum { TSB_SRC_DC = 0, TSB_SRC_SIN = 1, TSB_SRC_PULSE = 2, TSB_SRC_PWL = 3 };

/* Analysis kinds (pkg/analysis/anlysis.go:11-16). */
enum { TSB_AN_OP = 0, TSB_AN_TRAN = 1, TSB_AN_AC = 2, TSB_AN_DC = 3,
       TSB_AN_DC2 = 4   /* column layout of a nested DC sweep (SWEEP1, SWEEP2, signals; dc.go:272-288) for tsb_plan_num_columns / _column_name */ };

/* Per-instance status (tsb_result_status). */
enum {
    TSB_ST_OK = 0,
    TSB_ST_OP_FAILED = 1,    /* "source stepping failed" / "final solution failed"   op.go:216-229 */
    TSB_ST_TRAN_FAILED = 2,  /* "failed to converge at t=%g"                         tran.go:119  */
    TSB_ST_DC_FAILED = 3,    /* "convergence error at %s=%g"                         dc.go:128    */
    TSB_ST_OVERFLOW = 4,     /* more stored rows than the waveform capacity; rows beyond it dropped */
    TSB_ST_AC_FAILED = 5     /* "matrix solve error at f=%g"                         ac.go:68     */
};

/* Convergence constants, defaults = NewBaseAnalysis (anlysis.go:35-44) and NewTransient (tran.go:51). */
typedef struct tsb_opts {
    int max_iter;       /* 100   */
    double abstol;      /* 1e-12 */
    double reltol;      /* 1e-6  */
    double gmin;        /* 1e-12 (only recorded in ckt.Status; the solves use 0, SURVEY Q5) */
    double trtol;       /* 7.0   */
    int strict_fp;      /* 1: reference rounding (no FMA contraction, IEEE division wherever the reference divides);
                           0: fast build (FMA, one reciprocal of dt per step, reciprocal-seed pivots; each
                              substituted operation within 1 ulp); -1 (default): 1 for circuits with mutual
                              couplings (condition numbers ~1e7 make 1-ulp differences visible at 1e-9), else 0 */
    int block_size;     /* 0: default (128); rounded up to a multiple of 32 (whole warps), at most 1024 */
    int skip_linear_resolve; /* 1 (default): circuits without nonlinear devices do not execute the reference's
                           second Newton solve per step — it re-stamps identical values, returns identical bits and
                           always passes the convergence test; counters still report it (reference-equivalent) */
    int min_blocks;     /* __launch_bounds__ min resident blocks per SM for the specialised kernels.  0 (default): chosen
                           by a spill rule and, on the first transient run of a batch of >= 32768 instances, by timing the
                           candidates on a sub-batch.  THAT FIRST CALL IS NOT ASYNCHRONOUS: it blocks the host for a
                           fraction of a second (event synchronisation, possibly NVRTC), so it must not happen under CUDA
                           graph capture — it is skipped when the stream is capturing, and $TSB_AUTOTUNE=0 or an explicit
                           min_blocks > 0 disables it; the choice is remembered per process and, in the kernel cache, per
                           GPU model.  Results never depend on the choice. */
    int lane_refill;    /* 1: circuits with nonlinear devices run on a resident grid whose lanes, once their instance has
                           finished, take the next unprocessed instance from a work counter (finished lanes never idle
                           beside slow neighbours) — for sweeps whose instances need very different numbers of steps;
                           0 (default): one thread per instance, static mapping (3-17 % faster on the bundled decks,
                           whose lanes finish together).  Results are bit-identical either way. */
    double grid_dt;     /* TSB_OUT_GRID: spacing of the output grid; 0 (default) = the analysis' tStep after
                           NewTransient's clamping (tran.go:31-33), i.e. >= 300 points */
    int share_time_grid; /* transient analysis of circuits without nonlinear devices: instances that have taken the same
                           accept / reject decisions are at the same (time, dt), and what depends on those two only (the
                           clamped step, 1/dt, the source values when no source parameter varies per instance, the key of
                           StoreTimeResult's de-duplication) is the same for all of them.  1: a pilot launch (one instance,
                           beside the main launch) publishes these per attempt, every other instance looks them up and
                           verifies (time, dt) bit for bit, computing them itself on a miss — results are bit-identical
                           with and without; 0: off; -1 (default): on for batches of >= 2^18 instances */
    int coop_parts;     /* transient analysis, fast build: 2, 4 or 8 = the cooperative mapping — the netlist is cut into that many
                           sub-circuits joined by a small separator, and one instance is advanced by that many threads in
                           different warps of a block (each eliminates its own sub-circuit; a few doubles per step attempt —
                           per Newton iteration for circuits with diodes / MOSFETs — cross shared memory around named
                           barriers).  For circuits too large for one thread's registers.  The elimination order is a
                           nested-dissection order: results differ from the thread-per-circuit mapping by rounding (like the
                           fast build's other re-associations).  An explicit value fails with TSB_E_UNSUPPORTED when the
                           circuit has no such partition (tsb_plan_coop_info), has BJTs (generated dense) or mutual couplings,
                           or with strict_fp / TSB_OUT_GRID.  0: off.  -1 (default): two parts for circuits of >= 16 unknowns
                           where all of the above holds (measured on B200: RC ladders n = 18 1.6x, n = 26 2.1x, diode-clamped
                           ladder n = 26 1.8x the thread-per-circuit rate), else off */
} tsb_opts;

/* The partition behind tsb_opts.coop_parts (parts = 2 or 4): owner[u] for every unknown u = 1..n (external numbering: nodes,
   then branches; owner[0] unused) = the part that eliminates it, -1 = separator.  Returns TSB_E_UNSUPPORTED when the plan has
   no partition into `parts` sub-circuits.  `owner` holds n + 1 ints; either pointer may be NULL. */
int tsb_plan_coop_info(const tsb_plan* plan, int parts, int* owner, int* n_separator);

/* Output selection for tsb_run_tran / tsb_run_dc. */
enum {
    TSB_OUT_WAVE = 1,   /* every stored row: wave[row][column][instance]          */
    TSB_OUT_STATS = 2,  /* min / max / sum / last per column over the stored rows */
    TSB_OUT_GRID = 4,   /* transient only: the reference's result series resampled ON THE DEVICE onto the fixed grid
                           t_k = tstart + (k+1)*grid_dt <= tstop (k = 0..), by linear interpolation between
                           consecutive stored rows (constant before the first / after the last one):
                           wave[k][column][instance], column 0 = t_k.  This is how instances whose adaptive step
                           sequences differ are compared point by point, and what makes waveform output of the
                           ~2e4-step inductor decks fit in HBM for 1M+ instances.  Implies TSB_OUT_STATS; excludes
                           TSB_OUT_WAVE.  rows[inst] = grid rows written; counters[7] = rows of the reference series */
    TSB_OUT_AC_REFREAD = 8  /* AC analysis only, a modifier: read the solution out as the reference's accessor does when the
                           un-vendored sparse module follows Sparse 1.3's interleaved vectors — GetComplexSolution(i) returns
                           (solution[i], solution[i+Size]) (matrix/circuit.go:168-173) while the vector is laid out
                           solution[2k] = re x_k, solution[2k+1] = im x_k (:41-44, :85-97).  Default (flag clear): entry i is
                           (re x_i, im x_i) — what the accessor means if the module returns split halves.  The module's
                           source is not available, so both read-outs are offered (DESIGN.md, quirk Q28). */,
    TSB_OUT_MEAS = 16   /* tsb_run_tran / tsb_run_dc / tsb_run_ac: the measurements of the batch's measurement table
                           (tsb_batch_set_measures), reduced on the device from the stored rows as they are produced;
                           read with tsb_result_measures.  Implies TSB_OUT_STATS; combines with WAVE and GRID. */
};

/* ---- measurements (the SPICE .meas family, reduced on the device) -------------------------------------------------
 * The series of one instance is its stored rows (x_r, y_r), r = 0 .. last: exactly the rows TSB_OUT_WAVE would write,
 * rows beyond wave_cap_rows included; x is column 0 (TIME / SWEEP1 / FREQ), y is `column`.  Every operation below is
 * individually rounded in both builds, so a result is a function of the stored rows alone (independent of strict_fp,
 * the mapping, the processing order, lane refill and the shared time grid).
 *   WHEN   segment (r, r+1) rises when t_r < L <= t_r+1 and falls when t_r > L >= t_r+1 (t = trig_column, L = level; a
 *          NaN sample never crosses); CROSS is either.  f = (L - t_r) / (t_r+1 - t_r), x* = x_r + f (x_r+1 - x_r),
 *          value = y_r + f (y_r+1 - y_r).  Crossings with from <= x* <= to count; the result is (value, x*) of the
 *          count-th (1-based) or, count = -1, of the last one; (NaN, NaN) when there is none.  A delay (TRIG / TARG) is
 *          the difference of two WHEN abscissas.
 *   AT     r+1 = the first row with x_r+1 >= level: value = y_r+1 if x_r+1 == level, else
 *          y_r + ((level - x_r) / (x_r+1 - x_r)) (y_r+1 - y_r).  Result (value, level); value NaN for a level outside
 *          [x_0, x_last].
 *   MAX / MIN   over the rows with from <= x_r <= to, NaN samples ignored, a tie goes to the first row: (extreme, its x_r);
 *          (NaN, NaN) when no row is in the window.
 *   INTEG / AVG / RMS   window [a, b]: a = x_0 if from = -inf else from, b = x_last if to = +inf else to; NaN when
 *          a < x_0, b > x_last (an instance that failed before the window ended) or a > b.  Trapezoid rule over the
 *          segments clipped to [a, b] (an endpoint inside a segment takes its value as AT does), summed in row order
 *          from 0.0: INTEG = sum (x_hi - x_lo) (y_lo + y_hi) 0.5, AVG = INTEG / (b - a),
 *          RMS = sqrt(sum (x_hi - x_lo) (y_lo^2 + y_hi^2) 0.5 / (b - a)).  Abscissa NaN.  Zero width: INTEG 0, AVG and
 *          RMS NaN.
 * Kind, column and trig_column are compiled into the kernels (a new set of them compiles once, NVRTC); level, count,
 * edge and the window are run-time arguments.  Refused (before anything is launched): TSB_OUT_MEAS without a table or with
 * a column outside 1 .. n_columns-1 of the analysis (TSB_E_INVALID), on the nested DC sweep or with an explicit
 * coop_parts > 0 (TSB_E_UNSUPPORTED); coop_parts = -1 takes the thread-per-circuit mapping. */
enum { TSB_MEAS_WHEN = 0, TSB_MEAS_AT = 1, TSB_MEAS_MAX = 2, TSB_MEAS_MIN = 3, TSB_MEAS_AVG = 4, TSB_MEAS_INTEG = 5, TSB_MEAS_RMS = 6 };
enum { TSB_EDGE_CROSS = 0, TSB_EDGE_RISE = 1, TSB_EDGE_FALL = 2 };
enum { TSB_MEAS_CAP = 16 };
typedef struct tsb_meas {
    int kind;
    int column;        /* result column measured, 1 .. n_columns-1 of the analysis (tsb_plan_column_name) */
    int trig_column;   /* WHEN: the column whose crossing is sought (may equal `column`) */
    int edge;          /* WHEN: TSB_EDGE_* */
    int count;         /* WHEN: the count-th such crossing, 1-based; -1 = the last one */
    double level;      /* WHEN: crossing level; AT: the abscissa */
    double from, to;   /* window on column 0; -inf / +inf = the whole series */
} tsb_meas;

void tsb_default_opts(tsb_opts* o);
const char* tsb_version(void);

/* ---- context ------------------------------------------------------------------------------ */
int tsb_ctx_create(int device_ordinal, tsb_ctx** out);
void tsb_ctx_destroy(tsb_ctx* ctx);
const char* tsb_last_error(tsb_ctx* ctx);
/* Launch on an existing CUDA stream (cudaStream_t / CUstream as an integer); 0 = the context's own. */
int tsb_ctx_set_stream(tsb_ctx* ctx, uint64_t stream);
/* The stream the context launches on (cudaStream_t as an integer). */
int tsb_ctx_get_stream(tsb_ctx* ctx, uint64_t* stream);
/* Stream ordering contract for BORROWED device buffers (tsb_batch_set_param_dev, tsb_batch_stamp_dev,
 * tsb_lu_solve_batched_dev): the library reads / writes them on the context's stream and knows nothing about the stream
 * that produced them.  Either launch on that stream (tsb_ctx_set_stream), or record a cudaEvent_t on it after the producer
 * and hand it to tsb_ctx_wait_event: everything the context launches afterwards waits for the event on the device.  The
 * caller keeps borrowed buffers alive until the work that uses them has finished (tsb_batch_sync). */
int tsb_ctx_wait_event(tsb_ctx* ctx, uint64_t event);
/* Directory of the specialised-kernel cache (cubin files).  Default: $TSB_KCACHE or <lib dir>/_kcache. */
int tsb_ctx_set_cache_dir(tsb_ctx* ctx, const char* dir);
/* FP64 DFMA-chain microbenchmark on this GPU: TFLOP/s (the FP64 roof used by bench.py). */
int tsb_ctx_measure_fp64_peak(tsb_ctx* ctx, double* tflops);
int tsb_ctx_sm_count(tsb_ctx* ctx, int* sms);

/* ---- plan: one numbered netlist -------------------------------------------------------------
 * Replaces circuit.NewWithComplex + CreateMatrix + SetupDevices (circuit.go:31-163) for the batch.
 * `ctx` may be NULL for host-only use (structure queries, code generation at build time). */
int tsb_plan_create(tsb_ctx* ctx, int n_nodes, int n_branches, tsb_plan** out);
/* Host front-end convenience: C++ restatement of netlist.Parse + AssignNodeBranchMaps + CreateDevice
 * (parser.go:75-915, circuit.go:48-71) for hosts that do not bring the reference's Go parser. */
int tsb_plan_from_netlist(tsb_ctx* ctx, const char* text, tsb_plan** out);
int tsb_plan_add_device(tsb_plan* plan, int kind, const char* name, const int* nodes, int n_nodes, int branch,
                        const double* p, int n_p, const int* ip, int n_ip);
/* Freezes the plan: Translate order, stamped pattern, nominal first-factor pivot order
 * (the reference's symbolic pass), fill pattern. */
int tsb_plan_finalize(tsb_plan* plan);
void tsb_plan_destroy(tsb_plan* plan);
const char* tsb_plan_error(tsb_plan* plan);

int tsb_plan_size(const tsb_plan* plan, int* n_nodes, int* n_branches);
int tsb_plan_num_devices(const tsb_plan* plan);
int tsb_plan_device_info(const tsb_plan* plan, int dev, int* kind, const char** name, int nodes[4], int* branch,
                         int* n_p, int* n_ip);
int tsb_plan_device_params(const tsb_plan* plan, int dev, double* p, int cap_p, int* ip, int cap_ip);
int tsb_plan_find_device(const tsb_plan* plan, const char* name);            /* index or -1 */
int tsb_plan_node_name(const tsb_plan* plan, int node, const char** name);   /* from_netlist plans only */
/* What the netlist's dot-cards asked for (from_netlist plans). */
int tsb_plan_analysis(const tsb_plan* plan, int* analysis, double tran[4] /*tstart,tstop,tstep,tmax*/, int* uic,
                      int* dc_src_dev, double dc[3] /*start,stop,inc*/);
/* The rest of the dot-cards: the second source of `.dc src1 a b inc src2 a b inc` (-1: none; the reference's parser stops
 * after the first source, SURVEY Q20 — accepting the second one, `.end` and inline diode parameters `D1 a k MODEL Is=..`
 * are this front-end's hardenings), and the `.ac` card: sweep type (0 DEC, 1 OCT, 2 LIN), number of points, fstart, fstop. */
int tsb_plan_analysis2(const tsb_plan* plan, int* dc2_src_dev, double dc2[3], int* ac_sweep, int* ac_points, double ac_f[2]);
/* Structure (finalized plans).  All index arrays are 1-based with n+1 entries ([0] unused).
 *   ext2int    Sparse `Translate` numbering of the main matrix (first-touch order)
 *   pivot_row / pivot_col   external row / column of the pivot chosen at each elimination step */
int tsb_plan_structure(const tsb_plan* plan, int* ext2int, int* pivot_row, int* pivot_col);
/* Stamped pattern in first-touch order: rows[k], cols[k]; mode 0 = OP-mode stamps, 1 = + transient-only. */
int tsb_plan_pattern(const tsb_plan* plan, int mode, int* rows, int* cols, int cap, int* nnz);
/* Column names of a result row for `analysis` (TIME | SWEEP1, V(node..), I(branch..), I(R..)). */
int tsb_plan_num_columns(const tsb_plan* plan, int analysis);
int tsb_plan_column_name(const tsb_plan* plan, int analysis, int col, char* buf, int cap);

/* ---- batch: N instances of a plan -----------------------------------------------------------*/
int tsb_batch_create(tsb_plan* plan, int64_t n_inst, tsb_batch** out);
void tsb_batch_destroy(tsb_batch* batch);
/* Per-instance parameter values for (dev, param): n_inst doubles, host memory of any kind.  COPY semantics: the values
 * are staged through a library-owned pinned buffer, the caller's buffer is free again when the call returns. */
int tsb_batch_set_param(tsb_batch* batch, int dev, int param, const double* values);
/* Zero-copy variant for pinned host buffers: the H2D DMA reads `values` later.  The buffer must stay valid and unmodified
 * until the next tsb_batch_sync() (or a blocking tsb_result_* read of a run launched after this call).
 * Both variants copy on an upload stream of the context: behind this batch's own last launch and ahead of its next one, but
 * BESIDE whatever another batch of the context is running — a host that alternates two batches uploads the parameters of
 * step i + 1 while step i computes. */
int tsb_batch_set_param_async(tsb_batch* batch, int dev, int param, const double* values);
/* Same, values already resident in HBM (device pointer, n_inst doubles; borrowed until the batch
 * is destroyed or the parameter is set again). */
int tsb_batch_set_param_dev(tsb_batch* batch, int dev, int param, uint64_t dev_ptr);
/* One value for all instances (replaces the netlist value). */
int tsb_batch_set_param_uniform(tsb_batch* batch, int dev, int param, double value);

/* Optional processing order: slot s of the launch works on instance perm[s] (a permutation of 0..n_inst-1, host
 * memory, copied).  Lanes of a warp advance together, so grouping instances that need similar Newton iteration counts
 * (e.g. sorted by the parameter that drives them) removes waiting; parameters and results keep the caller's order and
 * do not change by a bit.  NULL removes the order. */
int tsb_batch_set_order(tsb_batch* batch, const int64_t* perm);

/* Measurement table of the batch (copied; n_meas <= TSB_MEAS_CAP; (NULL, 0) clears).  TSB_E_INVALID for an unknown kind, a
 * column or trig_column < 1, a NaN window or from > to, and for WHEN / AT a NaN level, for WHEN an unknown edge or count 0.
 * The columns are checked against the analysis when a run selects TSB_OUT_MEAS.  Setting a table discards the measurements
 * of the last run (tsb_result_measures fails until the next TSB_OUT_MEAS run). */
int tsb_batch_set_measures(tsb_batch* batch, const tsb_meas* m, int n_meas);

/* Analyses — the batch equivalents of analysis.NewOP / NewTransient / NewDCSweep + Setup + Execute. */
int tsb_run_op(tsb_batch* batch, const tsb_opts* opts);
int tsb_run_tran(tsb_batch* batch, double tstart, double tstop, double tstep, double tmax, int uic,
                 int out_flags, int64_t wave_cap_rows, const tsb_opts* opts);
int tsb_run_dc(tsb_batch* batch, int src_dev, double start, double stop, double inc, int out_flags,
               const tsb_opts* opts);
/* Nested sweep of two voltage sources (DCSweep.nestedSweep, dc.go:205-270): for every value of source 1 (outer loop)
 * source 2 runs through its whole range (inner loop); device state carries over from point to point exactly as in the
 * reference.  Rows are [SWEEP1, SWEEP2, signals...] (StoreNestedResult, dc.go:272-288; column names: analysis code
 * TSB_AN_DC2), n1 * n2 of them per instance.  A failing instance stops at its first non-converging point:
 * status = TSB_ST_DC_FAILED, rows[inst] = index of that point, counters[5] = the outer source's value there. */
int tsb_run_dc2(tsb_batch* batch, int src1_dev, double start1, double stop1, double inc1, int src2_dev, double start2,
                double stop2, double inc2, int out_flags, const tsb_opts* opts);
/* AC analysis (analysis.NewAC(fStart, fStop, nPoints, pType) + Setup + Execute, ac.go:21-126) of circuits WITHOUT nonlinear
 * devices: n_points frequencies in total between fstart and fstop (sweep_type 0 DEC / 1 OCT: logarithmic, 2 LIN; Go's
 * math.Log10 / Log2 / Pow restated for the point values), one complex solve per frequency and instance in the pivot order the
 * operating point of ACAnalysis.Setup froze, with what every device's Stamp does in Mode == ACAnalysis — quirks included:
 *   - an inductor is stamped as the ADMITTANCE j*omega*L between its nodes and leaves its branch row empty (inductor.go:43-57);
 *   - Mutual and MagneticInductor stamp nothing at all (their Stamp has no AC case, mutual.go:63-65, magnetic.go:205-273; the
 *     StampAC methods they define are never called by circuit.Stamp, circuit.go:165-176);
 *   so a circuit with any inductor fails with TSB_ST_AC_FAILED at the first frequency, as the reference's "matrix solve error
 *   at f=..." does (rows stored so far are kept; counters[5] = that frequency).  RC networks with V / I sources work.
 * Rows: [FREQ, V(node)_MAG, V(node)_PHASE (degrees) ..., I(vsource)_MAG, I(vsource)_PHASE ...] (StoreACResult,
 * anlysis.go:87-111: cmplx.Abs = Go's math.Hypot, cmplx.Phase*180/pi; column names: analysis code TSB_AN_AC).  AC magnitude /
 * phase of a source: parameters 1 and 2 of a DC source (`V1 1 0 AC mag [phase]`, vsource.go:98-111), sweepable per instance
 * like any other parameter.  out_flags: TSB_OUT_WAVE and / or TSB_OUT_STATS, optionally | TSB_OUT_AC_REFREAD.
 * Circuits with nonlinear devices: TSB_E_UNSUPPORTED.  The reference runs their operating point on the COMPLEX matrix with a
 * real-indexed right-hand side (AddRHS writes rhs[i], SolveComplex reads re/im pairs; matrix/circuit.go:99-105 vs :126-150),
 * Bjt.Stamp never dispatches to StampAC (bjt.go:315-374), and the small-signal values of diodes and MOSFETs come from that
 * scrambled point: a result that depends on the vector layout of a module whose source is not available. */
int tsb_run_ac(tsb_batch* batch, int sweep_type, int n_points, double fstart, double fstop, int out_flags, const tsb_opts* opts);
/* Block until the last run OF THIS BATCH has finished, its asynchronous read-back (tsb_result_fetch_async) and its parameter
 * uploads included (runs are asynchronous on the context's stream; another batch's run queued behind it is not waited for). */
int tsb_batch_sync(tsb_batch* batch);

/* ---- results of the last run -----------------------------------------------------------------
 * Layout in HBM (structure of arrays, instance is the fastest index so warps store coalesced):
 *   wave     [cap_rows][n_columns][n_inst]    stats [4: min,max,sum,last][n_columns][n_inst]
 *   rows     [n_inst] int64                   status [n_inst] int32
 *   counters [8][n_inst] int64: 0 accepted steps, 1 rejected steps, 2 transient solves, 3 OP solves (2, 3: as the
 *            reference would count them), 4 OP path (0 direct, 1 Gmin stepping, 2 source stepping),
 *            5 failure time/value (double bits), 6 factor+solve passes actually executed,
 *            7 rows of the reference's result series (== rows[] unless TSB_OUT_GRID) */
int tsb_result_dims(const tsb_batch* batch, int64_t* n_inst, int* n_columns, int64_t* cap_rows);
int tsb_result_dev_ptrs(const tsb_batch* batch, uint64_t* wave, uint64_t* stats, uint64_t* rows, uint64_t* status,
                        uint64_t* counters);
int tsb_result_rows(tsb_batch* batch, int64_t* rows /*[n_inst]*/);
int tsb_result_status(tsb_batch* batch, int32_t* status /*[n_inst]*/);
int tsb_result_counters(tsb_batch* batch, int64_t* counters /*[8][n_inst]*/);
/* Waveform of one instance, row-major [rows][n_columns]; returns the row count in *n_rows. */
int tsb_result_waveform(tsb_batch* batch, int64_t inst, double* out, int64_t cap_rows, int64_t* n_rows);
/* Whole wave / stats arrays in the device layout above. */
int tsb_result_wave_all(tsb_batch* batch, double* out, int64_t n_doubles);
int tsb_result_stats_all(tsb_batch* batch, double* out /*[4][n_columns][n_inst]*/);
/* Measurements of the last run (TSB_OUT_MEAS): out[0][m][inst] = value, out[1][m][inst] = abscissa, for the table the run
 * used.  TSB_E_INVALID after a run without measurements. */
int tsb_result_measures(tsb_batch* batch, double* out /*[2][n_meas][n_inst]*/);
/* Batch totals computed on the GPU: sum over instances of accepted steps, rejected steps, transient solves,
 * OP solves (reference-equivalent counts) and executed factor+solve passes. */
int tsb_result_totals(tsb_batch* batch, int64_t totals[5]);

/* Asynchronous read-back of the last run's per-instance results into caller-owned PINNED host buffers (NULL = not
 * wanted): stats [4][n_columns][n_inst], rows [n_inst], status [n_inst], counters [8][n_inst].  The copies run on a copy
 * stream of the context behind the run and overlap whatever is launched next (another batch's run); the buffers are
 * complete after tsb_batch_sync(batch).  A later run on the SAME batch waits for them before overwriting the results. */
int tsb_result_fetch_async(tsb_batch* batch, double* stats, int64_t* rows, int32_t* status, int64_t* counters);
/* Batch summary reduced ON THE DEVICE: out[3][n_columns] = per column the minimum, maximum and sum over all instances and
 * stored rows (NaN samples ignored); *rows_total = stored rows of the whole batch (mean = sum / rows_total).  A few KB
 * cross the bus instead of 32 * n_columns bytes per instance.  Needs TSB_OUT_STATS in the last run. */
int tsb_result_summary(tsb_batch* batch, double* out, int64_t* rows_total);

/* ---- job: one sweep over several GPUs of one box, from ONE host process ------------------------------------------------
 * (SURVEY §8(b): `tsb_ctx_create(const int* gpu_ids, int n, ...)`; §8(e).)  A job owns a context + plan + batch per GPU
 * and splits the instance range contiguously: shard g = instances [g*N/G, (g+1)*N/G).  No exchange between GPUs during a
 * run; every call fans out to the shards from one host thread per GPU.  Parameter arrays and per-instance results are in
 * JOB order (length n_inst); summaries are reduced on each device first.  gpu_ids may repeat a device (several contexts
 * on one GPU).  Replaces, for the sweep, what a Go host would do with one analysis.Analysis per goroutine. */
int tsb_job_create(const int* gpu_ids, int n_gpus, const char* netlist_text, int64_t n_inst, tsb_job** out);
void tsb_job_destroy(tsb_job* job);
const char* tsb_job_error(tsb_job* job);
int tsb_job_num_shards(const tsb_job* job);
int tsb_job_shard(const tsb_job* job, int g, tsb_batch** batch, int64_t* lo, int64_t* hi);   /* borrowed handle of shard g */
tsb_plan* tsb_job_plan(const tsb_job* job);                                                  /* structure / column queries */
int tsb_job_set_param(tsb_job* job, int dev, int param, const double* values /*[n_inst], host*/);
int tsb_job_set_param_uniform(tsb_job* job, int dev, int param, double value);
int tsb_job_run_op(tsb_job* job, const tsb_opts* opts);
int tsb_job_run_tran(tsb_job* job, double tstart, double tstop, double tstep, double tmax, int uic, int out_flags,
                     int64_t wave_cap_rows, const tsb_opts* opts);
int tsb_job_run_dc(tsb_job* job, int src_dev, double start, double stop, double inc, int out_flags, const tsb_opts* opts);
int tsb_job_sync(tsb_job* job);
int tsb_job_result_status(tsb_job* job, int32_t* status /*[n_inst]*/);
int tsb_job_result_rows(tsb_job* job, int64_t* rows /*[n_inst]*/);
int tsb_job_result_stats(tsb_job* job, double* stats /*[4][n_columns][n_inst]*/);
int tsb_job_set_measures(tsb_job* job, const tsb_meas* m, int n_meas);
int tsb_job_result_measures(tsb_job* job, double* out /*[2][n_meas][n_inst], JOB order*/);
int tsb_job_result_waveform(tsb_job* job, int64_t inst, double* out, int64_t cap_rows, int64_t* n_rows);
/* out[3][n_columns] (min, max, sum), stored rows and the five totals of tsb_result_totals, merged over the GPUs. */
int tsb_job_result_summary(tsb_job* job, double* out, int64_t* rows_total, int64_t totals[5]);

/* ---- operator level: batched factor + solve -------------------------------------------------------
 * Drop-in for the reference's matrix OPERATOR (pkg/matrix/circuit.go:126-150 Solve() = sparse Factor + Solve, fed by
 * AddElement / AddRHS, matrix/device.go:3-8) for hosts that stamp themselves: n_inst systems A x = b of one order
 * n <= 32 that share one pivot order.  One circuit per 4 / 8 / 16 lanes of a warp (2 or 3 rows per lane), matrix in registers,
 * pivot-row broadcast by warp shuffles (csrc/lu_warp.cu).  Layout: instance-major, A[inst][row][col] row-major
 * (0-based), b[inst][row], x[inst][col]; status[inst] = 0, or 1 for a zero pivot ("matrix factorization failed").
 * pivot_row[k] / pivot_col[k] (k = 0..n-1): 1-based external row / column eliminated at step k+1.
 * strict_fp = 1 reproduces Sparse 1.3's rounding (no FMA contraction, IEEE reciprocals, spSolve's summation order; a -0.0
 * entry of A counts as +0.0, as AddElement onto a cleared element makes it).
 * x of a status-1 system is unspecified (the reference leaves no solution).  Non-finite data is data: an infinite pivot has
 * the reciprocal 0 in both builds (x of its column = 0).  The fast build's reciprocals come from a flush-to-zero seed:
 * subnormal pivots and pivots above 2^1022 in magnitude lose accuracy there (the strict build divides).
 * Refusals, before anything is launched or written: n outside 1..32 (TSB_E_INVALID; tsb_lu_solve_batched_dev:
 * TSB_E_UNSUPPORTED), a pivot order that is not a permutation of 1..n (TSB_E_INVALID).  n_inst = 0 is a no-op (TSB_OK). */
/* The reference's symbolic pass on a nominal matrix: the order its first Factor() picks (Markowitz products over the
 * structurally dense matrix, relative threshold 1e-3, diagonal preference; SURVEY Appendix C), Translate numbering =
 * row-major first touch.  Host only (ctx not needed). */
int tsb_lu_order(int n, const double* A_nominal, int* pivot_row, int* pivot_col);
/* The device-stamp kernel on its own (pkg/device Stamp of every device of every instance, circuit.go:165-176): the
 * dense system after mat.Clear(); ckt.Stamp(status); mat.LoadGmin(gmin) on a freshly set-up circuit, status =
 * {Mode = mode (TSB_AN_OP or TSB_AN_TRAN), Time = time, TimeStep = dt, Gmin = gmin}, written to device memory as
 * A[inst][n][n] (row-major) and b[inst][n], 0-based = MNA index - 1.  With tsb_lu_solve_batched_dev and the plan's
 * own pivot order (tsb_plan_structure) it forms the two-kernel version of one Newton iteration.  Asynchronous. */
int tsb_batch_stamp_dev(tsb_batch* batch, int mode, double time, double dt, double gmin, uint64_t A_dev, uint64_t b_dev,
                        const tsb_opts* opts);
int tsb_lu_solve_batched(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, const double* A, const double* b,
                         double* x, int32_t* status, int64_t n_inst, int strict_fp);
/* Same with every array already in HBM (device pointers); asynchronous on the context's stream. */
int tsb_lu_solve_batched_dev(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, uint64_t A_dev, uint64_t b_dev,
                             uint64_t x_dev, uint64_t status_dev, int64_t n_inst, int strict_fp);
/* Complex systems: the reference's FactorComplex + SolveComplex (pkg/matrix/circuit.go:130, 140), i.e. one AC frequency
 * point of a host that stamps itself, over a batch.  Layout: interleaved complex, A[inst][row][col][re, im],
 * b[inst][row][re, im], x[inst][col][re, im] — the layout of C99 double _Complex, std::complex<double>, Go's complex128 and
 * torch.complex128 (x is the solution vector itself, not the analysis read-out of tsb_run_ac).  The pivot order, n, status
 * and the refusals are those of tsb_lu_solve_batched.  In the reference the AC order is the one its real operating point
 * froze (ac.go:33-49): take it from tsb_lu_order on the REAL nominal matrix (e.g. the conductance part G), or from
 * tsb_plan_structure; no order is chosen on complex values.  A pivot is zero when |re| + |im| == 0 (status 1; x of that
 * system is unspecified).
 * strict_fp = 1 reproduces Sparse 1.3's complex arithmetic bit for bit: CMPLX_RECIPROCAL as Smith's scaled division with its
 * branch predicates, CMPLX_MULT / CMPLX_MULT_SUBT_ASSIGN without contraction, forward substitution skipped when both parts
 * of an entry are zero, back substitution by ascending columns, -0.0 in either part of an entry of A counted as +0.0.
 * The fast build contracts to FMA, forms multipliers, and takes the two real quotients of Smith's form from the fast
 * reciprocal (subnormal and huge parts are limited as for the real fast build).  A pivot with one infinite and one finite
 * part has the reciprocal 0 in both builds (x of its column = 0).  Pointers need 8-byte alignment only. */
int tsb_lu_solve_batched_complex(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, const double* A,
                                 const double* b, double* x, int32_t* status, int64_t n_inst, int strict_fp);
/* Same with every array already in HBM (device pointers); asynchronous on the context's stream. */
int tsb_lu_solve_batched_complex_dev(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, uint64_t A_dev,
                                     uint64_t b_dev, uint64_t x_dev, uint64_t status_dev, int64_t n_inst, int strict_fp);

/* ---- introspection / build-time support -------------------------------------------------------*/
/* CUDA source of the kernels specialised for this batch configuration (which parameters vary). */
int tsb_batch_kernel_source(tsb_batch* batch, const tsb_opts* opts, char* buf, int64_t cap, int64_t* needed);
/* Which specialisation the two calls below describe: dc_src_dev >= 0 selects the DC-sweep kernel for that source
 * (dc_src2_dev >= 0: the nested sweep), grid != 0 the TSB_OUT_GRID kernels; (-1, -1, 0) = the default OP / transient
 * kernels.  The bit TSB_OUT_MEAS in `grid` selects the kernels of the batch's measurement table instead (grid ==
 * TSB_OUT_MEAS) or in addition (grid == TSB_OUT_GRID | TSB_OUT_MEAS).  A batch used this way is for introspection only (build step), do not run analyses on it. */
int tsb_batch_kernel_variant(tsb_batch* batch, int dc_src_dev, int dc_src2_dev, int grid);
/* Cache key (hex) of that source + compile options; the cubin is looked up as <cache_dir>/<key>.cubin. */
int tsb_batch_kernel_key(tsb_batch* batch, const tsb_opts* opts, char* buf, int cap);
/* Number of kernels launched by this context so far (bench.py's gpu_launches). */
int64_t tsb_ctx_launch_count(const tsb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* TSPICE_B200_H */
