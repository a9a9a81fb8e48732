// job.cpp — one sweep over several GPUs of one box, driven from ONE host process (include/tspice_b200.h, tsb_job_*).
//
// The reference is single-threaded Go; a Go host that adopts the batched engine is still one process.  A job owns one
// context + plan + batch per GPU, splits the instance range contiguously ([g*N/G, (g+1)*N/G), SURVEY §8(e)), launches
// every shard from a host thread of its own (so the first-call work of each context — kernel load, launch-bounds timing —
// overlaps too) and merges results: per-instance reads are routed to the owning GPU, batch summaries are reduced on each
// device to a few KB before they cross the bus.  There is no exchange between the GPUs during a run: instances are
// independent.  Built on the public C ABI only.
#include <cmath>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#include "../../include/tspice_b200.h"

struct tsb_job {
    struct Shard {
        tsb_ctx* ctx = nullptr;
        tsb_plan* plan = nullptr;
        tsb_batch* batch = nullptr;
        int64_t lo = 0, hi = 0;       // instances [lo, hi) of the job
    };
    std::vector<Shard> shards;
    int64_t n_inst = 0;
    int n_meas = 0;                   // measurement table of every shard (tsb_job_set_measures)
    int four_rows = 0;                // output rows of the Fourier table of every shard (tsb_job_set_fourier)
    std::string err;
};

namespace {
int job_fail(tsb_job* j, int code, const std::string& msg) { if (j) j->err = msg; return code; }

template <class F> int for_all_shards(tsb_job* j, F f) {
    std::vector<int> rc(j->shards.size(), TSB_OK);
    std::vector<std::thread> th;
    for (size_t g = 0; g < j->shards.size(); ++g) th.emplace_back([&, g] { rc[g] = f(j->shards[g]); });
    for (auto& t : th) t.join();
    for (size_t g = 0; g < rc.size(); ++g)
        if (rc[g] != TSB_OK) return job_fail(j, rc[g], std::string("GPU shard ") + std::to_string(g) + ": " + tsb_last_error(j->shards[g].ctx));
    return TSB_OK;
}
tsb_job::Shard* owner(tsb_job* j, int64_t inst) {
    for (auto& s : j->shards) if (inst >= s.lo && inst < s.hi) return &s;
    return nullptr;
}
}  // namespace

extern "C" {

int tsb_job_create(const int* gpu_ids, int n_gpus, const char* netlist_text, int64_t n_inst, tsb_job** out) {
    if (!out || !gpu_ids || n_gpus < 1 || !netlist_text || n_inst < n_gpus) return TSB_E_INVALID;
    *out = nullptr;
    tsb_job* j = new tsb_job;
    j->n_inst = n_inst;
    for (int g = 0; g < n_gpus; ++g) {
        tsb_job::Shard s;
        s.lo = n_inst * g / n_gpus; s.hi = n_inst * (g + 1) / n_gpus;
        int rc = tsb_ctx_create(gpu_ids[g], &s.ctx);
        if (rc == TSB_OK) rc = tsb_plan_from_netlist(s.ctx, netlist_text, &s.plan);
        if (rc == TSB_OK) rc = tsb_batch_create(s.plan, s.hi - s.lo, &s.batch);
        j->shards.push_back(s);
        if (rc != TSB_OK) { tsb_job_destroy(j); return rc; }
    }
    *out = j;
    return TSB_OK;
}
void tsb_job_destroy(tsb_job* j) {
    if (!j) return;
    for (auto& s : j->shards) {
        if (s.batch) tsb_batch_destroy(s.batch);
        if (s.plan) tsb_plan_destroy(s.plan);
        if (s.ctx) tsb_ctx_destroy(s.ctx);
    }
    delete j;
}
const char* tsb_job_error(tsb_job* j) { return j ? j->err.c_str() : ""; }
int tsb_job_num_shards(const tsb_job* j) { return j ? (int)j->shards.size() : TSB_E_INVALID; }
int tsb_job_shard(const tsb_job* j, int g, tsb_batch** batch, int64_t* lo, int64_t* hi) {
    if (!j || g < 0 || g >= (int)j->shards.size()) return TSB_E_INVALID;
    if (batch) *batch = j->shards[g].batch;
    if (lo) *lo = j->shards[g].lo;
    if (hi) *hi = j->shards[g].hi;
    return TSB_OK;
}
tsb_plan* tsb_job_plan(const tsb_job* j) { return j && !j->shards.empty() ? j->shards[0].plan : nullptr; }

int tsb_job_set_param(tsb_job* j, int dev, int param, const double* values) {
    if (!j || !values) return TSB_E_INVALID;
    for (auto& s : j->shards) {
        int rc = tsb_batch_set_param(s.batch, dev, param, values + s.lo);
        if (rc != TSB_OK) return job_fail(j, rc, tsb_last_error(s.ctx));
    }
    return TSB_OK;
}
int tsb_job_set_param_uniform(tsb_job* j, int dev, int param, double value) {
    if (!j) return TSB_E_INVALID;
    for (auto& s : j->shards) {
        int rc = tsb_batch_set_param_uniform(s.batch, dev, param, value);
        if (rc != TSB_OK) return job_fail(j, rc, tsb_last_error(s.ctx));
    }
    return TSB_OK;
}

int tsb_job_run_op(tsb_job* j, const tsb_opts* opts) {
    if (!j) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) { return tsb_run_op(s.batch, opts); });
}
int tsb_job_run_tran(tsb_job* j, double tstart, double tstop, double tstep, double tmax, int uic, int out_flags, int64_t wave_cap_rows,
                     const tsb_opts* opts) {
    if (!j) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) { return tsb_run_tran(s.batch, tstart, tstop, tstep, tmax, uic, out_flags, wave_cap_rows, opts); });
}
int tsb_job_run_dc(tsb_job* j, int src_dev, double start, double stop, double inc, int out_flags, const tsb_opts* opts) {
    if (!j) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) { return tsb_run_dc(s.batch, src_dev, start, stop, inc, out_flags, opts); });
}
int tsb_job_sync(tsb_job* j) {
    if (!j) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) { return tsb_batch_sync(s.batch); });
}

// Per-instance results in JOB order: each shard copies into its slice of the caller's arrays.
int tsb_job_result_status(tsb_job* j, int32_t* status) {
    if (!j || !status) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) { return tsb_result_status(s.batch, status + s.lo); });
}
int tsb_job_result_rows(tsb_job* j, int64_t* rows) {
    if (!j || !rows) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) { return tsb_result_rows(s.batch, rows + s.lo); });
}
// stats [4][n_columns][n_inst] in job order (each shard's block is copied column by column into place)
int tsb_job_result_stats(tsb_job* j, double* stats) {
    if (!j || !stats) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) {
        int64_t n = 0; int ncol = 0;
        int rc = tsb_result_dims(s.batch, &n, &ncol, nullptr);
        if (rc != TSB_OK) return rc;
        std::vector<double> tmp((size_t)4 * ncol * n);
        rc = tsb_result_stats_all(s.batch, tmp.data());
        if (rc != TSB_OK) return rc;
        for (int k = 0; k < 4 * ncol; ++k) std::memcpy(stats + (size_t)k * j->n_inst + s.lo, tmp.data() + (size_t)k * n, (size_t)n * sizeof(double));
        return (int)TSB_OK;
    });
}
int tsb_job_set_measures(tsb_job* j, const tsb_meas* m, int n_meas) {
    if (!j) return TSB_E_INVALID;
    for (auto& s : j->shards) {
        int rc = tsb_batch_set_measures(s.batch, m, n_meas);
        if (rc != TSB_OK) return job_fail(j, rc, tsb_last_error(s.ctx));
    }
    j->n_meas = n_meas;
    return TSB_OK;
}
// measurements [2][n_meas][n_inst] in job order (each shard's block is copied row by row into place)
int tsb_job_result_measures(tsb_job* j, double* out) {
    if (!j || !out) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) {
        int64_t n = 0;
        int rc = tsb_result_dims(s.batch, &n, nullptr, nullptr);
        if (rc != TSB_OK) return rc;
        const size_t rows = 2 * (size_t)j->n_meas;
        std::vector<double> tmp(rows * n);
        rc = tsb_result_measures(s.batch, tmp.data());
        if (rc != TSB_OK) return rc;
        for (size_t k = 0; k < rows; ++k) std::memcpy(out + k * j->n_inst + s.lo, tmp.data() + k * n, (size_t)n * sizeof(double));
        return (int)TSB_OK;
    });
}
int tsb_job_set_fourier(tsb_job* j, const tsb_four* f, int n) {
    if (!j) return TSB_E_INVALID;
    for (auto& s : j->shards) {
        int rc = tsb_batch_set_fourier(s.batch, f, n);
        if (rc != TSB_OK) return job_fail(j, rc, tsb_last_error(s.ctx));
    }
    j->four_rows = 0;
    for (int k = 0; k < n; ++k) j->four_rows += 1 + 2 * f[k].n_harm;
    return TSB_OK;
}
// Fourier coefficients [sum (1 + 2H)][n_inst] in job order (each shard's block is copied row by row into place)
int tsb_job_result_fourier(tsb_job* j, double* out) {
    if (!j || !out) return TSB_E_INVALID;
    return for_all_shards(j, [&](tsb_job::Shard& s) {
        int64_t n = 0;
        int rc = tsb_result_dims(s.batch, &n, nullptr, nullptr);
        if (rc != TSB_OK) return rc;
        const size_t rows = (size_t)j->four_rows;
        std::vector<double> tmp(rows * n);
        rc = tsb_result_fourier(s.batch, tmp.data());
        if (rc != TSB_OK) return rc;
        for (size_t k = 0; k < rows; ++k) std::memcpy(out + k * j->n_inst + s.lo, tmp.data() + k * n, (size_t)n * sizeof(double));
        return (int)TSB_OK;
    });
}
int tsb_job_result_waveform(tsb_job* j, int64_t inst, double* out, int64_t cap_rows, int64_t* n_rows) {
    if (!j) return TSB_E_INVALID;
    tsb_job::Shard* s = owner(j, inst);
    if (!s) return job_fail(j, TSB_E_INVALID, "instance out of range");
    int rc = tsb_result_waveform(s->batch, inst - s->lo, out, cap_rows, n_rows);
    return rc == TSB_OK ? rc : job_fail(j, rc, tsb_last_error(s->ctx));
}
// Job summary: every GPU reduces its shard on the device (tsb_result_summary), the host merges G x 3 x n_columns numbers.
int tsb_job_result_summary(tsb_job* j, double* out /*[3][n_columns]*/, int64_t* rows_total, int64_t totals[5]) {
    if (!j || !out) return TSB_E_INVALID;
    int ncol = 0;
    tsb_result_dims(j->shards[0].batch, nullptr, &ncol, nullptr);
    if (ncol <= 0) return job_fail(j, TSB_E_INVALID, "no run yet");
    const size_t G = j->shards.size();
    std::vector<double> part(G * 3 * ncol);
    std::vector<int64_t> rows(G, 0), tot(G * 5, 0);
    int rc = for_all_shards(j, [&](tsb_job::Shard& s) {
        const size_t g = &s - j->shards.data();
        int r = tsb_result_summary(s.batch, part.data() + g * 3 * ncol, &rows[g]);
        if (r == TSB_OK) r = tsb_result_totals(s.batch, tot.data() + g * 5);
        return r;
    });
    if (rc != TSB_OK) return rc;
    for (int c = 0; c < ncol; ++c) {
        double mn = HUGE_VAL, mx = -HUGE_VAL, sm = 0.0;
        for (size_t g = 0; g < G; ++g) {
            const double* p = part.data() + g * 3 * ncol;
            mn = std::fmin(mn, p[c]); mx = std::fmax(mx, p[ncol + c]); sm += p[2 * ncol + c];
        }
        out[c] = mn; out[ncol + c] = mx; out[2 * ncol + c] = sm;
    }
    if (rows_total) { *rows_total = 0; for (int64_t r : rows) *rows_total += r; }
    if (totals) for (int k = 0; k < 5; ++k) { totals[k] = 0; for (size_t g = 0; g < G; ++g) totals[k] += tot[g * 5 + k]; }
    return TSB_OK;
}

}  // extern "C"
