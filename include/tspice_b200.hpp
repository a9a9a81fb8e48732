// tspice_b200.hpp — C++ host-side mirror of the reference's analysis API over the C ABI (tspice_b200.h).
//
// The reference's host language is Go; where no Go toolchain exists the host side is C++.  The classes keep the
// reference's names, call sequence and error behaviour so that host code ports line by line:
//
//   reference (Go)                                              here (C++)
//   ------------------------------------------------------------------------------------------------------
//   nl, err := netlist.Parse(text)                              tsb::Circuit ckt = tsb::Circuit::FromNetlist(ctx, text);
//   ckt := circuit.NewWithComplex(...); AssignNodeBranchMaps;     (one call: parser.go:75, circuit.go:31-163)
//   CreateMatrix; SetupDevices
//   tr := analysis.NewTransient(tStart,tStop,tStep,tMax,uic)    auto tr = tsb::analysis::NewTransient(tStart,tStop,tStep,tMax,uic);
//   err = tr.Setup(ckt); err = tr.Execute()                     tr.Setup(ckt); tr.Execute();          // throw tsb::Error
//   res := tr.GetResults()   // map[string][]float64            auto res = tr.GetResults();           // std::map<std::string, std::vector<double>>
//
// plus the batch axis the reference does not have: Setup(batch) on a tsb::Batch with per-instance parameters,
// GetResults(instance), Status().  Go `error` returns become tsb::Error exceptions carrying the reference's
// message text; Go panics (inconsistent DC sweep lengths, dc.go:21-23) become std::invalid_argument.
// Header-only; link with -ltspice_b200.
#pragma once
#include <complex>
#include <cstdint>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>
#include "tspice_b200.h"

namespace tsb {

struct Error : std::runtime_error { using std::runtime_error::runtime_error; };

class Context {
public:
    explicit Context(int device = 0) {
        if (tsb_ctx_create(device, &h_) != TSB_OK) throw Error(std::string("tsb_ctx_create: ") + tsb_last_error(nullptr));
    }
    ~Context() { tsb_ctx_destroy(h_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    tsb_ctx* get() const { return h_; }
    std::string last_error() const { return tsb_last_error(h_); }
private:
    tsb_ctx* h_ = nullptr;
};

class Circuit {
public:
    static Circuit FromNetlist(Context& ctx, const std::string& text) {
        tsb_plan* p = nullptr;
        if (tsb_plan_from_netlist(ctx.get(), text.c_str(), &p) != TSB_OK) throw Error("Error parsing netlist: " + ctx.last_error());
        return Circuit(ctx, p);
    }
    Circuit(Circuit&& o) noexcept : ctx_(o.ctx_), h_(o.h_) { o.h_ = nullptr; }
    Circuit(const Circuit&) = delete;
    ~Circuit() { if (h_) tsb_plan_destroy(h_); }
    tsb_plan* get() const { return h_; }
    Context& ctx() const { return *ctx_; }
    int FindDevice(const std::string& name) const { return tsb_plan_find_device(h_, name.c_str()); }
    std::vector<std::string> Columns(int analysis) const {
        std::vector<std::string> out;
        char buf[128];
        for (int k = 0, n = tsb_plan_num_columns(h_, analysis); k < n; ++k) { tsb_plan_column_name(h_, analysis, k, buf, sizeof buf); out.push_back(buf); }
        return out;
    }
    void Card(int& analysis, double tran[4], int& uic, int& dc_src, double dc[3]) const { tsb_plan_analysis(h_, &analysis, tran, &uic, &dc_src, dc); }
private:
    Circuit(Context& ctx, tsb_plan* p) : ctx_(&ctx), h_(p) {}
    Context* ctx_;
    tsb_plan* h_;
};

class Batch {
public:
    Batch(Circuit& ckt, int64_t n) : ckt_(&ckt), n_(n) {
        if (tsb_batch_create(ckt.get(), n, &h_) != TSB_OK) throw Error("tsb_batch_create failed: " + ckt.ctx().last_error());
    }
    ~Batch() { if (h_) tsb_batch_destroy(h_); }
    Batch(const Batch&) = delete;
    void SetParam(const std::string& device, int param, const std::vector<double>& values) {
        int d = ckt_->FindDevice(device);
        if (d < 0) throw Error("device " + device + " not found");
        if ((int64_t)values.size() != n_) throw std::invalid_argument("values must have one entry per instance");
        if (tsb_batch_set_param(h_, d, param, values.data()) != TSB_OK) throw Error(ckt_->ctx().last_error());
    }
    // Measurement table (TSB_OUT_MEAS; definitions in tspice_b200.h); an empty vector clears it.
    void SetMeasures(const std::vector<tsb_meas>& m) {
        if (tsb_batch_set_measures(h_, m.empty() ? nullptr : m.data(), (int)m.size()) != TSB_OK) throw Error(ckt_->ctx().last_error());
        n_meas_ = (int)m.size();
    }
    // [2: value, abscissa][n_meas][n_inst] of the last run with TSB_OUT_MEAS.
    std::vector<double> Measures() const {
        std::vector<double> out((size_t)2 * n_meas_ * n_);
        if (tsb_result_measures(h_, out.data()) != TSB_OK) throw Error(ckt_->ctx().last_error());
        return out;
    }
    // Fourier table (TSB_OUT_FOUR; definitions in tspice_b200.h); an empty vector clears it.
    void SetFourier(const std::vector<tsb_four>& f) {
        if (tsb_batch_set_fourier(h_, f.empty() ? nullptr : f.data(), (int)f.size()) != TSB_OK) throw Error(ckt_->ctx().last_error());
        four_rows_ = 0;
        for (const tsb_four& e : f) four_rows_ += 1 + 2 * e.n_harm;
    }
    // [sum (1 + 2 n_harm)][n_inst] of the last run with TSB_OUT_FOUR: per entry a0, A_1, B_1, ..., A_H, B_H.
    std::vector<double> Fourier() const {
        std::vector<double> out((size_t)four_rows_ * n_);
        if (tsb_result_fourier(h_, out.data()) != TSB_OK) throw Error(ckt_->ctx().last_error());
        return out;
    }
    tsb_batch* get() const { return h_; }
    Circuit& circuit() const { return *ckt_; }
    int64_t size() const { return n_; }
private:
    Circuit* ckt_;
    int64_t n_;
    int n_meas_ = 0;
    int four_rows_ = 0;
    tsb_batch* h_ = nullptr;
};

namespace analysis {

using Results = std::map<std::string, std::vector<double>>;

// analysis.Analysis (pkg/analysis/anlysis.go:18-22)
class Analysis {
public:
    virtual ~Analysis() = default;
    void Setup(Circuit& ckt) { own_.reset(new Batch(ckt, 1)); batch_ = own_.get(); }     // nominal values, batch of one
    void Setup(Batch& batch) { own_.reset(); batch_ = &batch; }
    virtual void Execute() = 0;
    Results GetResults(int64_t inst = 0) const {
        require();
        int64_t n = 0, cap = 0; int ncol = 0;
        tsb_result_dims(batch_->get(), &n, &ncol, &cap);
        std::vector<double> w((size_t)(cap > 0 ? cap : 1) * ncol);
        int64_t rows = 0;
        if (tsb_result_waveform(batch_->get(), inst, w.data(), cap, &rows) != TSB_OK) throw Error(batch_->circuit().ctx().last_error());
        Results out;
        std::vector<std::string> names = batch_->circuit().Columns(kind());
        for (int k = 0; k < ncol; ++k) {
            std::vector<double>& col = out[names[k]];
            for (int64_t r = 0; r < rows; ++r) col.push_back(w[(size_t)r * ncol + k]);
        }
        return out;
    }
    std::vector<int32_t> Status() const {
        require();
        std::vector<int32_t> st((size_t)batch_->size());
        tsb_result_status(batch_->get(), st.data());
        return st;
    }
    tsb_opts opts;
protected:
    Analysis() { tsb_default_opts(&opts); }
    virtual int kind() const = 0;
    void require() const { if (!batch_) throw Error("circuit not set"); }              // tran.go:78-80
    void check(int rc) const { if (rc != TSB_OK) throw Error(batch_->circuit().ctx().last_error()); }
    // The reference's Execute() returns the solver error of its single circuit; for a batch of one do the same.
    void raise_single_instance_failure(const char* what) const {
        if (batch_->size() != 1) return;
        int32_t st = 0; tsb_result_status(batch_->get(), &st);
        if (st == TSB_ST_OP_FAILED) throw Error("operating point analysis error: final solution failed");       // op.go:228
        if (st == TSB_ST_TRAN_FAILED || st == TSB_ST_DC_FAILED) throw Error(std::string(what));
    }
    Batch* batch_ = nullptr;
    std::unique_ptr<Batch> own_;
};

class OperatingPoint : public Analysis {
public:
    void Execute() override { require(); check(tsb_run_op(batch_->get(), &opts)); check(tsb_batch_sync(batch_->get())); raise_single_instance_failure("failed to converge"); }
protected:
    int kind() const override { return TSB_AN_OP; }
};

class Transient : public Analysis {
public:
    Transient(double tStart, double tStop, double tStep, double tMax, bool uic)
        : tStart_(tStart), tStop_(tStop), tStep_(tStep), tMax_(tMax), uic_(uic) {}
    int out = TSB_OUT_WAVE;      // TSB_OUT_WAVE | TSB_OUT_STATS | TSB_OUT_GRID (results resampled onto a fixed time grid) | TSB_OUT_MEAS | TSB_OUT_FOUR
    int64_t cap_rows = 16384;
    double grid_dt = 0.0;        // TSB_OUT_GRID: grid spacing (0: the clamped tStep)
    void Execute() override {
        require();
        if (out & TSB_OUT_GRID) opts.grid_dt = grid_dt;
        check(tsb_run_tran(batch_->get(), tStart_, tStop_, tStep_, tMax_, uic_ ? 1 : 0, out, cap_rows, &opts));
        check(tsb_batch_sync(batch_->get()));
        raise_single_instance_failure("failed to converge at t");                      // tran.go:119
    }
protected:
    int kind() const override { return TSB_AN_TRAN; }
private:
    double tStart_, tStop_, tStep_, tMax_;
    bool uic_;
};

class DCSweep : public Analysis {
public:
    DCSweep(std::vector<std::string> sources, std::vector<double> starts, std::vector<double> stops, std::vector<double> incs)
        : src_(std::move(sources)), start_(std::move(starts)), stop_(std::move(stops)), inc_(std::move(incs)) {
        if (src_.size() != start_.size() || src_.size() != stop_.size() || src_.size() != inc_.size())
            throw std::invalid_argument("inconsistent parameter lengths");               // dc.go:21-23 (panic)
    }
    int out = TSB_OUT_WAVE;
    void Execute() override {
        require();
        if (src_.size() != 1) throw Error("unsupported number of sweep sources: " + std::to_string(src_.size()));   // dc.go:86
        int d = batch_->circuit().FindDevice(src_[0]);
        if (d < 0) throw Error("source " + src_[0] + " not found");                      // dc.go:64-66
        check(tsb_run_dc(batch_->get(), d, start_[0], stop_[0], inc_[0], out, &opts));
        check(tsb_batch_sync(batch_->get()));
        raise_single_instance_failure("convergence error");
    }
protected:
    int kind() const override { return TSB_AN_DC; }
private:
    std::vector<std::string> src_;
    std::vector<double> start_, stop_, inc_;
};

inline OperatingPoint NewOP() { return OperatingPoint(); }
inline Transient NewTransient(double tStart, double tStop, double tStep, double tMax, bool uic) { return Transient(tStart, tStop, tStep, tMax, uic); }
inline DCSweep NewDCSweep(std::vector<std::string> s, std::vector<double> a, std::vector<double> b, std::vector<double> c) {
    return DCSweep(std::move(s), std::move(a), std::move(b), std::move(c));
}

}  // namespace analysis

// Operator level (pkg/matrix: Clear / AddElement / AddRHS / Solve over a batch of stamped systems).
struct PivotOrder { std::vector<int> row, col; };
inline PivotOrder LuOrder(int n, const std::vector<double>& A_nominal) {
    if ((int)A_nominal.size() != n * n) throw std::invalid_argument("A_nominal must be n*n");
    PivotOrder o; o.row.resize(n); o.col.resize(n);
    if (tsb_lu_order(n, A_nominal.data(), o.row.data(), o.col.data()) != TSB_OK) throw Error("matrix factorization failed (nominal matrix is singular)");
    return o;
}
// A: [n_inst][n][n] row-major, b: [n_inst][n]; returns x [n_inst][n]; status[inst] = 1 marks a zero pivot.
inline std::vector<double> LuSolveBatched(Context& ctx, int n, const PivotOrder& o, const std::vector<double>& A,
                                          const std::vector<double>& b, std::vector<int32_t>& status, bool strict = false) {
    const int64_t n_inst = (int64_t)b.size() / n;
    if ((int64_t)A.size() != n_inst * n * n) throw std::invalid_argument("A must be n_inst*n*n");
    std::vector<double> x((size_t)n_inst * n);
    status.assign((size_t)n_inst, 0);
    if (tsb_lu_solve_batched(ctx.get(), n, o.row.data(), o.col.data(), A.data(), b.data(), x.data(), status.data(), n_inst, strict ? 1 : 0) != TSB_OK)
        throw Error(ctx.last_error());
    return x;
}
// Complex systems (FactorComplex + SolveComplex): A [n_inst][n][n], b [n_inst][n] as std::complex<double> (interleaved re, im);
// returns x [n_inst][n].  The order is the real one: LuOrder on the real nominal matrix, or the plan's.
inline std::vector<std::complex<double>> LuSolveBatchedComplex(Context& ctx, int n, const PivotOrder& o,
                                                               const std::vector<std::complex<double>>& A,
                                                               const std::vector<std::complex<double>>& b,
                                                               std::vector<int32_t>& status, bool strict = false) {
    const int64_t n_inst = (int64_t)b.size() / n;
    if ((int64_t)A.size() != n_inst * n * n) throw std::invalid_argument("A must be n_inst*n*n");
    std::vector<std::complex<double>> x((size_t)n_inst * n);
    status.assign((size_t)n_inst, 0);
    if (tsb_lu_solve_batched_complex(ctx.get(), n, o.row.data(), o.col.data(), reinterpret_cast<const double*>(A.data()),
                                     reinterpret_cast<const double*>(b.data()), reinterpret_cast<double*>(x.data()), status.data(),
                                     n_inst, strict ? 1 : 0) != TSB_OK)
        throw Error(ctx.last_error());
    return x;
}

}  // namespace tsb
