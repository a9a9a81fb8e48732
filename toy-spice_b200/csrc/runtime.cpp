// runtime.cpp — the C ABI (include/tspice_b200.h): contexts, plans, batches, runs, results.
//
// GPU plumbing: CUDA runtime API for memory / streams / launches; the netlist-specialised kernels
// are loaded as cubins (cudaLibraryLoadData) either from the in-tree kernel cache (built by
// __graft_entry__.build() with nvcc) or, on a miss, compiled with NVRTC (dlopen'ed lazily, so the
// library loads and exports its symbols on machines without a GPU or without NVRTC).
// There is NO CPU execution path for batches: if CUDA is unavailable every run_* call fails loudly.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <memory>
#include <mutex>
#include <sstream>
#include "tsb_internal.hpp"
#include "hostlu.hpp"

namespace tsb {
cudaError_t launch_fp64_peak(double* scratch, int blocks, int iters, cudaStream_t s);
cudaError_t launch_totals(const long long* counters, long long n_inst, unsigned long long* totals, int sms, cudaStream_t s);
cudaError_t launch_fill_i64(long long* p, long long n, long long v, int sms, cudaStream_t s);
cudaError_t launch_summary(const double* stats, long long n_inst, int ncol, double* partial, int blocks_x, cudaStream_t s);
cudaError_t launch_lu_warp(const double* A, const double* b, double* x, int* status, long long n_inst, int n, const int* prow,
                           const int* pcol, int strict, int sms, cudaStream_t s);
cudaError_t launch_clu_warp(const double* A, const double* b, double* x, int* status, long long n_inst, int n, const int* prow,
                            const int* pcol, int strict, int sms, cudaStream_t s);
}

using namespace tsb;

// Mirror of the device-side TsbArgs (device/skeleton.cuh) — keep in sync.
#define TSB_MAX_VARYING 128
struct TsbArgsHost {
    long long n_inst;
    const double* pv[TSB_MAX_VARYING];
    const double* U;
    int analysis;
    int uic;
    double tstart, tstop, tstep, maxstep, minstep;
    int max_iter;
    double abstol, reltol, trtol;
    int out_flags;
    long long cap_rows;
    double* wave;
    double* stats;
    long long* rows;
    int* status;
    long long* counters;
    double* scratch;
    const double* sweep;
    int n_sweep;
    int skip_linear_resolve;
    unsigned long long* work_counter;
    long long first_free;
    double grid_dt;
    int n_grid;
    long long n_run;
    const long long* order;
    const double* sweep2;
    double* tgrid;
    unsigned long long* tgrid_pub;
    int tgrid_cap;
    int tgrid_role;
    double Uc[32];
    double* coop_state;
    double meas_level[16], meas_from[16], meas_to[16];
    int meas_count[16], meas_edge[16];
    double* meas_out;
    double four_s[8], four_dt[8];
    int four_g[8], four_tw_off[8];
    const double* four_tw;
    double* four_out;
};
static_assert(sizeof(TsbArgsHost) <= 4096, "the kernel argument block must stay within the 4 KB kernel-parameter limit");

struct KernelModule {
    cudaLibrary_t lib = nullptr;
    cudaKernel_t optran = nullptr, dc = nullptr, stamp = nullptr, stamp_staged = nullptr, ac = nullptr, coop = nullptr;
    int info_regs = -1, info_spill = -1, min_blocks = 0;
};

struct tsb_ctx {
    int device = 0;
    int sms = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_stream = nullptr;                // tsb_result_fetch_async: device -> host copies beside the next launches
    cudaStream_t upload_stream = nullptr;              // tsb_batch_set_param*: host -> device copies beside another batch's running launch
    cudaStream_t pilot_stream = nullptr;               // shared time grid: the pilot launch runs beside the main one
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::string err;
    std::string cache_dir;
    std::map<std::string, KernelModule> modules;      // key -> loaded module
    std::map<std::string, int> auto_choice;            // key of the min_blocks=auto source -> chosen min blocks
    std::map<std::string, int> tuned;                  // ... -> choice confirmed by timing (autotune_min_blocks)
    int64_t launches = 0;
    // Lifetime: plans hold a reference to their context, batches to their plan, so the destroy calls may come in any
    // order (a garbage-collected host language releases them in no particular one): an object is torn down when its
    // owner has destroyed it AND nothing refers to it any more.
    std::atomic<int> refs{1};
    bool guard = false;                                // $TSB_GUARD=1: result buffers carry guard bands checked at every sync
    long long choice_epoch = 0;                        // bumped whenever auto_choice changes (invalidates batch memos)
    std::string tuned_suffix = ".tuned";               // ".<gpu name>-<SMs>sm.tuned": a timed choice holds for one GPU model only
};

struct tsb_plan {
    Plan p;
    tsb_ctx* ctx = nullptr;
    std::string err;
    std::atomic<int> refs{1};
};

struct tsb_batch {
    tsb_plan* plan = nullptr;
    tsb_ctx* ctx = nullptr;
    int64_t n_inst = 0;
    std::vector<double> uniform;                       // flat parameter space
    std::vector<char> varying;
    std::vector<int> var_slot;
    std::vector<double*> slot_ptr;                     // device pointer per slot
    std::vector<char> slot_owned;
    std::vector<double*> slot_stage;                   // per slot: library-owned pinned staging buffer of tsb_batch_set_param
    std::vector<cudaEvent_t> slot_staged;              //           and the event that marks its H2D copy as done
    double* d_uniform = nullptr;
    // results of the last run
    int analysis = -1, ncol = 0, out_flags = 0;
    int64_t cap_rows = 0;
    double *d_wave = nullptr, *d_stats = nullptr, *d_scratch = nullptr, *d_sweep = nullptr;
    long long *d_rows = nullptr, *d_counters = nullptr;
    int* d_status = nullptr;
    unsigned long long* d_totals = nullptr;
    unsigned long long* d_work = nullptr;              // lane-refill work counter
    bool grid_kernel = false;                          // the next module request wants the TSB_OUT_GRID specialisation
    bool dc_nested = false;                            // ... the nested-sweep specialisation of tsb_dc (rows carry SWEEP1 and SWEEP2)
    int dc_param2 = -1;                                //     and the inner source's parameter
    double* d_sweep2 = nullptr;
    int intro_dc_param = -1;                           // tsb_batch_kernel_variant: what kernel_source / kernel_key describe
    double* d_tgrid = nullptr;                         // shared time grid of the last transient run (skeleton.cuh)
    unsigned long long* d_tgrid_pub = nullptr;
    int tgrid_cap = 0, tgrid_nd = 0;
    int tgrid_used = 0;                                // the last transient run had a pilot
    std::string tgrid_sig;                             // what the table on the device was built for (analysis + uniform values)
    cudaEvent_t ev_run = nullptr, ev_fetch = nullptr;  // tsb_result_fetch_async: run finished / copies finished
    // Parameter uploads run on the context's upload stream: behind this batch's own last launch (ev_launched, recorded on the
    // launch stream after every launch of this batch) and ahead of its next one (ev_params, waited for in fill_common) — but
    // beside whatever ANOTHER batch is running, so a host that alternates two batches uploads step i + 1 during step i.
    cudaEvent_t ev_launched = nullptr, ev_params = nullptr;
    bool params_pending = false;
    bool fetch_pending = false;
    double* d_partial = nullptr;                       // tsb_result_summary: per-block partial results
    std::map<void*, size_t> guarded;                   // TSB_GUARD: user pointer -> payload bytes of every guarded buffer
    // memo of the last module request: generating the kernel source to derive its cache key costs ~0.3 ms of host
    // time, which is the length of a short launch (the stamp kernel); identical requests skip it
    std::string memo_sig, memo_autokey;
    KernelModule* memo_module = nullptr;
    long long* d_order = nullptr;                      // tsb_batch_set_order: processing order (device copy)
    double* d_coop_state = nullptr;                    // cooperative mapping: hand-over of the operating point, [n_state + n + 1][n_inst]
    size_t wave_bytes = 0, stats_bytes = 0;
    std::vector<tsb_meas> meas;                        // tsb_batch_set_measures
    bool meas_kernel = false;                          // the next module request wants the kernels of this table (TSB_MEAS)
    double* d_meas = nullptr;                          // [2][n_meas][n_inst] of the last TSB_OUT_MEAS run
    size_t meas_bytes = 0;
    int meas_last = 0;                                 // measurements the last run produced (0: it had no TSB_OUT_MEAS)
    std::vector<tsb_four> four;                        // tsb_batch_set_fourier
    std::vector<double> four_tw;                       // its twiddles, per entry cos[G] then sin[G] (host libm)
    bool four_tw_sent = false;                         // d_four_tw holds four_tw
    bool four_kernel = false;                          // the next module request wants the kernels of this table (TSB_FOUR)
    double* d_four = nullptr;                          // [sum (1 + 2H)][n_inst] of the last TSB_OUT_FOUR run
    double* d_four_tw = nullptr;
    size_t four_bytes = 0;
    int four_last = 0;                                 // Fourier entries the last run produced (0: it had no TSB_OUT_FOUR)
    int four_rows = 0;                                 // their output rows, sum (1 + 2H)
};

namespace {

std::string g_global_err;

int fail(tsb_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg; else g_global_err = msg;
    return code;
}
#define CU(ctx, call)                                                                              \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) return fail(ctx, TSB_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    } while (0)

std::string lib_dir() {
    Dl_info info;
    if (dladdr((void*)&lib_dir, &info) && info.dli_fname) {
        std::string p = info.dli_fname;
        size_t s = p.rfind('/');
        return s == std::string::npos ? "." : p.substr(0, s);
    }
    return ".";
}

uint64_t fnv1a(const std::string& s, uint64_t h) {
    for (unsigned char c : s) { h ^= c; h *= 1099511628211ULL; }
    return h;
}
std::string source_key(const std::string& src, const std::string& opts) {
    char buf[40];
    uint64_t a = fnv1a(opts, fnv1a(src, 14695981039346656037ULL));
    uint64_t b = fnv1a(src, fnv1a(opts, 0x9e3779b97f4a7c15ULL));
    snprintf(buf, sizeof buf, "%016llx%016llx", (unsigned long long)a, (unsigned long long)b);
    return buf;
}

// ---- NVRTC (lazy) -----------------------------------------------------------------------------
struct Nvrtc {
    void* h = nullptr;
    int (*CreateProgram)(void**, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*CompileProgram)(void*, int, const char* const*) = nullptr;
    int (*GetCUBINSize)(void*, size_t*) = nullptr;
    int (*GetCUBIN)(void*, char*) = nullptr;
    int (*GetProgramLogSize)(void*, size_t*) = nullptr;
    int (*GetProgramLog)(void*, char*) = nullptr;
    int (*DestroyProgram)(void**) = nullptr;
    bool load(std::string& err) {
        if (h) return true;
        // Absolute toolkit paths FIRST: inside a PyTorch process the bare soname resolves to torch's
        // bundled NVRTC 12.8, whose sm_100a code for these kernels measured up to 8x slower than the
        // 12.9 toolkit's (profiles/r01_notes.md).  $TSB_NVRTC overrides.
        const char* env = getenv("TSB_NVRTC");
        const char* names[] = {env && *env ? env : "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12",
                               "/usr/local/cuda/lib64/libnvrtc.so", "libnvrtc.so.12", "libnvrtc.so"};
        for (const char* n : names) { h = dlopen(n, RTLD_NOW | RTLD_LOCAL); if (h) break; }
        if (!h) { err = "NVRTC not found (libnvrtc.so.12) and no cached cubin for this kernel"; return false; }
#define SYM(f) *(void**)(&f) = dlsym(h, "nvrtc" #f); if (!f) { err = "nvrtc" #f " missing"; return false; }
        SYM(CreateProgram) SYM(CompileProgram) SYM(GetCUBINSize) SYM(GetCUBIN) SYM(GetProgramLogSize) SYM(GetProgramLog) SYM(DestroyProgram)
#undef SYM
        return true;
    }
};
Nvrtc g_nvrtc;
std::mutex g_nvrtc_mu;

std::string compile_options_string(const tsb_opts& o) {
    std::string s = "--gpu-architecture=sm_100a --std=c++17 -lineinfo";
    s += o.strict_fp ? " --fmad=false" : " --fmad=true";
    return s;
}

// ptxas -v figures of the transient kernel: what the launch-bounds auto-selection looks at.
struct KernelInfo { int regs = -1, spill_st = -1, spill_ld = -1; };

void parse_ptxas_log(const std::string& log, KernelInfo& info) {
    size_t p = log.find("'tsb_optran'");
    if (p == std::string::npos) return;
    size_t s1 = log.find("bytes spill stores", p);
    size_t u = log.find("Used ", p);
    if (s1 != std::string::npos) {
        size_t c = log.rfind(',', s1);
        if (c != std::string::npos) info.spill_st = atoi(log.c_str() + c + 1);
        size_t c2 = log.find(',', s1);
        if (c2 != std::string::npos) info.spill_ld = atoi(log.c_str() + c2 + 1);
    }
    if (u != std::string::npos) info.regs = atoi(log.c_str() + u + 5);
}

bool nvrtc_compile(const std::string& src, const std::string& name, const tsb_opts& o, std::vector<char>& cubin,
                   KernelInfo& info, std::string& err) {
    std::lock_guard<std::mutex> lk(g_nvrtc_mu);
    if (!g_nvrtc.load(err)) return false;
    void* prog = nullptr;
    if (g_nvrtc.CreateProgram(&prog, src.c_str(), name.c_str(), 0, nullptr, nullptr) != 0) { err = "nvrtcCreateProgram failed"; return false; }
    std::vector<const char*> opts = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo", o.strict_fp ? "--fmad=false" : "--fmad=true",
                                     "--ptxas-options=-v", "-diag-suppress=550"};
    int rc = g_nvrtc.CompileProgram(prog, (int)opts.size(), opts.data());
    size_t n = 0; g_nvrtc.GetProgramLogSize(prog, &n);
    std::string log(n, '\0'); if (n) g_nvrtc.GetProgramLog(prog, &log[0]);
    if (rc != 0) {
        err = "NVRTC compile failed:\n" + log.substr(0, 4000);
        g_nvrtc.DestroyProgram(&prog);
        return false;
    }
    parse_ptxas_log(log, info);
    n = 0; g_nvrtc.GetCUBINSize(prog, &n);
    cubin.resize(n);
    g_nvrtc.GetCUBIN(prog, cubin.data());
    g_nvrtc.DestroyProgram(&prog);
    return n > 0;
}

CodegenConfig make_config(const tsb_batch* b, const tsb_opts& o, int dc_param) {
    CodegenConfig cfg;
    cfg.varying = b->varying; cfg.var_slot = b->var_slot; cfg.n_var = (int)b->slot_ptr.size();
    cfg.block_size = o.block_size > 0 ? o.block_size : 128;
    cfg.dc_param = dc_param;
    cfg.fast_div = !o.strict_fp;
    cfg.min_blocks = o.min_blocks;            // 0 = "auto" placeholder (never compiled as such)
    cfg.skip_linear = o.skip_linear_resolve != 0;
    cfg.lane_refill = o.lane_refill != 0;
    cfg.tgrid = o.share_time_grid != 0;
    cfg.coop_parts = o.coop_parts > 0 ? o.coop_parts : 0;
    if (cfg.coop_parts) cfg.tgrid = false;
    if (const char* tf = getenv("TSB_TRANFAST")) cfg.tranfast = *tf != '0';       // development knob: A/B of the condensed elimination
    cfg.grid = b->grid_kernel;
    if (b->meas_kernel)
        for (const tsb_meas& m : b->meas) { cfg.meas.push_back(m.kind); cfg.meas.push_back(m.column); cfg.meas.push_back(m.trig_column); }
    if (b->four_kernel)
        for (const tsb_four& f : b->four) { cfg.four.push_back(f.column); cfg.four.push_back(f.n_harm); }
    cfg.dc_nested = b->dc_nested; cfg.dc_param2 = b->dc_param2;
    cfg.order = b->d_order != nullptr;
    if (const char* x = getenv("TSB_EXTRA_DEFINES")) {          // development knob for A/B kernel experiments
        std::string item;
        for (const char* c = x;; ++c) {
            if (*c == ';' || *c == '\0') {
                size_t eq = item.find('=');
                if (!item.empty()) {
                    std::string name = eq == std::string::npos ? item : item.substr(0, eq);
                    cfg.extra_defines += "#undef " + name + "\n#define " + name + " " + (eq == std::string::npos ? "1" : item.substr(eq + 1)) + "\n";
                }
                item.clear();
                if (*c == '\0') break;
            } else item += *c;
        }
    }
    return cfg;
}

bool read_file(const std::string& path, std::vector<char>& out) {
    std::ifstream f(path, std::ios::binary);
    if (!f) return false;
    out.assign(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
    return !out.empty();
}

// Small cache files (<autokey>.auto, <autokey>.<gpu>.tuned) are written under a private name and renamed into place like
// the cubins: ranks of one job share the directory.
void write_small_file(const std::string& path, const std::string& content) {
    const std::string tmp = path + ".tmp" + std::to_string((long long)getpid());
    { std::ofstream f(tmp); f << content; }
    rename(tmp.c_str(), path.c_str());
}

// cubin (+ ptxas figures) of one fully specified source: kernel cache first, NVRTC on a miss.
int obtain_cubin(tsb_ctx* ctx, const std::string& src, const std::string& key, const tsb_opts& o, std::vector<char>& cubin, KernelInfo& info) {
    const std::string base = ctx->cache_dir + "/" + key;
    if (read_file(base + ".cubin", cubin)) {
        std::ifstream f(base + ".info");
        if (f) f >> info.regs >> info.spill_st >> info.spill_ld;
        return TSB_OK;
    }
    std::string err;
    mkdir(ctx->cache_dir.c_str(), 0755);
    // Several ranks of one job share this directory: every file is written under a private name and renamed into
    // place (atomic on POSIX), so a reader sees either nothing (and compiles for itself) or a complete file.
    const std::string tmp = base + ".tmp" + std::to_string((long long)getpid());
    { std::ofstream f(tmp + ".cu"); f << src; }
    rename((tmp + ".cu").c_str(), (base + ".cu").c_str());
    if (!nvrtc_compile(src, base + ".cu", o, cubin, info, err)) return fail(ctx, TSB_E_COMPILE, err);
    { std::ofstream f(tmp + ".info"); f << info.regs << " " << info.spill_st << " " << info.spill_ld << "\n"; }
    rename((tmp + ".info").c_str(), (base + ".info").c_str());
    { std::ofstream f(tmp + ".cubin", std::ios::binary); f.write(cubin.data(), (std::streamsize)cubin.size()); }
    rename((tmp + ".cubin").c_str(), (base + ".cubin").c_str());
    return TSB_OK;
}

// Launch bounds of the transient kernel.  One circuit per thread keeps everything in registers, so
// occupancy is bought with the register cap: the kernels are latency-bound (dependent FP64 chains),
// more resident warps help until the cap forces spills into the Newton loop.  Rule (measured on B200,
// profiles/r01_notes.md): the largest min-blocks-per-SM in {6..1} whose ptxas report shows at most
// TSB_SPILL_OK bytes of spill stores; __graft_entry__.build() applies the same rule with nvcc.
const int TSB_SPILL_OK = 100;
const int TSB_MAX_MIN_BLOCKS = 6;

int get_module_uncached(tsb_batch* b, tsb_opts o, int dc_param, KernelModule** out, std::string* autokey_out);

int get_module(tsb_batch* b, tsb_opts o, int dc_param, KernelModule** out, std::string* autokey_out = nullptr) {
    tsb_ctx* ctx = b->ctx;
    std::string sig;
    sig.reserve(b->varying.size() + 96);
    sig.append(b->varying.begin(), b->varying.end());
    const char* xd = getenv("TSB_EXTRA_DEFINES");
    char tail[200];
    snprintf(tail, sizeof tail, "|%d|%d|%d|%d|%d|%d|%d|%d|%d|%d|%d|%d|%lld|%p|", o.coop_parts, o.share_time_grid != 0, o.strict_fp, o.block_size, o.skip_linear_resolve, o.min_blocks, o.lane_refill,
             (int)b->grid_kernel, (int)(b->d_order != nullptr), dc_param, (int)b->dc_nested, b->dc_param2, ctx->choice_epoch, (void*)ctx);
    sig += tail;
    if (b->meas_kernel)
        for (const tsb_meas& m : b->meas) sig += std::to_string(m.kind) + "," + std::to_string(m.column) + "," + std::to_string(m.trig_column) + ";";
    if (b->four_kernel) {
        sig += "|four:";
        for (const tsb_four& f : b->four) sig += std::to_string(f.column) + "," + std::to_string(f.n_harm) + ";";
    }
    if (xd) sig += xd;
    if (const char* tf = getenv("TSB_TRANFAST")) { sig += "|tf"; sig += tf; }
    if (b->memo_module && sig == b->memo_sig) {
        *out = b->memo_module;
        if (autokey_out) *autokey_out = b->memo_autokey;
        return TSB_OK;
    }
    std::string autokey;
    const long long epoch0 = ctx->choice_epoch;
    int rc = get_module_uncached(b, o, dc_param, out, &autokey);
    if (rc != TSB_OK) return rc;
    if (autokey_out) *autokey_out = autokey;
    if (ctx->choice_epoch == epoch0) { b->memo_sig = sig; b->memo_autokey = autokey; b->memo_module = *out; }   // pointers into ctx->modules are stable (std::map)
    else b->memo_module = nullptr;
    return TSB_OK;
}

int get_module_uncached(tsb_batch* b, tsb_opts o, int dc_param, KernelModule** out, std::string* autokey_out) {
    tsb_ctx* ctx = b->ctx;
    std::vector<char> cubin;
    KernelInfo info;
    std::string src, key;
    if (o.min_blocks <= 0) {
        o.min_blocks = 0;
        std::string autokey = source_key(generate_source(b->plan->p, make_config(b, o, dc_param)), compile_options_string(o));
        if (autokey_out) *autokey_out = autokey;
        auto ch = ctx->auto_choice.find(autokey);
        int chosen = ch != ctx->auto_choice.end() ? ch->second : 0;
        if (!chosen) {                       // a choice timed by an earlier process on this machine
            std::ifstream f(ctx->cache_dir + "/" + autokey + ctx->tuned_suffix);
            if (f && (f >> chosen) && chosen >= 1 && chosen <= 8) ctx->tuned[autokey] = chosen; else chosen = 0;
        }
        if (!chosen) {
            std::ifstream f(ctx->cache_dir + "/" + autokey + ".auto");
            if (f) f >> chosen;
        }
        if (chosen < 1 || chosen > 8) {
            int best = 1, best_spill = 1 << 30;
            for (int mb = TSB_MAX_MIN_BLOCKS; mb >= 1; --mb) {
                o.min_blocks = mb;
                src = generate_source(b->plan->p, make_config(b, o, dc_param));
                key = source_key(src, compile_options_string(o));
                KernelInfo ki;
                int rc = obtain_cubin(ctx, src, key, o, cubin, ki);
                if (rc != TSB_OK) return rc;
                int sp = ki.spill_st < 0 ? 0 : ki.spill_st;
                if (sp < best_spill) { best_spill = sp; best = mb; }
                if (sp <= TSB_SPILL_OK) { best = mb; break; }
            }
            chosen = best;
            write_small_file(ctx->cache_dir + "/" + autokey + ".auto", std::to_string(chosen) + "\n");
        }
        if (!ctx->auto_choice.count(autokey) || ctx->auto_choice[autokey] != chosen) { ctx->auto_choice[autokey] = chosen; ++ctx->choice_epoch; }
        o.min_blocks = chosen;
    }
    src = generate_source(b->plan->p, make_config(b, o, dc_param));
    key = source_key(src, compile_options_string(o));
    auto it = ctx->modules.find(key);
    if (it != ctx->modules.end()) { *out = &it->second; return TSB_OK; }
    int rc = obtain_cubin(ctx, src, key, o, cubin, info);
    if (rc != TSB_OK) return rc;
    KernelModule m;
    CU(ctx, cudaLibraryLoadData(&m.lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
    CU(ctx, cudaLibraryGetKernel(&m.optran, m.lib, "tsb_optran"));
    CU(ctx, cudaLibraryGetKernel(&m.dc, m.lib, "tsb_dc"));
    CU(ctx, cudaLibraryGetKernel(&m.stamp, m.lib, "tsb_stamp"));
    CU(ctx, cudaLibraryGetKernel(&m.stamp_staged, m.lib, "tsb_stamp_staged"));
    CU(ctx, cudaLibraryGetKernel(&m.ac, m.lib, "tsb_ac"));
    if (src.find("tsb_coop_tran(TsbArgs a)") != std::string::npos) CU(ctx, cudaLibraryGetKernel(&m.coop, m.lib, "tsb_coop_tran"));
    m.info_regs = info.regs; m.info_spill = info.spill_st; m.min_blocks = o.min_blocks;
    ctx->modules[key] = m;
    *out = &ctx->modules[key];
    return TSB_OK;
}

// Debug aid ($TSB_GUARD=1; compute-sanitizer is not available on every pool): every result buffer is allocated with a
// 256-byte band of 0xA5 on each side; tsb_batch_sync() reads the bands back and fails with the name of the buffer
// whose neighbourhood a kernel wrote to.  With small batches the structure-of-arrays strides are within a band, so
// an off-by-one in a row / column / instance count is caught.
const size_t TSB_GUARD_BYTES = 256;

cudaError_t galloc(tsb_batch* b, void** p, size_t bytes) {
    if (!b->ctx->guard) return cudaMalloc(p, bytes);
    char* base = nullptr;
    const size_t payload = (bytes + 15) / 16 * 16;
    cudaError_t e = cudaMalloc((void**)&base, payload + 2 * TSB_GUARD_BYTES);
    if (e != cudaSuccess) return e;
    cudaMemsetAsync(base, 0xA5, payload + 2 * TSB_GUARD_BYTES, b->ctx->stream);
    *p = base + TSB_GUARD_BYTES;
    b->guarded[*p] = payload;
    return cudaSuccess;
}
template <class P> void gfree(tsb_batch* b, P*& p) {
    if (!p) return;
    auto it = b->guarded.find((void*)p);
    if (it != b->guarded.end()) { cudaFree((char*)p - TSB_GUARD_BYTES); b->guarded.erase(it); }
    else cudaFree(p);
    p = nullptr;
}
int guard_check(tsb_batch* b) {
    tsb_ctx* ctx = b->ctx;
    if (!ctx->guard) return TSB_OK;
    std::vector<unsigned char> h(TSB_GUARD_BYTES);
    auto name_of = [&](void* p) -> const char* {
        const std::pair<const void*, const char*> known[] = {
            {b->d_wave, "wave"}, {b->d_stats, "stats"}, {b->d_rows, "rows"}, {b->d_status, "status"},
            {b->d_counters, "counters"}, {b->d_scratch, "scratch"}, {b->d_sweep, "sweep"}, {b->d_meas, "meas"}, {b->d_four, "four"},
            {b->d_four_tw, "four twiddles"}};
        for (const auto& kn : known)
            if (p == kn.first) return kn.second;
        return "buffer";
    };
    for (auto& kv : b->guarded) {
        for (int side = 0; side < 2; ++side) {
            const char* src = side == 0 ? (char*)kv.first - TSB_GUARD_BYTES : (char*)kv.first + kv.second;
            CU(ctx, cudaMemcpy(h.data(), src, TSB_GUARD_BYTES, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < TSB_GUARD_BYTES; ++i)
                if (h[i] != 0xA5)
                    return fail(ctx, TSB_E_CUDA, std::string("TSB_GUARD: a kernel wrote ") + (side ? "past the end of" : "before the start of") +
                                " the `" + name_of(kv.first) + "` buffer (offset " + std::to_string(side ? (long long)i : (long long)i - (long long)TSB_GUARD_BYTES) + ")");
        }
    }
    return TSB_OK;
}

void free_results(tsb_batch* b) {
    gfree(b, b->d_wave); gfree(b, b->d_stats); gfree(b, b->d_rows); gfree(b, b->d_status);
    gfree(b, b->d_counters); gfree(b, b->d_scratch); gfree(b, b->d_sweep); gfree(b, b->d_sweep2); gfree(b, b->d_meas); gfree(b, b->d_four); gfree(b, b->d_four_tw); cudaFree(b->d_totals); cudaFree(b->d_work);
    b->d_work = nullptr;
    b->d_wave = b->d_stats = b->d_scratch = b->d_sweep = b->d_sweep2 = nullptr;
    b->d_rows = b->d_counters = nullptr; b->d_status = nullptr; b->d_totals = nullptr;
    b->wave_bytes = b->stats_bytes = b->meas_bytes = b->four_bytes = 0;
    b->meas_last = b->four_last = b->four_rows = 0;
    b->four_tw_sent = false;
}

int alloc_results(tsb_batch* b, int analysis, int out_flags, int64_t cap_rows, int n_sweep) {
    tsb_ctx* ctx = b->ctx;
    const Plan& p = b->plan->p;
    const int64_t N = b->n_inst;
    int ncol = p.num_columns(analysis);
    size_t wave_bytes = (out_flags & (TSB_OUT_WAVE | TSB_OUT_GRID)) ? (size_t)cap_rows * ncol * N * sizeof(double) : 0;
    size_t stats_bytes = (out_flags & TSB_OUT_STATS) ? (size_t)4 * ncol * N * sizeof(double) : 0;
    if (wave_bytes != b->wave_bytes) {
        gfree(b, b->d_wave); b->wave_bytes = 0;
        if (wave_bytes) { CU(ctx, galloc(b, (void**)&b->d_wave, wave_bytes)); b->wave_bytes = wave_bytes; }
    }
    if (stats_bytes != b->stats_bytes) {
        gfree(b, b->d_stats); b->stats_bytes = 0;
        if (stats_bytes) { CU(ctx, galloc(b, (void**)&b->d_stats, stats_bytes)); b->stats_bytes = stats_bytes; }
    }
    b->meas_last = 0;
    if (out_flags & TSB_OUT_MEAS) {
        const size_t meas_bytes = (size_t)2 * b->meas.size() * N * sizeof(double);
        if (meas_bytes != b->meas_bytes) {
            gfree(b, b->d_meas); b->meas_bytes = 0;
            CU(ctx, galloc(b, (void**)&b->d_meas, meas_bytes)); b->meas_bytes = meas_bytes;
        }
        b->meas_last = (int)b->meas.size();
    }
    b->four_last = b->four_rows = 0;
    if (out_flags & TSB_OUT_FOUR) {
        int rows = 0;
        for (const tsb_four& f : b->four) rows += 1 + 2 * f.n_harm;
        const size_t four_bytes = (size_t)rows * N * sizeof(double);
        if (four_bytes != b->four_bytes) {
            gfree(b, b->d_four); b->four_bytes = 0;
            CU(ctx, galloc(b, (void**)&b->d_four, four_bytes)); b->four_bytes = four_bytes;
        }
        if (!b->four_tw_sent) {          // once per table
            gfree(b, b->d_four_tw);
            CU(ctx, galloc(b, (void**)&b->d_four_tw, b->four_tw.size() * sizeof(double)));
            CU(ctx, cudaMemcpyAsync(b->d_four_tw, b->four_tw.data(), b->four_tw.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            CU(ctx, cudaStreamSynchronize(ctx->stream));     // a new table may replace the host copy
            b->four_tw_sent = true;
        }
        b->four_last = (int)b->four.size();
        b->four_rows = rows;
    }
    if (!b->d_rows) CU(ctx, galloc(b, (void**)&b->d_rows, N * sizeof(long long)));
    if (!b->d_status) CU(ctx, galloc(b, (void**)&b->d_status, N * sizeof(int)));
    if (!b->d_counters) CU(ctx, galloc(b, (void**)&b->d_counters, 8 * N * sizeof(long long)));
    if (!b->d_scratch) CU(ctx, galloc(b, (void**)&b->d_scratch, (size_t)(p.n() + 1) * N * sizeof(double)));
    if (!b->d_totals) CU(ctx, cudaMalloc(&b->d_totals, 6 * sizeof(unsigned long long)));
    if (!b->d_work) CU(ctx, cudaMalloc(&b->d_work, sizeof(unsigned long long)));
    if (n_sweep > 0) {
        gfree(b, b->d_sweep); CU(ctx, galloc(b, (void**)&b->d_sweep, (size_t)n_sweep * sizeof(double)));
        gfree(b, b->d_sweep2);
        if (analysis == TSB_AN_DC2) CU(ctx, galloc(b, (void**)&b->d_sweep2, (size_t)n_sweep * sizeof(double)));
    }
    b->analysis = analysis; b->ncol = ncol; b->out_flags = out_flags; b->cap_rows = cap_rows;
    return TSB_OK;
}

// Marks "everything of this batch queued on the launch stream so far": the next parameter upload waits for it.
int note_launched(tsb_batch* b) {
    tsb_ctx* ctx = b->ctx;
    if (!b->ev_launched) CU(ctx, cudaEventCreateWithFlags(&b->ev_launched, cudaEventDisableTiming));
    CU(ctx, cudaEventRecord(b->ev_launched, ctx->stream));
    return TSB_OK;
}

int launch(tsb_batch* b, const tsb_opts& o, cudaKernel_t kernel, TsbArgsHost& args, bool persistent = false, int min_blocks = 0) {
    tsb_ctx* ctx = b->ctx;
    int block = o.block_size > 0 ? o.block_size : 128;
    const int ncol_smem = b->plan->p.num_columns(b->analysis == TSB_AN_DC2 ? TSB_AN_DC2 : b->analysis == TSB_AN_AC ? TSB_AN_AC : TSB_AN_TRAN);
    size_t smem = (args.out_flags & (TSB_OUT_STATS | TSB_OUT_GRID)) ? (size_t)4 * ncol_smem * block * sizeof(double) : 0;
    if (args.out_flags & TSB_OUT_MEAS) smem += (size_t)4 * b->meas_last * block * sizeof(double);     // 32 bytes per measurement
    if (args.out_flags & TSB_OUT_FOUR) smem += (size_t)2 * b->four_last * block * sizeof(double);     // 16 bytes per Fourier entry
    if (smem > 48 * 1024) CU(ctx, cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long blocks = (args.n_run + block - 1) / block;
    if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;
    if (blocks < 1) blocks = 1;
    if (!persistent) {
        args.work_counter = b->d_work;          // static mapping: the first fetch of every lane is already out of range
        args.first_free = args.n_run;
    } else {
        // Lane refill (skeleton.cuh): a resident grid of SMs x blocks-per-SM; lanes that finish an instance take
        // the next one from the work counter.  Sized from the occupancy the launch-bounds choice bought.
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)kernel, block, smem) != cudaSuccess || per_sm < 1) {
            cudaGetLastError();
            per_sm = min_blocks > 0 ? min_blocks : 2;
        }
        long long resident = (long long)ctx->sms * per_sm;
        if (blocks > resident) blocks = resident;
        CU(ctx, cudaMemsetAsync(b->d_work, 0, sizeof(unsigned long long), ctx->stream));
        args.work_counter = b->d_work;
        args.first_free = blocks * block;
    }
    void* kargs[] = {&args};
    CU(ctx, cudaLaunchKernel((const void*)kernel, dim3((unsigned)blocks), dim3((unsigned)block), kargs, smem, ctx->stream));
    ++ctx->launches;
    return note_launched(b);
}

int fill_common(tsb_batch* b, const tsb_opts& o, TsbArgsHost& a) {
    tsb_ctx* ctx = b->ctx;
    if (b->fetch_pending) {            // results of the previous run are still being copied out: the next run overwrites them
        CU(ctx, cudaStreamWaitEvent(ctx->stream, b->ev_fetch, 0));
        b->fetch_pending = false;
    }
    if (b->params_pending) {           // parameter uploads of tsb_batch_set_param* are on the upload stream
        CU(ctx, cudaStreamWaitEvent(ctx->stream, b->ev_params, 0));
        b->params_pending = false;
    }
    memset(&a, 0, sizeof a);
    a.n_inst = b->n_inst;
    a.n_run = b->n_inst;
    a.order = b->d_order;
    if (b->slot_ptr.size() > TSB_MAX_VARYING) return fail(ctx, TSB_E_UNSUPPORTED, "too many per-instance parameters (max 128)");
    for (size_t s = 0; s < b->slot_ptr.size(); ++s) a.pv[s] = b->slot_ptr[s];
    size_t ub = b->uniform.size() * sizeof(double);
    if (!b->d_uniform) CU(ctx, cudaMalloc(&b->d_uniform, ub ? ub : 8));
    if (ub) CU(ctx, cudaMemcpyAsync(b->d_uniform, b->uniform.data(), ub, cudaMemcpyHostToDevice, ctx->stream));
    a.U = b->d_uniform;
    for (size_t k = 0; k < b->uniform.size() && k < 32; ++k) a.Uc[k] = b->uniform[k];
    a.max_iter = o.max_iter; a.abstol = o.abstol; a.reltol = o.reltol; a.trtol = o.trtol;
    a.wave = b->d_wave; a.stats = b->d_stats; a.rows = b->d_rows; a.status = b->d_status;
    a.counters = b->d_counters; a.scratch = b->d_scratch;
    a.out_flags = b->out_flags; a.cap_rows = b->cap_rows;
    a.skip_linear_resolve = o.skip_linear_resolve;
    if (b->out_flags & TSB_OUT_MEAS) {
        for (int m = 0; m < b->meas_last; ++m) {
            const tsb_meas& t = b->meas[m];
            a.meas_level[m] = t.level; a.meas_from[m] = t.from; a.meas_to[m] = t.to; a.meas_count[m] = t.count; a.meas_edge[m] = t.edge;
        }
        a.meas_out = b->d_meas;
    }
    return TSB_OK;
}

tsb_opts resolve(const tsb_opts* o, const Plan& plan) {
    tsb_opts r; tsb_default_opts(&r);
    if (o) {
        r = *o;
        if (r.max_iter <= 0) r.max_iter = 100;
        if (r.block_size <= 0) r.block_size = 128;
        // whole warps only: the Newton loops of nonlinear circuits are warp-synchronous (full-mask votes)
        r.block_size = (r.block_size + 31) / 32 * 32;
        if (r.block_size > 1024) r.block_size = 1024;
    }
    const char* env = getenv("TSB_STRICT_FP");
    if (env && *env) r.strict_fp = *env != '0';
    // auto: circuits with mutual couplings have MNA matrices with condition numbers ~1e7-1e8 (the
    // (1-k^2) L/dt block next to 1e-4 S conductances), where ANY re-association of the arithmetic is
    // visible at the 1e-9 parity tolerance — they run in the reference-rounding build.
    if (r.strict_fp < 0) r.strict_fp = plan.has_mutual ? 1 : 0;
    return r;
}

// Per-thread statistics live in shared memory (32 bytes per result column): a circuit with many result columns does not fit
// 128 threads' worth into an SM's 227 KB.  The block shrinks (whole warps) until it does; the block size is part of the
// kernel's specialisation, so this happens before the module is requested.
void fit_block_to_shared_memory(tsb_opts& o, int ncol, int out_flags, int n_meas, int n_four = 0) {
    if (!(out_flags & (TSB_OUT_STATS | TSB_OUT_GRID))) return;
    // a column and a measurement take 4 doubles per thread, a Fourier entry 2
    const int per_thread = 4 * ncol + ((out_flags & TSB_OUT_MEAS) ? 4 * n_meas : 0) + ((out_flags & TSB_OUT_FOUR) ? 2 * n_four : 0);
    while (o.block_size > 32 && (size_t)per_thread * o.block_size * sizeof(double) > (size_t)226 * 1024) o.block_size -= 32;
}

// TSB_OUT_FOUR: the table is checked against the transient's columns before anything is allocated or launched.
int check_fourier(tsb_batch* b, int out_flags) {
    if (!(out_flags & TSB_OUT_FOUR)) return TSB_OK;
    if (b->four.empty()) return fail(b->ctx, TSB_E_INVALID, "TSB_OUT_FOUR: the batch has no Fourier table (tsb_batch_set_fourier)");
    const int ncol = b->plan->p.num_columns(TSB_AN_TRAN);
    for (const tsb_four& f : b->four)
        if (f.column >= ncol)
            return fail(b->ctx, TSB_E_INVALID, "TSB_OUT_FOUR: column " + std::to_string(f.column) + " is out of range for the transient (" +
                                                   std::to_string(ncol) + " columns)");
    return TSB_OK;
}

// TSB_OUT_FOUR: the run-time half of the table.  Window and grid as the header defines them, one IEEE operation per step.
void fill_fourier(const tsb_batch* b, TsbArgsHost& a, double tstop) {
    int off = 0;
    for (int e = 0; e < b->four_last; ++e) {
        const tsb_four& f = b->four[e];
        const double T = 1.0 / f.freq;
        const double end = std::isinf(f.t_end) ? tstop : f.t_end;
        a.four_s[e] = end - T;
        a.four_dt[e] = T / f.n_grid;
        a.four_g[e] = f.n_grid;
        a.four_tw_off[e] = off;
        off += 2 * f.n_grid;
    }
    a.four_tw = b->d_four_tw;
    a.four_out = b->d_four;
}

// TSB_OUT_MEAS: the table is checked against the columns of the analysis before anything is allocated or launched.
int check_measures(tsb_batch* b, int analysis, int out_flags) {
    if (!(out_flags & TSB_OUT_MEAS)) return TSB_OK;
    if (b->meas.empty()) return fail(b->ctx, TSB_E_INVALID, "TSB_OUT_MEAS: the batch has no measurement table (tsb_batch_set_measures)");
    const int ncol = b->plan->p.num_columns(analysis);
    for (const tsb_meas& m : b->meas)
        if (m.column >= ncol || m.trig_column >= ncol)
            return fail(b->ctx, TSB_E_INVALID, "TSB_OUT_MEAS: measurement column " + std::to_string(m.column >= ncol ? m.column : m.trig_column) +
                                                   " is out of range for the analysis (" + std::to_string(ncol) + " columns)");
    return TSB_OK;
}

// Launch-bounds autotuning.  The spill rule above is a static prior; what it trades (resident warps against spilled
// bytes) moves with every change of the generated code, and the measured optimum was 1-2 blocks/SM above the rule
// for the nonlinear decks (profiles/r01_notes.md).  So the first transient run of a large batch times the
// candidates {rule, rule+1, rule+2} on a sub-batch of two waves of instances — the very analysis that is about to
// run, writing into the result arrays the real run overwrites — and keeps the fastest for the process (and, via
// <autokey>.tuned in the kernel cache, for later processes).  Results do not depend on the choice: register
// allocation does not change the arithmetic.  $TSB_AUTOTUNE=0 disables.
const int64_t TSB_TUNE_MIN_INSTANCES = 1 << 15;

int autotune_min_blocks(tsb_batch* b, const tsb_opts& o_auto, const std::string& autokey, int rule_choice,
                        const TsbArgsHost& a_full, bool persistent) {
    tsb_ctx* ctx = b->ctx;
    const int block = o_auto.block_size > 0 ? o_auto.block_size : 128;
    cudaEvent_t e0, e1;
    CU(ctx, cudaEventCreate(&e0)); CU(ctx, cudaEventCreate(&e1));
    int best = rule_choice; double best_per = 0.0;
    for (int mb = rule_choice; mb <= TSB_MAX_MIN_BLOCKS && mb <= rule_choice + 2; ++mb) {
        tsb_opts o = o_auto; o.min_blocks = mb;
        KernelModule* m = nullptr;
        int rc = get_module(b, o, -1, &m);
        if (rc != TSB_OK) { cudaEventDestroy(e0); cudaEventDestroy(e1); return rc; }
        // three FULL waves of this candidate's own residency, compared per instance: one sub-batch size for all candidates
        // (round 1: two waves of the largest) is a whole number of waves for that one only and charges the others a
        // nearly empty tail wave — measured on rlc.cir: 6 blocks/SM won the sub-batch and lost the real run, 191 vs 184 ms
        long long n_sub = (long long)ctx->sms * mb * block * 3;
        if (n_sub > b->n_inst) n_sub = b->n_inst;
        float ms = 0.f;
        for (int rep = 0; rep < 2; ++rep) {              // rep 0 loads the module and warms the clocks
            TsbArgsHost a = a_full; a.n_run = n_sub;
            CU(ctx, cudaEventRecord(e0, ctx->stream));
            if ((rc = launch(b, o, m->optran, a, persistent, m->min_blocks)) != TSB_OK) { cudaEventDestroy(e0); cudaEventDestroy(e1); return rc; }
            CU(ctx, cudaEventRecord(e1, ctx->stream));
            CU(ctx, cudaEventSynchronize(e1));
            CU(ctx, cudaEventElapsedTime(&ms, e0, e1));
        }
        const double per = (double)ms / (double)n_sub;
        if (mb == rule_choice || per < best_per * 0.97) { best = mb; best_per = per; }     // a later candidate must win by 3 %
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    ctx->auto_choice[autokey] = best;
    ++ctx->choice_epoch;
    ctx->tuned[autokey] = best;
    write_small_file(ctx->cache_dir + "/" + autokey + ctx->tuned_suffix, std::to_string(best) + "\n");
    return TSB_OK;
}

// Shared time grid (device/skeleton.cuh): the pilot — one more launch of the transient kernel, ONE instance (slot 0),
// no result output, on a stream of its own so that it runs beside the main launch, with enough dynamic shared memory
// that no other block shares its SM — publishes what depends on (time, dt) only for every attempt of its run.  Worth it
// only when the main launch lasts many times longer than the pilot (one instance alone is latency-bound: ~10-20 ms
// for the 2.4e4 attempts of an inductor deck), hence the instance threshold of the automatic mode.
const int64_t TSB_TGRID_MIN_INSTANCES = 1 << 18;
const int TSB_COOP_AUTO_MIN_N = 16;        // tsb_opts.coop_parts = -1: two parts from this many unknowns up
const int TSB_TGRID_CAP = 1 << 16;

// The table is a pure function of the analysis arguments, the tolerances that steer the step control, the uniform
// parameter values (sources included) and the pilot's decisions; readers verify every entry against their own (time, dt).
// So a table built by an earlier run of this batch with the same arguments is still right — and complete, because runs
// are ordered on the context's stream — and the pilot need not run again (a different pilot instance could at worst
// lower the hit rate, never change a result).
std::string tgrid_signature(const tsb_batch* b, const tsb_opts& o, const TsbArgsHost& a, const void* kernel) {
    std::string s;
    auto add = [&](const void* p, size_t n) { s.append((const char*)p, n); };
    add(&a.tstart, sizeof(double) * 5); add(&a.uic, sizeof a.uic); add(&a.trtol, sizeof a.trtol); add(&a.max_iter, sizeof a.max_iter);
    add(&o.strict_fp, sizeof o.strict_fp); add(&kernel, sizeof kernel); add(&b->d_order, sizeof b->d_order);
    add(b->uniform.data(), b->uniform.size() * sizeof(double));
    add(b->varying.data(), b->varying.size());
    return s;
}

int launch_pilot(tsb_batch* b, const tsb_opts& o, cudaKernel_t kernel, TsbArgsHost& a) {
    tsb_ctx* ctx = b->ctx;
    const int nsrc = b->plan->p.n_src > 1 ? b->plan->p.n_src : 1;
    const int nd = ((3 + nsrc + 1) / 2) * 2;      // TsbTgLayout (device/skeleton.cuh)
    if (!b->d_tgrid || b->tgrid_nd != nd) {
        cudaFree(b->d_tgrid); b->d_tgrid = nullptr;
        CU(ctx, cudaMalloc(&b->d_tgrid, (size_t)TSB_TGRID_CAP * nd * sizeof(double)));
        b->tgrid_nd = nd; b->tgrid_cap = TSB_TGRID_CAP;
    }
    if (!b->d_tgrid_pub) CU(ctx, cudaMalloc(&b->d_tgrid_pub, sizeof(unsigned long long)));
    if (!ctx->pilot_stream) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        CU(ctx, cudaStreamCreateWithPriority(&ctx->pilot_stream, cudaStreamNonBlocking, hi));
        CU(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        CU(ctx, cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    }
    a.tgrid = b->d_tgrid; a.tgrid_pub = b->d_tgrid_pub; a.tgrid_cap = b->tgrid_cap; a.tgrid_role = 0;
    const std::string sig = tgrid_signature(b, o, a, (const void*)kernel);
    const char* reuse_env = getenv("TSB_TGRID_REUSE");
    if (sig == b->tgrid_sig && !(reuse_env && *reuse_env == '0')) return TSB_OK;      // the table of the previous run stands
    b->tgrid_sig = sig;
    // only the published count is reset: readers never look at entries at or above it
    CU(ctx, cudaMemsetAsync(b->d_tgrid_pub, 0, sizeof(unsigned long long), ctx->stream));
    CU(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));          // parameters, uniform table and the reset are in place
    CU(ctx, cudaStreamWaitEvent(ctx->pilot_stream, ctx->ev_fork, 0));
    TsbArgsHost ap = a;
    ap.tgrid_role = 1; ap.n_run = 1; ap.out_flags = 0; ap.work_counter = b->d_work; ap.first_free = 1;
    const int block = o.block_size > 0 ? o.block_size : 128;
    const size_t smem = 208 * 1024;                                // > 227 KB - one main-launch block: the SM is the pilot's alone
    CU(ctx, cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    void* kargs[] = {&ap};
    CU(ctx, cudaLaunchKernel((const void*)kernel, dim3(1), dim3((unsigned)block), kargs, smem, ctx->pilot_stream));
    ++ctx->launches;
    b->tgrid_used = 1;
    return TSB_OK;
}

int check_batch(tsb_batch* b) {
    if (!b || !b->plan) return TSB_E_INVALID;
    if (!b->ctx) return fail(nullptr, TSB_E_CUDA, "batch has no GPU context (host-only plan): analyses run on the GPU only");
    return TSB_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

void tsb_default_opts(tsb_opts* o) {
    if (!o) return;
    o->max_iter = 100; o->abstol = 1e-12; o->reltol = 1e-6; o->gmin = 1e-12; o->trtol = 7.0;
    o->strict_fp = -1; o->block_size = 128; o->skip_linear_resolve = 1; o->min_blocks = 0; o->lane_refill = 0; o->grid_dt = 0.0;
    o->share_time_grid = -1;
    o->coop_parts = -1;
}
const char* tsb_version(void) { return "tspice_b200 0.1 (sm_100a)"; }

int tsb_ctx_create(int device_ordinal, tsb_ctx** out) {
    if (!out) return TSB_E_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0)
        return fail(nullptr, TSB_E_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device_ordinal < 0 || device_ordinal >= count) return fail(nullptr, TSB_E_INVALID, "device ordinal out of range");
    std::unique_ptr<tsb_ctx> ctx(new tsb_ctx);
    ctx->device = device_ordinal;
    CU(nullptr, cudaSetDevice(device_ordinal));
    CU(nullptr, cudaFree(0));
    CU(nullptr, cudaDeviceGetAttribute(&ctx->sms, cudaDevAttrMultiProcessorCount, device_ordinal));
    CU(nullptr, cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    const char* env = getenv("TSB_KCACHE");
    ctx->cache_dir = env && *env ? env : lib_dir() + "/_kcache";
    {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device_ordinal) == cudaSuccess) {
            std::string nm;
            for (const char* c = prop.name; *c; ++c) nm += (isalnum((unsigned char)*c) ? *c : '_');
            ctx->tuned_suffix = "." + nm + "-" + std::to_string(ctx->sms) + "sm.tuned";
        } else cudaGetLastError();
    }
    const char* g = getenv("TSB_GUARD");
    ctx->guard = g && *g && *g != '0';
    *out = ctx.release();
    return TSB_OK;
}
static void ctx_release(tsb_ctx* ctx) {
    if (!ctx || ctx->refs.fetch_sub(1) != 1) return;
    cudaSetDevice(ctx->device);
    for (auto& kv : ctx->modules) if (kv.second.lib) cudaLibraryUnload(kv.second.lib);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->pilot_stream) cudaStreamDestroy(ctx->pilot_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->upload_stream) cudaStreamDestroy(ctx->upload_stream);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    delete ctx;
}
static void plan_release(tsb_plan* plan) {
    if (!plan || plan->refs.fetch_sub(1) != 1) return;
    ctx_release(plan->ctx);
    delete plan;
}
void tsb_ctx_destroy(tsb_ctx* ctx) { ctx_release(ctx); }
const char* tsb_last_error(tsb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_global_err.c_str(); }
int tsb_ctx_set_stream(tsb_ctx* ctx, uint64_t stream) {
    if (!ctx) return TSB_E_INVALID;
    ctx->stream = stream ? (cudaStream_t)(uintptr_t)stream : ctx->own_stream;
    return TSB_OK;
}
int tsb_ctx_get_stream(tsb_ctx* ctx, uint64_t* stream) {
    if (!ctx || !stream) return TSB_E_INVALID;
    *stream = (uint64_t)(uintptr_t)ctx->stream;
    return TSB_OK;
}
// Orders everything launched on the context's stream from now on after `event` (a cudaEvent_t recorded by the caller on
// the stream that produced borrowed device buffers: tsb_batch_set_param_dev, tsb_batch_stamp_dev, tsb_lu_solve_batched_dev).
int tsb_ctx_wait_event(tsb_ctx* ctx, uint64_t event) {
    if (!ctx || !event) return TSB_E_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamWaitEvent(ctx->stream, (cudaEvent_t)(uintptr_t)event, 0));
    return TSB_OK;
}
int tsb_ctx_set_cache_dir(tsb_ctx* ctx, const char* dir) {
    if (!ctx || !dir) return TSB_E_INVALID;
    ctx->cache_dir = dir;
    return TSB_OK;
}
int tsb_ctx_sm_count(tsb_ctx* ctx, int* sms) { if (!ctx || !sms) return TSB_E_INVALID; *sms = ctx->sms; return TSB_OK; }
int64_t tsb_ctx_launch_count(const tsb_ctx* ctx) { return ctx ? ctx->launches : 0; }

int tsb_ctx_measure_fp64_peak(tsb_ctx* ctx, double* tflops) {
    if (!ctx || !tflops) return TSB_E_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    const int blocks = ctx->sms * 8, iters = 4096;
    double* scratch = nullptr;
    CU(ctx, cudaMalloc(&scratch, (size_t)blocks * 256 * sizeof(double)));
    cudaEvent_t e0, e1;
    CU(ctx, cudaEventCreate(&e0)); CU(ctx, cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 6; ++rep) {
        CU(ctx, cudaEventRecord(e0, ctx->stream));
        CU(ctx, launch_fp64_peak(scratch, blocks, iters, ctx->stream));
        ++ctx->launches;
        CU(ctx, cudaEventRecord(e1, ctx->stream));
        CU(ctx, cudaEventSynchronize(e1));
        float ms = 0; CU(ctx, cudaEventElapsedTime(&ms, e0, e1));
        double flops = 2.0 * 64.0 * iters * 256.0 * blocks;     // 64 DFMA per iteration per thread
        double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(scratch);
    *tflops = best;
    return TSB_OK;
}

// ---- plan -------------------------------------------------------------------------------------
int tsb_plan_create(tsb_ctx* ctx, int n_nodes, int n_branches, tsb_plan** out) {
    if (!out || n_nodes < 0 || n_branches < 0) return TSB_E_INVALID;
    tsb_plan* p = new tsb_plan; p->ctx = ctx; p->p.ctx = ctx;
    if (ctx) ctx->refs.fetch_add(1);
    p->p.n_nodes = n_nodes; p->p.n_branches = n_branches;
    *out = p;
    return TSB_OK;
}
int tsb_plan_from_netlist(tsb_ctx* ctx, const char* text, tsb_plan** out) {
    if (!out || !text) return TSB_E_INVALID;
    *out = nullptr;
    std::unique_ptr<tsb_plan> p(new tsb_plan); p->ctx = ctx; p->p.ctx = ctx;
    std::string err;
    int rc = plan_from_netlist(text, p->p, err);
    if (rc != TSB_OK) return fail(ctx, rc, err);
    rc = plan_finalize(p->p);
    if (rc != TSB_OK) return fail(ctx, rc, p->p.error);
    if (ctx) ctx->refs.fetch_add(1);
    *out = p.release();
    return TSB_OK;
}
int tsb_plan_add_device(tsb_plan* plan, int kind, const char* name, const int* nodes, int n_nodes, int branch,
                        const double* p, int n_p, const int* ip, int n_ip) {
    if (!plan || plan->p.finalized || n_nodes < 0 || n_nodes > 4 || n_p < 0 || n_ip < 0) return TSB_E_INVALID;
    Dev d; d.kind = kind; d.name = name ? name : ""; d.n_nodes = n_nodes; d.branch = branch;
    for (int i = 0; i < n_nodes; ++i) d.nodes[i] = nodes[i];
    if (n_p) d.p.assign(p, p + n_p);
    if (n_ip) d.ip.assign(ip, ip + n_ip);
    plan->p.devs.push_back(d);
    return (int)plan->p.devs.size() - 1;
}
int tsb_plan_finalize(tsb_plan* plan) {
    if (!plan) return TSB_E_INVALID;
    int rc = plan_finalize(plan->p);
    if (rc != TSB_OK) { plan->err = plan->p.error; return fail(plan->ctx, rc, plan->p.error); }
    return TSB_OK;
}
void tsb_plan_destroy(tsb_plan* plan) { plan_release(plan); }
const char* tsb_plan_error(tsb_plan* plan) { return plan ? plan->p.error.c_str() : ""; }

int tsb_plan_coop_info(const tsb_plan* plan, int parts, int* owner, int* n_separator) {
    if (!plan || !plan->p.finalized) return TSB_E_INVALID;
    auto it = plan->p.coop.find(parts);
    if (it == plan->p.coop.end()) return TSB_E_UNSUPPORTED;
    const CoopPlan& cp = it->second;
    if (owner) for (int u = 0; u <= plan->p.n(); ++u) owner[u] = u == 0 ? -1 : cp.owner[u];
    if (n_separator) *n_separator = plan->p.n() - cp.n_int;
    return TSB_OK;
}
int tsb_plan_size(const tsb_plan* plan, int* n_nodes, int* n_branches) {
    if (!plan) return TSB_E_INVALID;
    if (n_nodes) *n_nodes = plan->p.n_nodes;
    if (n_branches) *n_branches = plan->p.n_branches;
    return TSB_OK;
}
int tsb_plan_num_devices(const tsb_plan* plan) { return plan ? (int)plan->p.devs.size() : TSB_E_INVALID; }
int tsb_plan_device_info(const tsb_plan* plan, int dev, int* kind, const char** name, int nodes[4], int* branch, int* n_p, int* n_ip) {
    if (!plan || dev < 0 || dev >= (int)plan->p.devs.size()) return TSB_E_INVALID;
    const Dev& d = plan->p.devs[dev];
    if (kind) *kind = d.kind;
    if (name) *name = d.name.c_str();
    if (nodes) for (int i = 0; i < 4; ++i) nodes[i] = i < d.n_nodes ? d.nodes[i] : 0;
    if (branch) *branch = d.branch;
    if (n_p) *n_p = (int)d.p.size();
    if (n_ip) *n_ip = (int)d.ip.size();
    return d.n_nodes;
}
int tsb_plan_device_params(const tsb_plan* plan, int dev, double* p, int cap_p, int* ip, int cap_ip) {
    if (!plan || dev < 0 || dev >= (int)plan->p.devs.size()) return TSB_E_INVALID;
    const Dev& d = plan->p.devs[dev];
    for (int i = 0; i < cap_p && i < (int)d.p.size(); ++i) p[i] = d.p[i];
    for (int i = 0; i < cap_ip && i < (int)d.ip.size(); ++i) ip[i] = d.ip[i];
    return TSB_OK;
}
int tsb_plan_find_device(const tsb_plan* plan, const char* name) {
    if (!plan || !name) return -1;
    for (size_t i = 0; i < plan->p.devs.size(); ++i) if (plan->p.devs[i].name == name) return (int)i;
    return -1;
}
int tsb_plan_node_name(const tsb_plan* plan, int node, const char** name) {
    if (!plan || !name || node < 0 || node >= (int)plan->p.node_names.size()) return TSB_E_INVALID;
    *name = plan->p.node_names[node].c_str();
    return TSB_OK;
}
int tsb_plan_analysis(const tsb_plan* plan, int* analysis, double tran[4], int* uic, int* dc_src_dev, double dc[3]) {
    if (!plan) return TSB_E_INVALID;
    if (analysis) *analysis = plan->p.analysis;
    if (tran) for (int i = 0; i < 4; ++i) tran[i] = plan->p.tran[i];
    if (uic) *uic = plan->p.uic;
    if (dc_src_dev) *dc_src_dev = plan->p.dc_src_dev;
    if (dc) for (int i = 0; i < 3; ++i) dc[i] = plan->p.dc[i];
    return TSB_OK;
}
int tsb_plan_analysis2(const tsb_plan* plan, int* dc2_src_dev, double dc2[3], int* ac_sweep, int* ac_points, double ac_f[2]) {
    if (!plan) return TSB_E_INVALID;
    if (dc2_src_dev) *dc2_src_dev = plan->p.dc2_src_dev;
    if (dc2) for (int i = 0; i < 3; ++i) dc2[i] = plan->p.dc2[i];
    if (ac_sweep) *ac_sweep = plan->p.ac_sweep;
    if (ac_points) *ac_points = plan->p.ac_points;
    if (ac_f) { ac_f[0] = plan->p.ac_f[0]; ac_f[1] = plan->p.ac_f[1]; }
    return TSB_OK;
}
int tsb_plan_structure(const tsb_plan* plan, int* ext2int, int* pivot_row, int* pivot_col) {
    if (!plan || !plan->p.finalized) return TSB_E_INVALID;
    int n = plan->p.n();
    for (int i = 0; i <= n; ++i) {
        if (ext2int) ext2int[i] = plan->p.order_main.ext2int[i];
        if (pivot_row) pivot_row[i] = plan->p.order_main.prow[i];
        if (pivot_col) pivot_col[i] = plan->p.order_main.pcol[i];
    }
    return TSB_OK;
}
int tsb_plan_pattern(const tsb_plan* plan, int mode, int* rows, int* cols, int cap, int* nnz) {
    if (!plan || !plan->p.finalized) return TSB_E_INVALID;
    std::vector<std::pair<int, int>> pat = plan->p.pattern_op;
    if (mode == 1) pat.insert(pat.end(), plan->p.pattern_tran_extra.begin(), plan->p.pattern_tran_extra.end());
    if (nnz) *nnz = (int)pat.size();
    for (int i = 0; i < cap && i < (int)pat.size(); ++i) { if (rows) rows[i] = pat[i].first; if (cols) cols[i] = pat[i].second; }
    return TSB_OK;
}
int tsb_plan_num_columns(const tsb_plan* plan, int analysis) { return plan ? plan->p.num_columns(analysis) : TSB_E_INVALID; }
int tsb_plan_column_name(const tsb_plan* plan, int analysis, int col, char* buf, int cap) {
    if (!plan || !buf || cap <= 0 || col < 0 || col >= plan->p.num_columns(analysis)) return TSB_E_INVALID;
    snprintf(buf, cap, "%s", plan->p.column_name(analysis, col).c_str());
    return TSB_OK;
}

// ---- batch ------------------------------------------------------------------------------------
int tsb_batch_create(tsb_plan* plan, int64_t n_inst, tsb_batch** out) {
    if (!plan || !out || n_inst <= 0) return TSB_E_INVALID;
    if (!plan->p.finalized) return fail(plan->ctx, TSB_E_INVALID, "plan is not finalized");
    tsb_batch* b = new tsb_batch;
    b->plan = plan; b->ctx = plan->ctx; b->n_inst = n_inst;
    plan->refs.fetch_add(1);
    b->uniform = plan->p.nominal;
    b->varying.assign(plan->p.n_params, 0);
    b->var_slot.assign(plan->p.n_params, -1);
    *out = b;
    return TSB_OK;
}
void tsb_batch_destroy(tsb_batch* b) {
    if (!b) return;
    if (b->ctx) {
        cudaSetDevice(b->ctx->device);
        for (size_t s = 0; s < b->slot_ptr.size(); ++s) {
            if (b->slot_owned[s]) cudaFree(b->slot_ptr[s]);
            if (b->slot_stage[s]) { cudaEventSynchronize(b->slot_staged[s]); cudaFreeHost(b->slot_stage[s]); cudaEventDestroy(b->slot_staged[s]); }
        }
        cudaFree(b->d_uniform);
        cudaFree(b->d_order);
        cudaFree(b->d_coop_state);
        cudaFree(b->d_tgrid); cudaFree(b->d_tgrid_pub); cudaFree(b->d_partial);
        if (b->ev_fetch) { cudaEventSynchronize(b->ev_fetch); cudaEventDestroy(b->ev_fetch); }
        if (b->ev_run) cudaEventDestroy(b->ev_run);
        if (b->ev_params) { cudaEventSynchronize(b->ev_params); cudaEventDestroy(b->ev_params); }
        if (b->ev_launched) cudaEventDestroy(b->ev_launched);
        free_results(b);
    }
    plan_release(b->plan);
    delete b;
}

static int param_index(tsb_batch* b, int dev, int param, int* flat) {
    if (!b) return TSB_E_INVALID;
    const Plan& p = b->plan->p;
    if (dev < 0 || dev >= (int)p.devs.size()) return fail(b->ctx, TSB_E_INVALID, "device index out of range");
    const Dev& d = p.devs[dev];
    if (param < 0 || param >= (int)d.p.size()) return fail(b->ctx, TSB_E_INVALID, "parameter index out of range for " + d.name);
    if ((d.kind == TSB_V || d.kind == TSB_I) && d.src_type() == TSB_SRC_PWL)
        return fail(b->ctx, TSB_E_UNSUPPORTED, "PWL tables are not sweepable");
    *flat = d.p_off + param;
    return TSB_OK;
}
static int claim_slot(tsb_batch* b, int flat) {
    if (b->var_slot[flat] >= 0) return b->var_slot[flat];
    b->varying[flat] = 1;
    b->var_slot[flat] = (int)b->slot_ptr.size();
    b->slot_ptr.push_back(nullptr);
    b->slot_owned.push_back(0);
    b->slot_stage.push_back(nullptr);
    b->slot_staged.push_back(nullptr);
    return b->var_slot[flat];
}
// Host values -> the parameter's device array.  `staged`: the values are first copied into a library-owned pinned
// buffer, so the caller's buffer is free again when the call returns whatever memory it is (with pinned caller memory
// cudaMemcpyAsync is a true DMA that reads the buffer later).  !staged (tsb_batch_set_param_async): zero-copy, the
// caller keeps the buffer valid and unmodified until the next tsb_batch_sync / result read.
static int set_param_host(tsb_batch* b, int dev, int param, const double* values, bool staged) {
    int flat = 0, rc = param_index(b, dev, param, &flat);
    if (rc != TSB_OK) return rc;
    if (!values) return TSB_E_INVALID;
    int slot = claim_slot(b, flat);
    if (!b->ctx) return TSB_OK;      // host-only plan: only the "varies per instance" fact is recorded
    tsb_ctx* ctx = b->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)b->n_inst * sizeof(double);
    if (!b->slot_owned[slot]) {
        double* p = nullptr;
        CU(ctx, cudaMalloc(&p, bytes));
        b->slot_ptr[slot] = p; b->slot_owned[slot] = 1;
    }
    const double* src = values;
    if (staged) {
        if (!b->slot_stage[slot]) {
            CU(ctx, cudaMallocHost((void**)&b->slot_stage[slot], bytes));
            CU(ctx, cudaEventCreateWithFlags(&b->slot_staged[slot], cudaEventDisableTiming));
        } else CU(ctx, cudaEventSynchronize(b->slot_staged[slot]));      // the previous copy out of this staging buffer
        memcpy(b->slot_stage[slot], values, bytes);
        src = b->slot_stage[slot];
    }
    // On the upload stream (see tsb_batch.ev_launched) unless the launch stream is being captured into a graph, where the
    // copy has to be a node of that graph.
    cudaStream_t up = ctx->stream;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(ctx->stream, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; }
    const bool beside = cap == cudaStreamCaptureStatusNone;
    if (beside) {
        if (!ctx->upload_stream) CU(ctx, cudaStreamCreateWithFlags(&ctx->upload_stream, cudaStreamNonBlocking));
        up = ctx->upload_stream;
        if (b->ev_launched) CU(ctx, cudaStreamWaitEvent(up, b->ev_launched, 0));     // this batch's last launch has read the old values
    }
    CU(ctx, cudaMemcpyAsync(b->slot_ptr[slot], src, bytes, cudaMemcpyHostToDevice, up));
    if (staged) CU(ctx, cudaEventRecord(b->slot_staged[slot], up));
    if (beside) {
        if (!b->ev_params) CU(ctx, cudaEventCreateWithFlags(&b->ev_params, cudaEventDisableTiming));
        CU(ctx, cudaEventRecord(b->ev_params, up));
        b->params_pending = true;
    }
    return TSB_OK;
}
int tsb_batch_set_param(tsb_batch* b, int dev, int param, const double* values) { return set_param_host(b, dev, param, values, true); }
int tsb_batch_set_param_async(tsb_batch* b, int dev, int param, const double* values) { return set_param_host(b, dev, param, values, false); }
int tsb_batch_set_param_dev(tsb_batch* b, int dev, int param, uint64_t dev_ptr) {
    int flat = 0, rc = param_index(b, dev, param, &flat);
    if (rc != TSB_OK) return rc;
    if (!dev_ptr) return TSB_E_INVALID;
    int slot = claim_slot(b, flat);
    if (b->slot_owned[slot]) { cudaFree(b->slot_ptr[slot]); b->slot_owned[slot] = 0; }
    b->slot_ptr[slot] = (double*)(uintptr_t)dev_ptr;
    return TSB_OK;
}
int tsb_batch_set_param_uniform(tsb_batch* b, int dev, int param, double value) {
    int flat = 0, rc = param_index(b, dev, param, &flat);
    if (rc != TSB_OK) return rc;
    if (b->varying[flat]) return fail(b->ctx, TSB_E_INVALID, "parameter already set per instance");
    b->uniform[flat] = value;
    return TSB_OK;
}

// ---- analyses ----------------------------------------------------------------------------------
int tsb_run_op(tsb_batch* b, const tsb_opts* opts) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    tsb_opts o = resolve(opts, b->plan->p);
    o.coop_parts = 0;          // the cooperative mapping is a transient-only specialisation
    CU(ctx, cudaSetDevice(ctx->device));
    KernelModule* m = nullptr;
    if ((rc = get_module(b, o, -1, &m)) != TSB_OK) return rc;
    if ((rc = alloc_results(b, TSB_AN_OP, TSB_OUT_WAVE, 1, 0)) != TSB_OK) return rc;
    TsbArgsHost a;
    if ((rc = fill_common(b, o, a)) != TSB_OK) return rc;
    a.analysis = TSB_AN_OP;
    return launch(b, o, m->optran, a, b->plan->p.has_nonlinear && o.lane_refill != 0, m->min_blocks);
}

int tsb_run_tran(tsb_batch* b, double tstart, double tstop, double tstep, double tmax, int uic, int out_flags,
                 int64_t wave_cap_rows, const tsb_opts* opts) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    if (!(tstop > 0) || !(tstep > 0)) return fail(ctx, TSB_E_INVALID, "tstop and tstep must be positive");
    if (!(out_flags & (TSB_OUT_WAVE | TSB_OUT_STATS | TSB_OUT_GRID | TSB_OUT_MEAS | TSB_OUT_FOUR))) return fail(ctx, TSB_E_INVALID, "no output selected");
    if ((out_flags & TSB_OUT_WAVE) && (out_flags & TSB_OUT_GRID)) return fail(ctx, TSB_E_INVALID, "TSB_OUT_WAVE and TSB_OUT_GRID share the waveform buffer: select one");
    if ((out_flags & TSB_OUT_WAVE) && wave_cap_rows <= 0) return fail(ctx, TSB_E_INVALID, "wave_cap_rows must be positive");
    if ((rc = check_measures(b, TSB_AN_TRAN, out_flags)) != TSB_OK) return rc;
    if ((rc = check_fourier(b, out_flags)) != TSB_OK) return rc;
    if (out_flags & (TSB_OUT_MEAS | TSB_OUT_FOUR)) out_flags |= TSB_OUT_STATS;     // the previous stored row lives in the statistics' `last` slots
    tsb_opts o = resolve(opts, b->plan->p);
    // NewTransient (tran.go:29-55)
    if (tstep > tstop / 300) tstep = tstop / 300;
    double minstep = tstep / 50.0;
    if (tmax == 0) tmax = tstep;
    double grid_dt = 0.0; int64_t n_grid = 0;
    if (out_flags & TSB_OUT_GRID) {
        out_flags |= TSB_OUT_STATS;          // the previous stored row lives in the statistics' `last` slots
        grid_dt = o.grid_dt > 0 ? o.grid_dt : tstep;
        double span = tstop - tstart;
        if (!(span > 0) || !(grid_dt > 0)) return fail(ctx, TSB_E_INVALID, "TSB_OUT_GRID needs tstart < tstop and a positive grid spacing");
        double q = span / grid_dt;
        if (q > 1e7) return fail(ctx, TSB_E_INVALID, "TSB_OUT_GRID: more than 1e7 grid points");
        n_grid = (int64_t)floor(q * (1.0 + 1e-12) + 1e-9);
        if (n_grid < 1) n_grid = 1;
        wave_cap_rows = n_grid;
    }
    CU(ctx, cudaSetDevice(ctx->device));
    if (const char* ce = getenv("TSB_COOP")) { if (*ce) o.coop_parts = atoi(ce); }      // development / A-B knob
    if (o.coop_parts < 0) {
        // auto: the cooperative mapping where it measured faster than one thread per circuit (RC ladders on B200: n = 14
        // 0.86x, n = 18 1.6x, n = 26 2.1x with two parts; diode-clamped ladders: n = 14 1.1x, n = 26 1.8x) and everything it
        // needs holds; otherwise thread-per-circuit
        const Plan& cpl = b->plan->p;
        o.coop_parts = 0;
        if (!cpl.has_bjt && !cpl.has_mutual && !o.strict_fp && !(out_flags & (TSB_OUT_GRID | TSB_OUT_MEAS | TSB_OUT_FOUR)) && o.skip_linear_resolve && !o.lane_refill) {
            // two parts where they fit; more parts only when the statistics of fewer do not leave an SM two blocks
            if (cpl.n() >= TSB_COOP_AUTO_MIN_N)
                for (int pick : {2, 4, 8}) {
                    if (!cpl.coop.count(pick)) continue;
                    const int nx = cpl.coop.at(pick).nx, nown = cpl.coop.at(pick).nown_max;
                    if (((size_t)4 * nown * 32 * pick + (size_t)2 * pick * nx * 32) * sizeof(double) <= 110 * 1024) { o.coop_parts = pick; break; }
                }
        }
    }
    if (o.coop_parts != 0) {
        // cooperative mapping (device/coop.cuh): an explicit request is refused where it does not apply, never silently replaced
        const Plan& cpl = b->plan->p;
        if (o.coop_parts != 2 && o.coop_parts != 4 && o.coop_parts != 8) return fail(ctx, TSB_E_INVALID, "coop_parts must be -1, 0, 2, 4 or 8");
        if (cpl.has_bjt || cpl.has_mutual) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts: circuits with BJTs or mutual couplings run thread-per-circuit");
        if (!cpl.coop.count(o.coop_parts)) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts: the netlist has no partition into that many sub-circuits (tsb_plan_coop_info)");
        if (o.strict_fp) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts: the nested-dissection order is a re-association, not available in the strict build");
        if (out_flags & TSB_OUT_GRID) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts: TSB_OUT_GRID is not available on the cooperative mapping");
        if (out_flags & TSB_OUT_MEAS) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts: TSB_OUT_MEAS is not available on the cooperative mapping");
        if (out_flags & TSB_OUT_FOUR) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts: TSB_OUT_FOUR is not available on the cooperative mapping");
        if (!o.skip_linear_resolve || o.lane_refill) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts needs skip_linear_resolve = 1 and lane_refill = 0");
        if (o.min_blocks <= 0) o.min_blocks = 2;          // tsb_optran only runs the operating point here: no launch-bounds search
    } else fit_block_to_shared_memory(o, b->plan->p.num_columns(TSB_AN_TRAN), out_flags, (int)b->meas.size(), (int)b->four.size());
    KernelModule* m = nullptr;
    b->grid_kernel = (out_flags & TSB_OUT_GRID) != 0;
    b->meas_kernel = (out_flags & TSB_OUT_MEAS) != 0;
    b->four_kernel = (out_flags & TSB_OUT_FOUR) != 0;
    std::string autokey;
    rc = get_module(b, o, -1, &m, &autokey);
    if (rc != TSB_OK) { b->grid_kernel = b->meas_kernel = b->four_kernel = false; return rc; }
    if ((rc = alloc_results(b, TSB_AN_TRAN, out_flags, (out_flags & (TSB_OUT_WAVE | TSB_OUT_GRID)) ? wave_cap_rows : 0, 0)) != TSB_OK) return rc;
    TsbArgsHost a;
    if ((rc = fill_common(b, o, a)) != TSB_OK) return rc;
    a.analysis = TSB_AN_TRAN; a.uic = uic;
    a.tstart = tstart; a.tstop = tstop; a.tstep = tstep; a.maxstep = tmax; a.minstep = minstep;
    a.grid_dt = grid_dt; a.n_grid = (int)n_grid;
    if (out_flags & TSB_OUT_FOUR) fill_fourier(b, a, tstop);
    const bool persistent = b->plan->p.has_nonlinear && o.lane_refill != 0;
    const char* tune_env = getenv("TSB_AUTOTUNE");
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(ctx->stream, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; }
    if (o.coop_parts == 0 && o.min_blocks <= 0 && !autokey.empty() && b->n_inst >= TSB_TUNE_MIN_INSTANCES && !ctx->tuned.count(autokey) &&
        !(tune_env && *tune_env == '0') && cap == cudaStreamCaptureStatusNone) {
        rc = autotune_min_blocks(b, o, autokey, m->min_blocks, a, persistent);
        if (rc == TSB_OK) rc = get_module(b, o, -1, &m);
        if (rc != TSB_OK) { b->grid_kernel = b->meas_kernel = b->four_kernel = false; return rc; }
    }
    b->grid_kernel = b->meas_kernel = b->four_kernel = false;
    b->tgrid_used = 0;
    const Plan& pl = b->plan->p;
    if (o.coop_parts > 0) {
        if (!m->coop) return fail(ctx, TSB_E_COMPILE, "cooperative kernel missing from the module");
        const CoopPlan& cp = pl.coop.at(o.coop_parts);
        if (!b->d_coop_state) CU(ctx, cudaMalloc(&b->d_coop_state, (size_t)(pl.n_state + pl.n() + 1) * b->n_inst * sizeof(double)));
        a.coop_state = b->d_coop_state;
        // 1. operating point(s) thread-per-circuit, state handed over; 2. the transient on the cooperative mapping
        TsbArgsHost a1 = a;
        a1.out_flags = 0;
        if ((rc = launch(b, o, m->optran, a1, false, m->min_blocks)) != TSB_OK) return rc;
        const int nx = cp.nx, nown = cp.nown_max;
        const int groups = 1, block = 32 * cp.parts * groups;
        const size_t smem = ((size_t)4 * nown * block + (size_t)groups * 2 * cp.parts * nx * 32) * sizeof(double);
        if (smem > 227 * 1024) return fail(ctx, TSB_E_UNSUPPORTED, "coop_parts: the statistics of one block do not fit in shared memory");
        if (smem > 48 * 1024) CU(ctx, cudaFuncSetAttribute((const void*)m->coop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        long long blocks = (a.n_run + 32 * groups - 1) / (32 * groups);
        if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;
        if (blocks < 1) blocks = 1;
        void* kargs[] = {&a};
        CU(ctx, cudaLaunchKernel((const void*)m->coop, dim3((unsigned)blocks), dim3((unsigned)block), kargs, smem, ctx->stream));
        ++ctx->launches;
        return note_launched(b);
    }
    const bool tg_possible = !pl.has_nonlinear && o.skip_linear_resolve != 0 && o.share_time_grid != 0 && !persistent;
    if (tg_possible && (o.share_time_grid > 0 || b->n_inst >= TSB_TGRID_MIN_INSTANCES)) {
        if ((rc = launch_pilot(b, o, m->optran, a)) != TSB_OK) return rc;
    }
    rc = launch(b, o, m->optran, a, persistent, m->min_blocks);
    if (rc == TSB_OK && b->tgrid_used) {
        // join: whatever follows on the context's stream (result reads, the next run) also follows the pilot
        CU(ctx, cudaEventRecord(ctx->ev_join, ctx->pilot_stream));
        CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
        if ((rc = note_launched(b)) != TSB_OK) return rc;      // the pilot reads the parameters too
    }
    return rc;
}

// DC sweep, one source (dc.go:88-140) or two nested sources (dc.go:205-270; src2_dev >= 0: the outer loop runs over
// source 1, the inner over source 2).  The sweep axes are the same for every instance, so the host flattens them into
// one list of points and the device loop stays warp-uniform.
static int run_dc_impl(tsb_batch* b, int src_dev, double start, double stop, double inc, int src2_dev, double start2, double stop2,
                       double inc2, int out_flags, const tsb_opts* opts) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    const Plan& p = b->plan->p;
    const bool nested = src2_dev != -1;
    auto is_vsrc = [&](int d) { return d >= 0 && d < (int)p.devs.size() && p.devs[d].kind == TSB_V; };
    if (!is_vsrc(src_dev) || (nested && !is_vsrc(src2_dev)))
        return fail(ctx, TSB_E_INVALID, nested ? "source not found" : "source not found");       // dc.go:47-68, :226-228
    if (!(inc > 0) || (nested && !(inc2 > 0))) return fail(ctx, TSB_E_INVALID, "sweep increment must be positive");
    if (out_flags & TSB_OUT_GRID) return fail(ctx, TSB_E_INVALID, "TSB_OUT_GRID applies to transient analysis only");
    if (out_flags & TSB_OUT_FOUR) return fail(ctx, TSB_E_UNSUPPORTED, "TSB_OUT_FOUR applies to transient analysis only");
    if (!(out_flags & (TSB_OUT_WAVE | TSB_OUT_STATS | TSB_OUT_MEAS))) return fail(ctx, TSB_E_INVALID, "no output selected");
    if (nested && (out_flags & TSB_OUT_MEAS)) return fail(ctx, TSB_E_UNSUPPORTED, "TSB_OUT_MEAS: the nested DC sweep's column 0 is not monotone");
    if ((rc = check_measures(b, TSB_AN_DC, out_flags)) != TSB_OK) return rc;
    if (out_flags & TSB_OUT_MEAS) out_flags |= TSB_OUT_STATS;
    std::vector<double> s1, s2;
    for (double v = start; v <= stop; v += inc) { s1.push_back(v); if (s1.size() > (1u << 24)) break; }   // dc.go:36-42
    if (nested) for (double v = start2; v <= stop2; v += inc2) { s2.push_back(v); if (s2.size() > (1u << 24)) break; }
    std::vector<double> sweep, sweep2;
    if (!nested) sweep = s1;
    else {
        if ((double)s1.size() * (double)s2.size() > (double)(1u << 24)) return fail(ctx, TSB_E_INVALID, "nested sweep: more than 2^24 points");
        for (double v1 : s1) for (double v2 : s2) { sweep.push_back(v1); sweep2.push_back(v2); }
    }
    tsb_opts o = resolve(opts, b->plan->p);
    o.coop_parts = 0;          // the cooperative mapping is a transient-only specialisation
    fit_block_to_shared_memory(o, p.num_columns(nested ? (int)TSB_AN_DC2 : (int)TSB_AN_DC), out_flags, (int)b->meas.size());
    CU(ctx, cudaSetDevice(ctx->device));
    auto dc_param_of = [&](int d) {
        const Dev& sd = p.devs[d];
        const int st = sd.src_type();
        return (st == TSB_SRC_DC || st == TSB_SRC_SIN) ? sd.p_off : -1;          // SetValue only reaches dcValue
    };
    const int dc_param = dc_param_of(src_dev), dc_param2 = nested ? dc_param_of(src2_dev) : -1;
    if ((dc_param >= 0 && b->varying[dc_param]) || (dc_param2 >= 0 && b->varying[dc_param2]))
        return fail(ctx, TSB_E_INVALID, "the swept source value is set per instance");
    const int an = nested ? (int)TSB_AN_DC2 : (int)TSB_AN_DC;
    KernelModule* m = nullptr;
    b->dc_nested = nested; b->dc_param2 = dc_param2; b->meas_kernel = (out_flags & TSB_OUT_MEAS) != 0;
    rc = get_module(b, o, dc_param, &m);
    b->dc_nested = false; b->dc_param2 = -1; b->meas_kernel = false;
    if (rc != TSB_OK) return rc;
    if ((rc = alloc_results(b, an, out_flags, (out_flags & TSB_OUT_WAVE) ? (int64_t)sweep.size() : 0, (int)sweep.size())) != TSB_OK) return rc;
    TsbArgsHost a;
    if ((rc = fill_common(b, o, a)) != TSB_OK) return rc;
    if (!sweep.empty()) {
        CU(ctx, cudaMemcpyAsync(b->d_sweep, sweep.data(), sweep.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        if (nested) CU(ctx, cudaMemcpyAsync(b->d_sweep2, sweep2.data(), sweep2.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    CU(ctx, cudaStreamSynchronize(ctx->stream));     // `sweep` is a stack vector
    a.analysis = TSB_AN_DC; a.sweep = b->d_sweep; a.sweep2 = b->d_sweep2; a.n_sweep = (int)sweep.size();
    return launch(b, o, m->dc, a);
}
int tsb_run_dc(tsb_batch* b, int src_dev, double start, double stop, double inc, int out_flags, const tsb_opts* opts) {
    return run_dc_impl(b, src_dev, start, stop, inc, -1, 0, 0, 0, out_flags, opts);
}
int tsb_run_dc2(tsb_batch* b, int src1_dev, double start1, double stop1, double inc1, int src2_dev, double start2, double stop2,
                double inc2, int out_flags, const tsb_opts* opts) {
    if (src2_dev < 0) return fail(b ? b->ctx : nullptr, TSB_E_INVALID, "source not found");
    return run_dc_impl(b, src1_dev, start1, stop1, inc1, src2_dev, start2, stop2, inc2, out_flags, opts);
}

// AC analysis (analysis.NewAC + Setup + Execute, ac.go:21-126): frequency points as generateFrequencyPoints makes them
// (n_points in TOTAL between fstart and fstop, on a logarithmic or linear axis), one complex solve per point and instance.
int tsb_run_ac(tsb_batch* b, int sweep_type, int n_points, double fstart, double fstop, int out_flags, const tsb_opts* opts) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    const Plan& p = b->plan->p;
    if (p.has_nonlinear)
        return fail(ctx, TSB_E_UNSUPPORTED, "AC analysis of a circuit with nonlinear devices: the reference takes their small-signal values from an "
                                             "operating point it solves on a complex matrix with a real-indexed right-hand side (matrix/circuit.go:99-105, "
                                             ":126-150); that state is an artefact of the un-vendored sparse module and is not reproduced");
    if (sweep_type < 0 || sweep_type > 2 || n_points < 1 || n_points > (1 << 20)) return fail(ctx, TSB_E_INVALID, "invalid sweep type or number of points");
    if (out_flags & TSB_OUT_GRID) return fail(ctx, TSB_E_INVALID, "TSB_OUT_GRID applies to transient analysis only");
    if (out_flags & TSB_OUT_FOUR) return fail(ctx, TSB_E_UNSUPPORTED, "TSB_OUT_FOUR applies to transient analysis only");
    if (!(out_flags & (TSB_OUT_WAVE | TSB_OUT_STATS | TSB_OUT_MEAS))) return fail(ctx, TSB_E_INVALID, "no output selected");
    if ((rc = check_measures(b, TSB_AN_AC, out_flags)) != TSB_OK) return rc;
    if (out_flags & TSB_OUT_MEAS) out_flags |= TSB_OUT_STATS;
    std::vector<double> f;
    ac_frequency_points(sweep_type, n_points, fstart, fstop, f);       // ac.go:100-126
    tsb_opts o = resolve(opts, p);
    o.coop_parts = 0;          // the cooperative mapping is a transient-only specialisation
    fit_block_to_shared_memory(o, b->plan->p.num_columns(TSB_AN_AC), out_flags, (int)b->meas.size());
    CU(ctx, cudaSetDevice(ctx->device));
    KernelModule* m = nullptr;
    b->meas_kernel = (out_flags & TSB_OUT_MEAS) != 0;
    rc = get_module(b, o, -1, &m);
    b->meas_kernel = false;
    if (rc != TSB_OK) return rc;
    if ((rc = alloc_results(b, TSB_AN_AC, out_flags, (out_flags & TSB_OUT_WAVE) ? (int64_t)n_points : 0, n_points)) != TSB_OK) return rc;
    TsbArgsHost a;
    if ((rc = fill_common(b, o, a)) != TSB_OK) return rc;
    CU(ctx, cudaMemcpyAsync(b->d_sweep, f.data(), f.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));     // `f` is a stack vector
    a.analysis = TSB_AN_AC; a.sweep = b->d_sweep; a.n_sweep = n_points;
    return launch(b, o, m->ac, a);
}

// Operator level: the device-stamp kernel on its own.  Writes, for every instance, the dense MNA system the reference
// holds after mat.Clear(); ckt.Stamp(status); mat.LoadGmin(gmin) on a freshly set-up circuit (device state as
// SetupDevices leaves it), with status = {Mode, Time, TimeStep = dt, Gmin}: A[inst][n][n] row-major and b[inst][n]
// (0-based = MNA index - 1), device pointers.  Together with tsb_lu_solve_batched_dev (pivot order from
// tsb_plan_structure) this is the two-kernel form of one Newton iteration: an HBM-bound stamp kernel and a
// compute-bound factor + solve kernel.
int tsb_batch_stamp_dev(tsb_batch* b, int mode, double time, double dt, double gmin, uint64_t A_dev, uint64_t b_dev, const tsb_opts* opts) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    if (!A_dev || !b_dev || (mode != 0 && mode != 1)) return fail(ctx, TSB_E_INVALID, "tsb_batch_stamp_dev: mode must be 0 (OP) or 1 (transient), outputs non-null");
    // A transient stamp divides by the step (C/dt, M/dt, ...); the fast build multiplies by 1/dt instead, which the kernel
    // only forms for dt > 0, so a zero, negative or NaN step would stamp those conductances as 0 there and as +-Inf or a
    // negative conductance in the strict build.  No analysis takes such a step: refuse it.
    if (mode == TSB_AN_TRAN && !(dt > 0)) return fail(ctx, TSB_E_INVALID, "tsb_batch_stamp_dev: transient mode needs dt > 0");
    tsb_opts o = resolve(opts, b->plan->p);
    o.coop_parts = 0;          // the cooperative mapping is a transient-only specialisation
    CU(ctx, cudaSetDevice(ctx->device));
    KernelModule* m = nullptr;
    if ((rc = get_module(b, o, -1, &m)) != TSB_OK) return rc;
    TsbArgsHost a;
    if ((rc = fill_common(b, o, a)) != TSB_OK) return rc;       // parameters only: no result buffers are needed here
    a.analysis = mode; a.tstart = time; a.tstep = dt; a.minstep = gmin;    // tsb_stamp reads status.Gmin from `minstep`
    a.wave = (double*)(uintptr_t)A_dev; a.stats = (double*)(uintptr_t)b_dev;
    a.out_flags = 0;
    // Staged (coalesced) form whenever the block's systems fit in shared memory: threads per block = the largest
    // multiple of 32 (<= the configured block size) with threads * ((n*n+n)|1) doubles <= 200 KB.
    const int n = b->plan->p.n();
    const size_t per_thread = (size_t)(((n * n + n) | 1)) * sizeof(double);
    int block = o.block_size > 0 ? o.block_size : 128;
    int staged_threads = (int)(200 * 1024 / per_thread) / 32 * 32;
    if (staged_threads > block) staged_threads = block;
    const char* env = getenv("TSB_STAMP_DIRECT");
    const bool staged = staged_threads >= 32 && !(env && *env == '1');
    cudaKernel_t kern = staged ? m->stamp_staged : m->stamp;
    size_t smem = 0;
    if (staged) {
        block = staged_threads;
        smem = (size_t)block * per_thread;
        if (smem > 48 * 1024) CU(ctx, cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    long long blocks = (b->n_inst + block - 1) / block;
    long long resident = (long long)ctx->sms * 32;             // grid-stride over blocks of instances
    if (blocks > resident) blocks = resident;
    void* kargs[] = {&a};
    CU(ctx, cudaLaunchKernel((const void*)kern, dim3((unsigned)blocks), dim3((unsigned)block), kargs, smem, ctx->stream));
    ++ctx->launches;
    return note_launched(b);
}

// Processing order.  Instances are independent, so WHICH lane works on which instance is free; what is not free is
// that the lanes of a warp advance together (warp-synchronous Newton loops): a warp is as slow as its slowest lane.
// A caller who knows which parameter drives the iteration count can hand over a permutation that puts like with like
// (e.g. np.argsort of the diode emission coefficient: diode2.cir -20 %).  Parameters and results stay in the
// caller's order; results are bit-identical with and without an order.  perm == NULL removes it.
int tsb_batch_set_order(tsb_batch* b, const int64_t* perm) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (!perm) { CU(ctx, cudaStreamSynchronize(ctx->stream)); cudaFree(b->d_order); b->d_order = nullptr; return TSB_OK; }
    std::vector<char> seen((size_t)b->n_inst, 0);
    for (int64_t i = 0; i < b->n_inst; ++i) {
        if (perm[i] < 0 || perm[i] >= b->n_inst || seen[(size_t)perm[i]]) return fail(ctx, TSB_E_INVALID, "tsb_batch_set_order: not a permutation of 0..n_inst-1");
        seen[(size_t)perm[i]] = 1;
    }
    if (!b->d_order) CU(ctx, cudaMalloc(&b->d_order, (size_t)b->n_inst * sizeof(long long)));
    static_assert(sizeof(long long) == sizeof(int64_t), "order entries are 64-bit");
    CU(ctx, cudaMemcpyAsync(b->d_order, perm, (size_t)b->n_inst * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return TSB_OK;
}

int tsb_batch_set_measures(tsb_batch* b, const tsb_meas* m, int n_meas) {
    if (!b || n_meas < 0 || (n_meas > 0 && !m)) return TSB_E_INVALID;
    if (n_meas > TSB_MEAS_CAP) return fail(b->ctx, TSB_E_INVALID, "tsb_batch_set_measures: at most 16 measurements");
    std::vector<tsb_meas> t(m, m + n_meas);
    for (int k = 0; k < n_meas; ++k) {
        tsb_meas& e = t[k];
        const std::string at = "tsb_batch_set_measures: measurement " + std::to_string(k) + ": ";
        if (e.kind < TSB_MEAS_WHEN || e.kind > TSB_MEAS_RMS) return fail(b->ctx, TSB_E_INVALID, at + "unknown kind");
        if (e.column < 1) return fail(b->ctx, TSB_E_INVALID, at + "column must be >= 1 (column 0 is the abscissa)");
        if (std::isnan(e.from) || std::isnan(e.to) || e.from > e.to) return fail(b->ctx, TSB_E_INVALID, at + "window needs from <= to");
        if (e.kind == TSB_MEAS_WHEN) {
            if (e.trig_column < 1) return fail(b->ctx, TSB_E_INVALID, at + "trig_column must be >= 1");
            if (e.edge < TSB_EDGE_CROSS || e.edge > TSB_EDGE_FALL) return fail(b->ctx, TSB_E_INVALID, at + "unknown edge");
            if (e.count == 0 || e.count < -1) return fail(b->ctx, TSB_E_INVALID, at + "count must be >= 1 or -1 (the last crossing)");
        } else {
            e.trig_column = e.column; e.edge = 0; e.count = 1;      // unused: kept out of the kernel specialisation
        }
        if ((e.kind == TSB_MEAS_WHEN || e.kind == TSB_MEAS_AT) && std::isnan(e.level)) return fail(b->ctx, TSB_E_INVALID, at + "level is NaN");
    }
    b->meas = t;
    b->meas_last = 0;                  // the last run's results belong to the old table
    b->memo_module = nullptr;
    return TSB_OK;
}

int tsb_batch_set_fourier(tsb_batch* b, const tsb_four* f, int n) {
    if (!b || n < 0 || (n > 0 && !f)) return TSB_E_INVALID;
    if (n > TSB_FOUR_CAP) return fail(b->ctx, TSB_E_INVALID, "tsb_batch_set_fourier: at most 8 entries");
    std::vector<tsb_four> t(f, f + n);
    std::vector<double> tw;
    for (int k = 0; k < n; ++k) {
        const tsb_four& e = t[k];
        const std::string at = "tsb_batch_set_fourier: entry " + std::to_string(k) + ": ";
        if (e.column < 1) return fail(b->ctx, TSB_E_INVALID, at + "column must be >= 1 (column 0 is TIME)");
        if (e.n_harm < 1 || e.n_harm > TSB_FOUR_MAX_HARM) return fail(b->ctx, TSB_E_INVALID, at + "n_harm must be in 1 .. 32");
        if (e.n_grid < 2 * e.n_harm + 1 || e.n_grid > TSB_FOUR_MAX_GRID) return fail(b->ctx, TSB_E_INVALID, at + "n_grid must be in 2 n_harm + 1 .. 65536");
        if (!std::isfinite(e.freq) || !(e.freq > 0)) return fail(b->ctx, TSB_E_INVALID, at + "freq must be finite and positive");
        if (std::isnan(e.t_end) || e.t_end == -INFINITY) return fail(b->ctx, TSB_E_INVALID, at + "t_end must be finite or +inf");
        const size_t c0 = tw.size();
        tw.resize(c0 + 2 * (size_t)e.n_grid);
        for (int j = 0; j < e.n_grid; ++j) {           // evaluated left to right: ((2.0 pi) j) / G
            tw[c0 + j] = std::cos(2.0 * M_PI * j / e.n_grid);
            tw[c0 + e.n_grid + j] = std::sin(2.0 * M_PI * j / e.n_grid);
        }
    }
    b->four = t;
    b->four_tw = tw;
    b->four_tw_sent = false;
    b->four_last = b->four_rows = 0;   // the last run's results belong to the old table
    b->memo_module = nullptr;
    return TSB_OK;
}

int tsb_batch_sync(tsb_batch* b) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    CU(b->ctx, cudaSetDevice(b->ctx->device));
    // THIS batch's last launch (ev_launched is recorded on the launch stream after every launch of the batch), not the whole
    // stream: a host that alternates two batches must not wait here for the other batch's run that is computing right now
    if (b->ev_launched && !b->ctx->guard) CU(b->ctx, cudaEventSynchronize(b->ev_launched));
    else CU(b->ctx, cudaStreamSynchronize(b->ctx->stream));
    if (b->ev_fetch) CU(b->ctx, cudaEventSynchronize(b->ev_fetch));
    if (b->ev_params) CU(b->ctx, cudaEventSynchronize(b->ev_params));      // zero-copy uploads: the caller's buffers are free again
    return guard_check(b);
}

static int result_totals6(tsb_batch* b, int64_t totals[6]);

// Asynchronous read-back of the last run's per-instance results into (pinned) host buffers; NULL = not wanted.  The
// copies are queued on a copy stream of the context behind the run, so they overlap whatever is launched next on the
// context's stream (another batch's run); the buffers are complete after tsb_batch_sync(batch).  A later run on the SAME
// batch waits for them on the device before it overwrites the results.
int tsb_result_fetch_async(tsb_batch* b, double* stats, int64_t* rows, int32_t* status, int64_t* counters) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    if (stats && !b->d_stats) return fail(ctx, TSB_E_INVALID, "the last run did not keep statistics");
    if (!b->d_rows) return fail(ctx, TSB_E_INVALID, "no run yet");
    if (!ctx->copy_stream) CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    if (!b->ev_run) {
        CU(ctx, cudaEventCreateWithFlags(&b->ev_run, cudaEventDisableTiming));
        CU(ctx, cudaEventCreateWithFlags(&b->ev_fetch, cudaEventDisableTiming));
    }
    CU(ctx, cudaEventRecord(b->ev_run, ctx->stream));
    CU(ctx, cudaStreamWaitEvent(ctx->copy_stream, b->ev_run, 0));
    if (stats) CU(ctx, cudaMemcpyAsync(stats, b->d_stats, b->stats_bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (rows) CU(ctx, cudaMemcpyAsync(rows, b->d_rows, b->n_inst * sizeof(long long), cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (status) CU(ctx, cudaMemcpyAsync(status, b->d_status, b->n_inst * sizeof(int), cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (counters) CU(ctx, cudaMemcpyAsync(counters, b->d_counters, 8 * b->n_inst * sizeof(long long), cudaMemcpyDeviceToHost, ctx->copy_stream));
    CU(ctx, cudaEventRecord(b->ev_fetch, ctx->copy_stream));
    b->fetch_pending = true;
    return TSB_OK;
}

// Batch-level summary computed on the device: out[3][n_columns] = per column the minimum, the maximum and the sum over
// ALL instances and stored rows; *rows_total = number of stored rows of the batch (mean = sum / rows_total).  A few KB
// cross the bus instead of 32 * n_columns bytes per instance.
int tsb_result_summary(tsb_batch* b, double* out, int64_t* rows_total) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    if (!out) return TSB_E_INVALID;
    if (!b->d_stats) return fail(ctx, TSB_E_INVALID, "the last run did not keep statistics (TSB_OUT_STATS)");
    CU(ctx, cudaSetDevice(ctx->device));
    const int bx = 64, ncol = b->ncol;
    if (!b->d_partial) CU(ctx, cudaMalloc(&b->d_partial, (size_t)64 * 64 * 3 * sizeof(double) + 64));
    if (ncol > 64) return fail(ctx, TSB_E_UNSUPPORTED, "tsb_result_summary: more than 64 result columns");
    CU(ctx, launch_summary(b->d_stats, b->n_inst, ncol, b->d_partial, bx, ctx->stream));
    ++ctx->launches;
    std::vector<double> h((size_t)ncol * bx * 3);
    CU(ctx, cudaMemcpyAsync(h.data(), b->d_partial, h.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    int64_t totals[6];
    if ((rc = result_totals6(b, totals)) != TSB_OK) return rc;             // synchronises the stream
    for (int c = 0; c < ncol; ++c) {
        double mn = HUGE_VAL, mx = -HUGE_VAL, sm = 0.0;
        for (int k = 0; k < bx; ++k) {
            const double* p = &h[((size_t)c * bx + k) * 3];
            mn = fmin(mn, p[0]); mx = fmax(mx, p[1]); sm += p[2];
        }
        out[0 * ncol + c] = mn; out[1 * ncol + c] = mx; out[2 * ncol + c] = sm;
    }
    if (rows_total) *rows_total = totals[5];          // counters[7]: rows of the result series the statistics run over
    return TSB_OK;
}

// ---- results -----------------------------------------------------------------------------------
int tsb_result_dims(const tsb_batch* b, int64_t* n_inst, int* n_columns, int64_t* cap_rows) {
    if (!b) return TSB_E_INVALID;
    if (n_inst) *n_inst = b->n_inst;
    if (n_columns) *n_columns = b->ncol;
    if (cap_rows) *cap_rows = b->cap_rows;
    return TSB_OK;
}
int tsb_result_dev_ptrs(const tsb_batch* b, uint64_t* wave, uint64_t* stats, uint64_t* rows, uint64_t* status, uint64_t* counters) {
    if (!b) return TSB_E_INVALID;
    if (wave) *wave = (uint64_t)(uintptr_t)b->d_wave;
    if (stats) *stats = (uint64_t)(uintptr_t)b->d_stats;
    if (rows) *rows = (uint64_t)(uintptr_t)b->d_rows;
    if (status) *status = (uint64_t)(uintptr_t)b->d_status;
    if (counters) *counters = (uint64_t)(uintptr_t)b->d_counters;
    return TSB_OK;
}
static int d2h(tsb_batch* b, void* dst, const void* src, size_t bytes) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    if (!src) return fail(b->ctx, TSB_E_INVALID, "no such result for the last run");
    CU(b->ctx, cudaSetDevice(b->ctx->device));
    CU(b->ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, b->ctx->stream));
    CU(b->ctx, cudaStreamSynchronize(b->ctx->stream));
    return TSB_OK;
}
int tsb_result_rows(tsb_batch* b, int64_t* rows) { return b && rows ? d2h(b, rows, b->d_rows, b->n_inst * sizeof(long long)) : TSB_E_INVALID; }
int tsb_result_status(tsb_batch* b, int32_t* status) { return b && status ? d2h(b, status, b->d_status, b->n_inst * sizeof(int)) : TSB_E_INVALID; }
int tsb_result_counters(tsb_batch* b, int64_t* counters) { return b && counters ? d2h(b, counters, b->d_counters, 8 * b->n_inst * sizeof(long long)) : TSB_E_INVALID; }
int tsb_result_wave_all(tsb_batch* b, double* out, int64_t n_doubles) {
    if (!b || !out) return TSB_E_INVALID;
    if ((size_t)n_doubles * sizeof(double) < b->wave_bytes) return fail(b->ctx, TSB_E_INVALID, "output buffer too small");
    return d2h(b, out, b->d_wave, b->wave_bytes);
}
int tsb_result_stats_all(tsb_batch* b, double* out) { return b && out ? d2h(b, out, b->d_stats, b->stats_bytes) : TSB_E_INVALID; }
int tsb_result_measures(tsb_batch* b, double* out) {
    if (!b || !out) return TSB_E_INVALID;
    if (!b->meas_last) return fail(b->ctx, TSB_E_INVALID, "the last run had no TSB_OUT_MEAS");
    return d2h(b, out, b->d_meas, (size_t)2 * b->meas_last * b->n_inst * sizeof(double));
}
int tsb_result_fourier(tsb_batch* b, double* out) {
    if (!b || !out) return TSB_E_INVALID;
    if (!b->four_last) return fail(b->ctx, TSB_E_INVALID, "the last run had no TSB_OUT_FOUR");
    return d2h(b, out, b->d_four, (size_t)b->four_rows * b->n_inst * sizeof(double));
}
int tsb_result_waveform(tsb_batch* b, int64_t inst, double* out, int64_t cap_rows, int64_t* n_rows) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    if (!out || inst < 0 || inst >= b->n_inst) return TSB_E_INVALID;
    if (!b->d_wave) return fail(ctx, TSB_E_INVALID, "the last run did not store waveforms");
    CU(ctx, cudaSetDevice(ctx->device));
    long long rows = 0;
    CU(ctx, cudaMemcpyAsync(&rows, b->d_rows + inst, sizeof rows, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (rows > b->cap_rows) rows = b->cap_rows;
    if (n_rows) *n_rows = rows;
    if (rows > cap_rows) rows = cap_rows;
    if (rows <= 0) return TSB_OK;
    // gather the strided column: wave[(r*ncol + j)*n_inst + inst] -> out[r*ncol + j]
    CU(ctx, cudaMemcpy2DAsync(out, sizeof(double), b->d_wave + inst, (size_t)b->n_inst * sizeof(double), sizeof(double),
                              (size_t)rows * b->ncol, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return TSB_OK;
}
static int result_totals6(tsb_batch* b, int64_t totals[6]) {
    int rc = check_batch(b); if (rc != TSB_OK) return rc;
    tsb_ctx* ctx = b->ctx;
    if (!totals || !b->d_counters) return TSB_E_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemsetAsync(b->d_totals, 0, 6 * sizeof(unsigned long long), ctx->stream));
    CU(ctx, launch_totals(b->d_counters, b->n_inst, b->d_totals, ctx->sms, ctx->stream));
    ++ctx->launches;
    unsigned long long h[6];
    CU(ctx, cudaMemcpyAsync(h, b->d_totals, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 6; ++k) totals[k] = (int64_t)h[k];
    return TSB_OK;
}
int tsb_result_totals(tsb_batch* b, int64_t totals[5]) {
    int64_t t[6];
    int rc = result_totals6(b, t);
    if (rc != TSB_OK) return rc;
    for (int k = 0; k < 5; ++k) totals[k] = t[k];
    return TSB_OK;
}

// ---- operator level: batched factor + solve (lu_warp.cu) -------------------------------------------
int tsb_lu_order(int n, const double* A_nominal, int* pivot_row, int* pivot_col) {
    if (n < 1 || n > 32 || !A_nominal || !pivot_row || !pivot_col) return TSB_E_INVALID;
    MarkowitzLU lu(n);
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) lu.add(i + 1, j + 1, A_nominal[i * n + j]);      // dense structure, as SetupElements leaves it
    if (!lu.order_and_factor()) return TSB_E_INVALID;
    for (int k = 1; k <= n; ++k) { pivot_row[k - 1] = lu.pivot_row(k); pivot_col[k - 1] = lu.pivot_col(k); }
    return TSB_OK;
}

static int lu_check_order(tsb_ctx* ctx, int n, const int* pr, const int* pc, int* prow0, int* pcol0) {
    if (n < 1 || n > 32) return fail(ctx, TSB_E_UNSUPPORTED, "tsb_lu_solve_batched: order must be 1..32 (the matrix of a system lives in the registers of at most 16 lanes)");
    unsigned seen_r = 0, seen_c = 0;
    for (int k = 0; k < n; ++k) {
        if (pr[k] < 1 || pr[k] > n || pc[k] < 1 || pc[k] > n) return fail(ctx, TSB_E_INVALID, "pivot order: index out of range");
        seen_r |= 1u << (pr[k] - 1); seen_c |= 1u << (pc[k] - 1);
        prow0[k] = pr[k] - 1; pcol0[k] = pc[k] - 1;
    }
    const unsigned full = n == 32 ? 0xffffffffu : ((1u << n) - 1);
    if (seen_r != full || seen_c != full) return fail(ctx, TSB_E_INVALID, "pivot order: not a permutation");
    return TSB_OK;
}

// Real (words = 1) and complex (words = 2: interleaved re, im) systems share the checks, the launch accounting and the host
// staging; only the kernel family differs.
typedef cudaError_t (*LuLaunch)(const double*, const double*, double*, int*, long long, int, const int*, const int*, int, int,
                                cudaStream_t);

static int lu_solve_dev(tsb_ctx* ctx, LuLaunch launch, int n, const int* pivot_row, const int* pivot_col, uint64_t A_dev,
                        uint64_t b_dev, uint64_t x_dev, uint64_t status_dev, int64_t n_inst, int strict_fp) {
    if (!ctx) return TSB_E_CUDA;
    if (!pivot_row || !pivot_col || !A_dev || !b_dev || !x_dev || !status_dev || n_inst < 0) return TSB_E_INVALID;
    int h[64];
    int rc = lu_check_order(ctx, n, pivot_row, pivot_col, h, h + 32);
    if (rc != TSB_OK) return rc;
    if (n_inst == 0) return TSB_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    // the pivot order goes to the kernel by value (a kernel parameter): nothing to allocate or copy per call
    cudaError_t e = launch((const double*)(uintptr_t)A_dev, (const double*)(uintptr_t)b_dev, (double*)(uintptr_t)x_dev,
                           (int*)(uintptr_t)status_dev, n_inst, n, h, h + 32, strict_fp != 0, ctx->sms, ctx->stream);
    ++ctx->launches;
    CU(ctx, e);
    return TSB_OK;
}

static int lu_solve_host(tsb_ctx* ctx, LuLaunch launch, int words, const char* what, int n, const int* pivot_row,
                         const int* pivot_col, const double* A, const double* b, double* x, int32_t* status, int64_t n_inst,
                         int strict_fp) {
    if (!ctx) return TSB_E_CUDA;
    if (!A || !b || !x || !status || n_inst < 0 || n < 1 || n > 32) return TSB_E_INVALID;
    if (n_inst == 0) return TSB_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t na = (size_t)n_inst * n * n * words * sizeof(double), nb = (size_t)n_inst * n * words * sizeof(double);
    double *dA = nullptr, *db = nullptr, *dx = nullptr; int* dst = nullptr;
    CU(ctx, cudaMalloc(&dA, na));
    if (cudaMalloc(&db, nb) != cudaSuccess || cudaMalloc(&dx, nb) != cudaSuccess || cudaMalloc(&dst, (size_t)n_inst * sizeof(int)) != cudaSuccess) {
        cudaFree(dA); cudaFree(db); cudaFree(dx); cudaFree(dst); cudaGetLastError();
        return fail(ctx, TSB_E_NOMEM, std::string(what) + ": out of device memory");
    }
    int rc = TSB_OK;
    if (cudaMemcpyAsync(dA, A, na, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
        cudaMemcpyAsync(db, b, nb, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) rc = fail(ctx, TSB_E_CUDA, "H2D copy failed");
    if (rc == TSB_OK) rc = lu_solve_dev(ctx, launch, n, pivot_row, pivot_col, (uint64_t)(uintptr_t)dA, (uint64_t)(uintptr_t)db,
                                        (uint64_t)(uintptr_t)dx, (uint64_t)(uintptr_t)dst, n_inst, strict_fp);
    if (rc == TSB_OK && (cudaMemcpyAsync(x, dx, nb, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
                         cudaMemcpyAsync(status, dst, (size_t)n_inst * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
                         cudaStreamSynchronize(ctx->stream) != cudaSuccess))
        rc = fail(ctx, TSB_E_CUDA, std::string(what) + ": " + cudaGetErrorString(cudaGetLastError()));
    cudaFree(dA); cudaFree(db); cudaFree(dx); cudaFree(dst);
    return rc;
}

int tsb_lu_solve_batched_dev(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, uint64_t A_dev, uint64_t b_dev,
                             uint64_t x_dev, uint64_t status_dev, int64_t n_inst, int strict_fp) {
    return lu_solve_dev(ctx, launch_lu_warp, n, pivot_row, pivot_col, A_dev, b_dev, x_dev, status_dev, n_inst, strict_fp);
}

int tsb_lu_solve_batched(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, const double* A, const double* b,
                         double* x, int32_t* status, int64_t n_inst, int strict_fp) {
    return lu_solve_host(ctx, launch_lu_warp, 1, "tsb_lu_solve_batched", n, pivot_row, pivot_col, A, b, x, status, n_inst, strict_fp);
}

int tsb_lu_solve_batched_complex_dev(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, uint64_t A_dev,
                                     uint64_t b_dev, uint64_t x_dev, uint64_t status_dev, int64_t n_inst, int strict_fp) {
    return lu_solve_dev(ctx, launch_clu_warp, n, pivot_row, pivot_col, A_dev, b_dev, x_dev, status_dev, n_inst, strict_fp);
}

int tsb_lu_solve_batched_complex(tsb_ctx* ctx, int n, const int* pivot_row, const int* pivot_col, const double* A,
                                 const double* b, double* x, int32_t* status, int64_t n_inst, int strict_fp) {
    return lu_solve_host(ctx, launch_clu_warp, 2, "tsb_lu_solve_batched_complex", n, pivot_row, pivot_col, A, b, x, status,
                         n_inst, strict_fp);
}

// ---- introspection -------------------------------------------------------------------------------
// Selects which specialisation tsb_batch_kernel_source / _key describe (the build step pre-compiles them): the DC-sweep
// kernels are specialised for the swept source(s), the TSB_OUT_GRID kernels carry the resampling code.
int tsb_batch_kernel_variant(tsb_batch* b, int dc_src_dev, int dc_src2_dev, int grid) {
    if (!b) return TSB_E_INVALID;
    const Plan& p = b->plan->p;
    auto param_of = [&](int d, int* out) {
        if (d < 0) { *out = -1; return true; }
        if (d >= (int)p.devs.size() || p.devs[d].kind != TSB_V) return false;
        const int st = p.devs[d].src_type();
        *out = (st == TSB_SRC_DC || st == TSB_SRC_SIN) ? p.devs[d].p_off : -1;
        return true;
    };
    int p1 = -1, p2 = -1;
    if (!param_of(dc_src_dev, &p1) || !param_of(dc_src2_dev, &p2)) return fail(b->ctx, TSB_E_INVALID, "source not found");
    b->intro_dc_param = p1; b->dc_param2 = p2; b->dc_nested = dc_src2_dev >= 0;
    b->grid_kernel = (grid & ~(TSB_OUT_MEAS | TSB_OUT_FOUR)) != 0; b->meas_kernel = (grid & TSB_OUT_MEAS) != 0;
    b->four_kernel = (grid & TSB_OUT_FOUR) != 0;
    b->memo_module = nullptr;
    return TSB_OK;
}
int tsb_batch_kernel_source(tsb_batch* b, const tsb_opts* opts, char* buf, int64_t cap, int64_t* needed) {
    if (!b) return TSB_E_INVALID;
    tsb_opts o = resolve(opts, b->plan->p);
    std::string src = generate_source(b->plan->p, make_config(b, o, b->intro_dc_param));
    if (needed) *needed = (int64_t)src.size() + 1;
    if (buf && cap > 0) { snprintf(buf, (size_t)cap, "%s", src.c_str()); }
    return TSB_OK;
}
int tsb_batch_kernel_key(tsb_batch* b, const tsb_opts* opts, char* buf, int cap) {
    if (!b || !buf || cap < 33) return TSB_E_INVALID;
    tsb_opts o = resolve(opts, b->plan->p);
    std::string src = generate_source(b->plan->p, make_config(b, o, b->intro_dc_param));
    snprintf(buf, cap, "%s", source_key(src, compile_options_string(o)).c_str());
    return TSB_OK;
}

}  // extern "C"
