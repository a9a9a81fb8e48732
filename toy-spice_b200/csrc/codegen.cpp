// codegen.cpp — emits the netlist-specialised CUDA translation unit for one plan.
//
// Why specialise: every instance of a batch shares the netlist, so the stamp pattern, the pivot
// order and the fill pattern are compile-time facts.  The generated `struct Ckt` holds all per-
// instance data in arrays that are only ever indexed by literals — after inlining, ptxas keeps
// parameters, device state, the matrix and the solution vectors in registers, and the LU is a
// straight line of DFMA / DMUL / reciprocal instructions with no index arithmetic, no shared
// memory and no shuffles (one circuit per thread; the matrices are 1x1 .. ~12x12).
//
// What the generated code restates (per Newton iteration):
//   mat.Clear(); ckt.Stamp(status); mat.LoadGmin(gmin); mat.Solve()      op.go:46-65, tran.go:172-190
// with the per-device stamp arithmetic delegated to device/models.cuh and the analysis drivers
// to device/skeleton.cuh (both embedded verbatim so the unit compiles under NVRTC and nvcc alike).
#include <cstdio>
#include <algorithm>
#include <map>
#include <set>
#include <sstream>
#include <vector>
#include "tsb_internal.hpp"

namespace tsb {

static const char* k_models_src =
#include "models_src.inc"
    ;
static const char* k_skeleton_src =
#include "skeleton_src.inc"
    ;
static const char* k_coop_src =
#include "coop_src.inc"
    ;

namespace {

std::string dlit(double v) {
    char buf[64];
    if (v == (long long)v && v > -1e15 && v < 1e15) snprintf(buf, sizeof buf, "%lld.0", (long long)v);
    else snprintf(buf, sizeof buf, "%.17g", v);
    return buf;
}

struct Emitter {
    std::ostringstream os;
    int ind = 0;
    void line(const std::string& s) { for (int i = 0; i < ind; ++i) os << "    "; os << s << "\n"; }
};

const char* kind_name(int k) {
    static const char* n[] = {"R", "C", "L", "V", "I", "D", "Q", "M", "K", "LCORE"};
    return (k >= 0 && k < 10) ? n[k] : "?";
}

// o[] evaluation of one device inside a stamp routine
void emit_eval(Emitter& e, const Plan& pl, int di, const std::string& ov) {
    const Dev& d = pl.devs[di];
    std::string P = "P + " + std::to_string(d.p_off), S = "S + " + std::to_string(d.s_off);
    int no = device_num_outputs(d);
    if (no > 0) e.line("double " + ov + "[" + std::to_string(no) + "];");
    switch (d.kind) {
    case TSB_R: e.line(ov + "[0] = D[" + std::to_string(d.d_off) + "];"); break;
    case TSB_C: e.line("tsb_cap_eval(" + P + ", " + S + ", e, " + ov + ");"); break;
    case TSB_L: e.line("tsb_ind_eval(" + P + ", " + S + ", e, " + ov + ");"); break;
    case TSB_LCORE: e.line("tsb_lcore_eval(D[" + std::to_string(d.d_off) + "], e, " + ov + ");"); break;
    case TSB_D: e.line("tsb_dio_eval(" + P + ", D + " + std::to_string(d.d_off) + ", " + S + ", e, " + ov + ");"); break;
    case TSB_Q: e.line("tsb_bjt_eval(" + P + ", " + S + ", " + std::to_string(d.ip.empty() ? 0 : d.ip[0]) + ", " + ov + ");"); break;
    case TSB_M:
        e.line("tsb_mos_eval(" + P + ", " + S + ", " + std::to_string(d.ip.size() > 0 ? d.ip[0] : 1) + ", " +
               std::to_string(d.ip.size() > 1 ? d.ip[1] : 0) + ", e, " + ov + ");");
        break;
    case TSB_K: {
        int m = (int)d.ip.size(), q = 0;
        auto cur = [&](int idx) {
            const Dev& l = pl.devs[idx];
            return l.kind == TSB_LCORE ? std::string("0.0") : "S[" + std::to_string(l.s_off) + "]";
        };
        for (int i = 0; i < m; ++i)
            for (int j = i + 1; j < m; ++j, ++q)
                e.line("tsb_mut_eval(D[" + std::to_string(d.d_off + q) + "], " + cur(d.ip[i]) + ", " + cur(d.ip[j]) + ", e, " + ov +
                       " + " + std::to_string(3 * q) + ");");
        break;
    }
    default: break;
    }
}

// Targets ("A[k]" / "b[i]") written by the stamps of the listed devices.
std::set<std::string> stamp_targets(const Plan& pl, const LuProgram& lu, bool linear_only, bool op_only) {
    std::set<std::string> t;
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        if (linear_only && d.nonlinear()) continue;
        if (op_only && d.kind == TSB_K) continue;
        for (const StampEntry& s : pl.stamps[di]) {
            if (op_only && s.tran_only) continue;
            if (s.col == 0) t.insert("b[" + std::to_string(s.row) + "]");
            else {
                auto it = lu.index.find({s.row, s.col});
                if (it != lu.index.end()) t.insert("A[" + std::to_string(it->second) + "]");
            }
        }
    }
    return t;
}

// Zero-initialisation of A[] and b[] (mat.Clear()).  With `first_assign` only the entries no stamp writes are
// zeroed: the first stamp into an entry then ASSIGNS instead of accumulating onto 0.0 (emit_stamps) — ptxas cannot
// fold 0.0 + x (it is not x for x = -0.0) and the first profile showed one DADD RZ per stamped entry.  Values are
// unchanged (0.0 + x == x for every x but -0.0, whose sign no later operation of the solve can turn into a
// different number short of a division by that zero, i.e. a zero pivot, which is a failure either way), so the
// strict build uses it too; dense (BJT) builds keep the literal accumulate for their NaN / Inf bookkeeping.
void emit_clear(Emitter& e, const LuProgram& lu, int n, const std::set<std::string>* assigned) {
    for (size_t k = 0; k < lu.pos.size(); ++k) {
        std::string t = "A[" + std::to_string(k) + "]";
        if (assigned && assigned->count(t)) continue;
        e.line(t + " = 0.0;   // (" + std::to_string(lu.pos[k].first) + "," + std::to_string(lu.pos[k].second) + ")");
    }
    for (int i = 0; i <= n; ++i) {
        std::string t = "b[" + std::to_string(i) + "]";
        if (assigned && assigned->count(t)) continue;
        e.line(t + " = 0.0;");
    }
}

// Emits the stamps of the listed devices into A[] (indexed through `lu.index`) and b[].
// `deferred`: source-valued right-hand-side entries (b[row] = +-SV[slot]) that are the ONLY stamp into their row are not
// emitted here but collected (as ready-made statements) for the caller to place after the factorisation — nothing before
// the substitution reads them, so where they are assigned changes no value; a row that several stamps accumulate into
// keeps its position (the order of additions is part of the rounding).
void emit_stamps(Emitter& e, const Plan& pl, const LuProgram& lu, bool linear_only, bool op_only, bool first_assign = false,
                 std::vector<std::string>* deferred = nullptr) {
    std::set<std::string> touched;
    std::map<std::string, int> writers;
    if (deferred)
        for (int di : pl.stamp_order) {
            const Dev& d = pl.devs[di];
            if (linear_only && d.nonlinear()) continue;
            if (op_only && d.kind == TSB_K) continue;
            for (const StampEntry& s : pl.stamps[di])
                if (!(op_only && s.tran_only) && s.col == 0) ++writers["b[" + std::to_string(s.row) + "]"];
        }
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        if (linear_only && d.nonlinear()) continue;
        if (op_only && d.kind == TSB_K) continue;
        e.line("{   // " + std::string(kind_name(d.kind)) + " " + d.name);
        ++e.ind;
        std::string ov = "o";
        emit_eval(e, pl, di, ov);
        for (const StampEntry& s : pl.stamps[di]) {
            if (op_only && s.tran_only) continue;
            std::string val;
            if (s.out == -1) val = dlit(s.cval);
            else if (s.out == -2) val = "SV[" + std::to_string(d.src_slot) + "]";
            else val = ov + "[" + std::to_string(s.out) + "]";
            std::string tgt;
            if (s.col == 0) tgt = "b[" + std::to_string(s.row) + "]";
            else {
                auto it = lu.index.find({s.row, s.col});
                if (it == lu.index.end()) continue;     // cannot happen: pattern built from these entries
                tgt = "A[" + std::to_string(it->second) + "]";
            }
            const bool fresh = touched.insert(tgt).second;
            std::string stmt = (first_assign && fresh) ? tgt + (s.sign < 0 ? " = -" : " = ") + val + ";" : tgt + (s.sign < 0 ? " -= " : " += ") + val + ";";
            if (deferred && s.out == -2 && s.col == 0 && writers[tgt] == 1) deferred->push_back(stmt);
            else e.line(stmt);
        }
        --e.ind;
        e.line("}");
    }
}

// Factor + solve in the frozen order.  Same operation order per element as Sparse 1.3's
// spFactor/spSolve (u = a*(1/pivot); a_ij -= u_kj*l_ik for k ascending; forward with reciprocal
// pivots; back-substitution in ascending column order), so --fmad=false reproduces its rounding.
// `b_zero` (fast sparse builds): rows of b no stamp writes — forward / back substitution skips the operations whose
// operand is such a structural zero.  `early_cond`: condition under which a zero pivot returns before the solve.
void emit_lu(Emitter& e, const LuProgram& lu, bool load_gmin, const std::string& xout, const std::set<int>* b_zero = nullptr,
             const std::string& early_cond = "!lu_ok", const std::vector<std::string>* mid = nullptr) {
    const int n = lu.n;
    if (!lu.dense) e.line("bool lu_ok = true;");
    if (load_gmin) {
        e.line("if (gmin != 0.0) {   // LoadGmin: added to the pivot positions (Diags[i] after reordering, SURVEY Q17)");
        ++e.ind;
        for (int k = 1; k <= n; ++k) e.line("A[" + std::to_string(lu.steps[k].piv) + "] += gmin;");
        --e.ind;
        e.line("}");
    }
    for (int k = 1; k <= n; ++k) {
        const LuProgram::Step& st = lu.steps[k];
        std::string piv = "A[" + std::to_string(st.piv) + "]";
        e.line("// step " + std::to_string(k) + ": pivot (" + std::to_string(lu.prow[k]) + "," + std::to_string(lu.pcol[k]) + ")");
        // zero pivot = the reference's "matrix factorization failed".  Sparse builds test all pivots with ONE
        // branch after the elimination (a zero pivot only produces Inf/NaN in values that are then discarded);
        // the dense (BJT) build returns at once, as the reference does.
        if (lu.dense) e.line("if (" + piv + " == 0.0) return false;");
        else e.line("lu_ok = lu_ok & (" + piv + " != 0.0);");
        // dense (BJT) builds: Inf / NaN pivots must give what IEEE gives the reference (1/Inf = 0, NaN stays NaN) — tsb_qdiv keeps
        // the special values (the hardware seed wherever the correction did not converge) without the compiler's division
        // sequence, whose slow path is a CALL for every non-finite operand: 11.8 calls per accepted step on bjt2.cir, where
        // 99.8 % of the instances overflow to NaN as in the reference (r02_notes section 10)
        e.line(piv + " = " + std::string(lu.dense ? "tsb_qdiv(1.0, " + piv + ")" : "tsb_rcp(" + piv + ")") + ";");
        for (size_t ui = 0; ui < st.urow.size(); ++ui) {
            std::string u = "A[" + std::to_string(st.urow[ui]) + "]";
            e.line(u + " *= " + piv + ";");
            for (size_t li = 0; li < st.lcol.size(); ++li)
                e.line("A[" + std::to_string(st.target[ui][li]) + "] -= " + u + " * A[" + std::to_string(st.lcol[li]) + "];");
        }
    }
    if (!lu.dense) e.line("if (" + early_cond + ") return false;");
    if (mid) for (const std::string& st : *mid) e.line(st);
    e.line("double c[" + std::to_string(n + 1) + "];");
    std::vector<char> cz(n + 1, 0);          // c[k] is a structural zero so far
    for (int k = 1; k <= n; ++k) {
        cz[k] = (b_zero && !lu.dense && b_zero->count(lu.prow[k])) ? 1 : 0;
        e.line("c[" + std::to_string(k) + "] = " + (cz[k] ? std::string("0.0") : "b[" + std::to_string(lu.prow[k]) + "]") + ";");
    }
    for (int k = 1; k <= n; ++k) {
        const LuProgram::Step& st = lu.steps[k];
        std::string ck = "c[" + std::to_string(k) + "]";
        if (cz[k]) continue;
        if (lu.dense) { e.line("if (" + ck + " != 0.0) {"); ++e.ind; }
        e.line(ck + " *= A[" + std::to_string(st.piv) + "];");
        for (size_t li = 0; li < st.lcol.size(); ++li) {
            int j = st.lrow_step[li];
            std::string prod = ck + " * A[" + std::to_string(st.lcol[li]) + "]";
            if (cz[j]) { e.line("c[" + std::to_string(j) + "] = -(" + prod + ");"); cz[j] = 0; }
            else e.line("c[" + std::to_string(j) + "] -= " + prod + ";");
        }
        if (lu.dense) { --e.ind; e.line("}"); }
    }
    for (int k = n; k >= 1; --k) {
        const LuProgram::Step& st = lu.steps[k];
        for (size_t ui = 0; ui < st.urow.size(); ++ui) {
            int j = st.ucol_step[ui];
            if (cz[j]) continue;
            std::string prod = "A[" + std::to_string(st.urow[ui]) + "] * c[" + std::to_string(j) + "]";
            if (cz[k]) { e.line("c[" + std::to_string(k) + "] = -(" + prod + ");"); cz[k] = 0; }
            else e.line("c[" + std::to_string(k) + "] -= " + prod + ";");
        }
    }
    for (int k = 1; k <= n; ++k) e.line(xout + "[" + std::to_string(lu.pcol[k]) + "] = c[" + std::to_string(k) + "];");
}


// ---- transient solves of the fast build: static condensation (plan.cpp: build_tranfast) ---------------------------------
// The elimination program of pl.lu_tf is split in two by what each operation depends on:
//   prefactor()            every operation whose operands are invariant over the run (resistor conductances, +-1 incidence
//                          entries and whatever the elimination makes of them) — executed once per instance; the values
//                          later operations need are kept in AI[];
//   assemble_solve_tf()    the operations with at least one operand that changes from solve to solve (companion
//                          conductances C/dt, L/dt, M/dt, nonlinear stamps, the right-hand side), reading invariant operands
//                          from AI[].  An entry that collects invariant and variant contributions starts each solve from its
//                          invariant part (AI[]) — a re-association the fast build is allowed.
// Entry names: "T[k]" inside prefactor, "AI[q]" / "A[k]" inside the solve.
struct TfSplit {
    const Plan& pl;
    const LuProgram& lu;
    Emitter pre, step;
    std::vector<char> inv;            // entry k is (still) invariant
    std::vector<char> has_base;       // entry k has an invariant part computed in prefactor (T[k] is meaningful)
    std::vector<char> step_init;      // A[k] has been assigned in the per-solve code
    std::map<int, int> ai_slot;       // entry k -> AI index (value copied out of T[k] at the end of prefactor)
    int n_ai = 0;
    std::vector<char> base_final;     // (second pass) entry k ends up with an invariant part: decides how a solve initialises A[k]
    std::map<int, double> lit;        // T[k] currently holds this literal (+-1 incidence entries): rcp and products fold
    TfSplit(const Plan& p) : pl(p), lu(p.lu_tf), inv(p.lu_tf.pos.size(), 1), has_base(p.lu_tf.pos.size(), 0), step_init(p.lu_tf.pos.size(), 0) {
        for (size_t k = 0; k < lu.pos.size(); ++k) if (k < pl.tf_variant.size() && pl.tf_variant[k]) inv[k] = 0;
    }
    std::string T(int k) const { return "T[" + std::to_string(k) + "]"; }
    std::string A(int k) const { return "A[" + std::to_string(k) + "]"; }
    std::string AI(int k) {          // invariant operand of a per-solve operation
        auto it = ai_slot.find(k);
        if (it == ai_slot.end()) it = ai_slot.emplace(k, n_ai++).first;
        return "AI[" + std::to_string(it->second) + "]";
    }
    std::string opnd(int k) { return inv[k] ? AI(k) : A(k); }
    // first per-solve touch of a variant entry: start from its invariant part if it has one
    void ensure_init(int k) {
        if (step_init[k]) return;
        step_init[k] = 1;
        step.line(A(k) + " = " + (based(k) ? AI(k) : std::string("0.0")) + ";");
    }
    bool based(int k) const { return base_final.empty() ? has_base[k] != 0 : base_final[k] != 0; }
    // variant update A[k] -= expr (or first assignment)
    void sub_variant(int k, const std::string& expr) {
        if (!step_init[k] && !based(k)) { step_init[k] = 1; step.line(A(k) + " = -(" + expr + ");"); return; }
        ensure_init(k);
        step.line(A(k) + " -= " + expr + ";");
    }
};

void tranfast_walk(TfSplit& sp, const Plan& pl, std::vector<std::string>& late, std::set<std::string>& b_touched);

void emit_tranfast(Emitter& e, const Plan& pl, const CodegenConfig& cfg) {
    const LuProgram& lu = pl.lu_tf;
    const int n = lu.n;
    std::vector<char> base_final;
    {   // first pass: which entries end up with an invariant part
        TfSplit dry(pl);
        std::vector<std::string> l0; std::set<std::string> b0;
        tranfast_walk(dry, pl, l0, b0);
        base_final = dry.has_base;
    }
    TfSplit sp(pl);
    sp.base_final = base_final;
    sp.pre.ind = 2; sp.step.ind = 2;
    std::vector<std::string> late;
    std::set<std::string> b_touched;
    tranfast_walk(sp, pl, late, b_touched);
    // ---- substitution (always per solve: the right-hand side changes) ---------------------------------------------------
    Emitter& se = sp.step;
    se.line("if (EARLY && !lu_ok) return false;");
    se.line("mid();");
    for (const std::string& stt : late) se.line(stt);
    std::set<int> bz;
    for (int i = 1; i <= n; ++i) if (!b_touched.count("b[" + std::to_string(i) + "]")) bz.insert(i);
    se.line("double c[" + std::to_string(n + 1) + "];");
    std::vector<char> cz(n + 1, 0);
    for (int k = 1; k <= n; ++k) {
        cz[k] = bz.count(lu.prow[k]) ? 1 : 0;
        se.line("c[" + std::to_string(k) + "] = " + (cz[k] ? std::string("0.0") : "b[" + std::to_string(lu.prow[k]) + "]") + ";");
    }
    for (int k = 1; k <= n; ++k) {
        const LuProgram::Step& st = lu.steps[k];
        std::string ck = "c[" + std::to_string(k) + "]";
        if (cz[k]) continue;
        se.line(ck + " *= " + sp.opnd(st.piv) + ";");
        for (size_t li = 0; li < st.lcol.size(); ++li) {
            int j = st.lrow_step[li];
            std::string prod = ck + " * " + sp.opnd(st.lcol[li]);
            if (cz[j]) { se.line("c[" + std::to_string(j) + "] = -(" + prod + ");"); cz[j] = 0; }
            else se.line("c[" + std::to_string(j) + "] -= " + prod + ";");
        }
    }
    for (int k = n; k >= 1; --k) {
        const LuProgram::Step& st = lu.steps[k];
        for (size_t ui = 0; ui < st.urow.size(); ++ui) {
            int j = st.ucol_step[ui];
            if (cz[j]) continue;
            std::string prod = sp.opnd(st.urow[ui]) + " * c[" + std::to_string(j) + "]";
            if (cz[k]) { se.line("c[" + std::to_string(k) + "] = -(" + prod + ");"); cz[k] = 0; }
            else se.line("c[" + std::to_string(k) + "] -= " + prod + ";");
        }
    }
    for (int k = 1; k <= n; ++k) se.line("x[" + std::to_string(lu.pcol[k]) + "] = c[" + std::to_string(k) + "];");
    se.line("return lu_ok;");

    // ---- assemble the two member functions --------------------------------------------------------------------------------
    e.line("double AI[" + std::to_string(std::max(1, sp.n_ai)) + "];   // invariant factors / invariant parts of the condensed transient elimination");
    e.line("bool pf_ok;");
    e.line("// once per instance, after load(): everything of the transient elimination that does not change during the run");
    e.line("__device__ __forceinline__ void prefactor() {");
    ++e.ind;
    e.line("double T[" + std::to_string(lu.pos.size()) + "];");
    e.line("pf_ok = true;");
    e.os << sp.pre.os.str();
    for (auto& kv : sp.ai_slot) e.line("AI[" + std::to_string(kv.second) + "] = T[" + std::to_string(kv.first) + "];");
    --e.ind;
    e.line("}");
    e.line("// one transient solve: stamps and elimination of what changes, substitution.  `mid` as in assemble_solve.");
    e.line("template <bool EARLY, class Mid>");
    e.line("__device__ __forceinline__ bool assemble_solve_tf(double time, double dt, double rdt, Mid mid) {");
    ++e.ind;
    e.line("TsbEnv e; e.mode = TSB_MODE_TRAN; e.time = time; e.dt = dt; e.gmin = 0.0; e.rdt = rdt;");
    e.line("double A[" + std::to_string(lu.pos.size()) + "];");
    e.line("double b[" + std::to_string(n + 1) + "];");
    e.os << sp.step.os.str();
    --e.ind;
    e.line("}");
    (void)cfg;
}

void tranfast_walk(TfSplit& sp, const Plan& pl, std::vector<std::string>& late, std::set<std::string>& b_touched) {
    const LuProgram& lu = pl.lu_tf;
    const int n = lu.n;
    // ---- stamps: invariant ones into T[] (prefactor), variant ones into A[] (solve) --------------------------------------
    // (`late`: source-valued right-hand sides, placed after the factorisation)
    std::map<std::string, int> rhs_writers;
    for (int di : pl.stamp_order)
        for (const StampEntry& s : pl.stamps[di]) if (s.col == 0) ++rhs_writers["b[" + std::to_string(s.row) + "]"];
    std::set<int> pre_touched;
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        bool any_var = false, any_inv = false;
        for (const StampEntry& s : pl.stamps[di]) {
            const bool v = s.col == 0 || !(d.kind == TSB_R || d.kind == TSB_V || d.kind == TSB_I || ((d.kind == TSB_L || d.kind == TSB_LCORE) && s.out == -1));
            (v ? any_var : any_inv) = true;
        }
        if (any_inv) {
            sp.pre.line("{   // " + std::string(kind_name(d.kind)) + " " + d.name);
            ++sp.pre.ind;
            if (d.kind == TSB_R) sp.pre.line("const double o0 = D[" + std::to_string(d.d_off) + "];");
            for (const StampEntry& s : pl.stamps[di]) {
                if (s.col == 0) continue;
                const bool v = !(d.kind == TSB_R || d.kind == TSB_V || d.kind == TSB_I || ((d.kind == TSB_L || d.kind == TSB_LCORE) && s.out == -1));
                if (v) continue;
                const int k = lu.index.at({s.row, s.col});
                std::string val = s.out == -1 ? dlit(s.cval) : std::string("o0");
                if (pre_touched.insert(k).second) {
                    sp.pre.line(sp.T(k) + (s.sign < 0 ? " = -" : " = ") + val + ";");
                    if (s.out == -1) sp.lit[k] = s.sign * s.cval;
                } else { sp.pre.line(sp.T(k) + (s.sign < 0 ? " -= " : " += ") + val + ";"); sp.lit.erase(k); }
                sp.has_base[k] = 1;
            }
            --sp.pre.ind;
            sp.pre.line("}");
        }
        if (any_var) {
            sp.step.line("{   // " + std::string(kind_name(d.kind)) + " " + d.name);
            ++sp.step.ind;
            if (d.kind != TSB_R) emit_eval(sp.step, pl, di, "o");
            for (const StampEntry& s : pl.stamps[di]) {
                const bool v = s.col == 0 || !(d.kind == TSB_R || d.kind == TSB_V || d.kind == TSB_I || ((d.kind == TSB_L || d.kind == TSB_LCORE) && s.out == -1));
                if (!v) continue;
                std::string val = s.out == -1 ? dlit(s.cval) : (s.out == -2 ? "SV[" + std::to_string(d.src_slot) + "]" : "o[" + std::to_string(s.out) + "]");
                if (s.col == 0) {
                    std::string tgt = "b[" + std::to_string(s.row) + "]";
                    const bool fresh = b_touched.insert(tgt).second;
                    std::string stmt = fresh ? tgt + (s.sign < 0 ? " = -" : " = ") + val + ";" : tgt + (s.sign < 0 ? " -= " : " += ") + val + ";";
                    if (s.out == -2 && rhs_writers[tgt] == 1) late.push_back(stmt); else sp.step.line(stmt);
                } else {
                    const int k = lu.index.at({s.row, s.col});
                    if (!sp.step_init[k] && !sp.based(k)) { sp.step_init[k] = 1; sp.step.line(sp.A(k) + (s.sign < 0 ? " = -" : " = ") + val + ";"); }
                    else { sp.ensure_init(k); sp.step.line(sp.A(k) + (s.sign < 0 ? " -= " : " += ") + val + ";"); }
                }
            }
            --sp.step.ind;
            sp.step.line("}");
        }
    }
    // entries nothing stamps and nothing invariant has touched yet start at zero in prefactor (fill-in)
    // ---- elimination ---------------------------------------------------------------------------------------------------
    sp.step.line("bool lu_ok = pf_ok;");
    for (int k = 1; k <= n; ++k) {
        const LuProgram::Step& st = lu.steps[k];
        const int p = st.piv;
        if (sp.inv[p]) {
            if (!sp.has_base[p]) { sp.pre.line(sp.T(p) + " = 0.0;"); sp.has_base[p] = 1; }
            if (sp.lit.count(p) && (sp.lit[p] == 1.0 || sp.lit[p] == -1.0)) {
                // a +-1 incidence pivot: its reciprocal is itself (kept a literal so that the products below fold away)
            } else {
                sp.pre.line("pf_ok = pf_ok & (" + sp.T(p) + " != 0.0);");
                sp.pre.line(sp.T(p) + " = tsb_rcp(" + sp.T(p) + ");");
                sp.lit.erase(p);
            }
        } else {
            sp.ensure_init(p);
            sp.step.line("lu_ok = lu_ok & (" + sp.A(p) + " != 0.0);");
            sp.step.line(sp.A(p) + " = tsb_rcp(" + sp.A(p) + ");");
        }
        for (size_t ui = 0; ui < st.urow.size(); ++ui) {
            const int u = st.urow[ui];
            if (sp.inv[u] && !sp.has_base[u]) { sp.pre.line(sp.T(u) + " = 0.0;"); sp.has_base[u] = 1; }
            if (sp.inv[u] && sp.inv[p]) {
                if (sp.lit.count(p) && sp.lit[p] == 1.0) { /* u * 1 */ }
                else if (sp.lit.count(p) && sp.lit[p] == -1.0) { sp.pre.line(sp.T(u) + " = -" + sp.T(u) + ";"); if (sp.lit.count(u)) sp.lit[u] = -sp.lit[u]; }
                else { sp.pre.line(sp.T(u) + " *= " + sp.T(p) + ";"); sp.lit.erase(u); }
            }
            else {
                if (sp.inv[u]) { sp.inv[u] = 0; sp.step_init[u] = 1; sp.step.line(sp.A(u) + " = " + sp.AI(u) + " * " + sp.opnd(p) + ";"); }
                else { sp.ensure_init(u); sp.step.line(sp.A(u) + " *= " + sp.opnd(p) + ";"); }
            }
            for (size_t li = 0; li < st.lcol.size(); ++li) {
                const int l = st.lcol[li], t = st.target[ui][li];
                if (sp.inv[l] && !sp.has_base[l]) { sp.pre.line(sp.T(l) + " = 0.0;"); sp.has_base[l] = 1; }
                if (sp.inv[u] && sp.inv[l]) {
                    // invariant product: into the invariant part of the target, whether the target stays invariant or not
                    if (!sp.has_base[t]) { sp.pre.line(sp.T(t) + " = -(" + sp.T(u) + " * " + sp.T(l) + ");"); sp.has_base[t] = 1; }
                    else sp.pre.line(sp.T(t) + " -= " + sp.T(u) + " * " + sp.T(l) + ";");
                    sp.lit.erase(t);
                } else {
                    sp.inv[t] = 0;
                    sp.sub_variant(t, sp.opnd(u) + " * " + sp.opnd(l));
                }
            }
        }
    }
}

// ---- AC analysis (ac.go:51-98): one complex solve per frequency, linear circuits ------------------------------------------
// Complex entries as (Ar[k], Ai[k]); the elimination program is pl.lu_ac: the reference's order (its complex matrix is
// factored first during the operating point that precedes the sweep, with real values) over the StampAC pattern.
void emit_ac(Emitter& e, const Plan& pl) {
    const LuProgram& lu = pl.lu_ac;
    const int n = lu.n;
    auto S = [](int k) { return std::to_string(k); };
    e.line("// mat.Clear(); ckt.Stamp(status{Mode: ACAnalysis, Frequency}); mat.Solve()  ->  xr + j*xi   (ac.go:57-71)");
    e.line("__device__ __forceinline__ bool solve_ac(double omega, double* xr, double* xi) {");
    ++e.ind;
    e.line("double Ar[" + S((int)lu.pos.size()) + "], Ai[" + S((int)lu.pos.size()) + "], br[" + S(n + 1) + "], bi[" + S(n + 1) + "];");
    for (size_t k = 0; k < lu.pos.size(); ++k) e.line("Ar[" + S((int)k) + "] = 0.0; Ai[" + S((int)k) + "] = 0.0;");
    for (int i = 0; i <= n; ++i) e.line("br[" + S(i) + "] = 0.0; bi[" + S(i) + "] = 0.0;");
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        std::vector<AcEntry> ae;
        device_ac_entries(pl, di, ae);
        e.line("{   // " + std::string(kind_name(d.kind)) + " " + d.name);
        ++e.ind;
        for (const AcEntry& a : ae) {
            const std::string k = S(lu.index.at({a.row, a.col}));
            const std::string sg = a.sign < 0 ? " -= " : " += ";
            switch (a.code) {
            case 0: e.line("Ar[" + k + "]" + sg + "D[" + S(d.d_off) + "];"); break;
            case 1: e.line("Ai[" + k + "]" + sg + "omega * (P[" + S(d.p_off) + "] * 1.0);"); break;
            case 2: e.line("Ai[" + k + "]" + sg + "omega * P[" + S(d.p_off) + "];"); break;
            default: e.line("Ar[" + k + "]" + sg + "1.0;"); break;
            }
        }
        // right-hand sides: AC magnitude / phase of the sources (vsource.go:160-176, isource.go:149-165)
        if ((d.kind == TSB_V || d.kind == TSB_I) && d.src_type() == TSB_SRC_DC && d.p.size() >= 3) {
            e.line("const double ph = P[" + S(d.p_off + 2) + "] * TSB_PI / 180.0;");
            e.line("const double re = P[" + S(d.p_off + 1) + "] * cos(ph), im = P[" + S(d.p_off + 1) + "] * tsb_go_sin(ph);");
            if (d.kind == TSB_V) e.line("br[" + S(d.branch) + "] += re; bi[" + S(d.branch) + "] += im;");
            else {
                if (d.nodes[0] != 0) e.line("br[" + S(d.nodes[0]) + "] += re; bi[" + S(d.nodes[0]) + "] += im;");
                if (d.nodes[1] != 0) e.line("br[" + S(d.nodes[1]) + "] -= re; bi[" + S(d.nodes[1]) + "] -= im;");
            }
        }
        --e.ind;
        e.line("}");
    }
    e.line("double tr, ti;");
    for (int k = 1; k <= n; ++k) {
        const LuProgram::Step& st = lu.steps[k];
        const std::string p = S(st.piv);
        e.line("// step " + S(k) + ": pivot (" + S(lu.prow[k]) + "," + S(lu.pcol[k]) + ")");
        e.line("if (Ar[" + p + "] == 0.0 && Ai[" + p + "] == 0.0) return false;   // \"matrix factorization failed\"");
        e.line("tsb_crcp(Ar[" + p + "], Ai[" + p + "]);");
        for (size_t ui = 0; ui < st.urow.size(); ++ui) {
            const std::string u = S(st.urow[ui]);
            e.line("tr = Ar[" + u + "] * Ar[" + p + "] - Ai[" + u + "] * Ai[" + p + "]; ti = Ar[" + u + "] * Ai[" + p + "] + Ai[" + u + "] * Ar[" + p + "]; Ar[" + u + "] = tr; Ai[" + u + "] = ti;");
            for (size_t li = 0; li < st.lcol.size(); ++li) {
                const std::string l = S(st.lcol[li]), t = S(st.target[ui][li]);
                e.line("Ar[" + t + "] -= Ar[" + u + "] * Ar[" + l + "] - Ai[" + u + "] * Ai[" + l + "]; Ai[" + t + "] -= Ar[" + u + "] * Ai[" + l + "] + Ai[" + u + "] * Ar[" + l + "];");
            }
        }
    }
    e.line("double cr[" + S(n + 1) + "], ci[" + S(n + 1) + "];");
    for (int k = 1; k <= n; ++k) e.line("cr[" + S(k) + "] = br[" + S(lu.prow[k]) + "]; ci[" + S(k) + "] = bi[" + S(lu.prow[k]) + "];");
    for (int k = 1; k <= n; ++k) {
        const LuProgram::Step& st = lu.steps[k];
        const std::string p = S(st.piv), ck = S(k);
        e.line("tr = cr[" + ck + "] * Ar[" + p + "] - ci[" + ck + "] * Ai[" + p + "]; ti = cr[" + ck + "] * Ai[" + p + "] + ci[" + ck + "] * Ar[" + p + "]; cr[" + ck + "] = tr; ci[" + ck + "] = ti;");
        for (size_t li = 0; li < st.lcol.size(); ++li) {
            const std::string j = S(st.lrow_step[li]), l = S(st.lcol[li]);
            e.line("cr[" + j + "] -= cr[" + ck + "] * Ar[" + l + "] - ci[" + ck + "] * Ai[" + l + "]; ci[" + j + "] -= cr[" + ck + "] * Ai[" + l + "] + ci[" + ck + "] * Ar[" + l + "];");
        }
    }
    for (int k = n; k >= 1; --k) {
        const LuProgram::Step& st = lu.steps[k];
        for (size_t ui = 0; ui < st.urow.size(); ++ui) {
            const std::string j = S(st.ucol_step[ui]), u = S(st.urow[ui]), ck = S(k);
            e.line("cr[" + ck + "] -= Ar[" + u + "] * cr[" + j + "] - Ai[" + u + "] * ci[" + j + "]; ci[" + ck + "] -= Ar[" + u + "] * ci[" + j + "] + Ai[" + u + "] * cr[" + j + "];");
        }
    }
    for (int k = 1; k <= n; ++k) e.line("xr[" + S(lu.pcol[k]) + "] = cr[" + S(k) + "]; xi[" + S(lu.pcol[k]) + "] = ci[" + S(k) + "];");
    e.line("return true;");
    --e.ind;
    e.line("}");
    // result row of one frequency (ac.go:73-95, StoreACResult anlysis.go:87-111): magnitude = cmplx.Abs, phase in degrees
    // refread: GetComplexSolution(i) = (solution[i], solution[i+Size]) taken literally over Sparse 1.3's interleaved vector
    // (solution[2i] = re x_i, solution[2i+1] = im x_i, entries 0 and 1 unused), matrix/circuit.go:168-173 vs :41-44
    e.line("__device__ __forceinline__ void signals_ac(const double* xr, const double* xi, bool refread, double* out) const {");
    ++e.ind;
    int c = 0;
    auto flat = [&](int q) -> std::string {            // entry q of the interleaved vector
        if (q < 2 || q > 2 * n + 1) return "0.0";
        return std::string(q % 2 == 0 ? "xr[" : "xi[") + S(q / 2) + "]";
    };
    auto emit_mp = [&](int idx) {
        e.line("{ const double re = refread ? " + flat(idx) + " : xr[" + S(idx) + "], im = refread ? " + flat(idx + n) + " : xi[" + S(idx) + "];");
        e.line("  out[" + S(c) + "] = tsb_go_hypot(re, im); out[" + S(c + 1) + "] = atan2(im, re) * 180.0 / TSB_PI; }");
        c += 2;
    };
    for (int i = 1; i <= pl.n_nodes; ++i) emit_mp(i);
    for (const Dev& d : pl.devs) if (d.kind == TSB_V) emit_mp(d.branch);
    --e.ind;
    e.line("}");
}


// ---- cooperative mapping (CoopPlan, device/coop.cuh): one struct per part ----------------------------------------------------
// The elimination program cp.lu is in nested-dissection order: steps 1..n_int eliminate the interiors (part 0's first),
// the rest the separator.  Part p emits, for a solve,
//   phase_a   the stamps of the devices it owns, the elimination steps of its interior, the forward substitution of its
//             interior; what these add to separator entries / separator right-hand sides is its CONTRIBUTION, written to the
//             exchange buffer (one slot per contributed value);
//   phase_b   (after the barrier) the separator system summed over the contributions of all parts in part order — the same
//             additions in the same order in every part, so every part holds the same bits — eliminated and solved by every
//             part for itself, then the back substitution of the part's own interior.
// Structural zeros are tracked symbolically per part (an entry no own device stamps and no own step fills does not exist
// for that part), so a part touches only what its sub-circuit makes non-zero.
struct CoopSym {
    std::vector<int> devs;                 // own devices, stamp order
    std::set<int> a_assigned, b_assigned;  // entries / rhs rows stamped by own devices
    std::set<int> touched;                 // entries structurally non-zero in this part's view after its own elimination
    std::vector<int> steps;                // own elimination steps, ascending
    std::vector<int> xe, xc;               // contributed separator entries / separator steps with a rhs contribution
    std::set<int> cnz;                     // steps (own and separator) whose c[] is structurally non-zero after the own forward pass
    std::vector<int> cols;                 // own result columns, ascending (part 0: column 0 = TIME first)
};

static const int COOP_HDR = 3;             // exchange slots 0 (flags of phase_a), 1 (result-store key, part 0), 2 (flags of phase_b: Newton loops)

void coop_analyse(const Plan& pl, const CoopPlan& cp, std::vector<CoopSym>& sym, int& nx) {
    const LuProgram& lu = cp.lu;
    const int n = lu.n;
    sym.assign(cp.parts, CoopSym());
    for (int di : pl.stamp_order) sym[cp.dev_owner[di]].devs.push_back(di);
    for (int k = 1; k <= n; ++k) if (cp.step_owner[k] >= 0) sym[cp.step_owner[k]].steps.push_back(k);
    for (size_t c = 0; c < cp.col_owner.size(); ++c) sym[cp.col_owner[c]].cols.push_back((int)c);
    auto is_sep_entry = [&](int e) { return cp.owner[lu.pos[e].first] < 0 && cp.owner[lu.pos[e].second] < 0; };
    nx = COOP_HDR;
    for (int p = 0; p < cp.parts; ++p) {
        CoopSym& y = sym[p];
        for (int di : y.devs)
            for (const StampEntry& s : pl.stamps[di]) {
                if (s.col == 0) y.b_assigned.insert(s.row);
                else y.a_assigned.insert(lu.index.at({s.row, s.col}));
            }
        y.touched = y.a_assigned;
        for (int k : y.steps) {
            const LuProgram::Step& st = lu.steps[k];
            for (size_t ui = 0; ui < st.urow.size(); ++ui) {
                if (!y.touched.count(st.urow[ui])) continue;
                for (size_t li = 0; li < st.lcol.size(); ++li) if (y.touched.count(st.lcol[li])) y.touched.insert(st.target[ui][li]);
            }
        }
        for (int e : y.touched) if (is_sep_entry(e)) y.xe.push_back(e);
        for (int k = 1; k <= n; ++k) if (y.b_assigned.count(lu.prow[k]) && (cp.step_owner[k] == p || cp.step_owner[k] < 0)) y.cnz.insert(k);
        for (int k : y.steps) {
            if (!y.cnz.count(k)) continue;
            const LuProgram::Step& st = lu.steps[k];
            for (size_t li = 0; li < st.lcol.size(); ++li) if (y.touched.count(st.lcol[li])) y.cnz.insert(st.lrow_step[li]);
        }
        for (int k = cp.n_int + 1; k <= n; ++k) if (y.cnz.count(k)) y.xc.push_back(k);
        nx = std::max(nx, COOP_HDR + (int)y.xe.size() + (int)y.xc.size());
    }
}

void emit_coop(Emitter& e, const Plan& pl, const CoopPlan& cp, const CodegenConfig& cfg) {
    const LuProgram& lu = cp.lu;
    const int n = lu.n, NP = cp.parts;
    auto S = [](int k) { return std::to_string(k); };
    std::vector<CoopSym> sym;
    int nx = 0;
    coop_analyse(pl, cp, sym, nx);
    int nown_max = 0;
    for (const CoopSym& y : sym) nown_max = std::max(nown_max, (int)y.cols.size());
    e.line("#define TSB_COOP_PARTS " + S(NP));
    e.line("#define TSB_COOP_NX " + S(nx) + "          // exchange slots per part and attempt");
    e.line("#define TSB_COOP_NOWN_MAX " + S(nown_max) + "   // result columns of the widest part");
    e.line("#define TSB_COOP_NCOL " + S((int)cp.col_owner.size()));
    e.line("#define TSB_COOP_NL " + std::string(pl.has_nonlinear ? "1" : "0") + "            // Newton loop (two barriers per iteration) / one solve per step");
    // the separator system after the gather: which entries / right-hand sides exist, for every part alike
    std::set<int> sep_touched, sep_cnz;
    for (const CoopSym& y : sym) { sep_touched.insert(y.xe.begin(), y.xe.end()); sep_cnz.insert(y.xc.begin(), y.xc.end()); }
    for (int p = 0; p < NP; ++p) {
        const CoopSym& y = sym[p];
        Plan sub = pl;                          // same numbering, own devices only: the stamp emitters work unchanged
        sub.stamp_order = y.devs;
        e.line("struct CoopPart" + S(p) + " {");
        ++e.ind;
        e.line("static constexpr int PART = " + S(p) + ", NOWN = " + S((int)y.cols.size()) + ", N = " + S(n) + ";");
        e.line("double xo[" + S(n + 1) + "];   // oldSolution of the Newton loop (circuits with nonlinear devices)");
        e.line("double P[" + S(std::max(1, pl.n_params)) + "], S[" + S(std::max(1, pl.n_state)) + "], D[" + S(std::max(1, pl.n_derived)) + "], SV[" +
               S(std::max(1, pl.n_src)) + "], x[" + S(n + 1) + "];     // global numbering; only this part's elements are ever touched");
        e.line("double A[" + S((int)lu.pos.size()) + "], c[" + S(n + 1) + "];   // factors / substitution vector kept from phase_a to phase_b");
        e.line("const double* U_;");
        e.line("__device__ __forceinline__ int col(int j) const {");
        {
            std::string tab;
            for (size_t j = 0; j < y.cols.size(); ++j) tab += (j ? ", " : "") + S(y.cols[j]);
            e.line("    constexpr int C[" + S(std::max<size_t>(1, y.cols.size())) + "] = {" + (tab.empty() ? "0" : tab) + "};");
            e.line("    return C[j];");
        }
        e.line("}");
        // ---- load: own parameters, derived values, the state the operating point left (tsb_optran's hand-over) ----
        e.line("__device__ __forceinline__ void load(const TsbArgs& a, long long inst) {");
        ++e.ind;
        e.line("U_ = a.U;");
        for (int di : y.devs) {
            const Dev& d = pl.devs[di];
            if (!((d.kind == TSB_V || d.kind == TSB_I) && d.src_type() == TSB_SRC_PWL))
                for (size_t j = 0; j < d.p.size(); ++j) {
                    int k = d.p_off + (int)j;
                    if (cfg.varying[k]) e.line("P[" + S(k) + "] = __ldcs(a.pv[" + S(cfg.var_slot[k]) + "] + inst);   // " + d.name + " p" + S((int)j));
                    else e.line("P[" + S(k) + "] = a." + (k < 32 ? "Uc[" : "U[") + S(k) + "];");
                }
            std::string P = "P + " + S(d.p_off);
            if (d.kind == TSB_R) e.line("D[" + S(d.d_off) + "] = tsb_res_g(" + P + ");");
            else if (d.kind == TSB_L) e.line("tsb_ind_derive(" + P + ", D + " + S(d.d_off) + ");");
            else if (d.kind == TSB_LCORE) e.line("D[" + S(d.d_off) + "] = tsb_lcore_L0(" + P + ");");
            else if (d.kind == TSB_D) e.line("tsb_dio_derive(" + P + ", D + " + S(d.d_off) + ");");
            for (int q = 0; q < d.n_state; ++q) e.line("S[" + S(d.s_off + q) + "] = a.coop_state[(long long)" + S(d.s_off + q) + " * a.n_inst + inst];");
            if (d.src_slot >= 0) e.line("SV[" + S(d.src_slot) + "] = 0.0;");
        }
        for (int u = 1; u <= n; ++u)
            if (cp.owner[u] == p || cp.owner[u] < 0) e.line("x[" + S(u) + "] = a.coop_state[(long long)" + S(pl.n_state + u) + " * a.n_inst + inst]; xo[" + S(u) + "] = x[" + S(u) + "];");
        e.line("x[0] = 0.0; xo[0] = 0.0;");
        --e.ind;
        e.line("}");
        // ---- sources --------------------------------------------------------------------------------------------
        for (int nb = 0; nb < 2; ++nb) {
            e.line(nb ? "__device__ __forceinline__ bool eval_sources_nb(double t) {" : "__device__ __forceinline__ void eval_sources(double t, double fac) {");
            ++e.ind;
            if (nb) e.line("bool ok = true;");
            for (int di : y.devs) {
                const Dev& d = pl.devs[di];
                if (d.src_slot < 0) continue;
                std::string sv = "SV[" + S(d.src_slot) + "]", P = "P + " + S(d.p_off);
                std::string fac = nb ? "1.0" : (d.kind == TSB_V ? "fac" : "1.0");
                switch (d.src_type()) {
                case TSB_SRC_DC: e.line(sv + " = P[" + S(d.p_off) + "] * " + fac + ";"); break;
                case TSB_SRC_SIN: e.line(sv + (nb ? " = tsb_src_sin_nb(" + P + ", t, ok);" : " = tsb_src_sin(" + P + ", t, " + fac + ");")); break;
                case TSB_SRC_PULSE: e.line(sv + " = tsb_src_pulse(" + P + ", t);"); break;
                case TSB_SRC_PWL: e.line(sv + " = tsb_src_pwl(U_ + " + S(d.p_off) + ", " + S((int)d.p.size() / 2) + ", t);"); break;
                }
            }
            e.line(nb ? "(void)t; return ok;" : "(void)t; (void)fac;");
            --e.ind;
            e.line("}");
        }
        // ---- truncation-error decisions of the own devices (Ckt::lte_flags restricted; OR / AND over parts is exact) ----
        e.line("__device__ __forceinline__ void lte_flags(double dt, double rdt, double trtol, double thr, bool& gt, bool& small) {");
        ++e.ind;
        e.line("gt = false; small = 0.0 < thr;");
        e.line("double trtol2 = trtol, thr2 = thr; TSB_OPAQUE(trtol2); TSB_OPAQUE(thr2);");
        for (int di : y.devs) {
            const Dev& d = pl.devs[di];
            if (d.kind == TSB_C)
                e.line("{ const double l = tsb_cap_lte(P + " + S(d.p_off) + ", S + " + S(d.s_off) + ", dt, rdt); gt = gt | (l > trtol); small = small & !(l >= thr); }");
            else if (d.kind == TSB_L) {
                e.line("{ double cu, vo; tsb_ind_lte2(S + " + S(d.s_off) + ", dt, rdt, cu, vo);");
                e.line("  const bool nan = ((cu != cu) | (vo != vo)) & !((cu == TSB_INF) | (vo == TSB_INF));");
                e.line("  gt = gt | (!nan & ((cu > trtol) | (vo > trtol2))); small = small & !(!nan & ((cu >= thr) | (vo >= thr2))); }");
            }
        }
        e.line("(void)dt; (void)rdt; (void)trtol; (void)trtol2; (void)thr2;");
        --e.ind;
        e.line("}");
        // ---- phase_a ----------------------------------------------------------------------------------------------
        e.line("// stamps, own elimination, own forward substitution; contributions -> xb[slot * 32] (this lane's column of the buffer)");
        e.line("__device__ __forceinline__ bool phase_a(double time, double dt, double rdt, double* xb) {");
        ++e.ind;
        e.line("TsbEnv e; e.mode = TSB_MODE_TRAN; e.time = time; e.dt = dt; e.gmin = 0.0; e.rdt = rdt;");
        e.line("double b[" + S(n + 1) + "];");
        for (int k : y.touched) if (!y.a_assigned.count(k)) e.line("A[" + S(k) + "] = 0.0;   // fill (" + S(lu.pos[k].first) + "," + S(lu.pos[k].second) + ")");
        emit_stamps(e, sub, lu, false, false, true, nullptr);
        e.line("bool lu_ok = true;");
        for (int k : y.steps) {
            const LuProgram::Step& st = lu.steps[k];
            const std::string piv = "A[" + S(st.piv) + "]";
            e.line("// step " + S(k) + ": pivot (" + S(lu.prow[k]) + "," + S(lu.pcol[k]) + ")");
            if (!y.touched.count(st.piv)) e.line(piv + " = 0.0;");
            e.line("lu_ok = lu_ok & (" + piv + " != 0.0);");
            e.line(piv + " = tsb_rcp(" + piv + ");");
            for (size_t ui = 0; ui < st.urow.size(); ++ui) {
                if (!y.touched.count(st.urow[ui])) continue;
                const std::string u = "A[" + S(st.urow[ui]) + "]";
                e.line(u + " *= " + piv + ";");
                for (size_t li = 0; li < st.lcol.size(); ++li)
                    if (y.touched.count(st.lcol[li])) e.line("A[" + S(st.target[ui][li]) + "] -= " + u + " * A[" + S(st.lcol[li]) + "];");
            }
        }
        {   // forward substitution over the own steps; separator rows collect this part's share
            std::set<int> nz;                      // c[k] assigned so far
            auto init_c = [&](int k) {
                if (nz.count(k)) return;
                nz.insert(k);
                e.line("c[" + S(k) + "] = " + (y.b_assigned.count(lu.prow[k]) ? "b[" + S(lu.prow[k]) + "]" : std::string("0.0")) + ";");
            };
            for (int k = 1; k <= n; ++k) if (y.cnz.count(k) && y.b_assigned.count(lu.prow[k])) init_c(k);
            for (int k : y.steps) {
                if (!y.cnz.count(k)) continue;
                init_c(k);
                const LuProgram::Step& st = lu.steps[k];
                e.line("c[" + S(k) + "] *= A[" + S(st.piv) + "];");
                for (size_t li = 0; li < st.lcol.size(); ++li) {
                    if (!y.touched.count(st.lcol[li])) continue;
                    const int j = st.lrow_step[li];
                    const std::string prod = "c[" + S(k) + "] * A[" + S(st.lcol[li]) + "]";
                    if (!nz.count(j)) { nz.insert(j); e.line("c[" + S(j) + "] = -(" + prod + ");"); }
                    else e.line("c[" + S(j) + "] -= " + prod + ";");
                }
            }
        }
        {
            int slot = COOP_HDR;
            for (int k : y.xe) e.line("xb[" + S(slot++) + " * 32] = A[" + S(k) + "];");
            for (int k : y.xc) e.line("xb[" + S(slot++) + " * 32] = c[" + S(k) + "];");
        }
        e.line("(void)b; (void)e;");
        e.line("return lu_ok;");
        --e.ind;
        e.line("}");
        // ---- phase_b ----------------------------------------------------------------------------------------------
        e.line("// xall: the attempt's exchange buffer, [part][slot][lane] with this lane's offset already applied");
        e.line("__device__ __forceinline__ bool phase_b(const double* xall) {");
        ++e.ind;
        e.line("bool lu_ok = true;");
        auto gather = [&](const std::string& tgt, bool entry, int k) {
            std::string sum;
            for (int q = 0; q < NP; ++q) {
                const std::vector<int>& lst = entry ? sym[q].xe : sym[q].xc;
                auto it = std::find(lst.begin(), lst.end(), k);
                if (it == lst.end()) continue;
                const int slot = COOP_HDR + (int)(it - lst.begin()) + (entry ? 0 : (int)sym[q].xe.size());
                sum += (sum.empty() ? "" : " + ") + std::string("xall[") + S(q * nx + slot) + " * 32]";
            }
            e.line(tgt + " = " + (sum.empty() ? "0.0" : sum) + ";");
        };
        std::set<int> st_touched = sep_touched;
        for (int k : sep_touched) gather("A[" + S(k) + "]", true, k);
        std::vector<char> cz(n + 1, 1);
        for (int k = cp.n_int + 1; k <= n; ++k) if (sep_cnz.count(k)) { gather("c[" + S(k) + "]", false, k); cz[k] = 0; }
        for (int k : y.steps) cz[k] = y.cnz.count(k) ? 0 : 1;
        for (int k = cp.n_int + 1; k <= n; ++k) {         // the separator's elimination steps, by every part alike
            const LuProgram::Step& st = lu.steps[k];
            const std::string piv = "A[" + S(st.piv) + "]";
            e.line("// separator step " + S(k) + ": pivot (" + S(lu.prow[k]) + "," + S(lu.pcol[k]) + ")");
            if (!st_touched.count(st.piv)) { e.line(piv + " = 0.0;"); st_touched.insert(st.piv); }
            e.line("lu_ok = lu_ok & (" + piv + " != 0.0);");
            e.line(piv + " = tsb_rcp(" + piv + ");");
            for (size_t ui = 0; ui < st.urow.size(); ++ui) {
                if (!st_touched.count(st.urow[ui])) continue;
                const std::string u = "A[" + S(st.urow[ui]) + "]";
                e.line(u + " *= " + piv + ";");
                for (size_t li = 0; li < st.lcol.size(); ++li) {
                    if (!st_touched.count(st.lcol[li])) continue;
                    const int t = st.target[ui][li];
                    const std::string prod = u + " * A[" + S(st.lcol[li]) + "]";
                    if (!st_touched.count(t)) { st_touched.insert(t); e.line("A[" + S(t) + "] = -(" + prod + ");"); }
                    else e.line("A[" + S(t) + "] -= " + prod + ";");
                }
            }
        }
        for (int k = cp.n_int + 1; k <= n; ++k) {         // forward
            if (cz[k]) continue;
            const LuProgram::Step& st = lu.steps[k];
            e.line("c[" + S(k) + "] *= A[" + S(st.piv) + "];");
            for (size_t li = 0; li < st.lcol.size(); ++li) {
                if (!st_touched.count(st.lcol[li])) continue;
                const int j = st.lrow_step[li];
                const std::string prod = "c[" + S(k) + "] * A[" + S(st.lcol[li]) + "]";
                if (cz[j]) { cz[j] = 0; e.line("c[" + S(j) + "] = -(" + prod + ");"); }
                else e.line("c[" + S(j) + "] -= " + prod + ";");
            }
        }
        auto back = [&](int k, const std::set<int>& tch) {
            const LuProgram::Step& st = lu.steps[k];
            for (size_t ui = 0; ui < st.urow.size(); ++ui) {
                if (!tch.count(st.urow[ui])) continue;
                const int j = st.ucol_step[ui];
                if (cz[j]) continue;
                const std::string prod = "A[" + S(st.urow[ui]) + "] * c[" + S(j) + "]";
                if (cz[k]) { cz[k] = 0; e.line("c[" + S(k) + "] = -(" + prod + ");"); }
                else e.line("c[" + S(k) + "] -= " + prod + ";");
            }
        };
        for (int k = n; k > cp.n_int; --k) back(k, st_touched);
        for (auto it = y.steps.rbegin(); it != y.steps.rend(); ++it) back(*it, y.touched);
        for (int k = cp.n_int + 1; k <= n; ++k) e.line("x[" + S(lu.pcol[k]) + "] = " + (cz[k] ? std::string("0.0") : "c[" + S(k) + "]") + ";");
        for (int k : y.steps) e.line("x[" + S(lu.pcol[k]) + "] = " + (cz[k] ? std::string("0.0") : "c[" + S(k) + "]") + ";");
        e.line("return lu_ok;");
        --e.ind;
        e.line("}");
        // ---- state of the own time-dependent devices, own result columns --------------------------------------------
        // ---- Newton loop helpers (circuits with nonlinear devices): own devices, own unknowns ------------------------------
        e.line("__device__ __forceinline__ void update_nl(const double* v) {   // circuit.UpdateNonlinearVoltages, own devices");
        ++e.ind;
        for (int di : y.devs) {
            const Dev& d = pl.devs[di];
            if (!d.nonlinear()) continue;
            std::string Sx = "S + " + S(d.s_off);
            auto v = [&](int k) { return "v[" + S(d.nodes[k]) + "]"; };
            if (d.kind == TSB_D) e.line("S[" + S(d.s_off) + "] = " + v(0) + " - " + v(1) + ";");
            else if (d.kind == TSB_M) e.line("tsb_mos_update(" + Sx + ", " + S(d.ip.size() > 1 ? d.ip[1] : 0) + ", " + v(0) + ", " + v(1) + ", " + v(2) + ", " + v(3) + ");");
        }
        e.line("(void)v;");
        --e.ind;
        e.line("}");
        {
            // convergence of the own unknowns (tran.go:192-207; the two-tolerance form of tsb_converged); the separator's
            // unknowns are the same bits in every part: part 0 tests them
            e.line("__device__ __forceinline__ bool converged_own(double reltol, double abstol) const {");
            ++e.ind;
            e.line("bool ok = true;");
            for (int u = 1; u <= n; ++u)
                if (cp.owner[u] == p || (cp.owner[u] < 0 && p == 0))
                    e.line("{ const double diff = fabs(x[" + S(u) + "] - xo[" + S(u) + "]); if ((diff > reltol * fabs(x[" + S(u) + "]) + abstol) & (diff > reltol * fabs(xo[" + S(u) +
                           "]) + abstol)) ok = false; }");
            e.line("return ok;");
            --e.ind;
            e.line("}");
            e.line("__device__ __forceinline__ void keep_old() {   // oldSolution = solution, own and separator unknowns");
            for (int u = 1; u <= n; ++u) if (cp.owner[u] == p || cp.owner[u] < 0) e.line("    xo[" + S(u) + "] = x[" + S(u) + "];");
            e.line("}");
        }
        auto vd_expr = [&](const Dev& d) { return "(x[" + S(d.nodes[0]) + "] - x[" + S(d.nodes[1]) + "])"; };
        e.line("__device__ __forceinline__ void load_state(double dt) {");
        ++e.ind;
        for (int di : y.devs) {
            const Dev& d = pl.devs[di];
            if (d.kind == TSB_L) e.line("tsb_ind_load(P + " + S(d.p_off) + ", D + " + S(d.d_off) + ", S + " + S(d.s_off) + ", " + vd_expr(d) + ", dt);");
        }
        e.line("(void)dt;");
        --e.ind;
        e.line("}");
        e.line("__device__ __forceinline__ void update_state() {");
        ++e.ind;
        for (int di : y.devs) {
            const Dev& d = pl.devs[di];
            if (d.kind == TSB_C) e.line("tsb_cap_update(P + " + S(d.p_off) + ", S + " + S(d.s_off) + ", " + vd_expr(d) + ");");
            if (d.kind == TSB_L) e.line("tsb_ind_update(D + " + S(d.d_off) + ", S + " + S(d.s_off) + ", " + vd_expr(d) + ");");
        }
        --e.ind;
        e.line("}");
        e.line("__device__ __forceinline__ void signals(double time, double* out) const {   // own columns of [TIME, GetSolution()...]");
        ++e.ind;
        {
            std::map<int, int> rcol;                // result column -> resistor device
            int c = n + 1;
            for (size_t di = 0; di < pl.devs.size(); ++di) if (pl.devs[di].kind == TSB_R) rcol[c++] = (int)di;
            for (size_t j = 0; j < y.cols.size(); ++j) {
                const int col = y.cols[j];
                std::string v;
                if (col == 0) v = "time";
                else if (col <= pl.n_nodes) v = "x[" + S(col) + "]";
                else if (col <= n) v = "-x[" + S(col) + "]";
                else { const Dev& d = pl.devs[rcol.at(col)]; v = "tsb_div_by(x[" + S(d.nodes[0]) + "] - x[" + S(d.nodes[1]) + "], P[" + S(d.p_off) + "], D[" + S(d.d_off) + "])"; }
                e.line("out[" + S((int)j) + "] = " + v + ";");
            }
        }
        e.line("(void)time; (void)out;");
        --e.ind;
        e.line("}");
        --e.ind;
        e.line("};");
    }
}

}  // namespace

void coop_dimensions(const Plan& pl, const CoopPlan& cp, int& nx, int& nown_max) {
    std::vector<CoopSym> sym;
    coop_analyse(pl, cp, sym, nx);
    nown_max = 0;
    for (const CoopSym& y : sym) nown_max = std::max(nown_max, (int)y.cols.size());
}

std::string generate_source(const Plan& pl, const CodegenConfig& cfg) {
    Emitter e;
    const int n = pl.n();
    const int ncol_tran = pl.num_columns(TSB_AN_TRAN);
    e.line("// Generated by tspice_b200 codegen: n=" + std::to_string(n) + ", " +
           std::to_string(pl.devs.size()) + " devices, " + std::to_string(pl.lu_main.pos.size()) + " matrix entries incl. fill" +
           (pl.lu_main.dense ? " (dense)" : "") + ".");
    e.line("#define TSB_BLOCK " + std::to_string(cfg.block_size));
    if (cfg.fast_div) e.line("#define TSB_FAST_DIV 1");
    e.line("#define TSB_MIN_BLOCKS " + std::to_string(cfg.min_blocks));
    e.line("#define TSB_SKIP_LINEAR_RESOLVE " + std::to_string(cfg.skip_linear ? 1 : 0));
    e.line("#define TSB_LANE_REFILL " + std::to_string(cfg.lane_refill && pl.has_nonlinear ? 1 : 0));
    e.line("#define TSB_GRID " + std::to_string(cfg.grid ? 1 : 0));
    e.line("#define TSB_ORDER " + std::to_string(cfg.order ? 1 : 0));
    e.line("#define TSB_TGRID " + std::to_string(cfg.tgrid && !pl.has_nonlinear && cfg.skip_linear ? 1 : 0));
    const CoopPlan* coop = nullptr;          // cooperative transient kernels ride along (device/coop.cuh)
    if (cfg.coop_parts > 0 && cfg.fast_div) { auto it = pl.coop.find(cfg.coop_parts); if (it != pl.coop.end()) coop = &it->second; }
    if (coop) e.line("#define TSB_COOP 1");
    if (!cfg.meas.empty()) {             // measurement table: the compile-time half (skeleton.cuh, TsbSink::emit_meas)
        std::string spec;
        for (size_t k = 0; k + 2 < cfg.meas.size(); k += 3)
            spec += (k ? ", {" : "{") + std::to_string(cfg.meas[k]) + ", " + std::to_string(cfg.meas[k + 1]) + ", " + std::to_string(cfg.meas[k + 2]) + "}";
        e.line("#define TSB_MEAS " + std::to_string(cfg.meas.size() / 3));
        e.line("#define TSB_MEAS_SPEC " + spec);
    }
    if (!cfg.extra_defines.empty()) e.os << cfg.extra_defines << "\n";     // development knob ($TSB_EXTRA_DEFINES)
    e.os << k_models_src << "\n" << k_skeleton_src << "\n";

    e.line("struct Ckt {");
    ++e.ind;
    e.line("static constexpr int N = " + std::to_string(n) + ";");
    e.line("static constexpr int NCOL_MAX = " + std::to_string(ncol_tran) + ";");
    e.line("static constexpr bool HAS_NL = " + std::string(pl.has_nonlinear ? "true" : "false") + ";");
    {
        // SRC_UNIFORM: no parameter of any source varies per instance, so the source values at a given time are the same
        // in every instance (what the shared time grid may hand from the pilot to the others)
        bool uniform = true;
        for (const Dev& d : pl.devs)
            if (d.src_slot >= 0 && d.src_type() != TSB_SRC_PWL)
                for (size_t j = 0; j < d.p.size(); ++j) if (cfg.varying[d.p_off + (int)j]) uniform = false;
        e.line("static constexpr int NSRC = " + std::to_string(std::max(1, pl.n_src)) + ";");
        e.line("static constexpr bool SRC_UNIFORM = " + std::string(uniform ? "true" : "false") + ";");
    }
    e.line("static constexpr int DC_NESTED = " + std::string(cfg.dc_nested ? "1" : "0") + ";   // tsb_dc: rows carry SWEEP1 and SWEEP2 (dc.go:272-288)");
    e.line("double P[" + std::to_string(std::max(1, pl.n_params)) + "];      // parameters");
    e.line("double S[" + std::to_string(std::max(1, pl.n_state)) + "];      // device state carried between solves");
    e.line("double D[" + std::to_string(std::max(1, pl.n_derived)) + "];      // per-instance constants derived from P (1/R, L0, M)");
    e.line("double SV[" + std::to_string(std::max(1, pl.n_src)) + "];     // source values of the current solve context");
    e.line("double x[" + std::to_string(n + 1) + "], xo[" + std::to_string(n + 1) + "];   // mat.Solution() and oldSolution (index 0 = ground)");
    e.line("const double* U_;");
    e.line("");

    // ---- load -----------------------------------------------------------------------------
    e.line("__device__ __forceinline__ void load(const TsbArgs& a, long long inst) {");
    ++e.ind;
    e.line("U_ = a.U;");
    for (const Dev& d : pl.devs) {
        if ((d.kind == TSB_V || d.kind == TSB_I) && d.src_type() == TSB_SRC_PWL) continue;   // PWL tables stay in global memory
        for (size_t j = 0; j < d.p.size(); ++j) {
            int k = d.p_off + (int)j;
            if (cfg.varying[k])
                e.line("P[" + std::to_string(k) + "] = __ldcs(a.pv[" + std::to_string(cfg.var_slot[k]) + "] + inst);   // " + d.name + " p" + std::to_string(j));
            else
                e.line("P[" + std::to_string(k) + "] = a." + (k < 32 ? "Uc[" : "U[") + std::to_string(k) + "];");
        }
    }
    for (int i = 0; i < std::max(1, pl.n_state); ++i) e.line("S[" + std::to_string(i) + "] = 0.0;");
    for (int i = 0; i <= n; ++i) e.line("x[" + std::to_string(i) + "] = 0.0; xo[" + std::to_string(i) + "] = 0.0;");
    for (int i = 0; i < std::max(1, pl.n_src); ++i) e.line("SV[" + std::to_string(i) + "] = 0.0;");
    e.line("D[0] = 0.0;");
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        std::string P = "P + " + std::to_string(d.p_off);
        if (d.kind == TSB_R) e.line("D[" + std::to_string(d.d_off) + "] = tsb_res_g(" + P + ");");
        else if (d.kind == TSB_L) e.line("tsb_ind_derive(" + P + ", D + " + std::to_string(d.d_off) + ");");
        else if (d.kind == TSB_LCORE) e.line("D[" + std::to_string(d.d_off) + "] = tsb_lcore_L0(" + P + ");");
        else if (d.kind == TSB_D) e.line("tsb_dio_derive(" + P + ", D + " + std::to_string(d.d_off) + ");");
        else if (d.kind == TSB_M) e.line("tsb_mos_init_state(" + P + ", S + " + std::to_string(d.s_off) + ");");
        else if (d.kind == TSB_K) {
            int m = (int)d.ip.size(), q = 0;
            auto val = [&](int idx) {
                const Dev& l = pl.devs[idx];
                return l.kind == TSB_LCORE ? "D[" + std::to_string(l.d_off) + "]" : "P[" + std::to_string(l.p_off) + "]";
            };
            for (int i = 0; i < m; ++i)
                for (int j = i + 1; j < m; ++j, ++q)
                    e.line("D[" + std::to_string(d.d_off + q) + "] = tsb_mut_M(P[" + std::to_string(d.p_off) + "], " + val(d.ip[i]) + ", " + val(d.ip[j]) + ");");
        }
    }
    --e.ind;
    e.line("}");

    // ---- init: side effects of SetupDevices' initial stamp (circuit.go:154-156) on device state
    e.line("__device__ __forceinline__ void init() {");
    ++e.ind;
    if (pl.has_nonlinear) {
        e.line("TsbEnv e; e.mode = TSB_MODE_OP; e.time = 0.0; e.dt = 0.0; e.gmin = 0.0; e.rdt = 0.0;");
        for (int di : pl.stamp_order) {
            if (!pl.devs[di].nonlinear()) continue;
            e.line("{");
            ++e.ind;
            emit_eval(e, pl, di, "o");
            e.line("(void)o;");
            --e.ind;
            e.line("}");
        }
    }
    --e.ind;
    e.line("}");

    // ---- sources ----------------------------------------------------------------------------
    e.line("// VoltageSource.GetVoltage / CurrentSource.GetCurrent at Status.Time; `fac` = source-stepping factor");
    e.line("__device__ __forceinline__ void eval_sources(double t, double fac) {");
    ++e.ind;
    for (const Dev& d : pl.devs) {
        if (d.src_slot < 0) continue;
        std::string sv = "SV[" + std::to_string(d.src_slot) + "]";
        std::string P = "P + " + std::to_string(d.p_off);
        // source stepping scales VoltageSource.dcValue only (op.go:118-124)
        std::string fac = d.kind == TSB_V ? "fac" : "1.0";
        switch (d.src_type()) {
        case TSB_SRC_DC: e.line(sv + " = P[" + std::to_string(d.p_off) + "] * " + fac + ";"); break;
        case TSB_SRC_SIN: e.line(sv + " = tsb_src_sin(" + P + ", t, " + fac + ");"); break;
        case TSB_SRC_PULSE: e.line(sv + " = tsb_src_pulse(" + P + ", t);"); break;
        case TSB_SRC_PWL: e.line(sv + " = tsb_src_pwl(U_ + " + std::to_string(d.p_off) + ", " + std::to_string(d.p.size() / 2) + ", t);"); break;
        }
    }
    e.line("(void)t; (void)fac;");
    --e.ind;
    e.line("}");

    e.line("// Same at fac = 1 with the branch-free math.Sin restatement; false when an argument is outside its range");
    e.line("// (|x| >= 2^29) — the caller then re-evaluates with eval_sources().");
    e.line("__device__ __forceinline__ bool eval_sources_nb(double t) {");
    ++e.ind;
    e.line("bool ok = true;");
    for (const Dev& d : pl.devs) {
        if (d.src_slot < 0) continue;
        std::string sv = "SV[" + std::to_string(d.src_slot) + "]";
        std::string P = "P + " + std::to_string(d.p_off);
        switch (d.src_type()) {
        case TSB_SRC_DC: e.line(sv + " = P[" + std::to_string(d.p_off) + "] * 1.0;"); break;
        case TSB_SRC_SIN: e.line(sv + " = tsb_src_sin_nb(" + P + ", t, ok);"); break;
        case TSB_SRC_PULSE: e.line(sv + " = tsb_src_pulse(" + P + ", t);"); break;
        case TSB_SRC_PWL: e.line(sv + " = tsb_src_pwl(U_ + " + std::to_string(d.p_off) + ", " + std::to_string(d.p.size() / 2) + ", t);"); break;
        }
    }
    e.line("(void)t;");
    e.line("return ok;");
    --e.ind;
    e.line("}");

    // ---- DC sweep source override --------------------------------------------------------------
    e.line("__device__ __forceinline__ void set_dc(double v) {");
    ++e.ind;
    if (cfg.dc_param >= 0) e.line("P[" + std::to_string(cfg.dc_param) + "] = v;   // VoltageSource.SetValue (vsource.go:241-244)");
    e.line("(void)v;");
    --e.ind;
    e.line("}");
    e.line("__device__ __forceinline__ void set_dc2(double v) {   // the inner source of a nested sweep (dc.go:236)");
    ++e.ind;
    if (cfg.dc_param2 >= 0) e.line("P[" + std::to_string(cfg.dc_param2) + "] = v;");
    e.line("(void)v;");
    --e.ind;
    e.line("}");

    // ---- nonlinear voltage update ----------------------------------------------------------------
    e.line("__device__ __forceinline__ void update_nl(const double* v) {   // circuit.UpdateNonlinearVoltages");
    ++e.ind;
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        if (!d.nonlinear()) continue;
        std::string S = "S + " + std::to_string(d.s_off);
        auto v = [&](int k) { return "v[" + std::to_string(d.nodes[k]) + "]"; };
        if (d.kind == TSB_D) e.line("S[" + std::to_string(d.s_off) + "] = " + v(0) + " - " + v(1) + ";");
        else if (d.kind == TSB_Q) e.line("tsb_bjt_update(" + S + ", " + std::to_string(d.ip.empty() ? 0 : d.ip[0]) + ", " + v(0) + ", " + v(1) + ", " + v(2) + ");");
        else e.line("tsb_mos_update(" + S + ", " + std::to_string(d.ip.size() > 1 ? d.ip[1] : 0) + ", " + v(0) + ", " + v(1) + ", " + v(2) + ", " + v(3) + ");");
    }
    e.line("(void)v;");
    --e.ind;
    e.line("}");

    // ---- initial estimate -----------------------------------------------------------------------
    e.line("// OperatingPoint.calculateInitialEstimate (op.go:90-111): separate sparse matrix, linear devices only");
    e.line("__device__ __forceinline__ bool init_estimate(double status_dt, double* out) {");
    ++e.ind;
    if (pl.init_struct_singular) {
        e.line("(void)status_dt; (void)out;");
        e.line("return false;   // structurally singular without the nonlinear devices -> nil estimate");
    } else {
        e.line("TsbEnv e; e.mode = TSB_MODE_OP; e.time = 0.0; e.dt = status_dt; e.gmin = 0.0; e.rdt = status_dt > 0 ? 1.0 / status_dt : 0.0;");
        e.line("double A[" + std::to_string(pl.lu_init.pos.size()) + "];");
        e.line("double b[" + std::to_string(n + 1) + "];");
        {
            const bool fa = !pl.lu_init.dense;      // also in the strict build: only the sign of a zero can differ
            std::set<std::string> tg = stamp_targets(pl, pl.lu_init, true, true);
            std::set<int> bz;
            for (int i = 1; i <= n; ++i) if (!tg.count("b[" + std::to_string(i) + "]")) bz.insert(i);
            emit_clear(e, pl.lu_init, n, fa ? &tg : nullptr);
            emit_stamps(e, pl, pl.lu_init, true, true, fa);
            e.line("double xt[" + std::to_string(n + 1) + "];");
            emit_lu(e, pl.lu_init, false, "xt", fa ? &bz : nullptr);
        }
        for (int i = 1; i <= n; ++i) e.line("out[" + std::to_string(i) + "] = xt[" + std::to_string(i) + "];");
        e.line("return true;");
    }
    --e.ind;
    e.line("}");

    // ---- Newton body ----------------------------------------------------------------------------
    e.line("// mat.Clear(); ckt.Stamp(status); mat.LoadGmin(gmin); mat.Solve()  ->  x");
    e.line("// MODE >= 0 fixes the analysis mode at compile time (the dedicated transient loop): mode selects fold away.");
    e.line("// EARLY = false (the dedicated linear transient loop): a zero pivot does not return before the solve — the body");
    e.line("// stays one basic block; the caller discards x when the result is false.");
    e.line("// SOLVE = false: stamps only, for their side effects on device state (the DC sweep's discarded pass, dc.go:119-125).");
    e.line("// `mid` runs between the factorisation and the substitution: the source values SV[] that feed only the right-hand");
    e.line("// side are read after it, so a caller may produce them there (tsb_tran_linear: looked up in the shared time grid");
    e.line("// or computed) — off the critical path of the factorisation.");
    e.line("struct TsbNoMid { __device__ __forceinline__ void operator()() const {} };");
    e.line("template <int MODE, bool EARLY = true, bool SOLVE = true, class Mid = TsbNoMid>");
    e.line("__device__ __forceinline__ bool assemble_solve(int mode_rt, double time, double dt, double rdt, double gmin, Mid mid = Mid()) {");
    ++e.ind;
    e.line("const int mode = MODE >= 0 ? MODE : mode_rt;");
    e.line("TsbEnv e; e.mode = mode; e.time = time; e.dt = dt; e.gmin = gmin; e.rdt = rdt;");
    e.line("double A[" + std::to_string(pl.lu_main.pos.size()) + "];");
    e.line("double b[" + std::to_string(n + 1) + "];");
    {
        const bool fa = !pl.lu_main.dense;      // also in the strict build: only the sign of a zero can differ
        std::set<std::string> tg = stamp_targets(pl, pl.lu_main, false, false);
        std::set<int> bz;
        for (int i = 1; i <= n; ++i) if (!tg.count("b[" + std::to_string(i) + "]")) bz.insert(i);
        emit_clear(e, pl.lu_main, n, fa ? &tg : nullptr);
        std::vector<std::string> late;
        emit_stamps(e, pl, pl.lu_main, false, false, fa, &late);
        late.insert(late.begin(), "mid();");
        e.line("if (!SOLVE) return true;");
        e.line("double xt[" + std::to_string(n + 1) + "];");
        emit_lu(e, pl.lu_main, true, "xt", fa ? &bz : nullptr, "EARLY && !lu_ok", &late);
    }
    for (int i = 1; i <= n; ++i) e.line("x[" + std::to_string(i) + "] = xt[" + std::to_string(i) + "];");
    e.line(pl.lu_main.dense ? "return true;" : "return lu_ok;");
    --e.ind;
    e.line("}");

    // ---- fast build: condensed transient elimination ------------------------------------------------------
    const bool use_tf = pl.has_tranfast && cfg.fast_div && cfg.tranfast;
    e.line("static constexpr bool HAS_TF = " + std::string(use_tf ? "true" : "false") + ";");
    if (use_tf) emit_tranfast(e, pl, cfg);

    // ---- AC analysis (linear circuits) ----------------------------------------------------------------------
    e.line("static constexpr int NCOL_AC = " + std::to_string(pl.num_columns(TSB_AN_AC)) + ";");
    e.line("static constexpr bool HAS_AC = " + std::string(pl.has_nonlinear ? "false" : "true") + ";");
    if (!pl.has_nonlinear) emit_ac(e, pl);

    // ---- operator level: the stamped system itself -----------------------------------------------------
    // mat.Clear(); ckt.Stamp(status); mat.LoadGmin(gmin) as a DENSE n x n matrix + right-hand side written to
    // global memory, instance-major (A[inst][row][col], b[inst][row], 0-based = external index - 1): what a
    // host that keeps its own Solve() — or the warp-per-circuit LU operator — consumes.
    {
        LuProgram dn;                       // index map of the dense layout (no elimination program needed)
        dn.n = n;
        for (int r = 1; r <= n; ++r)
            for (int c2 = 1; c2 <= n; ++c2) { dn.index[{r, c2}] = (int)dn.pos.size(); dn.pos.push_back({r, c2}); }
        e.line("__device__ __forceinline__ void stamp_dense(int mode, double time, double dt, double rdt, double gmin, double* __restrict__ Aout, double* __restrict__ bout) {");
        ++e.ind;
        e.line("TsbEnv e; e.mode = mode; e.time = time; e.dt = dt; e.gmin = gmin; e.rdt = rdt;");
        e.line("double A[" + std::to_string(n * n) + "];");
        e.line("double b[" + std::to_string(n + 1) + "];");
        emit_clear(e, dn, n, nullptr);
        emit_stamps(e, pl, dn, false, false, false);
        e.line("if (gmin != 0.0) {   // LoadGmin: onto the pivot positions of the frozen order (SURVEY Q17)");
        for (int k = 1; k <= n; ++k)
            e.line("    A[" + std::to_string(dn.index[{pl.lu_main.prow[k], pl.lu_main.pcol[k]}]) + "] += gmin;");
        e.line("}");
        for (int k = 0; k < n * n; ++k) e.line("Aout[" + std::to_string(k) + "] = A[" + std::to_string(k) + "];");
        for (int i = 1; i <= n; ++i) e.line("bout[" + std::to_string(i - 1) + "] = b[" + std::to_string(i) + "];");
        --e.ind;
        e.line("}");
    }

    // ---- time-dependent device state -------------------------------------------------------------
    auto vd_expr = [&](const Dev& d) {
        return "(x[" + std::to_string(d.nodes[0]) + "] - x[" + std::to_string(d.nodes[1]) + "])";
    };
    e.line("__device__ __forceinline__ void load_state(double dt) {   // circuit.LoadState (circuit.go:192-201)");
    ++e.ind;
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        if (d.kind == TSB_L) e.line("tsb_ind_load(P + " + std::to_string(d.p_off) + ", D + " + std::to_string(d.d_off) + ", S + " + std::to_string(d.s_off) + ", " + vd_expr(d) + ", dt);");
    }
    e.line("(void)dt;");
    --e.ind;
    e.line("}");
    e.line("__device__ __forceinline__ void update_state() {   // circuit.Update (circuit.go:203-224)");
    ++e.ind;
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        if (d.kind == TSB_C) e.line("tsb_cap_update(P + " + std::to_string(d.p_off) + ", S + " + std::to_string(d.s_off) + ", " + vd_expr(d) + ");");
        if (d.kind == TSB_L) e.line("tsb_ind_update(D + " + std::to_string(d.d_off) + ", S + " + std::to_string(d.s_off) + ", " + vd_expr(d) + ");");
    }
    --e.ind;
    e.line("}");
    e.line("__device__ __forceinline__ double lte(double dt, double rdt) {   // Transient.calculateTruncError (tran.go:239-250)");
    ++e.ind;
    e.line("double m = 0.0, l;");
    {
        // maxLTE := 0.0; if lte > maxLTE { maxLTE = lte }.  Every term is >= +0 or NaN, so the first update is
        // "l unless NaN" (a compare-with-itself select instead of the max(0, l) NaN fix-up sequence).
        bool first = true;
        for (int di : pl.stamp_order) {
            const Dev& d = pl.devs[di];
            std::string call;
            if (d.kind == TSB_C) call = "tsb_cap_lte(P + " + std::to_string(d.p_off) + ", S + " + std::to_string(d.s_off) + ", dt, rdt)";
            if (d.kind == TSB_L) call = "tsb_ind_lte(S + " + std::to_string(d.s_off) + ", dt, rdt)";
            if (call.empty()) continue;
            if (first) e.line("l = " + call + "; m = (l != l) ? 0.0 : l;");
            else e.line("l = " + call + "; if (l > m) m = l;");
            first = false;
        }
    }
    e.line("(void)dt; (void)rdt; (void)l;");
    e.line("return m;");
    --e.ind;
    e.line("}");

    // the same as two decisions, without materialising the maximum: gt = maxLTE > trtol (reject), small = maxLTE < thr (the
    // step may double).  maxLTE is the largest device LTE that is not NaN (a NaN never wins `lte > maxLTE`), or 0; the
    // inductor's own LTE is math.Max(current, voltage): NaN when either is NaN unless the other is +Inf.
    e.line("__device__ __forceinline__ void lte_flags(double dt, double rdt, double trtol, double thr, bool& gt, bool& small) {");
    ++e.ind;
    e.line("gt = false; small = 0.0 < thr;");
    e.line("#if TSB_X_LTE_OPAQUE");
    e.line("double trtol2 = trtol, thr2 = thr; TSB_OPAQUE(trtol2); TSB_OPAQUE(thr2);     // see TSB_OPAQUE");
    e.line("#else");
    e.line("const double trtol2 = trtol, thr2 = thr;");
    e.line("#endif");
    for (int di : pl.stamp_order) {
        const Dev& d = pl.devs[di];
        if (d.kind == TSB_C) {
            e.line("{ const double l = tsb_cap_lte(P + " + std::to_string(d.p_off) + ", S + " + std::to_string(d.s_off) + ", dt, rdt); gt = gt | (l > trtol); small = small & !(l >= thr); }");
        } else if (d.kind == TSB_L) {
            e.line("{ double cu, vo; tsb_ind_lte2(S + " + std::to_string(d.s_off) + ", dt, rdt, cu, vo);");
            e.line("  const bool nan = ((cu != cu) | (vo != vo)) & !((cu == TSB_INF) | (vo == TSB_INF));");
            e.line("  gt = gt | (!nan & ((cu > trtol) | (vo > trtol2))); small = small & !(!nan & ((cu >= thr) | (vo >= thr2))); }");
        }
    }
    e.line("(void)dt; (void)rdt; (void)trtol; (void)trtol2; (void)thr2;");
    --e.ind;
    e.line("}");

    if (coop) {
        e.line("// hand-over to the cooperative transient kernel: device state and solution, instance-fastest");
        e.line("__device__ __forceinline__ void dump_state(double* o, long long n_inst, long long inst) const {");
        for (int i = 0; i < pl.n_state; ++i) e.line("    o[(long long)" + std::to_string(i) + " * n_inst + inst] = S[" + std::to_string(i) + "];");
        for (int i = 0; i <= n; ++i) e.line("    o[(long long)" + std::to_string(pl.n_state + i) + " * n_inst + inst] = x[" + std::to_string(i) + "];");
        e.line("}");
    }
    // ---- signals -----------------------------------------------------------------------------------
    e.line("__device__ __forceinline__ void signals(double* out) const {   // circuit.GetSolution (circuit.go:242-273)");
    ++e.ind;
    {
        int k = 0;
        for (int i = 1; i <= pl.n_nodes; ++i) e.line("out[" + std::to_string(k++) + "] = x[" + std::to_string(i) + "];");
        for (int b = pl.n_nodes + 1; b <= n; ++b) e.line("out[" + std::to_string(k++) + "] = -x[" + std::to_string(b) + "];");
        for (const Dev& d : pl.devs)
            if (d.kind == TSB_R)
                e.line("out[" + std::to_string(k++) + "] = tsb_div_by(x[" + std::to_string(d.nodes[0]) + "] - x[" + std::to_string(d.nodes[1]) + "], P[" + std::to_string(d.p_off) + "], D[" + std::to_string(d.d_off) + "]);   // I(" + d.name + ") = (v1 - v2) / R");
    }
    --e.ind;
    e.line("}");
    --e.ind;
    e.line("};");
    e.line("");
    if (coop) {
        const int groups = cfg.coop_groups > 0 ? cfg.coop_groups : 1;
        const int cblock = 32 * coop->parts * groups;
        e.line("#define TSB_COOP_BLOCK " + std::to_string(cblock));
        {
            // Launch bounds: the per-thread statistics (32 bytes per own result column) decide how many blocks an SM holds;
            // asking for more only lowers the register cap for nothing (measured: ladder n = 26, 4 parts: 14.5 ms at the
            // shared-memory limit of 3 blocks, 16.0 ms at 4, 20.2 ms at 2).
            int nx = 0, nown = 0;
            coop_dimensions(pl, *coop, nx, nown);
            const size_t smem = ((size_t)4 * nown * cblock + (size_t)groups * 2 * coop->parts * nx * 32) * sizeof(double) + 1024;
            int mb = (int)((227 * 1024) / smem);
            mb = std::max(1, std::min(mb, std::max(1, 512 / cblock)));        // at most what 128 registers per thread allow
            e.line("#ifndef TSB_COOP_MIN_BLOCKS");
            e.line("#define TSB_COOP_MIN_BLOCKS " + std::to_string(mb));
            e.line("#endif");
        }
        emit_coop(e, pl, *coop, cfg);
        e.os << k_coop_src << "\n";
        e.line("// One group of TSB_COOP_PARTS warps per 32 instances: warp w runs part w % PARTS of the instances of group w / PARTS.");
        e.line("// Every part is a loop nest of its own behind an early return (a switch inside one shared loop made ptxas spill");
        e.line("// ten times as much: 1432 instead of 140 bytes at 168 registers).");
        e.line("template <class Part> __device__ __forceinline__ void tsb_coop_loop(const TsbArgs& a, double* xg, int group, int lane) {");
        e.line("    constexpr int G = TSB_COOP_BLOCK / (32 * TSB_COOP_PARTS);");
        e.line("    for (long long base = (long long)blockIdx.x * (G * 32); base < a.n_run; base += (long long)gridDim.x * (G * 32)) {");
        e.line("        const long long slot = base + group * 32 + lane;");
        e.line("        const bool valid = slot < a.n_run;");
        e.line("        if (TSB_COOP_NL) tsb_coop_tran_nl_part<Part>(a, tsb_slot_instance(a, slot, valid), valid, xg, 1 + group);");
        e.line("        else tsb_coop_tran_part<Part>(a, tsb_slot_instance(a, slot, valid), valid, xg, 1 + group);");
        e.line("    }");
        e.line("}");
        e.line("extern \"C\" __global__ void __launch_bounds__(TSB_COOP_BLOCK, TSB_COOP_MIN_BLOCKS) tsb_coop_tran(TsbArgs a) {");
        e.line("    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;");
        e.line("    const int part = warp % TSB_COOP_PARTS, group = warp / TSB_COOP_PARTS;");
        e.line("    double* xg = tsb_smem + 4 * TSB_COOP_NOWN_MAX * TSB_COOP_BLOCK + group * (2 * TSB_COOP_PARTS * TSB_COOP_NX * 32);");
        for (int p2 = 0; p2 + 1 < coop->parts; ++p2)
            e.line("    if (part == " + std::to_string(p2) + ") { tsb_coop_loop<CoopPart" + std::to_string(p2) + ">(a, xg, group, lane); return; }");
        e.line("    tsb_coop_loop<CoopPart" + std::to_string(coop->parts - 1) + ">(a, xg, group, lane);");
        e.line("}");
    }
    e.line("extern \"C\" __global__ void __launch_bounds__(TSB_BLOCK, TSB_MIN_BLOCKS) tsb_optran(TsbArgs a) {");
    e.line("    if (Ckt::HAS_NL && TSB_LANE_REFILL) {   // persistent lanes: finished lanes refill themselves from a.work_counter");
    e.line("        long long inst = (long long)blockIdx.x * blockDim.x + threadIdx.x;");
    e.line("        tsb_run_optran_instance<Ckt>(a, tsb_slot_instance(a, inst, inst < a.n_run), inst < a.n_run);");
    e.line("        return;");
    e.line("    }");
    e.line("    // block-uniform trip count: every lane of a warp enters the driver (its Newton loops are warp-synchronous)");
    e.line("    for (long long base = (long long)blockIdx.x * blockDim.x; base < a.n_run; base += (long long)gridDim.x * blockDim.x)");
    e.line("        tsb_run_optran_instance<Ckt>(a, tsb_slot_instance(a, base + threadIdx.x, base + threadIdx.x < a.n_run), base + threadIdx.x < a.n_run);");
    e.line("}");
    e.line("// Operator level: stamp every instance (fresh device state, sources at a.tstart) -> a.wave = A, a.stats = b.");
    e.line("// tsb_stamp: every thread stores its own system straight to HBM (instances are (N*N+N)*8 bytes apart: 32 scattered");
    e.line("// 8-byte words per store instruction).  tsb_stamp_staged: the block's systems are contiguous in the instance-major");
    e.line("// layout, so they are assembled in shared memory (odd row stride: conflict-free) and written out with coalesced");
    e.line("// stores — the HBM-bound form; used whenever blockDim.x * ((N*N+N)|1) doubles fit in shared memory.");
    e.line("template <bool STAGED> __device__ __forceinline__ void tsb_stamp_body(const TsbArgs& a) {");
    e.line("    constexpr int NA = Ckt::N * Ckt::N, NB = Ckt::N, LD = (NA + NB) | 1;");
    e.line("    for (long long base = (long long)blockIdx.x * blockDim.x; base < a.n_run; base += (long long)gridDim.x * blockDim.x) {");
    e.line("        const long long inst = base + threadIdx.x;");
    e.line("        const bool valid = inst < a.n_run;");
    e.line("        double* mine = STAGED ? tsb_smem + (long long)threadIdx.x * LD : a.wave + inst * (long long)NA;");
    e.line("        double* mine_b = STAGED ? mine + NA : a.stats + inst * (long long)NB;");
    e.line("        if (valid) {");
    e.line("            Ckt c;");
    e.line("            c.load(a, inst);");
    e.line("            c.init();");
    e.line("            c.eval_sources(a.tstart, 1.0);");
    e.line("            const double dt = a.tstep;");
    e.line("            c.stamp_dense(a.analysis, a.tstart, dt, dt > 0 ? 1.0 / dt : 0.0, a.minstep, mine, mine_b);   // status.Gmin travels in `minstep`");
    e.line("        }");
    e.line("        if (STAGED) {");
    e.line("            __syncthreads();");
    e.line("            const long long left = a.n_run - base;");
    e.line("            const int nvalid = left < (long long)blockDim.x ? (int)left : (int)blockDim.x;");
    e.line("            double* ga = a.wave + base * (long long)NA;");
    e.line("            for (int q = threadIdx.x; q < nvalid * NA; q += blockDim.x) { const int t = q / NA; __stcs(ga + q, tsb_smem[t * LD + (q - t * NA)]); }");
    e.line("            double* gb = a.stats + base * (long long)NB;");
    e.line("            for (int q = threadIdx.x; q < nvalid * NB; q += blockDim.x) { const int t = q / NB; __stcs(gb + q, tsb_smem[t * LD + NA + (q - t * NB)]); }");
    e.line("            __syncthreads();");
    e.line("        }");
    e.line("    }");
    e.line("}");
    e.line("extern \"C\" __global__ void __launch_bounds__(TSB_BLOCK) tsb_stamp(TsbArgs a) { tsb_stamp_body<false>(a); }");
    e.line("extern \"C\" __global__ void __launch_bounds__(TSB_BLOCK) tsb_stamp_staged(TsbArgs a) { tsb_stamp_body<true>(a); }");
    e.line("extern \"C\" __global__ void __launch_bounds__(TSB_BLOCK) tsb_ac(TsbArgs a) {");
    e.line("    for (long long base = (long long)blockIdx.x * blockDim.x; base < a.n_run; base += (long long)gridDim.x * blockDim.x)");
    e.line("        if (base + threadIdx.x < a.n_run) tsb_run_ac_instance<Ckt>(a, tsb_slot_instance(a, base + threadIdx.x, true));");
    e.line("}");
    e.line("extern \"C\" __global__ void __launch_bounds__(TSB_BLOCK) tsb_dc(TsbArgs a) {");
    e.line("    for (long long base = (long long)blockIdx.x * blockDim.x; base < a.n_run; base += (long long)gridDim.x * blockDim.x)");
    e.line("        tsb_run_dc_instance<Ckt>(a, tsb_slot_instance(a, base + threadIdx.x, base + threadIdx.x < a.n_run), base + threadIdx.x < a.n_run);");
    e.line("}");
    return e.os.str();
}

}  // namespace tsb
