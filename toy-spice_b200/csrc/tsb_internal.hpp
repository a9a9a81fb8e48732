// tsb_internal.hpp — host-side data model of the batched engine (not part of the public ABI).
#pragma once
#include <cstdint>
#include <map>
#include <string>
#include <utility>
#include <vector>
#include "../../include/tspice_b200.h"

namespace tsb {

// ---- device table -------------------------------------------------------------------------
struct Dev {
    int kind = 0;
    std::string name;
    int nodes[4] = {0, 0, 0, 0};
    int n_nodes = 0;
    int branch = 0;
    std::vector<double> p;     // nominal parameters (layout: include/tspice_b200.h)
    std::vector<int> ip;
    // assigned by finalize
    int p_off = 0;             // offset of p[] in the flat parameter space
    int s_off = 0, n_state = 0;
    int src_slot = -1;         // V / I: index into the source-value array
    int d_off = -1;            // derived-value slot(s)
    bool nonlinear() const { return kind == TSB_D || kind == TSB_Q || kind == TSB_M; }
    bool time_dependent() const { return kind == TSB_C || kind == TSB_L; }   // SURVEY Q11
    int src_type() const { return ip.empty() ? TSB_SRC_DC : ip[0]; }
};

// One AddElement / AddRHS call of a device stamp: value = sign * o[out] (or a constant).
struct StampEntry {
    int row, col;      // external indices; col == 0 -> AddRHS(row)
    int out;           // index into the device's stamp-value array o[]; -1 -> constant `cval`
    double sign;       // +1 / -1
    double cval;       // constant value when out < 0 (the +-1 incidence entries)
    bool tran_only;    // emitted by the reference only when Mode == Transient (pattern bookkeeping)
};

struct PivotOrder {
    int n = 0;
    std::vector<int> ext2int;        // [n+1], Translate numbering
    std::vector<int> prow, pcol;     // [n+1], external row/col of the pivot of step k
    bool singular = false;
};

// Elimination program over a fixed pattern (symbolic factorisation result).
struct LuProgram {
    int n = 0;
    std::vector<std::pair<int, int>> pos;          // entry k -> (ext row, ext col), pattern + fill
    std::map<std::pair<int, int>, int> index;      // (ext row, ext col) -> k
    std::vector<int> prow, pcol;                   // [n+1]
    struct Step {
        int piv;                                   // entry index of the pivot
        std::vector<int> urow;                     // entries (prow[k], c) right of the pivot, in column-internal order
        std::vector<int> lcol;                     // entries (r, pcol[k]) below the pivot, in row-internal order
        std::vector<std::vector<int>> target;      // target[u][l] = entry (row of l, col of u)
        std::vector<int> lrow_step;                // for each l: elimination step index of its row
        std::vector<int> ucol_step;                // for each u: elimination step index of its column
    };
    std::vector<Step> steps;                       // [n+1], 1-based
    bool dense = false;
};

// Cooperative mapping (device/coop.cuh): one circuit is solved by P threads in P different warps of a block.  The unknowns
// are split into P interiors that do not touch each other and a separator; part p stamps the devices it owns, eliminates
// its interior (a nested-dissection order: interiors first, separator last) and hands its contribution to the separator
// system to the others through shared memory; every part then solves the (small) separator system and back-substitutes
// its interior.  Built by plan.cpp: build_coop for circuits without nonlinear devices and without mutual couplings.
struct CoopPlan {
    int parts = 0;
    std::vector<int> owner;          // [n+1] unknown (external index) -> part, -1: separator
    std::vector<int> dev_owner;      // [devs] device -> part
    std::vector<int> step_owner;     // [n+1] elimination step of `lu` -> part, -1: separator step
    std::vector<int> col_owner;      // [transient columns] result column -> part (column 0, TIME: part 0)
    int n_int = 0;                   // steps 1..n_int eliminate interiors (part 0's first, then part 1's, ...), the rest the separator
    LuProgram lu;                    // elimination program of the nested-dissection order over the stamped pattern
    int nx = 0, nown_max = 0;        // exchange slots per part and attempt, result columns of the widest part (codegen.cpp: coop_dimensions, filled at finalize)
};

struct Plan {
    tsb_ctx* ctx = nullptr;
    int n_nodes = 0, n_branches = 0;
    std::vector<Dev> devs;                          // netlist order
    std::vector<int> stamp_order;                   // device indices, K last (circuit.go:83-152)
    std::vector<std::string> node_names;            // [n_nodes+1], from_netlist plans
    std::string title;
    // dot-card request (from_netlist plans)
    int analysis = TSB_AN_OP;
    double tran[4] = {0, 0, 0, 0};
    int uic = 0;
    int dc_src_dev = -1;
    double dc[3] = {0, 0, 0};
    std::string dc_src_name;
    int dc2_src_dev = -1;                           // second .dc source (nested sweep), -1: none
    double dc2[3] = {0, 0, 0};
    int ac_sweep = 0, ac_points = 0;                // .ac card: 0 DEC, 1 OCT, 2 LIN; total number of points; fstart, fstop
    double ac_f[2] = {0, 0};
    // finalize results
    bool finalized = false;
    int n_params = 0, n_state = 0, n_src = 0, n_derived = 0;
    std::vector<double> nominal;                    // flat parameter space
    std::vector<double> pwl_table;                  // concatenated PWL tables (uniform data)
    std::vector<std::vector<StampEntry>> stamps;    // per device: ordered AddElement/AddRHS calls (OP + tran)
    std::vector<std::pair<int, int>> pattern_op, pattern_tran_extra;   // first-touch order
    PivotOrder order_main, order_init;
    LuProgram lu_main, lu_init;
    // Transient solves of the fast build (static condensation, plan.cpp: build_tranfast): an elimination order that
    // takes the pivots whose value is the same in every solve of a run first, and per entry of lu_tf.pos whether its
    // STAMPED value changes from solve to solve (time step, device state)
    LuProgram lu_ac;                                // AC analysis: the OP order (the reference factors first in its OP) over the StampAC pattern
    LuProgram lu_tf;
    std::vector<char> tf_variant;
    bool has_tranfast = false;
    std::map<int, CoopPlan> coop;                   // parts (2, 4) -> cooperative plan, where one exists
    bool init_struct_singular = false;
    bool has_nonlinear = false, has_time_dependent = false, has_bjt = false, has_mutual = false;
    std::string error;

    int n() const { return n_nodes + n_branches; }
    int num_columns(int analysis_) const;
    std::string column_name(int analysis_, int col) const;
};

// netlist.cpp
int plan_from_netlist(const std::string& text, Plan& plan, std::string& err);
// plan.cpp
int plan_finalize(Plan& plan);
void device_stamp_entries(const Plan& plan, int dev_index, std::vector<StampEntry>& out);
// AddComplexElement calls of one device's StampAC in call order: (row, col, code); codes are listed at the definition.
struct AcEntry { int row, col, code; double sign; };
void device_ac_entries(const Plan& plan, int dev_index, std::vector<AcEntry>& out);
void ac_frequency_points(int sweep_type, int n_points, double fstart, double fstop, std::vector<double>& f);
int device_num_outputs(const Dev& d);
// codegen.cpp
struct CodegenConfig {
    std::vector<char> varying;      // [n_params] 1 -> read per instance from the SoA parameter buffer
    std::vector<int> var_slot;      // [n_params] slot in the SoA buffer or -1
    int n_var = 0;
    int block_size = 128;
    int dc_param = -1;              // flat parameter index overwritten by the DC sweep value
    int dc_param2 = -1;             // nested sweep (dc.go:205-270): parameter of the inner source; dc_nested marks the kernel
    bool dc_nested = false;
    bool fast_div = false;          // TSB_FAST_DIV build (non-strict): see device/models.cuh
    int min_blocks = 1;             // __launch_bounds__ second argument of the transient kernel
    bool skip_linear = true;        // compile the redundant second linear solve away
    std::string extra_defines;      // development knob: extra #define lines ($TSB_EXTRA_DEFINES, ';'-separated NAME=VALUE)
    bool grid = false;              // kernels that carry the TSB_OUT_GRID resampling code
    std::vector<int> meas;          // TSB_OUT_MEAS kernels: {kind, column, trigger column} per measurement; empty: none
    bool order = false;             // kernels that map launch slots to instances through a processing order
    bool lane_refill = false;       // nonlinear circuits: resident grid, finished lanes fetch the next instance
    bool tgrid = false;             // linear circuits: kernels that can read / publish the shared time grid (skeleton.cuh)
    bool tranfast = true;           // fast build: transient solves use the condensed elimination (lu_tf) where the plan has one
    int coop_groups = 1;            // cooperative kernels: groups of `coop_parts` warps per block
    int coop_parts = 0;             // > 0: the unit also carries the cooperative transient kernels for plan.coop[coop_parts]
};
std::string generate_source(const Plan& plan, const CodegenConfig& cfg);
// cooperative kernels: exchange slots per part and attempt, result columns of the widest part (what sizes their shared memory)
void coop_dimensions(const Plan& plan, const CoopPlan& cp, int& nx, int& nown_max);

}  // namespace tsb
