// UNCOMPILED — no Go toolchain in the build image; see README.md.
//
// cgo shim over include/tspice_b200.h.  The numbered netlist comes from the NETLIST TEXT (tsb_plan_from_netlist restates
// netlist.Parse + AssignNodeBranchMaps + CreateDevice), and NewPlan verifies that the library numbered nodes and
// branches exactly like the *circuit.Circuit the caller built with the reference's own packages, so that "V(name)" /
// "I(name)" keys mean the same thing on both sides (circuit.go:48-71).
package batch

/*
#cgo CFLAGS: -I${SRCDIR}/../../third_party/tspice_b200/include
#cgo LDFLAGS: -L${SRCDIR}/../../third_party/tspice_b200 -ltspice_b200 -Wl,-rpath,${SRCDIR}/../../third_party/tspice_b200
#include "tspice_b200.h"
#include <stdlib.h>
*/
import "C"

import (
	"fmt"
	"runtime"
	"unsafe"

	"github.com/edp1096/toy-spice/pkg/circuit"
)

// Context drives one GPU (tsb_ctx).
type Context struct{ h *C.tsb_ctx }

func NewContext(gpu int) (*Context, error) {
	var h *C.tsb_ctx
	if rc := C.tsb_ctx_create(C.int(gpu), &h); rc != C.TSB_OK {
		return nil, fmt.Errorf("tsb_ctx_create(%d): %s", gpu, C.GoString(C.tsb_last_error(nil)))
	}
	c := &Context{h}
	runtime.SetFinalizer(c, func(c *Context) { c.Close() })
	return c, nil
}

func (c *Context) Close() {
	if c.h != nil {
		C.tsb_ctx_destroy(c.h)
		c.h = nil
	}
}

func (c *Context) lastErr(what string) error {
	return fmt.Errorf("%s: %s", what, C.GoString(C.tsb_last_error(c.h)))
}

// Plan is the numbered netlist of the batch (tsb_plan): Translate order, stamped pattern, frozen pivot order.
type Plan struct {
	h   *C.tsb_plan
	ctx *Context
}

// NewPlan builds the plan from the netlist text and checks it against the circuit the reference built from the same
// text (ckt may be nil to skip the check).
func NewPlan(ctx *Context, netlistText string, ckt *circuit.Circuit) (*Plan, error) {
	cs := C.CString(netlistText)
	defer C.free(unsafe.Pointer(cs))
	var h *C.tsb_plan
	if rc := C.tsb_plan_from_netlist(ctx.h, cs, &h); rc != C.TSB_OK {
		return nil, ctx.lastErr("Error parsing netlist")
	}
	p := &Plan{h, ctx}
	runtime.SetFinalizer(p, func(p *Plan) { p.Close() })
	if ckt != nil {
		var nNodes, nBranches C.int
		C.tsb_plan_size(h, &nNodes, &nBranches)
		if int(nNodes) != len(ckt.GetNodeMap()) || int(nBranches) != len(ckt.GetBranchMap()) {
			return nil, fmt.Errorf("plan has %d nodes / %d branches, circuit has %d / %d", nNodes, nBranches,
				len(ckt.GetNodeMap()), len(ckt.GetBranchMap()))
		}
		for name, idx := range ckt.GetNodeMap() {
			var s *C.char
			if C.tsb_plan_node_name(h, C.int(idx), &s) != C.TSB_OK || C.GoString(s) != name {
				return nil, fmt.Errorf("node %q is number %d in the circuit but %q in the plan", name, idx, C.GoString(s))
			}
		}
		for name, idx := range ckt.GetBranchMap() {
			d := p.FindDevice(name)
			var branch C.int
			if d < 0 || C.tsb_plan_device_info(h, C.int(d), nil, nil, nil, &branch, nil, nil) < 0 || int(branch) != idx {
				return nil, fmt.Errorf("branch of %q is %d in the circuit but %d in the plan", name, idx, branch)
			}
		}
	}
	return p, nil
}

func (p *Plan) Close() {
	if p.h != nil {
		C.tsb_plan_destroy(p.h)
		p.h = nil
	}
}

func (p *Plan) FindDevice(name string) int {
	cs := C.CString(name)
	defer C.free(unsafe.Pointer(cs))
	return int(C.tsb_plan_find_device(p.h, cs))
}

// Columns returns the result keys in row order: TIME | SWEEP1 [SWEEP2], V(node...), I(branch...), I(R...).
func (p *Plan) Columns(analysis int) []string {
	n := int(C.tsb_plan_num_columns(p.h, C.int(analysis)))
	out := make([]string, n)
	buf := (*C.char)(C.malloc(128))
	defer C.free(unsafe.Pointer(buf))
	for k := 0; k < n; k++ {
		C.tsb_plan_column_name(p.h, C.int(analysis), C.int(k), buf, 128)
		out[k] = C.GoString(buf)
	}
	return out
}

// CoopInfo returns the partition behind tsb_opts.coop_parts (the cooperative mapping: one instance advanced by `parts`
// GPU threads, each eliminating its own sub-circuit): owner[u] for every unknown u = 1..n is the part that eliminates it,
// -1 = separator (owner[0] is unused); ok = false when the netlist has no partition into that many sub-circuits.  Nothing has
// to be called for the mapping to be used: the default options pick it for circuits of >= 16 unknowns.
func (p *Plan) CoopInfo(parts int) (owner []int, nSeparator int, ok bool) {
	var nn, nb C.int
	C.tsb_plan_size(p.h, &nn, &nb)
	n := int(nn) + int(nb)
	buf := make([]C.int, n+1)
	var ns C.int
	if rc := C.tsb_plan_coop_info(p.h, C.int(parts), &buf[0], &ns); rc != C.TSB_OK {
		return nil, 0, false
	}
	owner = make([]int, n+1)
	for i := range buf {
		owner[i] = int(buf[i])
	}
	return owner, int(ns), true
}

// ParamRef names one sweepable parameter: device name + index into the device kind's parameter layout (tspice_b200.h).
type ParamRef struct {
	Device string
	Param  int
}

// Batch is N instances of a plan (tsb_batch).
type Batch struct {
	h     *C.tsb_batch
	plan  *Plan
	N     int64
	nMeas int
}

func NewBatch(plan *Plan, n int64) (*Batch, error) {
	var h *C.tsb_batch
	if rc := C.tsb_batch_create(plan.h, C.int64_t(n), &h); rc != C.TSB_OK {
		return nil, plan.ctx.lastErr("tsb_batch_create")
	}
	b := &Batch{h: h, plan: plan, N: n}
	runtime.SetFinalizer(b, func(b *Batch) { b.Close() })
	return b, nil
}

func (b *Batch) Close() {
	if b.h != nil {
		C.tsb_batch_destroy(b.h)
		b.h = nil
	}
}

// SetParam gives every instance its own value of one parameter.  The values are copied during the call
// (tsb_batch_set_param stages them through a library-owned pinned buffer).
func (b *Batch) SetParam(ref ParamRef, values []float64) error {
	if int64(len(values)) != b.N {
		return fmt.Errorf("SetParam(%s[%d]): %d values for %d instances", ref.Device, ref.Param, len(values), b.N)
	}
	d := b.plan.FindDevice(ref.Device)
	if d < 0 {
		return fmt.Errorf("device %s not found", ref.Device)
	}
	if rc := C.tsb_batch_set_param(b.h, C.int(d), C.int(ref.Param), (*C.double)(unsafe.Pointer(&values[0]))); rc != C.TSB_OK {
		return b.plan.ctx.lastErr("tsb_batch_set_param")
	}
	return nil
}

func (b *Batch) Sync() error {
	if rc := C.tsb_batch_sync(b.h); rc != C.TSB_OK {
		return b.plan.ctx.lastErr("tsb_batch_sync")
	}
	return nil
}

// Status returns the per-instance status words (TSB_ST_*): failures are data, never a call failure.
func (b *Batch) Status() ([]int32, error) {
	out := make([]int32, b.N)
	if rc := C.tsb_result_status(b.h, (*C.int32_t)(unsafe.Pointer(&out[0]))); rc != C.TSB_OK {
		return nil, b.plan.ctx.lastErr("tsb_result_status")
	}
	return out, nil
}

// FailurePoint returns counters[5] of instance i: the time ("failed to converge at t=%g", tran.go:119) or sweep value
// (dc.go:128) at which the instance failed.
func (b *Batch) FailurePoint(i int64) float64 {
	cnt := make([]int64, 8*b.N)
	C.tsb_result_counters(b.h, (*C.int64_t)(unsafe.Pointer(&cnt[0])))
	return *(*float64)(unsafe.Pointer(&cnt[5*b.N+i]))
}

// Instance returns the reference's result map of one instance (anlysis.go:113-115).
func (b *Batch) Instance(i int64, analysis int) (map[string][]float64, error) {
	var nInst, capRows C.int64_t
	var nCol C.int
	C.tsb_result_dims(b.h, &nInst, &nCol, &capRows)
	if capRows < 1 {
		capRows = 1
	}
	buf := make([]float64, int64(capRows)*int64(nCol))
	var nRows C.int64_t
	if rc := C.tsb_result_waveform(b.h, C.int64_t(i), (*C.double)(unsafe.Pointer(&buf[0])), capRows, &nRows); rc != C.TSB_OK {
		return nil, b.plan.ctx.lastErr("tsb_result_waveform")
	}
	cols := b.plan.Columns(analysis)
	out := make(map[string][]float64, len(cols))
	for k, name := range cols {
		s := make([]float64, int(nRows))
		for r := 0; r < int(nRows); r++ {
			s[r] = buf[r*int(nCol)+k]
		}
		out[name] = s
	}
	return out, nil
}

// Meas is one entry of a measurement table (tsb_meas; the .meas family: WHEN, AT, MAX, MIN, AVG, INTEG, RMS, defined
// in tspice_b200.h).  From / To = math.Inf(-1) / math.Inf(1): the whole series.
type Meas struct {
	Kind, Column, TrigColumn, Edge, Count int
	Level, From, To                       float64
}

func measTable(m []Meas) []C.tsb_meas {
	t := make([]C.tsb_meas, len(m))
	for k, e := range m {
		t[k] = C.tsb_meas{kind: C.int(e.Kind), column: C.int(e.Column), trig_column: C.int(e.TrigColumn), edge: C.int(e.Edge),
			count: C.int(e.Count), level: C.double(e.Level), from: C.double(e.From), to: C.double(e.To)}
	}
	return t
}

// SetMeasures sets the batch's measurement table (copied; nil clears); runs with TSB_OUT_MEAS reduce it on the device.
func (b *Batch) SetMeasures(m []Meas) error {
	t := measTable(m)
	var p *C.tsb_meas
	if len(t) > 0 {
		p = &t[0]
	}
	if rc := C.tsb_batch_set_measures(b.h, p, C.int(len(t))); rc != C.TSB_OK {
		return b.plan.ctx.lastErr("tsb_batch_set_measures")
	}
	b.nMeas = len(t)
	return nil
}

// Measures returns value[m][instance] and abscissa[m][instance] of the last TSB_OUT_MEAS run.
func (b *Batch) Measures() (value, abscissa [][]float64, err error) {
	flat := make([]float64, 2*int64(b.nMeas)*b.N+1)
	if rc := C.tsb_result_measures(b.h, (*C.double)(unsafe.Pointer(&flat[0]))); rc != C.TSB_OK {
		return nil, nil, b.plan.ctx.lastErr("tsb_result_measures")
	}
	value, abscissa = make([][]float64, b.nMeas), make([][]float64, b.nMeas)
	for m := 0; m < b.nMeas; m++ {
		value[m] = flat[int64(m)*b.N : int64(m+1)*b.N]
		abscissa[m] = flat[int64(b.nMeas+m)*b.N : int64(b.nMeas+m+1)*b.N]
	}
	return value, abscissa, nil
}

// Stats returns min / max / sum / last per column and instance: stats[q][column][instance] (TSB_OUT_STATS runs).
func (b *Batch) Stats() ([][][]float64, error) {
	var nInst C.int64_t
	var nCol C.int
	C.tsb_result_dims(b.h, &nInst, &nCol, nil)
	flat := make([]float64, 4*int64(nCol)*int64(nInst))
	if rc := C.tsb_result_stats_all(b.h, (*C.double)(unsafe.Pointer(&flat[0]))); rc != C.TSB_OK {
		return nil, b.plan.ctx.lastErr("tsb_result_stats_all")
	}
	out := make([][][]float64, 4)
	for q := 0; q < 4; q++ {
		out[q] = make([][]float64, int(nCol))
		for c := 0; c < int(nCol); c++ {
			off := (int64(q)*int64(nCol) + int64(c)) * int64(nInst)
			out[q][c] = flat[off : off+int64(nInst)]
		}
	}
	return out, nil
}
