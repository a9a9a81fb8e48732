// UNCOMPILED — no Go toolchain in the build image; see README.md.
//
// BatchOP / BatchTransient / BatchDCSweep implement the reference's analysis.Analysis interface
// (pkg/analysis/anlysis.go:18-22: Setup(*circuit.Circuit) error; Execute() error; GetResults() map[string][]float64)
// over a batch of N instances.  With N == 1 and no Sweep they behave like analysis.NewOP / NewTransient / NewDCSweep:
// the per-instance status is turned back into the error the reference's Execute() would have returned.
// Call sites (cmd/spice/main.go:403-448, cmd/examples/*) only swap the constructor and hand over the netlist text.
package batch

/*
#include "tspice_b200.h"
*/
import "C"

import (
	"fmt"

	"github.com/edp1096/toy-spice/pkg/circuit"
)

const (
	anOP   = int(C.TSB_AN_OP)
	anTran = int(C.TSB_AN_TRAN)
	anDC   = int(C.TSB_AN_DC)
	anDC2  = int(C.TSB_AN_DC2)
	anAC   = int(C.TSB_AN_AC)
)

// base holds what the three analyses share.
type base struct {
	Netlist string                 // the text netlist.Parse was given
	GPU     int                    // device ordinal
	N       int64                  // instances (default 1)
	Sweep   map[ParamRef][]float64 // per-instance parameter values, N each
	Out     int                    // TSB_OUT_WAVE (default) | TSB_OUT_STATS | TSB_OUT_GRID | TSB_OUT_MEAS

	ctx   *Context
	plan  *Plan
	batch *Batch
}

func (a *base) setup(ckt *circuit.Circuit) error {
	if a.N <= 0 {
		a.N = 1
	}
	if a.Out == 0 {
		a.Out = int(C.TSB_OUT_WAVE)
	}
	var err error
	if a.ctx, err = NewContext(a.GPU); err != nil {
		return err
	}
	if a.plan, err = NewPlan(a.ctx, a.Netlist, ckt); err != nil {
		return err
	}
	if a.batch, err = NewBatch(a.plan, a.N); err != nil {
		return err
	}
	for ref, vals := range a.Sweep {
		if err = a.batch.SetParam(ref, vals); err != nil {
			return err
		}
	}
	return nil
}

// firstFailure maps instance 0's status word to the reference's error text.
func (a *base) firstFailure() error {
	st, err := a.batch.Status()
	if err != nil {
		return err
	}
	switch st[0] {
	case C.TSB_ST_OP_FAILED:
		return fmt.Errorf("final solution failed: failed to converge in 100 iterations") // op.go:216-229
	case C.TSB_ST_TRAN_FAILED:
		return fmt.Errorf("failed to converge at t=%g", a.batch.FailurePoint(0)) // tran.go:119
	case C.TSB_ST_DC_FAILED:
		return fmt.Errorf("convergence error at sweep value %g", a.batch.FailurePoint(0)) // dc.go:128
	case C.TSB_ST_AC_FAILED:
		return fmt.Errorf("matrix solve error at f=%g: matrix factorization failed", a.batch.FailurePoint(0)) // ac.go:68
	}
	return nil
}

func (a *base) Batch() *Batch { return a.batch }

// ---------------------------------------------------------------------------------------------- operating point
type BatchOP struct{ base }

func NewBatchOP(netlistText string) *BatchOP { return &BatchOP{base{Netlist: netlistText}} } // op.go:14

func (o *BatchOP) Setup(ckt *circuit.Circuit) error { return o.setup(ckt) }

func (o *BatchOP) Execute() error {
	if o.batch == nil {
		return fmt.Errorf("circuit not set")
	}
	if rc := C.tsb_run_op(o.batch.h, nil); rc != C.TSB_OK { // nil opts = NewBaseAnalysis defaults (anlysis.go:35-44)
		return o.ctx.lastErr("tsb_run_op")
	}
	if err := o.batch.Sync(); err != nil {
		return err
	}
	return o.firstFailure()
}

func (o *BatchOP) GetResults() map[string][]float64 {
	r, _ := o.batch.Instance(0, anOP)
	return r
}

// ---------------------------------------------------------------------------------------------- transient
type BatchTransient struct {
	base
	tStart, tStop, tStep, tMax float64
	uic                        bool
	CapRows                    int64 // waveform capacity per instance (TSB_OUT_WAVE); 0 = 16384
}

// NewBatchTransient keeps analysis.NewTransient's parameter list (tran.go:29) after the netlist text.
func NewBatchTransient(netlistText string, tStart, tStop, tStep, tMax float64, uic bool) *BatchTransient {
	return &BatchTransient{base: base{Netlist: netlistText}, tStart: tStart, tStop: tStop, tStep: tStep, tMax: tMax, uic: uic}
}

func (t *BatchTransient) Setup(ckt *circuit.Circuit) error { return t.setup(ckt) }

func (t *BatchTransient) Execute() error {
	if t.batch == nil {
		return fmt.Errorf("circuit not set") // tran.go:78-80
	}
	capRows := t.CapRows
	if capRows == 0 {
		capRows = 16384
	}
	uic := C.int(0)
	if t.uic {
		uic = 1
	}
	rc := C.tsb_run_tran(t.batch.h, C.double(t.tStart), C.double(t.tStop), C.double(t.tStep), C.double(t.tMax), uic,
		C.int(t.Out), C.int64_t(capRows), nil)
	if rc != C.TSB_OK {
		return t.ctx.lastErr("tsb_run_tran")
	}
	if err := t.batch.Sync(); err != nil {
		return err
	}
	return t.firstFailure()
}

func (t *BatchTransient) GetResults() map[string][]float64 {
	r, _ := t.batch.Instance(0, anTran)
	return r
}

// ---------------------------------------------------------------------------------------------- DC sweep
type BatchDCSweep struct {
	base
	sources                    []string
	starts, stops, increments []float64
}

// NewBatchDCSweep keeps analysis.NewDCSweep's parameter list (dc.go:20) after the netlist text, panic included.
func NewBatchDCSweep(netlistText string, sources []string, starts, stops, increments []float64) *BatchDCSweep {
	if len(sources) != len(starts) || len(sources) != len(stops) || len(sources) != len(increments) {
		panic("inconsistent parameter lengths") // dc.go:21-23
	}
	return &BatchDCSweep{base: base{Netlist: netlistText}, sources: sources, starts: starts, stops: stops, increments: increments}
}

func (d *BatchDCSweep) Setup(ckt *circuit.Circuit) error {
	if err := d.setup(ckt); err != nil {
		return err
	}
	for _, s := range d.sources {
		if d.plan.FindDevice(s) < 0 {
			return fmt.Errorf("source %s not found", s) // dc.go:64-66
		}
	}
	return nil
}

func (d *BatchDCSweep) Execute() error {
	if d.batch == nil {
		return fmt.Errorf("circuit not set")
	}
	var rc C.int
	switch len(d.sources) {
	case 1: // singleSweep, dc.go:88-140
		rc = C.tsb_run_dc(d.batch.h, C.int(d.plan.FindDevice(d.sources[0])), C.double(d.starts[0]), C.double(d.stops[0]),
			C.double(d.increments[0]), C.int(d.Out), nil)
	case 2: // nestedSweep, dc.go:205-270: source 0 is the outer loop
		rc = C.tsb_run_dc2(d.batch.h, C.int(d.plan.FindDevice(d.sources[0])), C.double(d.starts[0]), C.double(d.stops[0]),
			C.double(d.increments[0]), C.int(d.plan.FindDevice(d.sources[1])), C.double(d.starts[1]), C.double(d.stops[1]),
			C.double(d.increments[1]), C.int(d.Out), nil)
	default:
		return fmt.Errorf("unsupported number of sweep sources: %d", len(d.sources)) // dc.go:86
	}
	if rc != C.TSB_OK {
		return d.ctx.lastErr("tsb_run_dc")
	}
	if err := d.batch.Sync(); err != nil {
		return err
	}
	return d.firstFailure()
}

func (d *BatchDCSweep) GetResults() map[string][]float64 {
	an := anDC
	if len(d.sources) == 2 {
		an = anDC2
	}
	r, _ := d.batch.Instance(0, an)
	return r
}

// ---------------------------------------------------------------------------------------------- AC analysis
// BatchAC keeps analysis.NewAC's parameter list (ac.go:21) after the netlist text.  Linear circuits only (tspice_b200.h:
// tsb_run_ac); a circuit with an inductor fails at the first frequency exactly as the reference's does.
type BatchAC struct {
	base
	fStart, fStop float64
	nPoints       int
	pType         string
	RefRead       bool // TSB_OUT_AC_REFREAD: GetComplexSolution's literal index arithmetic over interleaved vectors
}

func NewBatchAC(netlistText string, fStart, fStop float64, nPoints int, pType string) *BatchAC {
	return &BatchAC{base: base{Netlist: netlistText}, fStart: fStart, fStop: fStop, nPoints: nPoints, pType: pType}
}

func (a *BatchAC) Setup(ckt *circuit.Circuit) error { return a.setup(ckt) } // the operating point of ac.go:33-49 has no effect on a linear circuit's sweep

func (a *BatchAC) Execute() error {
	if a.batch == nil {
		return fmt.Errorf("circuit not set") // ac.go:52-54
	}
	sweep := map[string]C.int{"DEC": 0, "OCT": 1, "LIN": 2}[a.pType]
	out := C.int(a.Out)
	if a.RefRead {
		out |= C.TSB_OUT_AC_REFREAD
	}
	if rc := C.tsb_run_ac(a.batch.h, sweep, C.int(a.nPoints), C.double(a.fStart), C.double(a.fStop), out, nil); rc != C.TSB_OK {
		return a.ctx.lastErr("tsb_run_ac")
	}
	if err := a.batch.Sync(); err != nil {
		return err
	}
	return a.firstFailure()
}

func (a *BatchAC) GetResults() map[string][]float64 { // keys FREQ, V(n)_MAG, V(n)_PHASE, I(Vsrc)_MAG, I(Vsrc)_PHASE (anlysis.go:87-111)
	r, _ := a.batch.Instance(0, anAC)
	return r
}
