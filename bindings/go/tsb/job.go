// UNCOMPILED — no Go toolchain in the build image; see README.md.
//
// Job: one parameter sweep over several GPUs of one box from ONE Go process (tsb_job_*).  Instances are split
// contiguously over the GPUs ([g*N/G, (g+1)*N/G)); there is no exchange between GPUs during a run; summaries are reduced
// on every device before they cross the bus.
package batch

/*
#include "tspice_b200.h"
#include <stdlib.h>
*/
import "C"

import (
	"fmt"
	"unsafe"
)

type Job struct {
	h     *C.tsb_job
	N     int64
	nMeas int
	nFour int
}

func NewJob(gpus []int, netlistText string, n int64) (*Job, error) {
	ids := make([]C.int, len(gpus))
	for i, g := range gpus {
		ids[i] = C.int(g)
	}
	cs := C.CString(netlistText)
	defer C.free(unsafe.Pointer(cs))
	var h *C.tsb_job
	if rc := C.tsb_job_create(&ids[0], C.int(len(ids)), cs, C.int64_t(n), &h); rc != C.TSB_OK {
		return nil, fmt.Errorf("tsb_job_create: %s", C.GoString(C.tsb_last_error(nil)))
	}
	return &Job{h: h, N: n}, nil
}

func (j *Job) Close() { C.tsb_job_destroy(j.h); j.h = nil }

func (j *Job) err(what string) error { return fmt.Errorf("%s: %s", what, C.GoString(C.tsb_job_error(j.h))) }

// SetParam takes N values in job order; every GPU receives its slice.
func (j *Job) SetParam(device string, param int, values []float64) error {
	cs := C.CString(device)
	defer C.free(unsafe.Pointer(cs))
	d := C.tsb_plan_find_device(C.tsb_job_plan(j.h), cs)
	if d < 0 {
		return fmt.Errorf("device %s not found", device)
	}
	if rc := C.tsb_job_set_param(j.h, d, C.int(param), (*C.double)(unsafe.Pointer(&values[0]))); rc != C.TSB_OK {
		return j.err("tsb_job_set_param")
	}
	return nil
}

func (j *Job) RunTransient(tStart, tStop, tStep, tMax float64, uic bool, out int, capRows int64) error {
	u := C.int(0)
	if uic {
		u = 1
	}
	if rc := C.tsb_job_run_tran(j.h, C.double(tStart), C.double(tStop), C.double(tStep), C.double(tMax), u, C.int(out),
		C.int64_t(capRows), nil); rc != C.TSB_OK {
		return j.err("tsb_job_run_tran")
	}
	if rc := C.tsb_job_sync(j.h); rc != C.TSB_OK {
		return j.err("tsb_job_sync")
	}
	return nil
}

// Summary returns per column the minimum, maximum and sum over all instances and stored rows, the number of stored
// rows, and the job totals (accepted steps, rejected steps, transient solves, OP solves, executed solves).
func (j *Job) Summary(nColumns int) (min, max, sum []float64, rows int64, totals [5]int64, err error) {
	buf := make([]float64, 3*nColumns)
	var r C.int64_t
	var t [5]C.int64_t
	if rc := C.tsb_job_result_summary(j.h, (*C.double)(unsafe.Pointer(&buf[0])), &r, &t[0]); rc != C.TSB_OK {
		return nil, nil, nil, 0, totals, j.err("tsb_job_result_summary")
	}
	for k := range totals {
		totals[k] = int64(t[k])
	}
	return buf[:nColumns], buf[nColumns : 2*nColumns], buf[2*nColumns:], int64(r), totals, nil
}

// SetMeasures sets the measurement table of every GPU's shard.
func (j *Job) SetMeasures(m []Meas) error {
	t := measTable(m)
	var p *C.tsb_meas
	if len(t) > 0 {
		p = &t[0]
	}
	if rc := C.tsb_job_set_measures(j.h, p, C.int(len(t))); rc != C.TSB_OK {
		return j.err("tsb_job_set_measures")
	}
	j.nMeas = len(t)
	return nil
}

// Measures returns value[m][instance] and abscissa[m][instance] in job order.
func (j *Job) Measures() (value, abscissa [][]float64, err error) {
	flat := make([]float64, 2*int64(j.nMeas)*j.N+1)
	if rc := C.tsb_job_result_measures(j.h, (*C.double)(unsafe.Pointer(&flat[0]))); rc != C.TSB_OK {
		return nil, nil, j.err("tsb_job_result_measures")
	}
	value, abscissa = make([][]float64, j.nMeas), make([][]float64, j.nMeas)
	for m := 0; m < j.nMeas; m++ {
		value[m] = flat[int64(m)*j.N : int64(m+1)*j.N]
		abscissa[m] = flat[int64(j.nMeas+m)*j.N : int64(j.nMeas+m+1)*j.N]
	}
	return value, abscissa, nil
}

// SetFourier sets the Fourier table of every GPU's shard.
func (j *Job) SetFourier(f []Four) error {
	t, rows := fourTable(f)
	var p *C.tsb_four
	if len(t) > 0 {
		p = &t[0]
	}
	if rc := C.tsb_job_set_fourier(j.h, p, C.int(len(t))); rc != C.TSB_OK {
		return j.err("tsb_job_set_fourier")
	}
	j.nFour = rows
	return nil
}

// Fourier returns coeff[row][instance] in job order.
func (j *Job) Fourier() ([][]float64, error) {
	flat := make([]float64, int64(j.nFour)*j.N+1)
	if rc := C.tsb_job_result_fourier(j.h, (*C.double)(unsafe.Pointer(&flat[0]))); rc != C.TSB_OK {
		return nil, j.err("tsb_job_result_fourier")
	}
	out := make([][]float64, j.nFour)
	for r := range out {
		out[r] = flat[int64(r)*j.N : int64(r+1)*j.N]
	}
	return out, nil
}

func (j *Job) Status() ([]int32, error) {
	out := make([]int32, j.N)
	if rc := C.tsb_job_result_status(j.h, (*C.int32_t)(unsafe.Pointer(&out[0]))); rc != C.TSB_OK {
		return nil, j.err("tsb_job_result_status")
	}
	return out, nil
}
