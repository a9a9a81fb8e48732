"""toy-spice_b200 — B200-native batched FP64 circuit simulation (OP / DC sweep / transient) behind
the analysis API of edp1096/toy-spice.  See DESIGN.md.  The CUDA extension
(libtspice_b200.so, built by __graft_entry__.build()) is mandatory: there is no CPU path."""
from .api import (ACAnalysis, NewAC, OUT_AC_REFREAD, ST_AC_FAILED, AN_AC, AN_DC, AN_DC2, AN_OP, AN_TRAN, OUT_FOUR, OUT_GRID, OUT_MEAS, OUT_STATS, OUT_WAVE, EDGE_CROSS, EDGE_FALL, EDGE_RISE,
                  MEAS_AT, MEAS_AVG, MEAS_INTEG, MEAS_MAX, MEAS_MIN, MEAS_RMS, MEAS_WHEN, Meas, meas, Four, four, fourier_summary, Batch, Circuit, Context, DCSweep, Job, NewDCSweep,
                  NewOP, NewTransient, OperatingPoint, Opts, Transient, TsbError, analysis_from_card, default_opts,
                  lib, lib_path, lu_order)
from .report import format_results, format_value_factor, write_raw
from .workloads import BUNDLED

__all__ = [n for n in dir() if not n.startswith("_")]
