"""Test infrastructure: the device source of the TSB_OUT_MEAS kernels on the host, through tests/host_emul.py.

host_emul compiles a netlist's kernel source with g++ behind a shim of the CUDA built-ins and runs whole analyses one
instance at a time.  This module reuses all of it and adds what a measurement run needs:
  * the kernel source of the batch's measurement table (`Batch.kernel_variant(meas=True)`: kind and columns are
    compiled in);
  * `__dsqrt_rn`, the one built-in the measurement code uses that the shim does not spell;
  * a driver that sets the table's run-time half (level, window, count, edge), adds TSB_OUT_MEAS to the run and writes
    the [2][n_meas][n] results after host_emul's own output.
The run-time half travels in the environment variable TSB_HOST_MEAS, so a new level reuses the compiled program, as it
reuses the kernel on the GPU."""
import os
import re
import subprocess

import numpy as np

import host_emul as H

T = H.T

_SHIM_EXTRA = "static inline double __dsqrt_rn(double a) { return sqrt(a); }\n"

_ANCHOR_ARGS = "    a.out_flags = (int)out_flags; a.cap_rows = cap_rows;"
_ARGS = _ANCHOR_ARGS + r'''
    // TSB_OUT_MEAS: level, from, to, count, edge per entry, whitespace-separated, in $TSB_HOST_MEAS
    std::vector<double> meas_out((size_t)2 * TSB_MEAS * n, 0.0);
    {
        const char* env = getenv("TSB_HOST_MEAS");
        char* q = (char*)env;
        for (int m = 0; m < TSB_MEAS; ++m) {
            a.meas_level[m] = strtod(q, &q); a.meas_from[m] = strtod(q, &q); a.meas_to[m] = strtod(q, &q);
            a.meas_count[m] = (int)strtod(q, &q); a.meas_edge[m] = (int)strtod(q, &q);
        }
    }
    a.out_flags |= TSB_OUT_MEAS | TSB_OUT_STATS;
    a.meas_out = meas_out.data();'''
_ANCHOR_OUT = "    fclose(f);\n    return 0;"
_OUT = "    fwrite(meas_out.data(), 8, meas_out.size(), f);\n" + _ANCHOR_OUT

_BUILT = {}


def _build(meas):
    """host_emul.build for the kernels of measurement table `meas` (same signature, same cache discipline)."""
    def build(text, overrides, tmpdir, strict=True, dc_src=-1, dc_src2=-1, opts_kw=None, grid=False):
        ckt = T.Circuit.from_netlist(text)
        b = ckt.batch(2)
        b.set_measures(meas)
        if dc_src != -1:
            b.kernel_variant(dc_src, dc_src2, meas=True)
        else:
            b.kernel_variant(grid=grid, meas=True)
        for (dev, par), vals in overrides.items():
            b.set_param(dev, par, np.resize(np.asarray(vals, dtype=np.float64), 2))
        opts = T.default_opts(**{**dict(strict_fp=1 if strict else 0, min_blocks=1, block_size=32, share_time_grid=0, coop_parts=0),
                                 **(opts_kw or {})})
        src = b.kernel_source(opts)
        info = dict(ckt=ckt, opts=opts,
                    slots=[(int(s), int(k)) for k, s in re.findall(r"P\[(\d+)\] = __ldcs\(a\.pv\[(\d+)\]", src)],
                    ncol_max=int(re.search(r"NCOL_MAX = (\d+)", src).group(1)), n=int(re.search(r"static constexpr int N = (\d+)", src).group(1)))
        key = (src, strict, tmpdir)
        if key in _BUILT:
            return _BUILT[key], info
        tag = f"m{len(_BUILT)}"
        cpp, exe = os.path.join(tmpdir, tag + ".cpp"), os.path.join(tmpdir, tag)
        host_src = src.replace("extern __shared__ double tsb_smem[];", "")
        for ptx, c in H._ASM_HOST:
            host_src = host_src.replace(ptx, c)
        assert H.MAIN.count(_ANCHOR_ARGS) == 1 and H.MAIN.count(_ANCHOR_OUT) == 1
        main = H.MAIN.replace(_ANCHOR_ARGS, _ARGS).replace(_ANCHOR_OUT, _OUT)
        with open(cpp, "w") as f:
            f.write(H.SHIM + _SHIM_EXTRA + host_src + main)
        flags = ["-O1", "-std=c++17", "-ffp-contract=off", "-w"] + ([] if strict else ["-DTSB_FAST_DIV"])
        r = subprocess.run(["g++"] + flags + ["-o", exe, cpp], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-4000:]
        _BUILT[key] = exe
        return exe, info
    return build


def run(text, n, overrides, tmpdir, meas, **kw):
    """host_emul.run with the measurement table `meas` (list of Meas) added to the run; returns (circuit, HostBatch,
    column names) with HostBatch.meas = [2: value, abscissa][n_meas][n]."""
    meas = list(meas)
    env_old = os.environ.get("TSB_HOST_MEAS")
    build_old = H.build
    os.environ["TSB_HOST_MEAS"] = " ".join(repr(float(v)) for m in meas for v in (m.level, m.from_, m.to, m.count, m.edge))
    H.build = _build(meas)            # host_emul.run looks its builder up by name at call time
    try:
        ckt, hb, cols = H.run(text, n, overrides, tmpdir, **kw)
    finally:
        H.build = build_old
        if env_old is None:
            del os.environ["TSB_HOST_MEAS"]
        else:
            os.environ["TSB_HOST_MEAS"] = env_old
    k = 2 * len(meas) * n
    raw = np.fromfile(os.path.join(tmpdir, "out.bin"), dtype=np.uint8)
    hb.meas = raw[raw.size - 8 * k:].view(np.float64).reshape(2, len(meas), n)
    return ckt, hb, cols
