"""Test infrastructure: the device source of the TSB_OUT_FOUR kernels on the host, through tests/host_emul.py.

As tests/meas_host_emul.py does for measurements, this reuses host_emul's g++ build of a netlist's kernel source and adds
what a Fourier run needs:
  * the kernel source of the batch's Fourier table (`Batch.kernel_variant(four=True)`: columns and harmonics compiled in);
  * a driver that sets the table's run-time half (window start, grid spacing, G, the twiddles — computed with libm by the
    same expression the library uses), adds TSB_OUT_FOUR to the run and writes the coefficients after host_emul's output.
The run-time half travels in the environment variable TSB_HOST_FOUR, so a new window reuses the compiled program."""
import os
import re
import subprocess

import numpy as np

import four_ref as F
import host_emul as H

T = H.T

_ANCHOR_ARGS = "    a.out_flags = (int)out_flags; a.cap_rows = cap_rows;"
_ARGS = _ANCHOR_ARGS + r'''
    // TSB_OUT_FOUR: s, dt, G per entry, whitespace-separated, in $TSB_HOST_FOUR
    std::vector<double> four_tw;
    size_t four_rows = 0;
    {
        char* q = (char*)getenv("TSB_HOST_FOUR");
        for (int e = 0; e < TSB_FOUR; ++e) {
            a.four_s[e] = strtod(q, &q); a.four_dt[e] = strtod(q, &q); a.four_g[e] = (int)strtod(q, &q);
            const int G = a.four_g[e];
            a.four_tw_off[e] = (int)four_tw.size();
            four_tw.resize(four_tw.size() + 2 * (size_t)G);
            for (int j = 0; j < G; ++j) {
                four_tw[a.four_tw_off[e] + j] = cos(2.0 * M_PI * j / G);
                four_tw[a.four_tw_off[e] + G + j] = sin(2.0 * M_PI * j / G);
            }
            four_rows += 1 + 2 * tsb_four_spec(e).harm;
        }
    }
    std::vector<double> four_out(four_rows * n, 0.0);
    a.four_tw = four_tw.data(); a.four_out = four_out.data();
    a.out_flags |= TSB_OUT_FOUR | TSB_OUT_STATS;'''
_ANCHOR_OUT = "    fclose(f);\n    return 0;"
_OUT = "    fwrite(four_out.data(), 8, four_out.size(), f);\n" + _ANCHOR_OUT

_BUILT = {}


def _build(table):
    """host_emul.build for the kernels of Fourier table `table` (same signature, same cache discipline)."""
    def build(text, overrides, tmpdir, strict=True, dc_src=-1, dc_src2=-1, opts_kw=None, grid=False):
        ckt = T.Circuit.from_netlist(text)
        b = ckt.batch(2)
        b.set_fourier(table)
        b.kernel_variant(grid=grid, four=True)
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
        tag = f"f{len(_BUILT)}"
        cpp, exe = os.path.join(tmpdir, tag + ".cpp"), os.path.join(tmpdir, tag)
        host_src = src.replace("extern __shared__ double tsb_smem[];", "")
        for ptx, c in H._ASM_HOST:
            host_src = host_src.replace(ptx, c)
        assert H.MAIN.count(_ANCHOR_ARGS) == 1 and H.MAIN.count(_ANCHOR_OUT) == 1
        main = H.MAIN.replace(_ANCHOR_ARGS, _ARGS).replace(_ANCHOR_OUT, _OUT)
        with open(cpp, "w") as f:
            f.write(H.SHIM + host_src + main)
        flags = ["-O1", "-std=c++17", "-ffp-contract=off", "-w"] + ([] if strict else ["-DTSB_FAST_DIV"])
        r = subprocess.run(["g++"] + flags + ["-o", exe, cpp], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-4000:]
        _BUILT[key] = exe
        return exe, info
    return build


def run(text, n, overrides, tmpdir, table, tstop, **kw):
    """host_emul.run with the Fourier table `table` (list of Four) added to the run; `tstop` is the transient's (it ends
    a window with t_end = +inf).  Returns (circuit, HostBatch, column names) with HostBatch.four = [sum (1 + 2H)][n]."""
    table = list(table)
    env_old = os.environ.get("TSB_HOST_FOUR")
    build_old = H.build
    os.environ["TSB_HOST_FOUR"] = " ".join(f"{s!r} {dt!r} {f.n_grid}" for f in table for s, dt in [F.window(f, tstop)])
    H.build = _build(table)           # host_emul.run looks its builder up by name at call time
    try:
        ckt, hb, cols = H.run(text, n, overrides, tmpdir, **kw)
    finally:
        H.build = build_old
        if env_old is None:
            del os.environ["TSB_HOST_FOUR"]
        else:
            os.environ["TSB_HOST_FOUR"] = env_old
    k = sum(1 + 2 * f.n_harm for f in table) * n
    raw = np.fromfile(os.path.join(tmpdir, "out.bin"), dtype=np.uint8)
    hb.four = raw[raw.size - 8 * k:].view(np.float64).reshape(-1, n)
    return ckt, hb, cols
