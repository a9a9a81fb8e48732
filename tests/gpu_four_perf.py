"""Cost of TSB_OUT_FOUR on the GPU: rlc and diode2 at 2^20 instances, statistics only against statistics plus one Fourier
entry (rlc: V(3), diode2: the output node V(2); 1 kHz, H = 9, G = 200, the last period), the two alternated three times
each in one process after a warm-up of each.
Reports ms per launch (host clock around run + sync), and per kernel the registers (ptxas, from the kernel cache) and the
blocks per SM those registers and the block's shared memory allow.  Development driver (not part of the suite):
    python tests/gpu_four_perf.py [out_file]"""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import parity_util as PU  # noqa: E402

T = PU.T
N = 1 << 20
REPS = 3
COLUMN = {"rlc": 3, "diode2": 2}          # V(3) of rlc, the output node V(2) of diode2


def card_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def kernel_figures(deck, table, opts_kw):
    """(registers, blocks per SM) of the transient kernel the run used: the launch-bounds choice recorded in the kernel
    cache (<autokey>.<gpu>.tuned, else .auto), then ptxas' register count of that kernel (<key>.info)."""
    cache = os.path.join(os.path.dirname(T.lib_path()), "_kcache")
    b = T.Circuit.from_netlist(T.BUNDLED[deck]).batch(2)
    for (dev, par), vals in PU.draws(deck, T.Circuit.from_netlist(T.BUNDLED[deck]), 2).items():
        b.set_param(dev, par, vals)
    if table:
        b.set_fourier(table)
        b.kernel_variant(four=True)
    autokey = b.kernel_key(T.default_opts(min_blocks=0, **opts_kw))
    mb = None
    for f in sorted(os.listdir(cache)):
        if f.startswith(autokey) and f.endswith(".tuned"):
            mb = int(open(os.path.join(cache, f)).read())
    if mb is None and os.path.exists(os.path.join(cache, autokey + ".auto")):
        mb = int(open(os.path.join(cache, autokey + ".auto")).read())
    key = b.kernel_key(T.default_opts(min_blocks=mb or 1, **opts_kw))
    regs = int(open(os.path.join(cache, key + ".info")).read().split()[0])
    ncol = len(T.Circuit.from_netlist(T.BUNDLED[deck]).columns(T.AN_TRAN))
    block = 128
    smem = (4 * ncol + 2 * len(table)) * block * 8 + 1024
    by_regs = 65536 // (((regs + 7) // 8) * 8 * block)
    by_smem = (228 * 1024) // smem
    return mb, regs, min(by_regs, by_smem)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    lines = [f"card: {card_info()}", f"instances: {N}, alternated {REPS}x, ms per launch (run_tran + sync, host clock)"]
    ctx = T.Context(0)
    for deck in ("rlc", "diode2"):
        text = T.BUNDLED[deck]
        ckt = T.Circuit.from_netlist(text, ctx)
        card = ckt.analysis_card()
        tran = (card["tstart"], card["tstop"], card["tstep"], card["tmax"], card["uic"])
        draws = PU.draws(deck, T.Circuit.from_netlist(text), N)
        batches = {}
        for name in ("stats", "stats+four"):
            b = ckt.batch(N)
            for (dev, par), vals in draws.items():
                b.set_param(dev, par, vals)
            batches[name] = b
        table = [T.four(COLUMN[deck], 1e3, n_harm=9, n_grid=200)]
        b0, b1 = batches["stats"], batches["stats+four"]
        b0.run_tran(*tran, out=T.OUT_STATS)          # warm-up (module load, launch-bounds timing)
        b0.sync()
        st = b0.stats_all()
        b1.set_fourier(table)
        b1.run_tran(*tran, out=T.OUT_STATS | T.OUT_FOUR)
        b1.sync()
        assert np.array_equal(b1.stats_all(), st, equal_nan=True), "statistics changed with the Fourier table on"
        times = {"stats": [], "stats+four": []}
        for _ in range(REPS):
            for name, flags in (("stats", T.OUT_STATS), ("stats+four", T.OUT_STATS | T.OUT_FOUR)):
                b = batches[name]
                t0 = time.perf_counter()
                b.run_tran(*tran, out=flags)
                b.sync()
                times[name].append((time.perf_counter() - t0) * 1e3)
        four = b1.fourier()
        m1 = T.fourier_summary(four, table)[0]["M"][0]
        for name, tab in (("stats", []), ("stats+four", table)):
            mb, regs, bps = kernel_figures(deck, tab, {})
            ts = times[name]
            lines.append(f"{deck:7s} {name:11s} ms/launch: " + " ".join(f"{t:8.2f}" for t in ts) +
                         f"   median {np.median(ts):8.2f}   min_blocks {mb}  regs {regs}  blocks/SM {bps}")
        ratio = np.median(times["stats+four"]) / np.median(times["stats"])
        lines.append(f"{deck:7s} overhead (median ratio): {100 * (ratio - 1):+.1f} %   "
                     f"finite coefficients: {np.isfinite(four).all(axis=0).mean():.3f}   median M_1: {np.nanmedian(m1):.4g}")
    text = "\n".join(lines)
    print(text)
    if out:
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
