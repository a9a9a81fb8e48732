"""Cost of TSB_OUT_MEAS on the GPU: rlc and diode2 at 2^20 instances, statistics only against statistics plus four
measurements (WHEN, AT, MAX, RMS), the two alternated three times each in one process after a warm-up of each.
Reports ms per launch (host clock around run + sync), and per kernel the registers (ptxas, from the kernel cache) and the
blocks per SM those registers and the block's shared memory allow.  Development driver (not part of the suite):
    python tests/gpu_meas_perf.py [out_file]"""
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
        b.set_measures(table)
        b.kernel_variant(meas=True)
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
    smem = (4 * ncol + 4 * len(table)) * block * 8 + 1024
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
        for name in ("stats", "stats+meas"):
            b = ckt.batch(N)
            for (dev, par), vals in draws.items():
                b.set_param(dev, par, vals)
            batches[name] = b
        b0 = batches["stats"]
        b0.run_tran(*tran, out=T.OUT_STATS)          # warm-up (module load, launch-bounds timing); gives the levels below
        b0.sync()
        st = b0.stats_all()
        level = float(0.5 * (st[0, 2, 0] + st[1, 2, 0]))
        table = [T.meas(T.MEAS_WHEN, 2, level), T.meas(T.MEAS_AT, 2, 0.5 * card["tstop"]), T.meas(T.MEAS_MAX, 1),
                 T.meas(T.MEAS_RMS, 2)]
        b1 = batches["stats+meas"]
        b1.set_measures(table)
        b1.run_tran(*tran, out=T.OUT_STATS | T.OUT_MEAS)
        b1.sync()
        assert np.array_equal(b1.stats_all(), st, equal_nan=True), "statistics changed with measurements on"
        times = {"stats": [], "stats+meas": []}
        for _ in range(REPS):
            for name, flags in (("stats", T.OUT_STATS), ("stats+meas", T.OUT_STATS | T.OUT_MEAS)):
                b = batches[name]
                t0 = time.perf_counter()
                b.run_tran(*tran, out=flags)
                b.sync()
                times[name].append((time.perf_counter() - t0) * 1e3)
        meas = b1.measures()
        for name, tab in (("stats", []), ("stats+meas", table)):
            mb, regs, bps = kernel_figures(deck, tab, {})
            ts = times[name]
            lines.append(f"{deck:7s} {name:11s} ms/launch: " + " ".join(f"{t:8.2f}" for t in ts) +
                         f"   median {np.median(ts):8.2f}   min_blocks {mb}  regs {regs}  blocks/SM {bps}")
        ratio = np.median(times["stats+meas"]) / np.median(times["stats"])
        lines.append(f"{deck:7s} overhead (median ratio): {100 * (ratio - 1):+.1f} %   "
                     f"finite WHEN results: {np.isfinite(meas[0, 0]).mean():.3f}")
    text = "\n".join(lines)
    print(text)
    if out:
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
