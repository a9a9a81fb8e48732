"""Test infrastructure: the generated `tsb_stamp` kernel (the direct-store form of tsb_batch_stamp_dev) compiled for the
host through tests/host_emul.py and run one "thread" per instance.

host_emul.build compiles a netlist's kernel source behind the CUDA shim; this module hands it a driver of its own instead
of host_emul.MAIN: it sets what tsb_batch_stamp_dev sets (mode, time, dt, gmin in `minstep`, A into `wave`, b into
`stats`, the flat parameters) and writes A [n_inst][n][n] and b [n_inst][n].  Several (mode, time, dt, gmin) cases run in
one process."""
import os
import subprocess

import numpy as np

import host_emul as H

T = H.T

MAIN = r'''
// ---- stamp driver: tsb_stamp, one kernel "thread" per instance, sequentially ----------------------------------------
static std::vector<char> slurp(const char* path) {
    FILE* f = fopen(path, "rb"); if (!f) { perror(path); exit(2); }
    fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
    std::vector<char> b(n); if (fread(b.data(), 1, n, f) != (size_t)n) exit(2); fclose(f); return b;
}
int main(int argc, char** argv) {
    std::vector<char> in = slurp(argv[1]);
    const long long* h = (const long long*)in.data();
    const long long n = h[0], nvar = h[1], npar = h[2], ncase = h[3];
    const double* cases = (const double*)(h + 4);             // ncase x {mode, time, dt, gmin}
    const double* p = cases + 4 * ncase;
    TsbArgs a; memset(&a, 0, sizeof a);
    a.n_inst = n; a.n_run = n;
    a.U = p; for (long long k = 0; k < npar && k < TSB_UC_MAX; ++k) a.Uc[k] = p[k];
    p += npar;
    for (long long s = 0; s < nvar; ++s) { a.pv[s] = p; p += n; }
    constexpr int NA = Ckt::N * Ckt::N, NB = Ckt::N;
    std::vector<double> A((size_t)n * NA), B((size_t)n * NB);
    a.wave = A.data(); a.stats = B.data();
    blockDim.x = TSB_BLOCK;
    FILE* f = fopen(argv[2], "wb");
    for (long long c = 0; c < ncase; ++c) {
        a.analysis = (int)cases[4 * c]; a.tstart = cases[4 * c + 1]; a.tstep = cases[4 * c + 2]; a.minstep = cases[4 * c + 3];
        std::fill(A.begin(), A.end(), 0.0); std::fill(B.begin(), B.end(), 0.0);
        for (long long i = 0; i < n; ++i) {
            blockIdx.x = (unsigned)(i / TSB_BLOCK); threadIdx.x = (unsigned)(i % TSB_BLOCK);
            tsb_stamp(a);
        }
        fwrite(A.data(), 8, A.size(), f); fwrite(B.data(), 8, B.size(), f);
    }
    fclose(f);
    return 0;
}
'''


def run(text, params, cases, tmpdir):
    """Stamp every instance of `params` {(device name, param): array [n_inst]} at every case (mode, time, dt, gmin) with the
    strict build of the host-compiled device source.  Returns [(A [n_inst][n][n], b [n_inst][n]) per case]."""
    exe, info = H.build(text, params, tmpdir, strict=True, main=MAIN)
    ckt = info["ckt"]
    n_inst = len(next(iter(params.values())))
    nominal, index = H._flat_parameters(ckt)
    flat_to_key = {v: k for k, v in index.items()}
    slot_of = dict(info["slots"])
    pv = [np.ascontiguousarray(params[flat_to_key[slot_of[s]]], dtype=np.float64) for s in range(len(slot_of))]
    hdr = np.array([n_inst, len(pv), len(nominal), len(cases)], dtype=np.int64)
    blob = hdr.tobytes() + np.asarray(cases, dtype=np.float64).reshape(-1).tobytes() + np.asarray(nominal, dtype=np.float64).tobytes() \
        + b"".join(v.tobytes() for v in pv)
    fin, fout = os.path.join(tmpdir, "stamp_in.bin"), os.path.join(tmpdir, "stamp_out.bin")
    with open(fin, "wb") as f:
        f.write(blob)
    r = subprocess.run([exe, fin, fout], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stderr[-2000:])
    n = info["n"]
    raw = np.fromfile(fout, dtype=np.float64).reshape(len(cases), -1)
    return [(row[: n_inst * n * n].reshape(n_inst, n, n), row[n_inst * n * n:].reshape(n_inst, n)) for row in raw]
