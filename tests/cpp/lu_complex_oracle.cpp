// ORACLE — TEST INFRASTRUCTURE ONLY (tests/test_lu_operator_complex.py compiles it into a temporary directory).
// The reference's complex matrix operator on a batch of dense systems, written over the oracle's Sparse 1.3 restatement
// (oracle/sparse13.hpp), with the call sequence of its AC analysis: the first Factor() — order-and-factor — runs on the
// REAL nominal matrix and freezes the order (ac.go:33-49: the operating point goes through the same matrix first); every
// instance is then Clear / AddElement + AddComplexElement (get_element / get_element_imag) / FactorComplex / SolveComplex
// (pkg/matrix/circuit.go:73-83, 130, 140).  A, b, x interleaved complex: A[inst][row][col][re, im], b / x [inst][i][re, im].
// prow / pcol (n entries, 1-based external) return the frozen order.  Checker for tsb_lu_solve_batched_complex.
#include <cstdint>
#include <vector>

#include "sparse13.hpp"

using namespace orc;

extern "C" int orc_lu_batch_complex(int n, const double* A_nominal, int64_t n_inst, const double* A, const double* b, double* x,
                                    int32_t* status, int* prow, int* pcol) {
    Sparse13 m(n);
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) m.get_element(i + 1, j + 1) += A_nominal[i * n + j];
    if (m.factor() >= SP_ZERO_DIAG) return -1;
    for (int k = 1; k <= n; ++k) { prow[k - 1] = m.pivot_ext_row(k); pcol[k - 1] = m.pivot_ext_col(k); }
    std::vector<double> rre(n + 1), rim(n + 1), sre, sim;
    for (int64_t q = 0; q < n_inst; ++q) {
        m.clear();
        const double* Aq = A + q * n * n * 2;
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) {
                m.get_element(i + 1, j + 1) += Aq[(i * n + j) * 2];
                m.get_element_imag(i + 1, j + 1) += Aq[(i * n + j) * 2 + 1];
            }
        double* xq = x + q * n * 2;
        if (m.factor_complex() >= SP_ZERO_DIAG) {
            status[q] = 1;
            for (int i = 0; i < 2 * n; ++i) xq[i] = 0.0;
            continue;
        }
        rre[0] = rim[0] = 0.0;
        for (int i = 0; i < n; ++i) { rre[i + 1] = b[(q * n + i) * 2]; rim[i + 1] = b[(q * n + i) * 2 + 1]; }
        m.solve_complex(rre, rim, sre, sim);
        for (int i = 0; i < n; ++i) { xq[2 * i] = sre[i + 1]; xq[2 * i + 1] = sim[i + 1]; }
        status[q] = 0;
    }
    return 0;
}
