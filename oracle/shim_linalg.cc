// oracle/shim_linalg.cc -- builds oracle/_build/libsmcmc_shim.so.
//
// The ROOT linear algebra the reference calls, as restated in oracle/rootshim (ROOT itself is
// absent): exposed so that tests/test_oracle.py can hold it against LAPACK (numpy) -- an
// independent implementation -- on random symmetric positive definite matrices.  The shim is
// repository code and compiles on its own, so this check does not need the reference tree.
// TEST INFRASTRUCTURE ONLY.
#include <exception>
#include <string>

#include <TDecompChol.h>
#include <TMatrixD.h>
#include <TMatrixDSymEigen.h>
#include <TVectorD.h>

namespace {
std::string gLastError;
}

extern "C" {

const char* shim_last_error(void) { return gLastError.c_str(); }

//   which 0: TDecompChol::Decompose -> U (upper, U^T U = a)          TSimpleMCMC.H:1100-1118
//   which 1: TMatrixD::Invert                                          TSimpleHMC.H:806-812
//   which 2: TMatrixDSymEigen -> out = eigenvectors in columns, values = eigenvalues descending
//            (TSimpleMCMC.H:1287-1301, TSimpleHMC.H:786-800)
// Returns 0, 1 when the Cholesky factorisation fails, -1 on an exception (shim_last_error()).
int shim_linalg(int which, int n, const double* a, double* out, double* values) {
    try {
        if (which == 2) {
            TMatrixDSym m(n);
            for (int i = 0; i < n; ++i)
                for (int j = 0; j < n; ++j) m(i, j) = a[(size_t)i * n + j];
            TMatrixDSymEigen eig(m);
            const TMatrixD& v = eig.GetEigenVectors();
            const TVectorD& w = eig.GetEigenValues();
            for (int i = 0; i < n; ++i) {
                values[i] = w(i);
                for (int j = 0; j < n; ++j) out[(size_t)i * n + j] = v(i, j);
            }
            return 0;
        }
        TMatrixD m(n, n);
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) m(i, j) = a[(size_t)i * n + j];
        if (which == 0) {
            TDecompChol chol(m);
            if (!chol.Decompose()) return 1;
            const TMatrixD& u = chol.GetU();
            for (int i = 0; i < n; ++i)
                for (int j = 0; j < n; ++j) out[(size_t)i * n + j] = u(i, j);
            return 0;
        }
        m.Invert();
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) out[(size_t)i * n + j] = m(i, j);
        return 0;
    } catch (std::exception& e) {
        gLastError = e.what();
        return -1;
    }
}

}  // extern "C"
