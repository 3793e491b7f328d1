// Test harness for the variances of the drop-in C++ header (RcppSparse::Matrix::colVars / rowVars): user-level code
// against include/RcppSparse.h, compiled with the Rcpp stand-in and linked to libsparse_b200 by tests/test_vars_cpu.py.
// The extern "C" wrapper only moves raw arrays in and out so that pytest can drive it with ctypes.
#include <RcppSparse.h>  // the drop-in header from include/

#include <cstdint>
#include <cstring>
#include <string>

namespace {
thread_local std::string g_err;
}  // namespace

extern "C" {
const char* vars_shim_last_error() { return g_err.c_str(); }

// rows = 0: out[ncol] = A.colVars(); rows = 1: out[nrow] = A.rowVars().  0 on success, 2 when the header threw.
int vars_shim(int rows, const int* i, const int* p, const double* x, int nrow, int ncol, int64_t nnz, double* out) {
  try {
    RcppSparse::Matrix A(Rcpp::NumericVector::view(const_cast<double*>(x), long(nnz)),
                         Rcpp::IntegerVector::view(const_cast<int*>(i), long(nnz)),
                         Rcpp::IntegerVector::view(const_cast<int*>(p), long(ncol) + 1), Rcpp::IntegerVector({nrow, ncol}));
    Rcpp::NumericVector v = rows ? A.rowVars() : A.colVars();
    if (v.size() != (rows ? nrow : ncol)) throw std::runtime_error("vars: wrong length");
    if (v.size() > 0) std::memcpy(out, v.begin(), sizeof(double) * size_t(v.size()));
    return 0;
  } catch (const std::exception& e) {
    g_err = std::string("runtime_error: ") + e.what();
    return 2;
  }
}
}
