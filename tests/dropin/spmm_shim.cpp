// Test harness for the block products of the drop-in C++ header (RcppSparse::Matrix::spmm / spmm_t): user-level code
// against include/RcppSparse.h, compiled with the Rcpp stand-in and linked to libsparse_b200 by tests/test_spmm_gpu.py.
// The extern "C" wrapper only moves raw arrays in and out so that pytest can drive it with ctypes.
#include <RcppSparse.h>  // the drop-in header from include/

#include <cstdint>
#include <cstring>
#include <string>

namespace {
thread_local std::string g_err;

RcppSparse::Matrix view(const int* i, const int* p, const double* x, int nrow, int ncol, int64_t nnz) {
  return RcppSparse::Matrix(Rcpp::NumericVector::view(const_cast<double*>(x), long(nnz)),
                            Rcpp::IntegerVector::view(const_cast<int*>(i), long(nnz)),
                            Rcpp::IntegerVector::view(const_cast<int*>(p), long(ncol) + 1),
                            Rcpp::IntegerVector({nrow, ncol}));
}
template <typename F>
int guarded(F f) {
  try {
    f();
    return 0;
  } catch (const std::invalid_argument& e) {
    g_err = std::string("invalid_argument: ") + e.what();
    return 1;
  } catch (const std::exception& e) {
    g_err = std::string("runtime_error: ") + e.what();
    return 2;
  }
}
}  // namespace

extern "C" {
const char* spmm_shim_last_error() { return g_err.c_str(); }

// Y = A B (transposed = 0) or A^T B through the header's NumericMatrix methods; B is b_rows x k column-major
int spmm_shim(int transposed, const int* i, const int* p, const double* x, int nrow, int ncol, int64_t nnz, const double* B,
              int64_t b_rows, int64_t k, double* Y) {
  return guarded([&] {
    RcppSparse::Matrix A = view(i, p, x, nrow, ncol, nnz);
    Rcpp::NumericMatrix b(b_rows, k);
    if (b_rows * k > 0) std::memcpy(b.begin(), B, sizeof(double) * size_t(b_rows * k));
    Rcpp::NumericMatrix y = transposed ? A.spmm_t(b) : A.spmm(b);
    if (y.nrow() != (transposed ? ncol : nrow) || y.ncol() != k) throw std::runtime_error("spmm: wrong shape");
    if (y.nrow() * k > 0) std::memcpy(Y, y.begin(), sizeof(double) * size_t(y.nrow() * k));
  });
}
}
