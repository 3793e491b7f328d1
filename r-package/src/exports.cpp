// Exported functions of the B200-backed RcppSparse package (SURVEY.md 8f N1).
//
// columnSums keeps the reference's name, signature and result (reference src/example.cpp:26-32); its body is
// now the class call, which the drop-in header serves from the device.  The b200_* functions are additions:
// thin wrappers over the class methods (reference inst/include/RcppSparse.h:131-156, 375-385, the SpMV idiom
// and its k-column form spmm, and the column / row variances), and a persistent handle — an external pointer to a heap RcppSparse::Matrix whose device mirror
// therefore survives across .Call()s (one .Call otherwise builds a fresh Matrix, i.e. a fresh upload:
// reference src/RcppExports.cpp:20).
#include <RcppSparse.h>

//' Column sums of a dgCMatrix (same contract as the reference's exported example)
//' @param A a \code{dgCMatrix}
//' @return numeric vector of length \code{ncol(A)}
//' @export
//[[Rcpp::export]]
Rcpp::NumericVector columnSums(RcppSparse::Matrix& A) {
    return A.colSums();
}

//[[Rcpp::export]]
Rcpp::NumericVector b200_colSums(RcppSparse::Matrix& A) { return A.colSums(); }

//[[Rcpp::export]]
Rcpp::NumericVector b200_rowSums(RcppSparse::Matrix& A) { return A.rowSums(); }

//[[Rcpp::export]]
Rcpp::NumericVector b200_colMeans(RcppSparse::Matrix& A) { return A.colMeans(); }

//[[Rcpp::export]]
Rcpp::NumericVector b200_rowMeans(RcppSparse::Matrix& A) { return A.rowMeans(); }

//[[Rcpp::export]]
Rcpp::NumericVector b200_colVars(RcppSparse::Matrix& A) { return A.colVars(); }

//[[Rcpp::export]]
Rcpp::NumericVector b200_rowVars(RcppSparse::Matrix& A) { return A.rowVars(); }

//[[Rcpp::export]]
Rcpp::NumericVector b200_spmv(RcppSparse::Matrix& A, const Rcpp::NumericVector& v) { return A.spmv(v); }

//[[Rcpp::export]]
Rcpp::NumericVector b200_spmv_t(RcppSparse::Matrix& A, const Rcpp::NumericVector& v) { return A.spmv_t(v); }

//[[Rcpp::export]]
Rcpp::S4 b200_transpose(RcppSparse::Matrix& A) { return A.transpose().wrap(); }

//[[Rcpp::export]]
Rcpp::NumericMatrix b200_crossprod(RcppSparse::Matrix& A) { return A.crossprod(); }

//[[Rcpp::export]]
Rcpp::NumericMatrix b200_spmm(RcppSparse::Matrix& A, const Rcpp::NumericMatrix& B) { return A.spmm(B); }

//[[Rcpp::export]]
Rcpp::NumericMatrix b200_spmm_t(RcppSparse::Matrix& A, const Rcpp::NumericMatrix& B) { return A.spmm_t(B); }

// ---- persistent device-resident handle ---------------------------------------------------------------------
// The external pointer owns a heap Matrix; the Matrix holds Rcpp handles to the dgCMatrix slots (so R keeps them
// alive) and, after its first sweep, the device mirror.  The finalizer deletes the Matrix, which releases the
// mirror (sb200_matrix_destroy) — also reachable early through b200_release().
typedef Rcpp::XPtr<RcppSparse::Matrix> MatrixPtr;

//[[Rcpp::export]]
SEXP b200_device_matrix(const Rcpp::S4& A) {
    MatrixPtr ptr(new RcppSparse::Matrix(A), true);  // true: delete on garbage collection
    return ptr;
}

//[[Rcpp::export]]
Rcpp::NumericVector b200_dm_sweep(SEXP handle, int op) {
    MatrixPtr A(handle);
    switch (op) {
        case 0: return A->colSums();
        case 1: return A->rowSums();
        case 2: return A->colMeans();
        case 3: return A->rowMeans();
        case 4: return A->colVars();
        case 5: return A->rowVars();
        default: throw std::invalid_argument("b200_dm_sweep: unknown op");
    }
}

//[[Rcpp::export]]
Rcpp::NumericVector b200_dm_spmv(SEXP handle, const Rcpp::NumericVector& v, bool transposed) {
    MatrixPtr A(handle);
    return transposed ? A->spmv_t(v) : A->spmv(v);
}

//[[Rcpp::export]]
Rcpp::NumericMatrix b200_dm_spmm(SEXP handle, const Rcpp::NumericMatrix& B, bool transposed) {
    MatrixPtr A(handle);
    return transposed ? A->spmm_t(B) : A->spmm(B);
}

//[[Rcpp::export]]
Rcpp::NumericMatrix b200_dm_crossprod(SEXP handle) {
    MatrixPtr A(handle);
    return A->crossprod();
}

//[[Rcpp::export]]
Rcpp::S4 b200_dm_transpose(SEXP handle) {
    MatrixPtr A(handle);
    return A->transpose().wrap();
}

// after x was modified in place from R/C++ (the by-reference semantics of the reference's vignette,
// vignettes/Documentation.Rmd:325-347): re-upload the values
//[[Rcpp::export]]
void b200_refresh(SEXP handle) {
    MatrixPtr A(handle);
    A->refresh();
}

//[[Rcpp::export]]
void b200_release(SEXP handle) {
    MatrixPtr A(handle);
    A->release();
}
