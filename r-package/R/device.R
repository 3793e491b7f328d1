# R-level surface of the persistent handle (SURVEY.md 8f N1).  A handle is an external pointer; methods take
# either a dgCMatrix (one upload per call) or a handle (mirror kept on the GPU between calls).

b200_device_matrix <- function(A) {
    stopifnot(methods::is(A, "dgCMatrix"))
    structure(list(ptr = .Call(`_RcppSparse_b200_device_matrix`, A), dim = dim(A)), class = "b200_matrix")
}

.b200_is_handle <- function(A) inherits(A, "b200_matrix")

.b200_sweep <- function(A, op, direct) {
    if (.b200_is_handle(A)) .Call(`_RcppSparse_b200_dm_sweep`, A$ptr, op) else direct(A)
}

b200_colSums  <- function(A) .b200_sweep(A, 0L, function(M) .Call(`_RcppSparse_b200_colSums`, M))
b200_rowSums  <- function(A) .b200_sweep(A, 1L, function(M) .Call(`_RcppSparse_b200_rowSums`, M))
b200_colMeans <- function(A) .b200_sweep(A, 2L, function(M) .Call(`_RcppSparse_b200_colMeans`, M))
b200_rowMeans <- function(A) .b200_sweep(A, 3L, function(M) .Call(`_RcppSparse_b200_rowMeans`, M))
# sample variances of the columns / rows (implicit zeros included, over n - 1, as var(A[, j]); NaN where var gives NA)
b200_colVars  <- function(A) .b200_sweep(A, 4L, function(M) .Call(`_RcppSparse_b200_colVars`, M))
b200_rowVars  <- function(A) .b200_sweep(A, 5L, function(M) .Call(`_RcppSparse_b200_rowVars`, M))

b200_spmv <- function(A, v) {
    v <- as.double(v)
    if (.b200_is_handle(A)) .Call(`_RcppSparse_b200_dm_spmv`, A$ptr, v, FALSE) else .Call(`_RcppSparse_b200_spmv`, A, v)
}

b200_spmv_t <- function(A, v) {
    v <- as.double(v)
    if (.b200_is_handle(A)) .Call(`_RcppSparse_b200_dm_spmv`, A$ptr, v, TRUE) else .Call(`_RcppSparse_b200_spmv_t`, A, v)
}

# A B (B: ncol(A) x k) and A^T B (B: nrow(A) x k) for a dense matrix of k right-hand sides, one sweep of A
b200_spmm <- function(A, B) {
    B <- as.matrix(B)
    storage.mode(B) <- "double"
    if (.b200_is_handle(A)) .Call(`_RcppSparse_b200_dm_spmm`, A$ptr, B, FALSE) else .Call(`_RcppSparse_b200_spmm`, A, B)
}

b200_spmm_t <- function(A, B) {
    B <- as.matrix(B)
    storage.mode(B) <- "double"
    if (.b200_is_handle(A)) .Call(`_RcppSparse_b200_dm_spmm`, A$ptr, B, TRUE) else .Call(`_RcppSparse_b200_spmm_t`, A, B)
}

b200_transpose <- function(A) {
    if (.b200_is_handle(A)) .Call(`_RcppSparse_b200_dm_transpose`, A$ptr) else .Call(`_RcppSparse_b200_transpose`, A)
}

b200_crossprod <- function(A) {
    if (.b200_is_handle(A)) .Call(`_RcppSparse_b200_dm_crossprod`, A$ptr) else .Call(`_RcppSparse_b200_crossprod`, A)
}

b200_refresh <- function(A) { stopifnot(.b200_is_handle(A)); invisible(.Call(`_RcppSparse_b200_refresh`, A$ptr)) }
b200_release <- function(A) { stopifnot(.b200_is_handle(A)); invisible(.Call(`_RcppSparse_b200_release`, A$ptr)) }

print.b200_matrix <- function(x, ...) cat("<b200 device-resident dgCMatrix ", x$dim[1], " x ", x$dim[2], ">\n", sep = "")
