// RcppSparse.h — drop-in replacement header: the same RcppSparse::Matrix class, with the
// data-parallel sweeps served by libsparse_b200 (NVIDIA B200, sm_100a) through the C ABI in
// sparse_b200.h.  No CPU fallback: if the library reports an error the method throws.
//
// Same public surface as the reference header (zdebruine/RcppSparse, inst/include/RcppSparse.h):
//   members x, i, p, Dim                                   reference :29-30   (zero-copy Rcpp handles)
//   constructors (4 vectors / S4 / default)                reference :33-42
//   rows cols nrow ncol n_nonzero nonzeros innerIndexPtr outerIndexPtr InnerNNZs   :44-51, :357-359
//   colSums rowSums colMeans rowMeans                      reference :131-156  -> sb200_col_sums ... sb200_row_means
//   crossprod                                              reference :158-194  -> sb200_crossprod / sb200_sharded_crossprod
//   transpose (and the vignette's t)                       reference :375-385  -> sb200_transpose / sb200_sharded_transpose
//   wrap, clone, at, operator(), operator[]                reference :387-394, :54-73 (host side, unchanged semantics)
//   InnerIterator                                          reference :218-233 (host side, unchanged)
//   Rcpp::traits::Exporter<RcppSparse::Matrix>             reference :398-423
// Additions: spmv(v) = A v and spmv_t(v) = A^T v (the reference only has the iterator idiom), spmm(B) = A B and
// spmm_t(B) = A^T B for a dense NumericMatrix of k right-hand sides (one sweep instead of k spmv calls),
// colVars() / rowVars() = the sample variance of every column / row (sparseMatrixStats::colVars / rowVars: implicit
// zeros included, over n - 1; NaN where R's var gives NA, n < 2), resident() to keep the device mirror between calls (then refresh() after mutating x in place, release() to
// drop it); SB200_GPUS=n runs the device ops on n GPUs of this process (sb200_sharded_*).
//   dense copies (operator()(rows, cols), col, row), InnerIndices, emptyInnerIndices, isAppxSymmetric,
//   InnerIteratorInRange / NotInRange, InnerRowIterator       reference :75-128, :196-216, :238-373 (host side; the
//   row iterator and the symmetry test do what their interfaces promise — the reference's own walk is broken)
//
// Include order: like the reference, this header must come BEFORE <Rcpp.h> in a translation unit
// (it forward-declares the Exporter specialisation between <RcppCommon.h> and <Rcpp.h>).
#ifndef RCPPSPARSE_B200_DROPIN_H
#define RCPPSPARSE_B200_DROPIN_H

#include <RcppCommon.h>

namespace RcppSparse {
class Matrix;
}

namespace Rcpp {
namespace traits {
template <>
class Exporter<RcppSparse::Matrix>;
}
}  // namespace Rcpp

#include <Rcpp.h>

#include <cstdlib>
#include <memory>
#include <vector>
#include <stdexcept>
#include <string>

#include "sparse_b200.h"

namespace RcppSparse {

namespace b200 {

// status -> C++ exception; BEGIN_RCPP/END_RCPP turn it into an R error (reference src/RcppExports.cpp:17,23)
inline void check(int status) {
  if (status == SB200_OK) return;
  const std::string what = std::string("libsparse_b200: ") + sb200_last_error();
  if (status == SB200_E_INVALID || status == SB200_E_STRUCTURE) throw std::invalid_argument(what);
  throw std::runtime_error(what);
}

inline int device_from_env() {
  const char* e = std::getenv("SB200_DEVICE");
  return e ? std::atoi(e) : 0;
}

inline int gpus_from_env() {
  const char* e = std::getenv("SB200_GPUS");
  const int n = e ? std::atoi(e) : 1;
  return n < 1 ? 1 : n;
}

// Owner of the device state of one Matrix.  Held through a shared_ptr: copies of a Matrix alias the same R
// vectors (Rcpp handle semantics), so they share it too; it is destroyed with the last copy.  There is no cache
// keyed by host address across objects — R may reuse addresses after a GC (SURVEY.md H4).
//
// The reference reads x / i / p LIVE on every call (its methods are loops over the R vectors, RcppSparse.h:131-156)
// and its vignette mutates them in place (Documentation.Rmd:325-347).  So by default nothing outlives a call here
// either: every method uploads the slots as they are NOW, runs, and drops the mirror — exactly what a fresh Matrix per
// .Call pays anyway (src/RcppExports.cpp:20).  Matrix::resident(true) opts into keeping the mirror (and the layouts
// the library caches on it) between calls; then an in-place change of x must be followed by refresh(), a change of
// i / p by release().
struct Mirror {
  sb200_matrix* handle = nullptr;    // one GPU
  sb200_sharded* sharded = nullptr;  // SB200_GPUS > 1: nnz-balanced column blocks on several GPUs of this process
  bool resident = false;
  // the slots the handles were uploaded from: if the public members are re-pointed afterwards
  // (m.x = other; the vignette allows it, Documentation.Rmd:235-236) a resident mirror is rebuilt
  const void *src_x = nullptr, *src_i = nullptr, *src_p = nullptr;
  long src_nnz = -1;
  int src_nrow = -1, src_ncol = -1;
  Mirror() = default;
  Mirror(const Mirror&) = delete;
  Mirror& operator=(const Mirror&) = delete;
  void drop() {
    if (handle) sb200_matrix_destroy(handle);
    if (sharded) sb200_sharded_destroy(sharded);
    handle = nullptr;
    sharded = nullptr;
  }
  ~Mirror() { drop(); }
};

}  // namespace b200

class Matrix {
public:
  // the dgCMatrix slots, aliased not copied
  Rcpp::NumericVector x;
  Rcpp::IntegerVector i, p, Dim;

  Matrix(Rcpp::NumericVector x_, Rcpp::IntegerVector i_, Rcpp::IntegerVector p_, Rcpp::IntegerVector Dim_)
      : x(x_), i(i_), p(p_), Dim(Dim_), mirror_(std::make_shared<b200::Mirror>()) {}

  Matrix(const Rcpp::S4& s) : mirror_(std::make_shared<b200::Mirror>()) {
    const char* needed[] = {"x", "p", "i", "Dim"};
    for (const char* name : needed)
      if (!s.hasSlot(name)) throw std::invalid_argument("Cannot construct RcppSparse::Matrix from this S4 object");
    x = s.slot("x");
    i = s.slot("i");
    p = s.slot("p");
    Dim = s.slot("Dim");
  }

  Matrix() : mirror_(std::make_shared<b200::Mirror>()) {}

  // ---- dimensions and handles ------------------------------------------------------------------
  unsigned int rows() { return Dim[0]; }
  unsigned int cols() { return Dim[1]; }
  unsigned int nrow() { return Dim[0]; }
  unsigned int ncol() { return Dim[1]; }
  unsigned int n_nonzero() { return x.size(); }
  Rcpp::NumericVector& nonzeros() { return x; }
  Rcpp::IntegerVector& innerIndexPtr() { return i; }
  Rcpp::IntegerVector& outerIndexPtr() { return p; }
  unsigned int InnerNNZs(int col) { return p[col + 1] - p[col]; }

  // deep copy of the four vectors; the copy gets its own (lazy) mirror
  Matrix clone() { return Matrix(Rcpp::clone(x), Rcpp::clone(i), Rcpp::clone(p), Rcpp::clone(Dim)); }

  // ---- point lookups stay on the host (latency-bound; rows are sorted inside a column) -------------
  double at(int row, int col) const {
    for (int k = p[col], end = p[col + 1]; k < end && i[k] <= row; ++k)
      if (i[k] == row) return x[k];
    return 0.0;
  }
  double operator()(int row, int col) const { return at(row, col); }
  double operator[](int index) const { return x[index]; }

  // ---- dense copies of parts of the matrix (reference :75-128; host side, same signatures) -------------
  // one row of selected columns, one column of selected rows, a block
  Rcpp::NumericVector operator()(int row, Rcpp::IntegerVector& col) {
    Rcpp::NumericVector out(col.size());
    for (long k = 0; k < col.size(); ++k) out[k] = at(row, col[k]);
    return out;
  }
  Rcpp::NumericVector operator()(Rcpp::IntegerVector& row, int col) {
    Rcpp::NumericVector out(row.size());
    for (long k = 0; k < row.size(); ++k) out[k] = at(row[k], col);
    return out;
  }
  Rcpp::NumericMatrix operator()(Rcpp::IntegerVector& row, Rcpp::IntegerVector& col) {
    Rcpp::NumericMatrix out(row.size(), col.size());
    for (long c = 0; c < col.size(); ++c)
      for (long r = 0; r < row.size(); ++r) out(r, c) = at(row[r], col[c]);
    return out;
  }
  // a column as a dense vector: scatter the stored entries over zeros
  Rcpp::NumericVector col(int c) {
    Rcpp::NumericVector dense(Dim[0]);
    for (int k = p[c], end = p[c + 1]; k < end; ++k) dense[i[k]] = x[k];
    return dense;
  }
  Rcpp::NumericMatrix col(Rcpp::IntegerVector& c) {
    Rcpp::NumericMatrix out(Dim[0], c.size());
    for (long j = 0; j < c.size(); ++j)
      for (int k = p[c[j]], end = p[c[j] + 1]; k < end; ++k) out(i[k], j) = x[k];
    return out;
  }
  // a row as a dense vector: one sorted lookup per column
  Rcpp::NumericVector row(int r) {
    Rcpp::NumericVector dense(Dim[1]);
    for (int c = 0; c < Dim[1]; ++c) {
      const int k = find_in_column(c, r);
      if (k >= 0) dense[c] = x[k];
    }
    return dense;
  }
  Rcpp::NumericMatrix row(Rcpp::IntegerVector& r) {
    Rcpp::NumericMatrix out(r.size(), Dim[1]);
    for (int c = 0; c < Dim[1]; ++c)
      for (long j = 0; j < r.size(); ++j) {
        const int k = find_in_column(c, r[j]);
        if (k >= 0) out(j, c) = x[k];
      }
    return out;
  }

  // rows with / without a stored entry in a column (reference :196-216)
  std::vector<unsigned int> InnerIndices(int col) {
    std::vector<unsigned int> rows_of;
    rows_of.reserve(p[col + 1] - p[col]);
    for (int k = p[col], end = p[col + 1]; k < end; ++k) rows_of.push_back(static_cast<unsigned int>(i[k]));
    return rows_of;
  }
  std::vector<unsigned int> emptyInnerIndices(int col) {
    std::vector<unsigned int> rows_without;
    rows_without.reserve(Dim[0] - (p[col + 1] - p[col]));
    int k = p[col];
    const int end = p[col + 1];
    for (int r = 0; r < Dim[0]; ++r) {
      if (k < end && i[k] == r)
        ++k;
      else
        rows_without.push_back(static_cast<unsigned int>(r));
    }
    return rows_without;
  }

  // A(r, c) == A(c, r) for every stored entry of a square matrix (what the reference's isAppxSymmetric, :362-373,
  // sets out to test; its own loop only compares the first column with a mis-walked first row)
  bool isAppxSymmetric() {
    if (Dim[0] != Dim[1]) return false;
    for (int c = 0; c < Dim[1]; ++c)
      for (int k = p[c], end = p[c + 1]; k < end; ++k)
        if (at(c, i[k]) != x[k]) return false;
    return true;
  }

  // ---- the sweeps: one kernel launch each behind the C ABI (per GPU when SB200_GPUS > 1) --------------------
  Rcpp::NumericVector colSums() {
    Rcpp::NumericVector sums(Dim[1]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_col_sums(l.s, sums.begin()) : sb200_col_sums(l.m, sums.begin()));
    return sums;
  }
  Rcpp::NumericVector rowSums() {
    Rcpp::NumericVector sums(Dim[0]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_row_sums(l.s, sums.begin()) : sb200_row_sums(l.m, sums.begin()));
    return sums;
  }
  Rcpp::NumericVector colMeans() {
    Rcpp::NumericVector means(Dim[1]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_col_means(l.s, means.begin()) : sb200_col_means(l.m, means.begin()));
    return means;
  }
  Rcpp::NumericVector rowMeans() {
    Rcpp::NumericVector means(Dim[0]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_row_means(l.s, means.begin()) : sb200_row_means(l.m, means.begin()));
    return means;
  }

  // sample variances, two passes around colMeans / rowMeans -> sb200_col_vars / sb200_row_vars (sb200_sharded_* on
  // several GPUs)
  Rcpp::NumericVector colVars() {
    Rcpp::NumericVector vars(Dim[1]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_col_vars(l.s, vars.begin()) : sb200_col_vars(l.m, vars.begin()));
    return vars;
  }
  Rcpp::NumericVector rowVars() {
    Rcpp::NumericVector vars(Dim[0]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_row_vars(l.s, vars.begin()) : sb200_row_vars(l.m, vars.begin()));
    return vars;
  }

  // dense A^T A (reference :158-194): ncol x ncol, exactly symmetric -> sb200_crossprod; on several GPUs
  // sb200_sharded_crossprod, which adds in the reference's row order (its result bit for bit)
  Rcpp::NumericMatrix crossprod() {
    Rcpp::NumericMatrix res(Dim[1], Dim[1]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_crossprod(l.s, res.begin()) : sb200_crossprod(l.m, res.begin()));
    return res;
  }

  // y = A v (v has ncol entries) and y = A^T v (v has nrow entries)
  Rcpp::NumericVector spmv(const Rcpp::NumericVector& v) {
    if (v.size() != Dim[1]) throw std::invalid_argument("spmv: v must have ncol entries");
    Rcpp::NumericVector y(Dim[0]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_spmv(l.s, v.begin(), y.begin()) : sb200_spmv(l.m, v.begin(), y.begin()));
    return y;
  }
  Rcpp::NumericVector spmv_t(const Rcpp::NumericVector& v) {
    if (v.size() != Dim[0]) throw std::invalid_argument("spmv_t: v must have nrow entries");
    Rcpp::NumericVector y(Dim[1]);
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_spmv_t(l.s, v.begin(), y.begin()) : sb200_spmv_t(l.m, v.begin(), y.begin()));
    return y;
  }

  // Y = A B (B: ncol x k) and Y = A^T B (B: nrow x k) for a dense block of k right-hand sides: one sweep of the matrix
  // instead of k calls of spmv / spmv_t, and one upload of it on a per-call mirror.  SB200_GPUS > 1: on that many GPUs.
  Rcpp::NumericMatrix spmm(const Rcpp::NumericMatrix& B) { return block_product(B, false); }
  Rcpp::NumericMatrix spmm_t(const Rcpp::NumericMatrix& B) { return block_product(B, true); }

  // canonical CSC of A^T; the result owns fresh R vectors (no call back into the R interpreter)
  Matrix transpose() {
    const long nnz = x.size();
    Rcpp::IntegerVector tp(long(Dim[0]) + 1), ti(nnz), tdim(2);
    Rcpp::NumericVector tx(nnz);
    tdim[0] = Dim[1];
    tdim[1] = Dim[0];
    Lease l(*this, true);
    b200::check(l.s ? sb200_sharded_transpose(l.s, tp.begin(), ti.begin(), tx.begin()) : sb200_transpose(l.m, tp.begin(), ti.begin(), tx.begin()));
    return Matrix(tx, ti, tp, tdim);
  }
  Matrix t() { return transpose(); }

  Rcpp::S4 wrap() {
    Rcpp::S4 s(std::string("dgCMatrix"));
    s.slot("x") = x;
    s.slot("i") = i;
    s.slot("p") = p;
    s.slot("Dim") = Dim;
    return s;
  }

  // Keep the device mirror (and the layouts the library caches on it) between calls instead of re-reading the R
  // vectors on every call like the reference does.  From then on: after changing x in place call refresh(), after
  // changing i / p call release().
  void resident(bool on = true) {
    mirror_->resident = on;
    if (!on) mirror_->drop();
  }
  bool is_resident() const { return mirror_->resident; }
  // re-upload x into a resident mirror (no-op otherwise: non-resident calls read x live)
  void refresh() {
    if (mirror_->handle) b200::check(sb200_matrix_refresh_values(mirror_->handle, x.begin()));
    if (mirror_->sharded) {  // the blocks are contiguous slices of x
      int n = 0;
      std::vector<int64_t> bounds(17, 0);
      b200::check(sb200_sharded_info(mirror_->sharded, &n, bounds.data()));
      for (int k = 0; k < n; ++k) {
        sb200_matrix* blk = nullptr;
        b200::check(sb200_sharded_block(mirror_->sharded, k, &blk));
        b200::check(sb200_matrix_refresh_values(blk, x.begin() + p[bounds[k]]));
      }
    }
  }
  void release() { mirror_->drop(); }

  // ---- column cursor, host side: same protocol as the reference ---------------------------------------
  class InnerIterator {
  public:
    InnerIterator(Matrix& m, int col) : m_(m), col_(col), at_(m.p[col]), end_(m.p[col + 1]) {}
    operator bool() const { return at_ < end_; }
    InnerIterator& operator++() {
      ++at_;
      return *this;
    }
    const double& value() const { return m_.x[at_]; }
    int row() const { return m_.i[at_]; }
    int col() const { return col_; }

  private:
    Matrix& m_;
    int col_, at_, end_;
  };

  // ---- stored entries of a column whose rows are (not) in a sorted list (reference :238-321, host side) ----
  // Same protocol as InnerIterator.  `rows` must be ascending; it is only read.  Two cursors advance in step
  // over the column's sorted rows and the list until they meet (InRange) / over the column skipping rows that
  // the list contains (NotInRange).
  class InnerIteratorInRange {
  public:
    InnerIteratorInRange(Matrix& m, int col, std::vector<unsigned int>& rows)
        : m_(m), rows_(rows), col_(col), at_(m.p[col]), end_(m.p[col + 1]), s_(0) {
      settle();
    }
    operator bool() const { return at_ < end_ && s_ < rows_.size(); }
    InnerIteratorInRange& operator++() {
      ++at_;
      ++s_;
      settle();
      return *this;
    }
    const double& value() const { return m_.x[at_]; }
    int row() const { return m_.i[at_]; }
    int col() const { return col_; }

  private:
    void settle() {  // advance whichever cursor is behind until both name the same row
      while (at_ < end_ && s_ < rows_.size()) {
        const unsigned int r = static_cast<unsigned int>(m_.i[at_]);
        if (r == rows_[s_]) return;
        if (r < rows_[s_])
          ++at_;
        else
          ++s_;
      }
    }
    Matrix& m_;
    const std::vector<unsigned int>& rows_;
    int col_, at_, end_;
    size_t s_;
  };

  class InnerIteratorNotInRange {
  public:
    InnerIteratorNotInRange(Matrix& m, int col, std::vector<unsigned int>& rows)
        : m_(m), rows_(rows), col_(col), at_(m.p[col]), end_(m.p[col + 1]), s_(0) {
      settle();
    }
    operator bool() const { return at_ < end_; }
    InnerIteratorNotInRange& operator++() {
      ++at_;
      settle();
      return *this;
    }
    const double& value() const { return m_.x[at_]; }
    int row() const { return m_.i[at_]; }
    int col() const { return col_; }

  private:
    void settle() {  // skip stored entries whose row the list contains
      while (at_ < end_) {
        const unsigned int r = static_cast<unsigned int>(m_.i[at_]);
        while (s_ < rows_.size() && rows_[s_] < r) ++s_;
        if (s_ < rows_.size() && rows_[s_] == r)
          ++at_;
        else
          return;
      }
    }
    Matrix& m_;
    const std::vector<unsigned int>& rows_;
    int col_, at_, end_;
    size_t s_;
  };

  // ---- stored entries of one row, in column order (reference :324-354; host side).  The reference's version
  // scans i[] as if it were laid out by row; this one does what its interface promises: a sorted lookup in each
  // column, cost O(ncol log(column length)).  For many rows use transpose() once instead. ----
  class InnerRowIterator {
  public:
    InnerRowIterator(Matrix& m, int row) : m_(m), row_(row), col_(-1), at_(-1) { ++(*this); }
    operator bool() const { return col_ < m_.Dim[1]; }
    InnerRowIterator& operator++() {
      for (++col_; col_ < m_.Dim[1]; ++col_) {
        at_ = m_.find_in_column(col_, row_);
        if (at_ >= 0) break;
      }
      return *this;
    }
    double& value() const { return m_.x[at_]; }
    int row() const { return row_; }
    int col() const { return col_; }

  private:
    Matrix& m_;
    int row_, col_, at_;
  };

private:
  Rcpp::NumericMatrix block_product(const Rcpp::NumericMatrix& B, bool transposed) {
    const long rows_b = transposed ? Dim[0] : Dim[1], rows_y = transposed ? Dim[1] : Dim[0];
    if (B.nrow() != rows_b)
      throw std::invalid_argument(transposed ? "spmm_t: B must have nrow rows" : "spmm: B must have ncol rows");
    Rcpp::NumericMatrix Y(rows_y, B.ncol());
    Lease l(*this, true);
    const double* b = const_cast<Rcpp::NumericMatrix&>(B).begin();  // only read
    if (l.s)
      b200::check(transposed ? sb200_sharded_spmm_t(l.s, b, B.ncol(), Y.begin()) : sb200_sharded_spmm(l.s, b, B.ncol(), Y.begin()));
    else
      b200::check(transposed ? sb200_spmm_t(l.m, b, B.ncol(), Y.begin()) : sb200_spmm(l.m, b, B.ncol(), Y.begin()));
    return Y;
  }

  // position of (row, col) in x / i, or -1: binary search in the column's sorted rows
  int find_in_column(int col, int row) const {
    int lo = p[col], hi = p[col + 1];
    while (lo < hi) {
      const int mid = lo + (hi - lo) / 2;
      if (i[mid] < row)
        lo = mid + 1;
      else
        hi = mid;
    }
    return (lo < p[col + 1] && i[lo] == row) ? lo : -1;
  }

  // Created with the object (empty), so that copies made at any time share one holder: a copy of a
  // Matrix aliases the same R vectors and must see the same device state.
  std::shared_ptr<b200::Mirror> mirror_;

  // The device handle(s) for one call: uploaded from the slots as they are now, dropped again at the end of the call
  // unless the Matrix is resident.  multi = the op has a several-GPU form (the sweeps, the block products, the
  // transpose and crossprod).
  struct Lease {
    b200::Mirror& mm;
    sb200_matrix* m = nullptr;
    sb200_sharded* s = nullptr;
    Lease(Matrix& A, bool multi) : mm(*A.mirror_) {
      const int gpus = multi ? b200::gpus_from_env() : 1;
      const bool same = mm.src_x == static_cast<const void*>(A.x.begin()) && mm.src_i == static_cast<const void*>(A.i.begin()) &&
                        mm.src_p == static_cast<const void*>(A.p.begin()) && mm.src_nnz == long(A.x.size()) &&
                        mm.src_nrow == A.Dim[0] && mm.src_ncol == A.Dim[1];
      if (!mm.resident || !same) mm.drop();
      if (A.Dim.size() != 2 || A.p.size() != long(A.Dim[1]) + 1 || A.i.size() != A.x.size())
        throw std::invalid_argument("RcppSparse::Matrix: slot lengths inconsistent with Dim");
      if (gpus > 1) {
        if (!mm.sharded)
          b200::check(sb200_sharded_create(A.i.begin(), A.p.begin(), A.x.begin(), A.Dim[0], A.Dim[1], A.x.size(), gpus, nullptr, 0u,
                                           &mm.sharded));
        s = mm.sharded;
      } else {
        if (!mm.handle)
          // a per-call mirror (dropped by ~Lease while the slots are still protected) leaves `i` on the host until an op
          // reads it: colSums / colMeans never do (reference :133-135), so they upload 8 of the 12 bytes per entry
          b200::check(sb200_matrix_create(A.i.begin(), A.p.begin(), A.x.begin(), A.Dim[0], A.Dim[1], A.x.size(),
                                          b200::device_from_env(), mm.resident ? 0u : SB200_LAZY_ROWS, &mm.handle));
        m = mm.handle;
      }
      mm.src_x = A.x.begin();
      mm.src_i = A.i.begin();
      mm.src_p = A.p.begin();
      mm.src_nnz = long(A.x.size());
      mm.src_nrow = A.Dim[0];
      mm.src_ncol = A.Dim[1];
    }
    ~Lease() {
      if (!mm.resident) mm.drop();
    }
    Lease(const Lease&) = delete;
    Lease& operator=(const Lease&) = delete;
  };
};

}  // namespace RcppSparse

namespace Rcpp {
namespace traits {

// Rcpp::as<RcppSparse::Matrix>: capture the four slot handles of a dgCMatrix, no copy
template <>
class Exporter<RcppSparse::Matrix> {
public:
  Exporter(SEXP obj) : s_(obj) {
    if (!s_.hasSlot("x") || !s_.hasSlot("p") || !s_.hasSlot("i") || !s_.hasSlot("Dim"))
      throw std::invalid_argument("Cannot construct RcppSparse::Matrix from this S4 object");
  }
  RcppSparse::Matrix get() { return RcppSparse::Matrix(s_); }

private:
  Rcpp::S4 s_;
};

}  // namespace traits
}  // namespace Rcpp

#endif  // RCPPSPARSE_B200_DROPIN_H
