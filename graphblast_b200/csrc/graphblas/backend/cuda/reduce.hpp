// graphblast_b200 backend — monoid reductions (vector -> scalar, matrix -> scalar,
// matrix rows -> vector).
//
// Replaces reference graphblas/backend/cuda/reduce.hpp:13-145.  Kept behaviour:
// an empty input returns the identity (:23-26); in struct-only mode a sparse
// vector / matrix reduces to its entry count (:71-72, :87-88).
// New: a dense 0/1 vector produced by the fused Boolean pull carries its count,
// so a plus-reduce over it is one 8-byte read instead of a pass over 4n bytes.
#ifndef GRAPHBLAS_BACKEND_CUDA_REDUCE_HPP_
#define GRAPHBLAS_BACKEND_CUDA_REDUCE_HPP_

#include <iostream>

#include "graphblas/backend/cuda/kernels/kernels.hpp"

namespace graphblas {
namespace backend {

// Second launch of a reduction: one CTA folds the per-CTA partials; a 32-bit
// result is posted to the host mailbox (no stream synchronisation).
template <typename T, typename MonoidT>
Info reduceFold(T* val, MonoidT op, T* partials, int grid) {
  T* d_out = partials + grid;
  cudaStream_t s = gbStream();
  const bool mail = sizeof(T) == 4;
  const unsigned long long ticket = mail ? runtime().mailTicket() : 0ull;
  reduceFinalKernel<<<1, GB_REDUCE_NT, 0, s>>>(d_out, partials, grid, op,
      static_cast<T>(op.identity()), mail ? runtime().mailSlot(2) : NULL, ticket);
  GB_KERNEL_CHECK();
  if (mail) {
    // fallback cell holds a T; read it as such if the post is lost
    volatile unsigned long long* slot = runtime().h_mail + 2;
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned long long spin = 0;; ++spin) {
      const unsigned long long v = *slot;
      if ((v >> 40) == ticket) {
        const unsigned int bits = static_cast<unsigned int>(v & 0xffffffffull);
        memcpy(val, &bits, 4);
        return GrB_SUCCESS;
      }
      if ((spin & 0x3ff) == 0x3ff &&
          std::chrono::steady_clock::now() - t0 > std::chrono::seconds(2))
        break;
    }
  }
  *val = runtime().fetch(d_out);
  return GrB_SUCCESS;
}

// Grid of the first launch and the scratch its partials (+ the result cell) live in.
template <typename T>
T* reducePartials(Index nvals, Descriptor* desc, int* grid) {
  *grid = gridFor(nvals, GB_REDUCE_NT, 4);
  return reinterpret_cast<T*>(desc->scratch(GB_SCRATCH_BLOCKSUM,
      (static_cast<size_t>(*grid) + 1)*sizeof(T)));
}

template <typename T, typename U,
          typename BinaryOpT, typename MonoidT>
Info reduceCommon(T* val, BinaryOpT accum, MonoidT op, const U* d_val, Index nvals,
    Descriptor* desc) {
  if (nvals == 0) {
    *val = op.identity();
    return GrB_SUCCESS;
  }
  int grid;
  T* partials = reducePartials<T>(nvals, desc, &grid);
  reducePartialKernel<<<grid, GB_REDUCE_NT, 0, gbStream()>>>(partials, d_val, nvals, op,
      static_cast<T>(op.identity()));
  GB_KERNEL_CHECK();
  return reduceFold(val, op, partials, grid);
}

// ---- container -> scalar ------------------------------------------------------------
// What a reduction folds: the stored values of a container and how many there are.
namespace reduce_detail {
template <typename U> const U* stored(const SparseVector<U>* x) { return x->d_val_; }
template <typename U> const U* stored(const SparseMatrix<U>* x) { return x->d_csrVal_; }
template <typename U> Index    count(const SparseVector<U>* x)  { return x->nvals_; }
template <typename U> Index    count(const SparseMatrix<U>* x)  { return x->nvals_; }
}  // namespace reduce_detail

// Sparse vector or sparse matrix: in struct-only mode the result is the entry count
// (reference :71-72, :87-88), else the fold of the stored values.
template <typename T, typename Container, typename BinaryOpT, typename MonoidT>
Info reduceStored(T* val, BinaryOpT accum, MonoidT op, const Container* x,
                  Descriptor* desc) {
  if (desc->struconly()) {
    *val = reduce_detail::count(x);
    return GrB_SUCCESS;
  }
  return reduceCommon(val, accum, op, reduce_detail::stored(x), reduce_detail::count(x),
                      desc);
}

// Dense vector.  A 0/1 vector left by the fused Boolean pull carries its count: a
// plus-like monoid over it is that count, no pass over the values.
template <typename T, typename U, typename BinaryOpT, typename MonoidT>
Info reduceDense(T* val, BinaryOpT accum, MonoidT op, DenseVector<U>* u,
                 Descriptor* desc) {
  const bool counts_ones = u->zero_one_ && op(3, 5) == 8 &&
                           op.identity() == static_cast<T>(0);
  if (counts_ones) {
    Index ones;
    CHECK(u->computeNnz(&ones, static_cast<U>(0), desc));
    *val = static_cast<T>(ones);
    return GrB_SUCCESS;
  }
  CHECK(u->materialize());
  return reduceCommon(val, accum, op, u->d_val_, u->nvals_, desc);
}

// ---- sparse matrix rows -> dense vector (out-degrees of PageRank) -------------------
// Struct-only mode leaves w untouched, as the reference does (:123-124).
template <typename W, typename a, typename MonoidT>
Info reduceRows(DenseVector<W>* w, MonoidT op, const SparseMatrix<a>* A, Descriptor* desc) {
  if (desc->struconly()) return GrB_SUCCESS;
  if (A->nrows_ == 0) return GrB_INVALID_OBJECT;
  CHECK(w->allocateGpu());
  const size_t lanes = static_cast<size_t>(A->nrows_)*32;          // a warp per row
  reduceRowsKernel<<<gridFor(lanes, 256), 256, 0, gbStream()>>>(w->d_val_,
      A->d_csrRowPtr_, A->d_csrVal_, A->nrows_, op, static_cast<W>(op.identity()));
  GB_KERNEL_CHECK();
  w->touched();
  w->nnz_ = A->nrows_;
  return GrB_SUCCESS;
}

}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_REDUCE_HPP_
