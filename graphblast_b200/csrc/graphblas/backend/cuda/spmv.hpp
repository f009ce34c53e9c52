// graphblast_b200 backend — pull-direction mxv host: w = A' (+.x) u with a dense
// u, A' = CSR rows of A, or CSC columns of A when the descriptor says transposed
// (vxm toggles GrB_INP1, so vxm pulls over the CSC).
//
// Replaces reference graphblas/backend/cuda/spmv.hpp:20-236.  Same decision:
//   mask given, --fusedmask 1 and the semiring's add is logical-or
//   (add_op(3,5) == 1, reference :84-96)  -> fused masked Boolean kernel;
//   otherwise                              -> generic merge-path SpMV, then the
//   mask pass that writes identity where masked out (:203-212), then the accum
//   pass that combines with the semiring's ADD (:213-219 — the reference ignores
//   the accum functor itself).
#ifndef GRAPHBLAS_BACKEND_CUDA_SPMV_HPP_
#define GRAPHBLAS_BACKEND_CUDA_SPMV_HPP_

#include <iostream>
#include <string>

#include "graphblas/backend/cuda/kernels/kernels.hpp"
#include "graphblas/backend/cuda/spmv_hub.hpp"

namespace graphblas {
namespace backend {

// Generic SpMV into `out` (raw result, no mask/accum).  2 launches (+1 the first
// time a matrix is used, to compute its tile partition).
template <typename W, typename a, typename U, typename SemiringT>
Info spmvMergeLaunch(W* out, const Index* tile_rows, SemiringT op, const Index* rowptr,
    const Index* colind, const a* val, const U* u, Index nrows, Index nnz,
    Descriptor* desc) {
  if (nrows <= 0) return GrB_SUCCESS;
  const long long total = static_cast<long long>(nrows) + nnz;
  const int nctas = static_cast<int>((total + GB_SPMV_TILE - 1)/GB_SPMV_TILE);
  Index* carry_row = reinterpret_cast<Index*>(desc->scratch(
      GB_SCRATCH_CARRY_ROW, static_cast<size_t>(nctas)*sizeof(Index)));
  W* carry_val = reinterpret_cast<W*>(desc->scratch(
      GB_SCRATCH_CARRY_VAL, static_cast<size_t>(nctas)*sizeof(W)));
  cudaStream_t s = gbStream();

  const bool aligned =
      (reinterpret_cast<uintptr_t>(colind) % 32 == 0) &&
      (reinterpret_cast<uintptr_t>(val)    % 32 == 0) &&
      sizeof(a) == 4 && sizeof(Index) == 4;
  const double alg_bytes = 8.0*nnz + 12.0*nrows + 4.0;
  profiler().begin(GB_PROF_SPMV_MERGE, s);
  typedef decltype(extractMul(op)) MulT;
  typedef decltype(extractAdd(op)) AddT;
  static bool configured = false;      // once per instantiation
  if (!configured) {
    cudaFuncSetAttribute(spmvMergeKernelT<GB_SPMV_NT, GB_SPMV_IPT, true, true, false, W, a, U, MulT, AddT>,
        cudaFuncAttributePreferredSharedMemoryCarveout, GB_SPMV_CARVEOUT);
    cudaFuncSetAttribute(spmvMergeKernelT<GB_SPMV_NT, GB_SPMV_IPT, false, true, true, W, a, U, MulT, AddT>,
        cudaFuncAttributePreferredSharedMemoryCarveout, GB_SPMV_CARVEOUT);
    configured = true;
  }
  // 256-bit loads, 8 consecutive nonzeros per thread, where the arrays are 32-byte
  // aligned; otherwise 32-bit loads, lanes on consecutive nonzeros.
  if (!aligned && sizeof(a) == 4)
    spmvMergeKernelT<GB_SPMV_NT, GB_SPMV_IPT, false, true, true><<<nctas, GB_SPMV_NT, 0, s>>>(out, tile_rows, carry_row,
        carry_val, rowptr, colind, val, u, nrows, nnz, op.identity(),
        extractMul(op), extractAdd(op));
  else if (aligned)
    spmvMergeKernelT<GB_SPMV_NT, GB_SPMV_IPT, true, true, false><<<nctas, GB_SPMV_NT, 0, s>>>(out, tile_rows, carry_row,
        carry_val, rowptr, colind, val, u, nrows, nnz, op.identity(),
        extractMul(op), extractAdd(op));
  else
    spmvMergeKernelT<GB_SPMV_NT, GB_SPMV_IPT, false, true, false><<<nctas, GB_SPMV_NT, 0, s>>>(out, tile_rows, carry_row,
        carry_val, rowptr, colind, val, u, nrows, nnz, op.identity(),
        extractMul(op), extractAdd(op));
  GB_KERNEL_CHECK();
  spmvCarryFixupKernel<<<(nctas + 255)/256, 256, 0, s>>>(out, carry_row,
      carry_val, nctas, extractAdd(op));
  GB_KERNEL_CHECK();
  profiler().end(GB_PROF_SPMV_MERGE, s, alg_bytes);
  return GrB_SUCCESS;
}

// Generic SpMV through the hub-cached kernel: 3 launches (pre-pass: hub values +
// identity for the empty rows; the persistent SpMV kernel; carry fix-up).
template <typename W, typename a, typename U, typename SemiringT>
Info spmvHubLaunch(W* out, const HubIndex& h, SemiringT op, const a* val, const U* u,
    Index nrows, Index nnz, Descriptor* desc) {
  Index* carry_row = reinterpret_cast<Index*>(desc->scratch(
      GB_SCRATCH_CARRY_ROW, static_cast<size_t>(h.ntiles)*sizeof(Index)));
  W* carry_val = reinterpret_cast<W*>(desc->scratch(
      GB_SCRATCH_CARRY_VAL, static_cast<size_t>(h.ntiles)*sizeof(W)));
  cudaStream_t s = gbStream();
  profiler().begin(GB_PROF_SPMV_MERGE, s);
  spmvHubRun<GB_HUB_GROUPS, GB_HUB_CAPACITY>(out, h, op, val, u, nnz, carry_row,
      carry_val, s);
  profiler().end(GB_PROF_SPMV_MERGE, s, 8.0*nnz + 12.0*nrows + 4.0);
  return GrB_SUCCESS;
}

template <typename W, typename a, typename U, typename M,
          typename BinaryOpT,      typename SemiringT>
Info spmv(DenseVector<W>* w, const Vector<M>* mask, BinaryOpT accum, SemiringT op,
    const SparseMatrix<a>* A, const DenseVector<U>* u, Descriptor* desc) {
  // Get descriptor parameters for SCMP, REPL, TRAN
  Desc_value scmp_mode, repl_mode, inp0_mode, inp1_mode;
  CHECK(desc->get(GrB_MASK, &scmp_mode));
  CHECK(desc->get(GrB_OUTP, &repl_mode));
  CHECK(desc->get(GrB_INP0, &inp0_mode));
  CHECK(desc->get(GrB_INP1, &inp1_mode));

  const bool use_mask  = (mask != NULL);
  const bool use_accum = !AccumIsNull<BinaryOpT>::value;
  const bool use_scmp  = (scmp_mode == GrB_SCMP);
  const bool use_repl  = (repl_mode == GrB_REPLACE);
  const bool use_tran  = (inp0_mode == GrB_TRAN || inp1_mode == GrB_TRAN);

  if (desc->debug()) {
    std::cout << "Executing Spmv\n";
    printState(use_mask, use_accum, use_scmp, use_repl, use_tran);
  }

  // Transpose (default is CSR):
  const Index* A_csrRowPtr = (use_tran) ? A->d_cscColPtr_ : A->d_csrRowPtr_;
  const Index* A_csrColInd = (use_tran) ? A->d_cscRowInd_ : A->d_csrColInd_;
  const a*     A_csrVal    = (use_tran) ? A->d_cscVal_    : A->d_csrVal_;
  const Index  A_nrows     = (use_tran) ? A->ncols_       : A->nrows_;
  if (A_csrRowPtr == NULL) return GrB_UNINITIALIZED_OBJECT;

  DenseVector<U>* u_t = const_cast<DenseVector<U>*>(u);
  CHECK(w->allocateGpu());
  CHECK(u_t->allocateGpu());

  // Which atomic the semiring's add behaves like (reference spmv.hpp:76-85).
  auto add_op = extractAdd(op);
  int functor = add_op(3, 5);

  if (desc->struconly() && functor != 1)
    std::cout << "Warning: Using structure-only mode and not using logical or "
        << "semiring may result in unintended behaviour. Is this intended?\n";

  cudaStream_t s = gbStream();

  if (use_mask && desc->fusedmask() && functor == 1) {
    Storage mask_vec_type;
    CHECK(mask->getStorage(&mask_vec_type));

    if (mask_vec_type == GrB_DENSE) {
      unsigned long long* ctr = w->countCell();
      CUDA_CALL(cudaMemsetAsync(ctr, 0, sizeof(unsigned long long), s));

      int variant = 0;
      variant |= use_scmp          ? 4 : 0;
      variant |= desc->earlyexit() ? 2 : 0;
      variant |= desc->opreuse()   ? 1 : 0;

      unsigned long long* prof_cell = NULL;
      if (profiler().enabled) {
        profiler().ensureCells();
        prof_cell = profiler().d_cells + GB_PROF_PULL_BOOL;
      }

      // Bitmap form whenever the Boolean semiring's identity is 0 (the test
      // "u[col] != identity" is then exactly a bit of u's shadow).  The shadows
      // of the visited mask and of the frontier are kept current by fill(),
      // assign() and this kernel itself, so inside a BFS no conversion pass runs;
      // a stale shadow costs one 4n-byte pass here.
      const bool bits_form = (op.identity() == static_cast<U>(0));
      unsigned long long mail_ticket = 0ull;
      double fixed_bytes;
      if (bits_form) {
        DenseVector<M>* mask_dense =
            const_cast<DenseVector<M>*>(&mask->dense_);
        const unsigned int* mask_bits = mask_dense->ensureBits();
        const unsigned int* u_bits =
            desc->opreuse() ? mask_bits : u_t->ensureBits();
        unsigned int* w_bits = w->bitsStorage();
        const int grid = gridFor(A_nrows, GB_PULL_NT, 8);
        // First-neighbour summary of this structure, computed once per matrix.
        SparseMatrix<a>* A_f = const_cast<SparseMatrix<a>*>(A);
        const int fw = use_tran ? 1 : 0;
        const Index* A_first = pullFirstNeighbours(A_f, fw, A_csrRowPtr, A_csrColInd,
                                                   A_nrows);
        // The 0/1 result is published through the bitmap shadow only; the value
        // array is written when somebody asks for it (DenseVector::materialize).
        W* const w_out = NULL;
        mail_ticket = runtime().mailTicket();
        unsigned long long* mail = runtime().mailSlot(1);
        unsigned long long* done = desc->counters() + 4;
#define GB_LAUNCH_PULL(SC, EE, OR)                                           \
        spmvMaskedOrPullBitsKernel<SC, EE, OR><<<grid, GB_PULL_NT, 0, s>>>(  \
            w_out, w_bits, mask_bits, u_bits, A_nrows, A_first,              \
            A_csrRowPtr, A_csrColInd, ctr, prof_cell, done, mail, mail_ticket)
        profiler().begin(GB_PROF_PULL_BOOL, s);
        switch (variant) {
          case 0: GB_LAUNCH_PULL(false, false, false); break;
          case 1: GB_LAUNCH_PULL(false, false, true ); break;
          case 2: GB_LAUNCH_PULL(false, true,  false); break;
          case 3: GB_LAUNCH_PULL(false, true,  true ); break;
          case 4: GB_LAUNCH_PULL(true,  false, false); break;
          case 5: GB_LAUNCH_PULL(true,  false, true ); break;
          case 6: GB_LAUNCH_PULL(true,  true,  false); break;
          case 7: GB_LAUNCH_PULL(true,  true,  true ); break;
          default: break;
        }
#undef GB_LAUNCH_PULL
        // Algorithmic bytes as SURVEY.md §8d defines them for a Boolean pull
        // level, at the API's types: 4(n+1) rowptr + 4n visited + 4n written,
        // plus 4 bytes per colind entry inspected (counted by the kernel; the
        // first-neighbour summary is colind[rowptr[row]]).  The kernel itself
        // moves fewer bytes (bitmaps, lazy values) — that is the saving.
        fixed_bytes = 12.0*A_nrows + 4.0;
      } else {
        CHECK(mask->materialize());
        CHECK(u_t->materialize());
        const M* mask_val = mask->dense_.d_val_;
        const int grid = gridFor(A_nrows, GB_PULL_NT, 8);
#define GB_LAUNCH_PULL(SC, EE, OR)                                           \
        spmvMaskedOrPullKernel<SC, EE, OR><<<grid, GB_PULL_NT, 0, s>>>(      \
            w->d_val_, mask_val, op.identity(), A_nrows, A_csrRowPtr,        \
            A_csrColInd, u_t->d_val_, ctr, prof_cell)
        profiler().begin(GB_PROF_PULL_BOOL, s);
        switch (variant) {
          case 0: GB_LAUNCH_PULL(false, false, false); break;
          case 1: GB_LAUNCH_PULL(false, false, true ); break;
          case 2: GB_LAUNCH_PULL(false, true,  false); break;
          case 3: GB_LAUNCH_PULL(false, true,  true ); break;
          case 4: GB_LAUNCH_PULL(true,  false, false); break;
          case 5: GB_LAUNCH_PULL(true,  false, true ); break;
          case 6: GB_LAUNCH_PULL(true,  true,  false); break;
          case 7: GB_LAUNCH_PULL(true,  true,  true ); break;
          default: break;
        }
#undef GB_LAUNCH_PULL
        fixed_bytes = 4.0*(A_nrows + 1) + 8.0*A_nrows;
      }
      GB_KERNEL_CHECK();
      // the inspected colind bytes are added on the device
      profiler().end(GB_PROF_PULL_BOOL, s, fixed_bytes);
      w->touched();
      w->bits_valid_ = bits_form;
      w->vals_stale_ = bits_form;
      // The kernel wrote 0/1 and counted the ones: the next convert() or
      // a PlusMonoid reduce can reuse the count (one 8-byte read, no pass).
      w->count_pending_ = true;
      w->count_ticket_  = mail_ticket;     // 0: not posted to the mailbox
      w->zero_one_      = true;
      w->nnz_identity_  = static_cast<W>(0);
      if (desc->debug())
        { w->materialize(); printDevice("w_val", w->d_val_, A_nrows); }
    } else if (mask_vec_type == GrB_SPARSE) {
      std::cout << "DeVec Sparse Mask logical_or Spmv\n";
      std::cout << "Error: Feature not implemented yet!\n";
    } else {
      return GrB_UNINITIALIZED_OBJECT;
    }
  } else {
    CHECK(u_t->materialize());
    if (use_mask) CHECK(mask->materialize());
    if (use_accum) CHECK(w->materialize());
    W* w_val;
    if (use_accum)
      w_val = reinterpret_cast<W*>(desc->scratch(GB_SCRATCH_VEC_A,
          static_cast<size_t>(A_nrows)*sizeof(W)));
    else
      w_val = w->d_val_;

    // Tile partition of this structure, computed once per matrix.
    SparseMatrix<a>* A_t = const_cast<SparseMatrix<a>*>(A);
    const int which = use_tran ? 1 : 0;
    const long long merge_total = static_cast<long long>(A_nrows) + A->nvals_;
    const int ntiles = static_cast<int>((merge_total + GB_SPMV_TILE - 1)/
        GB_SPMV_TILE);
    if (A_t->d_spmv_tiles_[which] == NULL ||
        A_t->spmv_tiles_key_[which] != A_csrRowPtr ||
        A_t->spmv_tiles_nvals_[which] != A->nvals_ ||
        A_t->spmv_tiles_count_[which] != ntiles) {
      if (A_t->d_spmv_tiles_[which] != NULL) gbFree(A_t->d_spmv_tiles_[which]);
      A_t->d_spmv_tiles_[which] = reinterpret_cast<Index*>(
          gbMalloc((static_cast<size_t>(ntiles) + 1)*sizeof(Index)));
      spmvMergePartitionKernel<<<(ntiles + 256)/256, 256, 0, s>>>(
          A_t->d_spmv_tiles_[which], A_csrRowPtr, A_nrows, A->nvals_, ntiles,
          GB_SPMV_TILE);
      GB_KERNEL_CHECK();
      A_t->spmv_tiles_key_[which]   = A_csrRowPtr;
      A_t->spmv_tiles_nvals_[which] = A->nvals_;
      A_t->spmv_tiles_count_[which] = ntiles;
    }
    // Large matrices whose entries mostly reference a few columns (power-law
    // graphs) take the hub-cached kernel (kernels/spmv_hub.cuh): hub columns are
    // served from shared memory, the rest as before.  The per-matrix index is
    // built on first use; matrices where the hubs cover too little keep the
    // merge kernel.  GB200_SPMV_HUB=0 forces the merge kernel.
    bool done = false;
    if (sizeof(W) == 4 && sizeof(a) == 4 && sizeof(U) == 4 && sizeof(Index) == 4) {
      static const int hub_mode = getEnv("GB200_SPMV_HUB", 1);
      static const int hub_min_nnz = getEnv("GB200_SPMV_HUB_MIN_NNZ", 1 << 22);
      static const int hub_min_pct = getEnv("GB200_SPMV_HUB_MIN_PCT", 30);
      const bool aligned32 =
          (reinterpret_cast<uintptr_t>(A_csrColInd) % 32 == 0) &&
          (reinterpret_cast<uintptr_t>(A_csrVal) % 32 == 0);
      if (hub_mode != 0 && A->nvals_ >= hub_min_nnz && aligned32) {
        const Index ncols_t = use_tran ? A->nrows_ : A->ncols_;
        HubIndex& h = A_t->hub_[which];
        if (A_t->hub_state_[which] == 0 || h.key != A_csrColInd ||
            h.key_nvals != A->nvals_) {
          buildHubIndex(&h, A_csrRowPtr, A_csrColInd, A_nrows, ncols_t, A->nvals_,
              GB_HUB_CAPACITY);
          A_t->hub_state_[which] = (100.0*h.coverage >= hub_min_pct) ? 1 : 2;
          if (A_t->hub_state_[which] == 2) {   // keep only the verdict
            const Index* key = h.key; const Index key_nvals = h.key_nvals;
            h.release();
            h.key = key; h.key_nvals = key_nvals;
          }
        }
        if (A_t->hub_state_[which] == 1) {
          CHECK(spmvHubLaunch(w_val, h, op, A_csrVal, u_t->d_val_, A_nrows,
              A->nvals_, desc));
          done = true;
        }
      }
    }
    if (!done)
    CHECK(spmvMergeLaunch(w_val, A_t->d_spmv_tiles_[which], op, A_csrRowPtr, A_csrColInd,
        A_csrVal, u_t->d_val_, A_nrows, A->nvals_, desc));

    if (use_mask) {
      Storage mask_vec_type;
      CHECK(mask->getStorage(&mask_vec_type));
      if (mask_vec_type != GrB_DENSE) {
        std::cout << "Spmv generic semiring with sparse mask\n";
        std::cout << "Error: Feature not implemented yet!\n";
        return GrB_NOT_IMPLEMENTED;
      }
      const int grid = gridFor(A_nrows, 256);
      // GrB_SCMP keeps entries whose mask is zero: overwrite where mask != 0.
      if (use_scmp)
        assignDenseDenseMaskKernel<false><<<grid, 256, 0, s>>>(w_val, A_nrows,
            mask->dense_.d_val_, static_cast<W>(op.identity()));
      else
        assignDenseDenseMaskKernel<true><<<grid, 256, 0, s>>>(w_val, A_nrows,
            mask->dense_.d_val_, static_cast<W>(op.identity()));
      GB_KERNEL_CHECK();
    }
    if (use_accum) {
      ewiseBinaryDenseKernel<<<gridFor(A_nrows, 256), 256, 0, s>>>(w->d_val_,
          extractAdd(op), w->d_val_, w_val, A_nrows);
      GB_KERNEL_CHECK();
    }
    w->touched();
    if (desc->debug())
      printDevice("w_val", w->d_val_, A_nrows);
  }
  return GrB_SUCCESS;
}
}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_SPMV_HPP_
