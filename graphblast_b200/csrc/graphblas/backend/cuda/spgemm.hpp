// graphblast_b200 backend — masked SpGEMM host (triangle counting path).
//
// Replaces reference graphblas/backend/cuda/spgemm.hpp:22-110 (spgemmMasked).
// C takes the mask's pattern (C->dup(mask)) and one value per mask entry is
// computed as the dot product A(i,:) . B(:,j).  The reference's unmasked
// cusparse_spgemm/cusparse_spgemm2 (:114-512) call cuSPARSE csrgemm2 entry
// points that no longer exist in CUDA 12 and are out of scope (SURVEY.md §2 #13).
#ifndef GRAPHBLAS_BACKEND_CUDA_SPGEMM_HPP_
#define GRAPHBLAS_BACKEND_CUDA_SPGEMM_HPP_

#include <iostream>

#include "graphblas/backend/cuda/kernels/kernels.hpp"

namespace graphblas {
namespace backend {

// One pass of the hash formulation: three launches, one per table size.  The
// largest tables go first (few items, long tails).
template <bool SWAP, typename c, typename TV, typename PV, typename m,
          typename MulOp, typename AddOp>
Info spgemmHashPass(c* C_val, const HashItem* lists, size_t stride,
    const unsigned int* counts, unsigned int* grabs,
    const Index* T_ptr, const Index* T_ind, const TV* T_val,
    const Index* P_ptr, const Index* P_ind, const PV* P_val,
    const Index* M_ptr, const Index* M_ind, const m* M_val,
    const Index* mask_rowptr, const Index* mask_colind,
    MulOp mul_op, AddOp add_op, c identity, unsigned long long* list_bytes,
    cudaStream_t s) {
  const int sms = runtime().sm_count;
  {
    typedef HashGroupSmem<GB_HASH_SLOTS_L, GB_HASH_CHUNK_L, TV> Smem;
    auto kernel = spgemmHashKernel<1024, false, GB_HASH_SLOTS_L, GB_HASH_SEG_L,
        GB_HASH_CHUNK_L, GB_HASH_UNROLL_L, SWAP, c, TV, PV, m, MulOp, AddOp>;
    static bool configured = false;          // per instantiation
    if (!configured) {
      CUDA_CALL(cudaFuncSetAttribute(kernel,
          cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(Smem))));
      configured = true;
    }
    kernel<<<sms*GB_HASH_CTAS_L, 1024, sizeof(Smem), s>>>(C_val, lists + 2*stride, counts + 2,
        grabs + 2, T_ptr, T_ind, T_val, P_ptr, P_ind, P_val, M_ptr, M_ind, M_val,
        mask_rowptr, mask_colind, mul_op, add_op, identity, list_bytes);
    GB_KERNEL_CHECK();
  }
  {
    typedef HashGroupSmem<GB_HASH_SLOTS_M, GB_HASH_CHUNK_M, TV> Smem;
    auto kernel = spgemmHashKernel<256, false, GB_HASH_SLOTS_M, GB_HASH_CAP_M,
        GB_HASH_CHUNK_M, GB_HASH_UNROLL_M, SWAP, c, TV, PV, m, MulOp, AddOp>;
    static bool configured = false;
    if (!configured) {
      CUDA_CALL(cudaFuncSetAttribute(kernel,
          cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(Smem))));
      configured = true;
    }
    kernel<<<sms*GB_HASH_CTAS_M, 256, sizeof(Smem), s>>>(C_val, lists + stride, counts + 1,
        grabs + 1, T_ptr, T_ind, T_val, P_ptr, P_ind, P_val, M_ptr, M_ind, M_val,
        mask_rowptr, mask_colind, mul_op, add_op, identity, list_bytes);
    GB_KERNEL_CHECK();
  }
  {
    typedef HashGroupSmem<GB_HASH_SLOTS_S, GB_HASH_CHUNK_S, TV> Smem;
    auto kernel = spgemmHashKernel<256, true, GB_HASH_SLOTS_S, GB_HASH_CAP_S,
        GB_HASH_CHUNK_S, 2, SWAP, c, TV, PV, m, MulOp, AddOp>;
    static bool configured = false;
    if (!configured) {
      CUDA_CALL(cudaFuncSetAttribute(kernel,
          cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(8*sizeof(Smem))));
      configured = true;
    }
    kernel<<<sms*4, 256, 8*sizeof(Smem), s>>>(C_val, lists, counts, grabs,
        T_ptr, T_ind, T_val, P_ptr, P_ind, P_val, M_ptr, M_ind, M_val,
        mask_rowptr, mask_colind, mul_op, add_op, identity, list_bytes);
    GB_KERNEL_CHECK();
  }
  return GrB_SUCCESS;
}

template <typename c, typename a, typename b, typename m,
          typename BinaryOpT,     typename SemiringT>
Info spgemmMasked(SparseMatrix<c>* C, const Matrix<m>* mask, BinaryOpT accum,
    SemiringT op, const SparseMatrix<a>* A, const SparseMatrix<b>* B,
    Descriptor* desc) {
  Desc_value scmp_mode, inp0_mode, inp1_mode;
  CHECK(desc->get(GrB_MASK, &scmp_mode));
  CHECK(desc->get(GrB_INP0, &inp0_mode));
  CHECK(desc->get(GrB_INP1, &inp1_mode));

  const bool use_mask   = (mask != NULL);
  const bool use_tran_A = inp0_mode == GrB_TRAN;
  const bool use_tran_B = inp1_mode == GrB_TRAN;

  const Index* A_csrRowPtr = (use_tran_A) ? A->d_cscColPtr_ : A->d_csrRowPtr_;
  const Index* A_csrColInd = (use_tran_A) ? A->d_cscRowInd_ : A->d_csrColInd_;
  const a*     A_csrVal    = (use_tran_A) ? A->d_cscVal_    : A->d_csrVal_;
  const Index  A_nrows     = (use_tran_A) ? A->ncols_       : A->nrows_;

  const Index* B_cscColPtr = (use_tran_B) ? B->d_csrRowPtr_ : B->d_cscColPtr_;
  const Index* B_cscRowInd = (use_tran_B) ? B->d_csrColInd_ : B->d_cscRowInd_;
  const b*     B_cscVal    = (use_tran_B) ? B->d_csrVal_    : B->d_cscVal_;

  if (A_csrRowPtr == NULL || B_cscColPtr == NULL)
    return GrB_UNINITIALIZED_OBJECT;

  if (use_mask) {
    Storage mask_mat_type;
    CHECK(mask->getStorage(&mask_mat_type));
    if (mask_mat_type == GrB_DENSE) {
      std::cout << "SpGEMM with dense mask\n";
      std::cout << "Error: Feature not implemented yet!\n";
    } else {
      if (reinterpret_cast<const void*>(C) != reinterpret_cast<const void*>(A) &&
          reinterpret_cast<const void*>(C) != reinterpret_cast<const void*>(B))
        CHECK(C->dup(&mask->sparse_));

      const SparseMatrix<m>* sparse_mask = &mask->sparse_;
      unsigned long long* work = desc->counters() + 3;
      cudaStream_t s = gbStream();
      CUDA_CALL(cudaMemsetAsync(work, 0, sizeof(unsigned long long), s));
      const int grid = runtime().sm_count*8;
      unsigned long long* prof_cell = NULL;
      if (profiler().enabled) {
        profiler().ensureCells();
        prof_cell = profiler().d_cells + GB_PROF_SPGEMM;
      }
      profiler().begin(GB_PROF_SPGEMM, s);
      // Hash formulation (kernels/spgemm_hash.cuh) when the mask can also be walked
      // by columns; otherwise the search kernels.  A symmetric matrix borrows its
      // CSR arrays for the column side, which is right only for the whole
      // pattern — tril drops the flag.
      static const bool hash_on = getEnv("GB200_SPGEMM_HASH", 1) != 0;
      const bool mask_by_cols = sparse_mask->format_ == GrB_SPARSE_MATRIX_CSRCSC &&
          sparse_mask->d_cscColPtr_ != NULL && sparse_mask->d_cscRowInd_ != NULL &&
          sparse_mask->d_cscVal_ != NULL;
      const Index B_ncols = use_tran_B ? B->nrows_ : B->ncols_;
      const bool hashed = hash_on && mask_by_cols &&
          sparse_mask->nrows_ == A_nrows && sparse_mask->ncols_ == B_ncols;
      if (hashed) {
        // work items per class: at most one partial chunk per owner plus the full ones
        const size_t stride = static_cast<size_t>(A_nrows > B_ncols ? A_nrows : B_ncols) +
            static_cast<size_t>(sparse_mask->nvals_)/GB_HASH_CHUNK_S + 1;
        const size_t list_ints = 2*2*GB_HASH_NCLASS*stride;
        Index* arena = reinterpret_cast<Index*>(desc->scratch(GB_SCRATCH_VEC_A,
            (list_ints + 32)*sizeof(Index)));
        HashItem* lists = reinterpret_cast<HashItem*>(arena);
        unsigned int* cells = reinterpret_cast<unsigned int*>(arena + list_ints);
        // cells: [0..2] item counts of pass 1, [4..6] of pass 2, [8..10] and
        // [12..14] the grab counters
        CUDA_CALL(cudaMemsetAsync(cells, 0, 32*sizeof(unsigned int), s));
        spgemmHashClassifyKernel<<<gridFor(A_nrows, 256), 256, 0, s>>>(A_csrRowPtr,
            sparse_mask->d_csrRowPtr_, A_nrows, false, lists, stride, cells);
        GB_KERNEL_CHECK();
        spgemmHashClassifyKernel<<<gridFor(B_ncols, 256), 256, 0, s>>>(B_cscColPtr,
            sparse_mask->d_cscColPtr_, B_ncols, true,
            lists + GB_HASH_NCLASS*stride, stride, cells + 4);
        GB_KERNEL_CHECK();
        CHECK((spgemmHashPass<false>(C->d_csrVal_, lists, stride, cells, cells + 8,
            A_csrRowPtr, A_csrColInd, A_csrVal, B_cscColPtr, B_cscRowInd, B_cscVal,
            sparse_mask->d_csrRowPtr_, sparse_mask->d_csrColInd_,
            sparse_mask->d_csrVal_, sparse_mask->d_csrRowPtr_,
            sparse_mask->d_csrColInd_, extractMul(op), extractAdd(op),
            static_cast<c>(op.identity()), prof_cell, s)));
        CHECK((spgemmHashPass<true>(C->d_csrVal_, lists + GB_HASH_NCLASS*stride,
            stride, cells + 4, cells + 12,
            B_cscColPtr, B_cscRowInd, B_cscVal, A_csrRowPtr, A_csrColInd, A_csrVal,
            sparse_mask->d_cscColPtr_, sparse_mask->d_cscRowInd_,
            sparse_mask->d_cscVal_, sparse_mask->d_csrRowPtr_,
            sparse_mask->d_csrColInd_, extractMul(op), extractAdd(op),
            static_cast<c>(op.identity()), prof_cell, s)));
      } else {
        // thread per mask entry; entries whose lists are both long are deferred
        // to a warp-per-entry kernel through a device-side list (`work` counts it)
        Index* heavy = reinterpret_cast<Index*>(desc->scratch(GB_SCRATCH_VEC_A,
            2*static_cast<size_t>(sparse_mask->nvals_ + 1)*sizeof(Index)));
        spgemmMaskedEdgeKernel<<<grid, GB_SPGEMM_NT, 0, s>>>(C->d_csrVal_,
            sparse_mask->d_csrRowPtr_, sparse_mask->d_csrColInd_,
            sparse_mask->d_csrVal_, extractMul(op), extractAdd(op),
            static_cast<c>(op.identity()), A_csrRowPtr, A_csrColInd, A_csrVal,
            B_cscColPtr, B_cscRowInd, B_cscVal, A_nrows, sparse_mask->nvals_,
            heavy, work, prof_cell);
        GB_KERNEL_CHECK();
        spgemmMaskedHeavyKernel<<<grid, GB_SPGEMM_NT, 0, s>>>(C->d_csrVal_,
            sparse_mask->d_csrColInd_, extractMul(op), extractAdd(op),
            static_cast<c>(op.identity()), A_csrRowPtr, A_csrColInd, A_csrVal,
            B_cscColPtr, B_cscRowInd, B_cscVal, heavy, work);
      }
      GB_KERNEL_CHECK();
      profiler().end(GB_PROF_SPGEMM, s, 8.0*(A_nrows + 1) +
          8.0*sparse_mask->nvals_);
    }
  }
  C->need_update_ = true;
  C->csr_initialized_ = true;
  C->csc_initialized_ = false;
  return GrB_SUCCESS;
}
}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_SPGEMM_HPP_
