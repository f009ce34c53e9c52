// graphblast_b200 backend — push-direction mxv host: sparse w = A'(:, f) (+.x) f
// for a sparse frontier f, A' rows = CSC columns of A by default and CSR rows
// when the descriptor says transposed (vxm toggles GrB_INP1, so vxm pushes along
// the CSR rows of A).
//
// Replaces reference graphblas/backend/cuda/spmspv.hpp:15-257 and
// spmspv_inner.hpp:62-320.  Launch sequence (5 launches + one cub scan, ONE
// 8-byte device-to-host read):
//   frontierDegreeKernel -> cub::DeviceScan::ExclusiveSum -> spmspvPushKernel
//   -> compactCount / compactScan / compactEmit (sorted, duplicate-free output).
// Scratch is O(|f| + n): a dense accumulator and a touched-bitmap that are kept
// "all identity / all zero" between calls by the compaction itself — not the
// (2n + 4*nnz*memusage) ints of the reference (spmspv.hpp:60-66), which is sized
// in `int` and overflows at RMAT-24.
//
// Quirks kept (SURVEY.md §8a):
//  * the mask is interpreted with the reference's inverted flag
//    (use_scmp = scmp_mode != GrB_SCMP, spmspv.hpp:33-37): result keeps entries
//    with mask == 0 under GrB_SCMP and entries with mask != 0 otherwise;
//  * masked key-value mode drops entries whose value is 0 (spmspv.hpp:203-243);
//  * struct-only mode carries no meaningful values (we store 1).
#ifndef GRAPHBLAS_BACKEND_CUDA_SPMSPV_HPP_
#define GRAPHBLAS_BACKEND_CUDA_SPMSPV_HPP_

#include <iostream>
#include <algorithm>
#include <string>

#include "graphblas/backend/cuda/kernels/kernels.hpp"
#include "graphblas/backend/cuda/compact.hpp"

namespace graphblas {
namespace backend {

// Makes the push arenas valid for (n outputs, identity): accumulator all
// identity, bitmap all zero.  A refill happens only when the identity's bit
// pattern or the size changes; steady-state calls skip it.
template <typename W>
Info preparePushArenas(Descriptor* desc, Index n, W identity, bool need_acc,
    unsigned int** bits_out, W** acc_out) {
  cudaStream_t s = gbStream();
  const size_t nwords = (static_cast<size_t>(n) + 31)/32;
  unsigned int* bits = reinterpret_cast<unsigned int*>(
      desc->scratch(GB_SCRATCH_BITS, nwords*sizeof(unsigned int)));
  if (!desc->bits_valid_ || desc->bits_words_ < nwords) {
    CUDA_CALL(cudaMemsetAsync(bits, 0, desc->slot_size_[GB_SCRATCH_BITS], s));
    desc->bits_valid_ = true;
    desc->bits_words_ = desc->slot_size_[GB_SCRATCH_BITS]/sizeof(unsigned int);
  }
  *bits_out = bits;
  *acc_out  = NULL;
  if (need_acc) {
    W* acc = reinterpret_cast<W*>(desc->scratch(GB_SCRATCH_ACC,
        static_cast<size_t>(n)*sizeof(W)));
    unsigned int id_bits = 0;
    memcpy(&id_bits, &identity, sizeof(W) < 4 ? sizeof(W) : 4);
    if (!desc->acc_valid_ || desc->acc_elems_ < static_cast<size_t>(n) ||
        desc->acc_identity_bits_ != id_bits ||
        desc->acc_elem_bytes_ != sizeof(W)) {
      const size_t cap = desc->slot_size_[GB_SCRATCH_ACC]/sizeof(W);
      fillKernel<<<gridFor(cap, 256), 256, 0, s>>>(acc, identity,
          static_cast<Index>(std::min<size_t>(cap, INT_MAX)));
      GB_KERNEL_CHECK();
      desc->acc_valid_         = true;
      desc->acc_elems_         = cap;
      desc->acc_identity_bits_ = id_bits;
      desc->acc_elem_bytes_    = sizeof(W);
    }
    *acc_out = acc;
  }
  return GrB_SUCCESS;
}

template <typename W, typename a, typename U, typename M,
          typename BinaryOpT, typename SemiringT>
Info spmspvMerge(SparseVector<W>* w, const Vector<M>* mask, BinaryOpT accum,
    SemiringT op, const SparseMatrix<a>* A, const SparseVector<U>* u, Descriptor* desc,
    bool* prefer_pull = NULL) {
  // prefer_pull != NULL: the caller can still take the pull direction.  If the
  // frontier's edges are more than 33 percent of all stored entries the
  // push is abandoned before it starts (*prefer_pull = true, w untouched): the
  // reference switches on the frontier's VERTEX share only (vector.hpp:318-342),
  // and a few hub vertices below that threshold can own most of the graph — at
  // RMAT-24 one such SSSP push expanded 2.9 GB of edges in 4.2 ms where the pull
  // over everything takes 2.1 ms.
  if (prefer_pull != NULL) *prefer_pull = false;
  // Get descriptor parameters for SCMP, REPL, TRAN
  Desc_value scmp_mode, repl_mode, inp0_mode, inp1_mode;
  CHECK(desc->get(GrB_MASK, &scmp_mode));
  CHECK(desc->get(GrB_OUTP, &repl_mode));
  CHECK(desc->get(GrB_INP0, &inp0_mode));
  CHECK(desc->get(GrB_INP1, &inp1_mode));

  const bool use_mask  = (mask != NULL);
  const bool use_accum = !AccumIsNull<BinaryOpT>::value;
  const bool keep_zero = (scmp_mode == GrB_SCMP);   // keep where mask == 0
  const bool use_repl  = (repl_mode == GrB_REPLACE);
  const bool use_tran  = (inp0_mode == GrB_TRAN || inp1_mode == GrB_TRAN);
  const bool struconly = desc->struconly();

  if (desc->debug()) {
    std::cout << "Executing Spmspv MERGE\n";
    std::cout << (struconly ? "In structure only mode\n"
                            : "In key-value mode\n");
    printState(use_mask, use_accum, !keep_zero, use_repl, use_tran);
  }

  // Transpose (default is CSC):
  const Index* A_csrRowPtr = (!use_tran) ? A->d_cscColPtr_ : A->d_csrRowPtr_;
  const Index* A_csrColInd = (!use_tran) ? A->d_cscRowInd_ : A->d_csrColInd_;
  const a*     A_csrVal    = (!use_tran) ? A->d_cscVal_    : A->d_csrVal_;
  // Output length = the other dimension of the traversed structure.
  const Index  out_size    = (!use_tran) ? A->nrows_       : A->ncols_;
  if (A_csrRowPtr == NULL) return GrB_UNINITIALIZED_OBJECT;

  const Index nf = u->nvals_;
  CHECK(w->allocateGpu());
  if (nf == 0) {
    w->nvals_       = 0;
    w->need_update_ = true;
    return GrB_SUCCESS;
  }

  const M* mask_val = NULL;
  const unsigned int* mask_bits = NULL;
  if (use_mask) {
    Storage mask_vec_type;
    CHECK(mask->getStorage(&mask_vec_type));
    if (mask_vec_type == GrB_DENSE) {
      mask_val = mask->dense_.d_val_;
      if (mask->dense_.bits_valid_) mask_bits = mask->dense_.d_bits_;
    } else if (mask_vec_type == GrB_SPARSE) {
      std::cout << "Spmspv Sparse Mask\n";
      std::cout << "Error: Feature not implemented yet!\n";
      return GrB_NOT_IMPLEMENTED;
    } else {
      return GrB_UNINITIALIZED_OBJECT;
    }
  }

  cudaStream_t s = gbStream();

  // 1) degrees of the frontier rows, scanned (offs[nf] = E_f).
  Index* offs = reinterpret_cast<Index*>(desc->scratch(GB_SCRATCH_OFFS,
      2*(static_cast<size_t>(nf) + 1)*sizeof(Index)));
  Index* deg  = offs + (nf + 1);
  if (nf + 1 <= GB_DEGSCAN_MAX) {
    frontierDegreeScanKernel<<<1, GB_DEGSCAN_NT, 0, s>>>(offs, A_csrRowPtr,
        u->d_ind_, nf);
    GB_KERNEL_CHECK();
  } else {
    frontierDegreeKernel<<<gridFor(nf + 1, 256), 256, 0, s>>>(deg, A_csrRowPtr,
        u->d_ind_, nf);
    GB_KERNEL_CHECK();
    size_t cub_bytes = 0;
    CUDA_CALL(cub::DeviceScan::ExclusiveSum(NULL, cub_bytes, deg, offs, nf + 1, s));
    void* cub_tmp = desc->scratch(GB_SCRATCH_CUB, cub_bytes);
    CUDA_CALL(cub::DeviceScan::ExclusiveSum(cub_tmp, cub_bytes, deg, offs, nf + 1, s));
  }

  // 1b) edge-based direction check (only for frontiers big enough to matter, so
  //     the small levels of a BFS pay nothing for it)
  const float edge_switch = 0.01f*33.f;     // share of the stored entries
  if (prefer_pull != NULL && nf >= 4096) {
    const unsigned long long ticket = runtime().mailTicket();
    postIndexKernel<<<1, 1, 0, s>>>(offs + nf, runtime().mailSlot(4), ticket);
    GB_KERNEL_CHECK();
    long long ef = -1;
    volatile unsigned long long* slot = runtime().h_mail + 4;
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned long long spin = 0;; ++spin) {
      const unsigned long long v = *slot;
      if ((v >> 40) == ticket) { ef = static_cast<long long>(v & 0xffffffffull); break; }
      if ((spin & 0x3ff) == 0x3ff &&
          std::chrono::steady_clock::now() - t0 > std::chrono::seconds(2))
        break;
    }
    if (ef < 0) ef = runtime().fetch(offs + nf);
    if (static_cast<double>(ef) > static_cast<double>(edge_switch)*A->nvals_) {
      if (desc->dirinfo())
        std::cout << "Frontier owns " << ef << " of " << A->nvals_
                  << " entries: pull instead of push\n";
      *prefer_pull = true;
      return GrB_SUCCESS;
    }
  }

  // 2) expand + combine into the accumulator / bitmap.
  unsigned int* bits;
  W*            acc;
  CHECK(preparePushArenas<W>(desc, out_size, op.identity(), !struconly, &bits, &acc));

  const int grid = runtime().sm_count*8;
  const int mask_mode = use_mask ? (keep_zero ? 2 : 1) : 0;
#define GB_LAUNCH_PUSH(SO, MM)                                               \
  spmspvPushKernel<SO, MM><<<grid, GB_PUSH_NT, 0, s>>>(bits, acc, mask_val,  \
      mask_bits, offs, u->d_ind_, u->d_val_, nf, A_csrRowPtr, A_csrColInd, A_csrVal,    \
      static_cast<W>(op.identity()), extractMul(op), extractAdd(op),      \
      add_kind, prof_cell)
  const int add_kind = static_cast<int>(extractAdd(op)(3, 5));
  unsigned long long* prof_cell = NULL;
  if (profiler().enabled) {
    profiler().ensureCells();
    prof_cell = profiler().d_cells + GB_PROF_PUSH;
  }
  profiler().begin(GB_PROF_PUSH, s);
  if (struconly) {
    if (mask_mode == 0)      GB_LAUNCH_PUSH(true, 0);
    else if (mask_mode == 1) GB_LAUNCH_PUSH(true, 1);
    else                     GB_LAUNCH_PUSH(true, 2);
  } else {
    if (mask_mode == 0)      GB_LAUNCH_PUSH(false, 0);
    else if (mask_mode == 1) GB_LAUNCH_PUSH(false, 1);
    else                     GB_LAUNCH_PUSH(false, 2);
  }
#undef GB_LAUNCH_PUSH
  GB_KERNEL_CHECK();
  profiler().end(GB_PROF_PUSH, s, 12.0*nf);   // ind + rowptr pair per frontier entry

  // 3) ordered compaction of the touched bitmap -> sorted unique output.
  const Index nwords = (out_size + 31)/32;
  Index count;
  if (struconly) {
    BitmapCompactSource<W, false, false> src;
    src.bits = bits; src.acc = acc; src.identity = op.identity();
    src.one = static_cast<W>(1);
    src.out_ind = w->d_ind_; src.out_val = w->d_val_;
    count = compactOrdered(src, nwords, desc);
  } else if (use_mask) {
    BitmapCompactSource<W, true, true> src;
    src.bits = bits; src.acc = acc; src.identity = op.identity();
    src.one = static_cast<W>(1);
    src.out_ind = w->d_ind_; src.out_val = w->d_val_;
    count = compactOrdered(src, nwords, desc);
  } else {
    BitmapCompactSource<W, true, false> src;
    src.bits = bits; src.acc = acc; src.identity = op.identity();
    src.one = static_cast<W>(1);
    src.out_ind = w->d_ind_; src.out_val = w->d_val_;
    count = compactOrdered(src, nwords, desc);
  }
  w->nvals_       = count;
  w->need_update_ = true;
  if (profiler().enabled)
    profiler().host_bytes[GB_PROF_PUSH] += 8.0*count;   // (ind, val) written

  if (desc->debug()) {
    std::cout << "Frontier size: " << w->nvals_ << std::endl;
    printDevice("w_ind", w->d_ind_, w->nvals_);
    if (!struconly) printDevice("w_val", w->d_val_, w->nvals_);
  }
  return GrB_SUCCESS;
}
}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_SPMSPV_HPP_
