// graphblast_b200 backend — masked SpGEMM (dot-product formulation) used by
// triangle counting: C(i,j) = add_k mul(A(i,k), B(k,j)) only for (i,j) in mask.
//
// These are the search kernels of spgemmMasked (spgemm.hpp), which run when the
// mask has no CSC to walk it by columns; otherwise the hash formulation
// (kernels/spgemm_hash.cuh) runs.
//
// Reference: the reference's spgemmMaskedKernel, kernels/spgemm.hpp:17-79 — one
// warp per mask row, every lane binary-searches A(i,:)'s columns in B(:,j) for each
// mask entry.  Here: one thread per mask entry walks the SHORTER of the two sorted
// lists and searches the longer one; entries whose lists are both long are
// deferred to a warp each (spgemmMaskedHeavyKernel).
#ifndef GRAPHBLAS_BACKEND_CUDA_KERNELS_SPGEMM_MASKED_CUH_
#define GRAPHBLAS_BACKEND_CUDA_KERNELS_SPGEMM_MASKED_CUH_

#include "graphblas/backend/cuda/kernels/common.cuh"

namespace graphblas {
namespace backend {

#define GB_SPGEMM_NT 256
#define GB_SPGEMM_HEAVY 32        // shorter list longer than this: warp per entry

// Edge-parallel form: one THREAD per mask entry (grid-stride).  In the triangle
// count both operands are rows of L = tril(A): a high-id vertex next to many hubs
// has a long row, and with one warp per mask row its tens of thousands of mask
// entries were processed one after the other by a single warp (RMAT-18: 105 ms,
// almost all of it in a handful of warps).  Here every mask entry is its own work
// item: the thread finds its row with a binary search over mask_rowptr (the top
// of the search tree is shared by neighbouring lanes and stays in L1), walks the
// SHORTER of the two sorted lists and looks each key up in the longer one, resuming
// every search where the previous one ended (keys ascend, so positions do too).
// Neighbouring lanes are mask entries of the same row, so the A-side list is a
// broadcast load.
template <typename c, typename a, typename b, typename m,
          typename MulOp, typename AddOp>
__global__ void __launch_bounds__(GB_SPGEMM_NT)
spgemmMaskedEdgeKernel(c* __restrict__           C_val,
                       const Index* __restrict__ mask_rowptr,
                       const Index* __restrict__ mask_colind,
                       const m* __restrict__     mask_val,
                       MulOp                     mul_op,
                       AddOp                     add_op,
                       c                         identity,
                       const Index* __restrict__ A_rowptr,
                       const Index* __restrict__ A_colind,
                       const a* __restrict__     A_val,
                       const Index* __restrict__ B_colptr,
                       const Index* __restrict__ B_rowind,
                       const b* __restrict__     B_val,
                       Index                     nrows,
                       Index                     nedges,
                       Index* __restrict__       heavy_list,   // (entry, row) pairs
                       unsigned long long*       heavy_count,
                       unsigned long long*       list_bytes) {
  long long scanned = 0;
  Index e = blockIdx.x*blockDim.x + threadIdx.x;
  const Index stride = gridDim.x*blockDim.x;
  for (; e < nedges; e += stride) {
    c accumulator = identity;
    if (mask_val[e]) {
      // row of mask entry e: the first r with mask_rowptr[r+1] > e
      Index lo = 0, hi = nrows;
      while (lo < hi) {
        const Index mid = lo + ((hi - lo) >> 1);
        if (__ldg(mask_rowptr + mid + 1) <= e) lo = mid + 1; else hi = mid;
      }
      const Index row   = lo;
      const Index j     = __ldg(mask_colind + e);
      const Index a_beg = __ldg(A_rowptr + row);
      const Index a_end = __ldg(A_rowptr + row + 1);
      const Index b_beg = __ldg(B_colptr + j);
      const Index b_end = __ldg(B_colptr + j + 1);
      scanned += (a_end - a_beg) + (b_end - b_beg);
      const Index shorter = (a_end - a_beg <= b_end - b_beg) ? (a_end - a_beg)
                                                             : (b_end - b_beg);
      if (shorter > GB_SPGEMM_HEAVY) {
        // long x long: a whole warp takes it in the second kernel
        const unsigned long long slot = atomicAdd(heavy_count, 1ull);
        heavy_list[2*slot]     = e;
        heavy_list[2*slot + 1] = row;
        continue;
      }
      if (a_end - a_beg <= b_end - b_beg) {
        Index q = b_beg;
        for (Index p = a_beg; p < a_end && q < b_end; ++p) {
          const Index key = __ldg(A_colind + p);
          q = findSorted(B_rowind, q, b_end, key);
          if (q < b_end && __ldg(B_rowind + q) == key)
            accumulator = add_op(mul_op(A_val[p], B_val[q]), accumulator);
        }
      } else {
        Index p = a_beg;
        for (Index q = b_beg; q < b_end && p < a_end; ++q) {
          const Index key = __ldg(B_rowind + q);
          p = findSorted(A_colind, p, a_end, key);
          if (p < a_end && __ldg(A_colind + p) == key)
            accumulator = add_op(mul_op(A_val[p], B_val[q]), accumulator);
        }
      }
    }
    C_val[e] = accumulator;
  }
  // algorithmic bytes: both index lists of every mask entry, 4 bytes per index
  unsigned long long total = static_cast<unsigned long long>(scanned);
  for (int d = 16; d > 0; d >>= 1)
    total += __shfl_down_sync(GB_FULL_MASK, total, d);
  if ((threadIdx.x & 31) == 0 && total && list_bytes != NULL)
    atomicAdd(list_bytes, 4ull*total);
}

// Second kernel of the edge-parallel form: one WARP per deferred mask entry (both
// lists longer than GB_SPGEMM_HEAVY).  Lanes take every 32nd key of the shorter
// list and search the longer one, each lane resuming where its last search ended.
template <typename c, typename a, typename b,
          typename MulOp, typename AddOp>
__global__ void __launch_bounds__(GB_SPGEMM_NT)
spgemmMaskedHeavyKernel(c* __restrict__           C_val,
                        const Index* __restrict__ mask_colind,
                        MulOp                     mul_op,
                        AddOp                     add_op,
                        c                         identity,
                        const Index* __restrict__ A_rowptr,
                        const Index* __restrict__ A_colind,
                        const a* __restrict__     A_val,
                        const Index* __restrict__ B_colptr,
                        const Index* __restrict__ B_rowind,
                        const b* __restrict__     B_val,
                        const Index* __restrict__ heavy_list,
                        const unsigned long long* __restrict__ heavy_count) {
  const int lane = threadIdx.x & 31;
  const unsigned long long nheavy = *heavy_count;
  unsigned long long w = (static_cast<unsigned long long>(blockIdx.x)*blockDim.x +
                          threadIdx.x) >> 5;
  const unsigned long long nwarps =
      (static_cast<unsigned long long>(gridDim.x)*blockDim.x) >> 5;
  for (; w < nheavy; w += nwarps) {
    const Index e     = heavy_list[2*w];
    const Index row   = heavy_list[2*w + 1];
    const Index j     = __ldg(mask_colind + e);
    const Index a_beg = __ldg(A_rowptr + row);
    const Index a_end = __ldg(A_rowptr + row + 1);
    const Index b_beg = __ldg(B_colptr + j);
    const Index b_end = __ldg(B_colptr + j + 1);
    c accumulator = identity;
    if (a_end - a_beg <= b_end - b_beg) {
      Index q = b_beg;
      for (Index p = a_beg + lane; p < a_end && q < b_end; p += 32) {
        const Index key = __ldg(A_colind + p);
        q = findSorted(B_rowind, q, b_end, key);
        if (q < b_end && __ldg(B_rowind + q) == key)
          accumulator = add_op(mul_op(A_val[p], B_val[q]), accumulator);
      }
    } else {
      Index p = a_beg;
      for (Index q = b_beg + lane; q < b_end && p < a_end; q += 32) {
        const Index key = __ldg(B_rowind + q);
        p = findSorted(A_colind, p, a_end, key);
        if (p < a_end && __ldg(A_colind + p) == key)
          accumulator = add_op(mul_op(A_val[p], B_val[q]), accumulator);
      }
    }
    accumulator = warpReduce(accumulator, add_op);
    if (lane == 0) C_val[e] = accumulator;
  }
}

}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_KERNELS_SPGEMM_MASKED_CUH_
