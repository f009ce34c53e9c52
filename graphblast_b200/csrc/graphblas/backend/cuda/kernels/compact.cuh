// graphblast_b200 backend — ORDERED stream compaction in two small kernels
// (count per CTA, whose last CTA scans the CTA counts -> emit).  Output order equals input
// order, so a compacted bitmap yields a sorted, duplicate-free index list with
// no sort at all — this is what replaces the reference's
// radix-sort + reduce-by-key in the push direction
// (reference spmspv_inner.hpp:233-316) and its updateFlag/Scan/streamCompact
// triples (reference kernels/util.hpp:52-148, spmspv.hpp:178-243,
// vector.hpp:391-413, assign.hpp:199-221).
//
// A "source" functor describes the items:
//   __device__ int  count(Index item) const;            // outputs of this item
//   __device__ void emit (Index item, Index pos) const; // write them at pos..
#ifndef GRAPHBLAS_BACKEND_CUDA_KERNELS_COMPACT_CUH_
#define GRAPHBLAS_BACKEND_CUDA_KERNELS_COMPACT_CUH_

#include "graphblas/backend/cuda/kernels/common.cuh"

namespace graphblas {
namespace backend {

#define GB_COMPACT_NT 256

// Count pass with the scan folded in: the CTA that finishes last (a counter that
// it leaves at zero again) scans the per-CTA counts in place, so the ordered
// compaction is two launches.
template <typename Source>
__global__ void __launch_bounds__(GB_COMPACT_NT)
compactCountScanKernel(Source src, Index nitems, int* __restrict__ block_counts,
                       int nblocks, unsigned long long* __restrict__ done,
                       unsigned long long* __restrict__ total_out,
                       unsigned long long* mail, unsigned long long ticket) {
  __shared__ int s_scan[GB_COMPACT_NT/32 + 1];
  __shared__ int s_carry;
  __shared__ bool s_last;
  // Source::kGroup consecutive items per thread (bitmap sources: 4 words): a
  // sparse frontier leaves almost every word empty, and a grid of one tiny item
  // per thread was launch- and tail-bound.
  const Index item0 = (static_cast<Index>(blockIdx.x)*GB_COMPACT_NT + threadIdx.x)
                      *Source::kGroup;
  int c = 0;
#pragma unroll
  for (int g = 0; g < Source::kGroup; ++g)
    if (item0 + g < nitems) c += src.count(item0 + g);
  int total = blockSum<GB_COMPACT_NT>(c, s_scan);
  if (threadIdx.x == 0) {
    block_counts[blockIdx.x] = total;
    __threadfence();
    s_last = (atomicAdd(done, 1ull) == gridDim.x - 1);
    s_carry = 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  volatile int* counts = block_counts;
  for (int base = 0; base < nblocks; base += GB_COMPACT_NT) {
    const int i = base + threadIdx.x;
    const int v = (i < nblocks) ? counts[i] : 0;
    int chunk_total;
    const int excl = blockExclusiveScan<GB_COMPACT_NT>(v, s_scan, &chunk_total);
    const int carry = s_carry;
    if (i < nblocks) counts[i] = carry + excl;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + chunk_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *total_out = static_cast<unsigned long long>(s_carry);
    *done = 0ull;
    if (mail != NULL) {          // post the total to the host (util.hpp mailbox)
      *reinterpret_cast<volatile unsigned long long*>(mail) =
          (ticket << 40) | static_cast<unsigned long long>(s_carry);
      __threadfence_system();
    }
  }
}

template <typename Source>
__global__ void __launch_bounds__(GB_COMPACT_NT)
compactEmitKernel(Source src, Index nitems,
                  const int* __restrict__ block_offsets) {
  __shared__ int s_scan[GB_COMPACT_NT/32 + 1];
  const Index item0 = (static_cast<Index>(blockIdx.x)*GB_COMPACT_NT + threadIdx.x)
                      *Source::kGroup;
  int cnt[Source::kGroup];
  int c = 0;
#pragma unroll
  for (int g = 0; g < Source::kGroup; ++g) {
    cnt[g] = (item0 + g < nitems) ? src.count(item0 + g) : 0;
    c += cnt[g];
  }
  int total;
  int excl = blockExclusiveScan<GB_COMPACT_NT>(c, s_scan, &total);
  int pos = block_offsets[blockIdx.x] + excl;
#pragma unroll
  for (int g = 0; g < Source::kGroup; ++g) {
    if (cnt[g] > 0) { src.emit(item0 + g, pos); pos += cnt[g]; }
    else if (item0 + g < nitems) src.finish(item0 + g);
  }
}

// ---------------------------------------------------------------------------
// Sources
// ---------------------------------------------------------------------------

// Dense vector -> sparse (ind, val) keeping entries != identity.
// One item = 8 consecutive elements.  StructOnly: values are not written.
template <typename T, bool StructOnly>
struct DenseCompactSource {
  static const int kGroup = 1;   // an item is already 8 contiguous values
  const T* u;
  T        identity;
  Index    n;
  Index*   out_ind;
  T*       out_val;

  __device__ int count(Index item) const {
    Index base = item*8;
    int c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (base + k < n) c += (u[base + k] != identity) ? 1 : 0;
    return c;
  }
  __device__ void emit(Index item, Index pos) const {
    Index base = item*8;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      if (base + k < n) {
        T v = u[base + k];
        if (v != identity) {
          out_ind[pos] = base + k;
          if (!StructOnly) out_val[pos] = v;
          ++pos;
        }
      }
    }
  }
  __device__ void finish(Index) const {}
};

// Touched-bitmap (+ dense accumulator) -> sorted sparse (ind, val).
// One item = one 32-bit word.  Restores the arena invariants on the way out:
// every visited accumulator cell goes back to `identity`, every word to 0.
//   KeyValue : values come from acc[]; otherwise the constant `one` is written.
//   DropZero : entries whose value == 0 are dropped (reference spmspv.hpp:203-243:
//              masked key-value push prunes zeros with updateFlag/streamCompact).
template <typename T, bool KeyValue, bool DropZero>
struct BitmapCompactSource {
  static const int kGroup = 4;   // 4 bitmap words per thread
  unsigned int* bits;
  T*            acc;
  T             identity;
  T             one;
  Index*        out_ind;
  T*            out_val;

  __device__ int count(Index item) const {
    unsigned int word = bits[item];
    if (!(KeyValue && DropZero)) return __popc(word);
    int c = 0;
    while (word) {
      int b = __ffs(word) - 1;
      word &= word - 1;
      if (acc[item*32 + b] != static_cast<T>(0)) ++c;
    }
    return c;
  }
  __device__ void emit(Index item, Index pos) const {
    unsigned int word = bits[item];
    while (word) {
      int b = __ffs(word) - 1;
      word &= word - 1;
      Index idx = item*32 + b;
      if (KeyValue) {
        T v = acc[idx];
        acc[idx] = identity;
        if (DropZero && v == static_cast<T>(0)) continue;
        out_ind[pos] = idx;
        out_val[pos] = v;
      } else {
        out_ind[pos] = idx;
        out_val[pos] = one;
      }
      ++pos;
    }
    bits[item] = 0u;
  }
  // Word had set bits but every value was dropped: still restore invariants.
  __device__ void finish(Index item) const {
    unsigned int word = bits[item];
    if (word == 0u) return;
    if (KeyValue) {
      while (word) {
        int b = __ffs(word) - 1;
        word &= word - 1;
        acc[item*32 + b] = identity;
      }
    }
    bits[item] = 0u;
  }
};

// Bitmap shadow of a dense vector (bit == value != 0) -> sparse (ind, val) for
// identity 0.  Read-only: one item = one word.
template <typename T, bool StructOnly>
struct DenseBitsCompactSource {
  static const int kGroup = 4;
  const unsigned int* bits;
  const T*            u;
  Index*              out_ind;
  T*                  out_val;

  __device__ int count(Index item) const { return __popc(bits[item]); }
  __device__ void emit(Index item, Index pos) const {
    unsigned int word = bits[item];
    while (word) {
      const int b = __ffs(word) - 1;
      word &= word - 1;
      const Index idx = item*32 + b;
      out_ind[pos] = idx;
      if (!StructOnly) out_val[pos] = u[idx];
      ++pos;
    }
  }
  __device__ void finish(Index) const {}
};

// Sparse vector filter: drop entries that the masked constant-assign would have
// overwritten with `val`, and entries already equal to `val`
// (reference assign.hpp:172-221: assignSparseKernel marks, updateFlag/scan/
// streamCompact prune "== val").  One item = one entry.
template <typename T, typename M, bool UseScmp>
struct SparseAssignFilterSource {
  static const int kGroup = 1;
  const Index* in_ind;
  const T*     in_val;
  const M*     mask;     // dense mask values
  T            val;
  Index*       out_ind;
  T*           out_val;

  __device__ bool keep(Index item) const {
    Index ind = in_ind[item];
    M m = mask[ind];
    bool overwritten = UseScmp ? (m == static_cast<M>(0))
                               : (m != static_cast<M>(0));
    return !overwritten && (in_val[item] != val);
  }
  __device__ int count(Index item) const { return keep(item) ? 1 : 0; }
  __device__ void emit(Index item, Index pos) const {
    out_ind[pos] = in_ind[item];
    out_val[pos] = in_val[item];
  }
  __device__ void finish(Index) const {}
};

}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_KERNELS_COMPACT_CUH_
