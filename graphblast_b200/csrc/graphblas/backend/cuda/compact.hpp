// graphblast_b200 backend — host driver for the ordered compaction kernels
// (kernels/compact.cuh).  Two launches (count pass whose last CTA scans the per-CTA
// counts, emit pass); the total reaches the host through the mailbox
// (util.hpp) while the emit pass is still running.
#ifndef GRAPHBLAS_BACKEND_CUDA_COMPACT_HPP_
#define GRAPHBLAS_BACKEND_CUDA_COMPACT_HPP_

#include "graphblas/backend/cuda/util.hpp"
#include "graphblas/backend/cuda/descriptor.hpp"
#include "graphblas/backend/cuda/kernels/kernels.hpp"

namespace graphblas {
namespace backend {

// Runs src over nitems items; returns the number of outputs emitted.
template <typename Source>
Index compactOrdered(Source src, Index nitems, Descriptor* desc) {
  if (nitems <= 0) return 0;
  const long long per_cta = static_cast<long long>(GB_COMPACT_NT)*Source::kGroup;
  const int nblocks = static_cast<int>((nitems + per_cta - 1) / per_cta);
  unsigned long long* ctr = desc->counters() + 1;
  cudaStream_t s = gbStream();
  int* block_counts = reinterpret_cast<int*>(
      desc->scratch(GB_SCRATCH_BLOCKSUM, static_cast<size_t>(nblocks)*sizeof(int)));
  // count + (last CTA) scan of the per-CTA counts, then emit: two launches
  // The total is posted to the host mailbox by the count pass, so the host
  // learns it while the emit pass is still running.
  const unsigned long long ticket = runtime().mailTicket();
  compactCountScanKernel<<<nblocks, GB_COMPACT_NT, 0, s>>>(src, nitems,
      block_counts, nblocks, desc->counters() + 2, ctr,
      runtime().mailSlot(0), ticket);
  GB_KERNEL_CHECK();
  compactEmitKernel<<<nblocks, GB_COMPACT_NT, 0, s>>>(src, nitems,
      block_counts);
  GB_KERNEL_CHECK();
  return static_cast<Index>(runtime().mailWait(0, ticket, ctr));
}

}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_COMPACT_HPP_
