// graphblast_b200 backend — host side of the fused BFS (kernels/bfs_fused.cuh):
// one cooperative launch per traversal.  Entered from algorithm::bfs of this
// project's frontend when the descriptor carries the BFS flags of the reference's
// benchmark script (run_bfs.sh:8-27: --struconly 1 --opreuse 1 --earlyexit 1,
// --fusedmask 1); every other combination runs the operation-by-operation loop.
#ifndef GRAPHBLAS_BACKEND_CUDA_BFS_FUSED_HPP_
#define GRAPHBLAS_BACKEND_CUDA_BFS_FUSED_HPP_

#include "graphblas/backend/cuda/kernels/bfs_fused.cuh"

namespace graphblas {
namespace backend {

// True when the traversal described by desc is the one the fused kernel computes.
inline bool bfsFusedApplies(Descriptor* desc) {
  static const int enabled = getEnv("GB200_BFS_FUSED", 1);
  if (!enabled) return false;
  Desc_value mask_mode, outp, inp0, inp1;
  if (desc->get(GrB_MASK, &mask_mode) != GrB_SUCCESS) return false;
  desc->get(GrB_OUTP, &outp); desc->get(GrB_INP0, &inp0); desc->get(GrB_INP1, &inp1);
  return desc->struconly() && desc->opreuse() && desc->earlyexit() && desc->fusedmask() &&
         mask_mode == GrB_DEFAULT && outp == GrB_DEFAULT && inp0 == GrB_DEFAULT &&
         inp1 == GrB_DEFAULT && !desc->debug() && desc->timing_ != 1;
}

__global__ void bfsAccountKernel(unsigned long long* cell,
                                 const unsigned long long* counters, Index n) {
  const unsigned long long bytes =
      counters[8]*(12ull*static_cast<unsigned long long>(n) + 4ull) + 4ull*counters[7] +
      12ull*counters[9] + 8ull*counters[10] + 8ull*counters[11];
  atomicAdd(cell, bytes);
}

// Work counters of the last fused traversal run with this descriptor: levels,
// entries inspected pulling, pull levels, vertices pushed, edges pushed, vertices
// discovered pushing.  Zeros when none has run.
inline void bfsFusedStats(Descriptor* desc, Index n, unsigned long long out[6]) {
  for (int i = 0; i < 6; ++i) out[i] = 0ull;
  const size_t nwords = (static_cast<size_t>(n) + 31)/32;
  const size_t words_bytes = ((nwords*sizeof(unsigned int) + 255)/256)*256;
  if (desc->scratchSize(GB_SCRATCH_BFS) < 4*words_bytes + 256) return;
  unsigned char* base = reinterpret_cast<unsigned char*>(desc->scratch(GB_SCRATCH_BFS, 0));
  CUDA_CALL(cudaMemcpyAsync(out, base + 4*words_bytes + 6*sizeof(unsigned long long),
      6*sizeof(unsigned long long), cudaMemcpyDeviceToHost, gbStream()));
  runtime().sync();
}

// v = BFS levels of A from s (source 1, unreached 0).  *depth = levels executed.
template <typename a>
Info bfsFused(Vector<float>* v, const Matrix<a>* A, Index s, Descriptor* desc, int* depth) {
  SparseMatrix<a>* S = const_cast<SparseMatrix<a>*>(&A->sparse_);
  const Index n = S->nrows_;
  if (n != S->ncols_) return GrB_DIMENSION_MISMATCH;
  if (S->d_csrRowPtr_ == NULL || S->d_cscColPtr_ == NULL) return GrB_UNINITIALIZED_OBJECT;
  cudaStream_t stream = gbStream();
  CHECK(v->setStorage(GrB_DENSE));
  CHECK(v->dense_.allocateGpu());

  // first-neighbour summary of the pulled structure (shared with the Boolean pull)
  const int fw = 1;                                   // vxm pulls over the CSC
  const Index* first = pullFirstNeighbours(S, fw, S->d_cscColPtr_, S->d_cscRowInd_, n);

  const size_t nwords = (static_cast<size_t>(n) + 31)/32;
  const size_t words_bytes = ((nwords*sizeof(unsigned int) + 255)/256)*256;
  unsigned char* base = reinterpret_cast<unsigned char*>(desc->scratch(GB_SCRATCH_BFS,
      4*words_bytes + 256 + GB_BFS_HEAVY_CAP*sizeof(Index)));
  BfsFusedArgs args;
  args.push_ptr = S->d_csrRowPtr_;  args.push_ind = S->d_csrColInd_;
  args.pull_ptr = S->d_cscColPtr_;  args.pull_ind = S->d_cscRowInd_;
  args.pull_first = first;
  args.pull_empty = pullEmptyRowBits(first, n);
  args.n = n;
  args.source = s;
  args.max_levels = desc->max_niter_;
  args.switchpoint = desc->switchpoint();
  Desc_value mode;
  CHECK(desc->get(GrB_MXVMODE, &mode));
  args.mode = (mode == GrB_PUSHONLY) ? 1 : (mode == GrB_PULLONLY ? 2 : 0);
  args.levels = v->dense_.d_val_;
  args.visited[0] = reinterpret_cast<unsigned int*>(base);
  args.visited[1] = reinterpret_cast<unsigned int*>(base + words_bytes);
  args.frontier   = reinterpret_cast<unsigned int*>(base + 2*words_bytes);
  args.next       = reinterpret_cast<unsigned int*>(base + 3*words_bytes);
  args.counters   = reinterpret_cast<unsigned long long*>(base + 4*words_bytes);
  args.heavy      = reinterpret_cast<Index*>(base + 4*words_bytes + 256);

  static int resident = 0;               // CTAs that fit at once (cooperative launch)
  void (*kernel)(BfsFusedArgs) = bfsFusedKernel<GB_BFS_MINB>;
  if (resident == 0) {
    int per_sm = 0;
    CUDA_CALL(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel,
        GB_BFS_NT, 0));
    resident = per_sm*runtime().sm_count;
    if (resident < 1) return GrB_PANIC;
  }
  void* params[] = { &args };
  profiler().begin(GB_PROF_PULL_BOOL, stream);
  CUDA_CALL(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel),
      dim3(resident), dim3(GB_BFS_NT), params, 0, stream));
  GB_KERNEL_CHECK();
  profiler().end(GB_PROF_PULL_BOOL, stream, 0.0);
  if (profiler().enabled) {
    // algorithmic bytes of the traversal (SURVEY.md §8d), from the kernel's own
    // work counters: per pull level 4(n+1) + 4n + 4n, 4 per inspected entry; per
    // push 12 per frontier entry, 8 per expanded edge (colind + visited lookup),
    // 8 per discovered vertex
    bfsAccountKernel<<<1, 1, 0, stream>>>(profiler().d_cells + GB_PROF_PULL_BOOL,
        args.counters, n);
    GB_KERNEL_CHECK();
  }
  v->dense_.touched();
  static const int trace = getEnv("GB200_BFS_TRACE", 0);
  if (trace) {                           // per-level times of this traversal
    unsigned long long cells[32];
    CUDA_CALL(cudaMemcpyAsync(cells, args.counters, sizeof(cells), cudaMemcpyDeviceToHost,
        stream));
    runtime().sync();
    const int levels = static_cast<int>(cells[6] < 15 ? cells[6] : 15);
    fprintf(stderr, "bfs trace: set-up %.1fus",
            1e-3*static_cast<double>((cells[12] >> 1) - cells[28]));
    for (int l = 1; l <= levels; ++l)
      fprintf(stderr, " L%d %s %.1fus", l, (cells[12 + l] & 1ull) ? "pull" : "push",
              1e-3*static_cast<double>((cells[12 + l] >> 1) - (cells[12 + l - 1] >> 1)));
    fprintf(stderr, " | L2 CTA0: scan %.1fus walk %.1fus parked %llu\n",
            1e-3*static_cast<double>(cells[29] - (cells[13] >> 1)),
            1e-3*static_cast<double>(cells[30] - cells[29]), cells[31]);
  }
  if (depth != NULL) {
    const unsigned long long levels = runtime().fetch(args.counters + 6);
    *depth = static_cast<int>(levels);
    desc->lastmxv_ = GrB_PULLONLY;
  }
  return GrB_SUCCESS;
}

}  // namespace backend
}  // namespace graphblas

#endif  // GRAPHBLAS_BACKEND_CUDA_BFS_FUSED_HPP_
