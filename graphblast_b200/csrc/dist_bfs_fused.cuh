// graphblast_b200 — the 1-D row-partitioned BFS as ONE persistent cooperative kernel
// per GPU (SURVEY.md §8e + f2): level loop, direction decision, frontier exchange
// over NVLink peer memory and the cross-GPU level barrier all run on the device.
// Included by capi.cu after dist_exchange.cuh, whose exchange block it uses:
//   data[2][total_words]  the replicated frontier bitmap, double buffered by epoch
//   flags2[world]         flags2[r] = (last epoch rank r has published << 32) | size of
//                         the slice it published
//
// A level loop on the host (r01) paid per level: bitmap export, publish kernel,
// one-warp wait kernel, a host mailbox read, OR / import passes and the generic
// assign + mxv launches — about 40 us of latency against 10..100 us of work, which
// is why two GPUs were slower than one in r01.  Here a level is:
//   local phase   push: scan the global frontier, expand the columns of the local
//                 CSC (owned out-neighbours), claiming owned vertices in the
//                 replicated visited bitmap; heavy columns by the whole grid.
//                 pull: every owned unvisited row probes the replicated visited
//                 bitmap (first-neighbour summary, early exit) — operand reuse in
//                 its global form (reference kernels/spmv.hpp:36-38).
//   publish       all threads store the owned slice of the new frontier into
//                 data[epoch & 1] of EVERY rank (peer stores), then one thread
//                 writes this rank's count and flag to every rank and spins on the
//                 local flags until all ranks have published the epoch.
//                 Together with the frontier slice the owner stores the merged
//                 visited words of its slice into the OTHER visited copy of every
//                 rank: level L reads copy L & 1, which nobody writes during L, so
//                 no merge pass and no extra barrier are needed.
// One grid-wide barrier per level (two on a push level with heavy columns); the
// cross-GPU barrier doubles as the second one.  A rank can be at most one epoch ahead of the
// slowest one, and that epoch writes the other data buffer.
#ifndef GRAPHBLAST_B200_DIST_BFS_FUSED_CUH_
#define GRAPHBLAST_B200_DIST_BFS_FUSED_CUH_

#include <cooperative_groups.h>

// CTA shape of the distributed traversal kernel (validated at 2 and 8 GPUs with this
// shape; the single-GPU kernel chooses its own, kernels/bfs_fused.cuh)
#ifndef GBX_BFS_NT
#define GBX_BFS_NT 1024
#endif

namespace gbx {

struct BfsDistArgs {
  // local (nl x n) matrix: CSR rows = owned vertices with their in-neighbours
  // (global ids); CSC = per global vertex its owned out-neighbours (local ids)
  const Index* pull_ptr;  const Index* pull_ind;  const Index* pull_first;
  const unsigned int* pull_empty;    // owned rows without in-neighbours (bitmap)
  const Index* push_ptr;  const Index* push_ind;
  Index n, nl, source;
  long long lo;                      // first owned vertex (multiple of 32)
  int   max_levels, mode;
  float switchpoint;
  float*        levels;              // [nl] result
  unsigned int* next_own;            // [nw + 8] owned slice of the next frontier
  unsigned int* seed;                // [total_words] level-1 frontier
  char* const*  peers;               // exchange block of every rank
  int    world, rank;
  size_t off_data[2], off_flags2, off_visited[2];
  size_t word_lo, nw, total_words;
  unsigned long long epoch0;         // publishes completed before this traversal
  unsigned long long* cells;         // [0..2] found (rotating) [3..5] heavy (rotating)
                                     // [6] unused [7] levels out [8] error
                                     // [9..11] CTA check-in of the publish (rotating)
  Index* heavy;
  long long timeout_cycles;
};

__device__ __forceinline__ bool distClaim(unsigned int* visited, long long vtx) {
  const unsigned int bit = 1u << (vtx & 31);
  unsigned int* word = visited + (vtx >> 5);
  if (*reinterpret_cast<volatile unsigned int*>(word) & bit) return false;
  return (atomicOr(word, bit) & bit) == 0;
}

__device__ __forceinline__ unsigned long long distNow() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// Phase time stamps of the first 12 levels (thread 0 of the grid, nanoseconds):
// cells[16 + 4*level + {0: level start, 1: local phase done, 2: barrier passed,
// 3: level end}]; read by the host when GB200_BFS_TRACE=1.
#define GBX_TRACE(slot) do {                                                  \
  if (gtid == 0 && level < 12) a.cells[16 + 8*level + (slot)] = distNow();    \
} while (0)

template <int MINB>
__global__ void __launch_bounds__(GBX_BFS_NT, MINB)
bfsFusedDistKernel(BfsDistArgs a) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  __shared__ int s_red[GBX_BFS_NT/32];
  __shared__ unsigned long long s_total;
  __shared__ bool s_failed;

  const int lane = threadIdx.x & 31;
  const Index gtid = blockIdx.x*blockDim.x + threadIdx.x;
  const Index gthreads = gridDim.x*blockDim.x;
  const Index gwarp = gtid >> 5;
  const Index gwarps = gthreads >> 5;
  const Index total_words = static_cast<Index>(a.total_words);
  const Index nw = static_cast<Index>(a.nw);
  const Index word_lo = static_cast<Index>(a.word_lo);
  char* const local = a.peers[a.rank];

  // ---- level 0 ---------------------------------------------------------------------
  const long long src_local = static_cast<long long>(a.source) - a.lo;
  for (Index i = gtid; i < a.nl; i += gthreads)
    a.levels[i] = (static_cast<long long>(i) == src_local) ? 1.f : 0.f;
  // Only the visited copy that level 1 reads is initialised here: the other one
  // is written in full by the owners during level 1 — possibly before this rank's
  // kernel has even started.
  unsigned int* const vis_copy[2] = {
      reinterpret_cast<unsigned int*>(local + a.off_visited[0]),
      reinterpret_cast<unsigned int*>(local + a.off_visited[1])};
  for (Index w = gtid; w < total_words; w += gthreads) {
    const unsigned int seed = (w == (a.source >> 5)) ? (1u << (a.source & 31)) : 0u;
    // owned rows nothing points at count as visited from the start (no level can
    // discover them; the owner's merged words carry the bits to the other ranks)
    const bool own = w >= word_lo && w < word_lo + nw;
    vis_copy[1][w] = seed | (own ? a.pull_empty[w - word_lo] : 0u);
    a.seed[w] = seed;
  }
  for (Index w = gtid; w < nw + 8; w += gthreads) a.next_own[w] = 0u;
  if (gtid < 12) a.cells[gtid] = 0ull;
  grid.sync();

  const unsigned int* F = a.seed;
  unsigned long long fcount = 1ull;
  bool dense = (a.mode == 2);
  float prev_ratio = 0.f;
  int level = 1;
  bool failed = false;

  for (; level <= a.max_levels && fcount > 0ull && !failed; ++level) {
    if (a.mode == 0) {
      const float ratio = static_cast<float>(fcount)/static_cast<float>(a.n);
      if (!dense) {
        if (ratio > a.switchpoint && ratio > prev_ratio) dense = true; else prev_ratio = ratio;
      } else {
        if (ratio <= a.switchpoint && ratio < prev_ratio) dense = false; else prev_ratio = ratio;
      }
    }
    unsigned long long* const found_cell = a.cells + (level % 3);
    unsigned long long* const heavy_cell = a.cells + 3 + (level % 3);
    if (gtid == 0) {
      a.cells[(level + 1) % 3] = 0ull;
      a.cells[3 + (level + 1) % 3] = 0ull;
    }
    const float next_level = static_cast<float>(level + 1);
    int found_here = 0;
    unsigned int* const vis = vis_copy[level & 1];     // as of the level's start
    GBX_TRACE(0);

    if (!dense) {
      // ---------------- push over the local CSC --------------------------------------
      for (Index w0 = gwarp*32; w0 < total_words; w0 += gwarps*32) {
        const Index mine = w0 + lane;
        const unsigned int my_bits = (mine < total_words) ? __ldcg(F + mine) : 0u;
        unsigned int pending = __ballot_sync(GB_FULL_MASK, my_bits != 0u);
        while (pending != 0u) {
          const int src_lane = __ffs(pending) - 1;
          pending &= pending - 1u;
          unsigned int bits = __shfl_sync(GB_FULL_MASK, my_bits, src_lane);
          const Index w = w0 + src_lane;
          while (bits != 0u) {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1u;
            const Index u = w*32 + b;
            const Index beg = __ldg(a.push_ptr + u);
            const Index deg = __ldg(a.push_ptr + u + 1) - beg;
            if (deg > GB_BFS_HEAVY) {
              unsigned long long slot = 0ull;
              if (lane == 0) slot = atomicAdd(heavy_cell, 1ull);
              slot = __shfl_sync(GB_FULL_MASK, slot, 0);
              if (slot < GB_BFS_HEAVY_CAP) {
                if (lane == 0) a.heavy[slot] = u;
                continue;
              }
            }
            for (Index k = lane; k < deg; k += 32) {
              const Index r = __ldg(a.push_ind + beg + k);      // owned, local id
              if (distClaim(vis, a.lo + r)) {
                a.levels[r] = next_level;
                atomicOr(a.next_own + (r >> 5), 1u << (r & 31));
                ++found_here;
              }
            }
          }
        }
      }
      grid.sync();
      unsigned long long nheavy = *reinterpret_cast<volatile unsigned long long*>(heavy_cell);
      if (nheavy > GB_BFS_HEAVY_CAP) nheavy = GB_BFS_HEAVY_CAP;
      for (unsigned long long h = 0; h < nheavy; ++h) {
        const Index u = a.heavy[h];
        const Index beg = __ldg(a.push_ptr + u);
        const Index deg = __ldg(a.push_ptr + u + 1) - beg;
        for (Index k = gtid; k < deg; k += gthreads) {
          const Index r = __ldg(a.push_ind + beg + k);
          if (distClaim(vis, a.lo + r)) {
            a.levels[r] = next_level;
            atomicOr(a.next_own + (r >> 5), 1u << (r & 31));
            ++found_here;
          }
        }
      }
    } else {
      // ---------------- pull over the owned rows ---------------------------------------
      const Index ngroups = (nw + 3) >> 2;
      for (Index g = gwarp; g < ngroups; g += gwarps) {
        unsigned int mword[4];
        Index f[4];
        unsigned int pword[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const Index word = g*4 + j;
          mword[j] = (word < nw) ? __ldcg(vis + word_lo + word) : 0xffffffffu;
        }
        if ((mword[0] & mword[1] & mword[2] & mword[3]) == 0xffffffffu) {
          if (lane < 4 && g*4 + lane < nw) a.next_own[g*4 + lane] = 0u;   // nothing to find
          continue;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const Index row = (g*4 + j)*32 + lane;
          const bool open = (row < a.nl) && !((mword[j] >> lane) & 1u);
          f[j] = open ? __ldg(a.pull_first + row) : static_cast<Index>(-1);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          pword[j] = 0u;
          if (f[j] != static_cast<Index>(-1)) pword[j] = vis[(f[j] & 0x7fffffff) >> 5];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const Index word = g*4 + j;
          const Index row = word*32 + lane;
          bool found = (pword[j] >> (f[j] & 31)) & 1u;
          if (f[j] >= 0 && !found) {
            Index k = __ldg(a.pull_ptr + row) + 1;
            const Index end = __ldg(a.pull_ptr + row + 1);
            for (; k < end; ++k) {
              const Index col = __ldg(a.pull_ind + k);
              if ((vis[col >> 5] >> (col & 31)) & 1u) { found = true; break; }
            }
          }
          const unsigned int out = __ballot_sync(GB_FULL_MASK, found);
          if (word < nw) {
            if (found) a.levels[row] = next_level;
            if (lane == 0) a.next_own[word] = out;
          }
          found_here += found ? 1 : 0;
        }
      }
    }
    const int block_found = blockSum<GBX_BFS_NT>(found_here, s_red);
    if (threadIdx.x == 0 && block_found)
      atomicAdd(found_cell, static_cast<unsigned long long>(block_found));
    grid.sync();
    GBX_TRACE(1);

    // ---------------- publish the owned slice, cross-GPU level barrier -----------------
    // Every CTA stores its share of the slice into every rank's buffer and checks
    // in; the last one to do so posts this rank's count and flag to all ranks.
    // Then every CTA waits on the LOCAL flags of all ranks (its own included): the
    // cross-GPU barrier doubles as the grid barrier, no grid.sync() in between.
    const unsigned long long epoch = a.epoch0 + static_cast<unsigned long long>(level);
    const int par = static_cast<int>(epoch & 1ull);
    const int vnext = (level + 1) & 1;
    // 16-byte peer stores (slices start and end on multiples of 1024 vertices)
    {
      uint4* const mine4 = reinterpret_cast<uint4*>(a.next_own);
      const uint4* const vis4 = reinterpret_cast<const uint4*>(vis + word_lo);
      const Index nw4 = nw >> 2;
      const Index lo4 = word_lo >> 2;
      for (Index i = gtid; i < nw4; i += gthreads) {
        const uint4 word = __ldcg(mine4 + i);
        mine4[i] = make_uint4(0u, 0u, 0u, 0u);
        uint4 merged = __ldcg(vis4 + i);     // push levels claimed in `vis` already
        merged.x |= word.x; merged.y |= word.y; merged.z |= word.z; merged.w |= word.w;
        for (int p = 0; p < a.world; ++p) {
          reinterpret_cast<uint4*>(a.peers[p] + a.off_data[par])[lo4 + i] = word;
          reinterpret_cast<uint4*>(a.peers[p] + a.off_visited[vnext])[lo4 + i] = merged;
        }
      }
      for (Index i = (nw4 << 2) + gtid; i < nw; i += gthreads) {   // < 4 words, if any
        const unsigned int word = __ldcg(a.next_own + i);
        a.next_own[i] = 0u;
        const unsigned int merged = __ldcg(vis + word_lo + i) | word;
        for (int p = 0; p < a.world; ++p) {
          reinterpret_cast<unsigned int*>(a.peers[p] + a.off_data[par])[word_lo + i] = word;
          reinterpret_cast<unsigned int*>(a.peers[p] + a.off_visited[vnext])[word_lo + i] = merged;
        }
      }
    }
    // one system-scope fence per CTA, after the CTA barrier: cumulativity carries
    // the other threads' peer stores
    __syncthreads();
    GBX_TRACE(4);
    if (threadIdx.x == 0) {
      __threadfence_system();
      GBX_TRACE(5);
      unsigned long long* const done_cell = a.cells + 9 + (level % 3);
      if (atomicAdd(done_cell, 1ull) == gridDim.x - 1) {
        a.cells[9 + (level + 1) % 3] = 0ull;           // next level's check-in counter
        __threadfence();
        const unsigned long long mine =
            *reinterpret_cast<volatile unsigned long long*>(found_cell);
        // one word per rank carries the epoch and this rank's count
        const unsigned long long word = (epoch << 32) | (mine & 0xffffffffull);
        for (int p = 0; p < a.world; ++p)
          reinterpret_cast<volatile unsigned long long*>(
              a.peers[p] + a.off_flags2)[a.rank] = word;
      }
      GBX_TRACE(6);
      const volatile unsigned long long* flags =
          reinterpret_cast<const volatile unsigned long long*>(local + a.off_flags2);
      const long long t0 = clock64();
      bool ok = true;
      unsigned long long total = 0ull;
      for (int p = 0; p < a.world && ok; ++p) {
        unsigned long long seen = flags[p];
        while ((seen >> 32) < (epoch & 0xffffffffull)) {
          if (clock64() - t0 > a.timeout_cycles) { ok = false; break; }
          __nanosleep(8);
          seen = flags[p];
        }
        total += seen & 0xffffffffull;
      }
      __threadfence_system();
      if (!ok) { total = 0ull; a.cells[8] = 1ull; }
      s_total = total;
      s_failed = !ok;
    }
    __syncthreads();
    fcount = s_total;
    failed = s_failed;
    GBX_TRACE(2);

    F = reinterpret_cast<const unsigned int*>(local + a.off_data[par]);
    GBX_TRACE(3);
  }
  if (gtid == 0) a.cells[7] = static_cast<unsigned long long>(level - 1);
}

}  // namespace gbx

extern "C" {

// Contract in include/graphblast_b200.h; one cooperative launch per traversal.
int gb200_dist_bfs_fused(gb200_xchg_t x, gb200_vector_t v, gb200_matrix_t M,
                         long long n, long long source, gb200_desc_t desc,
                         int* levels_out) {
  if (x == NULL || v == NULL || M == NULL || desc == NULL)
    return rc(graphblas::GrB_NULL_POINTER);
  if (!x->connected || M->f == NULL) return rc(graphblas::GrB_UNINITIALIZED_OBJECT);
  GB200_REQUIRE_DEVICE();
  using namespace graphblas;              // NOLINT(build/namespaces)
  using namespace graphblas::backend;     // NOLINT(build/namespaces)
  cudaStream_t s = gbStream();
  backend::SparseMatrix<float>& S = M->f->matrix_.sparse_;
  backend::Descriptor& d = desc->desc.descriptor_;
  Index nl;
  CHECK(v->f->size(&nl));
  if (S.d_csrRowPtr_ == NULL || S.d_cscColPtr_ == NULL) return rc(GrB_UNINITIALIZED_OBJECT);
  CHECK(v->f->vector_.setStorage(GrB_DENSE));
  CHECK(v->f->vector_.dense_.allocateGpu());

  // first-neighbour summary of the local rows (same cache as the Boolean pull)
  const int fw = 0;
  const Index* first = backend::pullFirstNeighbours(&S, fw, S.d_csrRowPtr_, S.d_csrColInd_,
                                                    S.nrows_);

  const size_t w_lo = x->word_off[x->rank];
  const size_t nw = x->word_off[x->rank + 1] - w_lo;
  const size_t own_bytes = ((nw + 8)*4 + 255)/256*256;
  unsigned char* base = reinterpret_cast<unsigned char*>(d.scratch(GB_SCRATCH_BFS,
      own_bytes + 1024 + GB_BFS_HEAVY_CAP*sizeof(Index)));
  gbx::BfsDistArgs a;
  a.pull_ptr = S.d_csrRowPtr_;  a.pull_ind = S.d_csrColInd_;
  a.pull_first = first;
  a.pull_empty = backend::pullEmptyRowBits(first, S.nrows_);
  a.push_ptr = S.d_cscColPtr_;  a.push_ind = S.d_cscRowInd_;
  a.n = static_cast<Index>(n);  a.nl = nl;  a.source = static_cast<Index>(source);
  a.lo = static_cast<long long>(w_lo)*32;
  a.max_levels = d.max_niter_;
  a.switchpoint = d.switchpoint();
  Desc_value mode;
  CHECK(desc->desc.get(GrB_MXVMODE, &mode));
  a.mode = (mode == GrB_PUSHONLY) ? 1 : (mode == GrB_PULLONLY ? 2 : 0);
  a.levels = v->f->vector_.dense_.d_val_;
  a.seed = x->d_seed;
  a.next_own = reinterpret_cast<unsigned int*>(base);
  a.cells = reinterpret_cast<unsigned long long*>(base + own_bytes);
  a.heavy = reinterpret_cast<Index*>(base + own_bytes + 1024);
  a.peers = x->d_peer;
  a.world = x->world;  a.rank = x->rank;
  a.off_data[0] = x->off_data[0];  a.off_data[1] = x->off_data[1];
  a.off_flags2 = x->off_flags2;
  a.off_visited[0] = x->off_visited[0];  a.off_visited[1] = x->off_visited[1];
  a.word_lo = w_lo;  a.nw = nw;  a.total_words = x->total_words;
  a.epoch0 = x->epoch;
  a.timeout_cycles = 20000000000ll;

  void (*kernel)(gbx::BfsDistArgs) = gbx::bfsFusedDistKernel<2>;
  static int resident = 0;
  if (resident == 0) {
    int per_sm = 0;
    CUDA_CALL(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, GBX_BFS_NT, 0));
    resident = per_sm*runtime().sm_count;
    if (resident < 1) return rc(GrB_PANIC);
  }
  void* params[] = { &a };
  profiler().begin(GB_PROF_PULL_BOOL, s);
  CUDA_CALL(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kernel), dim3(resident),
      dim3(GBX_BFS_NT), params, 0, s));
  GB_KERNEL_CHECK();
  profiler().end(GB_PROF_PULL_BOOL, s, 0.0);
  v->f->vector_.dense_.touched();
  // every rank ran the same number of levels = publishes
  unsigned long long out[2];
  CUDA_CALL(cudaMemcpyAsync(out, a.cells + 7, 2*sizeof(unsigned long long),
      cudaMemcpyDeviceToHost, s));
  runtime().sync();
  x->epoch += out[0];
  static const int trace = getEnv("GB200_BFS_TRACE", 0);
  if (trace) {
    unsigned long long t[112];
    CUDA_CALL(cudaMemcpy(t, a.cells + 16, sizeof(t), cudaMemcpyDeviceToHost));
    for (unsigned long long l = 1; l <= out[0] && l < 12; ++l)
      fprintf(stderr, "rank %d level %llu: local %.1f | stores %.1f fence %.1f check-in %.1f "
              "wait %.1f us\n", x->rank, l, (t[8*l + 1] - t[8*l])*1e-3,
              (t[8*l + 4] - t[8*l + 1])*1e-3, (t[8*l + 5] - t[8*l + 4])*1e-3,
              (t[8*l + 6] - t[8*l + 5])*1e-3, (t[8*l + 2] - t[8*l + 6])*1e-3);
  }
  if (levels_out != NULL) *levels_out = static_cast<int>(out[0]);
  return out[1] != 0ull ? rc(GrB_PANIC) : 0;
}

}  // extern "C"

#endif  // GRAPHBLAST_B200_DIST_BFS_FUSED_CUH_
