// graphblast_b200 — multi-GPU frontier exchange over peer memory and the native
// loops of the 1-D row-partitioned PageRank and SSSP (SURVEY.md §8e); the BFS is
// dist_bfs_fused.cuh.  Included by capi.cu.
//
// One process per GPU.  Every rank owns a block of device memory that all ranks
// map through CUDA IPC:
//
//   data[2][total_words]   the replicated frontier (bitmap words), double buffered
//   counts[2][world]       per-rank entry counts of the published slice
//   flags[world]           flags[r] = number of publishes rank r has completed
//   visited[2][total_words] (fused BFS only) replicated visited bitmap, by level parity
//
// publish(): ONE kernel stores the owned slice into data[parity] of EVERY peer
// (NVLink stores), then the last CTA writes the slice's count and the new flag
// value to every peer.  wait(): one warp spins on the local flags until every
// rank has published this epoch and sums the counts.  No NCCL call, no host
// round trip besides reading the 8-byte total that decides termination and
// direction.  Double buffering makes the scheme race free: a rank can only run
// one publish ahead of the slowest rank, and that publish goes to the other
// buffer.
#ifndef GRAPHBLAST_B200_DIST_EXCHANGE_CUH_
#define GRAPHBLAST_B200_DIST_EXCHANGE_CUH_

struct gb200_xchg_s {
  int    world, rank;
  size_t total_words;
  std::vector<size_t> word_off;          // world + 1
  size_t off_data[2], off_counts[2], off_flags, off_visited[2], off_flags2, bytes;
  char*  local;
  std::vector<char*> peer;               // peer[rank] == local
  char** d_peer;                         // device copy of peer[]
  unsigned long long  epoch;             // publishes issued so far
  unsigned long long* d_cells;           // [0] finished CTAs, [1] popcount, [2] total
  unsigned int*       d_seed;            // owned-slice scratch
  bool connected;
  // vectors of the PageRank loop: p_glob, p_prev_own, p_swap, r, r_temp
  graphblas::Vector<float>* pr_vec[5];
  // vectors of the SSSP loop: frontier_glob (view), relaxed, improved
  graphblas::Vector<float>* ss_vec[3];
};

namespace gbx {

using namespace graphblas::backend;  // NOLINT(build/namespaces)

#define GBX_NT 256

// Stores src[0..nwords) at word offset word_lo of data[] in every peer's block,
// then (last CTA) the count and the flag.  d_count_in != NULL: the count is
// already on the device; otherwise it is the popcount of the words.
__global__ void __launch_bounds__(GBX_NT)
xchgPublishKernel(const unsigned int* __restrict__ src, size_t nwords,
                  size_t word_lo, char* const* __restrict__ peers, int world,
                  int rank, size_t off_data, size_t off_counts, size_t off_flags,
                  unsigned long long epoch, unsigned long long* d_cells,
                  const unsigned long long* d_count_in, int use_imm,
                  unsigned long long imm) {
  __shared__ int s_red[GBX_NT/32];
  int pop = 0;
  size_t i = static_cast<size_t>(blockIdx.x)*GBX_NT + threadIdx.x;
  const size_t stride = static_cast<size_t>(gridDim.x)*GBX_NT;
  const bool vec = ((nwords | word_lo) & 3) == 0 &&
                   (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  if (vec) {
    // 16-byte loads and peer stores (the float payloads are megabytes per rank)
    const uint4* src4 = reinterpret_cast<const uint4*>(src);
    const size_t n4 = nwords >> 2;
    for (; i < n4; i += stride) {
      const uint4 w = src4[i];
      pop += __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
      for (int p = 0; p < world; ++p) {
        uint4* dst = reinterpret_cast<uint4*>(
            reinterpret_cast<unsigned int*>(peers[p] + off_data) + word_lo) + i;
        *dst = w;
      }
    }
  } else {
    for (; i < nwords; i += stride) {
      const unsigned int w = src[i];
      pop += __popc(w);
      for (int p = 0; p < world; ++p) {
        unsigned int* dst =
            reinterpret_cast<unsigned int*>(peers[p] + off_data) + word_lo + i;
        *dst = w;
      }
    }
  }
  const int total = blockSum<GBX_NT>(pop, s_red);
  if (threadIdx.x == 0 && total != 0 && d_count_in == NULL && !use_imm)
    atomicAdd(d_cells + 1, static_cast<unsigned long long>(total));
  __threadfence_system();          // this CTA's peer stores before its "done"
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long done = atomicAdd(d_cells, 1ull);
    if (done == gridDim.x - 1) {
      __threadfence();
      const unsigned long long cnt = use_imm ? imm : (d_count_in != NULL)
          ? *d_count_in
          : *reinterpret_cast<volatile unsigned long long*>(d_cells + 1);
      for (int p = 0; p < world; ++p) {
        volatile unsigned long long* c = reinterpret_cast<
            volatile unsigned long long*>(peers[p] + off_counts) + rank;
        *c = cnt;
      }
      __threadfence_system();      // data + counts before the flag
      for (int p = 0; p < world; ++p) {
        volatile unsigned long long* f = reinterpret_cast<
            volatile unsigned long long*>(peers[p] + off_flags) + rank;
        *f = epoch;
      }
      d_cells[0] = 0ull;
      d_cells[1] = 0ull;
    }
  }
}

// One warp: waits until every rank's flag has reached `epoch`, then
// d_cells[2] = sum of the published counts (all ones on timeout).
__global__ void xchgWaitKernel(const char* __restrict__ local, size_t off_counts,
                               size_t off_flags, int world,
                               unsigned long long epoch,
                               unsigned long long* d_cells,
                               long long timeout_cycles, int as_double,
                               unsigned long long* mail,
                               unsigned long long ticket) {
  const int lane = threadIdx.x;
  bool ok = true;
  if (lane < world) {
    const volatile unsigned long long* f = reinterpret_cast<
        const volatile unsigned long long*>(local + off_flags) + lane;
    const long long t0 = clock64();
    while (*f < epoch) {
      if (clock64() - t0 > timeout_cycles) { ok = false; break; }
      __nanosleep(64);
    }
  }
  ok = __all_sync(GB_FULL_MASK, ok);
  __threadfence_system();
  unsigned long long c = 0ull;
  if (ok && lane < world)
    c = *(reinterpret_cast<const volatile unsigned long long*>(
        local + off_counts) + lane);
  if (as_double) {
    // the per-rank cells hold doubles (partial sums); lane 0 adds them in rank
    // order so every rank computes the identical total
    double sum = 0.0;
    for (int p = 0; p < world; ++p) {
      const unsigned long long bits = __shfl_sync(GB_FULL_MASK, c, p);
      sum += __longlong_as_double(static_cast<long long>(bits));
    }
    if (lane == 0)
      d_cells[2] = ok ? static_cast<unsigned long long>(
          __double_as_longlong(sum)) : ~0ull;
    return;
  }
  for (int d = 16; d > 0; d >>= 1)
    c += __shfl_down_sync(GB_FULL_MASK, c, d);
  if (lane == 0) {
    d_cells[2] = ok ? c : ~0ull;
    if (mail != NULL && ok && c < (1ull << 40)) {   // host mailbox (util.hpp)
      *reinterpret_cast<volatile unsigned long long*>(mail) = (ticket << 40) | c;
      __threadfence_system();
    }
  }
}

inline int publish(gb200_xchg_s* x, const unsigned int* d_words,
                   const unsigned long long* d_count, int use_imm = 0,
                   unsigned long long imm = 0ull) {
  cudaStream_t s = gbStream();
  x->epoch += 1;
  const int par = static_cast<int>(x->epoch & 1ull);
  const size_t nw = x->word_off[x->rank + 1] - x->word_off[x->rank];
  int grid = static_cast<int>((nw/4 + GBX_NT - 1)/GBX_NT);
  if (grid > 4*runtime().sm_count) grid = 4*runtime().sm_count;
  if (grid < 1) grid = 1;
  xchgPublishKernel<<<grid, GBX_NT, 0, s>>>(d_words, nw, x->word_off[x->rank],
      x->d_peer, x->world, x->rank, x->off_data[par], x->off_counts[par],
      x->off_flags, x->epoch, x->d_cells, d_count, use_imm, imm);
  GB_KERNEL_CHECK();
  return 0;
}

// Waits for the epoch just published; returns the raw 8-byte total (integer
// sum of the ranks' cells, or the bits of their double sum), ~0 on timeout.
inline unsigned long long waitRaw(gb200_xchg_s* x, int as_double) {
  cudaStream_t s = gbStream();
  const int par = static_cast<int>(x->epoch & 1ull);
  // ~10 s at 2 GHz: a rank that died must not hang the others' GPUs
  // integer totals are posted to the host mailbox: no stream synchronisation
  const bool mail = !as_double;
  const unsigned long long ticket = mail ? runtime().mailTicket() : 0ull;
  xchgWaitKernel<<<1, 32, 0, s>>>(x->local, x->off_counts[par], x->off_flags,
      x->world, x->epoch, x->d_cells, 20000000000ll, as_double,
      mail ? runtime().mailSlot(3) : NULL, ticket);
  GB_KERNEL_CHECK();
  if (mail) return runtime().mailWait(3, ticket, x->d_cells + 2);
  return runtime().fetch(x->d_cells + 2);
}

// Returns the global count of the epoch just published, or -1 on timeout.
inline long long wait(gb200_xchg_s* x) {
  const unsigned long long total = waitRaw(x, 0);
  if (total == ~0ull) return -1;
  return static_cast<long long>(total);
}

inline const unsigned int* current(gb200_xchg_s* x) {
  const int par = static_cast<int>(x->epoch & 1ull);
  return reinterpret_cast<const unsigned int*>(x->local + x->off_data[par]);
}

}  // namespace gbx

extern "C" {

int gb200_xchg_create(gb200_xchg_t* out, int world, int rank,
                      const long long* word_offsets) {
  if (out == NULL || word_offsets == NULL || world < 1 || world > 32 ||
      rank < 0 || rank >= world)
    return rc(graphblas::GrB_INVALID_VALUE);
  GB200_REQUIRE_DEVICE();
  gb200_xchg_s* x = new gb200_xchg_s();
  x->world = world; x->rank = rank;
  x->word_off.resize(world + 1);
  for (int p = 0; p <= world; ++p)
    x->word_off[p] = static_cast<size_t>(word_offsets[p]);
  x->total_words = x->word_off[world];
  size_t off = 0;
  const size_t data_bytes = ((x->total_words + 8)*4 + 255) & ~size_t(255);
  for (int b = 0; b < 2; ++b) { x->off_data[b] = off; off += data_bytes; }
  for (int b = 0; b < 2; ++b) { x->off_counts[b] = off; off += 256; }
  x->off_flags = off; off += 256;
  // two replicated visited bitmaps for the fused BFS kernel (dist_bfs_fused.cuh):
  // owners store their slice of the NEXT level's copy into every rank
  for (int b = 0; b < 2; ++b) { x->off_visited[b] = off; off += data_bytes; }
  // flags of the fused kernel: one word per rank = (epoch << 32) | slice count, so
  // the count needs no store + fence of its own
  x->off_flags2 = off; off += 256;
  x->bytes = off;
  CUDA_CALL(cudaMalloc(&x->local, x->bytes));
  CUDA_CALL(cudaMemset(x->local, 0, x->bytes));
  CUDA_CALL(cudaMalloc(&x->d_cells, 8*sizeof(unsigned long long)));
  CUDA_CALL(cudaMemset(x->d_cells, 0, 8*sizeof(unsigned long long)));
  CUDA_CALL(cudaMalloc(&x->d_seed, (x->total_words + 8)*4));
  CUDA_CALL(cudaMalloc(&x->d_peer, world*sizeof(char*)));
  x->peer.assign(world, static_cast<char*>(NULL));
  x->peer[rank] = x->local;
  x->epoch = 0;
  x->connected = (world == 1);
  if (world == 1)
    CUDA_CALL(cudaMemcpy(x->d_peer, x->peer.data(), sizeof(char*),
        cudaMemcpyHostToDevice));
  for (int i = 0; i < 5; ++i) x->pr_vec[i] = NULL;
  for (int i = 0; i < 3; ++i) x->ss_vec[i] = NULL;
  *out = x;
  return 0;
}

int gb200_xchg_handle(gb200_xchg_t x, void* out64) {
  if (x == NULL || out64 == NULL) return rc(graphblas::GrB_NULL_POINTER);
  cudaIpcMemHandle_t h;
  CUDA_CALL(cudaIpcGetMemHandle(&h, x->local));
  static_assert(sizeof(h) == 64, "IPC handle size");
  memcpy(out64, &h, 64);
  return 0;
}

int gb200_xchg_connect(gb200_xchg_t x, const void* handles) {
  if (x == NULL || handles == NULL) return rc(graphblas::GrB_NULL_POINTER);
  for (int p = 0; p < x->world; ++p) {
    if (p == x->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char*>(handles) + 64*p, 64);
    void* ptr = NULL;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h,
        cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      std::cerr << "gb200_xchg_connect: cannot map rank " << p << ": "
                << cudaGetErrorString(e) << std::endl;
      cudaGetLastError();
      return rc(graphblas::GrB_PANIC);
    }
    x->peer[p] = static_cast<char*>(ptr);
  }
  CUDA_CALL(cudaMemcpy(x->d_peer, x->peer.data(), x->world*sizeof(char*),
      cudaMemcpyHostToDevice));
  x->connected = true;
  return 0;
}

int gb200_xchg_free(gb200_xchg_t x) {
  if (x == NULL) return 0;
  cudaDeviceSynchronize();
  for (int p = 0; p < x->world; ++p)
    if (p != x->rank && x->peer[p] != NULL) cudaIpcCloseMemHandle(x->peer[p]);
  cudaFree(x->local); cudaFree(x->d_cells);
  cudaFree(x->d_seed); cudaFree(x->d_peer);
  for (int i = 0; i < 5; ++i) delete x->pr_vec[i];
  for (int i = 0; i < 3; ++i) delete x->ss_vec[i];
  delete x;
  return 0;
}

// Publishes the owned slice held in vector v (dense or sparse, length = owned
// vertex count) and returns the global entry count once every rank has done so.
int gb200_xchg_allgather_bits(gb200_xchg_t x, gb200_vector_t v,
                              long long* total_out) {
  if (x == NULL || v == NULL || total_out == NULL)
    return rc(graphblas::GrB_NULL_POINTER);
  if (!x->connected) return rc(graphblas::GrB_UNINITIALIZED_OBJECT);
  GB200_REQUIRE_DEVICE();
  int info = gb200_vector_export_bits_async(v, x->d_seed, x->d_cells + 3);
  if (info != 0) return info;
  gbx::publish(x, x->d_seed, x->d_cells + 3);
  const long long total = gbx::wait(x);
  if (total < 0) return rc(graphblas::GrB_PANIC);
  *total_out = total;
  return 0;
}

int gb200_xchg_bits_ptr(gb200_xchg_t x, const uint32_t** d_bits) {
  if (x == NULL || d_bits == NULL) return rc(graphblas::GrB_NULL_POINTER);
  *d_bits = gbx::current(x);
  return 0;
}

// Generic form for 32-bit payloads (float vectors): publishes nwords_owned words
// from d_words with this rank's partial scalar; *sum_out = sum over ranks.
int gb200_xchg_allgather_words(gb200_xchg_t x, const void* d_words,
                               double partial, double* sum_out) {
  if (x == NULL || d_words == NULL || sum_out == NULL)
    return rc(graphblas::GrB_NULL_POINTER);
  if (!x->connected) return rc(graphblas::GrB_UNINITIALIZED_OBJECT);
  GB200_REQUIRE_DEVICE();
  unsigned long long bits;
  memcpy(&bits, &partial, 8);
  gbx::publish(x, static_cast<const unsigned int*>(d_words), NULL, 1, bits);
  const unsigned long long total = gbx::waitRaw(x, 1);
  if (total == ~0ull) return rc(graphblas::GrB_PANIC);
  memcpy(sum_out, &total, 8);
  return 0;
}

// PageRank over the 1-D row partition (the loop of algorithm/pr.hpp on the owned
// slice).  The exchange must have been created with one word per VERTEX
// (word_offsets = vertex bounds).  p (length nl) = owned ranks (output);
// M = owned rows of (alpha * A ./ outdeg)^T as an (nl x n) CSR matrix.
// Per iteration: p_swap = M (+.x) p_glob ; p = p_swap + (1-alpha)/n ;
// r = p - p_prev ; err_partial = sum(r.*r) ; peers exchange p and the partial.
int gb200_dist_pr(gb200_xchg_t x, gb200_vector_t p, gb200_matrix_t M,
                  long long n, float alpha, float eps, gb200_desc_t desc,
                  int* iters_out) {
  if (x == NULL || p == NULL || M == NULL || desc == NULL)
    return rc(graphblas::GrB_NULL_POINTER);
  if (!x->connected || M->f == NULL) return rc(graphblas::GrB_UNINITIALIZED_OBJECT);
  GB200_REQUIRE_DEVICE();
  using namespace graphblas;          // NOLINT(build/namespaces)
  Descriptor* d = &desc->desc;
  const size_t lo = x->word_off[x->rank];
  Index nl;
  CHECK(p->f->size(&nl));
  if (static_cast<size_t>(nl) != x->word_off[x->rank + 1] - lo ||
      x->total_words != static_cast<size_t>(n))
    return rc(GrB_DIMENSION_MISMATCH);
  if (x->pr_vec[0] == NULL) {
    x->pr_vec[0] = new Vector<float>(static_cast<Index>(n));   // p_glob (view)
    x->pr_vec[1] = new Vector<float>(nl);                      // p_prev (view)
    for (int i = 2; i < 5; ++i) x->pr_vec[i] = new Vector<float>(nl);
  }
  Vector<float>* p_glob = x->pr_vec[0];
  Vector<float>* p_prev = x->pr_vec[1];
  Vector<float>* p_swap = x->pr_vec[2];
  Vector<float>* r      = x->pr_vec[3];
  Vector<float>* r_temp = x->pr_vec[4];

  CHECK(p->f->fill(1.f/static_cast<float>(n)));
  void* p_dev = NULL;
  if (gb200_vector_device_ptr(p, &p_dev) != 0) return rc(GrB_PANIC);
  double total = 0.0;
  int info_i = gb200_xchg_allgather_words(x, p_dev, 0.0, &total);
  if (info_i != 0) return info_i;

  Desc_value saved_mode;
  CHECK(d->get(GrB_MXVMODE, &saved_mode));
  CHECK(d->set(GrB_MXVMODE, GrB_PULLONLY));
  const int max_niter = d->descriptor_.max_niter_;
  float error = 1.f;
  int iter;
  Info info = GrB_SUCCESS;
  for (iter = 1; error > eps && iter <= max_niter; ++iter) {
    float* data = const_cast<float*>(
        reinterpret_cast<const float*>(gbx::current(x)));
    info = p_glob->build(data, static_cast<Index>(n));          if (info) break;
    info = p_prev->build(data + lo, nl);                        if (info) break;
    info = mxv<float, float, float, float>(p_swap, GrB_NULL, GrB_NULL,
        PlusMultipliesSemiring<float>(), M->f, p_glob, d);      if (info) break;
    info = eWiseAdd<float, float, float, float>(p->f, GrB_NULL, GrB_NULL,
        PlusMultipliesSemiring<float>(), p_swap,
        (1.f - alpha)/static_cast<float>(n), d);                if (info) break;
    info = eWiseMult<float, float, float, float>(r, GrB_NULL, GrB_NULL,
        PlusMinusSemiring<float>(), p->f, p_prev, d);           if (info) break;
    info = eWiseAdd<float, float, float, float>(r_temp, GrB_NULL, GrB_NULL,
        MultipliesMultipliesSemiring<float>(), r, r, d);        if (info) break;
    float partial = 0.f;
    info = reduce<float, float>(&partial, GrB_NULL, PlusMonoid<float>(), r_temp,
        d);                                                     if (info) break;
    if (gb200_vector_device_ptr(p, &p_dev) != 0) { info = GrB_PANIC; break; }
    if (gb200_xchg_allgather_words(x, p_dev, static_cast<double>(partial),
                                   &total) != 0) { info = GrB_PANIC; break; }
    error = static_cast<float>(sqrt(total));
  }
  d->set(GrB_MXVMODE, saved_mode);
  if (iters_out != NULL) *iters_out = iter - 1;
  return rc(info);
}

// SSSP over the 1-D row partition: the loop of reference
// graphblas/algorithm/sssp.hpp:46-99 on the owned slice.  The exchange carries one
// word per VERTEX (the frontier's float values, FLT_MAX = absent) and the number of
// improved vertices as the partial.  v (length nl) = owned distances (output);
// M = owned rows of A^T (weights A(i,j) at M(j,i)), (nl x n), CSR + CSC.  The
// direction of every round is chosen by mxv itself (GrB_PUSHPULL: frontier ratio,
// hysteresis and the edge-share check), exactly as on one GPU.
int gb200_dist_sssp(gb200_xchg_t x, gb200_vector_t v, gb200_matrix_t M,
                    long long n, long long source, gb200_desc_t desc,
                    int* rounds_out) {
  if (x == NULL || v == NULL || M == NULL || desc == NULL)
    return rc(graphblas::GrB_NULL_POINTER);
  if (!x->connected || M->f == NULL) return rc(graphblas::GrB_UNINITIALIZED_OBJECT);
  GB200_REQUIRE_DEVICE();
  using namespace graphblas;          // NOLINT(build/namespaces)
  Descriptor* d = &desc->desc;
  const float kInf = std::numeric_limits<float>::max();
  const size_t lo = x->word_off[x->rank];
  Index nl;
  CHECK(v->f->size(&nl));
  if (static_cast<size_t>(nl) != x->word_off[x->rank + 1] - lo ||
      x->total_words != static_cast<size_t>(n))
    return rc(GrB_DIMENSION_MISMATCH);
  if (x->ss_vec[0] == NULL) {
    x->ss_vec[0] = new Vector<float>(static_cast<Index>(n));   // frontier (view)
    x->ss_vec[1] = new Vector<float>(nl);                      // relaxed
    x->ss_vec[2] = new Vector<float>(nl);                      // improved
  }
  Vector<float>* frontier = x->ss_vec[0];
  Vector<float>* relaxed  = x->ss_vec[1];
  Vector<float>* improved = x->ss_vec[2];
  gb200_vector_s relaxed_h = {GB200_FP32, relaxed};

  const bool own_src = source >= static_cast<long long>(lo) &&
                       source < static_cast<long long>(lo) + nl;
  CHECK(v->f->fill(kInf));
  CHECK(relaxed->fill(kInf));
  if (own_src) {
    CHECK(v->f->setElement(0.f, static_cast<Index>(source - lo)));
    CHECK(relaxed->setElement(0.f, static_cast<Index>(source - lo)));
  }
  void* r_dev = NULL;
  if (gb200_vector_device_ptr(&relaxed_h, &r_dev) != 0) return rc(GrB_PANIC);
  double total = 0.0;
  int info_i = gb200_xchg_allgather_words(x, r_dev, own_src ? 1.0 : 0.0, &total);
  if (info_i != 0) return info_i;

  const int max_niter = d->descriptor_.max_niter_;
  const float switchpoint = d->descriptor_.switchpoint();
  bool  sparse_mode = true;     // the source frontier is built sparse
  float prev_ratio  = 0.f;
  Info info = GrB_SUCCESS;
  int round;
  for (round = 1; round <= max_niter && total > 0.0; ++round) {
    float* data = const_cast<float*>(
        reinterpret_cast<const float*>(gbx::current(x)));
    info = frontier->build(data, static_cast<Index>(n));          if (info) break;
    // The gathered frontier arrives dense every round; on one GPU it would still
    // be SPARSE while it is small (it is the sparse output of the previous push),
    // and mxv's own conversion rule only turns a dense vector sparse when it
    // shrinks.  Carry the storage state of reference vector.hpp:318-342 across
    // rounds here and hand mxv the storage the single-GPU loop would have had.
    const float ratio = static_cast<float>(total/static_cast<double>(n));
    if (sparse_mode) {
      if (ratio > switchpoint && ratio > prev_ratio) sparse_mode = false;
      else prev_ratio = ratio;
    } else {
      if (ratio <= switchpoint && ratio < prev_ratio) sparse_mode = true;
      else prev_ratio = ratio;
    }
    if (sparse_mode) {
      info = frontier->vector_.dense2sparse(kInf, &d->descriptor_); if (info) break;
    }
    info = mxv<float, float, float, float>(relaxed, GrB_NULL, GrB_NULL,
        MinimumPlusSemiring<float>(), M->f, frontier, d);         if (info) break;
    info = eWiseAdd<float, float, float, float>(improved, GrB_NULL, GrB_NULL,
        CustomLessPlusSemiring<float>(), relaxed, v->f, d);       if (info) break;
    info = eWiseAdd<float, float, float, float>(v->f, GrB_NULL, GrB_NULL,
        MinimumPlusSemiring<float>(), v->f, relaxed, d);          if (info) break;
    CHECK(d->toggle(GrB_MASK));
    info = assign<float, float, float, Index>(relaxed, improved, GrB_NULL, kInf,
        GrB_ALL, nl, d);
    CHECK(d->toggle(GrB_MASK));
    if (info) break;
    // Owned part of the next frontier: its entry count is this rank's partial (the
    // single-GPU loop stops on "frontier empty or nothing improved"; nothing
    // improved means every entry was just masked back to FLT_MAX, so the count
    // covers both), its values go out as a dense float slice.
    Index cnt = 0;
    Storage r_type;
    CHECK(relaxed->vector_.getStorage(&r_type));
    if (r_type == GrB_SPARSE) {
      CHECK(relaxed->vector_.sparse_.nvals(&cnt));
      info = relaxed->vector_.sparse2dense(kInf, &d->descriptor_); if (info) break;
    } else {
      info = relaxed->vector_.dense_.computeNnz(&cnt, kInf, &d->descriptor_);
      if (info) break;
    }
    if (gb200_vector_device_ptr(&relaxed_h, &r_dev) != 0) { info = GrB_PANIC; break; }
    if (gb200_xchg_allgather_words(x, r_dev, static_cast<double>(cnt),
                                   &total) != 0) { info = GrB_PANIC; break; }
  }
  if (rounds_out != NULL) *rounds_out = round - 1;
  return rc(info);
}

}  // extern "C"

#endif  // GRAPHBLAST_B200_DIST_EXCHANGE_CUH_
