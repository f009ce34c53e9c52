/* graphblast_b200.h — C ABI of the B200-native GraphBLAS backend.
 *
 * The reference (gunrock/graphblast) is a header-only C++ template library with
 * no FFI of its own: its "plugin boundary" for this path is the compile-time
 * backend dispatch (graphblas/backend.hpp:4-15 -> graphblas/backend/cuda/), which
 * this repository replaces directory-for-directory (graphblast_b200/csrc/graphblas/
 * backend/cuda/, see INTEGRATION.md).  This C ABI is what a foreign-language
 * binding of the SAME path binds: every entry point is a thin extern "C" shim
 * over one frontend template of reference graphblas/operations.hpp or one method
 * of graphblas::{Matrix,Vector,Descriptor}, instantiated for the value types the
 * reference drivers use (float vectors/matrices; int matrices for triangle
 * counting) and for the 17 named semirings / 9 monoids of
 * reference graphblas/stddef.hpp:160-213.
 *
 * Conventions
 *   - every function returns a graphblas::Info code (0 = GrB_SUCCESS; values as in
 *     reference graphblas/types.hpp:30-44);
 *   - "h_" arguments are HOST pointers, "d_" arguments are DEVICE pointers;
 *     adopted device memory stays owned by the caller and must outlive the object;
 *   - no CPU fallback exists: without a CUDA device every compute entry fails.
 */
#ifndef GRAPHBLAST_B200_H_
#define GRAPHBLAST_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* The library is built with -fvisibility=hidden; only this ABI is exported. */
#pragma GCC visibility push(default)

typedef struct gb200_matrix_s* gb200_matrix_t;
typedef struct gb200_vector_s* gb200_vector_t;
typedef struct gb200_desc_s*   gb200_desc_t;

/* Value types. */
enum { GB200_FP32 = 0, GB200_INT32 = 1 };

/* Storage tags (reference graphblas/types.hpp:21-23). */
enum { GB200_UNKNOWN = 0, GB200_SPARSE = 1, GB200_DENSE = 2 };

/* Descriptor fields / values (reference graphblas/types.hpp:46-78). */
enum { GB200_MASK = 0, GB200_OUTP, GB200_INP0, GB200_INP1, GB200_MODE, GB200_TA,
       GB200_TB, GB200_NT, GB200_MXVMODE, GB200_TOL, GB200_BACKEND };
enum { GB200_SCMP = 0, GB200_REPLACE = 1, GB200_TRAN = 2, GB200_DEFAULT = 3,
       GB200_PUSHPULL = 10, GB200_PUSHONLY = 11, GB200_PULLONLY = 12,
       GB200_SEQUENTIAL = 13, GB200_CUDA = 14 };

/* Semirings, in REGISTER_SEMIRING order (reference graphblas/stddef.hpp:194-213). */
enum {
  GB200_LOGICAL_OR_AND = 0, GB200_PLUS_MULTIPLIES, GB200_MINIMUM_PLUS,
  GB200_MAXIMUM_MULTIPLIES, GB200_PLUS_DIVIDES, GB200_PLUS_GREATER,
  GB200_GREATER_PLUS, GB200_PLUS_MINUS, GB200_PLUS_LESS,
  GB200_CUSTOM_LESS_PLUS, GB200_MINIMUM_MULTIPLIES,
  GB200_MULTIPLIES_MULTIPLIES, GB200_NOT_EQUAL_TO_PLUS,
  GB200_MINIMUM_SELECT_SECOND, GB200_PLUS_NOT_EQUAL_TO,
  GB200_CUSTOM_LESS_LESS, GB200_MINIMUM_NOT_EQUAL_TO, GB200_NSEMIRINGS
};

/* Monoids, in REGISTER_MONOID order (reference graphblas/stddef.hpp:160-173). */
enum {
  GB200_PLUS_MONOID = 0, GB200_MULTIPLIES_MONOID, GB200_MINIMUM_MONOID,
  GB200_MAXIMUM_MONOID, GB200_LOGICAL_OR_MONOID, GB200_LOGICAL_AND_MONOID,
  GB200_GREATER_MONOID, GB200_CUSTOM_LESS_MONOID, GB200_NOT_EQUAL_TO_MONOID,
  GB200_NMONOIDS
};

/* ---- runtime ---------------------------------------------------------- */
/* Binds the calling process to `device` (one process per GPU) and creates the
 * backend runtime.  No reference counterpart (the reference uses device 0 and the
 * default stream, backend/cuda/descriptor.hpp:283-284 "TODO: Enable device selection"). */
int gb200_init(int device);
/* All backend kernels and copies are issued on `cuda_stream` (a cudaStream_t). */
int gb200_set_stream(void* cuda_stream);
int gb200_sync(void);
int gb200_sm_count(int* out);
const char* gb200_version(void);

/* ---- Descriptor: reference graphblas/descriptor.hpp:17-62 --------------- */
int gb200_desc_new(gb200_desc_t* out);
int gb200_desc_free(gb200_desc_t desc);
int gb200_desc_set(gb200_desc_t desc, int field, int value);       /* Descriptor::set   :41-47 */
int gb200_desc_get(gb200_desc_t desc, int field, int* value);      /* Descriptor::get   :49-52 */
int gb200_desc_toggle(gb200_desc_t desc, int field);               /* Descriptor::toggle:54-56 */
/* Named knobs = the command-line flags Descriptor::loadArgs reads
 * (reference backend/cuda/descriptor.hpp:207-287, graphblas/util.hpp:39-132):
 * "mxvmode" "switchpoint" "struconly" "opreuse" "earlyexit" "fusedmask" "sort"
 * "dirinfo" "debug" "timing" "max_niter" "memusage" "nthread".
 * gb200_desc_new() starts from the flag defaults of parseArgs. */
int gb200_desc_set_knob(gb200_desc_t desc, const char* name, double value);
int gb200_desc_get_knob(gb200_desc_t desc, const char* name, double* value);  /* + "lastmxv" */

/* ---- Matrix: reference graphblas/matrix.hpp:14-252 ---------------------- */
int gb200_matrix_new(gb200_matrix_t* out, int dtype, int nrows, int ncols);   /* Matrix(nrows,ncols) :20 */
int gb200_matrix_free(gb200_matrix_t A);
/* Matrix::build from host COO triples (:125-144): the triples are uploaded and
 * ordered into CSR + CSC on the device.  `undirected` plays the role of the ".ud."
 * cache name (structurally symmetric: CSC index arrays alias CSR on the device). */
int gb200_matrix_build_coo(gb200_matrix_t A, const int* h_rows, const int* h_cols,
                           const void* h_vals, int nvals, int undirected);
/* readMtx + Matrix::build, the loader path of every reference driver
 * (graphblas/util.hpp:364-430; example/gbfs.cu:57-69).  directed: 0/1/2.  The file
 * is parsed on the host; symmetrising, ordering and the removal of self-loops and
 * repeated entries run on the device with the loader's semantics. */
int gb200_matrix_load_mtx(gb200_matrix_t* out, int dtype, const char* path,
                          int directed);
/* ---- graph ingest on the device (no reference counterpart: the reference sorts
 * tuple vectors on the host, graphblas/util.hpp:170-195, 264-329, 502-600) --------
 * flags: the GB200_INGEST_* bits. */
#define GB200_INGEST_SYMMETRIZE          1   /* add (col,row) of every non-loop tuple */
#define GB200_INGEST_DROP_LOOPS          2   /* drop row == col */
#define GB200_INGEST_DEDUP               4   /* keep the first of equal (row,col) */
#define GB200_INGEST_SYMMETRIC_STRUCTURE 8   /* result is structurally symmetric:
                                                CSC index arrays alias the CSR */
/* Builds A (CSR + CSC, owned by A) from tuples in DEVICE memory; d_vals may be
 * NULL (value 1) and has A's element type otherwise. */
int gb200_matrix_build_coo_device(gb200_matrix_t A, const int* d_rows,
                                  const int* d_cols, const void* d_vals,
                                  long long ntuples, int flags);
/* Tuples -> sorted CSR held by the library; *nnz says how much room
 * gb200_ingest_export needs (d_rowptr[nrows+1], d_colind[nnz], d_val[nnz], any
 * of them NULL to skip). */
typedef struct gb200_ingest_s* gb200_ingest_t;
int gb200_ingest_coo(int nrows, int ncols, const int* d_rows, const int* d_cols,
                     const float* d_vals, long long ntuples, int flags,
                     gb200_ingest_t* out, long long* nnz);
int gb200_ingest_export(gb200_ingest_t h, int* d_rowptr, int* d_colind, float* d_val);
int gb200_ingest_free(gb200_ingest_t h);
/* CSC of a device CSR (csr2csc, reference graphblas/util.hpp:580-600); output
 * pointers may be NULL to skip that array. */
int gb200_csr_transpose_values(int nrows, int ncols, int nnz, const int* d_rowptr,
                               const int* d_colind, const float* d_val,
                               int* d_colptr_out, int* d_rowind_out,
                               float* d_cscval_out);
/* Stable LSD radix sort of 64-bit keys by their low `bits` bits, with an optional
 * 32-bit payload, in place (the sort the ingest is built on; exported for tests). */
int gb200_sort_pairs_u64(unsigned long long* d_keys, unsigned int* d_payload,
                         long long n, int bits);
/* Matrix::build(Index* row_ptr, Index* col_ind, T* values, Index nvals) (:152-161):
 * adopts DEVICE CSR arrays. */
int gb200_matrix_adopt_csr(gb200_matrix_t A, int* d_rowptr, int* d_colind,
                           void* d_val, int nvals);
/* Device CSC for the adopted matrix (no reference counterpart: the reference can
 * only adopt CSR).  symmetric != 0 with NULL index pointers aliases the CSR;
 * d_val == NULL makes an owned copy of the CSR values. */
int gb200_matrix_adopt_csc(gb200_matrix_t A, int* d_colptr, int* d_rowind,
                           void* d_val, int symmetric);
int gb200_matrix_nrows(gb200_matrix_t A, int* out);                 /* :104-108 */
int gb200_matrix_ncols(gb200_matrix_t A, int* out);                 /* :111-115 */
int gb200_matrix_nvals(gb200_matrix_t A, int* out);                 /* :118-122 */
/* Host copy of the CSR (what the reference CPU verifiers read,
 * algorithm/bfs.hpp:101-107).  Buffers: nrows+1, nvals, nvals. */
int gb200_matrix_extract_csr(gb200_matrix_t A, int* h_rowptr, int* h_colind,
                             void* h_val);
/* tril(A, A) under GrB_BACKEND = GrB_SEQUENTIAL (operations.hpp:872-886,
 * example/gtc.cu:80-82). */
int gb200_matrix_tril(gb200_matrix_t A, gb200_desc_t desc);
/* apply(A, set_uniform_random) under GrB_SEQUENTIAL (example/gsssp.cu:75-84,
 * algorithm/common.hpp:22-42): CSR-order draws of uniform_int[lo,hi] from
 * std::default_random_engine(seed). */
int gb200_matrix_apply_uniform_random(gb200_matrix_t A, gb200_desc_t desc,
                                      int seed, int lo, int hi);
/* The same random stream into a host array (no device needed). */
int gb200_host_uniform_weights(int seed, int lo, int hi, long long n, float* h_out);
/* A = alpha * A ./ rowsum(A): reduce + 2 x eWiseMult of example/gpr.cu:76-86. */
int gb200_pr_normalize(gb200_matrix_t A, float alpha, gb200_desc_t desc);

/* ---- Vector: reference graphblas/vector.hpp:13-264 ----------------------- */
int gb200_vector_new(gb200_vector_t* out, int dtype, int size);      /* Vector(nsize) :16 */
int gb200_vector_free(gb200_vector_t v);
int gb200_vector_fill(gb200_vector_t v, double val);                 /* fill :216-218 */
int gb200_vector_build_sparse(gb200_vector_t v, const int* h_ind,
                              const void* h_val, int nvals);         /* build(indices,values) :98-105 */
int gb200_vector_build_dense(gb200_vector_t v, const void* h_val, int n); /* build(values) :108-112 */
int gb200_vector_adopt_dense(gb200_vector_t v, void* d_val, int n);  /* build(T*,nvals) :125-130 */
int gb200_vector_adopt_sparse(gb200_vector_t v, int* d_ind, void* d_val,
                              int nvals);                            /* build(Index*,T*,nvals) :115-122 */
int gb200_vector_set_element(gb200_vector_t v, double val, int index);  /* :133-135 */
int gb200_vector_size(gb200_vector_t v, int* out);                   /* :82-86 */
int gb200_vector_nvals(gb200_vector_t v, int* out);                  /* :89-93 */
int gb200_vector_storage(gb200_vector_t v, int* out);                /* getStorage :243-246 */
/* extractTuples(values, n) (:154-158): a sparse vector is densified with 0. */
int gb200_vector_extract_dense(gb200_vector_t v, void* h_out, int n);
/* extractTuples(indices, values, n) (:145-151); *n_inout = capacity in, count out. */
int gb200_vector_extract_sparse(gb200_vector_t v, int* h_ind, void* h_val,
                                int* n_inout);
int gb200_vector_swap(gb200_vector_t a, gb200_vector_t b);           /* :259-262 */
int gb200_vector_dup(gb200_vector_t dst, gb200_vector_t src);        /* :71-73 */
int gb200_vector_clear(gb200_vector_t v);                            /* :76-78 */
int gb200_vector_sparse2dense(gb200_vector_t v, double identity, gb200_desc_t desc); /* :249-251 */
int gb200_vector_dense2sparse(gb200_vector_t v, double identity, gb200_desc_t desc); /* :254-256 */
/* Device address of the dense value array (valid while storage is dense). */
int gb200_vector_device_ptr(gb200_vector_t v, void** d_val);

/* ---- Operations: reference graphblas/operations.hpp ---------------------- */
/* mask may be NULL; use_accum != 0 passes a non-NULL accum (the reference then
 * accumulates with the semiring's ADD, backend/cuda/spmv.hpp:213-219). */
int gb200_vxm(gb200_vector_t w, gb200_vector_t mask, int use_accum, int semiring,
              gb200_vector_t u, gb200_matrix_t A, gb200_desc_t desc);      /* vxm :59-87 */
int gb200_mxv(gb200_vector_t w, gb200_vector_t mask, int use_accum, int semiring,
              gb200_matrix_t A, gb200_vector_t u, gb200_desc_t desc);      /* mxv :97-127 */
/* INT32 matrices, PlusMultiplies<int> (the triangle-counting instantiation). */
int gb200_mxm(gb200_matrix_t C, gb200_matrix_t mask, int semiring,
              gb200_matrix_t A, gb200_matrix_t B, gb200_desc_t desc);      /* mxm :22-49 */
int gb200_ewise_add(gb200_vector_t w, gb200_vector_t mask, int semiring,
                    gb200_vector_t u, gb200_vector_t v, gb200_desc_t desc); /* :277-299 */
int gb200_ewise_add_scalar(gb200_vector_t w, gb200_vector_t mask, int semiring,
                           gb200_vector_t u, double val, gb200_desc_t desc); /* :333-353 */
int gb200_ewise_mult(gb200_vector_t w, gb200_vector_t mask, int semiring,
                     gb200_vector_t u, gb200_vector_t v, gb200_desc_t desc); /* :137-158 */
/* assign(w, mask, GrB_NULL, val, GrB_ALL, size, desc) :509-530 */
int gb200_assign_scalar(gb200_vector_t w, gb200_vector_t mask, double val,
                        gb200_desc_t desc);
int gb200_reduce_vector(double* out, int monoid, gb200_vector_t u,
                        gb200_desc_t desc);                                 /* :640-653 */
int gb200_reduce_matrix(double* out, int monoid, gb200_matrix_t A,
                        gb200_desc_t desc);                                 /* :660-673 */
int gb200_reduce_matrix_rows(gb200_vector_t w, int monoid, gb200_matrix_t A,
                             gb200_desc_t desc);                            /* :620-633 */

/* ---- Algorithms: reference graphblas/algorithm/{bfs,sssp,pr,tc}.hpp ------ */
/* tight_ms receives the device time of the operation loop ("tight" in the
 * reference drivers, example/gbfs.cu:110-115). */
int gb200_bfs(gb200_vector_t v, gb200_matrix_t A, int source, gb200_desc_t desc,
              float* tight_ms);                                 /* algorithm/bfs.hpp:14-89 */
/* scatter (reference graphblas/operations.hpp:771): w[(int)u[i]] = val for every stored
 * value of u with 0 < (int)u[i] < size; assignScatter (:806): w[(int)ind[i]] = u[i];
 * extractGather (:839): w[i] = u[(int)ind[i]].  Dense float vectors. */
int gb200_scatter(gb200_vector_t w, gb200_vector_t u, float val, gb200_desc_t desc);
int gb200_assign_scatter(gb200_vector_t w, gb200_vector_t u, gb200_vector_t indices,
                         gb200_desc_t desc);
int gb200_extract_gather(gb200_vector_t w, gb200_vector_t u, gb200_vector_t indices,
                         gb200_desc_t desc);
/* Work counters of the last BFS that ran as the fused kernel with this descriptor:
 * levels, colind entries inspected while pulling, pull levels, frontier entries
 * pushed, edges pushed, vertices discovered while pushing (all zero if the
 * traversal ran operation by operation). */
int gb200_bfs_stats(gb200_desc_t desc, int n, unsigned long long* out6);
int gb200_sssp(gb200_vector_t v, gb200_matrix_t A, int source, gb200_desc_t desc,
               float* tight_ms);                                /* algorithm/sssp.hpp:15-103 */
int gb200_pr(gb200_vector_t p, gb200_matrix_t A, float alpha, float eps,
             gb200_desc_t desc, float* tight_ms);               /* algorithm/pr.hpp:15-94 */
int gb200_tc(long long* ntris, gb200_matrix_t A, gb200_matrix_t B,
             gb200_desc_t desc, float* tight_ms);               /* algorithm/tc.hpp:15-54 */

/* ---- Frontier exchange helpers for the 1-D row-partitioned multi-GPU path ----
 * (SURVEY.md §8e; the reference has no distributed path.)  A Boolean frontier
 * travels between ranks as a bitmap, n/8 bytes for n vertices. */
/* Bitmap (bit == value != 0) of v into DEVICE words d_bits[(size+31)/32]; works
 * for dense and sparse storage.  count_out (may be NULL) receives the popcount. */
int gb200_vector_export_bits(gb200_vector_t v, uint32_t* d_bits, long long* count_out);
/* Same, without any host synchronisation: the 64-bit popcount is written on the
 * device into d_count (8-byte aligned DEVICE address), e.g. the tail of the
 * record a rank contributes to the frontier all-gather. */
int gb200_vector_export_bits_async(gb200_vector_t v, uint32_t* d_bits,
                                   unsigned long long* d_count);
/* v becomes a dense 0/1 vector with the given bitmap (DEVICE words).
 * nnz >= 0 tells the number of set bits (saves the counting pass of the next
 * direction decision); pass -1 when unknown. */
int gb200_vector_import_bits(gb200_vector_t v, const uint32_t* d_bits, long long nnz);

/* ---- Measurement hooks (bench.py; no reference counterpart) --------------- */
/* Hot-kernel kinds: 0 merge-path SpMV (pull, generic semiring), 1 fused Boolean
 * pull, 2 push (SpMSpV expand), 3 masked SpGEMM.  When enabled every launch of
 * those kernels is bracketed by CUDA events on the launching stream. */
int gb200_profile_enable(int on);
int gb200_profile_reset(void);
/* Sum over the launches since the last reset: device milliseconds, launch count
 * and ALGORITHMIC bytes (SURVEY.md §8d definitions). */
int gb200_profile_read(int kind, double* ms, long long* launches, double* bytes);
/* Number of kernels this library has launched so far. */
int gb200_launch_count(unsigned long long* out);

/* ---- Graph ingest helpers (SURVEY.md §8f-1; ours, no reference counterpart) */
/* R-MAT (0.57,0.19,0.19,0.05) edges [first_edge, first_edge+nedges) into DEVICE
 * arrays; bit-identical to oracle/gb_oracle.c:orc_rmat_edges. */
int gb200_rmat_edges(int scale, long long nedges, unsigned long long seed,
                     long long first_edge, int* d_src, int* d_dst);

/* ---- Multi-GPU: frontier exchange over peer memory (SURVEY.md §8e) ----------
 * One process per GPU.  Each rank creates an exchange over the same partition of
 * the replicated bitmap (word_offsets[world+1], in 32-bit words; rank r owns words
 * [word_offsets[r], word_offsets[r+1])), passes its 64-byte IPC handle to every
 * other rank by any host channel (torch.distributed, MPI, a file), and connects.
 * After that the exchange needs no host library: the owner's kernel stores its
 * slice, count and epoch flag directly into every peer's copy over NVLink.
 * The reference has no multi-GPU code; this is the frontier all-gather that
 * BASELINE.json's north_star asks for after each mxv. */
typedef struct gb200_xchg_s* gb200_xchg_t;
int gb200_xchg_create(gb200_xchg_t* out, int world, int rank,
                      const long long* word_offsets);
int gb200_xchg_handle(gb200_xchg_t x, void* out64);
int gb200_xchg_connect(gb200_xchg_t x, const void* handles /* world x 64 bytes */);
int gb200_xchg_free(gb200_xchg_t x);
/* Publishes the owned slice (vector of the owned length, dense or sparse) and
 * waits for all ranks; *total_out = global number of entries. */
int gb200_xchg_allgather_bits(gb200_xchg_t x, gb200_vector_t v,
                              long long* total_out);
/* DEVICE pointer to the replicated bitmap of the last completed exchange. */
int gb200_xchg_bits_ptr(gb200_xchg_t x, const uint32_t** d_bits);
/* Level-synchronous BFS over the 1-D row partition as ONE persistent cooperative
 * kernel per GPU: level loop, direction decision, peer-memory exchange of the
 * frontier slice and the cross-GPU level barrier all on the device
 * (csrc/dist_bfs_fused.cuh).  v_own = levels of the owned vertices (length = owned
 * rows of M_local), M_local = the owned rows of A^T as an (owned x n) matrix with
 * CSR and CSC.  Collective: every rank calls it with the same n and source. */
int gb200_dist_bfs_fused(gb200_xchg_t x, gb200_vector_t v_own, gb200_matrix_t M_local,
                         long long n, long long source, gb200_desc_t desc,
                         int* levels_out);

/* Same exchange for 32-bit payloads (float vectors: create the exchange with one
 * word per vertex).  Publishes the owned words from DEVICE memory together with
 * this rank's partial scalar; *sum_out = the ranks' partials added in rank order
 * (identical on every rank). */
int gb200_xchg_allgather_words(gb200_xchg_t x, const void* d_words,
                               double partial, double* sum_out);
/* PageRank over the 1-D row partition: the loop of reference
 * graphblas/algorithm/pr.hpp:50-84 on the owned slice, p exchanged through peer
 * memory after every mxv.  p = owned ranks (length = owned rows of M); M = owned
 * rows of (alpha * A ./ outdeg)^T, (owned x n), CSR.  Runs until the global
 * residual norm <= eps or desc max_niter iterations. */
int gb200_dist_pr(gb200_xchg_t x, gb200_vector_t p, gb200_matrix_t M,
                  long long n, float alpha, float eps, gb200_desc_t desc,
                  int* iters_out);

/* SSSP over the 1-D row partition: the loop of reference
 * graphblas/algorithm/sssp.hpp:46-99 on the owned slice; frontier values (floats,
 * one word per vertex) and the number of improved vertices exchanged per round.
 * v = owned distances (FLT_MAX = unreachable); M = owned rows of A^T (owned x n,
 * CSR + CSC, weights).  Runs until no vertex improves or desc max_niter rounds. */
int gb200_dist_sssp(gb200_xchg_t x, gb200_vector_t v, gb200_matrix_t M,
                    long long n, long long source, gb200_desc_t desc,
                    int* rounds_out);

#pragma GCC visibility pop

#ifdef __cplusplus
}
#endif

#endif  /* GRAPHBLAST_B200_H_ */
