/*
 * bof_b200.h -- C ABI of the B200-native replacement for BLAS-on-Flash's tiled hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, `extern "C"`, no C++/torch types.
 * Every entry point names the reference interface it replaces (paths relative to the
 * reference tree, microsoft/BLAS-on-flash).  Three groups:
 *
 *   1. context / diagnostics
 *   2. device-tile kernels: operands already in HBM; `stream` is a cudaStream_t passed as void*
 *      (replace the per-tile `BaseTask::execute()` bodies, include/tasks/<task>.h, i.e. the MKL calls)
 *   3. host entry points: operands in host memory (pageable, pinned or a file mmap, i.e. the
 *      `flash_ptr<T>::ptr` of include/pointers/pointer.h:15-27); the library streams them through
 *      pinned staging buffers and CUDA streams (replace src/scheduler/ + src/file_handles/ for
 *      this path) and the result is in the host buffer when the call returns
 *      (reference contract: Scheduler::flush_cache() at kernel end, src/blas/gemm.cpp:200).
 *
 * Conventions
 *   - return value: 0 on success, negative on failure (BOF_E*), message via bof_last_error().
 *     The reference returns FBLAS_INT 0 / -1 (src/blas/csrmm.cpp:433-449); the C++ adapters in
 *     include/flash_blas.h map any negative code to -1.
 *   - fp32 values; CSR offsets are int64 (MKL_INT under ILP64, CMakeLists.txt:104); CSR column
 *     indices are int32 on the device (narrowed while staging) and int64 on the host/file side.
 *   - one call at a time per context (reference: Cache::flush asserts no active buffers,
 *     src/scheduler/cache.cpp:45-47).
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     BOF_ENODEV.
 */
#ifndef BOF_B200_H_
#define BOF_B200_H_

#include <stddef.h>
#include <stdint.h>

/* Every entry point is exported explicitly; the library itself is built with -fvisibility=hidden so that nothing
 * but this ABI leaves it. */
#if defined(__GNUC__)
#define BOF_API __attribute__((visibility("default")))
#else
#define BOF_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define BOF_OK 0
#define BOF_EINVAL (-1)  /* bad argument (reference: return -1 on bad char, csrmm.cpp:433-449) */
#define BOF_ECUDA (-2)   /* CUDA runtime/driver error */
#define BOF_ENOMEM (-3)  /* device or pinned allocation failed */
#define BOF_ENODEV (-4)  /* no CUDA device / wrong architecture */
#define BOF_EIO (-5)     /* host I/O failure */

typedef struct bof_ctx bof_ctx;

/* Runtime knobs.  Defaults mirror the reference's compile-time macros (CMakeLists.txt:38-63)
 * where a counterpart exists.  Zero in any field selects the default. */
typedef struct bof_config {
  int32_t device;            /* CUDA ordinal this context drives (one context per GPU/process)  */
  int32_t n_copy_threads;    /* host staging threads (reference N_IO_THR=4; default 8)          */
  uint64_t stage_bytes;      /* bytes per pinned staging buffer (default 16 MiB)                */
  int32_t n_stage_bufs;      /* pinned ring depth per direction (default 4)                     */
  uint64_t csrmm_max_nnz;    /* nnz budget per streamed CSR row block (reference MAX_NNZS=1e7;
                                default here 64 Mi so that a block amortises launch latency)    */
  uint64_t gemm_row_block;   /* rows of A/C per streamed GEMM block (reference GEMM_BLK_SIZE=8192)*/
  int32_t gemm_k_chunk;      /* k-extent accumulated inside the tensor core before the fp32
                                round-to-nearest fold (0 = default 256; <0 = whole k)           */
  int32_t gemm_force_path;   /* 0 auto, 1 tcgen05 1-CTA, 2 tcgen05 2-CTA, 3 CUDA-core FFMA      */
  int32_t gemm_wave_sync;    /* k-blocks (of 32) between wave lock-step points of the GEMM
                                kernel: 0 = default 64, <0 = off                                */
  int32_t gemm_split;        /* operand split of the fp32 GEMM: 0 = default, 1 = 3xTF32 (lo*hi + hi*lo +
                                hi*hi, all kind::tf32), 2 = hybrid (hi*hi kind::tf32, the two cross
                                terms on bf16 copies, kind::f16: 2/3 of the tensor time, cross-term
                                error <= 2^-19 relative).  With 1, an infinite input may give NaN
                                instead of +-Inf in its own row and column of C (hi*lo = Inf * 0 where
                                the partner is tf32-exact); other elements are unaffected.        */
  int32_t radix_max_bits;    /* digit width of the csrcsc / k-means radix passes: 0 = default 8; smaller values
                                force more passes (test knob)                                            */
  int32_t spmv_t_atomic;     /* csrgemv 'T': 0 = default, deterministic (products sorted by column, fixed-order sums,
                                no atomics); 1 = scatter with red.global.add.f32 (5x faster on the device, the
                                order of the additions -- like the reference's mutex'd adds -- is not fixed)  */
} bof_config;

/* Per-stage accounting of the last host entry point, for the out-of-core roofline
 * (no reference counterpart; the reference only logs wall time, drivers/csrmm.cpp:62-65). */
typedef struct bof_stats {
  double h2d_bytes, d2h_bytes;      /* bytes that crossed PCIe                                  */
  double h2d_ms, d2h_ms;            /* reserved (0 in this version)                             */
  double kernel_ms;                 /* CUDA-event time of the most recent tensor-core GEMM kernel */
  double stage_in_ms, stage_out_ms; /* host memcpy pageable<->pinned (wall, summed over threads)*/
  double total_ms;                  /* wall time of the call                                    */
  int64_t kernel_launches;          /* number of this library's kernels launched                */
} bof_stats;

/* ---- 1. context ----------------------------------------------------------------------- */

/* Replaces the static `flash::sched` + flash_setup() (src/lib_funcs.cpp:9,18-23). */
BOF_API int bof_ctx_create(const bof_config* cfg, bof_ctx** out);
BOF_API int bof_ctx_destroy(bof_ctx* ctx);
/* Message of the last failure on this context (ctx may be NULL: last failure of ctx creation). */
BOF_API const char* bof_last_error(const bof_ctx* ctx);
BOF_API int bof_get_stats(const bof_ctx* ctx, bof_stats* out);
/* Total kernels launched by this context since creation (bench.py's gpu_launches). */
BOF_API int64_t bof_launch_count(const bof_ctx* ctx);
/* Tell the library that host range [base, base+len) is the mmap of descriptor `fd` starting at byte
 * `file_offset` (what map_file() creates, include/pointers/allocator.h:19-45).  With BOF_STAGE_FD=1 in the
 * environment host entry points move such operands with pread/pwrite into their pinned staging buffers --
 * the reference's FlashFileHandle::read/write into cache buffers (src/file_handles/flash_file_handle.cpp:
 * 247-407) -- which pays off for cold files on real disks; by default they copy through the mapping, the
 * faster way for page-cache-resident files (measured).  Process-wide; include/pointers/allocator.h calls it. */
BOF_API int bof_register_mapping(const void* base, size_t len, int fd, uint64_t file_offset);
BOF_API int bof_unregister_mapping(const void* base);
/* ABI version, bumped on any signature change. */
BOF_API int bof_abi_version(void);

/* ---- 2. device-tile kernels ------------------------------------------------------------ */

/* K1/K2: C = alpha * A * B + beta * C, A in CSR (m x n), B n x k, C m x k.
 * Replaces mkl_scsrmm in SimpleCsrmmRmTask::execute (include/tasks/csrmm_task.h:219-228,
 * ord='R': row-major, 0-based) and SimpleCsrmmCmTask::execute (:290-312, ord='C': column-major;
 * indices stay 0-based here, the reference's in-place +1 is an MKL calling convention).
 * beta == 0 => C is not read (csrmm_task.h:194-196).  `offs` may be un-rebased (offs[0] != 0):
 * vals/idx are indexed by offs[i] - offs[0].  ord='C' needs workspace
 * bof_spmm_workspace_bytes(); ord='R' needs none. */
BOF_API int bof_spmm_csr_f32(bof_ctx* ctx, void* stream, char ord, int64_t m, int64_t n, int64_t k,
                     float alpha, const float* vals, const int32_t* idx, const int64_t* offs,
                     const float* B, int64_t ldb, float beta, float* C, int64_t ldc,
                     void* workspace, size_t workspace_bytes);
BOF_API size_t bof_spmm_workspace_bytes(char ord, int64_t m, int64_t n, int64_t k);

/* K4/K5: y = op(A) x, y overwritten (no alpha/beta).
 * Replaces mkl_cspblas_scsrgemv in CsrGemvNoTransInMem::execute
 * (include/tasks/csrgemv_task.h:60-83) and CsrGemvTransInMem::execute (:152-179; the mutex'd
 * `out[i] += v_out[i]` in task-completion order becomes a deterministic sort-by-column + ordered column sums, or
 * red.global.add.f32 with bof_config.spmv_t_atomic).  trans='N': x has n entries, y has m;
 * trans='T': x has m entries, y has n and is overwritten (src/blas/csrgemv.cpp:64); it synchronises the stream once
 * to read nnz from `offs` and takes its workspace from the context. */
BOF_API int bof_spmv_csr_f32(bof_ctx* ctx, void* stream, char trans, int64_t m, int64_t n,
                     const float* vals, const int32_t* idx, const int64_t* offs, const float* x,
                     float* y);

/* Index staging helpers: int64 (file format, misc/sparse_create.cpp:63-81) <-> int32 (device). */
BOF_API int bof_idx_narrow(bof_ctx* ctx, void* stream, const int64_t* in, int32_t* out, int64_t count);
BOF_API int bof_idx_widen(bof_ctx* ctx, void* stream, const int32_t* in, int64_t* out, int64_t count);

/* K3: C = alpha * op(A) * op(B) + beta * C, fp32 in/out, 3xTF32 on tcgen05 tensor cores.
 * Replaces cblas_sgemm in GemmTask::execute (include/tasks/gemm_task.h:67-93); argument meaning
 * as flash::gemm (include/flash_blas.h:14-18): ord 'R'/'C', ta/tb 'N'/'T', ld* = 0 => tight
 * (src/blas/gemm.cpp:63-67).  beta == 0 => C is not read (gemm_task.h:49-53).
 * Special values follow IEEE as cblas_sgemm does: an Inf or NaN in A, B or (beta != 0) C gives the Inf / NaN of
 * the exact dot product in the elements it meets and leaves every other element unchanged (gemm_split = 1: see
 * bof_config.gemm_split).  Finite inputs up to FLT_MAX keep the fp32 accuracy as long as the products are finite.
 * Needs workspace of bof_sgemm_workspace_bytes(m, n, k) bytes (the TF32 hi/lo operand planes). */
BOF_API int bof_sgemm_f32(bof_ctx* ctx, void* stream, char ord, char ta, char tb, int64_t m, int64_t n,
                  int64_t k, float alpha, const float* A, int64_t lda, const float* B,
                  int64_t ldb, float beta, float* C, int64_t ldc, void* workspace,
                  size_t workspace_bytes);
BOF_API size_t bof_sgemm_workspace_bytes(int64_t m, int64_t n, int64_t k);
/* Measurement aid (no reference counterpart): what the tensor pipe sustains for this library's own MMA instructions,
 * issued back to back by every CTA pair on one resident shared-memory stage (no TMA, no epilogue).  kind 0 =
 * kind::tf32, 1 = kind::f16 on bf16, 2 = the hybrid mix of the product kernel.  *mma_tflops counts 2*M*N*K per MMA,
 * *useful_tflops counts the fp32-equivalent flops of the mix (kind 2: one third of the MMA work).  Synchronises. */
BOF_API int bof_tc_issue_rate(bof_ctx* ctx, void* stream, int kind, int rounds, double* mma_tflops,
                      double* useful_tflops);

/* K6/K7: stable CSR -> CSC (A m x n  ->  A^T as CSR n x m): per output row ascending source
 * row, duplicates in storage order.  Replaces mkl_scsrcsc + index rebase in
 * BlockCsrCscTask::execute (include/tasks/csrcsc_task.h:42-92) and the row-block-ordered merge
 * BlockMergeTask::execute (:136-163).  Atomic-free: radix passes of histogram -> scan -> ranked
 * scatter.  offs/offs_t int64, idx/idx_t int32.  nnz = offs[m] - offs[0] must be < 2^31. */
BOF_API int bof_csr2csc(bof_ctx* ctx, void* stream, int64_t m, int64_t n, int64_t nnz,
                const int64_t* offs, const int32_t* idx, const float* vals, int64_t* offs_t,
                int32_t* idx_t, float* vals_t, void* workspace, size_t workspace_bytes);
BOF_API size_t bof_csr2csc_workspace_bytes(int64_t m, int64_t n, int64_t nnz);

/* K11: out[r] = sum_j X[r, j]^2 for a row-major rows x dim matrix.
 * Replaces the cblas_sdot loops of drivers/in_mem_kmeans.cpp:75-78,179-182. */
BOF_API int bof_row_sqnorm_f32(bof_ctx* ctx, void* stream, int64_t rows, int64_t dim, const float* X,
                       int64_t ldx, float* out);

/* K8+K9: assign[p] = first c minimising | fl(fl(-2 <x_p, mu_c> + c_l2sq[c]) + p_l2sq[p]) |.
 * Replaces KMeansTask::execute (include/tasks/kmeans_task.h:53-82: sgemm alpha=-2 + two rank-1
 * updates) fused with the cblas_isamin scan of drivers/in_mem_kmeans.cpp:82-85 -- the P x K
 * distance matrix is never materialised.  points P x dim, centers K x dim, row-major, tight.
 * The dot products are computed like bof_sgemm_f32's, with the same special-value contract and the same
 * bof_config.gemm_k_chunk fold of the accumulation (dim <= 256 is one chunk at the default).
 * Needs workspace bof_kmeans_workspace_bytes(). `points_planes` is optional: a caller iterating
 * on the same points passes the buffer filled by bof_kmeans_prepare_points() to skip the
 * per-call TF32 split of the points. */
BOF_API int bof_kmeans_assign(bof_ctx* ctx, void* stream, int64_t npoints, int64_t ncenters, int64_t dim,
                      const float* points, const float* centers, const float* c_l2sq,
                      const float* p_l2sq, int32_t* assign, const void* points_planes,
                      void* workspace, size_t workspace_bytes);
BOF_API size_t bof_kmeans_workspace_bytes(int64_t npoints, int64_t ncenters, int64_t dim,
                                  int with_point_planes);
BOF_API size_t bof_kmeans_point_planes_bytes(int64_t npoints, int64_t dim);
BOF_API int bof_kmeans_prepare_points(bof_ctx* ctx, void* stream, int64_t npoints, int64_t dim,
                              const float* points, void* points_planes);

/* K10: sums[c, :] = sum_{p: assign[p]==c} x_p, added sequentially in ascending p (point ids are
 * grouped by a stable radix sort on the assignment, then fixed 256-point segments of each cluster
 * are summed by one thread block each and combined in order: deterministic, no atomics), counts[c] = #points.  Replaces the bucket + cblas_saxpy loop of
 * drivers/in_mem_kmeans.cpp:105-125.  sums is K x dim fp32 followed by nothing; counts K fp32
 * (exact below 2^24 points per cluster and NCCL-allreduce friendly).  The caller all-reduces
 * [sums | counts] across GPUs and then calls bof_kmeans_finalize. */
BOF_API int bof_kmeans_reduce(bof_ctx* ctx, void* stream, int64_t npoints, int64_t ncenters, int64_t dim,
                      const float* points, const int32_t* assign, float* sums, float* counts,
                      void* workspace, size_t workspace_bytes);
BOF_API size_t bof_kmeans_reduce_workspace_bytes(int64_t npoints, int64_t ncenters, int64_t dim);
/* centers[c] = sums[c] / counts[c], empty cluster => zero vector (in_mem_kmeans.cpp:112);
 * also refreshes c_l2sq[c] (in_mem_kmeans.cpp:75-78). */
BOF_API int bof_kmeans_finalize(bof_ctx* ctx, void* stream, int64_t ncenters, int64_t dim,
                        const float* sums, const float* counts, float* centers, float* c_l2sq);

/* ---- 3. host entry points (what include/flash_blas.h's adapters call) -------------------- */

/* flash::csrmm (include/flash_blas.h:37-46; src/blas/csrmm.cpp:424-472).  a/ja are indexed
 * from ia[0]; ja/ia int64 as on disk.  trans_a='T' is csr2csc followed by 'N'. */
BOF_API int bof_host_csrmm(bof_ctx* ctx, char trans_a, int64_t m, int64_t n, int64_t k, float alpha,
                   float beta, const float* a, const int64_t* ia, const int64_t* ja, char ord_b,
                   const float* b, float* c);

/* flash::gemm (include/flash_blas.h:14-18; src/blas/gemm.cpp:27-202).  Operands may exceed HBM: when the resident
 * plan (the whole op(B)^T, or op(A) for column-major C, plus a ring of row blocks of the other operand) does not fit
 * the free device memory, C is computed in super-blocks of rows with k cut into panels whose fp32 partial sums stay
 * on the device (BOF_GEMM_HBM_BUDGET=<bytes> overrides the device memory for that decision, read on every call).
 * Panels start on gemm_k_chunk boundaries and resume the fold of the previous panel, so the result is bit-identical
 * to the resident one whatever the budget; the exception is gemm_k_chunk < 0 (whole k in TMEM), where out-of-core
 * calls fold at panel boundaries and match to rounding only.  BOF_ENOMEM, with the minimum in bof_last_error, when
 * not even 256 rows of C and one chunk of k fit.  Also true of bof_host_kmeans_dist. */
BOF_API int bof_host_gemm(bof_ctx* ctx, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k,
                  float alpha, float beta, const float* a, const float* b, float* c, int64_t lda,
                  int64_t ldb, int64_t ldc);

/* Variants for one-process-per-GPU sharding with the replicated dense operand already in this GPU's
 * HBM (SURVEY.md 8f-1): every rank uploads only 1/G of B and the ranks all-gather the rest over NVLink
 * (ncclAllGather, or blas-on-flash_b200/dist.py::allgather_dense); only the sharded operand and the
 * output rows cross PCIe.  b_dev is read-only.  Row-major, csrmm trans_a='N' only. */
BOF_API int bof_host_gemm_devb(bof_ctx* ctx, char ta, char tb, int64_t m, int64_t n, int64_t k, float alpha,
                       float beta, const float* a, const float* b_dev, float* c, int64_t lda,
                       int64_t ldb, int64_t ldc);
BOF_API int bof_host_csrmm_devb(bof_ctx* ctx, int64_t m, int64_t n, int64_t k, float alpha, float beta,
                        const float* a, const int64_t* ia, const int64_t* ja, const float* b_dev,
                        float* c);

/* ---- multi-GPU: one communicator rank per context (north_star (5); SURVEY.md 8e, 8f-1) ---------------
 * The reference is single-process, single-node, CPU only (SURVEY.md 2.3): there is nothing to replace; these entry
 * points are how its row-block tasks (src/blas/csrmm.cpp:64-126, src/blas/gemm.cpp:83-129) spread over the GPUs
 * of a node.  Output row blocks are sharded over the ranks with no collective on the compute path; NVLink carries
 * (i) the replicated dense operand, uploaded 1/world per rank and broadcast panel by panel while the tensor cores
 * / SpMM already work on what has arrived, and (ii) the k-means allreduce of centroid sums and counts.
 * NCCL is dlopen'ed on first use (libnccl.so.2): no link-time dependency, never loaded by single-GPU users.
 *   one process per GPU: rank 0 calls bof_comm_unique_id, the launcher distributes the 128 bytes, every rank calls
 *                        bof_comm_init on its context;
 *   one process, many GPUs: bof_mgpu_create below. */
#define BOF_COMM_ID_BYTES 128
BOF_API int bof_comm_unique_id(void* id_out /* BOF_COMM_ID_BYTES */);
BOF_API int bof_comm_init(bof_ctx* ctx, int world, int rank, const void* id);
BOF_API int bof_comm_finalize(bof_ctx* ctx);
BOF_API int bof_comm_world(const bof_ctx* ctx);   /* 1 without a communicator */
BOF_API int bof_comm_rank(const bof_ctx* ctx);
/* flash::gemm, row-major, on this rank's rows of op(A) and C (m_local of them); `b` is the WHOLE B in host memory
 * every rank can read (same contents on all ranks).  Collective: every rank of the communicator calls it with the
 * same n, k, tb.  Panel j of B is uploaded by rank j % world and broadcast; C leaves column slab by column slab. */
BOF_API int bof_dist_gemm(bof_ctx* ctx, char ta, char tb, int64_t m_local, int64_t n, int64_t k, float alpha,
                  float beta, const float* a_local, const float* b, float* c_local, int64_t lda,
                  int64_t ldb, int64_t ldc);
/* flash::csrmm('N', ..., 'R', ...) on this rank's row block of A (offsets may be un-rebased: values / indices are
 * addressed relative to ia[0]) and of C; `b` is the whole n x k B in host memory.  Collective. */
BOF_API int bof_dist_csrmm(bof_ctx* ctx, int64_t m_local, int64_t n, int64_t k, float alpha, float beta,
                   const float* a, const int64_t* ia, const int64_t* ja, const float* b, float* c_local);

/* One process, several GPUs (what flash_setup() + the flash:: entry points use when BOF_GPUS > 1): a context and a
 * communicator rank per device, one host thread per device inside every call, host operands shared by all of them
 * (one copy of B in host memory instead of one per process).  ndev <= 0: every visible device; devices may be NULL
 * (ordinals 0 .. ndev-1); cfg->device is ignored.  Same one-call-at-a-time rule as a single context. */
typedef struct bof_mgpu bof_mgpu;
BOF_API int bof_mgpu_create(const bof_config* cfg, int ndev, const int* devices, bof_mgpu** out);
BOF_API int bof_mgpu_destroy(bof_mgpu* mg);
BOF_API int bof_mgpu_count(const bof_mgpu* mg);
BOF_API bof_ctx* bof_mgpu_ctx(bof_mgpu* mg, int rank);
BOF_API const char* bof_mgpu_last_error(const bof_mgpu* mg);
/* flash::gemm: rows of C ('R') / columns of C ('C') sharded over the GPUs, the other operand panel-broadcast. */
BOF_API int bof_mgpu_gemm(bof_mgpu* mg, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k, float alpha,
                  float beta, const float* a, const float* b, float* c, int64_t lda, int64_t ldb, int64_t ldc);
/* flash::csrmm: trans_a='N', ord_b='R' = nnz-balanced row blocks per GPU; every other combination runs on GPU 0. */
BOF_API int bof_mgpu_csrmm(bof_mgpu* mg, char trans_a, int64_t m, int64_t n, int64_t k, float alpha, float beta,
                   const float* a, const int64_t* ia, const int64_t* ja, char ord_b, const float* b, float* c);
/* flash::csrgemv: 'N' disjoint row blocks; 'T' per-GPU partial y added on the host in GPU order (deterministic). */
BOF_API int bof_mgpu_csrgemv(bof_mgpu* mg, char trans_a, int64_t m, int64_t n, const float* a, const int64_t* ia,
                     const int64_t* ja, const float* x, float* y);
/* drivers/in_mem_kmeans.cpp:89-152 x iters: points sharded and resident, NCCL allreduce per iteration. */
BOF_API int bof_mgpu_kmeans_lloyd(bof_mgpu* mg, int64_t npoints, int64_t ncenters, int64_t dim,
                          const float* points_host, float* centers_host, int64_t iters, int64_t* assign_out);

/* flash::kmeans, the distance tile of k-means (include/flash_blas.h:20-25; KMeansTask::execute,
 * include/tasks/kmeans_task.h:53-82): the product of bof_host_gemm, then C(i, j) += c_l2sq[i] and
 * C(i, j) += p_l2sq[j] in that order (i over m, j over n), applied to each output block on the device
 * before it is downloaded.  c_l2sq (m entries) and p_l2sq (n entries) are host arrays. */
BOF_API int bof_host_kmeans_dist(bof_ctx* ctx, char mat_ord, char trans_a, char trans_b, int64_t m, int64_t n,
                         int64_t k, float alpha, float beta, const float* a, const float* b, float* c,
                         int64_t lda_a, int64_t lda_b, int64_t lda_c, const float* c_l2sq,
                         const float* p_l2sq);

/* flash::csrgemv (include/flash_blas.h:55-57; src/blas/csrgemv.cpp:82-97). */
BOF_API int bof_host_csrgemv(bof_ctx* ctx, char trans_a, int64_t m, int64_t n, const float* a,
                     const int64_t* ia, const int64_t* ja, const float* b, float* c);

/* flash::csrcsc (include/flash_blas.h:49-52; src/blas/csrcsc.cpp:32-159). */
BOF_API int bof_host_csrcsc(bof_ctx* ctx, int64_t m, int64_t n, const int64_t* ia, const int64_t* ja,
                    const float* a, int64_t* ia_tr, int64_t* ja_tr, float* a_tr);

/* A resident in HBM across calls (SURVEY 8(f)-2): the in-memory-B/C csrmm overload and csrgemv as the inner
 * loop of an eigensolver re-multiply the same A (include/flash_blas.h:43-46; src/blas/csrmm.cpp:453-472;
 * drivers/csrmm_pmem.cpp).  The reference re-reads A from flash every call because its Cache
 * (include/scheduler/cache.h:11-42) is flushed when a kernel returns; here bof_csr_open uploads A once
 * (host arrays as flash_ptr::ptr gives them; indices narrowed to int32 on the device) and bof_csr_mm /
 * bof_csr_mv take host B, C / x, y with the argument meaning of bof_host_csrmm / bof_host_csrgemv.
 * trans_a = 'T' products run on a resident copy of A^T (stable csr2csc, built on first use or by
 * bof_csr_build_transpose; it doubles the footprint); bof_csr_mv('T') without that copy uses the scatter
 * kernel on A.  bof_csr_arrays exposes the device arrays (int32 indices, int64 offsets) of A or A^T for
 * callers that keep B and C on the device and call bof_spmm_csr_f32 / bof_spmv_csr_f32 themselves.
 * One call at a time per context, like every other entry point. */
typedef struct bof_csr bof_csr;
BOF_API int bof_csr_open(bof_ctx* ctx, int64_t m, int64_t n, const float* a, const int64_t* ia, const int64_t* ja,
                 bof_csr** out);
BOF_API int bof_csr_build_transpose(bof_csr* h);
BOF_API int bof_csr_arrays(bof_csr* h, char trans_a, const float** vals, const int32_t** idx, const int64_t** offs,
                   int64_t* nnz);
BOF_API int bof_csr_mm(bof_csr* h, char trans_a, int64_t k, float alpha, float beta, char ord_b, const float* b,
               float* c);
BOF_API int bof_csr_mv(bof_csr* h, char trans_a, const float* x, float* y);
BOF_API int bof_csr_close(bof_csr* h);

/* One Lloyd iteration on this rank's shard of the points, device-resident across calls:
 * bof_kmeans_open uploads the shard once (drivers/kmeans.cpp:206-217: points mapped, norms
 * computed once); bof_kmeans_local_step = closest_centers + per-cluster partial sums
 * (drivers/in_mem_kmeans.cpp:69-125) leaving [K*dim sums | K (count & 4095) | K (count >> 12)] fp32 -- every entry
 * an exact integer or sum, also after adding the ranks' buffers -- in a device buffer
 * whose address is returned so that the caller can NCCL-allreduce it in place (the only
 * collective on the path); bof_kmeans_update divides and refreshes the resident centers.
 * assign_out (host, int64 as FBLAS_UINT center_index, in_mem_kmeans.cpp:82-85) may be NULL.
 * Out-of-core shards: when the shard with its operand planes and workspaces exceeds ~70 % of the device's memory
 * the points are NOT kept resident; every local_step then streams them from points_host in chunks through two
 * device buffers (upload of chunk c+1 overlapped with assign + reduce of chunk c; the reference re-reads its points
 * from flash every iteration the same way, drivers/kmeans.cpp:143-145), and points_host MUST stay valid and
 * unchanged until bof_kmeans_close. */
typedef struct bof_kmeans bof_kmeans;
BOF_API int bof_kmeans_open(bof_ctx* ctx, int64_t npoints, int64_t ncenters, int64_t dim,
                    const float* points_host, const float* centers_host, bof_kmeans** out);
BOF_API int bof_kmeans_local_step(bof_kmeans* km, void** dev_partial, size_t* partial_floats);
BOF_API int bof_kmeans_update(bof_kmeans* km);
/* In-place NCCL sum of the partial buffer over the ranks of the context's communicator, on the k-means stream (the
 * only reduction on the path); no-op at world 1.  bof_kmeans_lloyd = iters x (local_step, allreduce, update). */
BOF_API int bof_kmeans_allreduce(bof_kmeans* km);
BOF_API int bof_kmeans_lloyd(bof_kmeans* km, int64_t iters);
BOF_API int bof_kmeans_get(bof_kmeans* km, float* centers_host, int64_t* assign_host);
BOF_API void* bof_kmeans_stream(bof_kmeans* km);
BOF_API int bof_kmeans_close(bof_kmeans* km);

#ifdef __cplusplus
}
#endif
#endif /* BOF_B200_H_ */
