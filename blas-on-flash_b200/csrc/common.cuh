// Shared plumbing for the sm_100a kernels and the C ABI (include/bof_b200.h).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "bof_b200.h"

namespace bof {

constexpr int kNumSmsFallback = 148;

// One slot of the pinned staging ring used for pageable host operands (file mmaps).
struct StageSlot {
  void* ptr = nullptr;
  cudaEvent_t ev = nullptr;   // completion of the DMA that last used the slot
  bool in_flight = false;
  // pending device->host chunk: where the slot's contents go once the DMA has landed
  char* out_dst = nullptr;
  size_t out_pitch = 0, out_width = 0, out_rows = 0;
};

class CopyPool;  // host memcpy worker threads (capi.cu)
class Drainer;   // background thread that copies landed device->host chunks out of the pinned ring (capi.cu)

}  // namespace bof

// The opaque context of the C ABI: one per process/GPU (replaces the static flash::sched,
// src/lib_funcs.cpp:9 of the reference).
namespace bof { struct CommState; }

struct bof_ctx {
  bof_config cfg{};
  int device = 0;
  int num_sms = bof::kNumSmsFallback;
  size_t l2_bytes = 0;
  cudaStream_t compute = nullptr;  // kernels of the host entry points
  cudaStream_t h2d = nullptr;      // uploads
  cudaStream_t d2h = nullptr;      // downloads
  std::vector<bof::StageSlot> stage_in, stage_out;   // pinned rings, allocated on first pageable copy
  bof::CopyPool* pool = nullptr;       // workers of the calling thread (host -> pinned)
  bof::CopyPool* pool_out = nullptr;   // workers of the drainer thread (pinned -> host)
  bof::Drainer* drainer = nullptr;
  std::string err;
  bof_stats stats{};
  std::atomic<int64_t> launches{0};
  void* tmap_encode = nullptr;  // cuTensorMapEncodeTiled, fetched at ctx creation
  // Grow-only device buffers owned by the context and reused across host entry points, so that
  // steady-state calls do no cudaMalloc (the reference's counterpart is the Program Cache budget,
  // src/scheduler/cache.cpp).
  static constexpr int kSlots = 40;
  void* slot_ptr[kSlots] = {};
  size_t slot_bytes[kSlots] = {};
  std::vector<cudaEvent_t> events;
  // BOF_TRACE=1: timing events recorded along a host pipeline, printed (ms since the first) when it ends
  struct TraceMark { cudaEvent_t ev; const char* what; int idx; };
  std::vector<TraceMark> trace;
  std::vector<cudaEvent_t> trace_pool;
  struct HostMark { double ms; const char* what; long idx; };
  std::vector<HostMark> host_trace;   // wall-clock marks of the calling and the drainer thread
  std::mutex host_trace_mu;
  double trace_t0 = 0.0;
  // CUDA-event bracket of the most recent tensor-core GEMM kernel (for the roofline figure)
  cudaEvent_t tk0 = nullptr, tk1 = nullptr;
  bool tk_valid = false;
  uint32_t* sync_ctr = nullptr;   // wave lock-step counters of the GEMM kernel
  size_t sync_ctr_count = 0;
  // multi-GPU: communicator of this context's rank (comm.cu), collectives run on `coll`
  bof::CommState* comm = nullptr;
  cudaStream_t coll = nullptr;
  // SMs the persistent tensor-core kernels leave free while collectives of the same call may be waiting on the GPU:
  // an NCCL kernel that waits for a peer holds its CTAs, and a persistent grid that needs every SM would wait for it
  // (seen with BOF_TRACE at 2 GPUs: 20 ms stalls of the MMAs behind a broadcast whose root had not uploaded yet)
  int sm_reserve = 0;
};

namespace bof {

// cudaFuncSetAttribute applies to the CURRENT device only; one process may hold contexts on several GPUs
// (bof_config.device), so "already set" is remembered per device ordinal. Setting it twice is harmless.
struct PerDeviceOnce {
  std::atomic<uint64_t> mask{0};
  bool need(int dev) const { return ((mask.load(std::memory_order_acquire) >> (dev & 63)) & 1ull) == 0; }
  void done(int dev) { mask.fetch_or(1ull << (dev & 63), std::memory_order_release); }
};

inline int fail(bof_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  if (getenv("BOF_VERBOSE")) fprintf(stderr, "[bof_b200] error %d: %s\n", code, buf);
  return code;
}

#define BOF_CUDA(ctx, expr)                                                                  \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return bof::fail((ctx), BOF_ECUDA, "%s failed: %s (%s:%d)", #expr,                     \
                       cudaGetErrorString(e__), __FILE__, __LINE__);                         \
  } while (0)

#define BOF_LAUNCH_CHECK(ctx, what)                                                          \
  do {                                                                                       \
    cudaError_t e__ = cudaGetLastError();                                                    \
    if (e__ != cudaSuccess)                                                                  \
      return bof::fail((ctx), BOF_ECUDA, "launch of %s failed: %s (%s:%d)", (what),          \
                       cudaGetErrorString(e__), __FILE__, __LINE__);                         \
    (ctx)->launches.fetch_add(1, std::memory_order_relaxed);                                 \
  } while (0)

#define BOF_REQUIRE(ctx, cond, ...)                                                          \
  do {                                                                                       \
    if (!(cond)) return bof::fail((ctx), BOF_EINVAL, __VA_ARGS__);                           \
  } while (0)

template <typename T>
__host__ __device__ constexpr T ceil_div(T a, T b) {
  return (a + b - 1) / b;
}
template <typename T>
__host__ __device__ constexpr T round_up(T a, T b) {
  return ceil_div(a, b) * b;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Device buffer `slot` of at least `bytes` (contents are not preserved when it has to grow).
int slot_reserve(bof_ctx* ctx, int slot, size_t bytes, void** out);
template <typename T>
int slot_reserve(bof_ctx* ctx, int slot, size_t count, T** out) {
  void* p = nullptr;
  int rc = slot_reserve(ctx, slot, count * sizeof(T), &p);
  *out = static_cast<T*>(p);
  return rc;
}

// ---- kernel launchers implemented in the .cu files (device pointers, no validation) --------

// b_rows = number of rows of B (the gather target) when the caller knows it, 0 otherwise: it only steers the
// choice between kernel variants (L2 residency of the gather target).
int launch_spmm_rm(bof_ctx* ctx, cudaStream_t s, int64_t m, int64_t k, float alpha,
                   const float* vals, const int32_t* idx, const int64_t* offs, const float* B,
                   int64_t ldb, float beta, float* C, int64_t ldc, int64_t b_rows = 0);
// trans 'N'; 'T' (y zeroed first) / 't' (y += A^T x).  The transposed product is deterministic by default: products
// sorted stably by column, fixed-order column sums (radix.cu); bof_config.spmv_t_atomic = 1 selects the scatter kernel
// with red.global.add.f32 instead (faster, order of the additions varies from run to run).  nnz < 0: read from offs.
int launch_spmv(bof_ctx* ctx, cudaStream_t s, char trans, int64_t m, int64_t n, const float* vals,
                const int32_t* idx, const int64_t* offs, const float* x, float* y, int64_t nnz = -1);
size_t spmv_t_workspace_bytes(int64_t n, int64_t nnz);
int launch_spmv_t_sorted(bof_ctx* ctx, cudaStream_t s, int accumulate, int64_t m, int64_t n, int64_t nnz, const float* vals,
                         const int32_t* idx, const int64_t* offs, const float* x, float* y, void* ws, size_t ws_bytes);
constexpr int kSlotSpmvT = 35;      // context slot: workspace of the sorted A^T x path
constexpr int kSlotSpmmLong = 36;   // context slot: counters, deferred-row lists, grid-path partials of the SpMM
int launch_idx_narrow(bof_ctx* ctx, cudaStream_t s, const int64_t* in, int32_t* out, int64_t n);
int launch_idx_widen(bof_ctx* ctx, cudaStream_t s, const int32_t* in, int64_t* out, int64_t n);
// out[c * ldo + r] = in[r * ldi + c] for an rows x cols row-major input
int launch_transpose(bof_ctx* ctx, cudaStream_t s, int64_t rows, int64_t cols, const float* in,
                     int64_t ldi, float* out, int64_t ldo);
int launch_add_outer_terms(bof_ctx* ctx, cudaStream_t s, float* C, int64_t rows, int64_t cols, int64_t ldc,
                           const float* rowv, const float* colv, int row_first);
// out = alpha * in^T + beta * out, same indexing as launch_transpose (beta==0: out not read)
int launch_transpose_axpby(bof_ctx* ctx, cudaStream_t s, int64_t rows, int64_t cols, float alpha,
                           const float* in, int64_t ldi, float beta, float* out, int64_t ldo);

// TF32 split of a logical R x K operand whose element (r, kk) lives at src[r*s_r + kk*s_k]
// (exactly one of s_r, s_k is 1) into K-major planes hi/lo of row stride kp (multiple of 32).
int launch_split_planes(bof_ctx* ctx, cudaStream_t s, int64_t R, int64_t K, const float* src,
                        int64_t s_r, int64_t s_k, float* hi, float* lo, int64_t kp);

struct GemmEpilogue {
  // plain GEMM: Cout[i * ldc + j] = alpha * acc + beta * Cout
  float alpha = 1.f, beta = 0.f;
  float* C = nullptr;
  int64_t ldc = 0;
  // k-means assign epilogue (C == nullptr): per row running argmin over j of
  // |fl(fl(-2*acc + col_add[j]) + row_add[i])|
  const float* row_add = nullptr;
  const float* col_add = nullptr;
  int32_t* argmin_out = nullptr;
  // k-panels of one long k (plain GEMM only): each element's fold starts from carry[i * ld_carry + j] instead of 0,
  // and raw_out stores the fold itself to C (alpha and beta are applied by the last panel only)
  const float* carry = nullptr;
  int64_t ld_carry = 0;
  bool raw_out = false;
};

// Tensor-core core: acc[i, j] = sum_k P[i, k] * Q[j, k] with P = (p_hi, p_lo) M x kp planes and
// Q = (q_hi, q_lo) N x kp planes, 3xTF32 (lo*hi + hi*lo + hi*hi), fp32 accumulate in TMEM with an
// fp32 round-to-nearest fold every k_chunk elements of k.
int launch_gemm_tc(bof_ctx* ctx, cudaStream_t s, int cta_group, int64_t M, int64_t N, int64_t K,
                   int64_t kp, const float* p_hi, const float* p_lo, const float* q_hi,
                   const float* q_lo, const GemmEpilogue& ep, int64_t k_chunk);

int tc_issue_rate(bof_ctx* ctx, cudaStream_t s, int kind, int rounds, double* mma_tflops, double* useful_tflops);

// CUDA-core fp32 GEMM for ragged / unaligned shapes: C[i*ldc+j] = alpha*sum_k A(i,k)*B(k,j) +
// beta*C with A(i,k) = A[i*a_r + k*a_k], B(k,j) = B[k*b_k + j*b_c].
int launch_gemm_ffma(bof_ctx* ctx, cudaStream_t s, int64_t M, int64_t N, int64_t K, float alpha,
                     const float* A, int64_t a_r, int64_t a_k, const float* B, int64_t b_k,
                     int64_t b_c, float beta, float* C, int64_t ldc);

int launch_row_sqnorm(bof_ctx* ctx, cudaStream_t s, int64_t rows, int64_t dim, const float* X,
                      int64_t ldx, float* out);
size_t kmeans_reduce_workspace_bytes(int64_t npoints, int64_t ncenters, int64_t dim);
int launch_kmeans_reduce_ws(bof_ctx* ctx, cudaStream_t s, int64_t npoints, int64_t ncenters,
                            int64_t dim, const float* points, const int32_t* assign, float* sums,
                            float* counts, void* ws, size_t ws_bytes, float* counts_hi = nullptr);
// counts_hi != nullptr: the cluster sizes are split as counts = size & 4095, counts_hi = size >> 12 (both exact in fp32,
// also after a sum over ranks); otherwise `counts` holds the size itself (exact below 2^24)
int launch_kmeans_finalize(bof_ctx* ctx, cudaStream_t s, int64_t ncenters, int64_t dim,
                           const float* sums, const float* counts, float* centers, float* c_l2sq,
                           const float* counts_hi = nullptr);

size_t csr2csc_workspace_bytes(int64_t m, int64_t n, int64_t nnz);
int launch_csr2csc(bof_ctx* ctx, cudaStream_t s, int64_t m, int64_t n, int64_t nnz,
                   const int64_t* offs, const int32_t* idx, const float* vals, int64_t* offs_t,
                   int32_t* idx_t, float* vals_t, void* ws, size_t ws_bytes);

}  // namespace bof
