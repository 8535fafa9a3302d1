// The C ABI of include/bof_b200.h: context, argument validation, the device-tile entry points and
// the host entry points (per-GPU CUDA-stream tile pipelines: host buffer -> H2D -> kernel -> D2H
// -> host buffer).  The pipelines replace, for this path, the reference's scheduler / cache /
// io_executor / file_handle stack (src/scheduler/*.cpp, src/file_handles/*.cpp): residency is
// structural (every output row block is produced by one pass on one GPU), ordering is expressed
// with CUDA events instead of task parents and overlap checks.
#include "host_internal.cuh"

using namespace bof;

namespace {
thread_local std::string g_create_err;
}  // namespace

extern "C" {


int bof_abi_version(void) { return 1; }

int bof_ctx_create(const bof_config* cfg, bof_ctx** out) {
  if (!out) return BOF_EINVAL;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    g_create_err = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return BOF_ENODEV;
  }
  bof_ctx* ctx = new bof_ctx();
  if (cfg) ctx->cfg = *cfg;
  ctx->device = ctx->cfg.device;
  auto bail = [&](int code, const std::string& msg) {
    g_create_err = msg;
    delete ctx;
    return code;
  };
  if (ctx->device < 0 || ctx->device >= ndev) return bail(BOF_EINVAL, "device ordinal out of range");
  if ((e = cudaSetDevice(ctx->device)) != cudaSuccess) return bail(BOF_ECUDA, cudaGetErrorString(e));
  cudaDeviceProp prop{};
  if ((e = cudaGetDeviceProperties(&prop, ctx->device)) != cudaSuccess) return bail(BOF_ECUDA, cudaGetErrorString(e));
  if (prop.major != 10) {
    char buf[160];
    snprintf(buf, sizeof(buf), "device %d is sm_%d%d; this library only carries sm_100a code (B200)", ctx->device,
             prop.major, prop.minor);
    return bail(BOF_ENODEV, buf);
  }
  ctx->num_sms = prop.multiProcessorCount;
  ctx->l2_bytes = (size_t)prop.l2CacheSize;
  if (ctx->cfg.n_copy_threads <= 0) ctx->cfg.n_copy_threads = 8;
  if (ctx->cfg.stage_bytes == 0) ctx->cfg.stage_bytes = 16ull << 20;
  if (ctx->cfg.n_stage_bufs <= 0) ctx->cfg.n_stage_bufs = 4;
  if (ctx->cfg.csrmm_max_nnz == 0) ctx->cfg.csrmm_max_nnz = 64ull << 20;
  if (ctx->cfg.gemm_row_block == 0) ctx->cfg.gemm_row_block = 4096;
  cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&ctx->h2d, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&ctx->d2h, cudaStreamNonBlocking);
  cudaDriverEntryPointQueryResult qres;
  void* fn = nullptr;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
      qres == cudaDriverEntryPointSuccess)
    ctx->tmap_encode = fn;
  else
    cudaGetLastError();
  *out = ctx;
  return BOF_OK;
}

int bof_ctx_destroy(bof_ctx* ctx) {
  if (!ctx) return BOF_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (int i = 0; i < bof_ctx::kSlots; ++i)
    if (ctx->slot_ptr[i]) cudaFree(ctx->slot_ptr[i]);
  for (auto ev : ctx->events) cudaEventDestroy(ev);
  for (auto& m : ctx->trace) cudaEventDestroy(m.ev);
  for (auto ev : ctx->trace_pool) cudaEventDestroy(ev);
  comm_destroy(ctx);
  staging_destroy(ctx);  // copy pools, drainer thread (joined first), pinned rings
  if (ctx->sync_ctr) cudaFree(ctx->sync_ctr);
  if (ctx->tk0) cudaEventDestroy(ctx->tk0);
  if (ctx->tk1) cudaEventDestroy(ctx->tk1);
  if (ctx->compute) cudaStreamDestroy(ctx->compute);
  if (ctx->h2d) cudaStreamDestroy(ctx->h2d);
  if (ctx->d2h) cudaStreamDestroy(ctx->d2h);
  delete ctx;
  return BOF_OK;
}

const char* bof_last_error(const bof_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int bof_get_stats(const bof_ctx* ctx, bof_stats* out) {
  if (!ctx || !out) return BOF_EINVAL;
  *out = ctx->stats;
  // kernel_ms: device time of the most recent tensor-core GEMM kernel, once it has finished
  if (ctx->tk_valid && cudaEventQuery(ctx->tk1) == cudaSuccess) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->tk0, ctx->tk1) == cudaSuccess) out->kernel_ms = ms;
  }
  cudaGetLastError();
  return BOF_OK;
}

int64_t bof_launch_count(const bof_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }

// ---- device-tile entry points ---------------------------------------------------------------

size_t bof_spmm_workspace_bytes(char ord, int64_t m, int64_t n, int64_t k) {
  if (ord != 'C') return 0;
  return round_up<size_t>((size_t)n * k * 4, 256) + round_up<size_t>((size_t)m * k * 4, 256) + 256;
}

int bof_spmm_csr_f32(bof_ctx* ctx, void* stream, char ord, int64_t m, int64_t n, int64_t k, float alpha,
                     const float* vals, const int32_t* idx, const int64_t* offs, const float* B, int64_t ldb,
                     float beta, float* C, int64_t ldc, void* workspace, size_t workspace_bytes) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, is_rc(ord), "csrmm: ord_b must be 'R' or 'C' (got '%c')", ord);
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && k >= 0, "csrmm: negative dimension");
  BOF_REQUIRE(ctx, n < (1ll << 31), "csrmm: column count must fit int32 on the device");
  cudaStream_t s = as_stream(stream);
  if (m == 0 || k == 0) return BOF_OK;
  if (ord == 'R') {
    BOF_REQUIRE(ctx, ldb >= k && ldc >= k, "csrmm: leading dimension too small");
    return launch_spmm_rm(ctx, s, m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc, n);
  }
  // Column-major B (n x k, ldb >= n) and C (m x k, ldc >= m): transpose-on-stage around the
  // row-major kernel; the gathers need B rows contiguous.
  BOF_REQUIRE(ctx, ldb >= n && ldc >= m, "csrmm: leading dimension too small");
  BOF_REQUIRE(ctx, workspace && workspace_bytes >= bof_spmm_workspace_bytes(ord, m, n, k),
              "csrmm: column-major needs bof_spmm_workspace_bytes() of workspace");
  uint8_t* base = reinterpret_cast<uint8_t*>(round_up<uintptr_t>(reinterpret_cast<uintptr_t>(workspace), 256));
  float* Bt = reinterpret_cast<float*>(base);
  float* Ct = reinterpret_cast<float*>(base + round_up<size_t>((size_t)n * k * 4, 256));
  BOF_TRY(launch_transpose(ctx, s, k, n, B, ldb, Bt, k));
  BOF_TRY(launch_spmm_rm(ctx, s, m, k, 1.f, vals, idx, offs, Bt, k, 0.f, Ct, k, n));
  return launch_transpose_axpby(ctx, s, m, k, alpha, Ct, k, beta, C, ldc);
}

int bof_spmv_csr_f32(bof_ctx* ctx, void* stream, char trans, int64_t m, int64_t n, const float* vals,
                     const int32_t* idx, const int64_t* offs, const float* x, float* y) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, is_nt(trans), "csrgemv: trans_a must be 'N' or 'T' (got '%c')", trans);
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && n < (1ll << 31), "csrgemv: bad dimension");
  return launch_spmv(ctx, as_stream(stream), trans, m, n, vals, idx, offs, x, y);
}

int bof_idx_narrow(bof_ctx* ctx, void* stream, const int64_t* in, int32_t* out, int64_t count) {
  if (!ctx) return BOF_EINVAL;
  return launch_idx_narrow(ctx, as_stream(stream), in, out, count);
}
int bof_idx_widen(bof_ctx* ctx, void* stream, const int32_t* in, int64_t* out, int64_t count) {
  if (!ctx) return BOF_EINVAL;
  return launch_idx_widen(ctx, as_stream(stream), in, out, count);
}

size_t bof_sgemm_workspace_bytes(int64_t m, int64_t n, int64_t k) {
  const int64_t kp = padded_k(k);
  return 2 * plane_bytes(m, kp) + 2 * plane_bytes(n, kp) + 512;
}

int bof_sgemm_f32(bof_ctx* ctx, void* stream, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k,
                  float alpha, const float* A, int64_t lda, const float* B, int64_t ldb, float beta, float* C,
                  int64_t ldc, void* workspace, size_t workspace_bytes) {
  if (!ctx) return BOF_EINVAL;
  Canon c;
  BOF_TRY(canon_gemm(ctx, ord, ta, tb, m, n, k, A, lda, B, ldb, ldc, &c));
  return gemm_canon_device(ctx, as_stream(stream), c, alpha, beta, C, workspace, workspace_bytes);
}

int bof_tc_issue_rate(bof_ctx* ctx, void* stream, int kind, int rounds, double* mma_tflops, double* useful_tflops) {
  if (!ctx) return BOF_EINVAL;
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  return tc_issue_rate(ctx, as_stream(stream), kind, rounds, mma_tflops, useful_tflops);
}

size_t bof_csr2csc_workspace_bytes(int64_t m, int64_t n, int64_t nnz) { return csr2csc_workspace_bytes(m, n, nnz); }

int bof_csr2csc(bof_ctx* ctx, void* stream, int64_t m, int64_t n, int64_t nnz, const int64_t* offs,
                const int32_t* idx, const float* vals, int64_t* offs_t, int32_t* idx_t, float* vals_t,
                void* workspace, size_t workspace_bytes) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && nnz >= 0, "csrcsc: negative dimension");
  return launch_csr2csc(ctx, as_stream(stream), m, n, nnz, offs, idx, vals, offs_t, idx_t, vals_t, workspace,
                        workspace_bytes);
}

int bof_row_sqnorm_f32(bof_ctx* ctx, void* stream, int64_t rows, int64_t dim, const float* X, int64_t ldx,
                       float* out) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, rows >= 0 && dim >= 0 && ldx >= dim, "row_sqnorm: bad dimension");
  return launch_row_sqnorm(ctx, as_stream(stream), rows, dim, X, ldx, out);
}

size_t bof_kmeans_point_planes_bytes(int64_t npoints, int64_t dim) { return 2 * plane_bytes(npoints, padded_k(dim)) + 256; }

size_t bof_kmeans_workspace_bytes(int64_t npoints, int64_t ncenters, int64_t dim, int with_point_planes) {
  size_t b = 2 * plane_bytes(ncenters, padded_k(dim)) + 512;
  if (with_point_planes) b += bof_kmeans_point_planes_bytes(npoints, dim);
  return b;
}

int bof_kmeans_prepare_points(bof_ctx* ctx, void* stream, int64_t npoints, int64_t dim, const float* points,
                              void* points_planes) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, npoints >= 0 && dim > 0 && points_planes, "kmeans: bad argument");
  const int64_t kp = padded_k(dim);
  uint8_t* base = reinterpret_cast<uint8_t*>(round_up<uintptr_t>(reinterpret_cast<uintptr_t>(points_planes), 256));
  return launch_split_planes(ctx, as_stream(stream), npoints, dim, points, dim, 1, reinterpret_cast<float*>(base),
                             reinterpret_cast<float*>(base + plane_bytes(npoints, kp)), kp);
}

int bof_kmeans_assign(bof_ctx* ctx, void* stream, int64_t npoints, int64_t ncenters, int64_t dim,
                      const float* points, const float* centers, const float* c_l2sq, const float* p_l2sq,
                      int32_t* assign, const void* points_planes, void* workspace, size_t workspace_bytes) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, npoints >= 0 && ncenters > 0 && dim > 0, "kmeans: bad dimension");
  BOF_REQUIRE(ctx, workspace && workspace_bytes >= bof_kmeans_workspace_bytes(npoints, ncenters, dim, points_planes == nullptr),
              "kmeans: workspace too small");
  if (npoints == 0) return BOF_OK;
  cudaStream_t s = as_stream(stream);
  const int64_t kp = padded_k(dim);
  uint8_t* base = reinterpret_cast<uint8_t*>(round_up<uintptr_t>(reinterpret_cast<uintptr_t>(workspace), 256));
  float* c_hi = reinterpret_cast<float*>(base);
  float* c_lo = reinterpret_cast<float*>(base + plane_bytes(ncenters, kp));
  BOF_TRY(launch_split_planes(ctx, s, ncenters, dim, centers, dim, 1, c_hi, c_lo, kp));
  const uint8_t* pp;
  if (points_planes) {
    pp = reinterpret_cast<const uint8_t*>(round_up<uintptr_t>(reinterpret_cast<uintptr_t>(points_planes), 256));
  } else {
    uint8_t* mine = base + 2 * plane_bytes(ncenters, kp);
    BOF_TRY(bof_kmeans_prepare_points(ctx, stream, npoints, dim, points, mine));
    pp = reinterpret_cast<const uint8_t*>(round_up<uintptr_t>(reinterpret_cast<uintptr_t>(mine), 256));
  }
  GemmEpilogue ep;
  ep.C = nullptr;
  ep.row_add = p_l2sq;
  ep.col_add = c_l2sq;
  ep.argmin_out = assign;
  const int cg = ctx->cfg.gemm_force_path == 1 ? 1 : 2;
  return launch_gemm_tc(ctx, s, cg, npoints, ncenters, dim, kp, reinterpret_cast<const float*>(pp),
                        reinterpret_cast<const float*>(pp + plane_bytes(npoints, kp)), c_hi, c_lo, ep, k_chunk_of(ctx));
}

size_t bof_kmeans_reduce_workspace_bytes(int64_t npoints, int64_t ncenters, int64_t dim) {
  return kmeans_reduce_workspace_bytes(npoints, ncenters, dim);
}

int bof_kmeans_reduce(bof_ctx* ctx, void* stream, int64_t npoints, int64_t ncenters, int64_t dim,
                      const float* points, const int32_t* assign, float* sums, float* counts, void* workspace,
                      size_t workspace_bytes) {
  if (!ctx) return BOF_EINVAL;
  return launch_kmeans_reduce_ws(ctx, as_stream(stream), npoints, ncenters, dim, points, assign, sums, counts,
                                 workspace, workspace_bytes);
}

int bof_kmeans_finalize(bof_ctx* ctx, void* stream, int64_t ncenters, int64_t dim, const float* sums,
                        const float* counts, float* centers, float* c_l2sq) {
  if (!ctx) return BOF_EINVAL;
  return launch_kmeans_finalize(ctx, as_stream(stream), ncenters, dim, sums, counts, centers, c_l2sq);
}

}  // extern "C"
