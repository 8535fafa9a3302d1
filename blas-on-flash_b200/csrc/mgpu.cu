// One process, several GPUs: the flash:: entry points of a C++ application (and drivers/*.cpp) spread over the
// GPUs of the node without Python or a launcher.  A bof_mgpu owns one context + communicator rank per device;
// every call runs one host thread per device (north_star (5): output row blocks sharded with no collective; the
// replicated dense operand crosses PCIe once per node and is copied to the peers over NVLink; k-means allreduces
// centroid sums and counts).  Host operands are shared by all threads: one copy of B in host memory instead of N.
//
// Calls are organised in PHASES separated by a join of the per-device threads, and inside a phase no thread's
// progress depends on another thread's CUDA calls.  The flag-gated exchange of bof_dist_* (streams parked on
// cuStreamWaitValue32 until a peer's push arrives) is for one process per GPU only: inside one process, with peer
// access enabled, a cudaMalloc / cudaHostAlloc on one device can need the other devices' work to drain, which a
// parked stream never does -- seen as an intermittent hang at 4 GPUs (profiles/r02/t17_mgpu_check_hang.txt).
// Here the replicated operand is therefore completed on every device first (own slice uploaded, then pushed to the
// peers with copy-engine peer copies, everything stream-ordered on the pushing device), the threads join, and each
// device then runs the ordinary single-GPU pipeline against its resident copy (bof_host_*_devb).
#include "host_internal.cuh"

#include <thread>

using namespace bof;

extern "C" {
int bof_comm_unique_id(void* id_out);
int bof_comm_init(bof_ctx* ctx, int world, int rank, const void* id);
int bof_dist_gemm(bof_ctx* ctx, char ta, char tb, int64_t m_local, int64_t n, int64_t k, float alpha, float beta,
                  const float* a_local, const float* b, float* c_local, int64_t lda, int64_t ldb, int64_t ldc);
int bof_dist_csrmm(bof_ctx* ctx, int64_t m_local, int64_t n, int64_t k, float alpha, float beta, const float* a,
                   const int64_t* ia, const int64_t* ja, const float* b, float* c_local);
}

struct bof_mgpu {
  std::vector<bof_ctx*> ctx;
  std::vector<cudaStream_t> push;   // per device: peer copies of the replicated operand
  std::vector<float*> rep;          // per device: the replicated dense operand of the call in flight
  std::string err;
};

namespace {

// run fn(rank) on one thread per device; first failure wins
template <class F>
int for_each_rank(bof_mgpu* mg, F fn) {
  const int world = (int)mg->ctx.size();
  std::vector<int> rc((size_t)world, BOF_OK);
  std::vector<std::thread> th;
  for (int r = 1; r < world; ++r) th.emplace_back([&, r] { rc[r] = fn(r); });
  rc[0] = fn(0);
  for (auto& t : th) t.join();
  for (int r = 0; r < world; ++r)
    if (rc[r] != BOF_OK) {
      mg->err = "rank " + std::to_string(r) + ": " + bof_last_error(mg->ctx[r]);
      return rc[r];
    }
  return BOF_OK;
}

// rows [r0, r1) of rank r: equal shares rounded up to `align` rows
void split_rows(int64_t m, int world, int r, int64_t align, int64_t* r0, int64_t* r1) {
  int64_t per = ceil_div<int64_t>(m, world);
  per = round_up<int64_t>(std::max<int64_t>(per, 1), align);
  *r0 = std::min(m, (int64_t)r * per);
  *r1 = std::min(m, *r0 + per);
}

// rows [r0, r1) of rank r holding ~nnz / world nonzeros (the nnz-budget idea of get_next_blk_size,
// include/blas_utils.h:72-82, at the granularity of a GPU)
void split_nnz(const int64_t* ia, int64_t m, int world, int r, int64_t* r0, int64_t* r1) {
  const int64_t nnz = ia[m] - ia[0];
  auto cut = [&](int g) -> int64_t {
    if (g <= 0) return 0;
    if (g >= world) return m;
    const int64_t target = ia[0] + (int64_t)((__int128)nnz * g / world);
    return std::lower_bound(ia, ia + m + 1, target) - ia;
  };
  *r0 = std::min(cut(r), m);
  *r1 = std::max(*r0, std::min(cut(r + 1), m));
}

// Complete a host matrix of `rows` stored rows x `cols` floats (row pitch `ld`) on every device as a tight
// [rows x cols] array in mg->rep[r]: phase 1 reserves the buffers, phase 2 uploads 1/world of the rows per device
// (in pieces, so that pushes start while the rest uploads) and pushes each piece to every peer.
int replicate_rows(bof_mgpu* mg, const float* src, int64_t rows, int64_t cols, int64_t ld) {
  const int world = (int)mg->ctx.size();
  const size_t count = (size_t)std::max<int64_t>(rows * cols, 1);
  int rc = for_each_rank(mg, [&](int r) {
    bof_ctx* ctx = mg->ctx[r];
    BOF_CUDA(ctx, cudaSetDevice(ctx->device));
    return slot_reserve(ctx, S_DENSE, count, &mg->rep[r]);
  });
  if (rc != BOF_OK || rows == 0 || cols == 0) return rc;
  constexpr int kPieces = 4;
  return for_each_rank(mg, [&](int r) {
    bof_ctx* ctx = mg->ctx[r];
    BOF_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t base = rows / world, rem = rows % world;
    const int64_t r0 = r * base + std::min<int64_t>(r, rem), r1 = r0 + base + (r < rem ? 1 : 0);
    const int64_t per = ceil_div<int64_t>(std::max<int64_t>(r1 - r0, 1), kPieces);
    for (int q = 0; q < kPieces; ++q) {
      const int64_t p0 = std::min(r1, r0 + q * per), p1 = std::min(r1, p0 + per);
      if (p1 <= p0) continue;
      BOF_TRY(copy2d(ctx, mg->rep[r] + p0 * cols, (size_t)cols * 4, src + p0 * ld, (size_t)ld * 4, (size_t)cols * 4,
                     (size_t)(p1 - p0), cudaMemcpyHostToDevice, ctx->h2d));
      cudaEvent_t ev = get_event(ctx, 100 + q);
      BOF_CUDA(ctx, cudaEventRecord(ev, ctx->h2d));
      BOF_CUDA(ctx, cudaStreamWaitEvent(mg->push[r], ev, 0));
      for (int d = 1; d < world; ++d) {
        const int peer = (r + d) % world;   // every device starts with a different peer
        BOF_CUDA(ctx, cudaMemcpyPeerAsync(mg->rep[peer] + p0 * cols, mg->ctx[peer]->device, mg->rep[r] + p0 * cols, ctx->device,
                                          (size_t)(p1 - p0) * cols * 4, mg->push[r]));
      }
    }
    BOF_CUDA(ctx, cudaStreamSynchronize(ctx->h2d));
    BOF_CUDA(ctx, cudaStreamSynchronize(mg->push[r]));
    return (int)BOF_OK;
  });
}

}  // namespace

extern "C" {

int bof_mgpu_create(const bof_config* cfg, int ndev, const int* devices, bof_mgpu** out) {
  if (!out) return BOF_EINVAL;
  *out = nullptr;
  int have = 0;
  if (cudaGetDeviceCount(&have) != cudaSuccess || have == 0) { cudaGetLastError(); return BOF_ENODEV; }
  if (ndev <= 0) ndev = have;
  bof_mgpu* mg = new bof_mgpu();
  for (int i = 0; i < ndev; ++i) {
    bof_config c{};
    if (cfg) c = *cfg;
    c.device = devices ? devices[i] : i;
    bof_ctx* x = nullptr;
    const int rc = bof_ctx_create(&c, &x);
    if (rc != BOF_OK) {
      for (bof_ctx* y : mg->ctx) bof_ctx_destroy(y);
      delete mg;
      return rc;
    }
    mg->ctx.push_back(x);
    cudaStream_t st = nullptr;
    if (cudaSetDevice(c.device) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
      cudaGetLastError();
      for (bof_ctx* y : mg->ctx) bof_ctx_destroy(y);
      delete mg;
      return BOF_ECUDA;
    }
    mg->push.push_back(st);
    mg->rep.push_back(nullptr);
  }
  if (ndev > 1) {
    char id[128];
    int rc = bof_comm_unique_id(id);
    if (rc == BOF_OK) rc = for_each_rank(mg, [&](int r) { return bof_comm_init(mg->ctx[r], ndev, r, id); });
    if (rc != BOF_OK) {
      for (bof_ctx* y : mg->ctx) bof_ctx_destroy(y);
      delete mg;
      return rc;
    }
  }
  *out = mg;
  return BOF_OK;
}

int bof_mgpu_destroy(bof_mgpu* mg) {
  if (!mg) return BOF_OK;
  for (size_t i = 0; i < mg->ctx.size(); ++i) {
    if (i < mg->push.size() && mg->push[i] && cudaSetDevice(mg->ctx[i]->device) == cudaSuccess) cudaStreamDestroy(mg->push[i]);
    bof_ctx_destroy(mg->ctx[i]);
  }
  delete mg;
  return BOF_OK;
}

int bof_mgpu_count(const bof_mgpu* mg) { return mg ? (int)mg->ctx.size() : 0; }
bof_ctx* bof_mgpu_ctx(bof_mgpu* mg, int rank) { return mg && rank >= 0 && rank < (int)mg->ctx.size() ? mg->ctx[rank] : nullptr; }
const char* bof_mgpu_last_error(const bof_mgpu* mg) { return mg ? mg->err.c_str() : ""; }

// flash::gemm over the GPUs: rows of C (row-major) / columns of C (column-major) sharded, the other operand
// replicated by panel broadcast.
int bof_mgpu_gemm(bof_mgpu* mg, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k, float alpha, float beta,
                  const float* a, const float* b, float* c, int64_t lda, int64_t ldb, int64_t ldc) {
  if (!mg || mg->ctx.empty()) return BOF_EINVAL;
  const int world = (int)mg->ctx.size();
  if (world == 1) return bof_host_gemm(mg->ctx[0], ord, ta, tb, m, n, k, alpha, beta, a, b, c, lda, ldb, ldc);
  if (!is_rc(ord) || !is_nt(ta) || !is_nt(tb)) { mg->err = "gemm: mat_ord must be 'R'/'C', trans 'N'/'T'"; return BOF_EINVAL; }
  // column-major gemm(ta, tb, m, n, k, A, B, C) is row-major gemm(tb, ta, n, m, k, B, A, C)
  if (ord == 'C') { std::swap(ta, tb); std::swap(m, n); std::swap(a, b); std::swap(lda, ldb); }
  // row-major from here on: op(A) is m x k, its tight leading dimension k ('N') or m ('T')
  if (lda == 0) lda = ta == 'N' ? k : m;
  if (ldb == 0) ldb = tb == 'N' ? n : k;
  if (ldc == 0) ldc = n;
  // B as stored: k x n ('N') or n x k ('T'); every device gets a tight copy
  const int64_t b_rows = tb == 'N' ? k : n, b_cols = tb == 'N' ? n : k;
  if (int rc = replicate_rows(mg, b, b_rows, b_cols, ldb)) return rc;
  return for_each_rank(mg, [&](int r) {
    int64_t r0, r1;
    split_rows(m, world, r, 256, &r0, &r1);
    if (r1 == r0) return (int)BOF_OK;
    const float* a_loc = ta == 'N' ? a + r0 * lda : a + r0;   // 'T': a column range of the stored k x m matrix
    return bof_host_gemm_devb(mg->ctx[r], ta, tb, r1 - r0, n, k, alpha, beta, a_loc, mg->rep[r], c + r0 * ldc, lda, b_cols, ldc);
  });
}

// flash::csrmm over the GPUs ('N', row-major: nnz-balanced row blocks per GPU; anything else runs on GPU 0)
int bof_mgpu_csrmm(bof_mgpu* mg, char trans_a, int64_t m, int64_t n, int64_t k, float alpha, float beta, const float* a,
                   const int64_t* ia, const int64_t* ja, char ord_b, const float* b, float* c) {
  if (!mg || mg->ctx.empty()) return BOF_EINVAL;
  const int world = (int)mg->ctx.size();
  if (world == 1 || trans_a != 'N' || ord_b != 'R' || m < world)
    return bof_host_csrmm(mg->ctx[0], trans_a, m, n, k, alpha, beta, a, ia, ja, ord_b, b, c);
  if (int rc = replicate_rows(mg, b, n, k, k)) return rc;
  return for_each_rank(mg, [&](int r) {
    int64_t r0, r1;
    split_nnz(ia, m, world, r, &r0, &r1);
    if (r1 == r0) return (int)BOF_OK;
    const int64_t z0 = ia[r0] - ia[0];
    return bof_host_csrmm_devb(mg->ctx[r], r1 - r0, n, k, alpha, beta, a + z0, ia + r0, ja + z0, mg->rep[r], c + r0 * k);
  });
}

// flash::csrgemv over the GPUs.  'N': row blocks, disjoint y.  'T': every GPU produces a full-length partial y from
// its row block; the partials are added on the host in GPU order (deterministic; the reference adds task results
// in completion order under a mutex, include/tasks/csrgemv_task.h:170-176).
int bof_mgpu_csrgemv(bof_mgpu* mg, char trans_a, int64_t m, int64_t n, const float* a, const int64_t* ia,
                     const int64_t* ja, const float* x, float* y) {
  if (!mg || mg->ctx.empty()) return BOF_EINVAL;
  const int world = (int)mg->ctx.size();
  if (world == 1 || !is_nt(trans_a) || m < world) return bof_host_csrgemv(mg->ctx[0], trans_a, m, n, a, ia, ja, x, y);
  std::vector<std::vector<float>> part;
  if (trans_a == 'T') part.assign((size_t)world, std::vector<float>());
  int rc = for_each_rank(mg, [&](int r) {
    int64_t r0, r1;
    split_nnz(ia, m, world, r, &r0, &r1);
    const int64_t z0 = ia[r0] - ia[0];
    if (trans_a == 'N') return bof_host_csrgemv(mg->ctx[r], 'N', r1 - r0, n, a + z0, ia + r0, ja + z0, x, y + r0);
    float* dst = y;
    if (r > 0) { part[r].resize((size_t)n); dst = part[r].data(); }
    return bof_host_csrgemv(mg->ctx[r], 'T', r1 - r0, n, a + z0, ia + r0, ja + z0, x + r0, dst);
  });
  if (rc != BOF_OK || trans_a == 'N') return rc;
  for (int r = 1; r < world; ++r)
    for (int64_t j = 0; j < n; ++j) y[j] += part[r][j];
  return BOF_OK;
}

// flash::gemv over the GPUs: the outputs are split, never the reduction.  Row-dot shapes give each GPU a range of rows
// of the stored matrix, column sums a range of its columns (same lda, offset base); every GPU uploads its own x.
int bof_mgpu_gemv(bof_mgpu* mg, char ord, char trans, int64_t m, int64_t n, float alpha, float beta, const float* a,
                  int64_t lda, const float* x, float* y) {
  if (!mg || mg->ctx.empty()) return BOF_EINVAL;
  const int world = (int)mg->ctx.size();
  GemvCanon c;
  if (int rc = canon_gemv(mg->ctx[0], ord, trans, m, n, lda, &c)) {
    mg->err = bof_last_error(mg->ctx[0]);
    return rc;
  }
  if (world == 1 || c.nout() < world) {
    const int rc = bof_host_gemv(mg->ctx[0], ord, trans, m, n, alpha, beta, a, lda, x, y);
    if (rc != BOF_OK) mg->err = bof_last_error(mg->ctx[0]);
    return rc;
  }
  return for_each_rank(mg, [&](int r) {
    int64_t o0, o1;
    split_rows(c.nout(), world, r, 1, &o0, &o1);
    if (o1 == o0) return (int)BOF_OK;
    // the part as a row-major problem on the stored matrix: ('R','N') is a row-dot, ('R','T') a column sum
    if (c.rowdot)
      return bof_host_gemv(mg->ctx[r], 'R', 'N', o1 - o0, c.cols, alpha, beta, a + o0 * c.ld, c.ld, x, y + o0);
    return bof_host_gemv(mg->ctx[r], 'R', 'T', c.rows, o1 - o0, alpha, beta, a + o0, c.ld, x, y + o0);
  });
}

// `iters` Lloyd iterations (drivers/in_mem_kmeans.cpp:89-152), points sharded over the GPUs and resident, one NCCL
// allreduce of [sums | counts] per iteration.  centers_host: initial centres in, final centres out; assign_out
// (npoints entries, may be NULL): assignment of the last iteration.
int bof_mgpu_kmeans_lloyd(bof_mgpu* mg, int64_t npoints, int64_t ncenters, int64_t dim, const float* points_host,
                          float* centers_host, int64_t iters, int64_t* assign_out) {
  if (!mg || mg->ctx.empty()) return BOF_EINVAL;
  const int world = (int)mg->ctx.size();
  std::vector<float> c0((size_t)ncenters * dim);
  memcpy(c0.data(), centers_host, c0.size() * 4);   // every rank starts from the same centres; rank 0 writes the result
  // phases (see the top of the file): every shard opened (allocations) before the first NCCL kernel is enqueued,
  // every rank's iterations finished before anything is freed
  std::vector<bof_kmeans*> km((size_t)world, nullptr);
  int rc = for_each_rank(mg, [&](int r) {
    int64_t p0, p1;
    split_rows(npoints, world, r, 1, &p0, &p1);
    int rc1 = bof_kmeans_open(mg->ctx[r], p1 - p0, ncenters, dim, points_host + p0 * dim, c0.data(), &km[r]);
    if (rc1 == BOF_OK) rc1 = bof_kmeans_local_step(km[r], nullptr, nullptr);   // warm-up: workspaces and kernels in place
    if (rc1 == BOF_OK && cudaStreamSynchronize(as_stream(bof_kmeans_stream(km[r]))) != cudaSuccess) rc1 = BOF_ECUDA;
    return rc1;
  });
  if (rc == BOF_OK) rc = for_each_rank(mg, [&](int r) {
    int64_t p0, p1;
    split_rows(npoints, world, r, 1, &p0, &p1);
    int rc1 = bof_kmeans_lloyd(km[r], iters);
    if (rc1 == BOF_OK) rc1 = bof_kmeans_get(km[r], r == 0 ? centers_host : nullptr, assign_out ? assign_out + p0 : nullptr);
    return rc1;
  });
  const std::string first_err = mg->err;
  for_each_rank(mg, [&](int r) { if (km[r]) bof_kmeans_close(km[r]); return (int)BOF_OK; });
  if (rc != BOF_OK) mg->err = first_err;
  return rc;
}

}  // extern "C"
