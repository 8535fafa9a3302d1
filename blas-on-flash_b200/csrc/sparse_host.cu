// flash::csrmm / csrgemv / csrcsc on the host side: nnz-budgeted row blocks streamed through the GPU, and the
// resident-CSR handle (A kept in HBM across calls).  Reference: src/blas/csrmm.cpp, src/blas/csrgemv.cpp,
// src/blas/csrcsc.cpp, include/tasks/{csrmm,csrgemv,csrcsc}_task.h.
#include "host_internal.cuh"

#include <memory>

namespace bof {

constexpr cudaMemcpyKind H2D = cudaMemcpyHostToDevice, D2H = cudaMemcpyDeviceToHost;

// Event ids of the sparse host calls: + g per block generation, + gp per B panel, + q per piece of an exchanged B.
// No two of these calls run at once, so bof_csr_mm and csrcsc reuse the numbers of the streamed csrmm.
constexpr int kBPieces = 4;  // pieces of a rank's own rows of an exchanged B
enum SparseEvent : int {
  EV_B = 0,                              // dense operand uploaded (B of csrmm, x of csrgemv)
  EV_A = 1,                              // csrmm('T'): A uploaded for the device transpose
  EV_C0 = 2,                             // csrmm('T'): old C uploaded
  EV_UP = 4, EV_DONE = 6, EV_DOWN = 8,   // inputs of a block uploaded; its C rows computed; its C rows downloaded
  EV_PIECE = 100,                        // collective csrmm: own piece q of B uploaded
  EV_PAN = 0, EV_PAN_FREE = 2,           // bof_csr_mm: B panel uploaded; B panel consumed
  EV_CSC_A = 0, EV_CSC_T = 1,            // csrcsc: A uploaded; A^T built and widened
};
static_assert(EV_B < EV_A && EV_A < EV_C0 && EV_C0 < EV_UP && EV_UP + 2 <= EV_DONE && EV_DONE + 2 <= EV_DOWN &&
              EV_DOWN + 2 <= EV_PIECE, "csrmm / csrgemv: event ranges overlap");
static_assert(EV_PAN + 2 <= EV_PAN_FREE && EV_PAN_FREE + 2 <= EV_UP, "bof_csr_mm: event ranges overlap");

// Row-block partition by nnz budget (the idea of get_next_blk_size, include/blas_utils.h:72-82):
// blocks[i] .. blocks[i+1] are the rows of block i.
static std::vector<int64_t> partition_rows(const int64_t* ia, int64_t m, int64_t max_nnz) {
  std::vector<int64_t> cuts{0};
  int64_t r = 0;
  while (r < m) {
    const int64_t limit = ia[r] + max_nnz;
    int64_t e = std::upper_bound(ia + r + 1, ia + m + 1, limit) - ia - 1;  // last e with ia[e] <= limit
    if (e <= r) e = r + 1;  // a single row above the budget still forms a block
    cuts.push_back(e);
    r = e;
  }
  return cuts;
}

// A CSR matrix on the device with int32 column indices.
struct DevCsr { const int64_t* offs; const int32_t* idx; const float* vals; };

// The row blocks in which csrmm('N') and csrgemv stream A: block i is rows [cuts[i], cuts[i + 1]) and lands in
// generation i & 1 of the device buffers, which are sized for the largest block.
struct RowBlocks {
  std::vector<int64_t> cuts;
  int64_t max_rows = 1, max_nnz = 1;
  int64_t* offs[2]; int64_t* idx64[2]; int32_t* idx32[2]; float* vals[2];
  int count() const { return (int)cuts.size() - 1; }
};

static int plan_row_blocks(bof_ctx* ctx, const int64_t* ia, int64_t m, RowBlocks* rb) {
  const int64_t nnz = ia[m] - ia[0];
  int64_t budget = (int64_t)ctx->cfg.csrmm_max_nnz;
  budget = std::min(budget, std::max<int64_t>(nnz / 8, 1 << 20));  // >= 8 blocks when the matrix is big enough
  rb->cuts = partition_rows(ia, m, budget);
  for (int i = 0; i < rb->count(); ++i) {
    rb->max_rows = std::max(rb->max_rows, rb->cuts[i + 1] - rb->cuts[i]);
    rb->max_nnz = std::max(rb->max_nnz, ia[rb->cuts[i + 1]] - ia[rb->cuts[i]]);
  }
  for (int g = 0; g < 2; ++g) {
    BOF_TRY(slot_reserve(ctx, S_OFFS + g, (size_t)rb->max_rows + 1, &rb->offs[g]));
    BOF_TRY(slot_reserve(ctx, S_IDX64 + g, (size_t)rb->max_nnz, &rb->idx64[g]));
    BOF_TRY(slot_reserve(ctx, S_IDX32 + g, (size_t)rb->max_nnz, &rb->idx32[g]));
    BOF_TRY(slot_reserve(ctx, S_VALS + g, (size_t)rb->max_nnz, &rb->vals[g]));
  }
  return BOF_OK;
}

// Block i of A into its generation on the h2d stream; the caller narrows its indices once they have landed.
static int upload_a_block(bof_ctx* ctx, const RowBlocks& rb, int i, const float* a, const int64_t* ia, const int64_t* ja) {
  const int g = i & 1;
  const int64_t r0 = rb.cuts[i], r1 = rb.cuts[i + 1], z0 = ia[r0] - ia[0], bnnz = ia[r1] - ia[r0];
  BOF_TRY(copy1d(ctx, rb.offs[g], ia + r0, (size_t)(r1 - r0 + 1) * 8, H2D, ctx->h2d));
  BOF_TRY(copy1d(ctx, rb.idx64[g], ja + z0, (size_t)bnnz * 8, H2D, ctx->h2d));
  return copy1d(ctx, rb.vals[g], a + z0, (size_t)bnnz * 4, H2D, ctx->h2d);
}

// A^T of the device CSR A [m x n] into (offs_t, idx_t, vals_t) on the compute stream, with its workspace in S_WS.
static int transpose_csr(bof_ctx* ctx, int64_t m, int64_t n, int64_t nnz, const int64_t* offs, const int32_t* idx,
                         const float* vals, int64_t* offs_t, int32_t* idx_t, float* vals_t) {
  void* ws;
  const size_t wsb = csr2csc_workspace_bytes(m, n, nnz);
  BOF_TRY(slot_reserve(ctx, S_WS, wsb, &ws));
  return launch_csr2csc(ctx, ctx->compute, m, n, nnz, offs, idx, vals, offs_t, idx_t, vals_t, ws, wsb);
}

// A^T (K6) of the host CSR A [m x n] in S_OUT0..2: A is uploaded whole (event ev_up), narrowed and transposed on the
// compute stream.  Its int64 indices are staged in S_IDX64, which is free again once the transpose has run.
static int upload_transposed(bof_ctx* ctx, int64_t m, int64_t n, int64_t nnz, const float* a, const int64_t* ia,
                             const int64_t* ja, int ev_up, DevCsr* at) {
  const size_t z = (size_t)std::max<int64_t>(nnz, 1);
  int64_t *offs_d, *offs_t, *idx64;
  int32_t *idx32, *idx_t;
  float *vals_d, *vals_t;
  BOF_TRY(slot_reserve(ctx, S_OFFS, (size_t)m + 1, &offs_d));
  BOF_TRY(slot_reserve(ctx, S_IDX64, z, &idx64));
  BOF_TRY(slot_reserve(ctx, S_IDX32, z, &idx32));
  BOF_TRY(slot_reserve(ctx, S_VALS, z, &vals_d));
  BOF_TRY(slot_reserve(ctx, S_OUT0, (size_t)n + 1, &offs_t));
  BOF_TRY(slot_reserve(ctx, S_OUT1, z, &idx_t));
  BOF_TRY(slot_reserve(ctx, S_OUT2, z, &vals_t));
  BOF_TRY(copy1d(ctx, offs_d, ia, (size_t)(m + 1) * 8, H2D, ctx->h2d));
  BOF_TRY(copy1d(ctx, idx64, ja, (size_t)nnz * 8, H2D, ctx->h2d));
  BOF_TRY(copy1d(ctx, vals_d, a, (size_t)nnz * 4, H2D, ctx->h2d));
  BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, ev_up), ctx->h2d));
  BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, ev_up), 0));
  BOF_TRY(launch_idx_narrow(ctx, ctx->compute, idx64, idx32, nnz));
  BOF_TRY(transpose_csr(ctx, m, n, nnz, offs_d, idx32, vals_d, offs_t, idx_t, vals_t));
  *at = DevCsr{offs_t, idx_t, vals_t};
  return BOF_OK;
}

// Host C of a csrmm: row-major with pitch ld, or column-major with pitch ld (its row count).  The block of rows
// [r0, r0 + rows) x columns [j0, j0 + w) lies on the device tight: [rows x w], or [w x rows] for a column-major C.
struct HostC { float* c; int64_t ld; bool colmaj; };

static int upload_c_block(bof_ctx* ctx, const HostC& hc, int64_t r0, int64_t rows, int64_t j0, int64_t w, float* blk) {
  if (hc.colmaj)
    return copy2d(ctx, blk, (size_t)rows * 4, hc.c + j0 * hc.ld + r0, (size_t)hc.ld * 4, (size_t)rows * 4, (size_t)w, H2D, ctx->h2d);
  return copy2d(ctx, blk, (size_t)w * 4, hc.c + r0 * hc.ld + j0, (size_t)hc.ld * 4, (size_t)w * 4, (size_t)rows, H2D, ctx->h2d);
}

// The same block from the device to the host C, on the d2h stream (see d2h_transfer for the events and the ticket).
static int download_c_block(bof_ctx* ctx, const HostC& hc, int64_t r0, int64_t rows, int64_t j0, int64_t w,
                            const float* blk, cudaEvent_t wait_ev, cudaEvent_t record_ev, uint64_t* ticket) {
  if (hc.colmaj)
    return d2h_transfer(ctx, hc.c + j0 * hc.ld + r0, (size_t)hc.ld * 4, blk, (size_t)rows * 4, (size_t)rows * 4, (size_t)w,
                        ctx->d2h, wait_ev, record_ev, ticket);
  return d2h_transfer(ctx, hc.c + r0 * hc.ld + j0, (size_t)hc.ld * 4, blk, (size_t)w * 4, (size_t)w * 4, (size_t)rows,
                      ctx->d2h, wait_ev, record_ev, ticket);
}

// C block [rows x w] = alpha A_blk B + beta C block on the compute stream, B [b_rows x w] row-major.  A column-major
// C (cblk_t != nullptr) is computed into cblk and transposed into cblk_t [w x rows], which holds the old C block.
static int spmm_c_block(bof_ctx* ctx, int64_t rows, int64_t w, float alpha, const DevCsr& a, const float* B,
                        int64_t b_rows, float beta, float* cblk, float* cblk_t) {
  if (cblk_t == nullptr)
    return launch_spmm_rm(ctx, ctx->compute, rows, w, alpha, a.vals, a.idx, a.offs, B, w, beta, cblk, w, b_rows);
  BOF_TRY(launch_spmm_rm(ctx, ctx->compute, rows, w, 1.f, a.vals, a.idx, a.offs, B, w, 0.f, cblk, w, b_rows));
  return launch_transpose_axpby(ctx, ctx->compute, rows, w, alpha, cblk, w, beta, cblk_t, rows);
}

// bof_dist_csrmm: B [in_rows x k] is replicated over the ranks.  Every rank uploads rows [r0, r1) of it (1/world of
// the PCIe traffic) in a few pieces and pushes each piece into every peer's exchange buffer Bd with copy-engine peer
// copies over NVLink as soon as it has landed; meanwhile this rank's first A blocks upload behind the slice.  The
// SpMM gathers arbitrary rows of B, so the compute stream waits for every piece of every rank.
static int exchange_dense(bof_ctx* ctx, const float* b, int64_t in_rows, int64_t k, float* Bd) {
  const int world = comm_world(ctx), rank = comm_rank(ctx);
  auto piece = [&](int r, int q, int64_t* p0, int64_t* p1) {   // rows [p0, p1) of B: piece q of rank r's shard
    const int64_t base = in_rows / world, rem = in_rows % world;
    const int64_t r0 = r * base + std::min<int64_t>(r, rem), r1 = r0 + base + (r < rem ? 1 : 0);
    const int64_t per = ceil_div<int64_t>(r1 - r0, kBPieces);
    *p0 = std::min(r1, r0 + q * per);
    *p1 = std::min(r1, *p0 + per);
  };
  for (int q = 0; q < kBPieces; ++q) {
    int64_t p0, p1;
    piece(rank, q, &p0, &p1);
    if (p1 <= p0) continue;
    BOF_TRY(copy1d(ctx, Bd + p0 * k, b + p0 * k, (size_t)(p1 - p0) * k * 4, H2D, ctx->h2d));
    cudaEvent_t ev_own = get_event(ctx, EV_PIECE + q);
    BOF_CUDA(ctx, cudaEventRecord(ev_own, ctx->h2d));
    BOF_TRY(comm_push(ctx, (size_t)(p0 * k), (size_t)(p1 - p0) * k, rank * kBPieces + q, ev_own));
    if (q == kBPieces - 1) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, ev_own, 0));
  }
  trace_mark(ctx, ctx->h2d, "h2d: own slice of the dense operand landed", rank);
  for (int src = 0; src < world; ++src) {
    if (src == rank) continue;
    for (int q = 0; q < kBPieces; ++q) {
      int64_t p0, p1;
      piece(src, q, &p0, &p1);
      if (p1 > p0) BOF_TRY(comm_wait_item(ctx, ctx->compute, src * kBPieces + q));
    }
  }
  trace_mark(ctx, ctx->compute, "compute: dense operand complete on this rank", 0);
  return BOF_OK;
}

// csrmm's B [in_rows x k] row-major on the device for the compute stream: b_dev as it is, exchanged by a collective
// call, or uploaded from a host B, column-major or row-major with pitch ldb.
static int upload_dense(bof_ctx* ctx, const float* b, const float* b_dev, bool collective, bool colmaj, int64_t in_rows,
                        int64_t k, int64_t ldb, float** Bd) {
  if (b_dev != nullptr) {
    *Bd = const_cast<float*>(b_dev);  // already in HBM (e.g. all-gathered over NVLink); read-only here
    return BOF_OK;
  }
  if (collective) {
    BOF_TRY(comm_exchange_begin(ctx, (size_t)in_rows * k * sizeof(float), Bd));   // the buffer the peers push into
    return exchange_dense(ctx, b, in_rows, k, *Bd);
  }
  BOF_TRY(slot_reserve(ctx, S_DENSE, (size_t)in_rows * k, Bd));
  float* Braw = nullptr;
  if (colmaj) {
    BOF_TRY(slot_reserve(ctx, S_DENSE_T, (size_t)in_rows * k, &Braw));
    BOF_TRY(copy1d(ctx, Braw, b, (size_t)in_rows * k * 4, H2D, ctx->h2d));
  } else {
    BOF_TRY(copy2d(ctx, *Bd, (size_t)k * 4, b, (size_t)ldb * 4, (size_t)k * 4, (size_t)in_rows, H2D, ctx->h2d));
  }
  BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_B), ctx->h2d));
  BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_B), 0));
  if (colmaj) BOF_TRY(launch_transpose(ctx, ctx->compute, k, in_rows, Braw, in_rows, *Bd, k));
  return BOF_OK;
}

// csrmm('T'): A^T in CSR on the device, then the no-transpose kernel on its n rows into the whole C [n x k] on the
// device (beta needs the old C).
static int csrmm_transposed(bof_ctx* ctx, int64_t m, int64_t n, int64_t k, float alpha, float beta, const float* a,
                            const int64_t* ia, const int64_t* ja, const float* Bd, float* c, bool colmaj) {
  const int64_t nnz = ia[m] - ia[0];
  BOF_REQUIRE(ctx, nnz < (1ll << 31), "csrmm('T'): nnz must be below 2^31");
  DevCsr at;
  BOF_TRY(upload_transposed(ctx, m, n, nnz, a, ia, ja, EV_A, &at));
  float *Cd, *Ccm = nullptr;
  BOF_TRY(slot_reserve(ctx, S_CBLK, (size_t)n * k, &Cd));
  if (colmaj) BOF_TRY(slot_reserve(ctx, S_CBLK_T, (size_t)n * k, &Ccm));
  float* Cio = colmaj ? Ccm : Cd;  // what is copied from/to the host
  if (beta != 0.f) {
    BOF_TRY(copy1d(ctx, Cio, c, (size_t)n * k * 4, H2D, ctx->h2d));
    BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_C0), ctx->h2d));
    BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_C0), 0));
  }
  BOF_TRY(spmm_c_block(ctx, n, k, alpha, at, Bd, m, beta, Cd, Ccm));
  BOF_TRY(copy1d(ctx, c, Cio, (size_t)n * k * 4, D2H, ctx->compute));
  return sync_all(ctx);
}

// csrmm('N'): A streams in row blocks, C block by block.  Software-pipelined issue order: block i+1 is uploaded and
// launched before block i is downloaded, so a (host-blocking) staged download of block i overlaps the kernel of
// block i+1 and the copy engines never wait on the host.
static int csrmm_streamed(bof_ctx* ctx, int64_t m, int64_t n, int64_t k, float alpha, float beta, const float* a,
                          const int64_t* ia, const int64_t* ja, const float* Bd, const HostC& hc) {
  RowBlocks rb;
  BOF_TRY(plan_row_blocks(ctx, ia, m, &rb));
  float* cblk[2]; float* cblk_t[2] = {nullptr, nullptr};
  for (int g = 0; g < 2; ++g) {
    BOF_TRY(slot_reserve(ctx, S_CBLK + g, (size_t)rb.max_rows * k, &cblk[g]));
    if (hc.colmaj) BOF_TRY(slot_reserve(ctx, S_CBLK_T + g, (size_t)rb.max_rows * k, &cblk_t[g]));
  }
  bool used[2] = {false, false};
  uint64_t down_ticket[2] = {0, 0};  // pageable C: the drainer enqueues the download and records ev_down
  auto stage_block = [&](int i) -> int {
    const int g = i & 1;
    const int64_t r0 = rb.cuts[i], r1 = rb.cuts[i + 1], rows = r1 - r0;
    cudaEvent_t ev_up = get_event(ctx, EV_UP + g), ev_done = get_event(ctx, EV_DONE + g), ev_down = get_event(ctx, EV_DOWN + g);
    if (used[g]) {
      d2h_fence(ctx, down_ticket[g]);  // ev_down of block i-2 has been recorded (and ev_done may be re-recorded)
      BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, ev_done, 0));   // inputs of block i-2 consumed
      // Only an upload of old C rows (beta != 0) touches the C buffer from this stream; waiting for the download
      // unconditionally idled the H2D engine ~9 ms every other block (BOF_TRACE timeline, cfg-3: 419 -> 37x ms).
      if (beta != 0.f) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, ev_down, 0));   // its C rows left the device
    }
    BOF_TRY(upload_a_block(ctx, rb, i, a, ia, ja));
    if (beta != 0.f) BOF_TRY(upload_c_block(ctx, hc, r0, rows, 0, k, hc.colmaj ? cblk_t[g] : cblk[g]));
    BOF_CUDA(ctx, cudaEventRecord(ev_up, ctx->h2d));
    trace_mark(ctx, ctx->h2d, "h2d: A block landed", i);
    BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, ev_up, 0));
    if (used[g]) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, ev_down, 0));
    trace_mark(ctx, ctx->compute, "compute: block start", i);
    BOF_TRY(launch_idx_narrow(ctx, ctx->compute, rb.idx64[g], rb.idx32[g], ia[r1] - ia[r0]));
    BOF_TRY(spmm_c_block(ctx, rows, k, alpha, DevCsr{rb.offs[g], rb.idx32[g], rb.vals[g]}, Bd, n, beta, cblk[g], cblk_t[g]));
    BOF_CUDA(ctx, cudaEventRecord(ev_done, ctx->compute));
    trace_mark(ctx, ctx->compute, "compute: block end", i);
    used[g] = true;
    return BOF_OK;
  };
  const int nblk = rb.count();
  if (nblk > 0) BOF_TRY(stage_block(0));
  for (int i = 0; i < nblk; ++i) {
    if (i + 1 < nblk) BOF_TRY(stage_block(i + 1));
    const int g = i & 1;
    BOF_TRY(download_c_block(ctx, hc, rb.cuts[i], rb.cuts[i + 1] - rb.cuts[i], 0, k, hc.colmaj ? cblk_t[g] : cblk[g],
                             get_event(ctx, EV_DONE + g), get_event(ctx, EV_DOWN + g), &down_ticket[g]));
    trace_mark(ctx, ctx->d2h, "d2h: C block downloaded", i);
  }
  BOF_TRY(sync_all(ctx));
  trace_dump(ctx, "bof_host_csrmm");
  return BOF_OK;
}

}  // namespace bof

using namespace bof;

extern "C" {

static int host_csrmm_impl(bof_ctx* ctx, char trans_a, int64_t m, int64_t n, int64_t k, float alpha, float beta,
                           const float* a, const int64_t* ia, const int64_t* ja, char ord_b, const float* b, float* c,
                           const float* b_dev, bool dist_b = false, int64_t ldk = 0) {
  // ldk: leading dimension of the host B and C when this call works on a column panel of a wider product
  // (row-major, trans_a = 'N' only); 0 = tight (k)
  if (!ctx) return BOF_EINVAL;
  if (ldk == 0) ldk = k;
  BOF_REQUIRE(ctx, is_nt(trans_a), "csrmm: unrecognized value for param trans_a = '%c'", trans_a);
  BOF_REQUIRE(ctx, b_dev == nullptr || (trans_a == 'N' && ord_b == 'R'),
              "csrmm: a device-resident B is supported for trans_a='N', ord_b='R' only");
  BOF_REQUIRE(ctx, is_rc(ord_b), "csrmm: unrecognized value for param ord_b = '%c'", ord_b);
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && k >= 0 && m < (1ll << 31) && n < (1ll << 31), "csrmm: bad dimension");
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  trace_mark(ctx, ctx->h2d, "start", 0);
  const int64_t out_rows = trans_a == 'N' ? m : n;   // rows of C
  const int64_t in_rows = trans_a == 'N' ? n : m;    // rows of B
  // a collective call (bof_dist_csrmm) exchanges the dense operand on every rank, also on one that owns no rows of C
  const bool collective = dist_b && comm_world(ctx) > 1;
  if (k == 0 || (out_rows == 0 && !collective)) { stats_end(ctx); return call_guard.done(); }
  const bool colmaj = ord_b == 'C';
  float* Bd = nullptr;
  BOF_TRY(upload_dense(ctx, b, b_dev, collective, colmaj, in_rows, k, ldk, &Bd));
  if (out_rows == 0) {   // collective call, empty shard: my slice has been pushed and the peers' slices have arrived
    BOF_TRY(sync_all(ctx));
  } else {
    trace_mark(ctx, ctx->h2d, "h2d: dense operand landed", 0);
    if (trans_a == 'T') BOF_TRY(csrmm_transposed(ctx, m, n, k, alpha, beta, a, ia, ja, Bd, c, colmaj));
    else BOF_TRY(csrmm_streamed(ctx, m, n, k, alpha, beta, a, ia, ja, Bd, HostC{c, colmaj ? m : ldk, colmaj}));
  }
  stats_end(ctx);
  return call_guard.done();
}

// Widest column panel of B the device can hold next to the streamed blocks (0: the whole B fits).  The reference cuts B
// into column blocks of CSRMM_RM_CBLK_SIZE = 1024 for the same reason, a memory budget (src/blas/csrmm.cpp:64-126,
// include/tasks/csrmm_task.h:175-199); here the budget is HBM, and A is re-streamed once per panel.
static int64_t csrmm_column_panel(bof_ctx* ctx, int64_t in_rows, int64_t k) {
  static const int64_t forced = getenv("BOF_CSRMM_KPANEL") ? atoll(getenv("BOF_CSRMM_KPANEL")) : 0;   // test knob
  if (forced > 0) return forced < k ? forced : 0;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return 0; }
  const double budget = 0.6 * (double)total_b;
  if ((double)in_rows * k * 4 <= budget) return 0;
  int64_t kp = (int64_t)(budget / ((double)in_rows * 4));
  kp = (kp / 32) * 32;
  (void)ctx;
  return kp >= 32 ? kp : 32;
}

int bof_host_csrmm(bof_ctx* ctx, char trans_a, int64_t m, int64_t n, int64_t k, float alpha, float beta,
                   const float* a, const int64_t* ia, const int64_t* ja, char ord_b, const float* b, float* c) {
  if (ctx && trans_a == 'N' && ord_b == 'R' && m >= 0 && n > 0 && k > 0) {
    cudaSetDevice(ctx->device);
    const int64_t kp = csrmm_column_panel(ctx, n, k);
    if (kp > 0) {   // B does not fit in HBM: one pass over A per column panel of B and C
      bof_stats sum{};
      for (int64_t c0 = 0; c0 < k; c0 += kp) {
        const int rc = host_csrmm_impl(ctx, 'N', m, n, std::min(kp, k - c0), alpha, beta, a, ia, ja, 'R', b + c0, c + c0, nullptr,
                                       false, k);
        if (rc != BOF_OK) return rc;
        const bof_stats& st = ctx->stats;   // bof_get_stats reports the whole call, not the last panel
        sum.h2d_bytes += st.h2d_bytes; sum.d2h_bytes += st.d2h_bytes; sum.stage_in_ms += st.stage_in_ms;
        sum.stage_out_ms += st.stage_out_ms; sum.total_ms += st.total_ms; sum.kernel_launches += st.kernel_launches;
        sum.kernel_ms = st.kernel_ms;
      }
      ctx->stats = sum;
      return BOF_OK;
    }
  }
  return host_csrmm_impl(ctx, trans_a, m, n, k, alpha, beta, a, ia, ja, ord_b, b, c, nullptr);
}

int bof_host_csrmm_devb(bof_ctx* ctx, int64_t m, int64_t n, int64_t k, float alpha, float beta, const float* a,
                        const int64_t* ia, const int64_t* ja, const float* b_dev, float* c) {
  if (ctx && b_dev == nullptr) return fail(ctx, BOF_EINVAL, "csrmm_devb: b_dev is null");
  return host_csrmm_impl(ctx, 'N', m, n, k, alpha, beta, a, ia, ja, 'R', nullptr, c, b_dev);
}

int bof_dist_csrmm(bof_ctx* ctx, int64_t m_local, int64_t n, int64_t k, float alpha, float beta, const float* a,
                   const int64_t* ia, const int64_t* ja, const float* b, float* c_local) {
  return host_csrmm_impl(ctx, 'N', m_local, n, k, alpha, beta, a, ia, ja, 'R', b, c_local, nullptr, true);
}

// flash::csrgemv: x resident, A streams in row blocks; 'N' writes disjoint y rows, 'T' accumulates
// every block into the full y on the device (zeroed once, as src/blas/csrgemv.cpp:64 does).
int bof_host_csrgemv(bof_ctx* ctx, char trans_a, int64_t m, int64_t n, const float* a, const int64_t* ia,
                     const int64_t* ja, const float* b, float* c) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, is_nt(trans_a), "csrgemv trans_a error : expected=N or T, found=%c", trans_a);
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && m < (1ll << 31) && n < (1ll << 31), "csrgemv: bad dimension");
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  const bool tr = trans_a == 'T';
  const int64_t xlen = tr ? m : n, ylen = tr ? n : m;
  if (ylen == 0) { stats_end(ctx); return call_guard.done(); }
  float *xd, *yd;
  BOF_TRY(slot_reserve(ctx, S_DENSE, (size_t)std::max<int64_t>(xlen, 1), &xd));
  BOF_TRY(slot_reserve(ctx, S_CBLK, (size_t)ylen, &yd));
  BOF_TRY(copy1d(ctx, xd, b, (size_t)xlen * 4, H2D, ctx->h2d));
  BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_B), ctx->h2d));
  BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_B), 0));
  BOF_CUDA(ctx, cudaMemsetAsync(yd, 0, (size_t)ylen * 4, ctx->compute));

  RowBlocks rb;
  BOF_TRY(plan_row_blocks(ctx, ia, m, &rb));
  if (tr && ctx->cfg.spmv_t_atomic == 0) {   // workspace of the sorted A^T x path for the largest block, before the pipeline starts
    void* wsp = nullptr;
    BOF_TRY(slot_reserve(ctx, kSlotSpmvT, spmv_t_workspace_bytes(n, rb.max_nnz), &wsp));
  }
  bool used[2] = {false, false};
  for (int i = 0; i < rb.count(); ++i) {
    const int g = i & 1;
    const int64_t r0 = rb.cuts[i], r1 = rb.cuts[i + 1], rows = r1 - r0, bnnz = ia[r1] - ia[r0];
    cudaEvent_t ev_up = get_event(ctx, EV_UP + g), ev_done = get_event(ctx, EV_DONE + g);
    if (used[g]) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, ev_done, 0));
    BOF_TRY(upload_a_block(ctx, rb, i, a, ia, ja));
    BOF_CUDA(ctx, cudaEventRecord(ev_up, ctx->h2d));
    BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, ev_up, 0));
    BOF_TRY(launch_idx_narrow(ctx, ctx->compute, rb.idx64[g], rb.idx32[g], bnnz));
    if (!tr) {
      BOF_TRY(launch_spmv(ctx, ctx->compute, 'N', rows, n, rb.vals[g], rb.idx32[g], rb.offs[g], xd, yd + r0));
    } else {
      // y += A_blk^T x_blk : launch the accumulate kernel directly (y was zeroed once above)
      BOF_TRY(launch_spmv(ctx, ctx->compute, 't', rows, n, rb.vals[g], rb.idx32[g], rb.offs[g], xd + r0, yd, bnnz));
    }
    BOF_CUDA(ctx, cudaEventRecord(ev_done, ctx->compute));
    used[g] = true;
  }
  BOF_TRY(copy1d(ctx, c, yd, (size_t)ylen * 4, D2H, ctx->compute));
  BOF_TRY(sync_all(ctx));
  stats_end(ctx);
  return call_guard.done();
}

// flash::csrcsc: the whole matrix is transposed in HBM in one shot (the reference's two-phase
// row-block transpose + column-block merge exists only because a block had to fit in DRAM).
int bof_host_csrcsc(bof_ctx* ctx, int64_t m, int64_t n, const int64_t* ia, const int64_t* ja, const float* a,
                    int64_t* ia_tr, int64_t* ja_tr, float* a_tr) {
  if (!ctx) return BOF_EINVAL;
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && m < (1ll << 31) && n < (1ll << 31), "csrcsc: bad dimension");
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  const int64_t nnz = ia[m] - ia[0];
  BOF_REQUIRE(ctx, nnz >= 0 && nnz < (1ll << 31), "csrcsc: nnz must be in [0, 2^31)");
  DevCsr at;
  BOF_TRY(upload_transposed(ctx, m, n, nnz, a, ia, ja, EV_CSC_A, &at));
  // the int64 staging buffer of the input indices is free again: reuse it for the widened output
  int64_t* idx64 = static_cast<int64_t*>(ctx->slot_ptr[S_IDX64]);
  BOF_TRY(launch_idx_widen(ctx, ctx->compute, at.idx, idx64, nnz));
  BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_CSC_T), ctx->compute));
  BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->d2h, get_event(ctx, EV_CSC_T), 0));
  // values ride a second stream so that both copy engines' queues stay busy
  BOF_TRY(copy1d(ctx, a_tr, at.vals, (size_t)nnz * 4, D2H, ctx->d2h));
  BOF_TRY(copy1d(ctx, ja_tr, idx64, (size_t)nnz * 8, D2H, ctx->compute));
  BOF_TRY(copy1d(ctx, ia_tr, at.offs, (size_t)(n + 1) * 8, D2H, ctx->compute));  // offsets last, as csrcsc.cpp:150
  BOF_TRY(sync_all(ctx));
  stats_end(ctx);
  return call_guard.done();
}

// ---- resident CSR: A stays in HBM across calls (SURVEY 8(f)-2) -----------------------------------
// The reference re-reads A from flash on every flash::csrmm / flash::csrgemv call (its Cache is flushed when a
// kernel returns, src/blas/csrmm.cpp:259); the Krylov / eigensolver loops that call them re-multiply the same A.
// A bof_csr uploads A once (indices narrowed to int32), optionally keeps A^T next to it, and each product then
// moves only the dense operands over PCIe.

struct bof_csr {
  bof_ctx* ctx = nullptr;
  int64_t m = 0, n = 0, nnz = 0;
  // [0] = A (m rows), [1] = A^T in CSR (n rows), built on first use
  float* vals[2] = {nullptr, nullptr};
  int32_t* idx[2] = {nullptr, nullptr};
  int64_t* offs[2] = {nullptr, nullptr};
  std::vector<int64_t> offs_host[2];
  bool have_t = false;
};

static void csr_free(bof_csr* h) {
  if (!h) return;
  for (int t = 0; t < 2; ++t) {
    if (h->vals[t]) cudaFree(h->vals[t]);
    if (h->idx[t]) cudaFree(h->idx[t]);
    if (h->offs[t]) cudaFree(h->offs[t]);
  }
  delete h;
}

static int csr_alloc(bof_ctx* ctx, bof_csr* h, int t, int64_t rows) {
  const size_t z = (size_t)std::max<int64_t>(h->nnz, 1);
  struct Req { void** p; size_t bytes; } reqs[] = {
      {(void**)&h->vals[t], z * 4}, {(void**)&h->idx[t], z * 4}, {(void**)&h->offs[t], (size_t)(rows + 1) * 8}};
  for (auto& r : reqs) {
    if (cudaMalloc(r.p, r.bytes) != cudaSuccess) {
      cudaGetLastError();
      return fail(ctx, BOF_ENOMEM, "csr: cudaMalloc of %zu bytes failed", r.bytes);
    }
  }
  return BOF_OK;
}

int bof_csr_open(bof_ctx* ctx, int64_t m, int64_t n, const float* a, const int64_t* ia, const int64_t* ja,
                 bof_csr** out) {
  if (!ctx || !out) return BOF_EINVAL;
  *out = nullptr;
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && m < (1ll << 31) && n < (1ll << 31), "csr_open: bad dimension");
  BOF_REQUIRE(ctx, ia != nullptr, "csr_open: ia is null");
  const int64_t nnz = ia[m] - ia[0];
  BOF_REQUIRE(ctx, nnz >= 0 && nnz < (1ll << 31), "csr_open: nnz must be in [0, 2^31)");
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  // declared before the guard, so that a failed call quiesces the streams before the handle's memory is freed
  std::unique_ptr<bof_csr, void (*)(bof_csr*)> h(new bof_csr(), csr_free);
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  h->ctx = ctx; h->m = m; h->n = n; h->nnz = nnz;
  BOF_TRY(csr_alloc(ctx, h.get(), 0, m));
  h->offs_host[0].assign(ia, ia + m + 1);
  BOF_TRY(copy1d(ctx, h->offs[0], ia, (size_t)(m + 1) * 8, H2D, ctx->h2d));
  BOF_TRY(copy1d(ctx, h->vals[0], a, (size_t)nnz * 4, H2D, ctx->h2d));
  // int64 column indices cross PCIe as they are on disk and are narrowed chunk by chunk (two staging generations)
  const int64_t chunk = std::max<int64_t>(std::min<int64_t>((int64_t)ctx->cfg.csrmm_max_nnz, nnz), 1);
  int64_t* st[2];
  for (int g = 0; g < 2; ++g) BOF_TRY(slot_reserve(ctx, S_IDX64 + g, (size_t)chunk, &st[g]));
  bool used[2] = {false, false};
  int ci = 0;
  for (int64_t z = 0; z < nnz; z += chunk, ++ci) {
    const int g = ci & 1;
    const int64_t cnt = std::min(chunk, nnz - z);
    cudaEvent_t ev_up = get_event(ctx, EV_UP + g), ev_done = get_event(ctx, EV_DONE + g);
    if (used[g]) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, ev_done, 0));
    BOF_TRY(copy1d(ctx, st[g], ja + z, (size_t)cnt * 8, H2D, ctx->h2d));
    BOF_CUDA(ctx, cudaEventRecord(ev_up, ctx->h2d));
    BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, ev_up, 0));
    BOF_TRY(launch_idx_narrow(ctx, ctx->compute, st[g], h->idx[0] + z, cnt));
    BOF_CUDA(ctx, cudaEventRecord(ev_done, ctx->compute));
    used[g] = true;
  }
  BOF_TRY(sync_all(ctx));
  stats_end(ctx);
  *out = h.release();
  return call_guard.done();
}

int bof_csr_build_transpose(bof_csr* h) {
  if (!h) return BOF_EINVAL;
  if (h->have_t) return BOF_OK;
  bof_ctx* ctx = h->ctx;
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  CallGuard call_guard(ctx);
  BOF_TRY(csr_alloc(ctx, h, 1, h->n));
  BOF_TRY(transpose_csr(ctx, h->m, h->n, h->nnz, h->offs[0], h->idx[0], h->vals[0], h->offs[1], h->idx[1], h->vals[1]));
  h->offs_host[1].resize((size_t)h->n + 1);
  BOF_TRY(copy1d(ctx, h->offs_host[1].data(), h->offs[1], (size_t)(h->n + 1) * 8, D2H, ctx->compute));
  BOF_TRY(sync_all(ctx));
  h->have_t = true;
  return call_guard.done();
}

int bof_csr_arrays(bof_csr* h, char trans_a, const float** vals, const int32_t** idx, const int64_t** offs,
                   int64_t* nnz) {
  if (!h) return BOF_EINVAL;
  BOF_REQUIRE(h->ctx, is_nt(trans_a), "csr_arrays: unrecognized value for param trans_a = '%c'", trans_a);
  const int t = trans_a == 'T';
  if (t) BOF_TRY(bof_csr_build_transpose(h));
  if (vals) *vals = h->vals[t];
  if (idx) *idx = h->idx[t];
  if (offs) *offs = h->offs[t];
  if (nnz) *nnz = h->nnz;
  return BOF_OK;
}

// C = alpha op(A) B + beta C with host B, C.  The dense operands move in column panels of 64 (a panel is an
// independent product), so the upload of panel p+1, the kernels of panel p and the download of its row blocks
// overlap on the three streams; A is only read from HBM.
int bof_csr_mm(bof_csr* h, char trans_a, int64_t k, float alpha, float beta, char ord_b, const float* b, float* c) {
  if (!h) return BOF_EINVAL;
  bof_ctx* ctx = h->ctx;
  BOF_REQUIRE(ctx, is_nt(trans_a), "csrmm: unrecognized value for param trans_a = '%c'", trans_a);
  BOF_REQUIRE(ctx, is_rc(ord_b), "csrmm: unrecognized value for param ord_b = '%c'", ord_b);
  BOF_REQUIRE(ctx, k >= 0, "csrmm: bad dimension");
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  const int t = trans_a == 'T';
  if (t) BOF_TRY(bof_csr_build_transpose(h));
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  const int64_t out_rows = t ? h->n : h->m, in_rows = t ? h->m : h->n;
  if (out_rows == 0 || k == 0) { stats_end(ctx); return call_guard.done(); }
  const bool colmaj = ord_b == 'C';
  const HostC hc{c, colmaj ? out_rows : k, colmaj};
  const int64_t* oh = h->offs_host[t].data();

  // panel width: measured on the cfg-3 matrix at k = 256 (profiles/r01/resident_panel_sweep.txt): 32 -> 304 ms
  // (kernel-bound), 64 -> 217 ms, 128 -> 260 ms, 256 (no panels) -> 309 ms
  static const int64_t panel_cols = getenv("BOF_CSR_PANEL") ? std::max(4, atoi(getenv("BOF_CSR_PANEL"))) : 64;
  const int64_t kb = std::min<int64_t>(k, panel_cols);
  const int npan = (int)ceil_div<int64_t>(k, kb);
  const int64_t rows_blk = std::max<int64_t>(4096, (64ll << 20) / (kb * 4));
  const int nblk = (int)ceil_div<int64_t>(out_rows, rows_blk);
  const size_t pan_elems = (size_t)std::max<int64_t>(in_rows, 1) * kb;
  float *bpan_all, *braw_all = nullptr, *cblk[2], *cblk_t[2] = {nullptr, nullptr};
  BOF_TRY(slot_reserve(ctx, S_DENSE, 2 * pan_elems, &bpan_all));
  if (colmaj) BOF_TRY(slot_reserve(ctx, S_DENSE_T, 2 * pan_elems, &braw_all));
  for (int g = 0; g < 2; ++g) {
    BOF_TRY(slot_reserve(ctx, S_CBLK + g, (size_t)std::min(rows_blk, out_rows) * kb, &cblk[g]));
    if (colmaj) BOF_TRY(slot_reserve(ctx, S_CBLK_T + g, (size_t)std::min(rows_blk, out_rows) * kb, &cblk_t[g]));
  }
  bool pan_used[2] = {false, false}, blk_used[2] = {false, false};
  uint64_t down_ticket[2] = {0, 0};  // pageable C: the drainer enqueues the download and records EV_DOWN + g
  auto upload_panel = [&](int p) -> int {
    const int gp = p & 1;
    const int64_t j0 = (int64_t)p * kb, kbp = std::min(kb, k - j0);
    float* bp = bpan_all + (size_t)gp * pan_elems;
    if (pan_used[gp]) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, EV_PAN_FREE + gp), 0));
    if (in_rows > 0) {
      if (colmaj) {
        float* raw = braw_all + (size_t)gp * pan_elems;  // columns j0.. of a column-major B are contiguous
        BOF_TRY(copy1d(ctx, raw, b + j0 * in_rows, (size_t)in_rows * kbp * 4, H2D, ctx->h2d));
      } else {
        BOF_TRY(copy2d(ctx, bp, (size_t)kbp * 4, b + j0, (size_t)k * 4, (size_t)kbp * 4, (size_t)in_rows, H2D, ctx->h2d));
      }
    }
    BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_PAN + gp), ctx->h2d));
    pan_used[gp] = true;
    return BOF_OK;
  };
  int bc = 0;  // running block counter -> C buffer generation
  auto run_block = [&](int p, int i, int g) -> int {
    const int gp = p & 1;
    const int64_t j0 = (int64_t)p * kb, kbp = std::min(kb, k - j0);
    const int64_t r0 = (int64_t)i * rows_blk, rows = std::min(rows_blk, out_rows - r0);
    const int64_t z0 = oh[r0] - oh[0];
    float* bp = bpan_all + (size_t)gp * pan_elems;
    if (blk_used[g]) d2h_fence(ctx, down_ticket[g]);  // EV_DOWN + g recorded, EV_DONE + g may be re-recorded
    if (beta != 0.f) {
      if (blk_used[g]) {
        BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, EV_DONE + g), 0));
        BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, EV_DOWN + g), 0));
      }
      BOF_TRY(upload_c_block(ctx, hc, r0, rows, j0, kbp, colmaj ? cblk_t[g] : cblk[g]));
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_UP + g), ctx->h2d));
      BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_UP + g), 0));
    }
    if (i == 0) {
      BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_PAN + gp), 0));
      if (colmaj && in_rows > 0)
        BOF_TRY(launch_transpose(ctx, ctx->compute, kbp, in_rows, braw_all + (size_t)gp * pan_elems, in_rows, bp, kbp));
    }
    if (blk_used[g]) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_DOWN + g), 0));
    const DevCsr blk{h->offs[t] + r0, h->idx[t] + z0, h->vals[t] + z0};
    BOF_TRY(spmm_c_block(ctx, rows, kbp, alpha, blk, bp, 0, beta, cblk[g], cblk_t[g]));
    BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_DONE + g), ctx->compute));
    if (i == nblk - 1) BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_PAN_FREE + gp), ctx->compute));
    blk_used[g] = true;
    return BOF_OK;
  };
  auto fetch_block = [&](int p, int i, int g) -> int {
    const int64_t j0 = (int64_t)p * kb, kbp = std::min(kb, k - j0);
    const int64_t r0 = (int64_t)i * rows_blk, rows = std::min(rows_blk, out_rows - r0);
    return download_c_block(ctx, hc, r0, rows, j0, kbp, colmaj ? cblk_t[g] : cblk[g], get_event(ctx, EV_DONE + g),
                            get_event(ctx, EV_DOWN + g), &down_ticket[g]);
  };
  // software pipeline over (panel, block): launch step s, then download step s-1
  BOF_TRY(upload_panel(0));
  int prev_p = -1, prev_i = -1, prev_g = -1;
  for (int p = 0; p < npan; ++p) {
    if (beta == 0.f && p + 1 < npan) BOF_TRY(upload_panel(p + 1));
    for (int i = 0; i < nblk; ++i, ++bc) {
      const int g = bc & 1;
      BOF_TRY(run_block(p, i, g));
      if (prev_p >= 0) BOF_TRY(fetch_block(prev_p, prev_i, prev_g));
      prev_p = p; prev_i = i; prev_g = g;
    }
    // with beta != 0 the old-C uploads share the h2d stream, so the next panel is queued behind them
    if (beta != 0.f && p + 1 < npan) BOF_TRY(upload_panel(p + 1));
  }
  if (prev_p >= 0) BOF_TRY(fetch_block(prev_p, prev_i, prev_g));
  BOF_TRY(sync_all(ctx));
  stats_end(ctx);
  return call_guard.done();
}

// y = op(A) x with host x, y.  'T' uses the resident A^T when it has been built (a deterministic gather SpMV),
// else the scatter kernel on A.
int bof_csr_mv(bof_csr* h, char trans_a, const float* x, float* y) {
  if (!h) return BOF_EINVAL;
  bof_ctx* ctx = h->ctx;
  BOF_REQUIRE(ctx, is_nt(trans_a), "csrgemv trans_a error : expected=N or T, found=%c", trans_a);
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  const bool tr = trans_a == 'T';
  const int64_t xlen = tr ? h->m : h->n, ylen = tr ? h->n : h->m;
  if (ylen == 0) { stats_end(ctx); return call_guard.done(); }
  float *xd, *yd;
  BOF_TRY(slot_reserve(ctx, S_MISC, (size_t)std::max<int64_t>(xlen, 1), &xd));
  BOF_TRY(slot_reserve(ctx, S_OUT0, (size_t)ylen, &yd));
  cudaStream_t s = ctx->compute;
  BOF_TRY(copy1d(ctx, xd, x, (size_t)xlen * 4, H2D, s));
  if (!tr) BOF_TRY(launch_spmv(ctx, s, 'N', h->m, h->n, h->vals[0], h->idx[0], h->offs[0], xd, yd));
  else if (h->have_t) BOF_TRY(launch_spmv(ctx, s, 'N', h->n, h->m, h->vals[1], h->idx[1], h->offs[1], xd, yd));
  else BOF_TRY(launch_spmv(ctx, s, 'T', h->m, h->n, h->vals[0], h->idx[0], h->offs[0], xd, yd, h->nnz));
  BOF_TRY(copy1d(ctx, y, yd, (size_t)ylen * 4, D2H, s));
  BOF_TRY(sync_all(ctx));
  stats_end(ctx);
  return call_guard.done();
}

int bof_csr_close(bof_csr* h) {
  if (!h) return BOF_OK;
  cudaSetDevice(h->ctx->device);
  cudaDeviceSynchronize();
  csr_free(h);
  return BOF_OK;
}

}  // extern "C"
