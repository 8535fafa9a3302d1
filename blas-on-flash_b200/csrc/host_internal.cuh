// Internals shared by the host side of the library (staging, pipelines, C ABI); not part of the ABI.
#pragma once

#include "common.cuh"

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <string>
#include <vector>

#define BOF_TRY(expr)          \
  do {                         \
    int rc__ = (expr);         \
    if (rc__ != BOF_OK) return rc__; \
  } while (0)

namespace bof {

constexpr int kGemmRing = 5;  // P/C block generations in flight in bof_host_gemm

inline bool is_nt(char c) { return c == 'N' || c == 'T'; }
inline bool is_rc(char c) { return c == 'R' || c == 'C'; }
inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// slots of the context arena
enum Slot {
  S_DENSE = 0,     // resident dense operand (B of csrmm, x of csrgemv, Q source of gemm)
  S_DENSE_T,       // its transposed / split form
  S_BLK0 = 2,      // per-block buffers, two generations each (b = 0/1 added to the slot id)
  S_OFFS = 2, S_IDX64 = 4, S_IDX32 = 6, S_VALS = 8, S_CBLK = 10, S_CBLK_T = 12,
  S_WS = 18,       // kernel workspaces
  S_OUT0 = 19, S_OUT1, S_OUT2, S_MISC,
  // host gemm: ring of kGemmRing generations (g added to the slot id)
  S_PRAW = 24, S_PPLANES = 30, S_GCBLK = 32,
};

// ---- staging.cu: streams, events, host<->device copies, tracing ----
double now_ms();
cudaEvent_t get_event(bof_ctx* ctx, size_t i);
bool trace_on();
void trace_mark(bof_ctx* ctx, cudaStream_t s, const char* what, int idx);   // CUDA-event mark on a stream
void trace_host(bof_ctx* ctx, const char* what, long idx);                  // wall-clock mark (any thread)
void trace_dump(bof_ctx* ctx, const char* title);
bool host_is_pinned(const void* p);
int copy2d(bof_ctx* ctx, void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height,
           cudaMemcpyKind kind, cudaStream_t s);
int copy1d(bof_ctx* ctx, void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s);
int d2h_transfer(bof_ctx* ctx, void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height,
                 cudaStream_t s, cudaEvent_t wait_ev, cudaEvent_t record_ev, uint64_t* ticket);
void d2h_fence(bof_ctx* ctx, uint64_t ticket);
void stats_begin(bof_ctx* ctx);
void stats_end(bof_ctx* ctx);
int drain_wait(bof_ctx* ctx);
int sync_all(bof_ctx* ctx);
void quiesce(bof_ctx* ctx);
void staging_destroy(bof_ctx* ctx);   // copy pools, drainer thread, pinned rings

// Every host entry point holds one: any return that did not set `ok` leaves the context quiescent.
struct CallGuard {
  bof_ctx* ctx;
  bool ok = false;
  explicit CallGuard(bof_ctx* c) : ctx(c) {}
  ~CallGuard() { if (!ok && ctx) quiesce(ctx); }
  int done() { ok = true; return BOF_OK; }
};

// ---- gemm_host.cu ----
// Canonical form of a GEMM: Cout[Mo x No] (row-major, ldc) = P[Mo x K] * Q[No x K]^T where
// element (r, kk) of P is psrc[r*p_sr + kk*p_sk] (one of the strides is 1), same for Q.
struct Canon {
  int64_t Mo, No, K;
  const float* psrc; int64_t p_sr, p_sk;
  const float* qsrc; int64_t q_sr, q_sk;
  int64_t ldc;
};
int canon_gemm(bof_ctx* ctx, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k,
               const float* A, int64_t lda, const float* B, int64_t ldb, int64_t ldc, Canon* out);
int64_t padded_k(int64_t k);
size_t plane_bytes(int64_t rows, int64_t kp);
int pick_gemm_path(const bof_ctx* ctx, int64_t Mo, int64_t No, int64_t K);
int64_t k_chunk_of(const bof_ctx* ctx);
int gemm_canon_device(bof_ctx* ctx, cudaStream_t s, const Canon& c, float alpha, float beta, float* C,
                      void* ws, size_t ws_bytes);

// ---- gemv.cu / gemv_host.cu ----
// Canonical form of a gemv: the stored matrix S (rows x cols, row-major, pitch ld) and either one dot product per row
// of S (row-dot: ('R','N'), ('C','T')) or one sum per column (column-sum: ('R','T'), ('C','N')).
struct GemvCanon {
  int64_t rows, cols, ld;
  bool rowdot;
  int64_t nout() const { return rowdot ? rows : cols; }   // length of y
  int64_t nred() const { return rowdot ? cols : rows; }   // length of x
};
int canon_gemv(bof_ctx* ctx, char ord, char trans, int64_t m, int64_t n, int64_t lda, GemvCanon* out);
int64_t gemv_chunks(int64_t len);   // BOF_GEMV_CHUNK pieces of a reduction of length len
size_t gemv_workspace_bytes(const GemvCanon& c);
// y[o] (o < nout) of the canonical problem on device S, x, y.  carry (may be null) seeds the fold of every output with a
// partial sum of earlier reduction chunks (S and x then start on a chunk boundary of the whole reduction);
// final_out: y = alpha*acc + beta*y, else acc_out = acc (carry and acc_out may alias).  ws: gemv_workspace_bytes(c).
int launch_gemv(bof_ctx* ctx, cudaStream_t s, const GemvCanon& c, const float* S, const float* x, const float* carry,
                float* acc_out, float alpha, float beta, float* y, bool final_out, void* ws);

// ---- comm.cu: communicator rank of a context (world 1 / rank 0 without one) ----
int comm_world(const bof_ctx* ctx);
int comm_rank(const bof_ctx* ctx);
int comm_broadcast_f32(bof_ctx* ctx, float* buf, size_t count, int root);            // on ctx->coll
int comm_allreduce_sum_f32(bof_ctx* ctx, float* buf, size_t count, cudaStream_t s);
void comm_destroy(bof_ctx* ctx);
// peer exchange of the replicated operand (copy engines over NVLink + stream memory-op flags; comm.cu)
int comm_exchange_begin(bof_ctx* ctx, size_t bytes, float** xbuf_out);
int comm_push(bof_ctx* ctx, size_t offset, size_t count, int item, cudaEvent_t ready);
int comm_wait_item(bof_ctx* ctx, cudaStream_t s, int item);
void comm_sync_pushes(bof_ctx* ctx);

}  // namespace bof
