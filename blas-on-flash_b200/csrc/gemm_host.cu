// flash::gemm / flash::kmeans on the host side: canonical form of the 8 layout cases, the device-resident GEMM
// with a caller workspace, and the host pipeline (panelled upload of the resident operand, ring of row blocks,
// slab drain).  Reference: src/blas/gemm.cpp:27-202, include/tasks/gemm_task.h:67-93.
#include "host_internal.cuh"

namespace bof {

// Leading-dimension defaults and the row/col role table of src/blas/gemm.cpp:52-67.
int canon_gemm(bof_ctx* ctx, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k,
               const float* A, int64_t lda, const float* B, int64_t ldb, int64_t ldc, Canon* out) {
  BOF_REQUIRE(ctx, is_rc(ord), "gemm: mat_ord must be 'R' or 'C' (got '%c')", ord);
  BOF_REQUIRE(ctx, is_nt(ta), "gemm: trans_a must be 'N' or 'T' (got '%c')", ta);
  BOF_REQUIRE(ctx, is_nt(tb), "gemm: trans_b must be 'N' or 'T' (got '%c')", tb);
  BOF_REQUIRE(ctx, m >= 0 && n >= 0 && k >= 0, "gemm: negative dimension");
  const bool col = ord == 'C', tA = ta == 'T', tB = tb == 'T';
  const int64_t a_cols = (tA != col) ? m : k;  // contiguous extent of A as stored
  const int64_t b_cols = (tB != col) ? k : n;
  const int64_t c_cols = col ? m : n;
  if (lda == 0) lda = a_cols;
  if (ldb == 0) ldb = b_cols;
  if (ldc == 0) ldc = c_cols;
  BOF_REQUIRE(ctx, lda >= a_cols && ldb >= b_cols && ldc >= c_cols, "gemm: leading dimension too small");
  // op(A)(i, kk) = A[i*a_si + kk*a_sk]: contiguous in kk iff A is stored with k as its inner extent
  const int64_t a_si = (tA == col) ? lda : 1, a_sk = (tA == col) ? 1 : lda;
  // op(B)(kk, j) = B[j*b_sj + kk*b_sk]: contiguous in kk iff B is stored with k as its inner extent
  const int64_t b_sj = (tB != col) ? ldb : 1, b_sk = (tB != col) ? 1 : ldb;
  Canon c{};
  c.K = k;
  c.ldc = ldc;
  if (!col) {  // C[i*ldc + j]
    c.Mo = m; c.No = n;
    c.psrc = A; c.p_sr = a_si; c.p_sk = a_sk;
    c.qsrc = B; c.q_sr = b_sj; c.q_sk = b_sk;
  } else {     // column-major C is the row-major transpose: C^T = op(B)^T op(A)^T
    c.Mo = n; c.No = m;
    c.psrc = B; c.p_sr = b_sj; c.p_sk = b_sk;
    c.qsrc = A; c.q_sr = a_si; c.q_sk = a_sk;
  }
  *out = c;
  return BOF_OK;
}

int64_t padded_k(int64_t k) { return std::max<int64_t>(32, round_up<int64_t>(k, 32)); }
size_t plane_bytes(int64_t rows, int64_t kp) { return round_up<size_t>((size_t)rows * kp * 4, 256); }

int pick_gemm_path(const bof_ctx* ctx, int64_t Mo, int64_t No, int64_t K) {
  if (ctx->cfg.gemm_force_path) return ctx->cfg.gemm_force_path;
  if ((double)Mo * No * K < 2e6) return 3;  // launch-latency territory: CUDA cores, no planes
  return 2;
}

int64_t k_chunk_of(const bof_ctx* ctx) {
  if (ctx->cfg.gemm_k_chunk < 0) return 0;
  return ctx->cfg.gemm_k_chunk == 0 ? 256 : ctx->cfg.gemm_k_chunk;
}

// rows of the canonical P operand per block of the host pipeline
static int64_t host_row_block(const bof_ctx* ctx, int64_t Mo) {
  int64_t rb = (int64_t)ctx->cfg.gemm_row_block;
  rb = std::max<int64_t>(256, round_up<int64_t>(rb, 256));
  return std::min(rb, round_up<int64_t>(Mo, 256));
}

// Event ids of the host GEMM plans: + g per ring generation, + j per Q panel (out of core: per Q buffer).  The plans
// never run in one call, so EV_QFREE and EV_C0 (out of core) reuse numbers of the resident plan's Q panels.
constexpr int kMaxQPanels = 16;  // clamp of BOF_GEMM_QPANELS
enum GemmEvent : int {
  EV_TERMS = 3,                    // k-means terms uploaded
  EV_UP = 8, EV_SPLIT = 16,        // P rows uploaded; raw P split into planes (its buffer is free)
  EV_DONE = 24, EV_DOWN = 32,      // rows of C final; rows of C downloaded
  EV_QPAN = 40,                    // Q panel uploaded; also the column slabs of the resident drain
  EV_QFREE = 42, EV_C0 = 44,       // out of core: Q buffer consumed; old C of the super-block uploaded
  EV_SLAB = 88,                    // resident slab download: the slabs of Q panel j computed
};
static_assert(EV_TERMS < EV_UP && EV_UP + kGemmRing <= EV_SPLIT && EV_SPLIT + kGemmRing <= EV_DONE &&
              EV_DONE + kGemmRing <= EV_DOWN && EV_DOWN + kGemmRing <= EV_QPAN && EV_QPAN + kMaxQPanels <= EV_SLAB,
              "resident plan: event ranges overlap");
static_assert(EV_QPAN + 2 <= EV_QFREE && EV_QFREE + 2 <= EV_C0, "out-of-core plan: event ranges overlap");

// The device buffers of a host GEMM plan, (slot, bytes) in the order it reserves them; 0 bytes: a slot it leaves
// unused.  The same table gives the plan's footprint and the slots whose memory counts as available.
using SlotTable = std::vector<std::pair<int, size_t>>;
static size_t table_bytes(const SlotTable& t) { size_t n = 0; for (const auto& e : t) n += e.second; return n; }
static int reserve_slots(bof_ctx* ctx, const SlotTable& t) {
  void* p;
  for (const auto& e : t) if (e.second) BOF_TRY(slot_reserve(ctx, e.first, e.second, &p));
  return BOF_OK;
}
static float* slot_f32(const bof_ctx* ctx, int slot) { return static_cast<float*>(ctx->slot_ptr[slot]); }

// Device memory a host GEMM may plan with: BOF_GEMM_HBM_BUDGET=<bytes> when set (read on every call, so a test can
// force the out-of-core plan at a small size), otherwise the free memory plus what the context already holds in the
// slots of `t` (slot_reserve frees a slot before it grows it).  *forced tells which.
static size_t gemm_hbm_available(const bof_ctx* ctx, const SlotTable& t, bool* forced) {
  const char* e = getenv("BOF_GEMM_HBM_BUDGET");
  *forced = e != nullptr && *e != '\0';
  if (*forced) return (size_t)strtoull(e, nullptr, 10);
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return SIZE_MAX; }  // unknown: plan resident
  for (const auto& sl : t) free_b += ctx->slot_bytes[sl.first];
  return free_b;
}

// Resident plan, row blocks of rb: Q's raw copy (if it has a slot of its own), Q's planes, raw P per ring generation,
// the P planes and C blocks of all generations, the k-means terms.
static SlotTable resident_gemm_slots(const Canon& cn, int64_t rb, bool q_slot, bool tensor, bool with_terms) {
  const int64_t K = std::max<int64_t>(cn.K, 1), kp = padded_k(cn.K);
  const int ngen = (int)std::min<int64_t>(kGemmRing, ceil_div<int64_t>(cn.Mo, rb));
  SlotTable t;
  if (q_slot) t.push_back({S_DENSE, (size_t)cn.No * K * 4});
  if (tensor) t.push_back({S_DENSE_T, 2 * plane_bytes(cn.No, kp)});
  for (int g = 0; g < ngen; ++g) t.push_back({S_PRAW + g, (size_t)rb * K * 4});
  if (tensor) t.push_back({S_PPLANES, 2 * (size_t)ngen * plane_bytes(rb, kp)});
  t.push_back({S_GCBLK, (size_t)ngen * rb * cn.No * 4});
  if (with_terms) t.push_back({S_MISC, (size_t)(cn.Mo + cn.No) * 4});
  return t;
}

// Out-of-core plan, super-blocks of S rows, row blocks of rb, k-panels of L: two Q panels raw and split, the P planes
// and raw P of every ring generation, the fold of a super-block, its old C (beta != 0), the k-means terms.
static SlotTable ooc_gemm_slots(int64_t No, int64_t S, int64_t rb, int64_t L, bool with_c0, size_t terms) {
  SlotTable t = {{S_DENSE, (size_t)No * L * 8}, {S_DENSE_T, 4 * plane_bytes(No, L)},
                 {S_PPLANES, 2 * (size_t)kGemmRing * plane_bytes(rb, L)}};
  for (int g = 0; g < kGemmRing; ++g) t.push_back({S_PRAW + g, (size_t)rb * L * 4});
  t.insert(t.end(), {{S_GCBLK, (size_t)S * No * 4}, {S_CBLK, with_c0 ? (size_t)S * No * 4 : 0}, {S_MISC, terms}});
  return t;
}

// flash::kmeans' terms on the canonical C: += rows[r], += cols[j], the row term first iff row_first.
struct GemmTerms { const float* rows = nullptr; const float* cols = nullptr; int row_first = 0; };

// The terms into dst (rows, then columns); the compute stream waits for them.
static int upload_terms(bof_ctx* ctx, const GemmTerms& tm, int64_t Mo, int64_t No, float* dst) {
  BOF_TRY(copy1d(ctx, dst, tm.rows, (size_t)Mo * 4, cudaMemcpyHostToDevice, ctx->h2d));
  BOF_TRY(copy1d(ctx, dst + Mo, tm.cols, (size_t)No * 4, cudaMemcpyHostToDevice, ctx->h2d));
  BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_TERMS), ctx->h2d));
  BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_TERMS), 0));
  return BOF_OK;
}

// Strides (per row, per k) of `rows` rows x `len` k of a canonical operand uploaded as a tight block: [rows x len]
// when the source is contiguous in k (s_k == 1), [len x rows] otherwise.
struct Strides { int64_t r, k; };
static Strides tight_strides(int64_t s_k, int64_t rows, int64_t len) { return s_k == 1 ? Strides{len, 1} : Strides{1, rows}; }

// Rows [r0, r1) x k [k0, k1) of a canonical operand (element (r, kk) at src[r*s_r + kk*s_k]) into dst as that tight
// block, one pitched copy on stream s.
static int upload_operand(bof_ctx* ctx, const float* src, int64_t s_r, int64_t s_k, int64_t r0, int64_t r1, int64_t k0,
                          int64_t k1, float* dst, cudaStream_t s, Strides* st) {
  const int64_t rows = r1 - r0, len = k1 - k0;
  *st = tight_strides(s_k, rows, len);
  const cudaMemcpyKind H2D = cudaMemcpyHostToDevice;
  if (s_k == 1) return copy2d(ctx, dst, (size_t)len * 4, src + r0 * s_r + k0, (size_t)s_r * 4, (size_t)len * 4, (size_t)rows, H2D, s);
  // stored k-major: rows [k0, k1) of a [K x ld] matrix, columns [r0, r1)
  return copy2d(ctx, dst, (size_t)rows * 4, src + r0 + k0 * s_k, (size_t)s_k * 4, (size_t)rows * 4, (size_t)len, H2D, s);
}

// Rows [r0, r0 + rows) x columns [n0, n1) of C from the device block `blk` (pitch No, row r0 first), on the d2h stream.
static int download_c(bof_ctx* ctx, const Canon& cn, float* c, const float* blk, int64_t r0, int64_t rows, int64_t n0,
                      int64_t n1, cudaEvent_t wait_ev, cudaEvent_t record_ev, uint64_t* ticket) {
  return d2h_transfer(ctx, c + r0 * cn.ldc + n0, (size_t)cn.ldc * 4, blk + n0, (size_t)cn.No * 4, (size_t)(n1 - n0) * 4,
                      (size_t)rows, ctx->d2h, wait_ev, record_ev, ticket);
}

// GEMM on device-resident canonical operands with a caller-provided plane workspace.
int gemm_canon_device(bof_ctx* ctx, cudaStream_t s, const Canon& c, float alpha, float beta, float* C,
                      void* ws, size_t ws_bytes) {
  if (c.Mo == 0 || c.No == 0) return BOF_OK;
  const int path = pick_gemm_path(ctx, c.Mo, c.No, c.K);
  if (c.K == 0 || path == 3) {
    // K == 0 degenerates to C = beta*C, which the CUDA-core kernel handles as well
    return launch_gemm_ffma(ctx, s, c.Mo, c.No, c.K, alpha, c.psrc, c.p_sr, c.p_sk, c.qsrc, c.q_sk, c.q_sr,
                            beta, C, c.ldc);
  }
  const int64_t kp = padded_k(c.K);
  const size_t pb = plane_bytes(c.Mo, kp), qb = plane_bytes(c.No, kp);
  BOF_REQUIRE(ctx, ws != nullptr && ws_bytes >= 2 * pb + 2 * qb + 256, "gemm: workspace too small");
  uint8_t* base = reinterpret_cast<uint8_t*>(round_up<uintptr_t>(reinterpret_cast<uintptr_t>(ws), 256));
  float* p_hi = reinterpret_cast<float*>(base);
  float* p_lo = reinterpret_cast<float*>(base + pb);
  float* q_hi = reinterpret_cast<float*>(base + 2 * pb);
  float* q_lo = reinterpret_cast<float*>(base + 2 * pb + qb);
  BOF_TRY(launch_split_planes(ctx, s, c.Mo, c.K, c.psrc, c.p_sr, c.p_sk, p_hi, p_lo, kp));
  BOF_TRY(launch_split_planes(ctx, s, c.No, c.K, c.qsrc, c.q_sr, c.q_sk, q_hi, q_lo, kp));
  GemmEpilogue ep;
  ep.alpha = alpha; ep.beta = beta; ep.C = C; ep.ldc = c.ldc;
  return launch_gemm_tc(ctx, s, path == 1 ? 1 : 2, c.Mo, c.No, c.K, kp, p_hi, p_lo, q_hi, q_lo, ep, k_chunk_of(ctx));
}


}  // namespace bof

using namespace bof;

// Out-of-core plan of bof_host_gemm / bof_host_kmeans_dist, for operands whose resident plan does not fit the device.
// C is computed in super-blocks of S rows whose fp32 fold stays on the device for the whole k extent.  k is walked
// in panels of L elements, L a multiple of the fold chunk (launch_gemm_tc folds TMEM into fp32 every chunk), and each
// panel's launch resumes the fold the previous panel stored: the additions are the resident plan's, in its order,
// so the result is the same bits whatever the budget.  Per (super-block, panel) Q's panel is uploaded and split once
// into one of two buffers, so that panel p + 1 uploads while panel p multiplies; P's row blocks stream through the
// ring of kGemmRing generations, which cycles over (panel, row block) items.  The last panel applies alpha, beta
// (C0 read from its own buffer) and the k-means terms, and the rows of C are downloaded behind it.
// PCIe: H2D = sz(P) + n_super * sz(Q) [+ sz(C) when beta != 0], D2H = sz(C).
static int host_gemm_ooc(bof_ctx* ctx, const Canon& cn, int cg, float alpha, float beta, float* c, const GemmTerms& tm,
                         bool forced) {
  constexpr int NB = kGemmRing;
  const int64_t Mo = cn.Mo, No = cn.No, K = cn.K;
  const int64_t kc = k_chunk_of(ctx);
  const int64_t unit = 32 * (kc <= 0 ? 1 : std::max<int64_t>(1, kc / 32));  // a panel starts on a fold-chunk boundary
  const bool with_terms = tm.rows != nullptr;
  const int64_t rb0 = host_row_block(ctx, Mo);
  const size_t terms = with_terms ? (size_t)(Mo + No) * 4 : 0;
  auto slots_of = [&](int64_t S, int64_t rb, int64_t L) { return ooc_gemm_slots(No, S, rb, L, beta != 0.f, terms); };
  // the slots of the smallest plan are the plan's slots at any size: what they hold counts as available
  const SlotTable smallest = slots_of(std::min<int64_t>(Mo, 256), 256, unit);
  bool unused;
  size_t avail = gemm_hbm_available(ctx, smallest, &unused);
  if (!forced) avail -= std::min<size_t>(avail / 4, (size_t)1 << 30);  // allocation granularity, kernel workspaces
  auto fits = [&](int64_t S, int64_t rb, int64_t L) { return table_bytes(slots_of(S, rb, L)) <= avail; };

  const int64_t s_units = ceil_div<int64_t>(Mo, 256);
  const size_t need_min = table_bytes(smallest);
  if (need_min > avail)
    return fail(ctx, BOF_ENOMEM,
                "gemm: the operands exceed device memory and the out-of-core plan needs at least %zu bytes "
                "(256 rows of C, k-panels of %lld), %zu available", need_min, (long long)unit, avail);
  // S first, as large as fits with the shortest panel: every extra super-block re-streams Q
  int64_t lo = 1, hi = s_units;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) / 2;
    if (fits(std::min(Mo, mid * 256), std::min(rb0, mid * 256), unit)) lo = mid; else hi = mid - 1;
  }
  // whole row blocks of at most rb0 rows per super-block
  const int64_t blocks = ceil_div<int64_t>(lo * 256, rb0);
  const int64_t rb = lo / blocks * 256;
  const int64_t S = std::min(Mo, rb * blocks);
  // then L as long as the rest allows, evened out over the panels
  lo = 1; hi = ceil_div<int64_t>(K, unit);
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) / 2;
    if (fits(S, rb, mid * unit)) lo = mid; else hi = mid - 1;
  }
  const int64_t npan = ceil_div<int64_t>(K, lo * unit);
  const int64_t L = round_up<int64_t>(ceil_div<int64_t>(K, npan), unit);

  // ---- buffers: a slot that holds more than this plan needs is released, then the plan's table is reserved ----
  const SlotTable slots = slots_of(S, rb, L);
  bool synced = false;
  for (const auto& sb : slots) {
    if (ctx->slot_bytes[sb.first] <= sb.second) continue;
    if (!synced) { BOF_CUDA(ctx, cudaDeviceSynchronize()); synced = true; }   // a slot may still be in use by queued work
    BOF_CUDA(ctx, cudaFree(ctx->slot_ptr[sb.first]));
    ctx->slot_ptr[sb.first] = nullptr;
    ctx->slot_bytes[sb.first] = 0;
  }
  BOF_TRY(reserve_slots(ctx, slots));
  float* qraw = slot_f32(ctx, S_DENSE);
  float* fold = slot_f32(ctx, S_GCBLK);
  float* c0 = beta != 0.f ? slot_f32(ctx, S_CBLK) : nullptr;
  float* term_d = with_terms ? slot_f32(ctx, S_MISC) : nullptr;
  float* praw[NB];
  for (int g = 0; g < NB; ++g) praw[g] = slot_f32(ctx, S_PRAW + g);
  const size_t qpb = plane_bytes(No, L), ppb = plane_bytes(rb, L);
  auto q_hi = [&](int b) { return slot_f32(ctx, S_DENSE_T) + 2 * b * qpb / 4; };
  auto q_lo = [&](int b) { return slot_f32(ctx, S_DENSE_T) + (2 * b + 1) * qpb / 4; };
  auto p_hi = [&](int g) { return slot_f32(ctx, S_PPLANES) + g * ppb / 4; };
  auto p_lo = [&](int g) { return slot_f32(ctx, S_PPLANES) + (NB + g) * ppb / 4; };
  if (with_terms) BOF_TRY(upload_terms(ctx, tm, Mo, No, term_d));

  bool p_used[NB] = {}, q_used[2] = {}, down_used[NB] = {};
  uint64_t down_ticket[NB] = {};
  int64_t item = 0, qseq = 0;
  for (int64_t s0 = 0; s0 < Mo; s0 += S) {
    const int64_t s1 = std::min(Mo, s0 + S);
    const int64_t nb = ceil_div<int64_t>(s1 - s0, rb);
    // the rows of C of the previous super-block leave the buffer this one writes its result into first
    for (int g = 0; g < NB; ++g) {
      if (!down_used[g]) continue;
      d2h_fence(ctx, down_ticket[g]);
      BOF_CUDA(ctx, cudaStreamWaitEvent(beta != 0.f ? ctx->h2d : ctx->compute, get_event(ctx, EV_DOWN + g), 0));
    }
    if (beta != 0.f) {
      BOF_TRY(copy2d(ctx, c0, (size_t)No * 4, c + s0 * cn.ldc, (size_t)cn.ldc * 4, (size_t)No * 4, (size_t)(s1 - s0), cudaMemcpyHostToDevice, ctx->h2d));
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_C0), ctx->h2d));
    }
    for (int64_t p = 0; p < npan; ++p, ++qseq) {
      const int64_t k0 = p * L, k1 = std::min(K, k0 + L), len = k1 - k0, kpp = padded_k(len);
      const bool first = p == 0, last = p == npan - 1;
      const int b = (int)(qseq & 1);
      float* qbuf = qraw + (size_t)b * No * L;
      if (q_used[b]) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, EV_QFREE + b), 0));
      Strides qs;
      BOF_TRY(upload_operand(ctx, cn.qsrc, cn.q_sr, cn.q_sk, 0, No, k0, k1, qbuf, ctx->h2d, &qs));
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_QPAN + b), ctx->h2d));
      trace_mark(ctx, ctx->h2d, "h2d: Q k-panel landed", (int)p);
      for (int64_t i = 0; i < nb; ++i, ++item) {
        const int g = (int)(item % NB);
        const int64_t r0 = s0 + i * rb, rows = std::min(s1, r0 + rb) - r0;
        if (p_used[g]) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, EV_SPLIT + g), 0));  // raw P consumed
        Strides ps;
        BOF_TRY(upload_operand(ctx, cn.psrc, cn.p_sr, cn.p_sk, r0, r0 + rows, k0, k1, praw[g], ctx->h2d, &ps));
        BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_UP + g), ctx->h2d));
        if (i == 0) {
          BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_QPAN + b), 0));
          BOF_TRY(launch_split_planes(ctx, ctx->compute, No, len, qbuf, qs.r, qs.k, q_hi(b), q_lo(b), kpp));
        }
        BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_UP + g), 0));
        BOF_TRY(launch_split_planes(ctx, ctx->compute, rows, len, praw[g], ps.r, ps.k, p_hi(g), p_lo(g), kpp));
        BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_SPLIT + g), ctx->compute));
        p_used[g] = true;
        float* fold_rows = fold + (size_t)(r0 - s0) * No;
        float* out = (last && beta != 0.f) ? c0 + (size_t)(r0 - s0) * No : fold_rows;
        if (last && beta != 0.f && i == 0) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_C0), 0));
        GemmEpilogue ep;
        ep.alpha = alpha; ep.beta = beta; ep.C = out; ep.ldc = No;
        ep.carry = first ? nullptr : fold_rows; ep.ld_carry = No;
        ep.raw_out = !last;
        BOF_TRY(launch_gemm_tc(ctx, ctx->compute, cg, rows, No, len, kpp, p_hi(g), p_lo(g), q_hi(b), q_lo(b), ep, kc));
        if (!last) continue;
        if (with_terms)
          BOF_TRY(launch_add_outer_terms(ctx, ctx->compute, out, rows, No, No, term_d + r0, term_d + Mo, tm.row_first));
        if (down_used[g]) d2h_fence(ctx, down_ticket[g]);  // EV_DONE + g is waited on by that download
        BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_DONE + g), ctx->compute));
        BOF_TRY(download_c(ctx, cn, c, out, r0, rows, 0, No, get_event(ctx, EV_DONE + g), get_event(ctx, EV_DOWN + g),
                           &down_ticket[g]));
        down_used[g] = true;
      }
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_QFREE + b), ctx->compute));
      q_used[b] = true;
    }
  }
  BOF_TRY(sync_all(ctx));
  trace_dump(ctx, "bof_host_gemm (out of core)");
  return BOF_OK;
}

extern "C" {

// flash::gemm.  The canonical Q operand (op(B)^T for row-major problems) is uploaded and split
// into TF32 planes once; the canonical P operand and the output stream in row blocks,
// double-buffered (upload / split + MMA / download overlap).  The reference's k-dimension
// accumulate chain (src/blas/gemm.cpp:114-126) is an I/O artefact: the whole k extent is reduced
// on the device, so each C block crosses PCIe once.
static int host_gemm_impl(bof_ctx* ctx, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k, float alpha,
                          float beta, const float* a, const float* b, float* c, int64_t lda, int64_t ldb, int64_t ldc,
                          bool q_on_device, const float* term_m = nullptr, const float* term_n = nullptr,
                          bool dist_q = false) {
  if (!ctx) return BOF_EINVAL;
  Canon cn;
  BOF_TRY(canon_gemm(ctx, ord, ta, tb, m, n, k, a, lda, b, ldb, ldc, &cn));
  BOF_REQUIRE(ctx, !q_on_device || ord == 'R', "gemm: a device-resident B is supported for mat_ord='R' only");
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  // A collective call (bof_dist_gemm) must take the same decisions on every rank: N and K are common, the local M
  // is not -- a rank whose shard is empty or tiny still owns panels of Q and takes part in the exchange.
  const bool dist_call = dist_q && comm_world(ctx) > 1;
  if (cn.No == 0 || (cn.Mo == 0 && !dist_call)) { stats_end(ctx); return call_guard.done(); }
  const int path = dist_call ? (ctx->cfg.gemm_force_path ? ctx->cfg.gemm_force_path : 2) : pick_gemm_path(ctx, cn.Mo, cn.No, cn.K);
  const int64_t K = cn.K, kp = padded_k(K);
  const bool tensor = (K > 0 && path != 3);
  const int cg = path == 1 ? 1 : 2;
  // flash::kmeans: C(i, j) += term_m[i], then += term_n[j] (i over m, j over n), applied to each block on the
  // device before it is downloaded.  In canonical (row-major output) form the rows are m for 'R', n for 'C'.
  GemmTerms tm;
  if (term_m != nullptr && term_n != nullptr) tm = ord == 'R' ? GemmTerms{term_m, term_n, 1} : GemmTerms{term_n, term_m, 0};
  const bool with_terms = tm.rows != nullptr;

  int64_t rb = host_row_block(ctx, cn.Mo);
  // a rank's shard of a multi-GPU job can be a single block: cut it into four so that the first MMAs start after a
  // quarter of it has landed and the C slabs leave earlier
  if (dist_call && cn.Mo <= 4 * rb) rb = std::max<int64_t>(1024, round_up<int64_t>(ceil_div<int64_t>(cn.Mo, 4), 256));
  // Q has a slot of its own unless B is already in HBM or Q lives in the exchange buffer the peers push into
  const SlotTable slots = resident_gemm_slots(cn, rb, !q_on_device && !(dist_call && tensor), tensor, with_terms);
  if (tensor && !q_on_device && !dist_call) {
    // Operands whose resident plan does not fit the device take the out-of-core plan; every call that fits stays here.
    bool forced;
    if (table_bytes(slots) > gemm_hbm_available(ctx, slots, &forced)) {
      BOF_TRY(host_gemm_ooc(ctx, cn, cg, alpha, beta, c, tm, forced));
      stats_end(ctx);
      return call_guard.done();
    }
  }

  // ---- buffers ----
  float* qraw = nullptr;
  if (q_on_device) qraw = const_cast<float*>(cn.qsrc);  // B already in HBM in its source layout; read-only here
  else if (dist_call && tensor) BOF_TRY(comm_exchange_begin(ctx, (size_t)cn.No * std::max<int64_t>(K, 1) * sizeof(float), &qraw));
  static const int64_t n_q_panels_env =
      getenv("BOF_GEMM_QPANELS") ? std::min(kMaxQPanels, std::max(1, atoi(getenv("BOF_GEMM_QPANELS")))) : 0;
  const int64_t n_q_panels = n_q_panels_env ? n_q_panels_env : (dist_call && tensor ? (comm_world(ctx) >= 8 ? 16 : 8) : 8);
  if (dist_call && tensor && cn.Mo == 0) {
    // No rows of C on this rank: upload and push the Q panels it owns, and wait for the peers' panels so that no push
    // into this rank's exchange buffer is still in flight when the call returns.
    const int world = comm_world(ctx), rank = comm_rank(ctx);
    const int64_t rows_per = std::max<int64_t>(256, round_up<int64_t>(ceil_div<int64_t>(cn.No, n_q_panels), 256));
    const int npan = (int)ceil_div<int64_t>(cn.No, rows_per);
    for (int j = 0; j < npan; ++j) {
      const int64_t n0 = (int64_t)j * rows_per, n1 = std::min(cn.No, n0 + rows_per);
      if (j % world == rank) {
        Strides st;
        BOF_TRY(upload_operand(ctx, cn.qsrc, cn.q_sr, cn.q_sk, n0, n1, 0, K, qraw + n0 * K, ctx->h2d, &st));
        BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_QPAN + j), ctx->h2d));
        BOF_TRY(comm_push(ctx, (size_t)(n0 * K), (size_t)(n1 - n0) * K, j, get_event(ctx, EV_QPAN + j)));
      } else {
        BOF_TRY(comm_wait_item(ctx, ctx->compute, j));
      }
    }
    BOF_TRY(sync_all(ctx));
    stats_end(ctx);
    return call_guard.done();
  }
  // With no rows of C (a collective call without an exchange: K == 0 or the CUDA-core path) only Q's slot is non-empty.
  BOF_TRY(reserve_slots(ctx, slots));
  if (cn.Mo == 0) { stats_end(ctx); return call_guard.done(); }
  if (!qraw) qraw = slot_f32(ctx, S_DENSE);
  const size_t qb = plane_bytes(cn.No, kp);
  float* q_hi = tensor ? slot_f32(ctx, S_DENSE_T) : nullptr;
  float* q_lo = tensor ? q_hi + qb / 4 : nullptr;
  const int nblk = (int)ceil_div<int64_t>(cn.Mo, rb);
  const size_t pb = plane_bytes(rb, kp);
  constexpr int NB = kGemmRing;
  const int ngen = std::min(NB, nblk);
  // Ring of block generations.  Planes and C blocks of the ring are each ONE allocation (generation g at
  // row g*rb), so that consecutive generations can be multiplied in a single launch during the prologue.
  float* praw[NB];
  for (int g = 0; g < ngen; ++g) praw[g] = slot_f32(ctx, S_PRAW + g);
  float* hi_all = tensor ? slot_f32(ctx, S_PPLANES) : nullptr;
  float* lo_all = tensor ? hi_all + ngen * pb / 4 : nullptr;
  float* c_all = slot_f32(ctx, S_GCBLK);
  auto p_hi_of = [&](int g) { return hi_all + (size_t)g * rb * kp; };
  auto p_lo_of = [&](int g) { return lo_all + (size_t)g * rb * kp; };
  auto cblk_of = [&](int g) { return c_all + (size_t)g * rb * cn.No; };
  float* term_d = with_terms ? slot_f32(ctx, S_MISC) : nullptr;   // rows, then columns
  if (with_terms) BOF_TRY(upload_terms(ctx, tm, cn.Mo, cn.No, term_d));

  bool used[NB] = {};
  uint64_t down_ticket[NB] = {};  // pageable C: the drainer enqueues the download and records EV_DOWN
  Strides q_st{1, 1};  // of the raw Q copy on the device

  auto upload_block = [&](int i) -> int {  // P rows (+ old C rows when beta != 0) of block i
    const int g = i % NB;
    const int64_t r0 = (int64_t)i * rb, r1 = std::min(cn.Mo, r0 + rb), rows = r1 - r0;
    if (used[g]) {
      d2h_fence(ctx, down_ticket[g]);  // EV_DOWN of block i-NB has been recorded; its EV_DONE may be re-recorded
      BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, (tensor ? EV_SPLIT : EV_DONE) + g), 0));  // raw P of block i-NB consumed
      if (beta != 0.f) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, EV_DOWN + g), 0));       // C buffer free
    }
    Strides ps;
    trace_host(ctx, "caller: upload P block begin", i);
    if (K > 0) BOF_TRY(upload_operand(ctx, cn.psrc, cn.p_sr, cn.p_sk, r0, r1, 0, K, praw[g], ctx->h2d, &ps));
    trace_host(ctx, "caller: upload P block end", i);
    if (beta != 0.f)
      BOF_TRY(copy2d(ctx, cblk_of(g), (size_t)cn.No * 4, c + r0 * cn.ldc, (size_t)cn.ldc * 4, (size_t)cn.No * 4, (size_t)rows, cudaMemcpyHostToDevice, ctx->h2d));
    BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_UP + g), ctx->h2d));
    trace_mark(ctx, ctx->h2d, "h2d: P block landed", i);
    return BOF_OK;
  };
  // compute of block i against Q rows [n0, n1) (the whole Q when not panelled); `first`/`last` bracket the block
  auto rows_of = [&](int i) { return std::min(cn.Mo, (int64_t)(i + 1) * rb) - (int64_t)i * rb; };
  // wait for block i's upload (and for its buffers), split its rows into planes
  auto prepare_block = [&](int i) -> int {
    const int g = i % NB;
    const int64_t rows = rows_of(i);
    const Strides ps = tight_strides(cn.p_sk, rows, K);
    BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_UP + g), 0));
    if (used[g]) {
      d2h_fence(ctx, down_ticket[g]);
      BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_DOWN + g), 0));
    }
    if (tensor) {
      BOF_TRY(launch_split_planes(ctx, ctx->compute, rows, K, praw[g], ps.r, ps.k, p_hi_of(g), p_lo_of(g), kp));
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_SPLIT + g), ctx->compute));
    }
    return BOF_OK;
  };
  // blocks [i0, i0 + cnt) (consecutive generations, no ring wrap) against Q rows [n0, n1), one launch
  auto gemm_blocks = [&](int i0, int cnt, int64_t n0, int64_t n1) -> int {
    const int g = i0 % NB;
    int64_t rows = 0;
    for (int i = i0; i < i0 + cnt; ++i) rows += rows_of(i);
    if (tensor) {
      GemmEpilogue ep;
      ep.alpha = alpha; ep.beta = beta; ep.C = cblk_of(g) + n0; ep.ldc = cn.No;
      trace_mark(ctx, ctx->compute, "compute: gemm start, first block", i0);
      const int rc = launch_gemm_tc(ctx, ctx->compute, cg, rows, n1 - n0, K, kp, p_hi_of(g), p_lo_of(g), q_hi + n0 * kp,
                                    q_lo + n0 * kp, ep, k_chunk_of(ctx));
      trace_mark(ctx, ctx->compute, "compute: gemm end, rows", (int)rows);
      return rc;
    }
    const Strides ps = tight_strides(cn.p_sk, rows, K);  // cnt == 1 on this path
    return launch_gemm_ffma(ctx, ctx->compute, rows, n1 - n0, K, alpha, praw[g], ps.r, ps.k, qraw + n0 * q_st.r, q_st.k,
                            q_st.r, beta, cblk_of(g) + n0, cn.No);
  };
  auto finish_block = [&](int i) -> int {
    const int g = i % NB;
    if (with_terms)
      BOF_TRY(launch_add_outer_terms(ctx, ctx->compute, cblk_of(g), rows_of(i), cn.No, cn.No, term_d + (int64_t)i * rb,
                                     term_d + cn.Mo, tm.row_first));
    BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_DONE + g), ctx->compute));
    used[g] = true;
    return BOF_OK;
  };
  auto fetch_block = [&](int i) -> int {
    const int g = i % NB;
    BOF_TRY(download_c(ctx, cn, c, cblk_of(g), (int64_t)i * rb, rows_of(i), 0, cn.No, get_event(ctx, EV_DONE + g),
                       get_event(ctx, EV_DOWN + g), &down_ticket[g]));
    if (down_ticket[g] == 0) trace_mark(ctx, ctx->d2h, "d2h: C block downloaded", i);
    return BOF_OK;
  };

  // ---- Q (resident) and block 0 ----
  // When Q is K-major in the source its rows upload as contiguous panels: panel 0, then P block 0, then the
  // remaining panels; block 0 is computed panel by panel as they land, so only one panel and one P block of
  // PCIe time are exposed before the tensor cores start.
  // dist_q (bof_dist_gemm): Q is replicated over the ranks of the communicator.  Panel j is uploaded by rank
  // j % world only and broadcast over NVLink on the collective stream, so Q crosses PCIe once per node; every
  // rank consumes the panels in the same order as they arrive, exactly like its own uploads.
  const int world = dist_q ? comm_world(ctx) : 1, rank = comm_rank(ctx);
  const bool q_panels = tensor && !q_on_device && (dist_call || (size_t)cn.No * K * 4 >= (256u << 20));
  const int64_t qpan_rows = q_panels ? std::max<int64_t>(256, round_up<int64_t>(ceil_div<int64_t>(cn.No, n_q_panels), 256)) : cn.No;
  const int n_qpan = (int)ceil_div<int64_t>(cn.No, qpan_rows);
  // Every panel is kept as its own tight block at qraw + n0*K: [rows x K] when Q is K-major in the source,
  // [K x rows] (a column range of the stored matrix, pitched copy) when it is not.
  std::vector<Strides> pan_st((size_t)n_qpan, Strides{1, 1});
  auto upload_q_panel = [&](int j) -> int {
    const int64_t n0 = (int64_t)j * qpan_rows, n1 = std::min(cn.No, n0 + qpan_rows);
    if (dist_call && tensor) {
      const int owner = j % world;
      pan_st[j] = tight_strides(cn.q_sk, n1 - n0, K);  // what upload_operand produces
      if (owner == rank) {
        // upload my panel, then push it into every peer's exchange buffer with copy-engine peer copies (no SMs)
        BOF_TRY(upload_operand(ctx, cn.qsrc, cn.q_sr, cn.q_sk, n0, n1, 0, K, qraw + n0 * K, ctx->h2d, &pan_st[j]));
        BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_QPAN + j), ctx->h2d));
        trace_mark(ctx, ctx->h2d, "h2d: own Q panel landed", j);
        BOF_TRY(comm_push(ctx, (size_t)(n0 * K), (size_t)(n1 - n0) * K, j, get_event(ctx, EV_QPAN + j)));
      }
      return BOF_OK;
    }
    if (q_on_device) pan_st[j] = {cn.q_sr, cn.q_sk};  // single panel, source strides
    else if (K > 0) BOF_TRY(upload_operand(ctx, cn.qsrc, cn.q_sr, cn.q_sk, n0, n1, 0, K, qraw + n0 * K, ctx->h2d, &pan_st[j]));
    if (n_qpan == 1) q_st = pan_st[0];
    BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_QPAN + j), ctx->h2d));
    trace_mark(ctx, ctx->h2d, "h2d: Q panel landed", j);
    return BOF_OK;
  };
  auto split_q_panel = [&](int j) -> int {
    const int64_t n0 = (int64_t)j * qpan_rows, n1 = std::min(cn.No, n0 + qpan_rows);
    if (dist_call && tensor && j % world != rank) {
      BOF_TRY(comm_wait_item(ctx, ctx->compute, j));   // pushed by its owner: gate on the arrival flag
      trace_mark(ctx, ctx->compute, "compute: peer Q panel arrived", j);
    } else {
      BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_QPAN + j), 0));
    }
    if (!tensor) return BOF_OK;
    return launch_split_planes(ctx, ctx->compute, n1 - n0, K, qraw + n0 * K, pan_st[j].r, pan_st[j].k, q_hi + n0 * kp,
                               q_lo + n0 * kp, kp);
  };
  // Prologue: the first blocks ride between the Q panels (h2d order Q0 P0 Q1 P1 Q2 P2 Q3 P3 Q4 .. Qn) and are
  // computed against each panel as it lands (compute order = arrival order), so the tensor cores start after
  // one panel + one block of PCIe time and stay fed while the rest of Q uploads: every new panel unlocks one
  // tile per prologue block.
  trace_mark(ctx, ctx->h2d, "start", 0);
  // One generation stays out of the prologue: the prologue blocks all finish together (with the last panel), so
  // the first steady-state block would otherwise wait for a whole C block to be downloaded (11 ms at 32768^3,
  // seen with BOF_TRACE=1) before it could reuse generation 0.
  const int npro = n_qpan > 1 ? std::min({nblk, NB - 1, n_qpan}) : 1;  // blocks handled by the prologue
  auto pan = [&](int j, int64_t* n0, int64_t* n1) { *n0 = (int64_t)j * qpan_rows; *n1 = std::min(cn.No, *n0 + qpan_rows); };
  const bool merge = tensor;  // the CUDA-core path multiplies one block per launch
  // When every block rides in the prologue (a rank's shard of a multi-GPU job, or a small M), each (block, panel)
  // product completes a column slab of C for good: download slab by slab behind the compute instead of whole blocks
  // at the end, so only the last slab's download is exposed.
  const bool slab_download = tensor && !with_terms && n_qpan > 1 && nblk <= npro;
  uint64_t slab_ticket = 0;
  auto fetch_slab = [&](int i, int64_t n0, int64_t n1, cudaEvent_t after) -> int {
    return download_c(ctx, cn, c, cblk_of(i % NB), (int64_t)i * rb, rows_of(i), n0, n1, after, nullptr, &slab_ticket);
  };
  // Uploads and launches are issued panel by panel: with pinned memory the order of issue is immaterial (everything
  // is asynchronous), but a pageable upload blocks this thread while it is staged, and launching only after the
  // whole prologue had been uploaded left the GPU idle for the first 170 ms at 32768^3 (BOF_TRACE).
  for (int t = 0; t < n_qpan; ++t) {
    int64_t n0, n1;
    pan(t, &n0, &n1);
    BOF_TRY(upload_q_panel(t));
    if (t < npro) BOF_TRY(upload_block(t));
    BOF_TRY(split_q_panel(t));
    // panel t against the blocks that landed before it: one launch over those consecutive generations
    const int older = std::min(t, npro);
    if (older > 0) {
      if (merge) BOF_TRY(gemm_blocks(0, older, n0, n1));
      else for (int i = 0; i < older; ++i) BOF_TRY(gemm_blocks(i, 1, n0, n1));
    }
    // block t landed right after panel t: all panels so far at once
    if (t < npro) {
      BOF_TRY(prepare_block(t));
      BOF_TRY(gemm_blocks(t, 1, 0, n1));
    }
    if (slab_download) {
      cudaEvent_t ev = get_event(ctx, EV_SLAB + t);
      BOF_CUDA(ctx, cudaEventRecord(ev, ctx->compute));
      for (int i = 0; i < older; ++i) BOF_TRY(fetch_slab(i, n0, n1, ev));      // panel t of the earlier blocks
      if (t < npro) BOF_TRY(fetch_slab(t, 0, n1, ev));                          // panels 0..t of block t
      if (slab_ticket == 0) trace_mark(ctx, ctx->d2h, "d2h: slabs of panel downloaded", t);
    } else if (t == n_qpan - 1) {
      for (int i = 0; i < npro; ++i) BOF_TRY(finish_block(i));
    }
  }
  if (slab_download) {
    trace_host(ctx, "caller: everything issued", 0);
    BOF_TRY(sync_all(ctx));
    trace_host(ctx, "caller: sync_all returned", 0);
    trace_dump(ctx, "bof_host_gemm");
    stats_end(ctx);
    return call_guard.done();
  }
  // ---- steady state: Q complete; keep NB blocks in flight, fetch the oldest before reusing its buffers ----
  int next_fetch = 0;
  int fetch_end = nblk;  // blocks [next_fetch, fetch_end) still have to be downloaded whole
  for (int i = npro; i < nblk; ++i) {
    if (next_fetch < i) BOF_TRY(fetch_block(next_fetch++));            // keeps the downloads flowing
    while (next_fetch <= i - NB) BOF_TRY(fetch_block(next_fetch++));   // block i-NB owned these buffers
    BOF_TRY(upload_block(i));
    BOF_TRY(prepare_block(i));
    if (i == nblk - 1 && tensor && cn.No >= 2048) {
      // Drain: the last block is multiplied and downloaded in four column slabs, so only the last slab's
      // download (a quarter of a block) is exposed after the tensor cores stop.
      const int g = i % NB;
      const int64_t r0 = (int64_t)i * rb, rows = rows_of(i);
      const int64_t slab = round_up<int64_t>(ceil_div<int64_t>(cn.No, 4), 256);
      while (next_fetch < i) BOF_TRY(fetch_block(next_fetch++));  // d2h is FIFO: earlier blocks first
      int j = 0;
      for (int64_t n0 = 0; n0 < cn.No; n0 += slab, ++j) {
        const int64_t n1 = std::min(cn.No, n0 + slab);
        BOF_TRY(gemm_blocks(i, 1, n0, n1));
        if (with_terms)
          BOF_TRY(launch_add_outer_terms(ctx, ctx->compute, cblk_of(g) + n0, rows, n1 - n0, cn.No, term_d + r0,
                                         term_d + cn.Mo + n0, tm.row_first));
        BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_QPAN + j), ctx->compute));
        BOF_TRY(download_c(ctx, cn, c, cblk_of(g), r0, rows, n0, n1, get_event(ctx, EV_QPAN + j),
                           n1 == cn.No ? get_event(ctx, EV_DOWN + g) : nullptr, &down_ticket[g]));
        if (down_ticket[g] == 0) trace_mark(ctx, ctx->d2h, "d2h: last block, slab downloaded", j);
      }
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_DONE + g), ctx->compute));
      used[g] = true;
      fetch_end = i;
      break;
    }
    BOF_TRY(gemm_blocks(i, 1, 0, cn.No));
    BOF_TRY(finish_block(i));
  }
  while (next_fetch < fetch_end) BOF_TRY(fetch_block(next_fetch++));
  BOF_TRY(sync_all(ctx));
  trace_dump(ctx, "bof_host_gemm");
  stats_end(ctx);
  return call_guard.done();
}

int bof_host_gemm(bof_ctx* ctx, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k, float alpha,
                  float beta, const float* a, const float* b, float* c, int64_t lda, int64_t ldb, int64_t ldc) {
  return host_gemm_impl(ctx, ord, ta, tb, m, n, k, alpha, beta, a, b, c, lda, ldb, ldc, false);
}

int bof_host_kmeans_dist(bof_ctx* ctx, char ord, char ta, char tb, int64_t m, int64_t n, int64_t k, float alpha,
                         float beta, const float* a, const float* b, float* c, int64_t lda, int64_t ldb, int64_t ldc,
                         const float* c_l2sq, const float* p_l2sq) {
  if (ctx && (c_l2sq == nullptr || p_l2sq == nullptr)) return fail(ctx, BOF_EINVAL, "kmeans: c_l2sq / p_l2sq is null");
  return host_gemm_impl(ctx, ord, ta, tb, m, n, k, alpha, beta, a, b, c, lda, ldb, ldc, false, c_l2sq, p_l2sq);
}

int bof_host_gemm_devb(bof_ctx* ctx, char ta, char tb, int64_t m, int64_t n, int64_t k, float alpha, float beta,
                       const float* a, const float* b_dev, float* c, int64_t lda, int64_t ldb, int64_t ldc) {
  return host_gemm_impl(ctx, 'R', ta, tb, m, n, k, alpha, beta, a, b_dev, c, lda, ldb, ldc, true);
}

int bof_dist_gemm(bof_ctx* ctx, char ta, char tb, int64_t m_local, int64_t n, int64_t k, float alpha, float beta,
                  const float* a_local, const float* b, float* c_local, int64_t lda, int64_t ldb, int64_t ldc) {
  return host_gemm_impl(ctx, 'R', ta, tb, m_local, n, k, alpha, beta, a_local, b, c_local, lda, ldb, ldc, false, nullptr,
                        nullptr, true);
}

}  // extern "C"
