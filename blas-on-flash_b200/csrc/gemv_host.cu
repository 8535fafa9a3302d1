// flash::gemv with host operands (bof_host_gemv): A streams through the device in tiles and crosses PCIe exactly once,
// x and the fp32 fold of every output stay on the device, finished ranges of y leave behind the next tiles.
#include "host_internal.cuh"

namespace bof {

namespace {

constexpr cudaMemcpyKind H2D = cudaMemcpyHostToDevice;

enum : int {
  EV_IN = 0,     // x (and the old y) uploaded
  EV_UP = 2,     // tile g uploaded (g = 0/1 added)
  EV_DONE = 4,   // tile g consumed by its kernels
  EV_FIN = 6,    // a range of y final (alternating)
};

// Bytes per tile of A: BOF_GEMV_BLOCK_BYTES, or 128 MiB cut so that a large A makes at least 8 tiles.
size_t gemv_tile_bytes(size_t a_bytes) {
  if (const char* v = getenv("BOF_GEMV_BLOCK_BYTES")) {
    const long long b = atoll(v);
    if (b > 0) return (size_t)b;
  }
  return std::min<size_t>(128ull << 20, std::max<size_t>(a_bytes / 8, 16ull << 20));
}

}  // namespace

int canon_gemv(bof_ctx* ctx, char ord, char trans, int64_t m, int64_t n, int64_t lda, GemvCanon* out) {
  BOF_REQUIRE(ctx, is_rc(ord), "gemv: mat_ord must be 'R' or 'C' (got '%c')", ord);
  BOF_REQUIRE(ctx, is_nt(trans), "gemv: trans_a must be 'N' or 'T' (got '%c')", trans);
  BOF_REQUIRE(ctx, m >= 0 && n >= 0, "gemv: negative dimension (m = %lld, n = %lld)", (long long)m, (long long)n);
  // the stored matrix: m rows of n for 'R', n rows (the columns of A) of m for 'C'
  const int64_t rows = ord == 'R' ? m : n, cols = ord == 'R' ? n : m;
  if (lda == 0) lda = cols;
  BOF_REQUIRE(ctx, lda >= cols, "gemv: lda = %lld is smaller than %lld", (long long)lda, (long long)cols);
  *out = GemvCanon{rows, cols, lda, (ord == 'R') == (trans == 'N')};
  return BOF_OK;
}

}  // namespace bof

using namespace bof;

extern "C" {

int bof_host_gemv(bof_ctx* ctx, char ord, char trans, int64_t m, int64_t n, float alpha, float beta, const float* a,
                  int64_t lda, const float* x, float* y) {
  if (!ctx) return BOF_EINVAL;
  GemvCanon c;
  BOF_TRY(canon_gemv(ctx, ord, trans, m, n, lda, &c));
  BOF_CUDA(ctx, cudaSetDevice(ctx->device));
  stats_begin(ctx);
  CallGuard call_guard(ctx);
  const int64_t nout = c.nout(), nred = c.nred();
  if (nout == 0) { stats_end(ctx); return call_guard.done(); }

  // Tiles: whole rows of S while they fit the budget, else cuts along the reduction on chunk boundaries.  ostep x rstep
  // is a tile's extent along the outputs x along the reduction.
  const int64_t chunk = BOF_GEMV_CHUNK;
  const int64_t elems = std::max<int64_t>(1, (int64_t)(gemv_tile_bytes((size_t)c.rows * c.cols * 4) / 4));
  int64_t ostep, rstep;
  if (c.rowdot) {   // output = row of S, reduction along it
    if (nred <= elems) { rstep = std::max<int64_t>(nred, 1); ostep = std::max<int64_t>(1, elems / rstep); }
    else { rstep = std::max<int64_t>(chunk, elems / chunk * chunk); ostep = 1; }
  } else {          // output = column of S, reduction down it
    const int64_t h = std::max<int64_t>(1, std::min(nred, chunk));
    if (nout * h <= elems) { ostep = nout; rstep = std::max<int64_t>(1, elems / (nout * chunk)) * chunk; }
    else { rstep = chunk; ostep = std::max<int64_t>(1, elems / h); }
  }
  ostep = std::min(ostep, nout);
  rstep = std::min(rstep, std::max<int64_t>(nred, 1));
  // a tile on the device: `height` rows of S with pitch round_up(width, 4) so that its rows stay 16-byte aligned
  const int64_t width = c.rowdot ? rstep : ostep, height = c.rowdot ? ostep : rstep;
  const int64_t dpitch = round_up<int64_t>(width, 4);
  const GemvCanon tile_max{height, width, dpitch, c.rowdot};

  float *xd, *yd, *acc, *tile[2];
  void* ws = nullptr;
  BOF_TRY(slot_reserve(ctx, S_DENSE, (size_t)std::max<int64_t>(nred, 1), &xd));
  BOF_TRY(slot_reserve(ctx, S_GCBLK, (size_t)nout, &yd));
  BOF_TRY(slot_reserve(ctx, S_GCBLK + 1, (size_t)nout, &acc));
  for (int g = 0; g < 2; ++g) BOF_TRY(slot_reserve(ctx, S_PRAW + g, (size_t)(height * dpitch), &tile[g]));
  BOF_TRY(slot_reserve(ctx, S_WS, gemv_workspace_bytes(tile_max), &ws));

  BOF_TRY(copy1d(ctx, xd, x, (size_t)nred * 4, H2D, ctx->h2d));
  if (beta != 0.f) BOF_TRY(copy1d(ctx, yd, y, (size_t)nout * 4, H2D, ctx->h2d));
  BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_IN), ctx->h2d));
  BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_IN), 0));
  trace_mark(ctx, ctx->h2d, "h2d: x landed", 0);

  if (nred == 0) {
    BOF_TRY(launch_gemv(ctx, ctx->compute, c, nullptr, xd, nullptr, nullptr, alpha, beta, yd, true, ws));
    BOF_TRY(copy1d(ctx, y, yd, (size_t)nout * 4, cudaMemcpyDeviceToHost, ctx->compute));
  }
  int64_t tiles = 0, ranges = 0;
  uint64_t fin_ticket[2] = {0, 0};
  for (int64_t o0 = 0; o0 < nout && nred > 0; o0 += ostep, ++ranges) {
    const int64_t o1 = std::min(nout, o0 + ostep);
    for (int64_t r0 = 0; r0 < nred; r0 += rstep, ++tiles) {
      const int64_t r1 = std::min(nred, r0 + rstep);
      const int g = (int)(tiles & 1);
      if (tiles >= 2) BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->h2d, get_event(ctx, EV_DONE + g), 0));
      const int64_t w = c.rowdot ? r1 - r0 : o1 - o0, h = c.rowdot ? o1 - o0 : r1 - r0;
      const int64_t dp = round_up<int64_t>(w, 4);
      const float* src = c.rowdot ? a + o0 * c.ld + r0 : a + r0 * c.ld + o0;
      BOF_TRY(copy2d(ctx, tile[g], (size_t)dp * 4, src, (size_t)c.ld * 4, (size_t)w * 4, (size_t)h, H2D, ctx->h2d));
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_UP + g), ctx->h2d));
      trace_mark(ctx, ctx->h2d, "h2d: tile landed", (int)tiles);
      BOF_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, get_event(ctx, EV_UP + g), 0));
      const GemvCanon t{h, w, dp, c.rowdot};
      BOF_TRY(launch_gemv(ctx, ctx->compute, t, tile[g], xd + r0, r0 == 0 ? nullptr : acc + o0, acc + o0, alpha, beta,
                          yd + o0, r1 == nred, ws));
      BOF_CUDA(ctx, cudaEventRecord(get_event(ctx, EV_DONE + g), ctx->compute));
      trace_mark(ctx, ctx->compute, "compute: tile done", (int)tiles);
    }
    // y[o0, o1) is final: it leaves while the next tiles stream in
    const int f = (int)(ranges & 1);
    d2h_fence(ctx, fin_ticket[f]);   // the transfer that waited on this event two ranges ago has been issued
    cudaEvent_t ev_fin = get_event(ctx, EV_FIN + f);
    BOF_CUDA(ctx, cudaEventRecord(ev_fin, ctx->compute));
    BOF_TRY(d2h_transfer(ctx, y + o0, (size_t)(o1 - o0) * 4, yd + o0, (size_t)(o1 - o0) * 4, (size_t)(o1 - o0) * 4, 1,
                         ctx->d2h, ev_fin, nullptr, &fin_ticket[f]));
  }
  BOF_TRY(sync_all(ctx));
  trace_dump(ctx, "bof_host_gemv");
  stats_end(ctx);
  return call_guard.done();
}

}  // extern "C"
