// flash::gemv on sm_100a: y = alpha * op(A) x + beta * y, fp32, HBM-bound, deterministic.
//
// Every call is reduced to one stored row-major matrix S (rows x cols, pitch ld) and one of two shapes:
//   row-dot    out[r] = sum_c S[r][c] x[c]   (('R','N') and ('C','T'))
//   column-sum out[c] = sum_r S[r][c] x[r]   (('R','T') and ('C','N'))
// The reduction is cut into chunks of BOF_GEMV_CHUNK elements.  A chunk is summed by a tree that depends only on the
// element positions inside it (below); the chunk partials are folded in ascending chunk order into an fp32
// accumulator that starts at +0, and y = alpha*acc (+ beta*y) is applied once at the end.  Grid shape, tiling of the
// host pipeline, alignment, lda and the number of GPUs therefore never change a bit of the result.
//
// Row-dot chunk tree: element e of a chunk belongs to lane (e / 4) % 32, component e % 4, step e / 128.  Each
// (lane, component) runs an fma chain over its steps in ascending order, each lane adds (c0 + c1) + (c2 + c3), and the
// 32 lane sums meet in an xor butterfly (16, 8, 4, 2, 1).
// Column-sum chunk tree: the rows of a chunk form 16 groups (row % 16); each group runs an fma chain over its rows in
// ascending order, and the 16 group sums are added pairwise ((g0 + g1) + (g2 + g3)) + ... .
#include "host_internal.cuh"

// The kernels live in namespace bof (not an anonymous one) so that their symbol names stay the same from build to build.
namespace bof {

constexpr int kChunk = BOF_GEMV_CHUNK;
constexpr int kGroups = 16;   // row groups of the column-sum tree

__device__ __forceinline__ int64_t min64(int64_t a, int64_t b) { return a < b ? a : b; }
__device__ __forceinline__ float4 ld_stream4(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld_x4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// alpha * acc + beta * y; beta == 0 does not read y (a NaN there does not propagate)
__device__ __forceinline__ float gemv_out(float acc, float alpha, float beta, const float* y) {
  return beta == 0.f ? __fmul_rn(alpha, acc) : __fmaf_rn(beta, *y, __fmul_rn(alpha, acc));
}

__device__ __forceinline__ float warp_tree(float v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, m));
  return v;
}

// Elements e .. e+3 of a row (STREAM: of S, evict-first) or of x with n valid elements; invalid ones read as 0 and are
// never added (the caller skips steps past the last valid one, and a partial step only pads its own tail).
template <bool VEC, bool STREAM>
__device__ __forceinline__ float4 load4(const float* p, int e, int n) {
  if (VEC && e + 3 < n) return STREAM ? ld_stream4(p + e) : ld_x4(p + e);
  float a[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) a[j] = e + j < n ? (STREAM ? __ldcs(p + e + j) : __ldg(p + e + j)) : 0.f;
  return make_float4(a[0], a[1], a[2], a[3]);
}

// Chunk partials of ROWS rows of equal length that share x: s[rr] points at the chunk start of row rr (nullptr: no
// such row), x at the chunk start of x, n = valid elements of the chunk.  U steps are loaded before they are added.
template <bool VEC, int ROWS, int U>
__device__ __forceinline__ void rowdot_chunk(const float* const (&s)[ROWS], const float* x, int n, int lane,
                                             float (&out)[ROWS]) {
  float a[ROWS][4];
#pragma unroll
  for (int rr = 0; rr < ROWS; ++rr) a[rr][0] = a[rr][1] = a[rr][2] = a[rr][3] = 0.f;
  const int steps = (n + 127) / 128;
  for (int t0 = 0; t0 < steps; t0 += U) {
    float4 sv[ROWS][U], xv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int e = (t0 + u) * 128 + lane * 4;
      const bool live = t0 + u < steps;
      xv[u] = live ? load4<VEC, false>(x, e, n) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr)
        sv[rr][u] = live && s[rr] != nullptr ? load4<VEC, true>(s[rr], e, n) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (t0 + u >= steps) break;
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) {
        a[rr][0] = __fmaf_rn(sv[rr][u].x, xv[u].x, a[rr][0]);
        a[rr][1] = __fmaf_rn(sv[rr][u].y, xv[u].y, a[rr][1]);
        a[rr][2] = __fmaf_rn(sv[rr][u].z, xv[u].z, a[rr][2]);
        a[rr][3] = __fmaf_rn(sv[rr][u].w, xv[u].w, a[rr][3]);
      }
    }
  }
#pragma unroll
  for (int rr = 0; rr < ROWS; ++rr)
    out[rr] = warp_tree(__fadd_rn(__fadd_rn(a[rr][0], a[rr][1]), __fadd_rn(a[rr][2], a[rr][3])));
}

// Row-dot, whole rows per warp: ROWS consecutive rows, every chunk folded in registers.
// carry (may be null) seeds the fold; final: y = alpha*acc + beta*y, else acc_out = acc.
template <bool VEC, int ROWS, int U>
__global__ void __launch_bounds__(256) bof_gemv_rowdot_kernel(int64_t rows, int64_t cols, const float* __restrict__ S,
                                                              int64_t ld, const float* __restrict__ x,
                                                              const float* carry, float* acc_out, float alpha,
                                                              float beta, float* y, int final_out) {
  const int lane = threadIdx.x & 31;
  const int64_t r0 = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * ROWS;
  if (r0 >= rows) return;
  float acc[ROWS];
#pragma unroll
  for (int rr = 0; rr < ROWS; ++rr) acc[rr] = (carry != nullptr && r0 + rr < rows) ? carry[r0 + rr] : 0.f;
  for (int64_t c0 = 0; c0 < cols; c0 += kChunk) {
    const float* s[ROWS];
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) s[rr] = r0 + rr < rows ? S + (r0 + rr) * ld + c0 : nullptr;
    float part[ROWS];
    rowdot_chunk<VEC, ROWS, U>(s, x + c0, (int)min64(kChunk, cols - c0), lane, part);
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) acc[rr] = __fadd_rn(acc[rr], part[rr]);
  }
  if (lane != 0) return;
#pragma unroll
  for (int rr = 0; rr < ROWS; ++rr) {
    const int64_t r = r0 + rr;
    if (r >= rows) break;
    if (final_out) y[r] = gemv_out(acc[rr], alpha, beta, y + r);
    else acc_out[r] = acc[rr];
  }
}

// Row-dot for a few long rows: one warp per (row, chunk), chunk-major so that the warps of one chunk share x in L2;
// partial[ch * rows + r] is folded by bof_gemv_fold_*_kernel.
template <bool VEC>
__global__ void __launch_bounds__(256) bof_gemv_rowdot_split_kernel(int64_t rows, int64_t cols,
                                                                    const float* __restrict__ S, int64_t ld,
                                                                    const float* __restrict__ x, float* partial) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nchunks = (cols + kChunk - 1) / kChunk;
  if (w >= rows * nchunks) return;
  const int64_t ch = w / rows, r = w % rows, c0 = ch * kChunk;
  const float* s[1] = {S + r * ld + c0};
  float part[1];
  rowdot_chunk<VEC, 1, 8>(s, x + c0, (int)min64(kChunk, cols - c0), lane, part);
  if (lane == 0) partial[ch * rows + r] = part[0];
}

// Column-sum chunk partials: block (strip, chunk) of 16 * TPG threads covers 4 * TPG columns of one chunk of rows;
// thread (g, q) runs the fma chains of row group g for columns 4q .. 4q+3 of the strip.
template <bool VEC, int TPG>
__global__ void __launch_bounds__(kGroups * TPG) bof_gemv_colsum_kernel(int64_t rows, int64_t cols,
                                                                        const float* __restrict__ S, int64_t ld,
                                                                        const float* __restrict__ x, float* partial,
                                                                        int64_t nstrips) {
  constexpr int W = 4 * TPG;
  constexpr int U = 8;
  __shared__ float sm[kGroups][W];
  const int64_t strip = (int64_t)blockIdx.x % nstrips, ch = (int64_t)blockIdx.x / nstrips;
  const int g = threadIdx.x / TPG, q = threadIdx.x % TPG;
  const int64_t c = strip * W + 4 * q, row0 = ch * kChunk;
  const int n = (int)min64(kChunk, rows - row0);
  const int ncol = (int)min64(4, cols - c);   // <= 0: this thread's columns are past the edge
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  const float* base = S + row0 * ld + c;
  for (int i0 = g; i0 < n; i0 += U * kGroups) {
    float4 sv[U];
    float xr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * kGroups;
      sv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      xr[u] = 0.f;
      if (i < n && ncol > 0) {
        const float* p = base + (int64_t)i * ld;
        if (VEC && ncol == 4) {
          sv[u] = ld_stream4(p);
        } else {
          sv[u].x = __ldcs(p);
          if (ncol > 1) sv[u].y = __ldcs(p + 1);
          if (ncol > 2) sv[u].z = __ldcs(p + 2);
          if (ncol > 3) sv[u].w = __ldcs(p + 3);
        }
        xr[u] = __ldg(x + row0 + i);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i0 + u * kGroups >= n) break;
      a0 = __fmaf_rn(sv[u].x, xr[u], a0);
      a1 = __fmaf_rn(sv[u].y, xr[u], a1);
      a2 = __fmaf_rn(sv[u].z, xr[u], a2);
      a3 = __fmaf_rn(sv[u].w, xr[u], a3);
    }
  }
  sm[g][4 * q + 0] = a0;
  sm[g][4 * q + 1] = a1;
  sm[g][4 * q + 2] = a2;
  sm[g][4 * q + 3] = a3;
  __syncthreads();
  for (int j = threadIdx.x; j < W; j += blockDim.x) {
    if (strip * W + j >= cols) break;
    float v[kGroups];
#pragma unroll
    for (int k = 0; k < kGroups; ++k) v[k] = sm[k][j];
#pragma unroll
    for (int span = 1; span < kGroups; span *= 2)
#pragma unroll
      for (int k = 0; k < kGroups; k += 2 * span) v[k] = __fadd_rn(v[k], v[k + span]);
    partial[ch * cols + strip * W + j] = v[0];
  }
}

// Fold of chunk partials in ascending chunk order: acc = carry (or +0); acc += partial[ch * ldp + o] for every chunk.
// nchunks == 0 (empty reduction): y = beta * y, or 0 when beta == 0.
__device__ __forceinline__ void fold_store(int64_t o, float acc, bool empty, float* acc_out, float alpha, float beta,
                                           float* y, int final_out) {
  if (!final_out) acc_out[o] = acc;
  else if (empty) y[o] = beta == 0.f ? 0.f : __fmul_rn(beta, y[o]);
  else y[o] = gemv_out(acc, alpha, beta, y + o);
}

// one thread per output (few chunks)
__global__ void __launch_bounds__(256) bof_gemv_fold_thread_kernel(int64_t nout, int64_t nchunks,
                                                                   const float* __restrict__ partial, int64_t ldp,
                                                                   const float* carry, float* acc_out, float alpha,
                                                                   float beta, float* y, int final_out) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= nout) return;
  float acc = carry != nullptr ? carry[o] : 0.f;
  for (int64_t ch = 0; ch < nchunks; ++ch) acc = __fadd_rn(acc, partial[ch * ldp + o]);
  fold_store(o, acc, nchunks == 0 && carry == nullptr, acc_out, alpha, beta, y, final_out);
}

// one warp per output (many chunks): the lanes load 128 partials at a time, every lane adds them in chunk order
__global__ void __launch_bounds__(256) bof_gemv_fold_warp_kernel(int64_t nout, int64_t nchunks,
                                                                 const float* __restrict__ partial, int64_t ldp,
                                                                 const float* carry, float* acc_out, float alpha,
                                                                 float beta, float* y, int final_out) {
  const int lane = threadIdx.x & 31;
  const int64_t o = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (o >= nout) return;
  float acc = carry != nullptr ? carry[o] : 0.f;
  for (int64_t b = 0; b < nchunks; b += 128) {
    float v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t ch = b + lane * 4 + k;
      v[k] = ch < nchunks ? partial[ch * ldp + o] : 0.f;
    }
    const int64_t left = nchunks - b;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float p = __shfl_sync(0xffffffffu, v[k], j);
        if (j * 4 + k < left) acc = __fadd_rn(acc, p);
      }
    }
  }
  if (lane == 0) fold_store(o, acc, false, acc_out, alpha, beta, y, final_out);
}

static int launch_fold(bof_ctx* ctx, cudaStream_t s, int64_t nout, int64_t nchunks, const float* partial, int64_t ldp,
                const float* carry, float* acc_out, float alpha, float beta, float* y, bool final_out) {
  if (nchunks < 32) {
    bof_gemv_fold_thread_kernel<<<(unsigned)ceil_div<int64_t>(nout, 256), 256, 0, s>>>(
        nout, nchunks, partial, ldp, carry, acc_out, alpha, beta, y, final_out);
    BOF_LAUNCH_CHECK(ctx, "bof_gemv_fold_thread_kernel");
  } else {
    bof_gemv_fold_warp_kernel<<<(unsigned)ceil_div<int64_t>(nout, 8), 256, 0, s>>>(
        nout, nchunks, partial, ldp, carry, acc_out, alpha, beta, y, final_out);
    BOF_LAUNCH_CHECK(ctx, "bof_gemv_fold_warp_kernel");
  }
  return BOF_OK;
}

template <bool VEC>
static int launch_rowdot(bof_ctx* ctx, cudaStream_t s, const GemvCanon& c, const float* S, const float* x,
                  const float* carry, float* acc_out, float alpha, float beta, float* y, bool final_out, float* ws) {
  const int64_t nchunks = gemv_chunks(c.cols);
  // few rows: one warp per (row, chunk) and a fold, so that the whole GPU streams them
  const int64_t warps_whole_rows = c.cols <= 512 ? ceil_div<int64_t>(c.rows, 8) : c.rows;
  if (nchunks >= 2 && warps_whole_rows < (int64_t)ctx->num_sms * 16) {
    const int64_t items = c.rows * nchunks;
    bof_gemv_rowdot_split_kernel<VEC><<<(unsigned)ceil_div<int64_t>(items, 8), 256, 0, s>>>(c.rows, c.cols, S, c.ld,
                                                                                           x, ws);
    BOF_LAUNCH_CHECK(ctx, "bof_gemv_rowdot_split_kernel");
    return launch_fold(ctx, s, c.rows, nchunks, ws, c.rows, carry, acc_out, alpha, beta, y, final_out);
  }
  if (c.cols <= 512) {
    bof_gemv_rowdot_kernel<VEC, 8, 1><<<(unsigned)ceil_div<int64_t>(warps_whole_rows, 8), 256, 0, s>>>(
        c.rows, c.cols, S, c.ld, x, carry, acc_out, alpha, beta, y, final_out);
  } else {
    bof_gemv_rowdot_kernel<VEC, 1, 8><<<(unsigned)ceil_div<int64_t>(warps_whole_rows, 8), 256, 0, s>>>(
        c.rows, c.cols, S, c.ld, x, carry, acc_out, alpha, beta, y, final_out);
  }
  BOF_LAUNCH_CHECK(ctx, "bof_gemv_rowdot_kernel");
  return BOF_OK;
}

template <bool VEC, int TPG>
static int launch_colsum_tpg(bof_ctx* ctx, cudaStream_t s, const GemvCanon& c, const float* S, const float* x, float* ws) {
  const int64_t nstrips = ceil_div<int64_t>(c.cols, 4 * TPG), blocks = nstrips * gemv_chunks(c.rows);
  bof_gemv_colsum_kernel<VEC, TPG><<<(unsigned)blocks, kGroups * TPG, 0, s>>>(c.rows, c.cols, S, c.ld, x, ws, nstrips);
  BOF_LAUNCH_CHECK(ctx, "bof_gemv_colsum_kernel");
  return BOF_OK;
}

template <bool VEC>
static int launch_colsum(bof_ctx* ctx, cudaStream_t s, const GemvCanon& c, const float* S, const float* x, float* ws) {
  // columns per strip: the narrowest power-of-two multiple of 4 that covers them, at most 128
  if (c.cols <= 4) return launch_colsum_tpg<VEC, 1>(ctx, s, c, S, x, ws);
  if (c.cols <= 8) return launch_colsum_tpg<VEC, 2>(ctx, s, c, S, x, ws);
  if (c.cols <= 16) return launch_colsum_tpg<VEC, 4>(ctx, s, c, S, x, ws);
  if (c.cols <= 32) return launch_colsum_tpg<VEC, 8>(ctx, s, c, S, x, ws);
  if (c.cols <= 64) return launch_colsum_tpg<VEC, 16>(ctx, s, c, S, x, ws);
  return launch_colsum_tpg<VEC, 32>(ctx, s, c, S, x, ws);
}

int64_t gemv_chunks(int64_t len) { return ceil_div<int64_t>(len, kChunk); }

size_t gemv_workspace_bytes(const GemvCanon& c) {
  if (c.nout() == 0 || c.nred() == 0) return 0;
  return (size_t)gemv_chunks(c.nred()) * (size_t)c.nout() * sizeof(float) + 256;
}

int launch_gemv(bof_ctx* ctx, cudaStream_t s, const GemvCanon& c, const float* S, const float* x, const float* carry,
                float* acc_out, float alpha, float beta, float* y, bool final_out, void* ws) {
  const int64_t nout = c.nout(), nred = c.nred();
  if (nout == 0) return BOF_OK;
  if (nred == 0) return launch_fold(ctx, s, nout, 0, nullptr, 0, carry, acc_out, alpha, beta, y, final_out);
  float* part = reinterpret_cast<float*>(round_up<uintptr_t>(reinterpret_cast<uintptr_t>(ws), 256));
  const bool vec = aligned16(S) && c.ld % 4 == 0 && (!c.rowdot || aligned16(x));
  if (c.rowdot)
    return vec ? launch_rowdot<true>(ctx, s, c, S, x, carry, acc_out, alpha, beta, y, final_out, part)
               : launch_rowdot<false>(ctx, s, c, S, x, carry, acc_out, alpha, beta, y, final_out, part);
  BOF_TRY(vec ? launch_colsum<true>(ctx, s, c, S, x, part) : launch_colsum<false>(ctx, s, c, S, x, part));
  return launch_fold(ctx, s, c.cols, gemv_chunks(c.rows), part, c.cols, carry, acc_out, alpha, beta, y, final_out);
}

}  // namespace bof
