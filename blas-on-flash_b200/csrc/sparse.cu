// K1/K2/K4/K5: CSR x dense (SpMM) and CSR x vector (SpMV) for sm_100a, plus the small
// index/transposition helpers the staging path needs.
//
// Reference bodies replaced:
//   mkl_scsrmm            include/tasks/csrmm_task.h:219-228 (row-major), :290-312 (col-major)
//   mkl_cspblas_scsrgemv  include/tasks/csrgemv_task.h:60-83 ('N'), :152-179 ('T')
//
// Both are HBM/L2-bound gathers: one group of L lanes owns one output row; the (col, val) stream
// of the row is read coalesced with a streaming hint (it is touched exactly once) and each
// nonzero pulls one k-wide row of B as float4 per lane through the read-only path, several rows
// in flight per group so that the gather latency is covered.
#include "common.cuh"

#include <algorithm>

namespace bof {

namespace {

__device__ __forceinline__ float4 ldg_f4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ void fma4(float4& acc, float v, const float4& b) {
  acc.x = fmaf(v, b.x, acc.x);
  acc.y = fmaf(v, b.y, acc.y);
  acc.z = fmaf(v, b.z, acc.z);
  acc.w = fmaf(v, b.w, acc.w);
}

// ---- row splitting (north_star (1): "row-split / merge-path ... warp-per-row segments") ------------------------
// A row group (4..32 lanes) per row is the right shape for the short rows of the BASELINE matrices, but a power-law
// matrix has rows with 10^4..10^6 nonzeros, and one warp walking such a row would outlast the rest of the launch.
// The row kernel therefore only DEFERS them: rows longer than kMidRow go to a list (atomic append -- integer
// bookkeeping only; no floating-point value ever passes through an atomic) and a second, persistent kernel splits
// each of them into 32-nonzero segments over
//   * the 8 warps of one block (rows up to the long threshold), partial sums combined through shared memory in
//     warp order, or
//   * every warp of the grid (rows beyond max(16384, 64 x the mean row length)), block partials combined through a
//     fixed workspace in block order after a grid barrier (all blocks are co-resident),
// so no row occupies one warp for more than kMidRow nonzeros.  The result is deterministic: which tree sums a row
// depends only on its length and the launch's mean, never on the order in which rows were filed (each list has room
// for every row of the launch, so nothing spills from one path to the other).  No host round trip; the workspace is
// two m-entry lists and a grid of partials; a matrix without such rows pays one memset and one empty launch.
constexpr int kMidRow = 1024;            // nonzeros above which a row leaves the row-group kernel
constexpr int kLongRowMin = 16384;       // rows above max(this, kLongRowFactor x mean) are spread over the whole grid
constexpr int kLongRowFactor = 64;

struct LongRows {
  uint32_t* counters;   // [0] rows in mid_list, [1] rows in long_list, [2..3] grid barrier, [4] work ticket
  int32_t* mid_list;
  int32_t* long_list;
};

// L lanes per row, KV float4 per lane: one pass covers 4*L*KV columns starting at
// blockIdx.y * 4*L*KV.  Requires B, C 16-byte aligned, ldb/ldc multiples of 4; the column
// tail (k not a multiple of 4*L) is masked per float4, k itself must be a multiple of 4.
// U = B rows in flight per row group (registers), MINB = resident blocks per SM the register budget is cut
// for: together they set the bytes in flight per SM, which is what bounds this latency-limited gather.
template <int L, int KV, int U, int MINB>
__global__ void __launch_bounds__(256, MINB)
spmm_csr_rm_vec_kernel(int64_t m, int64_t k, float alpha, const float* __restrict__ vals,
                       const int32_t* __restrict__ idx, const int64_t* __restrict__ offs,
                       const float* __restrict__ B, int64_t ldb, float beta, float* __restrict__ C,
                       int64_t ldc, const LongRows lr) {
  constexpr int ROWS_PER_WARP = 32 / L;
  const int lane = threadIdx.x & 31;
  const int sub = lane / L;       // which row of the warp
  const int sl = lane % L;        // lane within the row group
  const int64_t warp_global = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t row = warp_global * ROWS_PER_WARP + sub;
  const int64_t col0 = (int64_t)blockIdx.y * (4 * L * KV) + 4 * sl;
  const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << (sub * L));
  bool row_ok = row < m;

  const int64_t base = offs[0];
  int64_t beg = 0, end = 0;
  if (row_ok) {
    beg = offs[row] - base;
    end = offs[row + 1] - base;
  }
  if (lr.counters != nullptr && end - beg > kMidRow) {
    // deferred to spmm_long_rows_kernel: every column chunk skips the row, chunk 0 files it.  Neither list can
    // overflow: each has room for all m rows.
    if (sl == 0 && blockIdx.y == 0) {
      const int64_t mean = (offs[m] - base) / m;
      if (end - beg > max((int64_t)kLongRowMin, (int64_t)kLongRowFactor * mean))
        lr.long_list[atomicAdd(&lr.counters[1], 1u)] = (int32_t)row;
      else
        lr.mid_list[atomicAdd(&lr.counters[0], 1u)] = (int32_t)row;
    }
    end = beg;
    row_ok = false;
  }

  bool col_ok[KV];
  float4 acc[KV];
#pragma unroll
  for (int v = 0; v < KV; ++v) {
    col_ok[v] = (col0 + (int64_t)v * 4 * L) < k;
    acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  }

  for (int64_t j = beg; j < end; j += L) {
    const int64_t mine = j + sl;
    int32_t c = 0;
    float a = 0.f;
    if (mine < end) {
      c = __ldcs(idx + mine);
      a = __ldcs(vals + mine);
    }
    const int cnt = (int)min((int64_t)L, end - j);  // nonzeros of this chunk (uniform inside the row group)
    int t = 0;
    for (; t + U <= cnt; t += U) {
      int32_t cc[U];
      float aa[U];
      float4 bb[U][KV];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        cc[u] = __shfl_sync(gmask, c, t + u, L);
        aa[u] = __shfl_sync(gmask, a, t + u, L);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float* brow = B + (int64_t)cc[u] * ldb + col0;
#pragma unroll
        for (int v = 0; v < KV; ++v)
          bb[u][v] = col_ok[v] ? ldg_f4(brow + v * 4 * L) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < KV; ++v) fma4(acc[v], aa[u], bb[u][v]);
    }
    for (; t < cnt; ++t) {
      const int32_t cc = __shfl_sync(gmask, c, t, L);
      const float aa = __shfl_sync(gmask, a, t, L);
      const float* brow = B + (int64_t)cc * ldb + col0;
#pragma unroll
      for (int v = 0; v < KV; ++v)
        if (col_ok[v]) fma4(acc[v], aa, ldg_f4(brow + v * 4 * L));
    }
  }

  if (!row_ok) return;
  float* crow = C + row * ldc + col0;
#pragma unroll
  for (int v = 0; v < KV; ++v) {
    if (!col_ok[v]) continue;
    float4 r;
    r.x = alpha * acc[v].x;
    r.y = alpha * acc[v].y;
    r.z = alpha * acc[v].z;
    r.w = alpha * acc[v].w;
    float4* dst = reinterpret_cast<float4*>(crow + v * 4 * L);
    if (beta != 0.f) {
      const float4 old = *dst;
      r.x = fmaf(beta, old.x, r.x);
      r.y = fmaf(beta, old.y, r.y);
      r.z = fmaf(beta, old.z, r.z);
      r.w = fmaf(beta, old.w, r.w);
    }
    __stcs(dst, r);
  }
}

// ---------------------------------------------------------------------------------------------
// TMA-staged variant for the wide shapes (k a multiple of 128): the block's slice of the A stream --
// the (col, val) pairs of its 8 consecutive rows, contiguous in CSR -- is brought into shared memory
// with two 1-D bulk TMA copies (cp.async.bulk + mbarrier complete_tx) issued by one thread, instead of
// per-warp register loads + shuffles; the warps then read (col, val) as smem broadcasts and keep U
// float4 gathers of B rows in flight each.  Slices whose ends are not 16-byte aligned (bulk copies need
// 16-byte aligned addresses and sizes) are staged with ordinary coalesced loads by the whole block.
// Slices larger than the staging buffer are walked in chunks.
// ---------------------------------------------------------------------------------------------
constexpr int SPMM_TMA_CAP = 2048;  // elements per staging chunk: 8 KiB of columns + 8 KiB of values

__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

template <int KV, int U>
__global__ void __launch_bounds__(256, 4)
spmm_csr_rm_tma_kernel(int64_t m, int64_t k, float alpha, const float* __restrict__ vals,
                       const int32_t* __restrict__ idx, const int64_t* __restrict__ offs,
                       const float* __restrict__ B, int64_t ldb, float beta, float* __restrict__ C,
                       int64_t ldc) {
  __shared__ __align__(16) int32_t s_idx[SPMM_TMA_CAP];
  __shared__ __align__(16) float s_val[SPMM_TMA_CAP];
  __shared__ __align__(8) uint64_t s_bar;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t row0 = (int64_t)blockIdx.x * 8;
  const int64_t row = row0 + warp;
  const int64_t col0 = (int64_t)blockIdx.y * (128 * KV) + 4 * lane;
  const int64_t base = offs[0];
  const int64_t seg_beg = offs[row0] - base;
  const int64_t seg_end = offs[min(row0 + 8, m)] - base;
  int64_t beg = 0, end = 0;
  if (row < m) { beg = offs[row] - base; end = offs[row + 1] - base; }

  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr_u32(&s_bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  bool col_ok[KV];
  float4 acc[KV];
#pragma unroll
  for (int v = 0; v < KV; ++v) {
    col_ok[v] = (col0 + (int64_t)v * 128) < k;
    acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  }

  uint32_t parity = 0;
  for (int64_t cs = seg_beg; cs < seg_end; cs += SPMM_TMA_CAP) {
    const int cnt = (int)min((int64_t)SPMM_TMA_CAP, seg_end - cs);
    const bool bulk_ok = ((reinterpret_cast<uintptr_t>(idx + cs) | reinterpret_cast<uintptr_t>(vals + cs)) & 15) == 0 &&
                         (cnt & 3) == 0;
    if (bulk_ok) {
      if (threadIdx.x == 0) {
        const uint32_t bytes = (uint32_t)cnt * 4u;
        const uint32_t bar = smem_addr_u32(&s_bar);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(2u * bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         smem_addr_u32(s_idx)),
                     "l"(idx + cs), "r"(bytes), "r"(bar)
                     : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         smem_addr_u32(s_val)),
                     "l"(vals + cs), "r"(bytes), "r"(bar)
                     : "memory");
      }
      uint32_t done = 0;
      while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_addr_u32(&s_bar)), "r"(parity)
            : "memory");
      }
      parity ^= 1u;
    } else {
      for (int i = threadIdx.x; i < cnt; i += 256) {
        s_idx[i] = __ldcs(idx + cs + i);
        s_val[i] = __ldcs(vals + cs + i);
      }
      __syncthreads();
    }

    // this warp's row, restricted to the chunk
    const int64_t jb = max(beg, cs), je = min(end, cs + cnt);
    int64_t j = jb;
    for (; j + U <= je; j += U) {
      int32_t cc[U];
      float aa[U];
      float4 bb[U][KV];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        cc[u] = s_idx[j - cs + u];
        aa[u] = s_val[j - cs + u];
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float* brow = B + (int64_t)cc[u] * ldb + col0;
#pragma unroll
        for (int v = 0; v < KV; ++v)
          bb[u][v] = col_ok[v] ? ldg_f4(brow + v * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < KV; ++v) fma4(acc[v], aa[u], bb[u][v]);
    }
    for (; j < je; ++j) {
      const int32_t cc = s_idx[j - cs];
      const float aa = s_val[j - cs];
      const float* brow = B + (int64_t)cc * ldb + col0;
#pragma unroll
      for (int v = 0; v < KV; ++v)
        if (col_ok[v]) fma4(acc[v], aa, ldg_f4(brow + v * 128));
    }
    __syncthreads();  // everyone is done with the staging buffers before the next chunk overwrites them
  }

  if (row >= m) return;
  float* crow = C + row * ldc + col0;
#pragma unroll
  for (int v = 0; v < KV; ++v) {
    if (!col_ok[v]) continue;
    float4 r;
    r.x = alpha * acc[v].x;
    r.y = alpha * acc[v].y;
    r.z = alpha * acc[v].z;
    r.w = alpha * acc[v].w;
    float4* dst = reinterpret_cast<float4*>(crow + v * 128);
    if (beta != 0.f) {
      const float4 old = *dst;
      r.x = fmaf(beta, old.x, r.x);
      r.y = fmaf(beta, old.y, r.y);
      r.z = fmaf(beta, old.z, r.z);
      r.w = fmaf(beta, old.w, r.w);
    }
    __stcs(dst, r);
  }
}


// ---- deferred (long) rows ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// all blocks of the (co-resident) grid meet; cnt / gen live in global memory, zero before the launch
__device__ __forceinline__ void grid_barrier(uint32_t* cnt, uint32_t* gen, unsigned nblocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t g = ld_acquire_u32(gen);
    __threadfence();
    if (atomicAdd(cnt, 1u) == nblocks - 1) {
      atomicExch(cnt, 0u);
      __threadfence();
      atomicAdd(gen, 1u);
    } else {
      while (ld_acquire_u32(gen) == g) {}
    }
    __threadfence();
  }
  __syncthreads();
}

constexpr int LR_WARPS = 8;

// Partial sums of the 32-nonzero segments seg0, seg0 + stride, ... of one row, for columns [c0, c0 + 128 KV):
// lane l holds float4 columns c0 + 4 l + 128 v.  U rows of B in flight per warp.
template <int KV>
__device__ __forceinline__ void row_segments(int64_t beg, int64_t end, int64_t seg0, int64_t stride, int64_t c0, int64_t k,
                                             const float* __restrict__ vals, const int32_t* __restrict__ idx,
                                             const float* __restrict__ B, int64_t ldb, float4 (&acc)[KV]) {
  constexpr int U = KV <= 2 ? 4 : 2;   // B rows in flight per warp (8 rows / 4 blocks per SM measured slower: 4.9 vs 3.9 ms)
  const int lane = threadIdx.x & 31;
  bool col_ok[KV];
#pragma unroll
  for (int v = 0; v < KV; ++v) {
    col_ok[v] = c0 + 4 * lane + 128 * v < k;
    acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int64_t nseg = (end - beg + 31) / 32;
  for (int64_t sg = seg0; sg < nseg; sg += stride) {
    const int64_t j = beg + sg * 32;
    const int64_t mine = j + lane;
    int32_t c = 0;
    float a = 0.f;
    if (mine < end) {
      c = __ldcs(idx + mine);
      a = __ldcs(vals + mine);
    }
    const int cnt = (int)min((int64_t)32, end - j);
    for (int t = 0; t < cnt; t += U) {
      int32_t cc[U];
      float aa[U];
      float4 bb[U][KV];
#pragma unroll
      for (int u = 0; u < U; ++u) {   // t, u, cnt are warp-uniform
        cc[u] = __shfl_sync(0xffffffffu, c, (t + u) & 31);
        aa[u] = __shfl_sync(0xffffffffu, a, (t + u) & 31);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const bool live = t + u < cnt;   // past the end of the segment nothing is read (0 * Inf would poison the sum)
        const float* brow = B + (int64_t)(live ? cc[u] : 0) * ldb + c0 + 4 * lane;
        if (!live) aa[u] = 0.f;
#pragma unroll
        for (int v = 0; v < KV; ++v) bb[u][v] = (live && col_ok[v]) ? ldg_f4(brow + 128 * v) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < KV; ++v) fma4(acc[v], aa[u], bb[u][v]);
    }
  }
}

// Persistent kernel over the rows the row-group kernel deferred (see LongRows above).  red: LR_WARPS x 128 KV floats.
template <int KV>
__global__ void __launch_bounds__(LR_WARPS * 32)
spmm_long_rows_kernel(int64_t k, float alpha, const float* __restrict__ vals, const int32_t* __restrict__ idx,
                      const int64_t* __restrict__ offs, const float* __restrict__ B, int64_t ldb, float beta,
                      float* __restrict__ C, int64_t ldc, const LongRows lr, float* __restrict__ partial_ws) {
  constexpr int CW = 128 * KV;   // columns per pass
  __shared__ __align__(16) float red[LR_WARPS][CW];
  __shared__ uint32_t ticket_s;
  const uint32_t n_mid = lr.counters[0], n_long = lr.counters[1];
  if (n_mid == 0 && n_long == 0) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t base = offs[0];
  const unsigned G = gridDim.x;

  auto stash = [&](const float4 (&acc)[KV]) {
#pragma unroll
    for (int v = 0; v < KV; ++v) *reinterpret_cast<float4*>(&red[warp][4 * lane + 128 * v]) = acc[v];
  };

  // ---- rows split over the warps of one block: blocks draw rows from a ticket counter
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) ticket_s = atomicAdd(&lr.counters[4], 1u);
    __syncthreads();
    const uint32_t t = ticket_s;
    if (t >= n_mid) break;
    const int64_t row = lr.mid_list[t];
    const int64_t beg = offs[row] - base, end = offs[row + 1] - base;
    for (int64_t c0 = 0; c0 < k; c0 += CW) {
      float4 acc[KV];
      row_segments<KV>(beg, end, warp, LR_WARPS, c0, k, vals, idx, B, ldb, acc);
      __syncthreads();   // red free again
      stash(acc);
      __syncthreads();
      for (int c = threadIdx.x; c < CW && c0 + c < k; c += LR_WARPS * 32) {
        float sum = 0.f;
#pragma unroll
        for (int w = 0; w < LR_WARPS; ++w) sum += red[w][c];   // warp order: deterministic
        float r = alpha * sum;
        float* dst = C + row * ldc + c0 + c;
        if (beta != 0.f) r = fmaf(beta, *dst, r);
        *dst = r;
      }
    }
  }

  // ---- rows split over every warp of the grid: all blocks walk the list together
  for (uint32_t i = 0; i < n_long; ++i) {
    const int64_t row = lr.long_list[i];
    const int64_t beg = offs[row] - base, end = offs[row + 1] - base;
    for (int64_t c0 = 0; c0 < k; c0 += CW) {
      float4 acc[KV];
      row_segments<KV>(beg, end, (int64_t)blockIdx.x * LR_WARPS + warp, (int64_t)G * LR_WARPS, c0, k, vals, idx, B, ldb, acc);
      __syncthreads();
      stash(acc);
      __syncthreads();
      float* mine = partial_ws + (size_t)blockIdx.x * CW;
      for (int c = threadIdx.x; c < CW; c += LR_WARPS * 32) {
        float sum = 0.f;
#pragma unroll
        for (int w = 0; w < LR_WARPS; ++w) sum += red[w][c];
        mine[c] = sum;
      }
      grid_barrier(&lr.counters[2], &lr.counters[3], G);
      if (blockIdx.x == i % G) {
        for (int c = threadIdx.x; c < CW && c0 + c < k; c += LR_WARPS * 32) {
          float sum = 0.f;
          for (unsigned b = 0; b < G; ++b) sum += __ldcg(partial_ws + (size_t)b * CW + c);   // block order: deterministic
          float r = alpha * sum;
          float* dst = C + row * ldc + c0 + c;
          if (beta != 0.f) r = fmaf(beta, *dst, r);
          *dst = r;
        }
      }
      grid_barrier(&lr.counters[2], &lr.counters[3], G);   // partial_ws may be overwritten again
    }
  }
  // the last block out leaves the counters zeroed for the next launch (an empty launch never touches them)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&lr.counters[5], 1u) == G - 1) {
      for (int i = 0; i < 8; ++i) lr.counters[i] = 0;
    }
  }
}

// Any k, any alignment: a warp owns a row and strides over the columns.
__global__ void __launch_bounds__(256)
spmm_csr_rm_generic_kernel(int64_t m, int64_t k, float alpha, const float* __restrict__ vals,
                           const int32_t* __restrict__ idx, const int64_t* __restrict__ offs,
                           const float* __restrict__ B, int64_t ldb, float beta,
                           float* __restrict__ C, int64_t ldc) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= m) return;
  const int64_t base = offs[0];
  const int64_t beg = offs[row] - base, end = offs[row + 1] - base;
  for (int64_t c0 = 0; c0 < k; c0 += 128) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int64_t j = beg; j < end; ++j) {
      const float a = __ldg(vals + j);
      const float* brow = B + (int64_t)__ldg(idx + j) * ldb + c0;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t cc = lane + 32 * u;
        if (c0 + cc < k) acc[u] = fmaf(a, __ldg(brow + cc), acc[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t cc = c0 + lane + 32 * u;
      if (cc < k) {
        float r = alpha * acc[u];
        if (beta != 0.f) r = fmaf(beta, C[row * ldc + cc], r);
        C[row * ldc + cc] = r;
      }
    }
  }
}

// y = A x : L lanes per row, U nonzeros per lane in flight (the (col, val) stream and the dependent
// x gathers need ~44 KB outstanding per SM to cover HBM latency), shuffle reduction inside the group.
template <int L, int U>
__global__ void __launch_bounds__(256)
spmv_csr_n_kernel(int64_t m, const float* __restrict__ vals, const int32_t* __restrict__ idx,
                  const int64_t* __restrict__ offs, const float* __restrict__ x,
                  float* __restrict__ y) {
  constexpr int ROWS_PER_WARP = 32 / L;
  const int lane = threadIdx.x & 31;
  const int sub = lane / L, sl = lane % L;
  const int64_t row =
      ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * ROWS_PER_WARP + sub;
  const int64_t base = offs[0];
  int64_t beg = 0, end = 0;
  if (row < m) {
    beg = offs[row] - base;
    end = offs[row + 1] - base;
  }
  float acc = 0.f;
  for (int64_t j = beg + sl; j < end; j += L * U) {
    int32_t c[U];
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t jj = j + u * L;
      const bool ok = jj < end;
      c[u] = ok ? __ldcs(idx + jj) : -1;
      v[u] = ok ? __ldcs(vals + jj) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (c[u] >= 0) acc = fmaf(v[u], __ldg(x + c[u]), acc);
  }
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o, L);
  if (row < m && sl == 0) y[row] = acc;
}

// y += A^T x : every nonzero (r, c, v) contributes v * x[r] to y[c]; red.global.add.f32
// replaces the reference's mutex-serialised vector add (csrgemv_task.h:170-176).
template <int L, int U>
__global__ void __launch_bounds__(256)
spmv_csr_t_kernel(int64_t m, const float* __restrict__ vals, const int32_t* __restrict__ idx,
                  const int64_t* __restrict__ offs, const float* __restrict__ x,
                  float* __restrict__ y) {
  constexpr int ROWS_PER_WARP = 32 / L;
  const int lane = threadIdx.x & 31;
  const int sub = lane / L, sl = lane % L;
  const int64_t row =
      ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * ROWS_PER_WARP + sub;
  if (row >= m) return;
  const int64_t base = offs[0];
  const int64_t beg = offs[row] - base, end = offs[row + 1] - base;
  const float xr = __ldg(x + row);
  for (int64_t j = beg + sl; j < end; j += L * U) {
    int32_t c[U];
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t jj = j + u * L;
      const bool ok = jj < end;
      c[u] = ok ? __ldcs(idx + jj) : -1;
      v[u] = ok ? __ldcs(vals + jj) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (c[u] >= 0) atomicAdd(y + c[u], v[u] * xr);
  }
}

__global__ void idx_narrow_kernel(const int64_t* __restrict__ in, int32_t* __restrict__ out,
                                  int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (int32_t)__ldcs(in + i);
}
__global__ void idx_widen_kernel(const int32_t* __restrict__ in, int64_t* __restrict__ out,
                                 int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (int64_t)__ldcs(in + i);
}

// out[c*ldo + r] = alpha * in[r*ldi + c] + beta * out[c*ldo + r]; 32x32 smem tiles, +1 padding.
template <bool AXPBY>
__global__ void __launch_bounds__(256)
transpose_kernel(int64_t rows, int64_t cols, float alpha, const float* __restrict__ in,
                 int64_t ldi, float beta, float* __restrict__ out, int64_t ldo,
                 unsigned tiles_c) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  // linear tile index: either extent may exceed the 65535 limit of grid.y
  const int64_t r0 = (int64_t)(blockIdx.x / tiles_c) * 32, c0 = (int64_t)(blockIdx.x % tiles_c) * 32;
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int64_t r = r0 + i, c = c0 + tx;
    tile[i][tx] = (r < rows && c < cols) ? in[r * ldi + c] : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int64_t c = c0 + i, r = r0 + tx;
    if (r < rows && c < cols) {
      float v = tile[tx][i];
      if (AXPBY) {
        v *= alpha;
        if (beta != 0.f) v = fmaf(beta, out[c * ldo + r], v);
      }
      out[c * ldo + r] = v;
    }
  }
}

template <int KV, int U>
int spmm_tma_launch(bof_ctx* ctx, cudaStream_t s, int64_t m, int64_t k, float alpha, const float* vals,
                    const int32_t* idx, const int64_t* offs, const float* B, int64_t ldb, float beta, float* C,
                    int64_t ldc) {
  dim3 grid((unsigned)ceil_div<int64_t>(m, 8), (unsigned)ceil_div<int64_t>(k, 128 * KV));
  spmm_csr_rm_tma_kernel<KV, U><<<grid, 256, 0, s>>>(m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc);
  BOF_LAUNCH_CHECK(ctx, "spmm_csr_rm_tma_kernel");
  return BOF_OK;
}


template <int KV>
int long_rows_launch(bof_ctx* ctx, cudaStream_t s, int grid, int64_t k, float alpha, const float* vals, const int32_t* idx,
                     const int64_t* offs, const float* B, int64_t ldb, float beta, float* C, int64_t ldc,
                     const LongRows& lr, float* partial_ws) {
  spmm_long_rows_kernel<KV><<<grid, LR_WARPS * 32, 0, s>>>(k, alpha, vals, idx, offs, B, ldb, beta, C, ldc, lr, partial_ws);
  BOF_LAUNCH_CHECK(ctx, "spmm_long_rows_kernel");
  return BOF_OK;
}

template <int L, int KV, int U = 4, int MINB = 4>
int spmm_vec_launch(bof_ctx* ctx, cudaStream_t s, int64_t m, int64_t k, float alpha,
                    const float* vals, const int32_t* idx, const int64_t* offs, const float* B,
                    int64_t ldb, float beta, float* C, int64_t ldc) {
  constexpr int ROWS_PER_BLOCK = 8 * (32 / L);
  dim3 grid((unsigned)ceil_div<int64_t>(m, ROWS_PER_BLOCK),
            (unsigned)ceil_div<int64_t>(k, 4 * L * KV));
  // state of the deferred-row path: [counters 256 B | long_list m_cap | partials G x 512 floats | mid_list m_cap]
  static const bool defer = getenv("BOF_SPMM_NO_SPLIT") == nullptr;
  LongRows lr{nullptr, nullptr, nullptr};
  float* partial_ws = nullptr;
  int lgrid = 0;
  if (defer && m < (1ll << 31)) {
    const int kv = k <= 128 ? 1 : (k <= 256 ? 2 : 4);
    static int occ[3] = {-1, -1, -1};   // blocks per SM of the three instantiations (same for every B200)
    int& per_sm = occ[kv == 1 ? 0 : (kv == 2 ? 1 : 2)];
    cudaError_t oe = cudaSuccess;
    if (per_sm < 0)
      oe = kv == 1 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, spmm_long_rows_kernel<1>, LR_WARPS * 32, 0)
         : kv == 2 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, spmm_long_rows_kernel<2>, LR_WARPS * 32, 0)
                   : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, spmm_long_rows_kernel<4>, LR_WARPS * 32, 0);
    if (oe == cudaSuccess && per_sm > 0) {
      lgrid = ctx->num_sms * std::min(per_sm, 2);   // co-resident by construction: the grid barrier relies on it
      size_t m_cap = 1024;
      while ((int64_t)m_cap < m) m_cap <<= 1;       // power-of-two sizing: a streamed pipeline regrows the slot rarely
      const size_t bytes = 256 + m_cap * 4 + (size_t)lgrid * 512 * 4 + m_cap * 4;
      void* p = nullptr;
      const size_t had = ctx->slot_bytes[kSlotSpmmLong];
      { const int rc_slot = slot_reserve(ctx, kSlotSpmmLong, bytes, &p); if (rc_slot != BOF_OK) return rc_slot; }
      // fresh memory: the counters start at zero; afterwards the long-row kernel leaves them zeroed itself
      if (ctx->slot_bytes[kSlotSpmmLong] != had) BOF_CUDA(ctx, cudaMemsetAsync(p, 0, 256, s));
      uint8_t* b8 = static_cast<uint8_t*>(p);
      lr.counters = reinterpret_cast<uint32_t*>(b8);
      lr.long_list = reinterpret_cast<int32_t*>(b8 + 256);
      partial_ws = reinterpret_cast<float*>(b8 + 256 + m_cap * 4);
      lr.mid_list = reinterpret_cast<int32_t*>(b8 + 256 + m_cap * 4 + (size_t)lgrid * 512 * 4);
    } else {
      cudaGetLastError();
    }
  }
  spmm_csr_rm_vec_kernel<L, KV, U, MINB><<<grid, 256, 0, s>>>(m, k, alpha, vals, idx, offs, B, ldb, beta,
                                                              C, ldc, lr);
  BOF_LAUNCH_CHECK(ctx, "spmm_csr_rm_vec_kernel");
  if (lr.counters != nullptr) {
    if (k <= 128) return long_rows_launch<1>(ctx, s, lgrid, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc, lr, partial_ws);
    if (k <= 256) return long_rows_launch<2>(ctx, s, lgrid, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc, lr, partial_ws);
    return long_rows_launch<4>(ctx, s, lgrid, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc, lr, partial_ws);
  }
  return BOF_OK;
}

}  // namespace

int launch_spmm_rm(bof_ctx* ctx, cudaStream_t s, int64_t m, int64_t k, float alpha,
                   const float* vals, const int32_t* idx, const int64_t* offs, const float* B,
                   int64_t ldb, float beta, float* C, int64_t ldc, int64_t b_rows) {
  if (m == 0 || k == 0) return BOF_OK;
  const bool vec_ok =
      (k % 4 == 0) && (ldb % 4 == 0) && (ldc % 4 == 0) && aligned16(B) && aligned16(C);
  if (!vec_ok) {
    spmm_csr_rm_generic_kernel<<<(unsigned)ceil_div<int64_t>(m, 8), 256, 0, s>>>(
        m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc);
    BOF_LAUNCH_CHECK(ctx, "spmm_csr_rm_generic_kernel");
    return BOF_OK;
  }
#define BOF_SPMM(L, KV) \
  return spmm_vec_launch<L, KV>(ctx, s, m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc)
  if (k <= 16) BOF_SPMM(4, 1);
  if (k <= 32) BOF_SPMM(8, 1);
  if (k <= 64) BOF_SPMM(16, 1);
  // Bytes-in-flight tuning of the two wide shapes (profiles/r01/spmm_variants.txt): with B ~ L2-sized (cfg-1)
  // 8 rows in flight at 4 blocks/SM is 31 % faster than 4 rows; with B >> L2 (cfg-3) every variant sits at the
  // DRAM gather limit.  BOF_SPMM_VARIANT overrides (0..5) for experiments.
  static const int variant = getenv("BOF_SPMM_VARIANT") ? atoi(getenv("BOF_SPMM_VARIANT")) : -1;
#define BOF_SPMM_V(L, KV, U, MINB) \
  return spmm_vec_launch<L, KV, U, MINB>(ctx, s, m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc)
  if (variant == 6 && k > 64)  // TMA-staged A stream
    return (k <= 128) ? spmm_tma_launch<1, 8>(ctx, s, m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc)
                      : spmm_tma_launch<2, 4>(ctx, s, m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc);
  if (variant == 7 && k > 64)
    return (k <= 128) ? spmm_tma_launch<1, 4>(ctx, s, m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc)
                      : spmm_tma_launch<2, 8>(ctx, s, m, k, alpha, vals, idx, offs, B, ldb, beta, C, ldc);
  // B larger than L2 can hold next to the A stream, but a 64-column slice of it fits: gather from one slice at a
  // time (cfg-1: B = 134 MB against 126 MB of L2; 0.675 -> 0.602 ms, profiles/r01/spmm_variants.txt).  For a B
  // far beyond L2 (cfg-3) the slices do not fit either and the extra passes over A would only cost.
  const bool l2_slices = b_rows > 0 && ldb == k && (double)b_rows * ldb * 4 > 0.5 * (double)ctx->l2_bytes &&
                         (double)b_rows * 64 * 4 <= 0.7 * (double)ctx->l2_bytes;
  if ((variant < 0 && l2_slices) || variant == 12) BOF_SPMM_V(16, 1, 8, 4);
  if (k <= 128) {
    switch (variant) {
      // 64-column chunks (grid.y = 2, all row blocks of chunk 0 are scheduled before chunk 1): half of B at a time
      // is the gather target, which fits L2 when the whole B does not
      case 8: BOF_SPMM_V(16, 1, 8, 4);
      case 9: BOF_SPMM_V(16, 1, 4, 4);
      case 10: BOF_SPMM_V(16, 1, 16, 2);
      case 11: BOF_SPMM_V(16, 1, 16, 3);
      case 1: BOF_SPMM_V(32, 1, 4, 5);
      case 2: BOF_SPMM_V(32, 1, 4, 6);
      case 3: BOF_SPMM_V(32, 1, 8, 3);
      case 4: BOF_SPMM_V(32, 1, 8, 4);
      case 5: BOF_SPMM_V(32, 1, 16, 2);
      case 0: BOF_SPMM_V(32, 1, 4, 4);
      default: BOF_SPMM_V(32, 1, 8, 4);
    }
  }
  switch (variant) {
    case 1: BOF_SPMM_V(32, 2, 4, 5);
    case 2: BOF_SPMM_V(32, 2, 4, 6);
    case 3: BOF_SPMM_V(32, 2, 8, 3);
    case 4: BOF_SPMM_V(32, 2, 8, 4);
    case 5: BOF_SPMM_V(32, 2, 16, 2);
    default: BOF_SPMM_V(32, 2, 4, 4);
  }
#undef BOF_SPMM_V
#undef BOF_SPMM
}

// KMeansTask::execute's two rank-1 updates (include/tasks/kmeans_task.h:74-80) on a row-major block:
// C[r, c] = (C[r, c] + first) + second with first/second = rowv[r], colv[c] in the order `row_first` says.
namespace {
__global__ void __launch_bounds__(256)
add_outer_terms_kernel(float* __restrict__ C, int64_t rows, int64_t cols, int64_t ldc, const float* __restrict__ rowv,
                       const float* __restrict__ colv, int row_first) {
  const int64_t total = rows * cols, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t r = i / cols, c = i - r * cols;
    float v = C[r * ldc + c];
    const float a = rowv[r], b = __ldg(colv + c);
    v = row_first ? __fadd_rn(__fadd_rn(v, a), b) : __fadd_rn(__fadd_rn(v, b), a);
    C[r * ldc + c] = v;
  }
}
}  // namespace

int launch_add_outer_terms(bof_ctx* ctx, cudaStream_t s, float* C, int64_t rows, int64_t cols, int64_t ldc,
                           const float* rowv, const float* colv, int row_first) {
  if (rows == 0 || cols == 0) return BOF_OK;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(rows * cols, 256), (int64_t)ctx->num_sms * 16);
  add_outer_terms_kernel<<<grid, 256, 0, s>>>(C, rows, cols, ldc, rowv, colv, row_first);
  BOF_LAUNCH_CHECK(ctx, "add_outer_terms_kernel");
  return BOF_OK;
}

int launch_spmv(bof_ctx* ctx, cudaStream_t s, char trans, int64_t m, int64_t n, const float* vals,
                const int32_t* idx, const int64_t* offs, const float* x, float* y, int64_t nnz) {
  // 'T' zeroes y first (src/blas/csrgemv.cpp:64); 't' accumulates into y as it is, which is
  // what a row-block pipeline needs for every block after the memset.
  if (trans == 'T' || trans == 't') {
    if (ctx->cfg.spmv_t_atomic != 0) {
      if (trans == 'T') BOF_CUDA(ctx, cudaMemsetAsync(y, 0, (size_t)n * sizeof(float), s));
      if (m == 0) return BOF_OK;
      spmv_csr_t_kernel<16, 4><<<(unsigned)ceil_div<int64_t>(m, 16), 256, 0, s>>>(m, vals, idx, offs, x, y);
      BOF_LAUNCH_CHECK(ctx, "spmv_csr_t_kernel");
      return BOF_OK;
    }
    if (nnz < 0 && m > 0) {   // device-tile callers hand over device offsets only: one small read-back
      int64_t ends[2] = {0, 0};
      BOF_CUDA(ctx, cudaMemcpyAsync(&ends[0], offs, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
      BOF_CUDA(ctx, cudaMemcpyAsync(&ends[1], offs + m, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
      BOF_CUDA(ctx, cudaStreamSynchronize(s));
      nnz = ends[1] - ends[0];
    }
    nnz = std::max<int64_t>(nnz, 0);
    const size_t wsb = spmv_t_workspace_bytes(n, nnz);
    void* ws = nullptr;
    { const int rc = slot_reserve(ctx, kSlotSpmvT, wsb, &ws); if (rc != BOF_OK) return rc; }
    return launch_spmv_t_sorted(ctx, s, trans == 't' ? 1 : 0, m, n, nnz, vals, idx, offs, x, y, ws, wsb);
  }
  if (m == 0) return BOF_OK;
  spmv_csr_n_kernel<16, 4><<<(unsigned)ceil_div<int64_t>(m, 16), 256, 0, s>>>(m, vals, idx, offs, x, y);
  BOF_LAUNCH_CHECK(ctx, "spmv_csr_n_kernel");
  return BOF_OK;
}

int launch_idx_narrow(bof_ctx* ctx, cudaStream_t s, const int64_t* in, int32_t* out, int64_t n) {
  if (n == 0) return BOF_OK;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(n, 256), (int64_t)ctx->num_sms * 16);
  idx_narrow_kernel<<<grid, 256, 0, s>>>(in, out, n);
  BOF_LAUNCH_CHECK(ctx, "idx_narrow_kernel");
  return BOF_OK;
}

int launch_idx_widen(bof_ctx* ctx, cudaStream_t s, const int32_t* in, int64_t* out, int64_t n) {
  if (n == 0) return BOF_OK;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(n, 256), (int64_t)ctx->num_sms * 16);
  idx_widen_kernel<<<grid, 256, 0, s>>>(in, out, n);
  BOF_LAUNCH_CHECK(ctx, "idx_widen_kernel");
  return BOF_OK;
}

int launch_transpose(bof_ctx* ctx, cudaStream_t s, int64_t rows, int64_t cols, const float* in,
                     int64_t ldi, float* out, int64_t ldo) {
  if (rows == 0 || cols == 0) return BOF_OK;
  const int64_t tiles_c = ceil_div<int64_t>(cols, 32), tiles_r = ceil_div<int64_t>(rows, 32);
  BOF_REQUIRE(ctx, tiles_c * tiles_r < (1ll << 31), "transpose: matrix too large for one launch");
  transpose_kernel<false><<<(unsigned)(tiles_c * tiles_r), 256, 0, s>>>(rows, cols, 1.f, in, ldi, 0.f,
                                                                       out, ldo, (unsigned)tiles_c);
  BOF_LAUNCH_CHECK(ctx, "transpose_kernel");
  return BOF_OK;
}

int launch_transpose_axpby(bof_ctx* ctx, cudaStream_t s, int64_t rows, int64_t cols, float alpha,
                           const float* in, int64_t ldi, float beta, float* out, int64_t ldo) {
  if (rows == 0 || cols == 0) return BOF_OK;
  const int64_t tiles_c = ceil_div<int64_t>(cols, 32), tiles_r = ceil_div<int64_t>(rows, 32);
  BOF_REQUIRE(ctx, tiles_c * tiles_r < (1ll << 31), "transpose: matrix too large for one launch");
  transpose_kernel<true><<<(unsigned)(tiles_c * tiles_r), 256, 0, s>>>(rows, cols, alpha, in, ldi, beta,
                                                                      out, ldo, (unsigned)tiles_c);
  BOF_LAUNCH_CHECK(ctx, "transpose_kernel");
  return BOF_OK;
}

}  // namespace bof
