// K3 / K8+K9: fp32 GEMM on the 5th-gen tensor cores (tcgen05 + TMEM) with a three-term operand split,
// and the k-means distance/argmin step that reuses the same main loop with a fused epilogue.
//
// Reference bodies replaced:
//   cblas_sgemm                 include/tasks/gemm_task.h:87-90
//   cblas_sgemm x3 (+ isamin)   include/tasks/kmeans_task.h:68-80, drivers/in_mem_kmeans.cpp:82-85
//
// Canonical form.  Every (order, transA, transB) combination is reduced by the caller to
//     acc[i, j] = sum_k P[i, k] * Q[j, k]
// with both operands K-major.  Each operand is stored as two planes produced by split_planes_* below
// (one pass over the operand, negligible next to the 2*M*N*K flops): hi = rna_tf32(x), and either
//   gemm_split = 1 ("3xTF32"): lo = rna_tf32(x - hi); product = lo*hi + hi*lo + hi*hi, all kind::tf32;
//   gemm_split = 2 (hybrid, default): bf16(hi) and bf16(x - hi) interleaved per 32-element k group;
//       hi*hi runs on the tf32 pipe, the two cross terms (each ~2^-11 of the product, so 8 mantissa
//       bits keep their error below 2^-19) on the bf16 pipe at twice the rate: 2/3 of the tensor time
//       of 3xTF32 and fewer truncating accumulations.  Measured at 32768^3: 337 vs 269 TFLOP/s,
//       rel. Frobenius error 1.8e-6 vs 2.3e-6 (profiles/r01/suite_split.json).
// lo*lo ~ 2^-22 is dropped in both.
//
// Kernel shape (per CTA; `CG` = tcgen05 cta_group, 1 or 2 SMs cooperating on one tile):
//   tile     (128*CG) x BLOCK_N, BLOCK_N = 128 (CG=1) or 256 (CG=2); every CTA owns 128 rows
//            (= 128 TMEM lanes) and loads 128 rows of Q per stage.
//   stage    32 k-elements (one 128-byte swizzle row): P_hi, P_lo, Q_hi, Q_lo = 4 x 16 KiB
//   warps    WG0: w0 TMA producer, w1 MMA issuer (leader CTA), w2 TMEM allocator
//            WG1+WG2: 8 epilogue warps, warp e reads TMEM lanes 32*(e%4).., column half e/4
//   TMEM     two accumulator buffers of BLOCK_N columns: the MMA warp fills one while the
//            epilogue drains the other.
//   k-chunks the tensor core accumulates at most `k_chunk` elements of k into TMEM; the epilogue
//            warps then fold the chunk into fp32 registers with round-to-nearest adds.  This
//            bounds the error of the tensor core's internal accumulation for very long k.
#include "common.cuh"

#include <cuda_bf16.h>

#ifndef BOF_DEFAULT_HYBRID
#define BOF_DEFAULT_HYBRID 1
#endif

namespace bof {
namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 32;  // fp32 elements per stage row: 128 bytes
constexpr int UMMA_K = 8;    // tf32 elements per tcgen05.mma
constexpr int LOAD_N = 128;  // rows of Q each CTA loads per stage
constexpr int STAGES = 3;
constexpr int PLANE_BYTES = 128 * BLOCK_K * 4;  // 16 KiB
constexpr int STAGE_BYTES = 4 * PLANE_BYTES;    // P_hi, P_lo, Q_hi, Q_lo
constexpr int NUM_THREADS = 384;
constexpr int NUM_EPI_WARPS = 8;
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;  // clears the CTA-pair peer bit of a smem address

enum EpiMode { EPI_GEMM = 0, EPI_ARGMIN = 1 };

struct Params {
  int64_t M, N;
  int32_t num_kb;         // k-blocks of 32
  int32_t kb_per_chunk;   // k-blocks per TMEM accumulation chunk
  int32_t tiles_m, tiles_n;
  int32_t n_per_item;     // EPI_GEMM: 1; EPI_ARGMIN: tiles_n (a work item walks all N tiles)
  float alpha, beta;
  float* C;
  int64_t ldc;
  const float* row_add;
  const float* col_add;
  int32_t* argmin_out;
  // Wave lock-step (EPI_GEMM, long k): every `sync_kb` k-blocks the leader producers of the
  // clusters working on the same wave of tiles meet at a global counter, so that the wave's
  // operand panels stay inside L2 (measured without it at 32768^3: L2 hit rate 36%, DRAM 59% busy).
  uint32_t* sync_counters;
  int32_t sync_kb;
  // FOLD variant (EPI_GEMM, k-panels of an out-of-core GEMM): chunk 0 of every element starts from
  // carry[row * ld_carry + col] when carry != nullptr; raw_out != 0 stores the un-scaled fold to C
  // (no alpha, no beta, C not read), so that the next k-panel can resume it.
  const float* carry;
  int64_t ld_carry;
  int32_t raw_out;
};

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Parity wait with a watchdog: a protocol bug traps (-> CUDA error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  uint64_t t0 = 0;
  uint32_t spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) break;
    if ((++spins & 0xfffu) == 0) {
      const uint64_t now = globaltimer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// Arrive on the barrier at the same smem offset in the pair's leader CTA (valid from either CTA).
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_BIT_MASK) : "memory");
}

template <int CG>
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* full_bar, void* dst,
                                            int32_t c_inner, int32_t c_outer) {
  if constexpr (CG == 2) {
    // Both CTAs of the pair signal the leader's barrier (peer bit cleared).
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(full_bar) & PEER_BIT_MASK), "r"(c_inner),
        "r"(c_outer)
        : "memory");
  } else {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(full_bar)), "r"(c_inner), "r"(c_outer)
        : "memory");
  }
}

template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  if constexpr (CG == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (CG == 2)
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// D[tmem] (+)= A[smem] * B[smem], kind::tf32
template <int CG>
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// D[tmem] (+)= A[smem] * B[smem], kind::f16 (bf16 operands selected by the instruction descriptor)
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// Arrive on `bar` (same offset in every CTA of the pair) once all previously issued MMAs retire.
template <int CG>
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  if constexpr (CG == 2) {
    const uint16_t mask = 0b11;
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"(mask)
        : "memory");
  } else {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  }
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (SBO), LBO unused.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);        // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                        // leading byte offset (ignored for SW128 K-major)
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                        // layout: SWIZZLE_128B
  return d;
}
// fp32 accumulate, both operands K-major; fmt: 2 = TF32 (kind::tf32), 1 = BF16 (kind::f16)
__host__ __device__ constexpr uint32_t make_idesc(int umma_m, int umma_n, uint32_t fmt = 2u) {
  return (1u << 4)                      // c_format = F32
         | (fmt << 7) | (fmt << 10)     // a_format = b_format
         | ((uint32_t)(umma_n >> 3) << 17) | ((uint32_t)(umma_m >> 4) << 24);
}

template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

struct SmemTail {
  uint64_t full[STAGES];
  uint64_t empty[STAGES];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
  float red_val[BLOCK_M];   // EPI_ARGMIN: exchange between the two column halves
  int32_t red_idx[BLOCK_M];
};

constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + sizeof(SmemTail) + 1024;

// ---------------------------------------------------------------------------------------------
// The kernel
// ---------------------------------------------------------------------------------------------
template <int CG, int EPI, bool CHUNKED, bool HYB, bool FOLD = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm3xtf32_kernel(const __grid_constant__ CUtensorMap map_p_hi, const __grid_constant__ CUtensorMap map_p_lo,
                  const __grid_constant__ CUtensorMap map_q_hi, const __grid_constant__ CUtensorMap map_q_lo,
                  const Params prm) {
  constexpr int BLOCK_N = (CG == 2) ? 256 : 128;
  constexpr int TILE_M = BLOCK_M * CG;
  constexpr int EPI_COLS = BLOCK_N / 2;  // columns per epilogue thread
  constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;
  constexpr uint32_t IDESC = make_idesc(BLOCK_M * CG, BLOCK_N, 2u);
  constexpr uint32_t IDESC_BF16 = make_idesc(BLOCK_M * CG, BLOCK_N, 1u);
  static_assert(!FOLD || (EPI == EPI_GEMM && CHUNKED), "the fold carry exists for the chunked GEMM epilogue only");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  SmemTail* tail = reinterpret_cast<SmemTail*>(smem + (size_t)STAGES * STAGE_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0u;
  const bool is_leader = cta_rank == 0;
  const int cluster_id = blockIdx.x / CG;
  const int num_clusters = gridDim.x / CG;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&tail->full[s], CG);   // one arrival per CTA's producer (+ the TMA bytes)
      mbar_init(&tail->empty[s], 1);   // tcgen05.commit
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tail->tmem_full[b], 1);                     // tcgen05.commit
      mbar_init(&tail->tmem_empty[b], NUM_EPI_WARPS * CG);   // every epilogue warp of the pair
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<CG>(&tail->tmem_base, TMEM_COLS);
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tail->tmem_base;

  const int num_items = (EPI == EPI_ARGMIN) ? prm.tiles_m : prm.tiles_m * prm.tiles_n;
  const int num_chunks = (prm.num_kb + prm.kb_per_chunk - 1) / prm.kb_per_chunk;

  // Grouped rasterisation: consecutive items walk 8 M-tiles before moving along N, so that the
  // clusters running concurrently share operand tiles in L2.
  auto decode_item = [&](int item, int& tm, int& tn0) {
    if (EPI == EPI_ARGMIN) { tm = item; tn0 = 0; return; }
    constexpr int GROUP = 8;
    const int per_group = GROUP * prm.tiles_n;
    const int g = item / per_group;
    const int first_m = g * GROUP;
    const int gsz = min(GROUP, prm.tiles_m - first_m);
    const int r = item - g * per_group;
    tm = first_m + r % gsz;
    tn0 = r / gsz;
  };

  if (warp < 4) {
    if constexpr (CHUNKED) setmaxnreg_dec<40>();
    if (warp == 0) {
      // ===================== TMA producer (every CTA) =====================
      int stage = 0;
      uint32_t phase = 0;
      for (int item = cluster_id; item < num_items; item += num_clusters) {
        int tm, tn0;
        decode_item(item, tm, tn0);
        const int32_t row_p = tm * TILE_M + (int)cta_rank * BLOCK_M;
        for (int nt = 0; nt < prm.n_per_item; ++nt) {
          const int32_t row_q = (tn0 + nt) * BLOCK_N + (int)cta_rank * LOAD_N;
          for (int kb = 0; kb < prm.num_kb; ++kb) {
            mbar_wait(&tail->empty[stage], phase ^ 1);
            if (EPI == EPI_GEMM && prm.sync_kb > 0 && is_leader && lane == 0 && kb % prm.sync_kb == 0) {
              // all clusters are co-resident (persistent grid <= #SMs, one CTA per SM): spinning is safe
              const int wave = (item - cluster_id) / num_clusters;
              const int syncs_per_tile = (prm.num_kb + prm.sync_kb - 1) / prm.sync_kb;
              const uint32_t expected = (uint32_t)min(num_clusters, num_items - wave * num_clusters);
              uint32_t* ctr = prm.sync_counters + (size_t)wave * syncs_per_tile + kb / prm.sync_kb;
              asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
              // Soft barrier: it only paces the producers for L2 locality, so a cluster that cannot see
              // its peers within 0.5 ms (e.g. the grid is not fully resident because another stream
              // holds SMs) simply goes on -- correctness never depends on the rendezvous.
              uint32_t seen = 0;
              const uint64_t t0 = globaltimer_ns();
              for (uint32_t spins = 0;; ++spins) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(ctr) : "memory");
                if (seen >= expected) break;
                __nanosleep(100);
                if ((spins & 0x3fu) == 0x3fu && globaltimer_ns() - t0 > 500000ull) break;
              }
            }
            if (lane == 0) {
              uint8_t* st = smem + (size_t)stage * STAGE_BYTES;
              if (is_leader) mbar_arrive_expect_tx(&tail->full[stage], STAGE_BYTES * CG);
              else mbar_arrive_leader(&tail->full[stage]);
              const int32_t kc = kb * BLOCK_K;
              tma_load_2d<CG>(&map_p_hi, &tail->full[stage], st, kc, row_p);
              tma_load_2d<CG>(&map_p_lo, &tail->full[stage], st + PLANE_BYTES, kc, row_p);
              tma_load_2d<CG>(&map_q_hi, &tail->full[stage], st + 2 * PLANE_BYTES, kc, row_q);
              tma_load_2d<CG>(&map_q_lo, &tail->full[stage], st + 3 * PLANE_BYTES, kc, row_q);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    } else if (warp == 1 && is_leader) {
      // ===================== MMA issuer (leader CTA of the pair) =====================
      int stage = 0;
      uint32_t phase = 0;
      uint32_t acc_iter = 0;
      for (int item = cluster_id; item < num_items; item += num_clusters) {
        for (int nt = 0; nt < prm.n_per_item; ++nt) {
          for (int c = 0; c < num_chunks; ++c, ++acc_iter) {
            const uint32_t buf = acc_iter & 1u;
            mbar_wait(&tail->tmem_empty[buf], ((acc_iter >> 1) & 1u) ^ 1u);
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + buf * BLOCK_N;
            const int kb_end = min(prm.num_kb, (c + 1) * prm.kb_per_chunk);
            for (int kb = c * prm.kb_per_chunk; kb < kb_end; ++kb) {
              mbar_wait(&tail->full[stage], phase);
              tc_fence_after();
              if (lane == 0) {
                const uint32_t st = smem_u32(smem + (size_t)stage * STAGE_BYTES);
                const uint64_t d_p_hi = make_smem_desc(st);
                const uint64_t d_p_lo = make_smem_desc(st + PLANE_BYTES);
                const uint64_t d_q_hi = make_smem_desc(st + 2 * PLANE_BYTES);
                const uint64_t d_q_lo = make_smem_desc(st + 3 * PLANE_BYTES);
                const uint32_t fresh = (kb == c * prm.kb_per_chunk) ? 0u : 1u;  // first MMA of a chunk overwrites
                if constexpr (HYB) {
                  // Second plane = bf16 pairs per 32-k group: bytes [0,64) bf16(hi), [64,128) bf16(lo).
                  // Cross terms on the bf16 pipe (K = 16 per MMA = 32 B), hi*hi on the tf32 pipe.
#pragma unroll
                  for (int kk = 0; kk < 2; ++kk) {
                    const uint64_t adv = (uint64_t)(kk * 2);                  // 32 B per k-step of 16 bf16
                    umma_bf16<CG>(tmem_d, d_p_lo + 4 + adv, d_q_lo + adv, IDESC_BF16, kk == 0 ? fresh : 1u);  // lo * hi
                    umma_bf16<CG>(tmem_d, d_p_lo + adv, d_q_lo + 4 + adv, IDESC_BF16, 1u);                    // hi * lo
                  }
#pragma unroll
                  for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
                    const uint64_t adv = (uint64_t)((kk * UMMA_K * 4) >> 4);
                    umma_tf32<CG>(tmem_d, d_p_hi + adv, d_q_hi + adv, IDESC, 1u);
                  }
                } else {
#pragma unroll
                  for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
                    const uint64_t adv = (uint64_t)((kk * UMMA_K * 4) >> 4);  // 32 B per k-step
                    umma_tf32<CG>(tmem_d, d_p_lo + adv, d_q_hi + adv, IDESC, kk == 0 ? fresh : 1u);
                    umma_tf32<CG>(tmem_d, d_p_hi + adv, d_q_lo + adv, IDESC, 1u);
                    umma_tf32<CG>(tmem_d, d_p_hi + adv, d_q_hi + adv, IDESC, 1u);
                  }
                }
                umma_commit<CG>(&tail->empty[stage]);  // frees the stage in both CTAs
                if (kb == kb_end - 1) umma_commit<CG>(&tail->tmem_full[buf]);
              }
              __syncwarp();
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else {
    // ===================== epilogue warps (every CTA) =====================
    if constexpr (CHUNKED) setmaxnreg_inc<232>();
    const int e = warp - 4;
    const int quarter = e & 3;  // TMEM lane quarter this warp may access
    const int half = e >> 2;    // which half of the BLOCK_N columns
    const int row_in_tile = (int)cta_rank * BLOCK_M + quarter * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    uint32_t acc_iter = 0;

    for (int item = cluster_id; item < num_items; item += num_clusters) {
      int tm, tn0;
      decode_item(item, tm, tn0);
      const int64_t row = (int64_t)tm * TILE_M + row_in_tile;
      float best = 3.402823466e+38f;
      int32_t best_idx = 0x7fffffff;
      float radd = 0.f;
      if (EPI == EPI_ARGMIN && row < prm.M) radd = __ldg(prm.row_add + row);

      for (int nt = 0; nt < prm.n_per_item; ++nt) {
        const int64_t col0 = (int64_t)(tn0 + nt) * BLOCK_N + half * EPI_COLS;
        float acc[CHUNKED ? EPI_COLS : 1];
        for (int c = 0; c < num_chunks; ++c, ++acc_iter) {
          const uint32_t buf = acc_iter & 1u;
          mbar_wait(&tail->tmem_full[buf], (acc_iter >> 1) & 1u);
          tc_fence_after();
          const uint32_t taddr = tmem_base + lane_addr + buf * BLOCK_N + half * EPI_COLS;
#pragma unroll
          for (int g = 0; g < EPI_COLS / 32; ++g) {
            uint32_t v[32];
            tmem_ld32(taddr + g * 32, v);
            tmem_ld_wait();
            if constexpr (CHUNKED) {
              if (FOLD && c == 0 && prm.carry != nullptr && row < prm.M) {
                // resume the fold of the previous k-panel: same additions, in the same order, as one long k
                const float* krow = prm.carry + row * prm.ld_carry + col0 + g * 32;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  acc[g * 32 + j] = (col0 + g * 32 + j < prm.N) ? krow[j] + __uint_as_float(v[j]) : __uint_as_float(v[j]);
              } else if (c == 0) {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[g * 32 + j] = __uint_as_float(v[j]);
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[g * 32 + j] += __uint_as_float(v[j]);
              }
            } else {
              // single chunk: consume the 32 columns right away
              if constexpr (EPI == EPI_GEMM) {
                if (row < prm.M) {
                  float* crow = prm.C + row * prm.ldc + col0 + g * 32;
#pragma unroll
                  for (int j = 0; j < 32; ++j) {
                    if (col0 + g * 32 + j < prm.N) {
                      float r = prm.alpha * __uint_as_float(v[j]);
                      if (prm.beta != 0.f) r = fmaf(prm.beta, crow[j], r);
                      crow[j] = r;
                    }
                  }
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const int64_t cj = col0 + g * 32 + j;
                  if (cj < prm.N) {
                    // reference order: D = -2*dot (exact scaling), D += c2, D += p2, then |D|
                    float d = __fadd_rn(__fadd_rn(-2.f * __uint_as_float(v[j]), __ldg(prm.col_add + cj)), radd);
                    d = fabsf(d);
                    if (d < best) { best = d; best_idx = (int32_t)cj; }
                  }
                }
              }
            }
          }
          // TMEM buffer drained: hand it back to the MMA warp of the leader CTA
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_leader(&tail->tmem_empty[buf]);
        }
        if constexpr (CHUNKED) {
          if constexpr (EPI == EPI_GEMM) {
            if (row < prm.M) {
              float* crow = prm.C + row * prm.ldc + col0;
#pragma unroll
              for (int j = 0; j < EPI_COLS; ++j) {
                if (FOLD && prm.raw_out) {
                  if (col0 + j < prm.N) crow[j] = acc[j];
                } else if (col0 + j < prm.N) {
                  float r = prm.alpha * acc[j];
                  if (prm.beta != 0.f) r = fmaf(prm.beta, crow[j], r);
                  crow[j] = r;
                }
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < EPI_COLS; ++j) {
              const int64_t cj = col0 + j;
              if (cj < prm.N) {
                float d = __fadd_rn(__fadd_rn(-2.f * acc[j], __ldg(prm.col_add + cj)), radd);
                d = fabsf(d);
                if (d < best) { best = d; best_idx = (int32_t)cj; }
              }
            }
          }
        }
      }

      if constexpr (EPI == EPI_ARGMIN) {
        // combine the two column halves: smaller |d| wins, ties go to the lower index
        // (cblas_isamin returns the first minimum, drivers/in_mem_kmeans.cpp:84-85)
        const int r_local = quarter * 32 + lane;
        if (half == 1) {
          tail->red_val[r_local] = best;
          tail->red_idx[r_local] = best_idx;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (half == 0) {
          const float ov = tail->red_val[r_local];
          const int32_t oi = tail->red_idx[r_local];
          if (ov < best || (ov == best && oi < best_idx)) { best = ov; best_idx = oi; }
          // a row whose distances are all NaN / +Inf never updates: keep the result in [0, N) like isamin does
          if ((uint32_t)best_idx >= (uint32_t)prm.N) best_idx = 0;
          if (row < prm.M) prm.argmin_out[row] = best_idx;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
    }
  }

  // teardown: nobody may exit (or free TMEM) while the pair can still signal its barriers
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) tmem_dealloc<CG>(tmem_base, TMEM_COLS);
}


// ---------------------------------------------------------------------------------------------
// Tensor-pipe issue-rate microbenchmark: the roofline denominator, measured with this library's own instructions.
// Every CTA pair issues the GEMM's MMAs (cta_group::2, 256 x 256 accumulator in TMEM) back to back on ONE resident
// shared-memory stage -- no TMA traffic, no epilogue -- so the number is what the tensor pipe sustains when nothing
// else is in its way: kind 0 = kind::tf32 only, 1 = kind::f16 (bf16) only, 2 = the hybrid mix of the product kernel
// (per 32 k-elements: four bf16 MMAs of K = 16 for the two cross terms + four tf32 MMAs of K = 8 for hi*hi).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128, 1)
tc_issue_rate_kernel(int kind, int rounds) {
  constexpr int CG = 2;
  constexpr int BLOCK_N = 256;
  constexpr uint32_t IDESC = make_idesc(BLOCK_M * CG, BLOCK_N, 2u);
  constexpr uint32_t IDESC_BF16 = make_idesc(BLOCK_M * CG, BLOCK_N, 1u);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t done_bar;
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool is_leader = cluster_ctarank() == 0;
  // operand planes: small integers as fp32 / bf16 bit patterns (finite, not all zero)
  uint32_t* w = reinterpret_cast<uint32_t*>(smem);
  for (int i = threadIdx.x; i < STAGE_BYTES / 4; i += blockDim.x) w[i] = 0x3f800000u + ((i * 2654435761u) & 0x007f0000u);
  if (threadIdx.x == 0) { mbar_init(&done_bar, 1); fence_barrier_init(); }
  if (warp == 2) tmem_alloc<CG>(&tmem_base_s, 2 * BLOCK_N);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes visible to the MMA's async proxy
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;
  if (warp == 1 && is_leader) {
    if (lane == 0) {
      const uint32_t st = smem_u32(smem);
      const uint64_t d_p_hi = make_smem_desc(st), d_p_lo = make_smem_desc(st + PLANE_BYTES);
      const uint64_t d_q_hi = make_smem_desc(st + 2 * PLANE_BYTES), d_q_lo = make_smem_desc(st + 3 * PLANE_BYTES);
      for (int r = 0; r < rounds; ++r) {
        if (kind != 0) {
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint64_t adv = (uint64_t)(kk * 2);
            umma_bf16<CG>(tmem_d, d_p_lo + 4 + adv, d_q_lo + adv, IDESC_BF16, (r | kk) == 0 ? 0u : 1u);
            umma_bf16<CG>(tmem_d, d_p_lo + adv, d_q_lo + 4 + adv, IDESC_BF16, 1u);
          }
        }
        if (kind != 1) {
#pragma unroll
          for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
            const uint64_t adv = (uint64_t)((kk * UMMA_K * 4) >> 4);
            umma_tf32<CG>(tmem_d, d_p_hi + adv, d_q_hi + adv, IDESC, (kind == 0 && (r | kk) == 0) ? 0u : 1u);
          }
        }
      }
      umma_commit<CG>(&done_bar);
    }
    __syncwarp();
  }
  // both CTAs wait for the pair's MMAs (the commit is multicast to the same barrier offset in both)
  if (warp == 0) mbar_wait(&done_bar, 0);
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc<CG>(tmem_d, 2 * BLOCK_N);
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------
// TF32 split (pre-pass)
// ---------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ float rna_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

// The planes of one operand element, for both splits: hi (tf32), lo = rna_tf32(x - hi) (the gemm_split = 1 plane)
// and the hybrid pair bh = bf16(hi), bl = bf16(x - hi).  Both split kernels call this one function.
//   - Non-finite x: hi = x and every residual 0, so that the cross terms vanish and hi*hi carries the IEEE Inf / NaN
//     (x - hi would be NaN).
//   - |x| >= 0x1.ffep127 (bits 0x7f7ff000): rna_tf32 would round to Inf, so hi truncates instead; x - hi stays exact
//     and lo keeps ~2^-21 relative.
//   - |hi| >= 0x1.ffp127 (bits 0x7f7f8000): bf16 round-to-nearest would overflow, so bh rounds toward zero (error
//     2^-8 of a cross term that is itself ~2^-11 of the product).
// Below these thresholds the planes are exactly rna_tf32 / bf16 round-to-nearest.
struct SplitElem {
  float hi, lo;
  uint16_t bh, bl;
};
__device__ __forceinline__ SplitElem split_elem(float x) {
  SplitElem s;
  const uint32_t ax = __float_as_uint(x) & 0x7fffffffu;
  if (ax >= 0x7f800000u) {
    s.hi = x; s.lo = 0.f; s.bh = 0; s.bl = 0;
    return s;
  }
  s.hi = ax >= 0x7f7ff000u ? __uint_as_float(__float_as_uint(x) & ~0x1fffu) : rna_tf32(x);
  const float e = x - s.hi;  // exact in fp32
  s.lo = rna_tf32(e);
  const uint32_t ah = __float_as_uint(s.hi) & 0x7fffffffu;
  s.bh = ah >= 0x7f7f8000u ? (uint16_t)(__float_as_uint(s.hi) >> 16) : __bfloat16_as_ushort(__float2bfloat16_rn(s.hi));
  s.bl = __bfloat16_as_ushort(__float2bfloat16_rn(e));
  return s;
}
// Hybrid second plane: per 32-element k group (128 bytes) 32 x bf16(hi) then 32 x bf16(lo), lo = x - hi exact.
__device__ __forceinline__ uint8_t* combo_ptr(float* plane, int64_t r, int64_t kp, int64_t kk, bool lo_half) {
  return reinterpret_cast<uint8_t*>(plane + r * kp) + (kk >> 5) * 128 + (lo_half ? 64 : 0) + (kk & 31) * 2;
}

// K contiguous in the source (s_k == 1): element-wise, 4 k-elements per thread.
__global__ void __launch_bounds__(256)
split_planes_kmajor_kernel(int64_t R, int64_t K, const float* __restrict__ src, int64_t s_r,
                           float* __restrict__ hi, float* __restrict__ lo, int64_t kp, bool vec, bool combo) {
  const int64_t quads_per_row = kp / 4;
  const int64_t total = R * quads_per_row;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += stride) {
    const int64_t r = q / quads_per_row, k0 = (q - r * quads_per_row) * 4;
    float x[4] = {0.f, 0.f, 0.f, 0.f};
    const float* p = src + r * s_r + k0;
    if (vec && k0 + 4 <= K) {
      const float4 t = __ldcs(reinterpret_cast<const float4*>(p));
      x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w;
    } else {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (k0 + u < K) x[u] = p[u];
    }
    const SplitElem s0 = split_elem(x[0]), s1 = split_elem(x[1]), s2 = split_elem(x[2]), s3 = split_elem(x[3]);
    *reinterpret_cast<float4*>(hi + r * kp + k0) = make_float4(s0.hi, s1.hi, s2.hi, s3.hi);
    if (!combo) {
      *reinterpret_cast<float4*>(lo + r * kp + k0) = make_float4(s0.lo, s1.lo, s2.lo, s3.lo);
    } else {
      uint2 ph, pl;
      ph.x = s0.bh | ((uint32_t)s1.bh << 16);
      ph.y = s2.bh | ((uint32_t)s3.bh << 16);
      pl.x = s0.bl | ((uint32_t)s1.bl << 16);
      pl.y = s2.bl | ((uint32_t)s3.bl << 16);
      *reinterpret_cast<uint2*>(combo_ptr(lo, r, kp, k0, false)) = ph;
      *reinterpret_cast<uint2*>(combo_ptr(lo, r, kp, k0, true)) = pl;
    }
  }
}

// R contiguous in the source (s_r == 1): 32x32 tiles through shared memory.
__global__ void __launch_bounds__(256)
split_planes_transpose_kernel(int64_t R, int64_t K, const float* __restrict__ src, int64_t s_k,
                              float* __restrict__ hi, float* __restrict__ lo, int64_t kp,
                              unsigned tiles_k, bool combo) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)(blockIdx.x / tiles_k) * 32, k0 = (int64_t)(blockIdx.x % tiles_k) * 32;
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int64_t kk = k0 + i, r = r0 + tx;
    tile[i][tx] = (kk < K && r < R) ? src[kk * s_k + r] : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int64_t r = r0 + i, kk = k0 + tx;
    if (r < R && kk < kp) {
      const SplitElem sp = split_elem(tile[tx][i]);
      hi[r * kp + kk] = sp.hi;
      if (!combo) {
        lo[r * kp + kk] = sp.lo;
      } else {
        *reinterpret_cast<uint16_t*>(combo_ptr(lo, r, kp, kk, false)) = sp.bh;
        *reinterpret_cast<uint16_t*>(combo_ptr(lo, r, kp, kk, true)) = sp.bl;
      }
    }
  }
}

// CUDA-core fp32 GEMM, 64x64 tile, 4x4 per thread, generic strides.
__global__ void __launch_bounds__(256)
gemm_ffma_kernel(int64_t M, int64_t N, int64_t K, float alpha, const float* __restrict__ A,
                 int64_t a_r, int64_t a_k, const float* __restrict__ B, int64_t b_k, int64_t b_c,
                 float beta, float* __restrict__ C, int64_t ldc) {
  constexpr int BM = 64, BN = 64, BK = 16;
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = (int64_t)blockIdx.y * BM, n0 = (int64_t)blockIdx.x * BN;
  float acc[4][4] = {};
  for (int64_t k0 = 0; k0 < K; k0 += BK) {
    for (int i = tid; i < BM * BK; i += 256) {
      // consecutive threads walk whichever index is contiguous in memory
      int mm, kk;
      if (a_k == 1) { kk = i % BK; mm = i / BK; } else { mm = i % BM; kk = i / BM; }
      const int64_t gm = m0 + mm, gk = k0 + kk;
      As[kk][mm] = (gm < M && gk < K) ? A[gm * a_r + gk * a_k] : 0.f;
    }
    for (int i = tid; i < BN * BK; i += 256) {
      int nn, kk;
      if (b_k == 1) { kk = i % BK; nn = i / BK; } else { nn = i % BN; kk = i / BN; }
      const int64_t gn = n0 + nn, gk = k0 + kk;
      Bs[kk][nn] = (gn < N && gk < K) ? B[gk * b_k + gn * b_c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { a[u] = As[kk][ty * 4 + u]; b[u] = Bs[kk][tx * 4 + u]; }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fmaf(a[u], b[v], acc[u][v]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t gm = m0 + ty * 4 + u;
    if (gm >= M) continue;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int64_t gn = n0 + tx * 4 + v;
      if (gn >= N) continue;
      float r = alpha * acc[u][v];
      if (beta != 0.f) r = fmaf(beta, C[gm * ldc + gn], r);
      C[gm * ldc + gn] = r;
    }
  }
}

// bof_config.gemm_split: 1 = pure 3xTF32; 2 = hybrid (TF32 hi*hi + two BF16 cross terms); 0 = default
bool hybrid_split(const bof_ctx* ctx) { return ctx->cfg.gemm_split == 2 || (ctx->cfg.gemm_split == 0 && BOF_DEFAULT_HYBRID); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

int make_plane_map(bof_ctx* ctx, CUtensorMap* map, const float* plane, int64_t rows, int64_t kp) {
  BOF_REQUIRE(ctx, ctx->tmap_encode != nullptr, "cuTensorMapEncodeTiled unavailable");
  const cuuint64_t dims[2] = {(cuuint64_t)kp, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)kp * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)tc::BLOCK_K, 128u};
  const cuuint32_t estr[2] = {1u, 1u};
  CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->tmap_encode)(
      map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(plane), dims, strides, box, estr,
      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ctx, BOF_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return BOF_OK;
}

template <int CG, int EPI, bool CHUNKED, bool HYB, bool FOLD = false>
int launch_variant(bof_ctx* ctx, cudaStream_t s, const CUtensorMap* maps, const tc::Params& prm, int num_items) {
  auto kern = tc::gemm3xtf32_kernel<CG, EPI, CHUNKED, HYB, FOLD>;
  static PerDeviceOnce attr_set;
  if (attr_set.need(ctx->device)) {
    BOF_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::SMEM_BYTES));
    attr_set.done(ctx->device);
  }
  const int max_clusters = std::max(1, (ctx->num_sms - ctx->sm_reserve) / CG);
  const int clusters = std::max(1, std::min(num_items, max_clusters));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(clusters * CG));
  cfg.blockDim = dim3(tc::NUM_THREADS);
  cfg.dynamicSmemBytes = tc::SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (!ctx->tk0) {
    BOF_CUDA(ctx, cudaEventCreate(&ctx->tk0));
    BOF_CUDA(ctx, cudaEventCreate(&ctx->tk1));
  }
  BOF_CUDA(ctx, cudaEventRecord(ctx->tk0, s));
  BOF_CUDA(ctx, cudaLaunchKernelEx(&cfg, kern, maps[0], maps[1], maps[2], maps[3], prm));
  BOF_LAUNCH_CHECK(ctx, "gemm3xtf32_kernel");
  BOF_CUDA(ctx, cudaEventRecord(ctx->tk1, s));
  ctx->tk_valid = true;
  return BOF_OK;
}

}  // namespace

int launch_split_planes(bof_ctx* ctx, cudaStream_t s, int64_t R, int64_t K, const float* src,
                        int64_t s_r, int64_t s_k, float* hi, float* lo, int64_t kp) {
  BOF_REQUIRE(ctx, kp % 32 == 0 && kp >= K, "split: bad padded k");
  if (R == 0) return BOF_OK;
  if (s_k == 1) {
    const bool vec = (s_r % 4 == 0) && aligned16(src);
    const int64_t total = R * (kp / 4);
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(total, 256), (int64_t)ctx->num_sms * 32);
    split_planes_kmajor_kernel<<<grid, 256, 0, s>>>(R, K, src, s_r, hi, lo, kp, vec, hybrid_split(ctx));
    BOF_LAUNCH_CHECK(ctx, "split_planes_kmajor_kernel");
  } else {
    BOF_REQUIRE(ctx, s_r == 1, "split: one of the operand strides must be 1");
    const int64_t tiles_k = kp / 32, tiles_r = ceil_div<int64_t>(R, 32);
    BOF_REQUIRE(ctx, tiles_k * tiles_r < (1ll << 31), "split: operand too large for one launch");
    split_planes_transpose_kernel<<<(unsigned)(tiles_k * tiles_r), 256, 0, s>>>(R, K, src, s_k, hi, lo, kp,
                                                                               (unsigned)tiles_k, hybrid_split(ctx));
    BOF_LAUNCH_CHECK(ctx, "split_planes_transpose_kernel");
  }
  return BOF_OK;
}

int launch_gemm_tc(bof_ctx* ctx, cudaStream_t s, int cta_group, int64_t M, int64_t N, int64_t K,
                   int64_t kp, const float* p_hi, const float* p_lo, const float* q_hi,
                   const float* q_lo, const GemmEpilogue& ep, int64_t k_chunk) {
  (void)K;
  if (M == 0 || N == 0) return BOF_OK;
  BOF_REQUIRE(ctx, cta_group == 1 || cta_group == 2, "gemm_tc: cta_group must be 1 or 2");
  BOF_REQUIRE(ctx, kp % 32 == 0 && kp > 0, "gemm_tc: padded k must be a positive multiple of 32");
  BOF_REQUIRE(ctx, M < (1ll << 31) && N < (1ll << 31) && kp < (1ll << 31), "gemm_tc: extent exceeds int32");
  CUtensorMap maps[4];
  int rc;
  if ((rc = make_plane_map(ctx, &maps[0], p_hi, M, kp))) return rc;
  if ((rc = make_plane_map(ctx, &maps[1], p_lo, M, kp))) return rc;
  if ((rc = make_plane_map(ctx, &maps[2], q_hi, N, kp))) return rc;
  if ((rc = make_plane_map(ctx, &maps[3], q_lo, N, kp))) return rc;

  const int block_n = cta_group == 2 ? 256 : 128;
  const int tile_m = 128 * cta_group;
  tc::Params prm{};
  prm.M = M;
  prm.N = N;
  prm.num_kb = (int32_t)(kp / 32);
  int64_t kbc = (k_chunk <= 0) ? prm.num_kb : std::max<int64_t>(1, k_chunk / 32);
  if (kbc > prm.num_kb) kbc = prm.num_kb;
  prm.kb_per_chunk = (int32_t)kbc;
  prm.tiles_m = (int32_t)ceil_div<int64_t>(M, tile_m);
  prm.tiles_n = (int32_t)ceil_div<int64_t>(N, block_n);
  const bool argmin = ep.C == nullptr;
  prm.n_per_item = argmin ? prm.tiles_n : 1;
  prm.alpha = ep.alpha;
  prm.beta = ep.beta;
  prm.C = ep.C;
  prm.ldc = ep.ldc;
  prm.row_add = ep.row_add;
  prm.col_add = ep.col_add;
  prm.argmin_out = ep.argmin_out;
  prm.carry = ep.carry;
  prm.ld_carry = ep.ld_carry;
  prm.raw_out = ep.raw_out ? 1 : 0;
  const bool fold = ep.carry != nullptr || ep.raw_out;
  if (argmin)
    BOF_REQUIRE(ctx, ep.row_add && ep.col_add && ep.argmin_out, "gemm_tc: argmin epilogue needs norms and an output");
  BOF_REQUIRE(ctx, !(argmin && fold), "gemm_tc: the fold carry needs the GEMM epilogue");
  const bool chunked = prm.kb_per_chunk < prm.num_kb;
  const int num_items = argmin ? prm.tiles_m : prm.tiles_m * prm.tiles_n;
  // wave lock-step only pays when a tile's k-panel outgrows L2 and there is more than one wave
  const int clusters = std::max(1, std::min(num_items, std::max(1, (ctx->num_sms - ctx->sm_reserve) / cta_group)));
  prm.sync_kb = 0;
  prm.sync_counters = nullptr;
  if (!argmin && ctx->cfg.gemm_wave_sync >= 0 && prm.num_kb >= 256 && num_items > clusters) {
    prm.sync_kb = ctx->cfg.gemm_wave_sync > 0 ? ctx->cfg.gemm_wave_sync : 64;
    const size_t waves = (size_t)ceil_div(num_items, clusters);
    const size_t n_ctr = waves * (size_t)ceil_div(prm.num_kb, prm.sync_kb);
    if (ctx->sync_ctr_count < n_ctr) {
      // Sized with headroom on first use: cudaFree / cudaMalloc synchronise the whole device, and in the middle of
      // a host pipeline (the first full-width block after narrower prologue launches) that stalled the caller for
      // as long as the drainer thread kept device->host copies in flight (BOF_TRACE: 0.9 s at 32768^3).
      size_t n_alloc = 1u << 16;
      while (n_alloc < n_ctr) n_alloc <<= 1;
      if (ctx->sync_ctr) BOF_CUDA(ctx, cudaFree(ctx->sync_ctr));
      ctx->sync_ctr = nullptr;
      ctx->sync_ctr_count = 0;
      BOF_CUDA(ctx, cudaMalloc(&ctx->sync_ctr, n_alloc * sizeof(uint32_t)));
      ctx->sync_ctr_count = n_alloc;
    }
    BOF_CUDA(ctx, cudaMemsetAsync(ctx->sync_ctr, 0, n_ctr * sizeof(uint32_t), s));
    prm.sync_counters = ctx->sync_ctr;
  }

  const bool hyb = hybrid_split(ctx);
  if (fold) {  // a k-panel shorter than one chunk still goes through the chunked epilogue that holds the fold
    if (cta_group == 2) {
      if (hyb) return launch_variant<2, tc::EPI_GEMM, true, true, true>(ctx, s, maps, prm, num_items);
      return launch_variant<2, tc::EPI_GEMM, true, false, true>(ctx, s, maps, prm, num_items);
    }
    if (hyb) return launch_variant<1, tc::EPI_GEMM, true, true, true>(ctx, s, maps, prm, num_items);
    return launch_variant<1, tc::EPI_GEMM, true, false, true>(ctx, s, maps, prm, num_items);
  }
#define BOF_TC(CG, EPI, CH)                                                            \
  do {                                                                                 \
    if (hyb) return launch_variant<CG, EPI, CH, true>(ctx, s, maps, prm, num_items);   \
    return launch_variant<CG, EPI, CH, false>(ctx, s, maps, prm, num_items);           \
  } while (0)
  if (cta_group == 2) {
    if (argmin) { if (chunked) BOF_TC(2, tc::EPI_ARGMIN, true); else BOF_TC(2, tc::EPI_ARGMIN, false); }
    if (chunked) BOF_TC(2, tc::EPI_GEMM, true); else BOF_TC(2, tc::EPI_GEMM, false);
  } else {
    if (argmin) { if (chunked) BOF_TC(1, tc::EPI_ARGMIN, true); else BOF_TC(1, tc::EPI_ARGMIN, false); }
    if (chunked) BOF_TC(1, tc::EPI_GEMM, true); else BOF_TC(1, tc::EPI_GEMM, false);
  }
#undef BOF_TC
}

int launch_gemm_ffma(bof_ctx* ctx, cudaStream_t s, int64_t M, int64_t N, int64_t K, float alpha,
                     const float* A, int64_t a_r, int64_t a_k, const float* B, int64_t b_k,
                     int64_t b_c, float beta, float* C, int64_t ldc) {
  if (M == 0 || N == 0) return BOF_OK;
  dim3 grid((unsigned)ceil_div<int64_t>(N, 64), (unsigned)ceil_div<int64_t>(M, 64));
  BOF_REQUIRE(ctx, grid.y <= 65535u, "gemm_ffma: too many row tiles (use the tensor-core path)");
  gemm_ffma_kernel<<<grid, 256, 0, s>>>(M, N, K, alpha, A, a_r, a_k, B, b_k, b_c, beta, C, ldc);
  BOF_LAUNCH_CHECK(ctx, "gemm_ffma_kernel");
  return BOF_OK;
}


// tensor-pipe issue rate in TFLOP/s of MMA work (2 * M * N * K per instruction) for `kind` (see tc_issue_rate_kernel);
// `useful` additionally returns the rate in USEFUL fp32 flops of the hybrid mix (2 * 256 * 256 * 32 per round)
int tc_issue_rate(bof_ctx* ctx, cudaStream_t s, int kind, int rounds, double* mma_tflops, double* useful_tflops) {
  BOF_REQUIRE(ctx, kind >= 0 && kind <= 2 && rounds > 0, "tc_issue_rate: bad kind / rounds");
  static PerDeviceOnce attr_set;
  const size_t smem = (size_t)tc::STAGE_BYTES + 2048;
  if (attr_set.need(ctx->device)) {
    BOF_CUDA(ctx, cudaFuncSetAttribute(tc::tc_issue_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set.done(ctx->device);
  }
  const int clusters = ctx->num_sms / 2;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(clusters * 2));
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaEvent_t e0, e1;
  BOF_CUDA(ctx, cudaEventCreate(&e0));
  BOF_CUDA(ctx, cudaEventCreate(&e1));
  BOF_CUDA(ctx, cudaLaunchKernelEx(&cfg, tc::tc_issue_rate_kernel, kind, 64));   // warm-up
  BOF_CUDA(ctx, cudaEventRecord(e0, s));
  BOF_CUDA(ctx, cudaLaunchKernelEx(&cfg, tc::tc_issue_rate_kernel, kind, rounds));
  BOF_LAUNCH_CHECK(ctx, "tc_issue_rate_kernel");
  BOF_CUDA(ctx, cudaEventRecord(e1, s));
  BOF_CUDA(ctx, cudaStreamSynchronize(s));
  float ms = 0.f;
  BOF_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  const double per_round_useful = 2.0 * 256 * 256 * 32;                     // one 32-element k-step of a 256 x 256 tile
  // MMA work per round: tf32 = one term, bf16 = the two cross terms, hybrid = all three
  const double mma_per_round = per_round_useful * (kind == 2 ? 3.0 : (kind == 1 ? 2.0 : 1.0));
  if (mma_tflops) *mma_tflops = mma_per_round * rounds * clusters / (ms * 1e-3) / 1e12;
  if (useful_tflops) *useful_tflops = per_round_useful * rounds * clusters / (ms * 1e-3) / 1e12;
  return BOF_OK;
}

}  // namespace bof
