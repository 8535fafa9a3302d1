// flash_blas.h -- the reference's public kernel API (include/flash_blas.h:14-57), kept signature for
// signature so that a BLAS-on-Flash application switches by relinking against libflashblas_b200.
// Every function is a thin adapter (blas-on-flash_b200/host/flash_blas.cpp) that flattens the
// flash_ptr arguments to host addresses and calls the C ABI of include/bof_b200.h; the arithmetic
// runs in hand-written sm_100a kernels.  Return convention as the reference: 0 on success, -1 on a
// bad argument (src/blas/csrmm.cpp:433-449) or any CUDA / I/O failure (message on stderr).
//
// Out of scope of the hot path (SURVEY.md section 2): sort, map, reduce.
#pragma once

#include "bof_types.h"
#include "pointers/allocator.h"
#include "pointers/pointer.h"

namespace flash {

// C = alpha * op(A) * op(B) + beta * C                                   [reference flash_blas.h:14-18]
//   mat_ord 'R' | 'C', trans_a / trans_b 'N' | 'T'; op(A) is m x k, op(B) is k x n
//   lda_* = 0 selects the tight leading dimension (src/blas/gemm.cpp:63-67)
FBLAS_INT gemm(CHAR mat_ord, CHAR trans_a, CHAR trans_b,
               FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k,
               FPTYPE alpha, FPTYPE beta,
               flash_ptr<FPTYPE> a, flash_ptr<FPTYPE> b, flash_ptr<FPTYPE> c,
               FBLAS_UINT lda_a = 0, FBLAS_UINT lda_b = 0, FBLAS_UINT lda_c = 0);

// c = alpha * op(A) * b + beta * c                            [declared, never defined: reference flash_blas.h:28-30]
//   A is m x n stored mat_ord 'R' | 'C' with leading dimension lda_a (0 = tight), trans_a 'N' | 'T';
//   b has n ('N') or m ('T') entries, c the other count.  beta == 0: c is not read.  Deterministic, and the same bits
//   on one GPU or several (bof_host_gemv / bof_mgpu_gemv).  The FPTYPE* overload takes b and c in host memory.
FBLAS_INT gemv(CHAR mat_ord, CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FPTYPE alpha, FPTYPE beta,
               flash_ptr<FPTYPE> a, flash_ptr<FPTYPE> b, flash_ptr<FPTYPE> c, FBLAS_UINT lda_a = 0);
FBLAS_INT gemv(CHAR mat_ord, CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FPTYPE alpha, FPTYPE beta,
               flash_ptr<FPTYPE> a, FPTYPE* b, FPTYPE* c, FBLAS_UINT lda_a = 0);

// Distance tile of k-means: C = alpha * op(A) * op(B) + beta * C + c_l2sq 1^T + 1 p_l2sq^T
//                                                                        [reference flash_blas.h:20-25]
//   the reference calls it as ('C','T','N', ncenters, npoints, dim, -2, 0, centers, points, dist, ...)
//   (drivers/kmeans.cpp:36-38); `ones` is accepted for source compatibility and not read.  The two rank-1
//   terms are added on the device (bof_host_kmeans_dist) before each block of C is downloaded.
//   Prefer kmeans_lloyd() below: it never materialises the distance matrix.
FBLAS_INT kmeans(CHAR mat_ord, CHAR trans_a, CHAR trans_b,
                 FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k,
                 FPTYPE alpha, FPTYPE beta,
                 flash_ptr<FPTYPE> a, flash_ptr<FPTYPE> b, flash_ptr<FPTYPE> c,
                 FBLAS_UINT lda_a, FBLAS_UINT lda_b, FBLAS_UINT lda_c,
                 FPTYPE* c_l2sq, FPTYPE* p_l2sq, FPTYPE* ones);

// C = alpha * op(A) * B + beta * C with A (m x n) in CSR                  [reference flash_blas.h:37-40]
//   trans_a 'N': B is n x k, C is m x k;  trans_a 'T': B is m x k, C is n x k
//   ord_b 'R' | 'C' is the layout of both B and C.  Mind the order: offsets `ia` come before indices `ja`.
FBLAS_INT csrmm(CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k,
                FPTYPE alpha, FPTYPE beta,
                flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja,
                CHAR ord_b, flash_ptr<FPTYPE> b, flash_ptr<FPTYPE> c);

// Same with B and C in host memory                                        [reference flash_blas.h:43-46]
//   (returns 0 on success; the reference's -1 on the row-major success path, csrmm.cpp:463-466, is a bug)
FBLAS_INT csrmm(CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k,
                FPTYPE alpha, FPTYPE beta,
                flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja,
                CHAR ord_b, FPTYPE* b, FPTYPE* c);

// CSR(ia, ja, a; m x n) -> CSR of the transpose (ia_tr, ja_tr, a_tr; n x m), stable    [flash_blas.h:49-52]
FBLAS_INT csrcsc(FBLAS_UINT m, FBLAS_UINT n,
                 flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja, flash_ptr<FPTYPE> a,
                 flash_ptr<MKL_INT> ia_tr, flash_ptr<MKL_INT> ja_tr, flash_ptr<FPTYPE> a_tr);

// c = op(A) b, A (m x n) in CSR on flash, b and c host vectors, c overwritten     [reference flash_blas.h:55-57]
FBLAS_INT csrgemv(CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n,
                  flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja,
                  FPTYPE* b, FPTYPE* c);

// ---- extension: keep a CSR matrix in HBM across calls ------------------------------------------
// Iterative callers (the block Krylov-Schur eigensolver of the paper, drivers/csrmm_pmem.cpp) multiply by the same
// A many times; the reference re-reads it from flash each call.  After csr_pin(m, n, a, ia, ja) every
// flash::csrmm / flash::csrgemv whose (a, ia, ja, m, n) match runs on the HBM-resident copy and moves only the
// dense operands.  The files behind a, ia, ja must not change while pinned.  with_transpose also keeps A^T
// (needed by trans_a = 'T' products; built on first use otherwise).  flash_destroy() unpins everything.
FBLAS_INT csr_pin(FBLAS_UINT m, FBLAS_UINT n, flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja,
                  bool with_transpose = false);
FBLAS_INT csr_unpin(flash_ptr<FPTYPE> a);

// ---- extension: the Lloyd loop that lives in the reference's drivers ---------------------------
// `n_iters` iterations of drivers/kmeans.cpp:103-189 (closest_centers + centroid update) with the
// points resident in HBM: fused distance-GEMM/argmin, deterministic centroid reduce.  `centers` is
// updated in place (file contents on return); closest_center (npoints entries, may be null) receives
// the assignment of the last iteration.  With more than one process/GPU each rank passes its shard
// and `allreduce` (may be null on one GPU) must sum the `count` floats at device address `buf` over
// all ranks on `stream` -- e.g. ncclAllReduce(buf, buf, count, ncclFloat, ncclSum, comm, stream).
using kmeans_allreduce_fn = int (*)(void* buf, size_t count, void* stream, void* user);
FBLAS_INT kmeans_lloyd(flash_ptr<FPTYPE> points, flash_ptr<FPTYPE> centers,
                       FBLAS_UINT npoints, FBLAS_UINT ndims, FBLAS_UINT ncenters, FBLAS_UINT n_iters,
                       FBLAS_UINT* closest_center = nullptr,
                       kmeans_allreduce_fn allreduce = nullptr, void* allreduce_user = nullptr);

}  // namespace flash
