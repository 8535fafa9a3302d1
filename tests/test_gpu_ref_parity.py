"""GPU parity against the REFERENCE ITSELF: the CUDA path, called through the C ABI host entry points, is compared
with (i) tests/golden/golden_ref.npz -- outputs written by the reference's own binaries -- and (ii) where
oracle/_ref has been built, live runs of those binaries on fresh, larger inputs (in_mem_* = the bare MKL
call; flash drivers = flash::gemm / csrmm / csrgemv / csrcsc through the reference's scheduler and file handles).
Tolerances are BASELINE.json's: relative Frobenius <= 1e-5 for gemm / csrmm / csrgemv / centroids, bit-exact for
csrcsc and for k-means assignments on ties-free points."""
import numpy as np
import pytest

import oracle
from golden_ref import G, TOL, csrcsc_cases, csrgemv_cases, csrmm_cases, gemm_cases, gemm_layout, same_csc, sparse_inputs
from oracle import ref_run as rr

pytestmark = pytest.mark.gpu
needs_ref = pytest.mark.skipif(not (rr.available() and rr.available("_small")),
                               reason="oracle/_ref not built (make -C oracle -f Makefile.ref REF=<reference sources>)")


@pytest.mark.parametrize("case", list(gemm_cases()), ids=lambda c: c[0])
def test_gemm_vs_reference_output(ctx, case):
    _, o, ta, tb, M, N, K, alpha, beta, a, b, c, want = case
    lda, ldb, ldc = gemm_layout(o, ta, tb, M, N, K)
    got = c.copy()
    ctx.host_gemm(o, ta, tb, M, N, K, alpha, beta, a, b, got, lda, ldb, ldc)
    assert oracle.rel_fro(got, want.reshape(-1)) <= TOL


@pytest.mark.parametrize("case", list(csrmm_cases()), ids=lambda c: c[0])
def test_csrmm_vs_reference_output(ctx, case):
    _, trans, k, alpha, beta, ord_b, B, C, want = case
    s = sparse_inputs()
    got = C.copy()
    ctx.host_csrmm(trans, s["m"], s["n"], k, alpha, beta, s["a"], s["ia"], s["ja"], ord_b, B, got)
    assert oracle.rel_fro(got, want.reshape(got.shape)) <= TOL


@pytest.mark.parametrize("case", list(csrgemv_cases()), ids=lambda c: c[0])
def test_csrgemv_vs_reference_output(ctx, case):
    _, trans, x, want = case
    s = sparse_inputs()
    y = np.full(want.shape, np.nan, np.float32)  # csrgemv overwrites (src/blas/csrgemv.cpp:82-97)
    ctx.host_csrgemv(trans, s["m"], s["n"], s["a"], s["ia"], s["ja"], x, y)
    assert oracle.rel_fro(y, want) <= TOL


@pytest.mark.parametrize("case", list(csrcsc_cases()), ids=lambda c: c[0])
def test_csrcsc_vs_reference_output_bit_exact(ctx, case):
    _, m, n, ia, ja, a, want = case
    nnz = int(ia[m])
    ia_t, ja_t, a_t = np.zeros(n + 1, np.int64), np.zeros(nnz, np.int64), np.zeros(nnz, np.float32)
    ctx.host_csrcsc(m, n, ia, ja, a, ia_t, ja_t, a_t)
    assert same_csc((ia_t, ja_t, a_t), want)


def _lloyd(bof, ctx, pts, cent, iters):
    P, d = pts.shape
    K = cent.shape[0]
    km = bof.KMeans(ctx, P, K, d, pts, cent)
    for _ in range(iters):
        km.local_step()
        km.update()
    c, a = np.zeros((K, d), np.float32), np.zeros(P, np.int64)
    km.get(c, a)
    km.close()
    return c, a


def test_kmeans_vs_reference_output(bof, ctx):
    pts, c0 = G["km_points"], G["km_centers0"]
    c1, _ = _lloyd(bof, ctx, pts, c0, 1)
    assert oracle.rel_fro(c1, G["km_centers_iter1"]) <= TOL
    c3, _ = _lloyd(bof, ctx, pts, c0, 3)
    assert oracle.rel_fro(c3, G["km_centers_iter3"]) <= TOL
    # assignments of the first 600 points against the reference's flash::kmeans distances (ties-free filter)
    p600 = np.ascontiguousarray(pts[:600])
    _, a600 = _lloyd(bof, ctx, p600, c0, 1)   # assignment is made with the INPUT centers
    D = G["km_dist_600"]
    part = np.partition(np.abs(D), 1, axis=1)
    clear = (part[:, 1] - part[:, 0]) > 1e-3 * (1 + part[:, 0])
    assert clear.mean() > 0.95
    assert np.array_equal(a600[clear], G["km_assign_600"][clear])
    # the distance tile itself, in the reference's call form (drivers/kmeans.cpp:37-39)
    K, d = c0.shape
    Dg = np.full(600 * K, np.nan, np.float32)
    ctx.host_kmeans_dist("C", "T", "N", K, 600, d, -2.0, 0.0, c0, p600, Dg, oracle.row_sqnorm(c0),
                         oracle.row_sqnorm(p600), lda=d, ldb=d, ldc=K)
    assert oracle.rel_fro(Dg.reshape(600, K), D) <= TOL


# ---------------------------------------------------------------- live reference binaries on this box
@needs_ref
def test_live_gemm_flash_driver(ctx):
    """the reference's gemm driver (default 8192 tiles: 2 k tiles -> a beta=1 chain) vs the tensor-core path"""
    M, N, K = 2048, 1536, 8300
    a, b, c = oracle.gen_dense(M * K, seed=51), oracle.gen_dense(K * N, seed=52), oracle.gen_dense(M * N, seed=53)
    want = rr.gemm("R", "N", "N", M, N, K, 1.0, 0.5, a, b, c, K, N, N, flash=True)
    got = c.copy()
    ctx.host_gemm("R", "N", "N", M, N, K, 1.0, 0.5, a, b, got, K, N, N)
    assert oracle.rel_fro(got, want.reshape(-1)) <= TOL
    want_t = rr.gemm("C", "T", "N", M, N, K, 1.0, 0.0, a, b, c, K, K, M)  # in_mem driver: one cblas_sgemm
    got = np.full(M * N, np.nan, np.float32)
    ctx.host_gemm("C", "T", "N", M, N, K, 1.0, 0.0, a, b, got, K, K, M)
    assert oracle.rel_fro(got, want_t.reshape(-1)) <= TOL


@needs_ref
def test_live_sparse_drivers(ctx):
    """in_mem_csrmm / flash csrmm / csrgemv / csrcsc of the reference on a 200k x 150k matrix with 32 nnz/row"""
    m, n, k = 200_000, 150_000, 128
    a, ia, ja = oracle.gen_csr(m, n, 32, seed=61)
    B, C0 = oracle.gen_dense((n, k), seed=62), oracle.gen_dense((m, k), seed=63)
    for flash in (False, True):
        want = rr.csrmm("N", m, n, k, 1.25, 0.75, a, ia, ja, "R", B, C0, flash=flash)
        got = C0.copy()
        ctx.host_csrmm("N", m, n, k, 1.25, 0.75, a, ia, ja, "R", B, got)
        assert oracle.rel_fro(got, want) <= TOL
    x, xt = oracle.gen_dense((n,), seed=64), oracle.gen_dense((m,), seed=65)
    for trans, v in (("N", x), ("T", xt)):
        want = rr.csrgemv(trans, m, n, a, ia, ja, v, flash=True)
        y = np.full(want.shape, np.nan, np.float32)
        ctx.host_csrgemv(trans, m, n, a, ia, ja, v, y)
        assert oracle.rel_fro(y, want) <= TOL
    want = rr.csrcsc(m, n, ia, ja, a, flash=True)
    nnz = int(ia[m])
    ia_t, ja_t, a_t = np.zeros(n + 1, np.int64), np.zeros(nnz, np.int64), np.zeros(nnz, np.float32)
    ctx.host_csrcsc(m, n, ia, ja, a, ia_t, ja_t, a_t)
    assert same_csc((ia_t, ja_t, a_t), want)


@needs_ref
def test_live_kmeans_driver_five_iterations(bof, ctx):
    """in_mem_kmeans_driver run 5 times (one Lloyd iteration per invocation) vs 5 resident iterations on the GPU"""
    rng = np.random.default_rng(71)
    K, d, P = 64, 64, 50_000
    mu = (rng.normal(size=(K, d)) * 4).astype(np.float32)
    pts = (mu[rng.integers(0, K, P)] + 0.3 * rng.normal(size=(P, d))).astype(np.float32)
    # ties-free start (BASELINE.json north_star): one initial centre inside every true cluster.  Starting from
    # the first K points instead puts several centres into one cluster; points between them have top-2 margins
    # down to exactly 0 in fp32 and MKL itself, the fp32 restatement and the GPU then each resolve them their own
    # way (reference vs oracle drift 4.8e-4 after 5 iterations on that start, see DESIGN.md section 2).
    c0 = (mu + 0.05 * rng.normal(size=(K, d))).astype(np.float32)
    _, margin = oracle.kmeans_assign(pts, c0)
    assert margin.min() > 1.0
    want = rr.kmeans_iters(pts, c0, iters=5)
    got, _ = _lloyd(bof, ctx, pts, c0, 5)
    assert oracle.rel_fro(got, want) <= TOL
