"""CPU tests that PIN THE ORACLE TO THE REFERENCE: oracle/oracle.c against tests/golden/golden_ref.npz, whose
outputs were written by the reference's own binaries (unmodified sources built by oracle/Makefile.ref), and --
where oracle/_ref has been built (make -C oracle -f Makefile.ref REF=<reference sources>) -- against live runs of
those binaries on fresh inputs, including sizes that take several tiles of the default build."""
import numpy as np
import pytest

import oracle
from golden_ref import G, TOL, csrcsc_cases, csrgemv_cases, csrmm_cases, gemm_cases, gemm_layout, same_csc, sparse_inputs
from oracle import ref_run as rr

needs_ref = pytest.mark.skipif(not (rr.available() and rr.available("_small")),
                               reason="oracle/_ref not built (make -C oracle -f Makefile.ref REF=<reference sources>)")


@pytest.mark.parametrize("case", list(gemm_cases()), ids=lambda c: c[0])
def test_oracle_gemm_vs_reference_output(case):
    _, o, ta, tb, M, N, K, alpha, beta, a, b, c, want = case
    lda, ldb, ldc = gemm_layout(o, ta, tb, M, N, K)
    got = oracle.gemm(o, ta, tb, M, N, K, alpha, beta, a, b, c, lda, ldb, ldc)
    assert oracle.rel_fro(got, want) <= TOL
    # the reference's own tiling + beta=1 chains (src/blas/gemm.cpp:83-129) restated: same result
    tiled = oracle.gemm(o, ta, tb, M, N, K, alpha, beta, a, b, c, lda, ldb, ldc, tiled_blk=256)
    assert oracle.rel_fro(tiled, want) <= TOL


@pytest.mark.parametrize("case", list(csrmm_cases()), ids=lambda c: c[0])
def test_oracle_csrmm_vs_reference_output(case):
    _, trans, k, alpha, beta, ord_b, B, C, want = case
    s = sparse_inputs()
    got = oracle.csrmm(trans, s["m"], s["n"], k, alpha, beta, s["a"], s["ia"], s["ja"], ord_b, B, C)
    assert oracle.rel_fro(got, want.reshape(got.shape)) <= TOL


@pytest.mark.parametrize("case", list(csrgemv_cases()), ids=lambda c: c[0])
def test_oracle_csrgemv_vs_reference_output(case):
    _, trans, x, want = case
    s = sparse_inputs()
    got = oracle.csrgemv(trans, s["m"], s["n"], s["a"], s["ia"], s["ja"], x)
    assert oracle.rel_fro(got, want) <= TOL


@pytest.mark.parametrize("case", list(csrcsc_cases()), ids=lambda c: c[0])
def test_oracle_csrcsc_vs_reference_output_bit_exact(case):
    _, m, n, ia, ja, a, want = case
    assert same_csc(oracle.csrcsc(m, n, ia, ja, a), want)
    assert same_csc(oracle.csrcsc(m, n, ia, ja, a, blocked_rblk=512, max_nnzs=6000), want)


def test_oracle_kmeans_vs_reference_output():
    pts, c0 = G["km_points"], G["km_centers0"]
    c = c0.copy()
    for it in range(3):
        c, assign, _ = oracle.lloyd_iter(pts, c)
        if it == 0:
            assert oracle.rel_fro(c, G["km_centers_iter1"]) <= TOL
    assert oracle.rel_fro(c, G["km_centers_iter3"]) <= TOL
    # flash::kmeans distance matrix and the isamin assignment derived from it
    a600, margin = oracle.kmeans_assign(pts[:600], c0)
    assert np.array_equal(a600, G["km_assign_600"])
    D = G["km_dist_600"].astype(np.float64)
    Dref = ((pts[:600, None, :].astype(np.float64) - c0[None].astype(np.float64)) ** 2).sum(-1)
    assert oracle.rel_fro(D, Dref) <= TOL


# ---------------------------------------------------------------- live reference binaries (fresh inputs)
@needs_ref
def test_live_reference_gemm_default_tiles():
    """1100 x 900 x 8300: two k tiles of the DEFAULT build (GEMM_BLK_SIZE = 8192) -> one beta=1 chain."""
    M, N, K = 1100, 900, 8300
    a, b = oracle.gen_dense(M * K, seed=31), oracle.gen_dense(K * N, seed=32)
    c = oracle.gen_dense(M * N, seed=33)
    got = rr.gemm("R", "N", "N", M, N, K, 1.0, 0.5, a, b, c, K, N, N, flash=True)
    want = oracle.gemm("R", "N", "N", M, N, K, 1.0, 0.5, a, b, c, K, N, N, acc64=True)
    assert oracle.rel_fro(got.reshape(M, N), want.reshape(M, N)) <= TOL


@needs_ref
@pytest.mark.parametrize("flash", [False, True], ids=["in_mem", "flash"])
def test_live_reference_sparse(flash):
    m, n, k = 5000, 4200, 128
    a, ia, ja = oracle.gen_csr(m, n, 24, seed=41)
    B, C0 = oracle.gen_dense((n, k), seed=42), oracle.gen_dense((m, k), seed=43)
    sfx = "_small" if flash else ""
    got = rr.csrmm("N", m, n, k, 1.25, 0.75, a, ia, ja, "R", B, C0, flash=flash, suffix=sfx)
    assert oracle.rel_fro(got, oracle.csrmm("N", m, n, k, 1.25, 0.75, a, ia, ja, "R", B, C0)) <= TOL
    x = oracle.gen_dense((n,), seed=44)
    xt = oracle.gen_dense((m,), seed=45)
    assert oracle.rel_fro(rr.csrgemv("N", m, n, a, ia, ja, x, flash=flash, suffix=sfx),
                          oracle.csrgemv("N", m, n, a, ia, ja, x)) <= TOL
    assert oracle.rel_fro(rr.csrgemv("T", m, n, a, ia, ja, xt, flash=flash, suffix=sfx),
                          oracle.csrgemv("T", m, n, a, ia, ja, xt)) <= TOL
    assert same_csc(rr.csrcsc(m, n, ia, ja, a, flash=flash, suffix=sfx), oracle.csrcsc(m, n, ia, ja, a))


@needs_ref
def test_live_reference_kmeans_five_iterations():
    rng = np.random.default_rng(7)
    K, d, P = 24, 48, 6000
    mu = (rng.normal(size=(K, d)) * 4).astype(np.float32)
    pts = (mu[rng.integers(0, K, P)] + 0.3 * rng.normal(size=(P, d))).astype(np.float32)
    c = pts[:K].copy()
    want = rr.kmeans_iters(pts, c, iters=5)
    for _ in range(5):
        c, _, _ = oracle.lloyd_iter(pts, c)
    assert oracle.rel_fro(c, want) <= TOL
