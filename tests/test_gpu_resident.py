"""GPU parity: A resident in HBM across calls (bof_csr_*, SURVEY 8(f)-2) -- the in-memory-B/C csrmm overload and
csrgemv as an eigensolver inner loop.  Same oracle and tolerance as the streamed entry points.  While every row has
at most 16384 nonzeros the resident products equal the streamed ones bit for bit (same per-row summation order).  A
longer row may be summed over the whole grid by one and over the 8 warps of a block by the other, so beyond that
only the error bound is shared (tests/test_gpu_sparse_numerics.py checks both sides of the line)."""
import numpy as np
import pytest
import torch

import oracle
from gpu_util import ragged_csr

pytestmark = pytest.mark.gpu
TOL = 1e-5


def dense_pair(rng, rows_b, rows_c, k, ord_b):
    B = rng.random((rows_b, k), dtype=np.float32)
    C0 = rng.random((rows_c, k), dtype=np.float32)
    if ord_b == "C":
        return B, C0, np.asfortranarray(B).T.copy().reshape(-1), np.asfortranarray(C0).T.copy().reshape(-1)
    return B, C0, B.reshape(-1).copy(), C0.reshape(-1).copy()


def unpack(flat, rows, k, ord_b):
    return flat.reshape(rows, k) if ord_b == "R" else flat.reshape(k, rows).T


@pytest.mark.parametrize("trans", ["N", "T"])
@pytest.mark.parametrize("ord_b", ["R", "C"])
@pytest.mark.parametrize("k", [8, 128, 200, 384])
def test_resident_mm_matches_oracle_and_streamed(bof, ctx, trans, ord_b, k):
    rng = np.random.default_rng(100 + k)
    m, n = 1500, 1100
    a, ia, ja = ragged_csr(rng, m, n, 30)
    rows_b, rows_c = (n, m) if trans == "N" else (m, n)
    h = bof.ResidentCsr(ctx, m, n, a, ia, ja)
    try:
        for alpha, beta in ((1.0, 0.0), (1.5, 0.5)):
            B, C0, bflat, cflat = dense_pair(rng, rows_b, rows_c, k, ord_b)
            c_res = cflat.copy() if beta else np.full_like(cflat, np.nan)  # beta == 0: C must not be read
            h.mm(trans, k, alpha, beta, ord_b, bflat, c_res)
            ref = oracle.csrmm(trans, m, n, k, alpha, beta, a, ia, ja, "R", B, C0, acc64=True)
            assert oracle.rel_fro(unpack(c_res, rows_c, k, ord_b), ref) <= TOL
            c_str = cflat.copy()
            ctx.host_csrmm(trans, m, n, k, alpha, beta, a, ia, ja, ord_b, bflat, c_str)
            assert np.array_equal(c_res, c_str)
    finally:
        h.close()


def test_resident_mm_many_row_blocks_and_repeat_calls(bof, ctx):
    """Wide enough that the output splits into several row blocks per panel; repeated calls reuse the handle."""
    rng = np.random.default_rng(7)
    m, n, k = 300_000, 4096, 256   # rows_blk = 262144 at 64-wide panels -> 2 row blocks x 4 panels
    nzr = 6
    ia = np.arange(m + 1, dtype=np.int64) * nzr
    ja = np.sort(rng.integers(0, n, size=(m, nzr)), axis=1).reshape(-1).astype(np.int64)
    a = (rng.integers(1, 10, size=m * nzr)).astype(np.float32)        # (i % 9) + 1 style integer data: exact
    B = rng.integers(0, 10, size=(n, k)).astype(np.float32)
    h = bof.ResidentCsr(ctx, m, n, a, ia, ja)
    try:
        Bt = torch.from_numpy(B).pin_memory()
        Ct = torch.empty((m, k), dtype=torch.float32).pin_memory()
        outs = []
        for _ in range(3):
            Ct.fill_(float("nan"))
            h.mm("N", k, 1.0, 0.0, "R", Bt, Ct)
            outs.append(Ct.numpy().copy())
        import scipy.sparse as sp
        ref = (sp.csr_matrix((a.astype(np.float64), ja, ia), shape=(m, n)) @ B.astype(np.float64)).astype(np.float32)
        assert np.array_equal(outs[0], ref)        # integer data: every fp32 sum is exact
        assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[1], outs[2])
    finally:
        h.close()


@pytest.mark.parametrize("with_t", [False, True])
def test_resident_mv(bof, ctx, with_t):
    rng = np.random.default_rng(9)
    m, n = 5000, 3700
    a, ia, ja = ragged_csr(rng, m, n, 50)
    h = bof.ResidentCsr(ctx, m, n, a, ia, ja)
    try:
        if with_t:
            h.build_transpose()
        for trans in "NT":
            x = rng.random(n if trans == "N" else m, dtype=np.float32)
            y = np.full(m if trans == "N" else n, np.nan, np.float32)
            h.mv(trans, x, y)
            assert oracle.rel_fro(y, oracle.csrgemv(trans, m, n, a, ia, ja, x, acc64=True)) <= TOL
            if trans == "T" and with_t:  # gather SpMV on the resident A^T: run-to-run deterministic
                y2 = np.empty_like(y); h.mv(trans, x, y2)
                assert np.array_equal(y, y2)
    finally:
        h.close()


def test_resident_arrays_feed_the_device_tile_kernels(bof, ctx):
    """bof_csr_arrays + bof_spmm_csr_f32 with B and C kept on the device (a fully device-side Krylov step)."""
    rng = np.random.default_rng(10)
    m, n, k = 900, 700, 64
    a, ia, ja = ragged_csr(rng, m, n, 25)
    h = bof.ResidentCsr(ctx, m, n, a, ia, ja)
    try:
        for trans, rows_c, rows_b in (("N", m, n), ("T", n, m)):
            vals, idx, offs, nnz = h.arrays(trans)
            assert nnz == int(ia[-1])
            B = rng.random((rows_b, k), dtype=np.float32)
            Bd = torch.from_numpy(B).cuda(); Cd = torch.empty((rows_c, k), device="cuda")
            ctx.spmm("R", rows_c, rows_b, k, 1.0, vals, idx, offs, Bd, k, 0.0, Cd, k)
            ref = oracle.csrmm(trans, m, n, k, 1.0, 0.0, a, ia, ja, "R", B, np.zeros((rows_c, k), np.float32), acc64=True)
            assert oracle.rel_fro(Cd.cpu().numpy(), ref) <= TOL
    finally:
        h.close()


def test_resident_edge_cases(bof, ctx):
    a = np.zeros(0, np.float32); ja = np.zeros(0, np.int64)
    ia = np.zeros(6, np.int64)                       # 5 x 4 matrix with no nonzeros
    h = bof.ResidentCsr(ctx, 5, 4, a, ia, ja)
    try:
        B = np.ones((4, 8), np.float32); C = np.full((5, 8), 3.0, np.float32)
        h.mm("N", 8, 1.0, 2.0, "R", B, C)
        assert np.all(C == 6.0)
        y = np.full(4, np.nan, np.float32)
        h.mv("T", np.ones(5, np.float32), y)
        assert np.all(y == 0.0)
        with pytest.raises(bof.BofError):
            h.mm("X", 8, 1.0, 0.0, "R", B, C)
    finally:
        h.close()
