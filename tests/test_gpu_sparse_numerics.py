"""GPU numerics of the sparse kernels (sparse.cu: SpMM on every launch path of launch_spmm_rm, SpMV 'N' / 'T') and of
the host pipelines around them, element by element against a float64 reference computed on the device.

Bound, for every element of C = alpha op(A) B + beta C0 with mixed-sign data in [-1, 1):

    |C - R| <= (d_r + 2) * 2^-24 * |alpha| * (|A||B|)_rj + 2^-23 * |beta * C0_rj|

d_r is the summation depth of output row r on the path the launcher takes (the +2 covers the product alpha * acc
and the final fmaf with beta):
  * rows of at most 1024 nonzeros, and every row in the generic, TMA and BOF_SPMM_NO_SPLIT kernels: d = nnz_r
    (one fmaf chain in nonzero order per column);
  * block-split rows (1024 < nnz_r <= max(16384, 64 x mean row length of the launch)):
    d = 32 * ceil(nseg / 8) + 8 with nseg = ceil(nnz_r / 32) (8 warps, then the warp-order sum);
  * grid-split rows (longer): d = 32 * ceil(nseg / (8 G)) + 8 + G with G = 2 x #SMs blocks (then the block-order sum);
  * host pipelines: which row block sets the mean is the pipeline's choice, so a row above 1024 nonzeros gets the
    larger of the two split depths;
  * SpMV 'N': d = ceil(nnz_r / 16) + 4 (16 lanes, then a shuffle tree);
  * SpMV 'T', sorted: d = ceil(nnz_c / 8) + 3, plus the number of row blocks in the host pipeline;
  * SpMV 'T', atomic: d = nnz_c.
Non-finite reference elements must be matched exactly (NaN by NaN, Inf by the same Inf); every other element must be
finite and within the bound.  A failure names the worst elements and the maximum ratio per row class (short, block,
grid) and per column chunk of 4 L KV columns.  The bound rejects a reference with one nonzero or one 32-nonzero
segment left out (test_bound_rejects_*), so a kernel that drops either cannot pass.

Exact properties, bit for bit: run-to-run and row-permutation equivariance (also with more than 4096 grid-split rows
in one launch), column-slice invariance for rows of at most 1024 nonzeros across the kernels (each accumulates one
column in nonzero order with fmaf, then alpha * acc and fmaf(beta, old, .)), and resident against streamed csrmm
while every row has at most 16384 nonzeros.

Knobs the library reads once per process (BOF_SPMM_VARIANT, BOF_SPMM_NO_SPLIT, BOF_CSRMM_KPANEL) run in a child
process, sparse_numerics_child.py, which also holds the reference and the bound."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from sparse_numerics_child import (BLOCK, GRID, MID_ROW, Csr, assert_bound, bound_ratio, cdiv, classes, from_lens, gen,
                                   long_rows_csr, nonfinite_case, padded, permute_rows, pipeline_depth, reference,
                                   run_spmm, same_bits, signed, spmm_depth, spmm_reference, unrebase, zipf_csr)

pytestmark = pytest.mark.gpu
CHILD = Path(__file__).parent / "sparse_numerics_child.py"
NAN = float("nan")

# 1024 / 1025: the edge of deferral; 16384 / 16385: the edge of the grid split at a mean that makes 16384 the threshold
LONG = [1024, 1025, 3000, 16384, 16385, 40000]


@pytest.fixture(scope="module")
def long_csr():
    """2000 rows of 0..48 nonzeros (mean ~63, so the grid threshold is 16384) and the LONG rows: 1024 stays in the
    row-group kernel, 1025, 3000 and 16384 are block-split, 16385 and 40000 grid-split."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    A = long_rows_csr(2000, 5000, LONG, seed=1)
    cls = classes(A.lens)
    assert int((cls == BLOCK).sum()) == 3 and int((cls == GRID).sum()) == 2
    return A


def spmm(ctx, A, B, k, ldb, alpha=1.0):
    C = torch.full((A.m, k), NAN, device="cuda")
    ctx.spmm("R", A.m, A.n, k, alpha, A.vals, A.idx, A.offs, B, ldb, 0.0, C, k)
    return C


# ---------------------------------------------------------------------------------------------------------------
# the harness itself
# ---------------------------------------------------------------------------------------------------------------
def test_bound_rejects_a_dropped_nonzero_and_a_dropped_segment(ctx, long_csr):
    A, k = long_csr, 32
    B = signed((A.n, k), gen(2))
    C = spmm(ctx, A, B, k, k)
    cls = classes(A.lens)
    depth = spmm_depth(A.lens, cls)
    R, S, _ = spmm_reference(A, B, k)
    assert float(bound_ratio(C, R, S, None, depth).max()) <= 1.0
    base = A.offs - A.offs[0]
    others = torch.ones(A.m, dtype=torch.bool, device="cuda")

    r = int(torch.nonzero((A.lens >= 8) & (A.lens <= 48))[0])
    keep = torch.ones(A.nnz, dtype=torch.bool, device="cuda")
    keep[int(base[r]) + 3] = False
    ratio = bound_ratio(C, spmm_reference(A, B, k, keep=keep)[0], S, None, depth)
    others[r] = False
    assert float(ratio[r].max()) > 1.0 and float(ratio[others].max()) <= 1.0, "one dropped nonzero of a short row"

    r = int(torch.argmax(A.lens))
    assert int(cls[r]) == GRID
    z0 = int(base[r]) + 32 * (int(A.lens[r]) // 64)
    keep = torch.ones(A.nnz, dtype=torch.bool, device="cuda")
    keep[z0:z0 + 32] = False
    ratio = bound_ratio(C, spmm_reference(A, B, k, keep=keep)[0], S, None, depth)
    assert float(ratio[r].max()) > 1.0, "one dropped 32-nonzero segment of the longest grid row"


# ---------------------------------------------------------------------------------------------------------------
# SpMM device paths within the bound
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [4, 12, 16, 28, 32, 48, 64, 100, 128, 132, 200, 256, 260, 640])
def test_spmm_row_group_kernels(ctx, long_csr, k):
    """L = 4, 8, 16, 32 lanes, KV = 1, 2, with long rows deferred (KV = 1, 2, 4 there): un-rebased offsets, padded ldb
    (NaN padding, never read) and ldc (padding untouched)."""
    run_spmm(ctx, unrebase(long_csr), signed((long_csr.n, k), gen(k)), k, ldb=k + 4, ldc=k + 8, split=True,
             what="row-group")


# case -> (k, ldb, ldc, B offset in floats)
GENERIC = {"k7": (7, 11, 9, 0), "k131": (131, 135, 133, 0), "k128_ldb130": (128, 130, 132, 0),
           "k128_B_unaligned": (128, 132, 132, 1)}


@pytest.mark.parametrize("case", list(GENERIC))
def test_spmm_generic_kernel(ctx, long_csr, case):
    """k not a multiple of 4, ldb not a multiple of 4, B not 16-byte aligned: the warp-per-row kernel, every row in
    nonzero order (no deferral)."""
    k, ldb, ldc, shift = GENERIC[case]
    run_spmm(ctx, unrebase(long_csr), signed((long_csr.n, k), gen(k)), k, ldb=ldb, ldc=ldc, split=False, b_shift=shift,
             what=case)


@pytest.mark.parametrize("k", [128, 200])
def test_spmm_l2_slice_policy(ctx, k):
    """B of 72-112 MB (more than half of L2; a 64-column slice fits): 16-lane row groups over 64-column chunks."""
    A = long_rows_csr(4096, 140_000, [1025, 3000, 20000], seed=23, hi=30)
    run_spmm(ctx, unrebase(A), signed((A.n, k), gen(k)), k, ldb=k, ldc=k + 4, split=True, what="l2-slice")


@pytest.mark.parametrize("k", [4, 32, 132, 640])
def test_spmm_zipf_rows(ctx, k):
    A = zipf_csr(6000, 40000, 1_200_000, seed=100 + k)
    cls = classes(A.lens)
    assert int((cls == GRID).sum()) >= 4 and int((cls == BLOCK).sum()) >= 20
    run_spmm(ctx, unrebase(A), signed((A.n, k), gen(k)), k, ldb=k, ldc=k + 4, split=True, what="zipf")


# case -> (k, ldb - n, ldc - m)
COLMAJ = {"k12": (12, 3, 11), "k7": (7, 0, 5), "k130": (130, 8, 4)}


@pytest.mark.parametrize("case", list(COLMAJ))
def test_spmm_column_major_entry(ctx, long_csr, case):
    """bof_spmm_csr_f32 with ord 'C': B (n x k, ldb > n) and C (m x k, ldc > m) column-major.  Within the bound, padding
    untouched, and the same bits as the row-major entry on the same kernel family."""
    k, pb, pc = COLMAJ[case]
    A = unrebase(long_csr)
    m, n = A.m, A.n
    ldb, ldc = n + pb, m + pc
    g = gen(k)
    Bdata, C0 = signed((n, k), g), signed((m, k), g)
    _, Bcm = padded(k, n, ldb, NAN, Bdata.T)
    cls = classes(A.lens, split=k % 4 == 0)
    depth = spmm_depth(A.lens, cls)
    for alpha, beta in ((1.0, 0.0), (1.5, 0.5)):
        _, Ccm = padded(k, m, ldc, NAN if beta == 0 else 7.0, None if beta == 0 else C0.T)
        before = Ccm[:, m:].clone()
        ctx.spmm("C", m, n, k, alpha, A.vals, A.idx, A.offs, Bcm, ldb, beta, Ccm, ldc)
        got = Ccm[:, :m].T
        assert_bound(got, spmm_reference(A, Bdata, k, alpha, beta, C0), depth, cls, 0, f"column-major {case}")
        assert same_bits(Ccm[:, m:], before)
        _, Brm = padded(n, k, k + 4 if k % 4 == 0 else k, NAN, Bdata)
        Crm = C0.clone() if beta else torch.full((m, k), NAN, device="cuda")
        ctx.spmm("R", m, n, k, alpha, A.vals, A.idx, A.offs, Brm, Brm.shape[1], beta, Crm, k)
        assert same_bits(got, Crm), f"column-major {case}: differs from row-major"


@pytest.mark.parametrize("k,split", [(32, True), (128, True), (131, False)])
def test_spmm_nonfinite(ctx, long_csr, k, split):
    """+Inf / -Inf in referenced rows of B (one column where both reach a row: NaN), NaN in A, 0 against Inf, on
    short, block and grid rows (split) and in the generic kernel.  Non-finite outputs exactly where the float64
    reference has them, with their sign; the rest finite and within the bound; padding untouched."""
    A, B = nonfinite_case(unrebase(long_csr), long_csr.n, k, seed=k)
    outs = run_spmm(ctx, A, B, k, ldb=k, ldc=k + 4 if split else k + 1, split=split, what="non-finite")
    assert not bool(torch.isfinite(outs[0]).all())


# ---------------------------------------------------------------------------------------------------------------
# exact properties
# ---------------------------------------------------------------------------------------------------------------
def test_zipf_row_permutation_equivariance(ctx):
    A = zipf_csr(6000, 40000, 1_200_000, seed=7)
    k = 128
    B = signed((A.n, k), gen(8))
    perm = torch.randperm(A.m, device="cuda", generator=gen(9))
    C = spmm(ctx, A, B, k, k, alpha=1.5)
    assert same_bits(spmm(ctx, permute_rows(A, perm), B, k, k, alpha=1.5), C[perm])


@pytest.fixture(scope="module")
def spill_csr():
    """300 000 rows, 4200 of them with 16 500 nonzeros, the rest 0..8 (~70 M nonzeros, mean ~235, so the threshold is
    16384): more grid-split rows than the 4096 a launch once took before spilling the rest to the block path."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    g = gen(42)
    m = 300_000
    lens = torch.randint(0, 9, (m,), device="cuda", generator=g)
    lens[torch.randperm(m, device="cuda", generator=g)[:4200]] = 16500
    A = from_lens(lens, 8192, g)
    assert int((classes(A.lens) == GRID).sum()) == 4200
    return A


def test_spill_matrix_repeat_runs_identical(ctx, spill_csr):
    A, k = spill_csr, 32
    B = signed((A.n, k), gen(43))
    runs = [spmm(ctx, A, B, k, k) for _ in range(3)]
    assert same_bits(runs[0], runs[1]) and same_bits(runs[0], runs[2])
    cls = classes(A.lens)
    assert_bound(runs[0], spmm_reference(A, B, k), spmm_depth(A.lens, cls), cls, 32, "spill matrix")


def test_spill_matrix_row_permutation_equivariance(ctx, spill_csr):
    A, k = spill_csr, 32
    B = signed((A.n, k), gen(43))
    perm = torch.randperm(A.m, device="cuda", generator=gen(44))
    assert same_bits(spmm(ctx, permute_rows(A, perm), B, k, k), spmm(ctx, A, B, k, k)[perm])


def test_column_slice_invariance(ctx, long_csr):
    """C(A, B[:, :16]) == C(A, B)[:, :16] for rows of at most 1024 nonzeros: L = 4 against L = 8, 16, 32 (KV 1, 2),
    the generic kernel (ldb = 130) and the column-major entry (k = 20 and 7 inside).  Block-split rows use the same
    8-warp tree at every k, so they match across the row-group kernels too."""
    A = unrebase(long_csr)
    m, n = A.m, A.n
    Bdata = signed((n, 640), gen(3))
    _, B = padded(n, 640, 644, NAN, Bdata)
    short = A.lens <= MID_ROW
    block = classes(A.lens) == BLOCK
    C16 = spmm(ctx, A, B, 16, 644, alpha=1.5)
    for k in (32, 64, 128, 256, 640):
        Ck = spmm(ctx, A, B, k, 644, alpha=1.5)
        assert same_bits(Ck[short, :16], C16[short]), f"k={k}: short rows"
        assert same_bits(Ck[block, :16], C16[block]), f"k={k}: block-split rows"
    _, Bg = padded(n, 128, 130, NAN, Bdata[:, :128])
    assert same_bits(spmm(ctx, A, Bg, 128, 130, alpha=1.5)[short, :16], C16[short]), "generic kernel"
    for k in (20, 7):
        _, Bcm = padded(k, n, n + 1, NAN, Bdata[:, :k].T)
        Ccm = torch.full((k, m), NAN, device="cuda")
        ctx.spmm("C", m, n, k, 1.5, A.vals, A.idx, A.offs, Bcm, n + 1, 0.0, Ccm, m)
        w = min(k, 16)
        assert same_bits(Ccm.T[short, :w], C16[short, :w]), f"column-major k={k}"


@pytest.mark.parametrize("longest", [16384, 30000])
def test_resident_against_streamed(bof, ctx, longest):
    """bof_csr_mm (64-column panels over 262144-row blocks, so rows of the second block have a nonzero base) against
    bof_host_csrmm (nnz budget 20000: the longest row forms a block of its own).  Same bits while every row has at
    most 16384 nonzeros; a longer row is grid-split by one and block-split by the other, so only the bound holds."""
    m, n, k = 300_000, 6000, 200
    g = gen(longest)
    lens = torch.randint(0, 5, (m,), device="cuda", generator=g)
    lens[[10, 262_150, 262_200, 299_000]] = torch.tensor([2000, 1025, longest, 16384], device="cuda")
    A = from_lens(lens, n, g)
    a, ia, ja = A.host()
    B, C0 = signed((n, k), g), signed((m, k), g)
    Bh = B.cpu().numpy()
    depth, cls = pipeline_depth(A.lens), classes(A.lens)
    h = bof.ResidentCsr(ctx, m, n, a, ia, ja)
    try:
        with bof.Context(device=0, csrmm_max_nnz=20000) as c2:
            for alpha, beta in ((1.0, 0.0), (1.5, 0.5)):
                ref = spmm_reference(A, B, k, alpha, beta, C0)
                fill = C0.cpu().numpy() if beta else np.full((m, k), np.nan, np.float32)
                c_res, c_str = fill.copy(), fill.copy()
                h.mm("N", k, alpha, beta, "R", Bh, c_res)
                c2.host_csrmm("N", m, n, k, alpha, beta, a, ia, ja, "R", Bh, c_str)
                for name, c in (("resident", c_res), ("streamed", c_str)):
                    assert_bound(torch.from_numpy(c).cuda(), ref, depth, cls, 64, f"{name} alpha={alpha} beta={beta}")
                if longest <= 16384:
                    assert np.array_equal(c_res.view(np.int32), c_str.view(np.int32))
    finally:
        h.close()


# ---------------------------------------------------------------------------------------------------------------
# SpMV
# ---------------------------------------------------------------------------------------------------------------
def spmv_n_check(ctx, A, x, what):
    y = torch.full((A.m,), NAN, device="cuda")
    ctx.spmv("N", A.m, A.n, A.vals, A.idx, A.offs, x, y)
    ref = reference(A.vals, A.rows(), A.idx, x, A.m, 0)
    assert_bound(y, ref, cdiv(A.lens, 16) + 4, classes(A.lens), 0, what)
    return y


def spmv_t_ref(A, x):
    R, S, _ = reference(A.vals, A.idx, A.rows(), x, A.n, 0)
    nnz_c = torch.bincount(A.idx.long(), minlength=A.n)
    return (R, S, None), nnz_c


def test_spmv_n_zipf_rows(ctx):
    A = unrebase(zipf_csr(6000, 40000, 1_200_000, seed=11))
    spmv_n_check(ctx, A, signed(A.n, gen(12)), "spmv N zipf")


def wide_t_csr():
    """n = 70000 > 2^16 columns (three radix passes), columns >= 60000 empty, a few rows of 3000..20000 nonzeros."""
    return unrebase(long_rows_csr(50_000, 70_000, [3000, 20000], seed=13, hi=40), lead=1)


def test_spmv_t_sorted_wide(ctx):
    A = wide_t_csr()
    A = Csr(A.vals, A.idx % 60000, A.offs, A.n)
    x = signed(A.m, gen(14))
    y = torch.full((A.n,), NAN, device="cuda")
    ctx.spmv("T", A.m, A.n, A.vals, A.idx, A.offs, x, y)
    ref, nnz_c = spmv_t_ref(A, x)
    assert_bound(y, ref, cdiv(nnz_c, 8) + 3, torch.zeros_like(nnz_c), 0, "spmv T sorted")
    assert bool((y[nnz_c == 0] == 0).all()) and int((nnz_c == 0).sum()) >= 10000


def test_spmv_t_atomic(bof, ctx):
    A = wide_t_csr()
    x = signed(A.m, gen(15))
    with bof.Context(device=0, spmv_t_atomic=1) as c2:
        y = torch.full((A.n,), NAN, device="cuda")
        c2.spmv("T", A.m, A.n, A.vals, A.idx, A.offs, x, y)
    ref, nnz_c = spmv_t_ref(A, x)
    assert_bound(y, ref, nnz_c, torch.zeros_like(nnz_c), 0, "spmv T atomic")


def row_blocks(ia, budget):
    """The host pipeline's nnz-budgeted row blocks (partition_rows in sparse_host.cu)."""
    m, r, nb = len(ia) - 1, 0, 0
    while r < m:
        e = int(np.searchsorted(ia, ia[r] + budget, side="right")) - 1
        r, nb = max(e, r + 1), nb + 1
    return nb


def test_host_csrgemv_t_row_blocks(bof):
    A = wide_t_csr()
    a, ia, ja = A.host()
    x = signed(A.m, gen(16))
    budget = 100_000
    nb = row_blocks(ia, budget)
    assert nb >= 8
    ys = []
    with bof.Context(device=0, csrmm_max_nnz=budget) as c2:
        for _ in range(2):
            y = np.full(A.n, np.nan, np.float32)
            c2.host_csrgemv("T", A.m, A.n, a, ia, ja, x.cpu().numpy(), y)
            ys.append(y)
    ref, nnz_c = spmv_t_ref(A, x)
    assert_bound(torch.from_numpy(ys[0]).cuda(), ref, cdiv(nnz_c, 8) + 3 + nb, torch.zeros_like(nnz_c), 0,
                 "host csrgemv T")
    assert np.array_equal(ys[0].view(np.int32), ys[1].view(np.int32))


def test_spmv_nonfinite_x(bof, ctx):
    """Inf and NaN in x reach exactly the outputs the float64 reference puts them in, with their sign."""
    A = unrebase(long_rows_csr(3000, 2000, [3000], seed=17, hi=20))
    x = signed(A.n, gen(18))
    x[[3, 4, 5]] = torch.tensor([float("inf"), float("-inf"), NAN], device="cuda")
    y = spmv_n_check(ctx, A, x, "spmv N non-finite x")
    assert not bool(torch.isfinite(y).all()) and bool(torch.isfinite(y).any())
    xt = signed(A.m, gen(19))
    xt[[3, 4, 5]] = torch.tensor([float("inf"), float("-inf"), NAN], device="cuda")
    ref, nnz_c = spmv_t_ref(A, xt)
    for atomic in (0, 1):
        with bof.Context(device=0, spmv_t_atomic=atomic) as c2:
            y = torch.full((A.n,), NAN, device="cuda")
            c2.spmv("T", A.m, A.n, A.vals, A.idx, A.offs, xt, y)
        depth = nnz_c if atomic else cdiv(nnz_c, 8) + 3
        assert_bound(y, ref, depth, torch.zeros_like(nnz_c), 0, f"spmv T non-finite x atomic={atomic}")


# ---------------------------------------------------------------------------------------------------------------
# host pipelines
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ord_b", ["R", "C"])
def test_host_csrmm_n_row_above_budget(bof, ord_b):
    """flash::csrmm 'N' with an nnz budget of 20000: rows of 30000 and 40000 nonzeros form blocks of their own."""
    A = long_rows_csr(3000, 2500, [1025, 5000, 17000, 30000, 40000], seed=31)
    m, n, k = A.m, A.n, 96
    a, ia, ja = A.host()
    g = gen(32)
    B, C0 = signed((n, k), g), signed((m, k), g)
    lay = (lambda X: X.cpu().numpy().copy()) if ord_b == "R" else (lambda X: X.T.contiguous().cpu().numpy())
    depth, cls = pipeline_depth(A.lens), classes(A.lens)
    with bof.Context(device=0, csrmm_max_nnz=20000) as c2:
        for alpha, beta in ((1.0, 0.0), (1.5, 0.5)):
            c = lay(C0) if beta else np.full((m, k), np.nan, np.float32)
            c2.host_csrmm("N", m, n, k, alpha, beta, a, ia, ja, ord_b, lay(B), c)
            got = torch.from_numpy(c).cuda()
            got = got if ord_b == "R" else got.view(k, m).T
            assert_bound(got, spmm_reference(A, B, k, alpha, beta, C0), depth, cls, 0, f"host csrmm N {ord_b}")


def test_host_csrmm_t_dense_columns(bof):
    """flash::csrmm 'T': columns 7, 8 and 9 of A are in every row, so after the transpose they are rows of 40000
    nonzeros, grid-split (the mean of A^T is ~250)."""
    m, n, k = 40_000, 3000, 64
    g = gen(33)
    A = from_lens(torch.randint(3, 12, (m,), device="cuda", generator=g), n, g)
    for j in range(3):
        A.idx[A.offs[:-1] + j] = 7 + j
    a, ia, ja = A.host()
    nnz_c = torch.bincount(A.idx.long(), minlength=n)
    cls = classes(nnz_c)
    assert int((cls == GRID).sum()) == 3
    B, C0 = signed((m, k), g), signed((n, k), g)
    with bof.Context(device=0) as c2:
        for alpha, beta in ((1.0, 0.0), (1.5, 0.5)):
            c = C0.cpu().numpy().copy() if beta else np.full((n, k), np.nan, np.float32)
            c2.host_csrmm("T", m, n, k, alpha, beta, a, ia, ja, "R", B.cpu().numpy(), c)
            ref = spmm_reference(A, B, k, alpha, beta, C0, trans=True)
            assert_bound(torch.from_numpy(c).cuda(), ref, pipeline_depth(nnz_c), cls, 0, "host csrmm T")


# ---------------------------------------------------------------------------------------------------------------
# knobs read once per process: child processes
# ---------------------------------------------------------------------------------------------------------------
def run_child(mode, env):
    r = subprocess.run([sys.executable, str(CHILD), mode], env=dict(os.environ, **env), capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "SPARSE_CHILD_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


KNOBS = {f"variant{v}": {"BOF_SPMM_VARIANT": str(v)} for v in range(13)}
KNOBS["no_split"] = {"BOF_SPMM_NO_SPLIT": "1"}


@pytest.mark.parametrize("knob", list(KNOBS))
def test_spmm_knob_paths_child_process(knob):
    """Every BOF_SPMM_VARIANT (0-12: register tunings, TMA-staged 6 and 7, the L2-slice kernel 12) and
    BOF_SPMM_NO_SPLIT at k = 128 and 256: bound, non-finite inputs, column-slice invariance against k = 16, aligned
    and unaligned A streams (TMA bulk and fallback staging, slices over 2048 elements)."""
    run_child("variant", KNOBS[knob])


def test_host_csrmm_column_panels_long_rows_child_process():
    run_child("kpanel", {"BOF_CSRMM_KPANEL": "64"})
