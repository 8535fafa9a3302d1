"""flash::gemv on the GPU: fp64 parity for every layout, the chunk contract (the same bits from the device entry point,
the host pipeline at any tiling, pinned or pageable buffers, and the two layouts that store the same matrix), IEEE
special values, PCIe accounting, argument errors and the C++ driver on mapped files."""
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
LAYOUTS = [("R", "N"), ("R", "T"), ("C", "N"), ("C", "T")]


def stored(A, ord_, pad=0, fill=np.nan):
    """A (m x n) as the library reads it: rows of A ('R') or of A^T ('C') with leading dimension tight + pad; the padding
    holds `fill` so that reading it shows up in the result."""
    S = A if ord_ == "R" else A.T
    buf = np.full((S.shape[0], S.shape[1] + pad), fill, dtype=np.float32)
    buf[:, :S.shape[1]] = S
    return buf, (S.shape[1] + pad if pad else 0)


def lens(trans, m, n):
    return (n, m) if trans == "N" else (m, n)   # (len x, len y)


def ref64(A, trans, alpha, beta, x, y0):
    """alpha * op(A) x + beta * y0 in fp64, elementwise IEEE (0 * Inf = NaN), and |alpha| |op(A)| |x| for the bound"""
    M = (A if trans == "N" else A.T).astype(np.float64)
    x64 = x.astype(np.float64)
    dot = (M * x64[None, :]).sum(axis=1) if M.size else np.zeros(M.shape[0])
    mag = (np.abs(M) * np.abs(x64)[None, :]).sum(axis=1) if M.size else np.zeros(M.shape[0])
    out = alpha * dot
    if beta != 0:
        out = out + beta * y0.astype(np.float64)
    return out, abs(alpha) * mag


def check_bound(y, y64, mag):
    err = np.abs(y.astype(np.float64) - y64)
    tol = 2.0 ** -16 * mag + 2.0 ** -22 * np.abs(y64)
    bad = ~(err <= tol)
    assert not bad.any(), f"{bad.sum()} outputs out of bound, worst {err[bad].max()} vs {tol[bad].min()}"


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def problem(m, n, trans, seed, beta):
    rng = np.random.default_rng(seed)
    A = (rng.random((m, n), dtype=np.float32) - 0.5)
    xl, yl = lens(trans, m, n)
    x = rng.random(xl, dtype=np.float32) - 0.5
    y0 = np.full(yl, np.nan, np.float32) if beta == 0 else rng.random(yl, dtype=np.float32)
    return A, x, y0


def host_run(ctx, ord_, trans, m, n, alpha, beta, A, x, y0, pad=0):
    buf, lda = stored(A, ord_, pad)
    y = y0.copy()
    ctx.host_gemv(ord_, trans, m, n, alpha, beta, buf, x, y, lda=lda)
    return y


def dev_run(ctx, ord_, trans, m, n, alpha, beta, A, x, y0, pad=0):
    buf, lda = stored(A, ord_, pad)
    Ad, xd, yd = (torch.from_numpy(v).cuda() for v in (buf, x, y0.copy()))
    ctx.sgemv(ord_, trans, m, n, alpha, Ad, lda, xd, beta, yd)
    torch.cuda.synchronize()
    return yd.cpu().numpy()


@pytest.mark.parametrize("ord_,trans", LAYOUTS)
@pytest.mark.parametrize("m,n", [(1537, 9001), (3, 100003), (100003, 5), (1, 1), (0, 7), (7, 0)])
@pytest.mark.parametrize("beta", [0.0, -0.75])
def test_parity_fp64(ctx, ord_, trans, m, n, beta):
    alpha = 1.25
    A, x, y0 = problem(m, n, trans, seed=m * 7 + n, beta=beta)
    y64, mag = ref64(A, trans, alpha, beta, x, y0)
    yh = host_run(ctx, ord_, trans, m, n, alpha, beta, A, x, y0, pad=3)
    check_bound(yh, y64, mag)
    yd = dev_run(ctx, ord_, trans, m, n, alpha, beta, A, x, y0, pad=3)
    assert np.array_equal(bits(yd), bits(yh)), "device entry point and host pipeline differ"


@pytest.mark.parametrize("rowdot", [True, False])
def test_same_memory_two_layouts(ctx, rowdot):
    """('R','N') on S and ('C','T') on the same memory are the same problem; so are ('R','T') and ('C','N')"""
    rng = np.random.default_rng(5)
    r, c, ld = 2049, 8195, 8200
    S = rng.random((r, ld), dtype=np.float32) - 0.5
    x = rng.random(c if rowdot else r, dtype=np.float32)
    y1 = np.zeros(r if rowdot else c, np.float32)
    y2 = y1.copy()
    ctx.host_gemv("R", "N" if rowdot else "T", r, c, 0.5, 0.0, S, x, y1, lda=ld)
    ctx.host_gemv("C", "T" if rowdot else "N", c, r, 0.5, 0.0, S, x, y2, lda=ld)
    assert np.array_equal(bits(y1), bits(y2))


@pytest.mark.parametrize("ord_,trans", LAYOUTS)
def test_pinned_and_pageable(ctx, ord_, trans):
    m, n, beta = 3001, 4099, 0.5
    A, x, y0 = problem(m, n, trans, seed=11, beta=beta)
    yp = host_run(ctx, ord_, trans, m, n, 2.0, beta, A, x, y0)
    buf, _ = stored(A, ord_)
    pin = [torch.from_numpy(v).pin_memory() for v in (buf, x, y0.copy())]
    ctx.host_gemv(ord_, trans, m, n, 2.0, beta, pin[0], pin[1], pin[2])
    assert np.array_equal(bits(pin[2].numpy()), bits(yp))


@pytest.mark.parametrize("ord_,trans", LAYOUTS)
@pytest.mark.parametrize("block_bytes", [16384, 3 * 16384 + 4, 1 << 20])
def test_tiling_is_bit_identical(ctx, monkeypatch, ord_, trans, block_bytes):
    """BOF_GEMV_BLOCK_BYTES that cut A on both axes (16 KiB: one chunk per tile) give the bits of the default tiling and
    of the device entry point"""
    beta = -0.75
    for (m, n) in [(1100, 9001), (20000, 300)]:
        A, x, y0 = problem(m, n, trans, seed=m + n, beta=beta)
        monkeypatch.delenv("BOF_GEMV_BLOCK_BYTES", raising=False)
        ref = host_run(ctx, ord_, trans, m, n, 1.5, beta, A, x, y0, pad=1)
        monkeypatch.setenv("BOF_GEMV_BLOCK_BYTES", str(block_bytes))
        got = host_run(ctx, ord_, trans, m, n, 1.5, beta, A, x, y0, pad=1)
        assert np.array_equal(bits(got), bits(ref)), (m, n)
        assert np.array_equal(bits(dev_run(ctx, ord_, trans, m, n, 1.5, beta, A, x, y0, pad=1)), bits(ref)), (m, n)


@pytest.mark.parametrize("ord_,trans,m,n", [("R", "N", 2, 30_000_001), ("C", "T", 30_000_001, 2),
                                            ("R", "T", 10_000_019, 3), ("C", "N", 3, 10_000_019)])
def test_long_rows_and_tall_skinny(ctx, ord_, trans, m, n):
    """row-dot of a few very long rows (split across CTAs, folded in a second pass) and column sums of a tall, narrow
    matrix (row-chunk parallelism) against fp64, device entry point and host pipeline bit-identical"""
    A, x, y0 = problem(m, n, trans, seed=3, beta=0.25)
    y64, mag = ref64(A, trans, 0.75, 0.25, x, y0)
    yd = dev_run(ctx, ord_, trans, m, n, 0.75, 0.25, A, x, y0)
    check_bound(yd, y64, mag)
    yh = host_run(ctx, ord_, trans, m, n, 0.75, 0.25, A, x, y0)
    assert np.array_equal(bits(yh), bits(yd))


@pytest.mark.parametrize("ord_,trans", LAYOUTS)
@pytest.mark.parametrize("alpha", [1.5, 0.0])
@pytest.mark.parametrize("where", ["A", "x"])
def test_special_values_reach_only_their_outputs(ctx, ord_, trans, alpha, where):
    """an Inf or NaN of A reaches only the output of its line; an Inf of x reaches every output, as NaN where it meets a
    zero of A; alpha = 0 is no shortcut (0 * Inf = NaN)"""
    m, n = 300, 5000
    rng = np.random.default_rng(9)
    A = rng.random((m, n), dtype=np.float32) + 0.5
    xl, yl = lens(trans, m, n)
    x = rng.random(xl, dtype=np.float32) + 0.5
    if where == "A":
        A[2, 5] = np.inf
        A[7, 4100] = np.nan
    else:
        A[9, 33] = 0.0
        x[33 if trans == "N" else 9] = -np.inf
    y0 = np.full(yl, np.nan, np.float32)
    y64, mag = ref64(A, trans, alpha, 0.0, x, y0)
    assert (~np.isfinite(y64)).any() and (where == "x" or np.isfinite(y64).sum() >= yl - 2)
    for y in (host_run(ctx, ord_, trans, m, n, alpha, 0.0, A, x, y0),
              dev_run(ctx, ord_, trans, m, n, alpha, 0.0, A, x, y0)):
        assert np.array_equal(np.isnan(y), np.isnan(y64))
        assert np.array_equal(np.isposinf(y), np.isposinf(y64)) and np.array_equal(np.isneginf(y), np.isneginf(y64))
        fin = np.isfinite(y64)
        check_bound(y[fin], y64[fin], mag[fin])


@pytest.mark.parametrize("beta", [0.0, 2.0])
@pytest.mark.parametrize("block_bytes", [None, 16384])
def test_pcie_accounting(ctx, monkeypatch, beta, block_bytes):
    """A crosses PCIe exactly once whatever the tiling; the old y only when beta != 0"""
    if block_bytes is None:
        monkeypatch.delenv("BOF_GEMV_BLOCK_BYTES", raising=False)
    else:
        monkeypatch.setenv("BOF_GEMV_BLOCK_BYTES", str(block_bytes))
    for ord_, trans in LAYOUTS:
        m, n = 1000, 3000
        A, x, y0 = problem(m, n, trans, seed=1, beta=beta)
        host_run(ctx, ord_, trans, m, n, 1.0, beta, A, x, y0, pad=2)
        st = ctx.stats()
        xl, yl = lens(trans, m, n)
        assert st.h2d_bytes == 4 * (m * n + xl + (yl if beta != 0 else 0)), (ord_, trans)
        assert st.d2h_bytes == 4 * yl
        assert st.kernel_launches >= 1


def test_bad_arguments(bof, ctx):
    A = np.ones((4, 5), np.float32)
    x = np.ones(5, np.float32)
    y = np.zeros(4, np.float32)
    bad = [dict(ord_="X", trans="N", m=4, n=5, lda=0), dict(ord_="R", trans="Q", m=4, n=5, lda=0),
           dict(ord_="R", trans="N", m=-1, n=5, lda=0), dict(ord_="R", trans="N", m=4, n=5, lda=4),
           dict(ord_="C", trans="N", m=4, n=5, lda=3)]
    for b in bad:
        with pytest.raises(bof.BofError) as ei:
            ctx.host_gemv(b["ord_"], b["trans"], b["m"], b["n"], 1.0, 0.0, A, x, y, lda=b["lda"])
        assert ei.value.code == -1 and "gemv" in str(ei.value)
        with pytest.raises(bof.BofError) as ei:
            ctx.sgemv(b["ord_"], b["trans"], b["m"], b["n"], 1.0, torch.ones(20, device="cuda"), b["lda"],
                      torch.ones(5, device="cuda"), 0.0, torch.zeros(5, device="cuda"), ws=torch.empty(1 << 16, dtype=torch.uint8, device="cuda"))
        assert ei.value.code == -1
    with pytest.raises(bof.BofError) as ei:   # workspace too small
        ctx.sgemv("R", "N", 4, 5, 1.0, torch.ones(20, device="cuda"), 0, torch.ones(5, device="cuda"), 0.0,
                  torch.zeros(4, device="cuda"), ws=torch.empty(0, dtype=torch.uint8, device="cuda"))
    assert ei.value.code == -1 and "workspace" in str(ei.value)
    ctx.host_gemv("R", "N", 4, 5, 2.0, 0.0, A, x, y)   # the context still works
    assert np.array_equal(y, np.full(4, 10.0, np.float32))


@pytest.mark.parametrize("ord_,trans", [("R", "N"), ("C", "N"), ("R", "T")])
def test_driver_on_files(ctx, tmp_path, ord_, trans):
    import __graft_entry__ as g
    if not (ROOT / "build" / "gemv").exists():
        g.build()
    m, n, pad, alpha, beta = 1300, 2100, 5, 0.5, 1.5
    A, x, y0 = problem(m, n, trans, seed=21, beta=beta)
    buf, lda = stored(A, ord_, pad)
    buf.tofile(tmp_path / "A.bin"); x.tofile(tmp_path / "x.bin"); y0.tofile(tmp_path / "y.bin")
    r = subprocess.run([str(ROOT / "build" / "gemv"), tmp_path / "A.bin", tmp_path / "x.bin", tmp_path / "y.bin", str(m),
                        str(n), str(alpha), str(beta), trans, ord_, str(lda)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "returned 0" in r.stdout, r.stdout + r.stderr
    want = host_run(ctx, ord_, trans, m, n, alpha, beta, A, x, y0, pad=pad)
    assert (tmp_path / "y.bin").read_bytes() == want.tobytes()
