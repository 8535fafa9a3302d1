"""flash::gemm on operands larger than the device: the out-of-core plan of bof_host_gemm / bof_host_kmeans_dist.

BOF_GEMM_HBM_BUDGET=<bytes> stands in for the device memory, so the plan runs at test size.  The plan cuts C into
super-blocks of S rows and k into panels of L elements (a multiple of the fold chunk); each panel's launch resumes the
fp32 fold the previous panel stored, so the result must be the same bits as the resident plan's whatever the budget.
Its device footprint, which the budgets below are computed from, is

    S*No*4 (fold) [+ S*No*4 (C0) if beta != 0] + 2 * (No*L*4 + 2 planes of No x L) + 5 * (rb*L*4 + 2 planes of rb x L)

in canonical terms (row-major C is Mo x No = m x n; column-major C is n x m), planes rounded up to 256 bytes, and
rb = gemm_row_block = 256 here."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

PATHS = {"tc1": (1, 1), "tc2": (2, 1), "hyb1": (1, 2), "hyb2": (2, 2)}  # name -> (gemm_force_path, gemm_split)
LAYOUTS = [(o, a, b) for o in "RC" for a in "NT" for b in "NT"]
M, N, K = 700, 520, 1000   # ragged against every tile, K neither a multiple of 32 nor of the 256 chunk
RB = 256
RING = 5
REL = 2.0 ** -16


def planes(rows, L):
    return -(-rows * L * 4 // 256) * 256


def ooc_bytes(S, No, L, beta):
    return S * No * 4 * (2 if beta else 1) + 2 * (No * L * 4 + 2 * planes(No, L)) + RING * (RB * L * 4 + 2 * planes(RB, L))


def canon(ord_):
    return (M, N) if ord_ == "R" else (N, M)


def budget_panels(ord_, beta, L=256):
    """One super-block (the fold of the whole C fits), k-panels of L."""
    Mo, No = canon(ord_)
    return ooc_bytes(Mo, No, L, beta)


def budget_super(ord_, beta, unit=256):
    """Super-blocks of 256 rows, k-panels of one chunk: the smallest plan there is."""
    _, No = canon(ord_)
    return ooc_bytes(256, No, unit, beta)


@pytest.fixture(scope="module")
def ctxs(bof):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    made = {name: bof.Context(device=0, gemm_force_path=p, gemm_split=s, gemm_row_block=RB) for name, (p, s) in PATHS.items()}
    yield made
    for c in made.values():
        c.close()


def stored(X, trans, ord_, pad):
    """X (logical op(X)) as the caller stores it for (trans, ord_), with `pad` extra elements per leading dimension."""
    S = X.T if trans == "T" else X          # the matrix as stored, logically
    S = S if ord_ == "R" else S.T           # row-major array holding it
    out = np.full((S.shape[0], S.shape[1] + pad), 7.0, np.float32)
    out[:, :S.shape[1]] = S
    return out


def logical_c(cst, ord_, m, n):
    return cst[:, :n] if ord_ == "R" else cst[:, :m].T


def operands(seed, m=M, n=N, k=K):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((m, k), dtype=np.float32)
    B = rng.standard_normal((k, n), dtype=np.float32)
    C0 = rng.standard_normal((m, n), dtype=np.float32)
    return A, B, C0


def run(c, lay, A, B, C0, alpha, beta, pad=3, nan_c=False, kmeans=None):
    """C as stored after the call (padding included) and the call's stats."""
    ord_, ta, tb = lay
    m, k = A.shape
    n = B.shape[1]
    a, b = stored(A, ta, ord_, pad), stored(B, tb, ord_, pad)
    cst = stored(C0, "N", ord_, pad)
    if nan_c:
        cst[:, :cst.shape[1] - pad] = np.nan
    if kmeans is None:
        c.host_gemm(ord_, ta, tb, m, n, k, alpha, beta, a, b, cst, a.shape[1], b.shape[1], cst.shape[1])
    else:
        c.host_kmeans_dist(ord_, ta, tb, m, n, k, alpha, beta, a, b, cst, kmeans[0], kmeans[1], a.shape[1], b.shape[1],
                           cst.shape[1])
    return cst, c.stats()


def check_bound(got, A, B, C0, alpha, beta):
    ref = alpha * (A.astype(np.float64) @ B.astype(np.float64)) + beta * C0.astype(np.float64)
    assert oracle.rel_fro(got, ref) <= 1e-5
    bound = REL * abs(alpha) * (np.abs(A).astype(np.float64) @ np.abs(B).astype(np.float64)) + 2.0 ** -22 * np.abs(ref)
    err = np.abs(got.astype(np.float64) - ref)
    worst = float((err / np.maximum(bound, 1e-300)).max())
    assert worst <= 1.0, f"max |C-R| / bound = {worst:.3g}"


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("lay", LAYOUTS, ids=["".join(l) for l in LAYOUTS])
@pytest.mark.parametrize("beta", [0.0, -0.75])
def test_bit_identical_to_resident(ctxs, monkeypatch, lay, path, beta):
    """Several k-panels in one super-block, and super-blocks of 256 rows: the same bits as the resident plan."""
    c = ctxs[path]
    A, B, C0 = operands(11)
    alpha = 1.25
    monkeypatch.delenv("BOF_GEMM_HBM_BUDGET", raising=False)
    ref, _ = run(c, lay, A, B, C0, alpha, beta, nan_c=beta == 0.0)
    for budget in (budget_panels(lay[0], beta), budget_super(lay[0], beta)):
        monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(budget))
        got, _ = run(c, lay, A, B, C0, alpha, beta, nan_c=beta == 0.0)
        assert np.array_equal(got, ref), f"budget {budget}: differs from the resident plan"
    check_bound(logical_c(got, lay[0], M, N), A, B, C0, alpha, beta)


@pytest.mark.parametrize("k_chunk", [128, 512, 96, -1])
def test_other_chunk_sizes(bof, monkeypatch, k_chunk):
    """Panels start on fold-chunk boundaries for any gemm_k_chunk; -1 (no fold) folds at panel boundaries only."""
    A, B, C0 = operands(12)
    lay = ("R", "N", "T")
    unit = 32 * max(1, k_chunk // 32) if k_chunk > 0 else 32
    with bof.Context(device=0, gemm_row_block=RB, gemm_k_chunk=k_chunk) as c:
        monkeypatch.delenv("BOF_GEMM_HBM_BUDGET", raising=False)
        ref, _ = run(c, lay, A, B, C0, 1.0, 0.5)
        for budget in (budget_panels("R", True, L=unit), budget_super("R", True, unit=unit)):
            monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(budget))
            got, _ = run(c, lay, A, B, C0, 1.0, 0.5)
            if k_chunk > 0:
                assert np.array_equal(got, ref), f"gemm_k_chunk {k_chunk}, budget {budget}"
            check_bound(logical_c(got, "R", M, N), A, B, C0, 1.0, 0.5)


@pytest.mark.parametrize("path", ["tc2", "hyb2"])
def test_special_values(ctxs, monkeypatch, path):
    """Inf and NaN inputs give what the resident plan gives."""
    c = ctxs[path]
    A, B, C0 = operands(13)
    A[3, 5] = np.inf; A[400, 900] = -np.inf; A[650, 10] = np.nan
    B[7, 11] = np.inf; B[999, 500] = np.nan
    lay = ("R", "N", "N")
    monkeypatch.delenv("BOF_GEMM_HBM_BUDGET", raising=False)
    ref, _ = run(c, lay, A, B, C0, 1.0, 1.0)
    monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(budget_super("R", True)))
    got, _ = run(c, lay, A, B, C0, 1.0, 1.0)
    assert np.array_equal(got, ref, equal_nan=True)


@pytest.mark.parametrize("lay", [("R", "N", "N"), ("C", "T", "N")], ids=["RNN", "CTN"])
@pytest.mark.parametrize("beta", [0.0, 0.5])
def test_pcie_accounting(ctxs, monkeypatch, lay, beta):
    """P and C cross PCIe once; Q once per super-block."""
    c = ctxs["hyb2"]
    A, B, C0 = operands(14)
    Mo, No = canon(lay[0])
    szP, szQ, szC = Mo * K * 4, No * K * 4, M * N * 4
    monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(budget_panels(lay[0], beta)))
    _, st = run(c, lay, A, B, C0, 1.0, beta)
    assert st.h2d_bytes == szP + szQ + (szC if beta else 0)
    assert st.d2h_bytes == szC
    monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(budget_super(lay[0], beta)))
    _, st = run(c, lay, A, B, C0, 1.0, beta)
    q = st.h2d_bytes - szP - (szC if beta else 0)
    assert q % szQ == 0 and q // szQ == -(-Mo // 256) >= 2
    assert st.d2h_bytes == szC


def test_budget_too_small(ctxs, monkeypatch):
    """Below the smallest plan the call fails with BOF_ENOMEM and says what it needs; the context stays usable."""
    c = ctxs["tc2"]
    A, B, C0 = operands(15)
    lay = ("R", "N", "N")
    need = budget_super("R", False)
    monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(need - 1))
    a, b, cst = stored(A, "N", "R", 0), stored(B, "N", "R", 0), stored(C0, "N", "R", 0)
    rc = c.lib.bof_host_gemm(c.h, b"R", b"N", b"N", M, N, K, 1.0, 0.0, a.ctypes.data, b.ctypes.data, cst.ctypes.data, 0, 0, 0)
    assert rc == -3
    assert f"at least {need} bytes" in c.last_error()
    monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(need))
    got, _ = run(c, lay, A, B, C0, 1.0, 0.0)
    check_bound(logical_c(got, "R", M, N), A, B, C0, 1.0, 0.0)


def test_one_context_resident_then_out_of_core(bof, monkeypatch):
    """Resident, out-of-core, resident on one context: every result right, the first and last the same bits."""
    A, B, C0 = operands(16)
    lay = ("C", "N", "T")
    with bof.Context(device=0, gemm_row_block=RB) as c:
        outs = []
        for budget in (None, budget_super("C", True), None):
            if budget is None:
                monkeypatch.delenv("BOF_GEMM_HBM_BUDGET", raising=False)
            else:
                monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(budget))
            got, _ = run(c, lay, A, B, C0, 2.0, 0.25)
            check_bound(logical_c(got, "C", M, N), A, B, C0, 2.0, 0.25)
            outs.append(got)
        assert np.array_equal(outs[0], outs[2])
        assert np.array_equal(outs[0], outs[1])


@pytest.mark.parametrize("ord_", ["R", "C"])
def test_kmeans_dist(ctxs, monkeypatch, ord_):
    """bof_host_kmeans_dist: the outer terms are added behind the last k-panel, in the resident order."""
    c = ctxs["hyb2"]
    A, B, _ = operands(17)
    C0 = np.zeros((M, N), np.float32)
    c_l2sq = (A.astype(np.float64) ** 2).sum(1).astype(np.float32)
    p_l2sq = (B.astype(np.float64) ** 2).sum(0).astype(np.float32)
    lay = (ord_, "N", "N")
    monkeypatch.delenv("BOF_GEMM_HBM_BUDGET", raising=False)
    ref, _ = run(c, lay, A, B, C0, -2.0, 0.0, kmeans=(c_l2sq, p_l2sq))
    for budget in (budget_panels(ord_, False), budget_super(ord_, False)):
        monkeypatch.setenv("BOF_GEMM_HBM_BUDGET", str(budget + (M + N) * 4))
        got, _ = run(c, lay, A, B, C0, -2.0, 0.0, kmeans=(c_l2sq, p_l2sq))
        assert np.array_equal(got, ref)
    d = c_l2sq[:, None].astype(np.float64) + p_l2sq[None, :] - 2.0 * (A.astype(np.float64) @ B.astype(np.float64))
    assert oracle.rel_fro(logical_c(got, ord_, M, N), d) <= 1e-5


def test_gemm_driver_under_budget(bof, tmp_path):
    """flash::gemm through the reference CLI (build/gemm) writes the same file with the plan forced as without."""
    exe = ROOT / "build" / "gemm"
    if not exe.exists():
        import __graft_entry__ as g
        g.build()
    A, B, C0 = operands(18)
    A.tofile(tmp_path / "A.bin"); B.tofile(tmp_path / "B.bin")
    outs = []
    for budget in (None, budget_panels("R", True)):
        C0.tofile(tmp_path / "C.bin")
        env = {k: v for k, v in os.environ.items() if k != "BOF_GEMM_HBM_BUDGET"}
        if budget is not None:
            env["BOF_GEMM_HBM_BUDGET"] = str(budget)
        r = subprocess.run([str(exe), *map(str, (tmp_path / "A.bin", tmp_path / "B.bin", tmp_path / "C.bin", M, K, N,
                                                 1.0, 0.5, "N", "N", "R", 0, 0, 0))],
                           capture_output=True, text=True, timeout=600, env=env)
        assert r.returncode == 0 and "returned 0" in r.stdout, r.stdout + r.stderr
        outs.append(np.fromfile(tmp_path / "C.bin", dtype=np.float32))
    assert np.array_equal(outs[0], outs[1])
    check_bound(outs[1].reshape(M, N), A, B, C0, 1.0, 0.5)
