"""GPU numerics of the tensor-core GEMM (gemm3xtf32_kernel<CG, EPI, CHUNKED, HYB>) and the fused k-means argmin,
element by element against float64 references: every kernel variant on the persistent schedule, power-of-two scale
equivariance, Inf / NaN propagation and finite inputs next to FLT_MAX.

Error measure unless a test says otherwise: |C - R| <= 2^-16 * (|A| @ |B|) for every element.  The split's error is
at most 2^-19 of each product for the cross terms plus the fp32 accumulation, so the bound leaves ~8x headroom;
dropping a cross term or a k-block of 32 breaks it.

Kernel variants: tile = (128 * CG) x BLOCK_N with BLOCK_N = 128 * CG; a launch has min(items, #SMs / CG) clusters of
CG CTAs, and each cluster walks items cluster_id, cluster_id + clusters, ... (EPI_GEMM: one item per tile, EPI_ARGMIN:
one item per M tile).  CHUNKED is selected when k_chunk / 32 < ceil(k / 32) (k_chunk = gemm_k_chunk, default 256)."""
import math

import numpy as np
import pytest
import torch

import oracle
from gpu_util import dev

pytestmark = pytest.mark.gpu

# name -> (gemm_force_path, gemm_split): tc = pure 3xTF32, hyb = TF32 hi*hi + BF16 cross terms, ffma = CUDA cores
PATHS = {"tc1": (1, 1), "tc2": (2, 1), "hyb1": (1, 2), "hyb2": (2, 2), "ffma": (3, 0)}
TC = ("tc1", "tc2", "hyb1", "hyb2")
CG = {"tc1": 1, "hyb1": 1, "tc2": 2, "hyb2": 2}
REL = 2.0 ** -16
FLT_MAX = float(np.finfo(np.float32).max)
LAYOUTS = [("R", "N", "N"), ("R", "T", "T")]  # between them each operand goes through both split kernels


@pytest.fixture(scope="module")
def ctxs(bof):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    made = {name: bof.Context(device=0, gemm_force_path=p, gemm_split=s) for name, (p, s) in PATHS.items()}
    for name, c in made.items():
        c.path = name
    yield made
    for c in made.values():
        c.close()


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def ratio_to_bound(got, ref, bound):
    """|got - ref| / bound element-wise in float64 (torch tensors on one device); 0 / 0 counts as 0."""
    err = (got.double() - ref.double()).abs()
    bound = bound.double()
    r = err / bound.clamp_min(torch.finfo(torch.float64).tiny)
    return torch.where((err == 0), torch.zeros_like(r), r)


def assert_bound(got, ref, bound, tile, what):
    """Every element within its bound; the message carries the per-tile maxima of the ratio, worst tiles first."""
    r = ratio_to_bound(got, ref, bound)
    worst = float(r.max())
    if worst <= 1.0:
        return worst
    M, N = r.shape
    tm, tn = -(-M // tile), -(-N // tile)
    pad = torch.zeros((tm * tile, tn * tile), dtype=r.dtype, device=r.device)
    pad[:M, :N] = r
    per_tile = pad.reshape(tm, tile, tn, tile).amax(dim=(1, 3)).cpu()
    bad = [(float(per_tile[i, j]), i, j) for i in range(tm) for j in range(tn) if per_tile[i, j] > 1.0]
    bad.sort(reverse=True)
    i, j = np.unravel_index(int(r.argmax()), r.shape)
    pytest.fail(f"{what}: max |C-R|/(2^-16 |A||B|) = {worst:.3g} at ({i}, {j}), got {float(got[i, j])!r} ref "
                f"{float(ref[i, j])!r}; {len(bad)} of {tm * tn} tiles ({tile}x{tile}) over the bound, worst "
                f"(ratio, tile_m, tile_n): {[(round(b[0], 2), b[1], b[2]) for b in bad[:8]]}")


def store(X, trans):
    """Row-major storage of X ('N') or of X^T ('T')."""
    return np.ascontiguousarray(X.T if trans == "T" else X)


def gemm_dev(c, lay, A, B, alpha=1.0, beta=0.0, C0=None):
    """C = alpha op(A) op(B) + beta C0 through bof_sgemm_f32, op(A) = A, op(B) = B logically (host arrays)."""
    ord_, ta, tb = lay
    M, K = A.shape
    N = B.shape[1]
    Cd = dev(C0) if C0 is not None else torch.empty((M, N), device="cuda")
    c.sgemm(ord_, ta, tb, M, N, K, alpha, dev(store(A, ta)), 0, dev(store(B, tb)), 0, beta, Cd, 0)
    return Cd.cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------
# (a) variant matrix, GEMM epilogue, persistent schedule
# ---------------------------------------------------------------------------------------------------------------
def persistent_shape(cg):
    """Ragged M x N with at least 2 * clusters + 1 tiles: every cluster takes two or three items, so the item loop
    and the TMEM double-buffer hand-over between items run."""
    clusters = num_sms() // cg
    tile = 128 * cg
    tiles = 2 * clusters + 1
    tm = math.isqrt(tiles - 1) + 1
    tn = -(-tiles // tm)
    return (tm - 1) * tile + 37, (tn - 1) * tile + 77, clusters, tm * tn


# case -> (K, gemm_k_chunk): 7 k-blocks in one chunk (CHUNKED=false); 35 k-blocks in chunks of 8, 8, 8, 8, 3
# (CHUNKED=true); 35 k-blocks accumulated whole in TMEM (gemm_k_chunk=-1, CHUNKED=false)
K_CASES = {"k200": (200, 0), "k1100_chunked": (1100, 0), "k1100_whole": (1100, -1)}


@pytest.mark.parametrize("case", list(K_CASES))
@pytest.mark.parametrize("path", TC)
def test_gemm_variants_persistent(bof, path, case):
    """EPI_GEMM on all eight <CG, CHUNKED, HYB> instantiations: tc1 / hyb1 run CG=1 (128 x 128 tiles, #SMs clusters;
    148 SMs: M x N = 2213 x 2125 = 18 x 17 = 306 tiles >= 297), tc2 / hyb2 run CG=2 (256 x 256 tiles, #SMs / 2
    clusters; 3109 x 2893 = 13 x 12 = 156 tiles >= 149).  M is not a multiple of the tile, N not of BLOCK_N, K not
    of 32.  k200 / k1100_whole select CHUNKED=false, k1100_chunked CHUNKED=true (5 chunks, the last one short).
    Mixed-sign N(0,1) data; a second call with beta != 0 writes into a padded ldc whose padding must stay intact."""
    fp, split = PATHS[path]
    K, k_chunk = K_CASES[case]
    M, N, clusters, tiles = persistent_shape(CG[path])
    assert tiles >= 2 * clusters + 1
    g = torch.Generator(device="cuda").manual_seed(K + 7 * CG[path] + split)
    A = torch.randn((M, K), device="cuda", generator=g)
    B = torch.randn((K, N), device="cuda", generator=g)
    C0 = torch.randn((M, N), device="cuda", generator=g)
    ref = A.double() @ B.double()
    absab = A.double().abs() @ B.double().abs()
    with bof.Context(device=0, gemm_force_path=fp, gemm_split=split, gemm_k_chunk=k_chunk) as c:
        ws = c.sgemm_workspace(M, N, K)
        C = torch.full((M, N), float("nan"), device="cuda")  # beta == 0: C is not read
        c.sgemm("R", "N", "N", M, N, K, 1.0, A, 0, B, 0, 0.0, C, 0, ws=ws)
        torch.cuda.synchronize()
        assert_bound(C, ref, REL * absab, 128 * CG[path], f"{path} {case} beta=0")
        ldc = N + 5
        Cp = torch.full((M, ldc), -12345.0, device="cuda")
        Cp[:, :N] = C0
        alpha, beta = -0.75, 1.5
        c.sgemm("R", "N", "N", M, N, K, alpha, A, 0, B, 0, beta, Cp, ldc, ws=ws)
        torch.cuda.synchronize()
    ref2 = alpha * ref + beta * C0.double()
    bound2 = REL * (abs(alpha) * absab + abs(beta) * C0.double().abs())
    assert_bound(Cp[:, :N], ref2, bound2, 128 * CG[path], f"{path} {case} beta={beta} ldc={ldc}")
    assert bool((Cp[:, N:] == -12345.0).all()), "padding columns of C were written"


# ---------------------------------------------------------------------------------------------------------------
# (b) variant matrix, argmin epilogue
# ---------------------------------------------------------------------------------------------------------------
_ASSIGN_REF = {}


def mixture(rng, P, K, d, sigma=0.05, spread=4.0):
    cent = (rng.normal(size=(K, d)) * spread).astype(np.float32)
    pts = (cent[rng.integers(0, K, P)] + sigma * rng.normal(size=(P, d))).astype(np.float32)
    return pts, cent


def assign_case(c, d):
    """Points (128 * #SMs + 77 of them: tiles_m > clusters for CG = 1 and 2), 1000 centers, the device norms and the
    oracle's float64-dot assignment on a row subset (every point up to dim 1000), cached per dim."""
    if d not in _ASSIGN_REF:
        P, K = 128 * num_sms() + 77, 1000
        rng = np.random.default_rng(1000 + d)
        pts, cent = mixture(rng, P, K, d)
        pd, cd = dev(pts), dev(cent)
        p2 = torch.empty(P, device="cuda"); c2 = torch.empty(K, device="cuda")
        c.row_sqnorm(P, d, pd, d, p2)
        c.row_sqnorm(K, d, cd, d, c2)
        p2h, c2h = p2.cpu().numpy(), c2.cpu().numpy()
        sel = np.arange(P) if d <= 1000 else np.unique(np.r_[0:P:4, P - 256:P])
        ref, margin = oracle.kmeans_assign(pts[sel], cent, c2h, p2h[sel], acc64=True)
        _ASSIGN_REF.clear()  # keep one dim resident at a time
        _ASSIGN_REF[d] = (pd, cd, p2, c2, sel, ref, margin, p2h)
    return _ASSIGN_REF[d]


@pytest.mark.parametrize("path", TC)
@pytest.mark.parametrize("d", [8, 256, 257, 1000, 4096])
def test_assign_variants(ctxs, path, d):
    """EPI_ARGMIN on all eight <CG, CHUNKED, HYB> instantiations: tc1 / hyb1 (gemm_force_path=1) run CG=1 with
    tiles_m = ceil(P / 128) = #SMs + 1 items over #SMs clusters; tc2 / hyb2 run CG=2 (the default shape) with
    ceil(P / 256) = #SMs / 2 + 1 items over #SMs / 2 clusters.  1000 centers: a ragged last N tile (7.8 of 128,
    3.9 of 256).  dim 8 and 256 fit one chunk of 256 (CHUNKED=false); 257 (2 chunks), 1000 (4) and 4096 (16) run
    CHUNKED=true.  Bit-exact against the float64-dot oracle on ties-free points."""
    c = ctxs[path]
    pd, cd, p2, c2, sel, ref, margin, p2h = assign_case(c, d)
    P, K = pd.shape[0], cd.shape[0]
    assert -(-P // (128 * CG[path])) > num_sms() // CG[path]
    out = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    c.kmeans_assign(P, K, d, pd, cd, c2, p2, out)
    got = out.cpu().numpy().astype(np.int64)
    assert got.min() >= 0 and got.max() < K
    ok = margin > 1e-3 * (1 + np.abs(p2h[sel]))
    assert ok.mean() > 0.95, ok.mean()
    g = got[sel]
    bad = np.nonzero(ok & (g != ref))[0]
    assert bad.size == 0, (f"{path} d={d}: {bad.size} mismatches on ties-free points, first rows "
                           f"{sel[bad[:8]].tolist()} got {g[bad[:8]].tolist()} ref {ref[bad[:8]].tolist()}")


# ---------------------------------------------------------------------------------------------------------------
# (c) power-of-two scale equivariance
# ---------------------------------------------------------------------------------------------------------------
# Smallest exponent e = s + t at which the |A||B| bound must hold for C(2^s A, 2^t B), inputs |x| in [2^-4, 2^4].
# Measured on a B200: every path keeps the bound, with the same worst ratio, at every exponent of the sweep down to
# -110, where the smallest cross products are below 2^-126, so tcgen05 loses nothing there that the bound would see.
SCALE_FLOOR = -110


def log_uniform(rng, shape):
    """|x| in [2^-4, 2^4], random sign and mantissa."""
    x = np.exp2(rng.uniform(-4, 4, size=shape)) * rng.choice([-1.0, 1.0], size=shape)
    return x.astype(np.float32)


@pytest.mark.parametrize("lay", LAYOUTS, ids=["RNN", "RTT"])
@pytest.mark.parametrize("path", list(PATHS))
def test_gemm_scale_equivariance(ctxs, path, lay):
    """C(2^s A, 2^t B) == 2^(s+t) C(A, B) bit for bit while every plane value and partial product stays normal:
    the scaling commutes with the split, the MMAs, the fp32 folds and alpha.  K = 300 (10 k-blocks, 2 chunks:
    CHUNKED=true on the tensor-core paths); 'RNN' splits A with split_planes_kmajor_kernel and B with
    split_planes_transpose_kernel, 'RTT' the other way round.  Beyond |s + t| = 64 the exponent is pushed towards
    -110 and towards the largest finite one, where the |A||B| bound is asserted against float64 from SCALE_FLOOR
    up."""
    c = ctxs[path]
    M, N, K = 300, 260, 300
    rng = np.random.default_rng(11)
    A, B = log_uniform(rng, (M, K)), log_uniform(rng, (K, N))
    alpha = -0.75
    base = gemm_dev(c, lay, A, B, alpha)
    for s in (-64, -32, 0, 32, 64):
        for t in (-64, -32, 0, 32, 64):
            if abs(s + t) > 64:
                continue
            got = gemm_dev(c, lay, np.ldexp(A, s), np.ldexp(B, t), alpha)
            want = np.ldexp(base, s + t)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), \
                (path, lay, s, t, int((got != want).sum()))

    A64, B64 = A.astype(np.float64), B.astype(np.float64)
    ref, absab = alpha * (A64 @ B64), abs(alpha) * (np.abs(A64) @ np.abs(B64))
    e_max = 126 - math.ceil(math.log2(absab.max()))
    holds = {}
    for e in [-72, -80, -88, -96, -100, -102, -104, -106, -108, -110, 72, 80, 88, 96, 104, e_max]:
        s = e // 2
        got = gemm_dev(c, lay, np.ldexp(A, s), np.ldexp(B, e - s), alpha)
        assert np.all(np.isfinite(got)), (path, lay, e)
        r = ratio_to_bound(torch.from_numpy(got), torch.from_numpy(np.ldexp(ref, e)),
                           torch.from_numpy(REL * np.ldexp(absab, e)))
        holds[e] = float(r.max())
    down = sorted(e for e in holds if e < 0)
    floor = max(down) + 1
    for e in sorted(down, reverse=True):
        if holds[e] > 1.0:
            break
        floor = e
    print(f"{path} {''.join(lay)}: |A||B| bound holds down to s+t = {floor}; max ratio per exponent "
          + ", ".join(f"{e}: {holds[e]:.3g}" for e in sorted(holds)))
    over = {e: holds[e] for e in holds if e >= SCALE_FLOOR and holds[e] > 1.0}
    assert not over, f"{path} {lay}: bound fails at exponents {over} (floor {SCALE_FLOOR})"


# ---------------------------------------------------------------------------------------------------------------
# (d) Inf / NaN propagation
# ---------------------------------------------------------------------------------------------------------------
def special_case():
    """A with +Inf, -Inf and NaN in separate rows and +Inf with -Inf in one row; B strictly positive and tf32-exact
    (1.0, 3.0) in the k rows those values meet, one +Inf in column J0; C0 with an Inf and a NaN (beta != 0)."""
    M, N, K = 200, 150, 300
    rng = np.random.default_rng(5)
    A = rng.normal(size=(M, K)).astype(np.float32)
    B = rng.normal(size=(K, N)).astype(np.float32)
    C0 = rng.normal(size=(M, N)).astype(np.float32)
    A0, B0, C00 = A.copy(), B.copy(), C0.copy()
    rows = {3: [(10, np.inf)], 17: [(45, -np.inf)], 40: [(130, np.nan)], 77: [(200, np.inf), (290, -np.inf)]}
    for r, hits in rows.items():
        for k, v in hits:
            A[r, k] = v
            A0[r, k] = 0.0
            B[k, :] = B0[k, :] = 1.0 if k % 2 == 0 else 3.0
    J0, K0 = 99, 260
    A[:, K0] = A0[:, K0] = np.where(np.abs(A[:, K0]) < 0.5, 0.5, A[:, K0])  # a finite non-zero partner for B's Inf
    B[K0, J0] = np.inf
    B0[K0, J0] = 0.0
    cspec = {(5, 7): np.inf, (9, 11): np.nan}
    for (i, j), v in cspec.items():
        C0[i, j] = v
        C00[i, j] = 0.0
    touched = np.zeros((M, N), bool)
    touched[list(rows)] = True
    touched[:, J0] = True
    for i, j in cspec:
        touched[i, j] = True
    return A, B, C0, A0, B0, C00, touched


def check_special(path, got, got0, A, B, C0, A0, B0, C00, touched, alpha, beta, what):
    ref = alpha * np.einsum("ik,kj->ij", A.astype(np.float64), B.astype(np.float64), optimize=False) \
        + beta * C0.astype(np.float64)
    cls = lambda x: np.select([np.isnan(x), np.isposinf(x), np.isneginf(x)], [1, 2, 3], 0)
    cg, cr = cls(got), cls(ref)
    if path in ("tc1", "tc2"):
        # gemm_split = 1: hi*lo of an infinite operand and a tf32-exact partner is Inf * 0, so an infinite input may
        # turn its own row and column into NaN -- but never into a finite number
        assert np.array_equal(cg != 0, cr != 0), (what, np.argwhere((cg != 0) != (cr != 0))[:8].tolist())
    else:
        assert np.array_equal(cg, cr), (what, [(i, j, got[i, j], ref[i, j]) for i, j in np.argwhere(cg != cr)[:8]])
    fin = cr == 0
    bound = REL * (abs(alpha) * (np.abs(A0.astype(np.float64)) @ np.abs(B0.astype(np.float64)))
                   + abs(beta) * np.abs(C00.astype(np.float64)))
    err = np.abs(got[fin].astype(np.float64) - ref[fin])
    assert np.all(err <= bound[fin]), (what, float((err / bound[fin]).max()))
    # isolation: an element that meets no special value is the same bits as with the specials replaced by 0
    iso = ~touched
    assert np.array_equal(got[iso].view(np.uint32), got0[iso].view(np.uint32)), \
        (what, int((got[iso] != got0[iso]).sum()))


@pytest.mark.parametrize("lay", LAYOUTS + ["host"], ids=["RNN", "RTT", "host"])
@pytest.mark.parametrize("path", list(PATHS))
def test_gemm_nonfinite_propagation(ctxs, path, lay):
    """IEEE classes of C (NaN, +Inf, -Inf) equal those of a float64 per-element dot (no BLAS, no skipped zeros) on
    the hybrid and CUDA-core paths; on gemm_split=1 a non-finite reference stays non-finite.  K = 300 (CHUNKED on
    the tensor-core paths); 'RNN' / 'RTT' put the special values through both split kernels on both operands,
    'host' goes through bof_host_gemm."""
    c = ctxs[path]
    A, B, C0, A0, B0, C00, touched = special_case()
    alpha, beta = 1.25, 0.5
    M, K = A.shape
    N = B.shape[1]
    if lay == "host":
        got, got0 = C0.copy(), C00.copy()
        c.host_gemm("R", "N", "N", M, N, K, alpha, beta, A, B, got)
        c.host_gemm("R", "N", "N", M, N, K, alpha, beta, A0, B0, got0)
    else:
        got = gemm_dev(c, lay, A, B, alpha, beta, C0)
        got0 = gemm_dev(c, lay, A0, B0, alpha, beta, C00)
    check_special(path, got, got0, A, B, C0, A0, B0, C00, touched, alpha, beta, f"{path} {lay}")


# ---------------------------------------------------------------------------------------------------------------
# (e) finite inputs next to FLT_MAX
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lay", LAYOUTS, ids=["RNN", "RTT"])
@pytest.mark.parametrize("path", list(PATHS))
def test_gemm_near_overflow_inputs(ctxs, path, lay):
    """|A| in {FLT_MAX, 3.402e38, 3.3962e38, 3.39e38, 2^127}: rna_tf32 rounds the first two up to Inf, bf16 rounds
    the first three up to Inf.  |B| ~ 2^-100, so every product (~2^27) and every result is an ordinary finite number
    and must meet the |A||B| bound.  K = 300 (CHUNKED on the tensor-core paths)."""
    c = ctxs[path]
    M, N, K = 160, 136, 300
    rng = np.random.default_rng(9)
    mags = np.array([FLT_MAX, 3.402e38, 3.3962e38, 3.39e38, 2.0 ** 127], np.float32)
    A = (mags[rng.integers(0, mags.size, (M, K))] * rng.choice(np.float32([-1, 1]), (M, K))).astype(np.float32)
    B = np.ldexp(rng.uniform(1, 2, (K, N)) * rng.choice([-1.0, 1.0], (K, N)), -101).astype(np.float32)
    got = gemm_dev(c, lay, A, B)
    A64, B64 = A.astype(np.float64), B.astype(np.float64)
    assert np.all(np.isfinite(got)), (path, lay, int((~np.isfinite(got)).sum()))
    assert_bound(torch.from_numpy(got), torch.from_numpy(A64 @ B64), torch.from_numpy(REL * (np.abs(A64) @ np.abs(B64))),
                 128, f"{path} {lay}")


# ---------------------------------------------------------------------------------------------------------------
# (f) k-means scale equivariance
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", TC)
@pytest.mark.parametrize("d", [100, 600])
def test_kmeans_scale_equivariance(ctxs, path, d):
    """row_sqnorm(2^s X) == 2^(2s) row_sqnorm(X) bit for bit, and assign(2^s P, 2^s C) == assign(P, C) for every
    point (ties included), s in {-40, -20, 20, 40}.  tc1 / hyb1 run CG=1, tc2 / hyb2 CG=2; dim 100 is one chunk,
    dim 600 three (CHUNKED=true).  |x| >= 2^-6, so every plane value and product stays normal at s = -40."""
    c = ctxs[path]
    P, K = 3000, 300
    rng = np.random.default_rng(d)
    pts, cent = mixture(rng, P, K, d, sigma=0.5, spread=1.0)
    pts = np.where(np.abs(pts) < 2.0 ** -6, np.copysign(np.float32(2.0 ** -6), pts), pts).astype(np.float32)
    cent = np.where(np.abs(cent) < 2.0 ** -6, np.copysign(np.float32(2.0 ** -6), cent), cent).astype(np.float32)

    def run(s):
        pd, cd = dev(np.ldexp(pts, s)), dev(np.ldexp(cent, s))
        p2 = torch.empty(P, device="cuda"); c2 = torch.empty(K, device="cuda")
        c.row_sqnorm(P, d, pd, d, p2)
        c.row_sqnorm(K, d, cd, d, c2)
        out = torch.full((P,), -1, dtype=torch.int32, device="cuda")
        c.kmeans_assign(P, K, d, pd, cd, c2, p2, out)
        return p2.cpu().numpy(), c2.cpu().numpy(), out.cpu().numpy()

    p2, c2, a = run(0)
    for s in (-40, -20, 20, 40):
        p2s, c2s, a_s = run(s)
        assert np.array_equal(p2s.view(np.uint32), np.ldexp(p2, 2 * s).view(np.uint32)), (path, d, s)
        assert np.array_equal(c2s.view(np.uint32), np.ldexp(c2, 2 * s).view(np.uint32)), (path, d, s)
        assert np.array_equal(a_s, a), (path, d, s, int((a_s != a).sum()))
