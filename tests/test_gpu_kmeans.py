"""GPU parity: k-means distance/argmin (fused 3xTF32 GEMM epilogue), centroid reduce, Lloyd iteration."""
from pathlib import Path

import numpy as np
import pytest
import torch

import oracle
from gpu_util import dev

pytestmark = pytest.mark.gpu
TOL = 1e-5
G = np.load(Path(__file__).parent / "golden" / "golden_small.npz")


def mixture(rng, P, K, d, sigma=0.05, spread=4.0):
    cent = (rng.normal(size=(K, d)) * spread).astype(np.float32)
    pts = (cent[rng.integers(0, K, P)] + sigma * rng.normal(size=(P, d))).astype(np.float32)
    return pts, cent


def gpu_assign(ctx, pts, cent):
    P, d = pts.shape
    K = cent.shape[0]
    pd, cd = dev(pts), dev(cent)
    p2 = torch.empty(P, device="cuda"); c2 = torch.empty(K, device="cuda")
    ctx.row_sqnorm(P, d, pd, d, p2)
    ctx.row_sqnorm(K, d, cd, d, c2)
    out = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    ctx.kmeans_assign(P, K, d, pd, cd, c2, p2, out)
    return out.cpu().numpy().astype(np.int64), p2.cpu().numpy(), c2.cpu().numpy()


@pytest.mark.parametrize("P,K,d", [(1000, 7, 16), (5000, 1024, 256), (777, 300, 100), (130, 1000, 33), (4096, 256, 64)])
def test_assign_bit_exact_on_ties_free_points(ctx, P, K, d):
    rng = np.random.default_rng(P + K + d)
    pts, cent = mixture(rng, P, K, d)
    got, p2, c2 = gpu_assign(ctx, pts, cent)
    assert oracle.rel_fro(p2, oracle.row_sqnorm(pts)) <= TOL and oracle.rel_fro(c2, oracle.row_sqnorm(cent)) <= TOL
    ref, margin = oracle.kmeans_assign(pts, cent)
    ok = margin > 1e-3 * (1 + np.abs(p2))  # ties-free: top-2 gap well above fp32 rounding of the distances
    assert ok.mean() > 0.95
    assert np.array_equal(got[ok], ref[ok]), f"{(got[ok] != ref[ok]).sum()} mismatches on ties-free points"
    assert got.min() >= 0 and got.max() < K


def test_assign_hybrid_split_mode(bof):
    """Same bit-exact-on-ties-free contract with the hybrid operand split (gemm_split=2)."""
    rng = np.random.default_rng(77)
    pts, cent = mixture(rng, 6000, 512, 128)
    with bof.Context(device=0, gemm_split=2) as c2:
        got, p2, _ = gpu_assign(c2, pts, cent)
    ref, margin = oracle.kmeans_assign(pts, cent)
    ok = margin > 1e-3 * (1 + np.abs(p2))
    assert ok.mean() > 0.95 and np.array_equal(got[ok], ref[ok])


def test_assign_golden(ctx):
    pts, cent = G["km_points"], G["km_centers"]
    got, _, _ = gpu_assign(ctx, pts, cent)
    _, margin = oracle.kmeans_assign(pts, cent)
    ok = margin > 1e-3
    assert np.array_equal(got[ok], G["km_assign"][ok])


def test_assign_isamin_semantics(bof):
    """first index of the minimum ABSOLUTE value (cblas_isamin, drivers/in_mem_kmeans.cpp:84-85), on both cluster
    shapes (force_path 0: cta_group=2, 256-column N tiles; 1: cta_group=1, 128-column N tiles) and with a chunked dim
    (300 > 256: CHUNKED=true).  Exact ties in integer arithmetic, placed inside one epilogue column half, across
    the two halves of a tile and across N tiles; the tie in the chunked case sits in the second k chunk."""
    for force_path, d in ((0, 8), (1, 8), (0, 300), (1, 300)):
        with bof.Context(device=0, gemm_force_path=force_path) as c:
            check_isamin_ties(c, force_path, d)


def check_isamin_ties(c, force_path, d):
    pts = np.zeros((128, d), np.float32)
    cent = np.zeros((300, d), np.float32)
    cent[:, 0] = 1.0
    cent[200, 0] = 0.5; cent[260, 0] = 0.5  # two equal minima -> first one wins
    got, _, _ = gpu_assign(c, pts, cent)
    assert np.all(got == 200), (force_path, d)
    cent[:, 0] = 1.0  # all tie -> index 0
    got, _, _ = gpu_assign(c, pts, cent)
    assert np.all(got == 0), (force_path, d)
    # points = v (small integers, nonzero dot products); centers v + 2 e_j at squared distance 4, two of them
    # v + e_a, v + e_b at distance 1: the tie must go to the lower index
    rng = np.random.default_rng(d)
    v = rng.integers(0, 4, d).astype(np.float32)
    pts = np.tile(v, (128, 1))
    cent = np.tile(v, (300, 1))
    cent[np.arange(300), np.arange(300) % d] += 2.0
    a = d - 1  # for d = 300 in the last k-block of the second chunk
    for i, j in ((30, 70), (100, 140), (120, 136), (200, 260)):  # halves of tile 0 (cg 1 / cg 2), across tiles
        cent[i] = v; cent[j] = v
        cent[i, a] += 1.0; cent[j, (a - 1) % d] -= 1.0 if v[(a - 1) % d] > 0 else -1.0
        got, _, _ = gpu_assign(c, pts, cent)
        assert np.all(got == i), (force_path, d, i, j, np.unique(got))
        cent[i] = v; cent[j] = v
        cent[i, i % d] += 2.0; cent[j, j % d] += 2.0


def test_reduce_and_finalize(ctx):
    rng = np.random.default_rng(5)
    P, K, d = 20000, 100, 48
    pts = rng.normal(size=(P, d)).astype(np.float32)
    assign = rng.integers(0, K, P).astype(np.int32)
    assign[assign == 7] = 8  # an empty cluster
    pd, ad = dev(pts), dev(assign)
    sums = torch.empty((K, d), device="cuda"); counts = torch.empty(K, device="cuda")
    ctx.kmeans_reduce(P, K, d, pd, ad, sums, counts)
    ref_c, ref_n = oracle.kmeans_update(pts, assign.astype(np.int64), K, mode=1)
    assert np.array_equal(counts.cpu().numpy().astype(np.int64), ref_n)
    # deterministic: same bits on a second run
    sums2 = torch.empty_like(sums); counts2 = torch.empty_like(counts)
    ctx.kmeans_reduce(P, K, d, pd, ad, sums2, counts2)
    assert torch.equal(sums, sums2)
    cent = torch.empty((K, d), device="cuda"); c2 = torch.empty(K, device="cuda")
    ctx.kmeans_finalize(K, d, sums, counts, cent, c2)
    got = cent.cpu().numpy()
    assert np.all(got[7] == 0)  # empty cluster => zero vector (in_mem_kmeans.cpp:112)
    assert oracle.rel_fro(got, ref_c) <= TOL
    assert oracle.rel_fro(got, oracle.kmeans_update(pts, assign.astype(np.int64), K, mode=0)[0]) <= TOL  # reference order
    assert oracle.rel_fro(c2.cpu().numpy(), oracle.row_sqnorm(got)) <= TOL


def test_lloyd_iterations_teacher_forced(bof, ctx):
    """Each iteration starts from the oracle's centroids of the previous one (SURVEY.md section 7, hard parts)."""
    rng = np.random.default_rng(6)
    P, K, d = 30000, 64, 32
    pts, cent_true = mixture(rng, P, K, d, sigma=0.3)
    cent = pts[:K].copy()
    for it in range(3):
        km = bof.KMeans(ctx, P, K, d, pts, cent)
        km.local_step()
        km.update()
        got_c = np.zeros((K, d), np.float32); got_a = np.zeros(P, np.int64)
        km.get(got_c, got_a)
        km.close()
        ref_c, ref_a, _ = oracle.lloyd_iter(pts, cent)
        _, margin = oracle.kmeans_assign(pts, cent)
        ok = margin > 1e-3 * (1 + np.einsum("ij,ij->i", pts, pts))
        assert np.array_equal(got_a[ok], ref_a[ok])
        if ok.all():
            assert oracle.rel_fro(got_c, ref_c) <= TOL
        cent = ref_c


@pytest.mark.parametrize("ord_", ["C", "R"])
def test_distance_tile_flash_kmeans(ctx, ord_):
    """flash::kmeans / KMeansTask::execute (include/tasks/kmeans_task.h:68-80): D = -2 mu^T X, then += c_l2sq[i],
    then += p_l2sq[j].  'C' is the reference's own call form ('C','T','N', ncenters, npoints, dim, -2, 0, centers,
    points, dist; drivers/kmeans.cpp:36-38); the rank-1 terms are added on the device, fp32, in that order."""
    rng = np.random.default_rng(31)
    K, P, d = 70, 5000, 48
    cent = rng.normal(size=(K, d)).astype(np.float32)
    pts = rng.normal(size=(P, d)).astype(np.float32)
    c2 = oracle.row_sqnorm(cent); p2 = oracle.row_sqnorm(pts)
    if ord_ == "C":
        # column-major: op(A) = centers^T^T ... A is d x K col-major = centers row-major; C is K x P col-major
        D = np.full(K * P, np.nan, np.float32)
        ctx.host_kmeans_dist("C", "T", "N", K, P, d, -2.0, 0.0, cent, pts, D, c2, p2, lda=d, ldb=d, ldc=K)
        got = D.reshape(P, K).T                      # D(i, j) at j*K + i
        prod = oracle.gemm("C", "T", "N", K, P, d, -2.0, 0.0, cent, pts, np.zeros(K * P, np.float32), d, d, K,
                           acc64=True).reshape(P, K).T
    else:
        D = np.full((K, P), np.nan, np.float32)
        ctx.host_kmeans_dist("R", "N", "T", K, P, d, -2.0, 0.0, cent, pts, D, c2, p2)
        got = D
        prod = oracle.gemm("R", "N", "T", K, P, d, -2.0, 0.0, cent, pts, np.zeros((K, P), np.float32), acc64=True)
    ref = (prod + c2[:, None]) + p2[None, :]
    assert oracle.rel_fro(got, ref) <= 1e-5
    # the argmin over centers of the tile reproduces the oracle's assignment (isamin semantics on ties-free data)
    a_ref, margin = oracle.kmeans_assign(pts, cent, c2, p2)
    clear = margin > 1e-3                       # top-2 gap well above fp32 rounding of the distances
    assert clear.mean() > 0.9
    assert np.array_equal(np.abs(got).argmin(axis=0)[clear], a_ref[clear])


def test_out_of_core_shard_child_process():
    """Shards larger than HBM are streamed chunk by chunk on every iteration (the reference re-reads its points from
    flash per iteration, drivers/kmeans.cpp:143-145).  BOF_KMEANS_CHUNK forces the mode at test size: 3 Lloyd
    iterations with a ragged last chunk must give the resident mode's assignments and, up to the order of the
    fp32 chunk sums, its centroids."""
    import os, subprocess, sys, textwrap
    code = textwrap.dedent('''
        import numpy as np, sys
        sys.path.insert(0, %r)
        import __graft_entry__ as g, oracle
        bof = g.load_package()
        rng = np.random.default_rng(12)
        P, K, d = 50000, 48, 40
        cent = (rng.normal(size=(K, d)) * 4).astype(np.float32)
        pts = (cent[rng.integers(0, K, P)] + 0.3 * rng.normal(size=(P, d))).astype(np.float32)
        c0 = (cent + 0.05 * rng.normal(size=(K, d))).astype(np.float32)
        with bof.Context(device=0) as ctx:
            km = bof.KMeans(ctx, P, K, d, pts, c0)
            for _ in range(3):
                km.local_step(); km.update()
            got_c = np.zeros((K, d), np.float32); got_a = np.zeros(P, np.int64)
            km.get(got_c, got_a); km.close()
        ref_c = c0
        for _ in range(3):
            prev = ref_c
            ref_c, ref_a, _ = oracle.lloyd_iter(pts, prev)
        _, margin = oracle.kmeans_assign(pts, prev)
        ok = margin > 1e-3 * (1 + np.einsum("ij,ij->i", pts, pts))
        assert ok.mean() > 0.99
        assert np.array_equal(got_a[ok], ref_a[ok])
        assert oracle.rel_fro(got_c, ref_c) <= 1e-5, oracle.rel_fro(got_c, ref_c)
        np.save(sys.argv[1], got_c)
        print("ok")
    ''' % str(Path(__file__).resolve().parent.parent))
    import tempfile
    outs = []
    with tempfile.TemporaryDirectory() as td:
        for name, chunk in (("resident", "0"), ("chunked", "7000")):
            f = os.path.join(td, name + ".npy")
            r = subprocess.run([sys.executable, "-c", code, f], env=dict(os.environ, BOF_KMEANS_CHUNK=chunk),
                               capture_output=True, text=True, timeout=300)
            assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr
            outs.append(np.load(f))
    assert oracle.rel_fro(outs[1], outs[0]) <= 2e-6
