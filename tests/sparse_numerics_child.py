"""Float64 reference and element-wise error bound of the sparse kernels, shared by test_gpu_sparse_numerics.py, and
the child process that file runs for the knobs the library reads once per process:

    BOF_SPMM_VARIANT=<v> python tests/sparse_numerics_child.py variant     (or BOF_SPMM_NO_SPLIT=1)
    BOF_CSRMM_KPANEL=64 python tests/sparse_numerics_child.py kpanel

The rule of the bound is stated in test_gpu_sparse_numerics.py.  Everything is computed on the device with torch:
the reference gathers the products in float64 and adds them per output row with index_add_."""
import math
import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
U = 2.0 ** -24
MID_ROW, LONG_MIN, LONG_FACTOR = 1024, 16384, 64   # sparse.cu: kMidRow, kLongRowMin, kLongRowFactor
SHORT, BLOCK, GRID = 0, 1, 2
CLASS_NAMES = ("short", "block", "grid")


class Csr:
    """A on the device in the kernels' layout: vals f32, idx i32, offs i64 (offs[0] may be nonzero)."""

    def __init__(self, vals, idx, offs, n):
        self.vals, self.idx, self.offs, self.n = vals, idx, offs, n
        self.m = offs.numel() - 1

    @property
    def nnz(self):
        return self.vals.numel()

    @property
    def lens(self):
        return self.offs[1:] - self.offs[:-1]

    def rows(self):
        return torch.repeat_interleave(torch.arange(self.m, device=self.offs.device), self.lens)

    def host(self):
        """(a f32, ia i64 from 0, ja i64) numpy arrays for the host entry points."""
        return (self.vals.cpu().numpy().copy(), (self.offs - self.offs[0]).cpu().numpy(),
                self.idx.long().cpu().numpy())


def gen(seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return g


def signed(shape, g):
    """Mixed-sign data in [-1, 1): cancellation keeps |result| well below |A||B|, so a lost term shows."""
    return torch.rand(shape, device="cuda", generator=g) * 2 - 1


def from_lens(lens, n, g, col_hi=None):
    """Rows of the given lengths, columns uniform in [0, col_hi or n) (duplicates allowed, unsorted), values in [-1, 1)."""
    lens = torch.as_tensor(lens, dtype=torch.int64, device="cuda")
    offs = torch.zeros(lens.numel() + 1, dtype=torch.int64, device="cuda")
    offs[1:] = torch.cumsum(lens, 0)
    nnz = int(offs[-1])
    idx = torch.randint(0, col_hi or n, (nnz,), device="cuda", generator=g, dtype=torch.int32)
    return Csr(signed(nnz, g), idx, offs, n)


def short_lens(m, hi, g):
    return torch.randint(0, hi + 1, (m,), device="cuda", generator=g)


def long_rows_csr(m, n, long_lens, seed, hi=48):
    """m rows of 0..hi nonzeros, with the given long rows spread over the matrix (mean stays small, so the grid
    threshold is 16384)."""
    g = gen(seed)
    lens = short_lens(m, hi, g)
    pos = torch.randperm(m, device="cuda", generator=g)[:len(long_lens)]
    lens[pos] = torch.tensor(long_lens, device="cuda")
    return from_lens(lens, n, g)


def zipf_csr(m, n, nnz_target, seed):
    """Power-law row lengths, as tools/bench_spmm_skew.py draws them: rank r gets ~ nnz_target / (r ln m) nonzeros."""
    g = gen(seed)
    ranks = torch.randperm(m, device="cuda", generator=g) + 1
    lens = torch.clamp((nnz_target / (ranks.double() * math.log(m))).long() + 1, max=n)
    return from_lens(lens, n, g)


def unrebase(A, lead=3, shift=1_000_003):
    """The same matrix as a row-block slice of a larger one: offs[0] != 0, and vals / idx start `lead` elements into
    their allocation (not 16-byte aligned unless lead % 4 == 0).  The elements in front are NaN and must not be read."""
    v = torch.full((A.nnz + lead,), float("nan"), device="cuda")
    i = torch.zeros(A.nnz + lead, dtype=torch.int32, device="cuda")
    v[lead:] = A.vals
    i[lead:] = A.idx
    return Csr(v[lead:], i[lead:], A.offs - A.offs[0] + shift, A.n)


def permute_rows(A, perm):
    """P A: row i of the result is row perm[i] of A, nonzeros in the same order."""
    lens = A.lens[perm]
    offs = torch.zeros(A.m + 1, dtype=torch.int64, device="cuda")
    offs[1:] = torch.cumsum(lens, 0)
    new_row = torch.repeat_interleave(torch.arange(A.m, device="cuda"), lens)
    src = (A.offs[perm] - A.offs[0])[new_row] + (torch.arange(A.nnz, device="cuda") - offs[new_row])
    return Csr(A.vals[src], A.idx[src], offs, A.n)


def padded(rows, k, ld, fill, data=None, shift=0):
    """(storage, view): a rows x ld row-major buffer filled with `fill`, the first k columns set to `data`, seen as a
    rows x ld tensor that starts `shift` floats into its allocation."""
    store = torch.full((rows * ld + shift,), fill, device="cuda")
    view = store[shift:].view(rows, ld)
    if data is not None:
        view[:, :k] = data
    return store, view


def same_bits(x, y):
    return torch.equal(x.contiguous().view(torch.int32), y.contiguous().view(torch.int32))


# ---- reference and bound ------------------------------------------------------------------------------------------
def reference(vals, out_idx, in_idx, X, out_rows, k, alpha=1.0, beta=0.0, C0=None, keep=None):
    """R = alpha * sum_z vals[z] X[in_idx[z], :k] into row out_idx[z] (+ beta C0) and S = |alpha| sum |vals X| in
    float64.  X is (rows x >= k) or a vector (k = 0).  keep: mask of nonzeros R keeps (S keeps all; self-check)."""
    vec = X.dim() == 1
    R = torch.zeros((out_rows,) if vec else (out_rows, k), dtype=torch.float64, device="cuda")
    S = torch.zeros_like(R)
    step = max(1, (1 << 26) // max(k, 1))
    for z0 in range(0, vals.numel(), step):
        z1 = min(vals.numel(), z0 + step)
        a = vals[z0:z1].double()
        xi = in_idx[z0:z1].long()
        p = a * X[xi].double() if vec else a[:, None] * X[xi, :k].double()
        o = out_idx[z0:z1].long()
        S.index_add_(0, o, p.abs())
        if keep is not None:
            p, o = p[keep[z0:z1]], o[keep[z0:z1]]
        R.index_add_(0, o, p)
    R *= alpha
    S *= abs(alpha)
    BT = None
    if beta != 0.0:
        BT = (beta * C0.double()).abs()
        R += beta * C0.double()
    return R, S, BT


def spmm_reference(A, B, k, alpha=1.0, beta=0.0, C0=None, keep=None, trans=False):
    """alpha op(A) B + beta C0 with op(A) = A or A^T (trans) for the device matrix A."""
    rows = A.rows()
    if trans:
        return reference(A.vals, A.idx, rows, B, A.n, k, alpha, beta, C0, keep)
    return reference(A.vals, rows, A.idx, B, A.m, k, alpha, beta, C0, keep)


def classes(lens, split=True):
    """Row class on the row-group kernels with deferral (split) or on a kernel that sums every row in order."""
    c = torch.zeros_like(lens)
    if split:
        thr = max(LONG_MIN, LONG_FACTOR * (int(lens.sum()) // max(lens.numel(), 1)))
        c[lens > MID_ROW] = BLOCK
        c[lens > thr] = GRID
    return c


def grid_blocks():
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count   # the launcher's lgrid on a B200


def cdiv(a, b):
    return (a + b - 1) // b


def block_depth(lens):
    return 32 * cdiv(cdiv(lens, 32), 8) + 8


def grid_depth(lens, G):
    return 32 * cdiv(cdiv(lens, 32), 8 * G) + 8 + G


def spmm_depth(lens, cls):
    """Summation depth per row: nnz in order, or the block / grid split trees of spmm_long_rows_kernel."""
    d = lens.clone()
    d = torch.where(cls == BLOCK, block_depth(lens), d)
    return torch.where(cls == GRID, grid_depth(lens, grid_blocks()), d)


def pipeline_depth(lens):
    """Host pipelines: the row block that sets the mean (and so block or grid) is the pipeline's choice; a row above
    1024 nonzeros gets the larger of the two depths."""
    return torch.where(lens > MID_ROW, torch.maximum(block_depth(lens), grid_depth(lens, grid_blocks())), lens)


def bound_ratio(got, R, S, BT, depth):
    """|got - R| / bound element-wise; non-finite R must be matched exactly (NaN by NaN, Inf by the same Inf) and
    counts as 0 when it is, inf when it is not.  A finite R with a non-finite got is inf."""
    g = got.double()
    d = depth.double() if g.dim() == 1 else depth.double()[:, None]
    bound = (d + 2) * U * S
    if BT is not None:
        bound = bound + 2 * U * BT
    err = (g - R).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    fin = torch.isfinite(R)
    match = (torch.isnan(R) & torch.isnan(g)) | (g == R)
    r = torch.where(fin, r, torch.where(match, torch.zeros_like(r), torch.full_like(r, math.inf)))
    return torch.nan_to_num(r, nan=math.inf)


def bound_report(got, R, r, cls, chunk):
    worst = float(r.max())
    flat = int(r.argmax())
    at = divmod(flat, r.shape[1]) if r.dim() == 2 else (flat,)
    lines = [f"max |C - R| / bound = {worst:.3g} at {at}, got {float(got[at])!r} ref {float(R[at])!r}; "
             f"{int((r > 1).sum())} elements over"]
    rowmax = r if r.dim() == 1 else r.amax(dim=1)
    for c, name in enumerate(CLASS_NAMES):
        sel = cls == c
        if bool(sel.any()):
            lines.append(f"  {name} rows ({int(sel.sum())}): max ratio {float(rowmax[sel].max()):.3g}")
    if r.dim() == 2 and chunk:
        per = [float(r[:, j:j + chunk].max()) for j in range(0, r.shape[1], chunk)]
        lines.append(f"  per column chunk of {chunk}: " + ", ".join(f"{x:.3g}" for x in per))
    top = torch.topk(r.reshape(-1), min(8, r.numel())).indices.tolist()
    for f in top:
        e = divmod(f, r.shape[1]) if r.dim() == 2 else (f,)
        lines.append(f"  {e}: ratio {float(r[e]):.3g} got {float(got[e])!r} ref {float(R[e])!r} "
                     f"class {CLASS_NAMES[int(cls[e[0]])]}")
    return "\n".join(lines)


def assert_bound(got, ref, depth, cls, chunk, what):
    """Every element of got within the bound of the reference (R, S, BT); non-finite ones exact."""
    R, S, BT = ref
    r = bound_ratio(got, R, S, BT, depth)
    worst = float(r.max())
    if worst > 1.0:
        raise AssertionError(f"{what}: " + bound_report(got, R, r, cls, chunk))
    return worst


def chunk_of(k):
    """4 L KV columns: the column chunk one row group of the launcher's kernel covers."""
    if k <= 16:
        return 16
    if k <= 32:
        return 32
    if k <= 64:
        return 64
    return 128 if k <= 128 else 256


# ---- one SpMM case on a device path -------------------------------------------------------------------------------
def run_spmm(ctx, A, Bdata, k, *, ldb, ldc, split, b_shift=0, what=""):
    """C = A B (beta = 0, NaN-filled C) and C = 1.5 A B + 0.5 C0 through bof_spmm_csr_f32 'R' with B and C padded to
    ldb / ldc.  Checks the bound, that C's padding is untouched and returns the two results (m x k views)."""
    g = gen(k + 17)
    m, n = A.m, A.n
    _, B = padded(n, k, ldb, float("nan"), Bdata[:, :k], shift=b_shift)   # B's padding is never read
    C0 = signed((m, k), g)
    cls = classes(A.lens, split)
    depth = spmm_depth(A.lens, cls)
    outs = []
    for alpha, beta in ((1.0, 0.0), (1.5, 0.5)):
        _, C = padded(m, k, ldc, float("nan") if beta == 0 else 7.0, None if beta == 0 else C0)
        before = C[:, k:].clone()
        ctx.spmm("R", m, n, k, alpha, A.vals, A.idx, A.offs, B, ldb, beta, C, ldc)
        ref = spmm_reference(A, B, k, alpha, beta, C0)
        assert_bound(C[:, :k], ref, depth, cls, chunk_of(k), f"{what} k={k} ldb={ldb} ldc={ldc} alpha={alpha} beta={beta}")
        assert same_bits(C[:, k:], before), f"{what}: padding of C written"
        outs.append(C[:, :k].clone())
    return outs


def nonfinite_case(A, n, k, seed):
    """B with +Inf and -Inf in rows that short, block and grid rows reference (one output column sees both: NaN),
    NaN in A values and an explicit 0 against Inf.  Returns (A', B data)."""
    g = gen(seed)
    B = signed((n, k), g)
    c_pos, c_neg, j = 11, 12, min(5, k - 1)
    B[c_pos, j] = math.inf
    B[c_neg, j] = -math.inf
    B[c_neg, k - 1] = -math.inf
    vals, idx = A.vals.clone(), A.idx.clone()
    lens = A.lens
    base = A.offs - A.offs[0]
    order = torch.argsort(lens, descending=True).tolist()
    shorts = [r for r in order if 4 <= int(lens[r]) <= MID_ROW][:6]
    longs = [r for r in order if int(lens[r]) > MID_ROW][:3]
    for i, r in enumerate(shorts[:3] + longs):
        z = int(base[r])
        idx[z] = c_pos
        if i % 2 == 0:
            idx[z + 1] = c_neg            # both infinities reach this row: NaN in column j
    idx[int(base[shorts[3]]) + 2] = c_pos
    vals[int(base[shorts[3]]) + 2] = 0.0   # 0 * Inf = NaN, as in IEEE
    vals[int(base[shorts[4]]) + 1] = math.nan
    if longs:
        vals[int(base[longs[-1]]) + 100] = math.nan
    return Csr(vals, idx, A.offs, A.n), B


# ---- child modes --------------------------------------------------------------------------------------------------
def variant_lens(m, g):
    """Short rows with ragged (odd) lengths, 8-row slices longer than the TMA staging chunk (2048), the first slice
    2400 elements from an aligned start (bulk copies), and rows of 1025 and 3000 nonzeros (block) and 60000 (grid:
    the mean is ~400, so the threshold is ~25600)."""
    lens = torch.randint(0, 700, (m,), device="cuda", generator=g) | 1
    lens[:8] = 300
    lens[[40, 333, 777]] = torch.tensor([1025, 3000, 60000], device="cuda")
    return lens


def child_variant(bof):
    v = os.environ.get("BOF_SPMM_VARIANT")
    no_split = os.environ.get("BOF_SPMM_NO_SPLIT") is not None
    variant = int(v) if v is not None else -1
    ctx = bof.Context(device=0)
    m, n = 1203, 3000
    A = from_lens(variant_lens(m, gen(5)), n, gen(6))
    Bdata = signed((n, 256), gen(7))
    ref16 = None
    for lead in (0, 3):
        Al = unrebase(A, lead)
        _, B16 = padded(n, 16, 20, float("nan"), Bdata[:, :16])
        C16 = torch.empty((m, 16), device="cuda")
        ctx.spmm("R", m, n, 16, 1.0, Al.vals, Al.idx, Al.offs, B16, 20, 0.0, C16, 16)
        ref16 = C16 if ref16 is None else ref16
        assert same_bits(C16, ref16)
        short = A.lens <= MID_ROW
        for k in (128, 256):
            tma = variant in (6, 7)
            split = not (tma or no_split)
            outs = run_spmm(ctx, Al, Bdata, k, ldb=k + 4, ldc=k + 8, split=split, what=f"variant {v} lead {lead}")
            assert same_bits(outs[0][short, :16], C16[short]), f"variant {v} k={k}: columns 0..15 differ from k=16"
            An, Bn = nonfinite_case(Al, n, k, 8)
            run_spmm(ctx, An, Bn, k, ldb=k, ldc=k + 4, split=split, what=f"variant {v} non-finite")
    ctx.close()


def child_kpanel(bof):
    """flash::csrmm in column panels (BOF_CSRMM_KPANEL=64): a long row above the nnz budget forms its own block."""
    m, n, k = 3000, 2500, 200
    A = long_rows_csr(m, n, [1025, 5000, 17000, 30000], seed=9)
    a, ia, ja = A.host()
    g = gen(10)
    B = signed((n, k), g)
    C0 = signed((m, k), g)
    depth = pipeline_depth(A.lens)
    cls = classes(A.lens)
    with bof.Context(device=0, csrmm_max_nnz=20000) as ctx:
        for alpha, beta in ((1.0, 0.0), (1.5, 0.5)):
            C = C0.cpu().numpy().copy() if beta else np.full((m, k), np.nan, np.float32)
            ctx.host_csrmm("N", m, n, k, alpha, beta, a, ia, ja, "R", B.cpu().numpy(), C)
            ref = spmm_reference(A, B, k, alpha, beta, C0)
            assert_bound(torch.from_numpy(C).cuda(), ref, depth, cls, 64, f"kpanel alpha={alpha} beta={beta}")


def main():
    sys.path.insert(0, str(ROOT))
    import __graft_entry__ as g
    bof = g.load_package()
    {"variant": child_variant, "kpanel": child_kpanel}[sys.argv[1]](bof)
    torch.cuda.synchronize()
    print("SPARSE_CHILD_OK")


if __name__ == "__main__":
    main()
