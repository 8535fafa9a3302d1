"""bof_b200 -- B200-native hot path of BLAS-on-Flash (csrmm, gemm, gemv, csrgemv, csrcsc, kmeans step).

The product is ``libbof_b200.so`` (hand-written sm_100a kernels + C ABI, ``include/bof_b200.h``)
and the C++ adapters that keep the reference's ``flash::`` signatures (``include/flash_blas.h``).
This Python package is the thin harness the tests and ``bench.py`` drive it with: it only moves
pointers.  PyTorch is used for device allocations, streams and ``torch.distributed``.

The directory name carries a hyphen (``blas-on-flash_b200``), so import it through
``__graft_entry__.load_package()`` which registers it as ``bof_b200``.
"""
from __future__ import annotations

import ctypes as C

from . import _capi
from ._capi import BofConfig, BofError, BofStats, ch, load, ptr

__all__ = ["Context", "KMeans", "ResidentCsr", "MultiGpu", "BofError", "BofStats", "load"]


def _cur_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream


class Context:
    """One per process/GPU; mirrors ``flash_setup``/``flash_destroy`` (reference src/lib_funcs.cpp:18-34)."""

    def __init__(self, device: int = 0, **cfg):
        self.lib = load()
        conf = BofConfig()
        conf.device = device
        for k, v in cfg.items():
            if not hasattr(conf, k):
                raise TypeError(f"unknown bof_config field {k!r}")
            setattr(conf, k, v)
        h = C.c_void_p()
        rc = self.lib.bof_ctx_create(C.byref(conf), C.byref(h))
        if rc != 0:
            raise BofError(rc, (self.lib.bof_last_error(None) or b"").decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.bof_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            raise BofError(rc, (self.lib.bof_last_error(self.h) or b"").decode())

    def last_error(self) -> str:
        return (self.lib.bof_last_error(self.h) or b"").decode()

    def stats(self) -> BofStats:
        s = BofStats()
        self._check(self.lib.bof_get_stats(self.h, C.byref(s)))
        return s

    def launch_count(self) -> int:
        return int(self.lib.bof_launch_count(self.h))

    def _ws(self, nbytes: int):
        import torch

        return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=f"cuda:{self.device}")

    # ---- device-tile kernels (torch CUDA tensors or raw device addresses) ----
    def spmm(self, ord_b, m, n, k, alpha, vals, idx, offs, B, ldb, beta, Cmat, ldc, stream=None):
        nb = self.lib.bof_spmm_workspace_bytes(ch(ord_b), m, n, k)
        ws = self._ws(nb) if nb else None
        self._check(self.lib.bof_spmm_csr_f32(self.h, stream or _cur_stream(), ch(ord_b), m, n, k, alpha, ptr(vals),
                                              ptr(idx), ptr(offs), ptr(B), ldb, beta, ptr(Cmat), ldc, ptr(ws), nb))

    def spmv(self, trans, m, n, vals, idx, offs, x, y, stream=None):
        self._check(self.lib.bof_spmv_csr_f32(self.h, stream or _cur_stream(), ch(trans), m, n, ptr(vals), ptr(idx),
                                              ptr(offs), ptr(x), ptr(y)))

    def idx_narrow(self, src, dst, count, stream=None):
        self._check(self.lib.bof_idx_narrow(self.h, stream or _cur_stream(), ptr(src), ptr(dst), count))

    def idx_widen(self, src, dst, count, stream=None):
        self._check(self.lib.bof_idx_widen(self.h, stream or _cur_stream(), ptr(src), ptr(dst), count))

    def sgemm_workspace(self, m, n, k):
        return self._ws(self.lib.bof_sgemm_workspace_bytes(m, n, k))

    def sgemm(self, ord_, ta, tb, m, n, k, alpha, A, lda, B, ldb, beta, Cmat, ldc, ws=None, stream=None):
        if ws is None:
            ws = self.sgemm_workspace(m, n, k)
        self._check(self.lib.bof_sgemm_f32(self.h, stream or _cur_stream(), ch(ord_), ch(ta), ch(tb), m, n, k, alpha,
                                           ptr(A), lda, ptr(B), ldb, beta, ptr(Cmat), ldc, ptr(ws), ws.numel()))

    def sgemv_workspace(self, ord_, trans, m, n):
        return self._ws(self.lib.bof_sgemv_workspace_bytes(ch(ord_), ch(trans), m, n))

    def sgemv(self, ord_, trans, m, n, alpha, A, lda, x, beta, y, ws=None, stream=None):
        """y = alpha * op(A) x + beta * y on device tensors (A stored 'R' / 'C' with leading dimension lda, 0 = tight)"""
        if ws is None:
            ws = self.sgemv_workspace(ord_, trans, m, n)
        self._check(self.lib.bof_sgemv_f32(self.h, stream or _cur_stream(), ch(ord_), ch(trans), m, n, alpha, ptr(A), lda,
                                           ptr(x), beta, ptr(y), ptr(ws), ws.numel()))

    def tc_issue_rate(self, kind: int, rounds: int = 20000, stream=None):
        """(mma_tflops, useful_tflops) of the tensor-pipe issue-rate microbenchmark; kind 0 tf32, 1 bf16, 2 hybrid mix"""
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.bof_tc_issue_rate(self.h, stream or _cur_stream(), kind, rounds, C.byref(a), C.byref(b)))
        return a.value, b.value

    def csr2csc_workspace(self, m, n, nnz):
        return self._ws(self.lib.bof_csr2csc_workspace_bytes(m, n, nnz))

    def csr2csc(self, m, n, nnz, offs, idx, vals, offs_t, idx_t, vals_t, ws=None, stream=None):
        if ws is None:
            ws = self.csr2csc_workspace(m, n, nnz)
        self._check(self.lib.bof_csr2csc(self.h, stream or _cur_stream(), m, n, nnz, ptr(offs), ptr(idx), ptr(vals),
                                         ptr(offs_t), ptr(idx_t), ptr(vals_t), ptr(ws), ws.numel()))

    def row_sqnorm(self, rows, dim, X, ldx, out, stream=None):
        self._check(self.lib.bof_row_sqnorm_f32(self.h, stream or _cur_stream(), rows, dim, ptr(X), ldx, ptr(out)))

    def kmeans_assign(self, npoints, ncenters, dim, points, centers, c_l2sq, p_l2sq, assign, planes=None, ws=None,
                      stream=None):
        if ws is None:
            ws = self._ws(self.lib.bof_kmeans_workspace_bytes(npoints, ncenters, dim, 0 if planes is not None else 1))
        self._check(self.lib.bof_kmeans_assign(self.h, stream or _cur_stream(), npoints, ncenters, dim, ptr(points),
                                               ptr(centers), ptr(c_l2sq), ptr(p_l2sq), ptr(assign), ptr(planes),
                                               ptr(ws), ws.numel()))

    def kmeans_prepare_points(self, npoints, dim, points, stream=None):
        planes = self._ws(self.lib.bof_kmeans_point_planes_bytes(npoints, dim))
        self._check(self.lib.bof_kmeans_prepare_points(self.h, stream or _cur_stream(), npoints, dim, ptr(points),
                                                       ptr(planes)))
        return planes

    def kmeans_reduce(self, npoints, ncenters, dim, points, assign, sums, counts, ws=None, stream=None):
        if ws is None:
            ws = self._ws(self.lib.bof_kmeans_reduce_workspace_bytes(npoints, ncenters, dim))
        self._check(self.lib.bof_kmeans_reduce(self.h, stream or _cur_stream(), npoints, ncenters, dim, ptr(points),
                                               ptr(assign), ptr(sums), ptr(counts), ptr(ws), ws.numel()))

    def kmeans_finalize(self, ncenters, dim, sums, counts, centers, c_l2sq, stream=None):
        self._check(self.lib.bof_kmeans_finalize(self.h, stream or _cur_stream(), ncenters, dim, ptr(sums),
                                                 ptr(counts), ptr(centers), ptr(c_l2sq)))

    # ---- host entry points (numpy arrays / pinned torch CPU tensors) ----
    def host_csrmm(self, trans_a, m, n, k, alpha, beta, a, ia, ja, ord_b, b, c):
        self._check(self.lib.bof_host_csrmm(self.h, ch(trans_a), m, n, k, alpha, beta, ptr(a), ptr(ia), ptr(ja),
                                            ch(ord_b), ptr(b), ptr(c)))

    def host_gemm(self, ord_, ta, tb, m, n, k, alpha, beta, a, b, c, lda=0, ldb=0, ldc=0):
        self._check(self.lib.bof_host_gemm(self.h, ch(ord_), ch(ta), ch(tb), m, n, k, alpha, beta, ptr(a), ptr(b),
                                           ptr(c), lda, ldb, ldc))

    def host_gemm_devb(self, ta, tb, m, n, k, alpha, beta, a, b_dev, c, lda=0, ldb=0, ldc=0):
        self._check(self.lib.bof_host_gemm_devb(self.h, ch(ta), ch(tb), m, n, k, alpha, beta, ptr(a), ptr(b_dev),
                                                ptr(c), lda, ldb, ldc))

    def host_csrmm_devb(self, m, n, k, alpha, beta, a, ia, ja, b_dev, c):
        self._check(self.lib.bof_host_csrmm_devb(self.h, m, n, k, alpha, beta, ptr(a), ptr(ia), ptr(ja), ptr(b_dev),
                                                 ptr(c)))

    def host_gemv(self, ord_, trans, m, n, alpha, beta, a, x, y, lda=0):
        self._check(self.lib.bof_host_gemv(self.h, ch(ord_), ch(trans), m, n, alpha, beta, ptr(a), lda, ptr(x), ptr(y)))

    def host_csrgemv(self, trans_a, m, n, a, ia, ja, b, c):
        self._check(self.lib.bof_host_csrgemv(self.h, ch(trans_a), m, n, ptr(a), ptr(ia), ptr(ja), ptr(b), ptr(c)))

    def host_kmeans_dist(self, ord_, ta, tb, m, n, k, alpha, beta, a, b, c, c_l2sq, p_l2sq, lda=0, ldb=0, ldc=0):
        self._check(self.lib.bof_host_kmeans_dist(self.h, ch(ord_), ch(ta), ch(tb), m, n, k, alpha, beta, ptr(a), ptr(b),
                                                  ptr(c), lda, ldb, ldc, ptr(c_l2sq), ptr(p_l2sq)))

    # ---- multi-GPU: one communicator rank per context (bof_comm_*, bof_dist_*) ----
    def comm_init(self, world: int, rank: int, unique_id: bytes):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(self.lib.bof_comm_init(self.h, world, rank, C.cast(buf, C.c_void_p)))

    def comm_world(self) -> int:
        return int(self.lib.bof_comm_world(self.h))

    def dist_gemm(self, ta, tb, m_local, n, k, alpha, beta, a_local, b, c_local, lda=0, ldb=0, ldc=0):
        self._check(self.lib.bof_dist_gemm(self.h, ch(ta), ch(tb), m_local, n, k, alpha, beta, ptr(a_local), ptr(b),
                                           ptr(c_local), lda, ldb, ldc))

    def dist_csrmm(self, m_local, n, k, alpha, beta, a, ia, ja, b, c_local):
        self._check(self.lib.bof_dist_csrmm(self.h, m_local, n, k, alpha, beta, ptr(a), ptr(ia), ptr(ja), ptr(b),
                                            ptr(c_local)))

    def host_csrcsc(self, m, n, ia, ja, a, ia_tr, ja_tr, a_tr):
        self._check(self.lib.bof_host_csrcsc(self.h, m, n, ptr(ia), ptr(ja), ptr(a), ptr(ia_tr), ptr(ja_tr),
                                             ptr(a_tr)))


class KMeans:
    """Resident-shard Lloyd iteration (reference drivers/in_mem_kmeans.cpp:89-152 / drivers/kmeans.cpp:103-189)."""

    def __init__(self, ctx: Context, npoints, ncenters, dim, points_host, centers_host):
        self.ctx = ctx
        self.npoints, self.ncenters, self.dim = npoints, ncenters, dim
        self._points_host = points_host   # out-of-core shards are streamed from this buffer on every step
        h = C.c_void_p()
        ctx._check(ctx.lib.bof_kmeans_open(ctx.h, npoints, ncenters, dim, ptr(points_host), ptr(centers_host),
                                           C.byref(h)))
        self.h = h

    def local_step(self):
        """assign + local partial sums; returns (device address, float count) of [K*dim sums | K counts]."""
        p, n = C.c_void_p(), C.c_size_t()
        self.ctx._check(self.ctx.lib.bof_kmeans_local_step(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def update(self):
        self.ctx._check(self.ctx.lib.bof_kmeans_update(self.h))

    def allreduce(self):
        """NCCL sum of the partial buffer over the ranks of the context's communicator (no-op at world 1)"""
        self.ctx._check(self.ctx.lib.bof_kmeans_allreduce(self.h))

    def lloyd(self, iters: int):
        """iters x (local_step, allreduce, update) inside the library; asynchronous until get()"""
        self.ctx._check(self.ctx.lib.bof_kmeans_lloyd(self.h, iters))

    def get(self, centers_host=None, assign_host=None):
        self.ctx._check(self.ctx.lib.bof_kmeans_get(self.h, ptr(centers_host), ptr(assign_host)))

    def stream(self) -> int:
        return int(self.ctx.lib.bof_kmeans_stream(self.h) or 0)

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.bof_kmeans_close(self.h)
            self.h = None


class ResidentCsr:
    """A kept in HBM across csrmm / csrgemv calls (bof_csr_*; the eigensolver inner loop of SURVEY 8(f)-2)."""

    def __init__(self, ctx: Context, m, n, a, ia, ja):
        self.ctx, self.m, self.n = ctx, m, n
        h = C.c_void_p()
        ctx._check(ctx.lib.bof_csr_open(ctx.h, m, n, ptr(a), ptr(ia), ptr(ja), C.byref(h)))
        self.h = h

    def build_transpose(self):
        self.ctx._check(self.ctx.lib.bof_csr_build_transpose(self.h))

    def arrays(self, trans_a="N"):
        """(vals, idx, offs) device addresses and nnz of A ('N') or A^T ('T')."""
        v, i, o, z = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_int64()
        self.ctx._check(self.ctx.lib.bof_csr_arrays(self.h, ch(trans_a), C.byref(v), C.byref(i), C.byref(o),
                                                    C.byref(z)))
        return v.value, i.value, o.value, z.value

    def mm(self, trans_a, k, alpha, beta, ord_b, b, c):
        self.ctx._check(self.ctx.lib.bof_csr_mm(self.h, ch(trans_a), k, alpha, beta, ch(ord_b), ptr(b), ptr(c)))

    def mv(self, trans_a, x, y):
        self.ctx._check(self.ctx.lib.bof_csr_mv(self.h, ch(trans_a), ptr(x), ptr(y)))

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.bof_csr_close(self.h)
            self.h = None


def comm_unique_id() -> bytes:
    """128-byte id for bof_comm_init; create on one rank and distribute (dist.init_comm does it over torch.distributed)."""
    lib = load()
    buf = C.create_string_buffer(128)
    rc = lib.bof_comm_unique_id(C.cast(buf, C.c_void_p))
    if rc != 0:
        raise BofError(rc, "bof_comm_unique_id failed (libnccl.so.2 not loadable?)")
    return buf.raw


class MultiGpu:
    """One process, several GPUs (bof_mgpu_*): what the C++ flash:: adapters use when BOF_GPUS > 1."""

    def __init__(self, ndev: int = 0, devices=None, **cfg):
        self.lib = load()
        conf = BofConfig()
        for k, v in cfg.items():
            setattr(conf, k, v)
        devs = (C.c_int * len(devices))(*devices) if devices else None
        h = C.c_void_p()
        rc = self.lib.bof_mgpu_create(C.byref(conf), len(devices) if devices else ndev, C.cast(devs, C.c_void_p) if devs else None,
                                      C.byref(h))
        if rc != 0:
            raise BofError(rc, (self.lib.bof_last_error(None) or b"").decode())
        self.h = h

    def count(self) -> int:
        return int(self.lib.bof_mgpu_count(self.h))

    def _check(self, rc):
        if rc != 0:
            raise BofError(rc, (self.lib.bof_mgpu_last_error(self.h) or b"").decode())

    def gemm(self, ord_, ta, tb, m, n, k, alpha, beta, a, b, c, lda=0, ldb=0, ldc=0):
        self._check(self.lib.bof_mgpu_gemm(self.h, ch(ord_), ch(ta), ch(tb), m, n, k, alpha, beta, ptr(a), ptr(b), ptr(c),
                                           lda, ldb, ldc))

    def csrmm(self, trans_a, m, n, k, alpha, beta, a, ia, ja, ord_b, b, c):
        self._check(self.lib.bof_mgpu_csrmm(self.h, ch(trans_a), m, n, k, alpha, beta, ptr(a), ptr(ia), ptr(ja), ch(ord_b),
                                            ptr(b), ptr(c)))

    def csrgemv(self, trans_a, m, n, a, ia, ja, x, y):
        self._check(self.lib.bof_mgpu_csrgemv(self.h, ch(trans_a), m, n, ptr(a), ptr(ia), ptr(ja), ptr(x), ptr(y)))

    def gemv(self, ord_, trans, m, n, alpha, beta, a, x, y, lda=0):
        self._check(self.lib.bof_mgpu_gemv(self.h, ch(ord_), ch(trans), m, n, alpha, beta, ptr(a), lda, ptr(x), ptr(y)))

    def kmeans_lloyd(self, npoints, ncenters, dim, points, centers, iters, assign=None):
        self._check(self.lib.bof_mgpu_kmeans_lloyd(self.h, npoints, ncenters, dim, ptr(points), ptr(centers), iters,
                                                   ptr(assign)))

    def close(self):
        if getattr(self, "h", None):
            self.lib.bof_mgpu_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
