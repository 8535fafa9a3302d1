"""Runs the reference's OWN drivers, built unmodified into ``oracle/_ref/`` by ``oracle/Makefile.ref``.
TEST INFRASTRUCTURE ONLY (same rule as ``oracle/__init__.py``): tests, golden-fixture generation and
``bench.py``'s CPU legs.  Nothing here reads ``/root/reference`` -- only the prebuilt binaries.

Each function writes its numpy operands in the reference's file formats (raw fp32 / int64, the
``.csr/.col/.off`` triple of misc/sparse_create.cpp), invokes one driver with the positional command
line of ``drivers/*.cpp`` and reads the output file back.  ``flash=True`` selects the out-of-core
driver (``drivers/gemm.cpp``, ``csrmm.cpp``, ``csrgemv.cpp``, ``kmeans.cpp``, and flash::csrcsc behind
``oracle/ref_shim/ref_csrcsc_main.cpp``), otherwise the ``in_mem_*`` driver -- a bare MKL call.
The flash drivers open files with O_DIRECT (src/file_handles/flash_file_handle.cpp:193), which works on
tmpfs from Linux 6.6 on; the scratch directory defaults to /dev/shm.
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_REF = Path(__file__).resolve().parent / "_ref"


def available(suffix: str = "") -> bool:
    return (_REF / f"in_mem_gemm_driver{suffix}").exists() and (_REF / "libmklshim.so").exists()


def exe(name: str, suffix: str = "") -> str:
    p = _REF / f"{name}{suffix}"
    if not p.exists():
        raise FileNotFoundError(f"{p} missing: run `make -C oracle -f Makefile.ref REF=<reference sources>`")
    return str(p)


class Scratch:
    """A private directory for one driver run (tmpfs by default), removed on exit."""

    def __init__(self, base: str | None = None):
        base = base or os.environ.get("BOF_REF_SCRATCH") or ("/dev/shm" if os.path.isdir("/dev/shm") else None)
        self.dir = Path(tempfile.mkdtemp(prefix="bofref_", dir=base))

    def put(self, name: str, arr: np.ndarray, pad_to: int = 4096) -> str:
        """Raw little-endian dump, zero-padded to a 4 KiB multiple: the flash file handle reads and writes
        whole sectors around unaligned ends (flash_file_handle.cpp:508-716)."""
        p = self.dir / name
        raw = np.ascontiguousarray(arr).tobytes()
        pad = (-len(raw)) % pad_to if pad_to else 0
        with open(p, "wb") as f:
            f.write(raw)
            if pad or not raw:
                f.write(b"\0" * (pad if raw else pad_to))
        return str(p)

    def get(self, name: str, dtype, count: int) -> np.ndarray:
        return np.fromfile(self.dir / name, dtype=dtype, count=count)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        shutil.rmtree(self.dir, ignore_errors=True)


def _run(cmd, cwd=None, threads: int | None = None, timeout: float | None = None) -> str:
    timeout = timeout or float(os.environ.get("BOF_REF_TIMEOUT", "3600"))
    env = dict(os.environ)
    if threads:
        env["OMP_NUM_THREADS"] = env["MKL_NUM_THREADS"] = str(threads)
    r = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError(f"{cmd[0]} exited {r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}")
    return r.stdout


def took(stdout: str, what: str) -> float | None:
    """Seconds the driver itself reports around the kernel call ('gemm() took 1.23', Timer in ms/1000)."""
    m = re.search(re.escape(what) + r"\(\) took\s+([0-9.eE+-]+)", stdout)
    return float(m.group(1)) if m else None


def gemm(ord_, ta, tb, m, n, k, alpha, beta, a, b, c, lda, ldb, ldc, flash=False, suffix="", threads=None,
         want_time=False):
    """drivers/in_mem_gemm.cpp:12-16 / drivers/gemm.cpp:17-21: <A> <B> <C> <m> <k> <n> <alpha> <beta> <ta> <tb> <ord>
    <lda> <ldb> <ldc>.  The in-memory driver reads m*k / k*n / m*n floats, i.e. tight leading dimensions."""
    with Scratch() as s:
        fa, fb, fc = s.put("A", a), s.put("B", b), s.put("C", c)
        args = [fa, fb, fc, str(m), str(k), str(n), repr(float(alpha)), repr(float(beta)), ta, tb, ord_, str(lda),
                str(ldb), str(ldc)]
        if flash:
            os.makedirs("/tmp/gemm_driver_temps", exist_ok=True)
        out = _run([exe("gemm_driver" if flash else "in_mem_gemm_driver", suffix), *args], cwd=s.dir, threads=threads)
        res = s.get("C", np.float32, np.asarray(c).size).reshape(np.asarray(c).shape)
    return (res, took(out, "gemm")) if want_time else res


def _put_csr(s, a, ia, ja):
    return s.put("A.csr", np.asarray(a, np.float32)), s.put("A.col", np.asarray(ja, np.int64)), s.put(
        "A.off", np.asarray(ia, np.int64))


def csrmm(trans, m, n, k, alpha, beta, a, ia, ja, ord_b, b, c, flash=False, suffix="", threads=None, want_time=False,
          pmem=False):
    """drivers/in_mem_csrmm.cpp:13-31 / drivers/csrmm.cpp:12-33: <vals> <idxs> <offs> <B> <C> <a_nrows> <a_ncols>
    <b_ncols> <alpha> <beta> <trans_a> <ord_b>; ord_b 'R' row-major / 'C' column-major."""
    with Scratch() as s:
        fv, fi, fo = _put_csr(s, a, ia, ja)
        fb, fc = s.put("B", b), s.put("C", c)
        name = "csrmm_pmem_driver" if pmem else ("csrmm_driver" if flash else "in_mem_csrmm_driver")
        out = _run([exe(name, suffix), fv, fi, fo, fb, fc, str(m), str(n), str(k), repr(float(alpha)),
                    repr(float(beta)), trans, ord_b], cwd=s.dir, threads=threads)
        res = s.get("C", np.float32, np.asarray(c).size).reshape(np.asarray(c).shape)
    return (res, took(out, "csrmm" if flash or pmem else "mkl_csrmm")) if want_time else res


def csrgemv(trans, m, n, a, ia, ja, x, flash=False, suffix="", threads=None):
    """drivers/in_mem_csrgemv.cpp:13-27 / drivers/csrgemv.cpp: <vals> <idxs> <offs> <b> <c> <a_nrows> <a_ncols> <trans>."""
    ylen = m if trans == "N" else n
    with Scratch() as s:
        fv, fi, fo = _put_csr(s, a, ia, ja)
        fb, fc = s.put("x", np.asarray(x, np.float32)), s.put("y", np.zeros(ylen, np.float32))
        _run([exe("ref_csrgemv" if flash else "in_mem_csrgemv_driver", suffix), fv, fi, fo, fb, fc, str(m), str(n),
              trans], cwd=s.dir, threads=threads)
        return s.get("y", np.float32, ylen)


def csrcsc(m, n, ia, ja, a, flash=False, suffix="", threads=None):
    """drivers/in_mem_csrcsc.cpp:12-27: <vals> <idxs> <offs> <valsT> <idxsT> <offsT> <n_rows> <n_cols>; the flash
    variant goes through ref_csrcsc (same arguments + scratch dir) -> flash::csrcsc."""
    nnz = int(ia[m] - ia[0])
    with Scratch() as s:
        fv, fi, fo = _put_csr(s, a, ia, ja)
        tv = s.put("T.csr", np.zeros(max(nnz, 1), np.float32))
        ti = s.put("T.col", np.zeros(max(nnz, 1), np.int64))
        to = s.put("T.off", np.zeros(n + 1, np.int64))
        if flash:
            _run([exe("ref_csrcsc", suffix), fv, fi, fo, tv, ti, to, str(m), str(n), str(s.dir) + "/"], cwd=s.dir,
                 threads=threads)
        else:
            _run([exe("in_mem_csrcsc_driver", suffix), fv, fi, fo, tv, ti, to, str(m), str(n)], cwd=s.dir,
                 threads=threads)
        return s.get("T.off", np.int64, n + 1), s.get("T.col", np.int64, nnz), s.get("T.csr", np.float32, nnz)


def kmeans_iters(points, centers, iters=1, suffix="", threads=None):
    """drivers/in_mem_kmeans.cpp:153-157: <points> <centers> <npoints> <ndims> <ncenters>; one Lloyd iteration per
    invocation, the centers file is overwritten in place -> run it `iters` times.  (drivers/kmeans.cpp, the flash
    variant, cannot run as shipped -- see oracle/ref_shim/ref_kmeans_dist_main.cpp.)"""
    points = np.ascontiguousarray(points, np.float32)
    centers = np.ascontiguousarray(centers, np.float32)
    P, d = points.shape
    K = centers.shape[0]
    with Scratch() as s:
        fp, fc = s.put("points", points, pad_to=0), s.put("centers", centers, pad_to=0)
        for _ in range(iters):
            _run([exe("in_mem_kmeans_driver", suffix), fp, fc, str(P), str(d), str(K)], cwd=s.dir, threads=threads)
        return s.get("centers", np.float32, K * d).reshape(K, d)


def kmeans_dist(points, centers, suffix="", threads=None):
    """flash::kmeans called as drivers/kmeans.cpp:37-39 does -> the P x K distance matrix (row p = point p)."""
    points = np.ascontiguousarray(points, np.float32)
    centers = np.ascontiguousarray(centers, np.float32)
    P, d = points.shape
    K = centers.shape[0]
    with Scratch() as s:
        fp, fc = s.put("points", points), s.put("centers", centers)
        fd = s.put("dist", np.zeros(P * K, np.float32))
        _run([exe("ref_kmeans_dist", suffix), fp, fc, fd, str(P), str(d), str(K)], cwd=s.dir, threads=threads)
        return s.get("dist", np.float32, P * K).reshape(P, K)
