#!/usr/bin/env python
"""flash::gemv on one B200.  Prints one JSON line:

  resident  bof_sgemv_f32 on a 4 GiB device-resident A (well past the 126 MB L2) for 32768 x 32768, 2^24 x 64 and
            64 x 2^24, both reduction shapes (row-dot = ('R','N'), column-sum = ('R','T')); CUDA events over --iters
            launches after a warm-up; GB/s counts A + x + y once, and the fraction is of the 7.7 TB/s data-sheet HBM rate.
  e2e       bof_host_gemv from a pinned 8 GiB A (32768 x 65536, ('R','N')) next to a pinned host-to-device copy of the
            same bytes, both measured here, best of --rounds.  The end-to-end call is bound by PCIe.
  cpu       torch.mv of the same 8 GiB A on the host, with its thread count.
  card      name and power limit from nvidia-smi in the same run.

    python tools/bench_gemv.py [--iters 20] [--rounds 3]"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402

GiB = 1 << 30
HBM_BPS = 7.7e12


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
    name, pl = [s.strip() for s in out.splitlines()[0].split(",")]
    return name, pl


def resident(ctx, iters):
    A = torch.rand(GiB, device="cuda") - 0.5   # 4 GiB, every shape below is a view of it
    res = []
    for (m, n) in [(32768, 32768), (1 << 24, 64), (64, 1 << 24)]:
        for trans in "NT":
            xl, yl = (n, m) if trans == "N" else (m, n)
            x = torch.rand(xl, device="cuda")
            y = torch.zeros(yl, device="cuda")
            ws = ctx.sgemv_workspace("R", trans, m, n)
            for _ in range(3):
                ctx.sgemv("R", trans, m, n, 1.0, A, 0, x, 0.0, y, ws=ws)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                ctx.sgemv("R", trans, m, n, 1.0, A, 0, x, 0.0, y, ws=ws)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            nbytes = 4 * (m * n + xl + yl)
            res.append({"m": m, "n": n, "trans": trans, "shape": "row-dot" if trans == "N" else "column-sum",
                        "ms": round(ms, 4), "GBps": round(nbytes / ms / 1e6, 1),
                        "frac_7p7TBps": round(nbytes / ms / 1e-3 / HBM_BPS, 3)})
    del A
    torch.cuda.empty_cache()
    return res


def end_to_end(ctx, rounds):
    m, n = 32768, 65536   # 8 GiB
    A = torch.empty((m, n), dtype=torch.float32, pin_memory=True)
    for r0 in range(0, m, 4096):   # fill through the GPU: a host-side rand of 2^31 floats takes minutes
        A[r0:r0 + 4096].copy_(torch.rand((4096, n), device="cuda") - 0.5)
    x = torch.rand(n).pin_memory()
    y = torch.zeros(m).pin_memory()
    dst = torch.empty((m, n), dtype=torch.float32, device="cuda")
    h2d, e2e = [], []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(A, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        h2d.append(e0.elapsed_time(e1))
    del dst
    torch.cuda.empty_cache()
    for _ in range(rounds):
        t0 = time.perf_counter()
        ctx.host_gemv("R", "N", m, n, 1.0, 0.0, A, x, y)
        e2e.append((time.perf_counter() - t0) * 1e3)
    st = ctx.stats()
    # CPU reference point on the same bytes
    cpu = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        yc = torch.mv(A, x)
        cpu.append((time.perf_counter() - t0) * 1e3)
    err = float((yc - y).abs().max() / yc.abs().max().clamp_min(1e-30))
    nbytes = 4 * m * n
    return {"m": m, "n": n, "A_GiB": nbytes / GiB,
            "pinned_h2d_ms": round(min(h2d), 2), "pinned_h2d_GBps": round(nbytes / min(h2d) / 1e6, 1),
            "host_gemv_ms": round(min(e2e), 2), "host_gemv_GBps": round(nbytes / min(e2e) / 1e6, 1),
            "host_gemv_over_h2d": round(min(e2e) / min(h2d), 3),
            "h2d_bytes": st.h2d_bytes, "d2h_bytes": st.d2h_bytes, "kernel_launches": st.kernel_launches,
            "cpu_torch_mv_ms": round(min(cpu), 2), "cpu_threads": torch.get_num_threads(),
            "cpu_torch_mv_GBps": round(nbytes / min(cpu) / 1e6, 1), "max_rel_diff_vs_cpu": err}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_gemv needs a GPU")
    bof = g.load_package()
    name, pl = gpu_info()
    ctx = bof.Context(device=0)
    try:
        out = {"bench": "gemv", "card": name, "power_limit": pl, "resident": resident(ctx, max(args.iters, 20)),
               "e2e": end_to_end(ctx, args.rounds)}
    finally:
        ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
