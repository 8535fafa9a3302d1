#!/usr/bin/env python
"""bof_host_gemm on operands larger than HBM (the out-of-core plan), from pinned host buffers.  Prints one JSON line per
case and a last one with everything, plus the card's name and power limit.

  (a) 32768 x 262144 x 32768 NN, the largest point of the paper's gemm figure (Fig. 5, d = 262144): 34 GB per input, at
      the default budget (really beyond HBM, nothing forced).  Time, 2mnk/t, PCIe bytes, the ratio to the PCIe bound
      (H2D bytes over the pinned H2D rate measured in the same run), and 128 seeded rows of C against float64.
  (b) A^T B with A, B 2^24 x 1024 ('T','N', m = n = 1024): the tall-skinny projection.  Scaled down when host memory
      is short, and then kept beyond the budget with BOF_GEMM_HBM_BUDGET.
  (c) 32768^3 NN, resident and forced out of core (BOF_GEMM_HBM_BUDGET = half the resident footprint), alternated.

    python tools/bench_gemm_ooc.py [--out profiles/gemm_ooc.json] [--rounds 3] [--skip a,b]"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402

GiB = 1 << 30


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, pl = [s.strip() for s in out.splitlines()[0].split(",")]
        return name, pl
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return torch.cuda.get_device_name(0), None


def mem_available():
    for line in open("/proc/meminfo"):
        if line.startswith("MemAvailable:"):
            return int(line.split()[1]) * 1024
    return 0


def pinned_random(rows, cols, seed):
    """rows x cols fp32 standard normal in pinned host memory, generated on the device slab by slab."""
    t = torch.empty((rows, cols), dtype=torch.float32, pin_memory=True)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    step = max(1, (1 << 28) // cols)
    for r0 in range(0, rows, step):
        r1 = min(rows, r0 + step)
        t[r0:r1].copy_(torch.randn((r1 - r0, cols), device="cuda", generator=gen), non_blocking=False)
    torch.cuda.synchronize()
    return t


def h2d_rate(nbytes=4 * GiB):
    src = torch.empty(nbytes // 4, dtype=torch.float32, pin_memory=True)
    dst = torch.empty_like(src, device="cuda")
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    rate = 3 * nbytes / (time.perf_counter() - t0)
    del src, dst
    torch.cuda.empty_cache()
    return rate


def timed_gemm(ctx, ta, tb, m, n, k, a, b, c, budget=None):
    """Wall time of one call (it returns after its last download) and its stats."""
    if budget is None:
        os.environ.pop("BOF_GEMM_HBM_BUDGET", None)
    else:
        os.environ["BOF_GEMM_HBM_BUDGET"] = str(budget)
    t0 = time.perf_counter()
    ctx.host_gemm("R", ta, tb, m, n, k, 1.0, 0.0, a, b, c)
    dt = time.perf_counter() - t0
    os.environ.pop("BOF_GEMM_HBM_BUDGET", None)
    return dt, ctx.stats()


def release():
    torch.cuda.empty_cache()
    torch._C._host_emptyCache()   # pinned blocks go back to the system


def check_rows(a, b, c, ta, rows):
    """max over the sampled rows of |C - R| / (2^-16 |A||B|), float64 on the device, k in slabs."""
    k = a.shape[0] if ta == "T" else a.shape[1]
    n = b.shape[1]
    ref = torch.zeros((len(rows), n), dtype=torch.float64, device="cuda")
    mag = torch.zeros_like(ref)
    idx = torch.as_tensor(rows)
    a_rows = None if ta == "T" else a[idx]
    step = 8192
    for k0 in range(0, k, step):
        k1 = min(k, k0 + step)
        ap = (a[k0:k1][:, idx].T if ta == "T" else a_rows[:, k0:k1]).cuda().double()
        bp = b[k0:k1].cuda().double()
        ref += ap @ bp
        mag += ap.abs() @ bp.abs()
    got = c[idx].cuda().double()
    ratio = ((got - ref).abs() / (2.0 ** -16 * mag).clamp_min(1e-300)).max().item()
    rel = ((got - ref).norm() / ref.norm()).item()
    return ratio, rel


def case_a(bof, rate, out):
    m, k, n = 32768, 262144, 32768
    a, b = pinned_random(m, k, 1), pinned_random(k, n, 2)
    c = torch.empty((m, n), dtype=torch.float32, pin_memory=True)
    release()
    with bof.Context(device=0) as ctx:   # two calls: the first also reserves the device buffers
        times = [timed_gemm(ctx, "N", "N", m, n, k, a, b, c)[0]]
        dt, st = timed_gemm(ctx, "N", "N", m, n, k, a, b, c)
        times.append(dt)
    rows = np.random.default_rng(5).choice(m, 128, replace=False)
    ratio, rel = check_rows(a, b, c, "N", rows)
    bound = st.h2d_bytes / rate
    r = dict(case="a_fig5_32768x262144x32768_NN", seconds_first_then_second=times, seconds=dt, tflops=2.0 * m * n * k / dt / 1e12,
             h2d_bytes=st.h2d_bytes, d2h_bytes=st.d2h_bytes, h2d_rate_gbs=rate / 1e9, pcie_bound_s=bound,
             x_of_pcie_bound=dt / bound, rows_checked=128, max_err_over_bound=ratio, rel_fro_rows=rel)
    print(json.dumps(r), flush=True)
    out.append(r)


def case_b(bof, rate, out):
    m = n = 1024
    k = 1 << 24
    need = 2 * k * 1024 * 4
    note, budget = None, None
    if mem_available() < need * 1.5:
        k = max(1 << 20, int(mem_available() / 1.5 / (2 * 1024 * 4)) >> 20 << 20)
        # resident footprint at this k is about 12 bytes per element of Q plus the P ring; half of it forces the plan
        budget = (n * k * 12) // 2
        note = (f"host memory available {mem_available() / GiB:.0f} GiB < {need * 1.5 / GiB:.0f} GiB: k scaled to {k}, "
                f"BOF_GEMM_HBM_BUDGET={budget}")
        print(note, flush=True)
    a, b = pinned_random(k, m, 3), pinned_random(k, n, 4)   # stored k x m and k x n: op(A) = A^T
    c = torch.empty((m, n), dtype=torch.float32, pin_memory=True)
    release()
    with bof.Context(device=0) as ctx:
        times = [timed_gemm(ctx, "T", "N", m, n, k, a, b, c, budget)[0]]
        dt, st = timed_gemm(ctx, "T", "N", m, n, k, a, b, c, budget)
        times.append(dt)
    rows = np.random.default_rng(6).choice(m, 128, replace=False)
    ratio, rel = check_rows(a, b, c, "T", rows)
    bound = st.h2d_bytes / rate
    r = dict(case=f"b_tall_skinny_AtB_m{m}_n{n}_k{k}", note=note, seconds_first_then_second=times, seconds=dt, tflops=2.0 * m * n * k / dt / 1e12,
             h2d_bytes=st.h2d_bytes, d2h_bytes=st.d2h_bytes, pcie_bound_s=bound, x_of_pcie_bound=dt / bound,
             rows_checked=128, max_err_over_bound=ratio, rel_fro_rows=rel)
    print(json.dumps(r), flush=True)
    out.append(r)


def case_c(bof, rounds, out):
    m = n = k = 32768
    a, b = pinned_random(m, k, 7), pinned_random(k, n, 8)
    c_res = torch.empty((m, n), dtype=torch.float32, pin_memory=True)
    c_ooc = torch.empty_like(c_res, pin_memory=True)
    # resident: Q raw + planes (12 B/elem) + 5 generations of 4096-row P blocks (12 B/elem) and C blocks (4 B/elem)
    resident = n * k * 12 + 5 * 4096 * (k * 12 + n * 4)
    budget = resident // 2
    release()
    with bof.Context(device=0) as res, bof.Context(device=0) as ooc:   # each keeps its plan's buffers
        timed_gemm(res, "N", "N", m, n, k, a, b, c_res)   # warm-up of both plans
        timed_gemm(ooc, "N", "N", m, n, k, a, b, c_ooc, budget)
        t_res, t_ooc = [], []
        for _ in range(rounds):
            t_res.append(timed_gemm(res, "N", "N", m, n, k, a, b, c_res)[0])
            dt, st = timed_gemm(ooc, "N", "N", m, n, k, a, b, c_ooc, budget)
            t_ooc.append(dt)
    r = dict(case="c_32768cubed_resident_vs_ooc", budget=budget, resident_s=t_res, ooc_s=t_ooc,
             overhead=min(t_ooc) / min(t_res) - 1.0, ooc_h2d_bytes=st.h2d_bytes,
             array_equal=bool(torch.equal(c_res, c_ooc)))
    print(json.dumps(r), flush=True)
    out.append(r)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the results to this JSON file")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--skip", default="", help="comma-separated cases to skip (a, b, c)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    bof = g.load_package()
    name, pl = gpu_info()
    rate = h2d_rate()
    print(json.dumps(dict(gpu=name, power_limit=pl, h2d_pinned_gbs=rate / 1e9)), flush=True)
    out = []
    skip = set(args.skip.split(","))
    for key, fn in (("a", lambda: case_a(bof, rate, out)), ("b", lambda: case_b(bof, rate, out)),
                    ("c", lambda: case_c(bof, args.rounds, out))):
        if key not in skip:
            fn()
            release()
    res = dict(gpu=name, power_limit=pl, h2d_pinned_gbs=rate / 1e9, cases=out)
    print(json.dumps(res), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
