#!/usr/bin/env python
"""Device time of bof_kmeans_assign with the accumulation folded into fp32 every gemm_k_chunk elements of k (default
256) against the whole k in TMEM (gemm_k_chunk=-1), CUDA events around back-to-back calls on prepared point planes;
also how many assignments the two settings disagree on.  Prints one JSON line with the card name and power limit.
    python tools/bench_kmeans_chunk.py [--points 1048576] [--centers 1024] [--dim 1024] [--iters 10]"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402

import __graft_entry__ as g  # noqa: E402


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=1 << 20)
    ap.add_argument("--centers", type=int, default=1024)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two settings")
    args = ap.parse_args()
    bof = g.load_package()
    P, K, d = args.points, args.centers, args.dim
    gen = torch.Generator(device="cuda").manual_seed(3)
    cent = torch.randn((K, d), device="cuda", generator=gen) * 4
    pts = cent[torch.randint(0, K, (P,), device="cuda", generator=gen)] + 0.05 * torch.randn((P, d), device="cuda",
                                                                                                generator=gen)
    res = {"points": P, "centers": K, "dim": d, "iters": args.iters, "gpu": torch.cuda.get_device_name(0),
           "power_limit_w": power_limit_w()}
    ctxs = {"k_chunk_256": bof.Context(device=0), "k_chunk_whole": bof.Context(device=0, gemm_k_chunk=-1)}
    try:
        c0 = ctxs["k_chunk_256"]
        p2 = torch.empty(P, device="cuda"); c2 = torch.empty(K, device="cuda")
        c0.row_sqnorm(P, d, pts, d, p2)
        c0.row_sqnorm(K, d, cent, d, c2)
        planes = c0.kmeans_prepare_points(P, d, pts)  # the same planes serve both contexts (same split)
        ws = c0._ws(c0.lib.bof_kmeans_workspace_bytes(P, K, d, 0))
        outs = {name: torch.empty(P, dtype=torch.int32, device="cuda") for name in ctxs}
        times = {name: [] for name in ctxs}
        for name, c in ctxs.items():  # warm-up
            c.kmeans_assign(P, K, d, pts, cent, c2, p2, outs[name], planes=planes, ws=ws)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):
            for name, c in ctxs.items():
                e0.record()
                for _ in range(args.iters):
                    c.kmeans_assign(P, K, d, pts, cent, c2, p2, outs[name], planes=planes, ws=ws)
                e1.record()
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) / args.iters)
        for name in ctxs:
            ms = min(times[name])
            res[name] = {"ms_per_call_min": ms, "ms_per_call_all": times[name],
                         "tflops_dot": 2.0 * P * K * d / (ms * 1e-3) / 1e12}
        res["assign_differ"] = int((outs["k_chunk_256"] != outs["k_chunk_whole"]).sum())
    finally:
        for c in ctxs.values():
            c.close()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
