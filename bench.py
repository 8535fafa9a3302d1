#!/usr/bin/env python
"""bench.py -- headline measurement for the B200-native BLAS-on-Flash hot path.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): flash::gemm sgemm 32768 x 32768 x 32768 fp32, row-major NN,
alpha 1 beta 0, output row blocks sharded over the N ranks with no collective (strong scaling:
the job is fixed, rank r owns C rows [r*M/N, (r+1)*M/N), B is replicated).
A "step" is one pass of the hot path over that job.

  value   whole-job GFLOP/s with the operands resident in HBM (bof_sgemm_f32: operand split of both
          matrices + the tcgen05 kernel), CUDA-event timed, max over ranks.
  e2e     the same metric through the host entry point bof_host_gemm (what flash::gemm calls):
          pinned host buffers, H2D of A-shard and B and D2H of C inside the timed region.
  roofline  dominant kernel gemm3xtf32_kernel: useful flops 2*m*n*k per launch / its CUDA-event
          duration, against 1/(1/TF32 + 2/BF16) (one tf32 and two bf16 MMAs per product), BF16 from
          MEASURED_PEAKS.json, TF32 from a cuBLAS measurement in the same run (sustained figures:
          the kernel runs ~0.2 s per launch).
  cpu_baseline  the reference's own in_mem_gemm driver (oracle/_ref, unmodified drivers/in_mem_gemm.cpp ->
          cblas_sgemm = MKL) on the box's host cores on a bounded sample: one 8192^3 GemmTask tile (1/64 of the
          job); MKL sgemm through ctypes if the binary is not on the box.
  extra   every other BASELINE.json config at the same world size (tools/bench_configs.py): csrmm_cfg1,
          csrmm_cfg3 (sharded; replicated and all-gathered B), csrgemv_N/T_cfg4, csrcsc_cfg4, kmeans_cfg5 (with the
          NCCL allreduce at N > 1), each with roofline, e2e (host buffers, byte counts), cpu_baseline and a parity
          figure on the timed buffers; plus the pinned PCIe bandwidth of all ranks copying at once.

--steps K sets the number of timed steps of both gemm legs.  --dump-outputs DIR writes, after the timed steps,
what the last step of each leg returned: DIR/gemm_C_rows.npy (bof_sgemm_f32) and DIR/host_gemm_C_rows.npy
(bof_host_gemm), fp32, the same DUMP_ROWS seeded rows of C in every run (rank 0's row block when N > 1).  The
inputs come from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
if "--impl" in sys.argv and "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host thread (must be set before
    # libgomp / MKL initialise, i.e. before numpy or torch are imported)
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    os.environ["MKL_NUM_THREADS"] = str(os.cpu_count() or 1)

M_FULL = N_FULL = K_FULL = 32768
# dram__bytes_read.sum + dram__bytes_write.sum of one full-size gemm3xtf32_kernel launch, from the
# ncu --set full capture summarised in profiles/ (None until that capture exists)
NCU_TRAFFIC_BYTES = 275551000000 + 4630000000  # profiles/r02/t14_per_launch_all_configs.txt (gemm3xtf32_kernel<2,0,1,1>, one launch)
TILE = 8192  # reference GEMM_BLK_SIZE (CMakeLists.txt:46-50 of the reference)
DUMP_ROWS = 128  # rows of C dumped per leg: 2 x 128 x 32768 fp32 = 32 MiB at the full size


def dump_rows(m: int):
    """The rows of an m-row C that --dump-outputs writes: a fixed seeded sample, sorted."""
    import numpy as np

    return np.sort(np.random.default_rng(0x5EED00D0).choice(m, size=min(m, DUMP_ROWS), replace=False))


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"],
                "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML in a thread every 10 ms (an nvidia-smi child
    takes longer to start than a short multi-GPU timed region lasts), nvidia-smi -lms as the fallback."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    # nvmlClocksEventReason* bits
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index: int, pci_bus_id: str = None):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self.thread, self.run = None, None, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = None
            for bus in ((pci_bus_id, pci_bus_id.encode()) if pci_bus_id else ()):
                try:
                    self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus)
                    break
                except Exception:
                    continue
            if self.handle is None:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while self.run:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append((sm, self.max_sm, mask))
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.nvml:
            self.run = True
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        sm, mx, reasons = [], [], set()
        if self.nvml:
            self.run = False
            self.thread.join(timeout=1)
            for s_, m_, mask in self.rows:
                sm.append(s_); mx.append(m_)
                reasons.update(k for k, bit in self.BITS.items() if mask & bit)
            src = "nvml"
        else:
            if self.proc:
                self.proc.terminate()
                try:
                    self.proc.wait(timeout=2)
                except Exception:
                    self.proc.kill()
            for r in self.rows:
                try:
                    sm.append(float(r[0])); mx.append(float(r[1]))
                except Exception:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            src = "nvidia-smi"
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": src}


def gpu_pci_bus_id(torch, local: int):
    """NVML's index ignores CUDA_VISIBLE_DEVICES; address the device torch uses by its PCI bus id."""
    try:
        p = torch.cuda.get_device_properties(local)
        return "%08X:%02X:%02X.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
    except Exception:
        return None


def ref_gemm_sample(reps: int = 1):
    """One reference GemmTask tile (8192^3) through the reference's OWN in_mem_gemm driver binary (oracle/_ref,
    built from the unmodified sources by oracle/Makefile.ref), timed by the driver's own chrono bracket around
    cblas_sgemm (drivers/in_mem_gemm.cpp:63-70).  Returns (cpu_baseline dict, seconds) or None if the binary is
    not on this box."""
    import numpy as np
    from oracle import ref_run as rr

    if not rr.available():
        return None
    n = TILE
    rng = np.random.default_rng(0)
    a = rng.random(n * n, dtype=np.float32)
    b = rng.random(n * n, dtype=np.float32)
    c = np.zeros(n * n, dtype=np.float32)
    best = float("inf")
    for _ in range(reps):
        _, secs = rr.gemm("R", "N", "N", n, n, n, 1.0, 0.0, a, b, c, n, n, n, want_time=True)
        if not secs:
            return None
        best = min(best, secs)
    return {"value": 2.0 * n ** 3 / best / 1e9, "unit": "GFLOP/s", "cores": os.cpu_count(), "kind": "reference",
            "sample": f"oracle/_ref/in_mem_gemm_driver (unmodified drivers/in_mem_gemm.cpp -> cblas_sgemm, MKL threads = all "
                      f"{os.cpu_count()} logical cpus) on one reference GemmTask tile {n}^3 = 1/64 of the job, its own timer: {best:.2f} s"}, best


def cpu_gemm_sample(reps: int = 2):
    """MKL sgemm on one reference GemmTask tile (8192^3), all host threads (fallback when oracle/_ref is absent)."""
    import numpy as np
    from oracle import mkl

    got = ref_gemm_sample(reps=1)
    if got is not None:
        return got

    n = TILE
    rng = np.random.default_rng(0)
    a = rng.random((n, n), dtype=np.float32)
    b = rng.random((n, n), dtype=np.float32)
    c = np.zeros((n, n), dtype=np.float32)
    mkl.sgemm_rowmajor(256, 256, 256, 1.0, a[:256, :256].copy(), b[:256, :256].copy(), 0.0, c[:256, :256].copy())
    best = float("inf")
    for _ in range(reps):
        t = time.perf_counter()
        mkl.sgemm_rowmajor(n, n, n, 1.0, a, b, 0.0, c)
        best = min(best, time.perf_counter() - t)
    return {"value": 2.0 * n ** 3 / best / 1e9, "unit": "GFLOP/s", "cores": mkl.max_threads(), "kind": "port",
            "sample": f"MKL sgemm_ (oneMKL via libtorch_cpu) on one reference GemmTask tile {n}^3 = 1/64 of the job, "
                      f"best of {reps}, {best:.2f} s; host has {os.cpu_count()} logical cpus"}, best


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of this workload -- oracle/_ref/in_mem_gemm_driver,
    the unmodified reference driver built by oracle/Makefile.ref (MKL sgemm through ctypes when it is absent)."""
    if rank != 0:
        return
    for _ in range(max(args.warmup, 1) - 1):
        pass  # warm-up happens inside cpu_gemm_sample (small call) -- each step is already seconds long
    times = []
    base = None
    for _ in range(args.steps):
        base, t = cpu_gemm_sample(reps=1)
        times.append(t)
    t_tile = sum(times) / len(times)
    gflops = 2.0 * TILE ** 3 / t_tile / 1e9
    base["value"] = gflops
    line = {
        "impl": "reference", "metric": "gemm_gflops", "value": gflops, "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_tile * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "flash::gemm sgemm 32768x32768x32768 fp32 (BASELINE.json configs[1])",
                   "sample": "each step = one 8192^3 GemmTask tile (1/64 of the job) through " + ("the reference's in_mem_gemm driver binary"
                             if base.get("kind") == "reference" else "MKL sgemm (ctypes)") + " on all host threads"},
        "cpu_baseline": base,
        "e2e": {"value": gflops, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def tf32_library_peak(torch, seconds=3.0):
    """Roofline denominator only (never on the product path): cuBLAS TF32 8192^3 via torch.matmul,
    burst = best of 10, sustained = back to back for `seconds` under the power cap -- the same
    protocol MEASURED_PEAKS.json uses for bf16, which has no TF32 entry."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.rand((n, n), device="cuda"); b = torch.rand((n, n), device="cuda")
        for _ in range(3):
            a @ b
        torch.cuda.synchronize()
        best = float("inf")
        for _ in range(10):
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record(); a @ b; e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        reps, t_end = 0, time.time() + seconds
        e0.record()
        while time.time() < t_end:
            for _ in range(25):
                a @ b
            reps += 25
            torch.cuda.synchronize()
        e1.record(); torch.cuda.synchronize()
        return {"burst": 2.0 * n ** 3 / (best * 1e-3) / 1e12,
                "sustained": 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def run_extras(args, bof, ctx, torch, dist, pk, tf32, rank, world, local):
    """All other BASELINE.json configs at this world size (collective: every rank takes part)."""
    from tools import bench_configs as bc

    pk2 = dict(pk); pk2["tf32_sustained"] = tf32["sustained"]; pk2["tf32_burst"] = tf32["burst"]
    env = bc.Env(bof, ctx, rank, world, local, pk2, dist=dist, cpu=not args.no_cpu)
    want = set(args.extra.split(","))
    extra = {}

    def guarded(name, fn):
        t0 = time.perf_counter()
        try:
            r = fn()
        except Exception as ex:  # the headline must still print
            import traceback
            r = {"error": repr(ex)[:300], "trace": traceback.format_exc()[-600:]}
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        if isinstance(r, dict):
            r["bench_seconds"] = round(time.perf_counter() - t0, 1)
        return r

    if "pcie" in want:
        extra["pcie"] = guarded("pcie", lambda: bc.pcie_bandwidth(env))
    if "cfg1" in want:
        extra["csrmm_cfg1"] = guarded("cfg1", lambda: bc.csrmm_cfg1(env))
    host_csr = None
    if "cfg3" in want or "cfg4" in want:
        t0 = time.perf_counter()
        try:
            rec, host_csr = bc.csrmm_cfg3(env, scale=args.scale)
            rec["bench_seconds"] = round(time.perf_counter() - t0, 1)
        except Exception as ex:
            import traceback
            rec = {"error": repr(ex)[:300], "trace": traceback.format_exc()[-600:]}
        extra["csrmm_cfg3"] = rec
        torch.cuda.synchronize(); torch.cuda.empty_cache()
    if "cfg4" in want and host_csr is not None:
        r = guarded("cfg4", lambda: bc.cfg4(env, host_csr, scale=args.scale))
        if "error" in r:
            extra["cfg4"] = r
        else:
            r.pop("bench_seconds", None)
            extra.update(r)
    host_csr = None
    if "cfg5" in want:
        extra["kmeans_cfg5"] = guarded("cfg5", lambda: bc.kmeans_cfg5(env, scale=args.scale))
    if "file" in want and world == 1:
        extra["e2e_file"] = guarded("file", lambda: bc.file_backed(env, scale=args.scale))
    if "pcie" in extra and "h2d_gbs_per_gpu" in extra["pcie"]:
        # out-of-core legs as multiples of the measured PCIe bound of THIS run (north_star: within 1.3x)
        h2d = extra["pcie"]["h2d_gbs_per_gpu"]
        ef = extra.get("e2e_file", {})
        if isinstance(ef.get("csrmm_cfg3"), dict) and "ms" in ef["csrmm_cfg3"]:
            ef["csrmm_cfg3"]["x_of_pcie_bound"] = ef["csrmm_cfg3"]["ms"] / ((18.723e9) / h2d / 1e6)
        if isinstance(ef.get("gemm_cfg2"), dict) and "ms" in ef["gemm_cfg2"]:
            ef["gemm_cfg2"]["x_of_pcie_or_kernel_bound"] = ef["gemm_cfg2"]["ms"] / max(8.59e9 / h2d / 1e6, 201.0)
        for key, sub in (("csrmm_cfg3", "e2e"), ("csrmm_cfg3", "e2e_shared_b"), ("csrgemv_N_cfg4", "e2e")):
            e = extra.get(key, {}).get(sub)
            if e and e.get("h2d_bytes_per_step"):
                bound_ms = e["h2d_bytes_per_step"] / h2d / 1e6
                e["pcie_h2d_bound_ms"] = bound_ms
                e["x_of_pcie_bound"] = e["ms"] / bound_ms
                both = extra["pcie"].get("both_gbs_per_gpu")
                if both:  # both directions busy at once: the host moves (h2d + d2h) bytes at the measured duplex rate
                    e["pcie_duplex_bound_ms"] = (e["h2d_bytes_per_step"] + e.get("d2h_bytes_per_step", 0)) / both / 1e6
                    e["x_of_pcie_duplex_bound"] = e["ms"] / e["pcie_duplex_bound_ms"]
    return extra


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=M_FULL, help="override m=n=k (debug only; invalid as a bench value)")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--extra", default="pcie,cfg1,cfg3,cfg4,cfg5,file", help="which other configs to measure into `extra`")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink cfg-3/4/5 (debug only; invalid as a bench value)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="leave the process on all CPUs (A/B of the NUMA binding)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write sampled rows of C from the last timed step of each gemm "
                                                          "leg as DIR/<name>.npy (fp32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as g

    bof = g.load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    # CPU baseline first: its OpenMP workers are created while the process may still run on every host core
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            cpu, _ = cpu_gemm_sample()
        except Exception as ex:
            cpu = {"value": None, "unit": "GFLOP/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex!r}"}
    from bof_b200 import dist as bdist
    cpus_before = len(os.sched_getaffinity(0))
    numa_cpus = 0 if args.no_numa_bind else bdist.bind_to_gpu_numa(local)  # pinned buffers next to this GPU's PCIe root
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pk = peaks()
    ctx = bof.Context(device=local)
    Mg = Ng = Kg = args.size
    assert Mg % world == 0
    Mr = Mg // world  # this rank's C / A rows

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident leg ------------------------------------------------------------------
    gen = torch.Generator(device="cuda"); gen.manual_seed(0x5EED0002 + rank)
    A = torch.rand((Mr, Kg), device="cuda", generator=gen)
    genb = torch.Generator(device="cuda"); genb.manual_seed(0x5EED0003)
    B = torch.rand((Kg, Ng), device="cuda", generator=genb)
    Cd = torch.empty((Mr, Ng), device="cuda")
    ws = ctx.sgemm_workspace(Mr, Ng, Kg)
    for _ in range(args.warmup):
        ctx.sgemm("R", "N", "N", Mr, Ng, Kg, 1.0, A, 0, B, 0, 0.0, Cd, 0, ws=ws)
    barrier()
    sampler = ClockSampler(local, gpu_pci_bus_id(torch, local)); sampler.start()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    kern_ms = []
    e0.record()
    for _ in range(args.steps):
        ctx.sgemm("R", "N", "N", Mr, Ng, Kg, 1.0, A, 0, B, 0, 0.0, Cd, 0, ws=ws)
    e1.record()
    barrier()
    t_dev = max_over_ranks(e0.elapsed_time(e1) * 1e-3) / args.steps
    kern_ms.append(ctx.stats().kernel_ms)  # last launch of gemm3xtf32_kernel, CUDA events on its stream
    launches_dev = ctx.launch_count() - l0
    clocks = sampler.stop()
    flops_job = 2.0 * Mg * Ng * Kg
    value = flops_job / t_dev / 1e9
    t_kernel = max_over_ranks(kern_ms[-1] * 1e-3)
    achieved = 2.0 * Mr * Ng * Kg / t_kernel / 1e12
    tf32 = tf32_library_peak(torch)
    # the kernel runs for ~0.3 s per launch under the power cap -> sustained figure; a short debug size -> burst
    long_run = t_kernel > 0.05
    tf32_peak = tf32["sustained"] if long_run else tf32["burst"]
    bf16_peak = pk["bf16_sustained"] if long_run else pk["bf16_burst"]
    # per useful flop the kernel issues one TF32 MMA flop (hi*hi) and two BF16 MMA flops (the cross terms)
    peak = 1.0 / (1.0 / tf32_peak + 2.0 / bf16_peak)
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "traffic": NCU_TRAFFIC_BYTES if world == 1 and Mg == 32768 else None,
                "kernel": "gemm3xtf32_kernel<2,EPI_GEMM,chunked,hybrid>", "kernel_ms": t_kernel * 1e3,
                "peak_note": "useful fp32 flops (2mnk) per launch against 1/(1/TF32 + 2/BF16): one tf32 MMA (hi*hi) and two "
                             f"bf16 MMAs (cross terms) per product; BF16 = MEASURED_PEAKS.json ({pk['src']}) "
                             f"{'sustained' if long_run else 'burst'} {bf16_peak:.0f}, TF32 = cuBLAS TF32 8192^3 measured in this "
                             f"run (burst {tf32['burst']:.0f}, sustained {tf32['sustained']:.0f} TFLOP/s; the file has no TF32 entry)",
                "alt_peak_3xtf32": tf32_peak / 3.0, "alt_frac_3xtf32": achieved / (tf32_peak / 3.0), "peaks_file": pk["src"]}
    # The same fractions against THIS library's own instructions: tc_issue_rate_kernel issues the product kernel's MMAs
    # (cta_group::2, 256x256 TMEM accumulator) back to back on one resident smem stage.  Burst = one 4000-round launch,
    # sustained = back-to-back launches for ~2 s (power cap).
    try:
        own = {}
        for kind, name in ((0, "tf32"), (1, "bf16"), (2, "hybrid_useful")):
            burst = ctx.tc_issue_rate(kind, 4000)[1 if kind == 2 else 0]
            t_end, vals = time.time() + 2.0, []
            while time.time() < t_end:
                vals.append(ctx.tc_issue_rate(kind, 40000)[1 if kind == 2 else 0])
            own[name] = {"burst": burst, "sustained": sum(vals[len(vals) // 2:]) / max(1, len(vals) - len(vals) // 2)}
        which = "sustained" if long_run else "burst"
        roofline["own_peaks_tflops"] = own
        roofline["frac_hybrid"] = achieved / own["hybrid_useful"][which]       # of the issue-rate ceiling of the actual MMA mix
        roofline["frac_3xtf32"] = achieved / (own["tf32"][which] / 3.0)         # SURVEY.md 8(d): TF32 peak / 3
        roofline["own_peaks_note"] = ("bof_tc_issue_rate: kind::tf32 / kind::f16(bf16) MMA flops and, for the hybrid mix, useful fp32 flops "
                                      f"(1/3 of the MMA work); fractions use the {which} figures")
    except Exception as ex:
        roofline["own_peaks_error"] = repr(ex)[:200]
    # spot check of the result on the timed buffers (cheap: 64 sampled entries in fp64)
    ii = torch.randint(0, Mr, (64,), device="cuda"); jj = torch.randint(0, Ng, (64,), device="cuda")
    ref = (A[ii].double() * B[:, jj].t().double()).sum(1)
    spot = float(((Cd[ii, jj].double() - ref).abs() / ref.abs()).max())
    dumps = {}
    if args.dump_outputs:
        rows = torch.from_numpy(dump_rows(Mr))
        dumps["gemm_C_rows"] = Cd[rows.to(Cd.device)].cpu().numpy()
    del A, B, Cd, ws
    torch.cuda.empty_cache()

    # ---- end-to-end leg: host buffers through the reference-facing entry point ------------------
    Ah = torch.empty((Mr, Kg), dtype=torch.float32, pin_memory=True)
    Bh = torch.empty((Kg, Ng), dtype=torch.float32, pin_memory=True)
    Ch = torch.empty((Mr, Ng), dtype=torch.float32, pin_memory=True)
    # fill on the GPU (host RNG over 2^30 elements would dominate the run time); B is the replicated operand:
    # every rank must hold the same values, A is this rank's shard
    for host, seed in ((Ah, 0x5EED0010 + rank), (Bh, 0x5EED0011)):
        gfill = torch.Generator(device="cuda"); gfill.manual_seed(seed)
        for r0 in range(0, host.shape[0], 4096):
            host[r0:r0 + 4096].copy_(torch.rand((min(4096, host.shape[0] - r0), host.shape[1]), device="cuda", generator=gfill))
    torch.cuda.synchronize()
    e2e_steps = args.steps
    from bof_b200 import dist as bdist
    if world > 1:
        bdist.init_comm(ctx)   # the library's own communicator rank: panel broadcasts of B on its collective stream

    def e2e_step():
        """One flash::gemm on this rank's row shard, host buffers in, host buffer out."""
        if world == 1:
            ctx.host_gemm("R", "N", "N", Mr, Ng, Kg, 1.0, 0.0, Ah, Bh, Ch)  # returns after the D2H completed
            st_ = ctx.stats()
            return st_.h2d_bytes, st_.d2h_bytes
        # N > 1: B is replicated.  bof_dist_gemm: panel j of B is uploaded by rank j % N only and pushed into every
        # peer's HBM by copy-engine peer copies over NVLink while the tensor cores work on the panels that have arrived;
        # only the A shard, 1/N of B and the C shard cross this GPU's PCIe link.
        ctx.dist_gemm("N", "N", Mr, Ng, Kg, 1.0, 0.0, Ah, Bh, Ch)
        st_ = ctx.stats()
        return st_.h2d_bytes, st_.d2h_bytes

    for _ in range(2):
        e2e_step()
    barrier()
    l1 = ctx.launch_count()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        h2d_b, d2h_b = e2e_step()
    barrier()
    t_e2e = max_over_ranks(time.perf_counter() - t0) / e2e_steps
    launches_e2e = ctx.launch_count() - l1
    e2e = {"value": flops_job / t_e2e / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": h2d_b,
           "d2h_bytes_per_step": d2h_b, "ms_per_step": t_e2e * 1e3, "steps": e2e_steps,
           "pcie_gbs": (h2d_b + d2h_b) / t_e2e / 1e9,
           "api": "bof_host_gemm (C ABI behind flash::gemm), pinned host A/B/C" if world == 1 else
                  "bof_dist_gemm (C ABI): per rank 1/N of B's column panels H2D, pushed to the peers' HBM by copy-engine peer copies "
                  "over NVLink (arrival flags, no SMs) overlapped with the MMAs, C downloaded slab by slab; pinned host A/B/C"}
    i0 = int(torch.randint(0, Mr, (1,))); j0 = int(torch.randint(0, Ng, (1,)))
    ref0 = float((Ah[i0].double() * Bh[:, j0].double()).sum())
    e2e["spot_rel_err"] = abs(float(Ch[i0, j0]) - ref0) / abs(ref0)
    if args.dump_outputs:
        dumps["host_gemm_C_rows"] = Ch[rows].numpy()
    del Ah, Bh, Ch

    torch.cuda.empty_cache()
    extra = {}
    l2 = ctx.launch_count()
    if not args.no_extra:
        extra = run_extras(args, bof, ctx, torch, dist, pk, tf32, rank, world, local)
    launches_extra = ctx.launch_count() - l2

    if "pcie" in extra and extra["pcie"].get("h2d_gbs_per_gpu"):
        pc = extra["pcie"]
        e2e["pcie_h2d_bound_ms"] = h2d_b / pc["h2d_gbs_per_gpu"] / 1e6
        e2e["pcie_duplex_bound_ms"] = (h2d_b + d2h_b) / pc["both_gbs_per_gpu"] / 1e6
        e2e["kernel_ms"] = t_kernel * 1e3
        e2e["x_of_bound"] = e2e["ms_per_step"] / max(e2e["pcie_h2d_bound_ms"], e2e["kernel_ms"])
        e2e["x_of_duplex_bound"] = e2e["ms_per_step"] / max(e2e["pcie_duplex_bound_ms"], e2e["kernel_ms"])
        e2e["bound_note"] = ("per-GPU bytes of this run / pinned-copy rates measured in this run with all ranks copying at once "
                             "(extra.pcie): H2D alone, and H2D + D2H at the both-directions rate")
    if rank == 0:
        if args.dump_outputs:
            out = Path(args.dump_outputs)
            out.mkdir(parents=True, exist_ok=True)
            for name, arr in dumps.items():
                np.save(out / f"{name}.npy", arr)
        line = {
            "metric": "gemm_gflops", "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_dev * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"flash::gemm sgemm {Mg}x{Ng}x{Kg} fp32 row-major NN alpha=1 beta=0 (BASELINE.json configs[1])",
                       "sharding": f"C/A row blocks over {world} rank(s), B replicated, no collective",
                       "arithmetic": "three-term split on tcgen05: hi*hi kind::tf32 + (lo*hi, hi*lo) on bf16 copies kind::f16, fp32 "
                                     "accumulate in TMEM folded in fp32 registers every 256 k",
                       "l2": "operands (4 GiB each) exceed the 126 MB L2; no flush needed",
                       "spot_check_max_rel_err": spot},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(launches_dev + launches_e2e + launches_extra),
            "gpu_launches_detail": {"gemm_device_leg": int(launches_dev), "gemm_e2e_leg": int(launches_e2e), "extra": int(launches_extra)},
            "host": {"cpus": cpus_before, "numa_bound_cpus": numa_cpus}, "extra": extra,
        }
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
