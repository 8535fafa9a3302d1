"""bench.py on the GPU at a small size: --steps sets the timed steps of both gemm legs, and --dump-outputs writes the
sampled rows of C that the last step computed from bench.py's seeded inputs."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import bench
import oracle

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
N = 1024


def run_bench(out, steps):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--size", str(N), "--steps", str(steps), "--warmup", "1",
                        "--no-extra", "--no-cpu", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def seeded_rand(seed):
    """An N x N operand as bench.py draws it at world size 1 (one 4096-row chunk for the host leg at this size)."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.rand((N, N), device="cuda", generator=g)


def test_steps_and_dump_outputs(tmp_path):
    d2 = run_bench(tmp_path / "a", 2)
    d3 = run_bench(tmp_path / "b", 3)
    for leg in ("gemm_device_leg", "gemm_e2e_leg"):
        l2, l3 = d2["gpu_launches_detail"][leg], d3["gpu_launches_detail"][leg]
        assert l2 > 0 and l3 * 2 == l2 * 3, (leg, l2, l3)
    rows = torch.from_numpy(bench.dump_rows(N)).cuda()
    for name, seed_a, seed_b in (("gemm_C_rows", 0x5EED0002, 0x5EED0003), ("host_gemm_C_rows", 0x5EED0010, 0x5EED0011)):
        want = (seeded_rand(seed_a)[rows].double() @ seeded_rand(seed_b).double()).cpu().numpy()
        for d in ("a", "b"):
            got = np.load(tmp_path / d / f"{name}.npy")
            assert got.dtype == np.float32 and got.shape == (bench.DUMP_ROWS, N)
            assert oracle.rel_fro(got, want) <= 1e-5, (name, d)
