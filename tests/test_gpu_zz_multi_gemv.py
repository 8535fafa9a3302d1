"""flash::gemv over several GPUs of one process (bof_mgpu_gemv, what flash::gemv uses with BOF_GPUS > 1): the outputs are
split, never the reduction, so every world size gives the bits of one GPU.  Skipped below 2 GPUs; sorts after the other
multi-GPU file for the same reason as that one."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
NGPU = torch.cuda.device_count() if torch.cuda.is_available() else 0
need2 = pytest.mark.skipif(NGPU < 2, reason="needs at least 2 GPUs")
LAYOUTS = [("R", "N"), ("R", "T"), ("C", "N"), ("C", "T")]


def operands(ord_, trans, m, n, pad, seed):
    rng = np.random.default_rng(seed)
    rows, cols = (m, n) if ord_ == "R" else (n, m)
    buf = rng.random((rows, cols + pad), dtype=np.float32) - 0.5
    x = rng.random(n if trans == "N" else m, dtype=np.float32)
    y0 = rng.random(m if trans == "N" else n, dtype=np.float32)
    return buf, cols + pad, x, y0


@need2
@pytest.mark.parametrize("ord_,trans", LAYOUTS)
def test_mgpu_gemv_matches_one_gpu(bof, ctx, ord_, trans):
    shapes = [(5001, 7003), (3, 9000), (9000, 3), (1, 40)]   # the last has fewer outputs than GPUs for 'N'
    ref = {}
    for (m, n) in shapes:
        buf, lda, x, y0 = operands(ord_, trans, m, n, 2, m + n)
        y = y0.copy()
        ctx.host_gemv(ord_, trans, m, n, 1.5, -0.5, buf, x, y, lda=lda)
        ref[(m, n)] = y
    for world in range(2, NGPU + 1):
        with bof.MultiGpu(devices=list(range(world))) as mg:
            for (m, n) in shapes:
                buf, lda, x, y0 = operands(ord_, trans, m, n, 2, m + n)
                y = y0.copy()
                mg.gemv(ord_, trans, m, n, 1.5, -0.5, buf, x, y, lda=lda)
                assert np.array_equal(y.view(np.uint32), ref[(m, n)].view(np.uint32)), (world, m, n)


@need2
def test_gemv_driver_with_bof_gpus(ctx, tmp_path):
    import __graft_entry__ as g
    if not (ROOT / "build" / "gemv").exists():
        g.build()
    m, n = 4100, 3000
    buf, lda, x, y0 = operands("R", "T", m, n, 0, 8)
    buf.tofile(tmp_path / "A.bin"); x.tofile(tmp_path / "x.bin")
    outs = []
    for gpus in ("1", "2"):
        y0.tofile(tmp_path / "y.bin")
        r = subprocess.run([str(ROOT / "build" / "gemv"), tmp_path / "A.bin", tmp_path / "x.bin", tmp_path / "y.bin", str(m),
                            str(n), "1.0", "0.5", "T", "R", "0"], capture_output=True, text=True, timeout=600,
                           env=dict(os.environ, BOF_GPUS=gpus))
        assert r.returncode == 0 and "returned 0" in r.stdout, r.stdout + r.stderr
        outs.append((tmp_path / "y.bin").read_bytes())
    assert outs[0] == outs[1]
