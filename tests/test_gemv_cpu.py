"""CPU-side checks of the gemv entry points: workspace sizes follow the chunk contract, and a missing context or a bad
argument is refused without a GPU."""
import ctypes as C


def test_workspace_bytes(bof):
    lib = bof.load()
    chunk = 4096
    # one fp32 partial per (chunk of the reduction, output) plus alignment slack
    assert lib.bof_sgemv_workspace_bytes(b"R", b"N", 64, 1 << 24) == 64 * ((1 << 24) // chunk) * 4 + 256
    assert lib.bof_sgemv_workspace_bytes(b"C", b"T", 1 << 24, 64) == 64 * ((1 << 24) // chunk) * 4 + 256
    assert lib.bof_sgemv_workspace_bytes(b"R", b"T", 4097, 10) == 10 * 2 * 4 + 256
    assert lib.bof_sgemv_workspace_bytes(b"R", b"N", 0, 10) == 0
    assert lib.bof_sgemv_workspace_bytes(b"R", b"N", 10, 0) == 0
    assert lib.bof_sgemv_workspace_bytes(b"X", b"N", 10, 10) == 0


def test_null_context_is_rejected(bof):
    lib = bof.load()
    x = (C.c_float * 4)()
    assert lib.bof_host_gemv(None, b"R", b"N", 2, 2, 1.0, 0.0, x, 0, x, x) == -1
    assert lib.bof_sgemv_f32(None, None, b"R", b"N", 2, 2, 1.0, x, 0, x, 0.0, x, None, 0) == -1
    assert lib.bof_mgpu_gemv(None, b"R", b"N", 2, 2, 1.0, 0.0, x, 0, x, x) == -1
