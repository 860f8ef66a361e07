"""16-bit layout canvases, the parts that need no GPU: the C ABI exports the bf16 / fp16 entry points, they report
size errors through the return code, and the Python layer refuses other canvas dtypes before touching a device."""
import ctypes

import pytest
import torch

from canonicalsg2im_b200 import _lib

NEW = ("csg_layout_fwd_bf16", "csg_layout_bwd_vecs_bf16", "csg_layout_bwd_geom_bf16", "csg_layout_occlude_fwd_bf16")


@pytest.fixture(scope="module")
def built():
    _lib.build()
    return _lib.load()


def test_16bit_entry_points_exported(built):
    protos = _lib.parse_header()
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in NEW:
        assert name in protos and hasattr(raw, name), name
    # void* data and a trailing int fp16 before the workspace / stream arguments
    assert protos["csg_layout_fwd_bf16"][1][6] == ctypes.c_void_p and protos["csg_layout_fwd_bf16"][1][-2] == ctypes.c_int


def test_16bit_size_error_is_reported(built):
    for fp16 in (0, 1):
        rc = built.csg_layout_fwd_bf16(0, 0, 0, 0, 0, 0, 0, 1, 6, 8, 8, 0, 0, 0, fp16, 0)    # D=6: not a multiple of 4
        assert rc != 0 and b"multiple of 4" in built.csg_last_error()


@pytest.mark.parametrize("dtype", [torch.float64, torch.int32, torch.float8_e4m3fn])
def test_other_canvas_dtypes_raise(dtype):
    from canonicalsg2im_b200 import layout as L
    v, b = torch.zeros(2, 8), torch.rand(2, 4)
    off = torch.tensor([0, 2], dtype=torch.int32)
    with pytest.raises(ValueError, match="out_dtype"):
        L.layout_batched(v, b, off, 16, out_dtype=dtype)
    with pytest.raises(ValueError, match="out_dtype"):
        L.layout_pyramid(v, b, off, 16, sizes=(8,), out_dtype=dtype)
    with pytest.raises(ValueError, match="out_dtype"):
        L.boxes_to_layout(v, b, 16, out_dtype=dtype)
    with pytest.raises(ValueError, match="out_dtype"):
        L.masks_to_layout(v, b, torch.ones(2, 4, 4), 16, out_dtype=dtype)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_cpu_tensors_still_refused(dtype):
    from canonicalsg2im_b200 import layout as L
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        L.boxes_to_layout(torch.zeros(2, 8), torch.rand(2, 4), 16, out_dtype=dtype)
