"""Host-only checks of the planner's arena layouts on a device-less context (MADM_PLAN_ONLY test hook)."""
import ctypes as C

import pytest

from helpers import meta_training_params, tensor_table


@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
def test_training_layout_leaves_the_forward_arena_alone(monkeypatch, dtype):
    """The input-gradient layout is built by a LAYOUT pass of the training traversal after the caller has sized the forward arena with
    madm_packed_bytes.  Every forward-arena entry that traversal reaches must already exist (operands only the training forward uses,
    such as the natural-order ff.net.0.proj weight, live in the dgrad arena), or the caller's packed arena would be too small."""
    from madm_b200 import _lib
    monkeypatch.setenv("MADM_PLAN_ONLY", "1")
    lib = _lib.load()
    h = C.c_void_p()
    _lib.check(lib.madm_create(C.byref(h), 0), None, "madm_create")
    try:
        _lib.check(lib.madm_set_compute_dtype(h, _lib.DTYPE_FP16 if dtype == "fp16" else _lib.DTYPE_BF16), h, "dtype")
        named = meta_training_params()
        arr, keep = tensor_table(named, 0x1000)
        _lib.check(lib.madm_set_tensors(h, arr, len(named)), h, "madm_set_tensors")
        fwd = lib.madm_packed_bytes(h)
        assert fwd > 2 ** 30, (fwd, lib.madm_last_error(h))
        assert lib.madm_dgrad_packed_bytes(h) > 2 ** 30, lib.madm_last_error(h)
        assert lib.madm_packed_bytes(h) == fwd
    finally:
        lib.madm_destroy(h)
