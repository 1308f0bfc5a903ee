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


def test_reregistered_shapes_lay_the_arenas_out_again(monkeypatch):
    """madm_set_tensors with a new shape under a name the context knows (here the four projections' bottleneck width 128 -> 256) changes
    the model like a new name does: the arena and workspace sizes must then be those of a fresh context registered with the same tensors.
    Re-registering the same shapes at new addresses (every Engine.bind) keeps them."""
    from madm_b200 import _lib
    monkeypatch.setenv("MADM_PLAN_ONLY", "1")
    lib = _lib.load()

    def sizes(h):
        got = (lib.madm_packed_bytes(h), lib.madm_dgrad_packed_bytes(h), lib.madm_workspace_bytes(h, 8),
               lib.madm_train_workspace_bytes(h, 2, b"Depth"))
        assert all(got), (got, lib.madm_last_error(h))
        return got

    def register(h, named, base):
        arr, keep = tensor_table(named, base)
        _lib.check(lib.madm_set_tensors(h, arr, len(named)), h, "madm_set_tensors")

    named = meta_training_params()
    wide = [(n, t) for n, t in meta_training_params(proj_width=256) if n.startswith("feature_projections.")]
    merged = dict(named)
    merged.update(wide)
    merged = list(merged.items())
    h, fresh = C.c_void_p(), C.c_void_p()
    _lib.check(lib.madm_create(C.byref(h), 0), None, "madm_create")
    _lib.check(lib.madm_create(C.byref(fresh), 0), None, "madm_create")
    try:
        register(h, named, 0x1000)
        narrow = sizes(h)
        register(h, wide, 0x10000000)
        register(fresh, merged, 0x1000)
        want = sizes(fresh)
        assert want != narrow
        assert sizes(h) == want
        register(h, merged, 0x20000000)
        assert sizes(h) == want
    finally:
        lib.madm_destroy(h)
        lib.madm_destroy(fresh)
