"""The single-precision validity kernels index the distance field with 32-bit ints, so every entry point that
installs a field refuses one of 2^31 cells or more with SMPLGPU_ERR_INVALID, before it allocates or reads anything,
and leaves the context's field and verdicts as they were."""
import numpy as np
import pytest

from smpl_b200 import api, scenes

pytestmark = pytest.mark.gpu

ERR_INVALID = -1
TOO_BIG = (2048, 1024, 1024)      # exactly 2^31 cells
LARGEST = (2047, 1024, 1024)      # 2^31 - 2^20 cells: would be accepted (not installed here)


def test_fields_of_2_31_cells_are_refused():
    scene = scenes.pr2_clutter_scene()
    ctx, tables = api.setup_context(scene)
    lo, hi, cont = tables.limits()
    q = scenes.random_states(20000, lo, hi, cont, seed=71)
    before = ctx.is_states_valid(q)
    field = ctx.download_distance_field()
    L, h = ctx.L, ctx.h
    origin = np.zeros(3)
    p_origin = origin.ctypes.data_as(api.c_double_p)
    d2 = np.zeros(8, np.uint16)
    assert np.prod(TOO_BIG, dtype=np.int64) == 1 << 31 and np.prod(LARGEST, dtype=np.int64) < 1 << 31

    assert L.smplgpu_set_distance_field(h, d2.ctypes.data_as(api.c_uint16_p), *TOO_BIG, p_origin, 0.02, 100, 0.0) == ERR_INVALID
    assert L.smplgpu_build_distance_field(h, None, 0, *TOO_BIG, p_origin, 0.02, 0.4, 0.0) == ERR_INVALID
    assert L.smplgpu_build_distance_field_from_meshes(h, None, 0, None, 0, None, 0, *TOO_BIG, p_origin, 0.02, 0.4,
                                                      0.0) == ERR_INVALID
    ptr, nb = api.C.c_void_p(), api.C.c_int64()
    assert L.smplgpu_reserve_distance_field(h, *TOO_BIG, api.C.byref(ptr), api.C.byref(nb)) == ERR_INVALID
    # int overflow of the product itself
    assert L.smplgpu_build_distance_field(h, None, 0, 1 << 16, 1 << 16, 1 << 16, p_origin, 0.02, 0.4, 0.0) == ERR_INVALID

    assert np.array_equal(ctx.download_distance_field(), field)
    assert np.array_equal(ctx.is_states_valid(q), before)
    ctx.close()
