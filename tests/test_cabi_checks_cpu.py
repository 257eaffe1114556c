"""Every C entry checks its arguments before its handle (include/gik.h: sizes, parameters, pointers, then the handle),
so each argument check answers here, with a null handle and no GPU.  x = c_void_p(8) is never dereferenced: every call
below is refused before any memory access."""
import ctypes
import math

import pytest

x = ctypes.c_void_p(8)
SIZE, NULL, PARAM, HANDLE = -2, -1, -5, -6


def _params(**kw):
    from gik_b200 import _cabi
    p = _cabi.GikParams(1e-3, 1e-2, 0.0, 1000, 0)
    for k, v in kw.items():
        setattr(p, k, v)
    return ctypes.byref(p)


# faults of the gik_params_t argument: all GIK_E_PARAM but the missing struct
PARAM_FAULTS = [(None, NULL), (_params(eps=0.0), PARAM), (_params(eps=math.nan), PARAM), (_params(dt=-1.0), PARAM),
                (_params(damping=-1.0), PARAM), (_params(max_iters=-1), PARAM), (_params(flags=1), PARAM),
                (_params(flags=2 | 4), PARAM)]

# entry -> (arguments between the handle and the stream that pass every check, faults): a fault is
# (argument index, value, code); code HANDLE marks an optional pointer (NULL is accepted, so the null handle answers)
ENTRIES = {
    "fk": ([4, x, x], [(0, -1, SIZE), (1, None, NULL), (2, None, NULL)]),
    "jac": ([4, x, x], [(0, -1, SIZE), (1, None, NULL), (2, None, NULL)]),
    "solve": ([4, x, x, _params(), x, x, x, x],
              [(0, -1, SIZE)] + [(3, p, c) for p, c in PARAM_FAULTS] +
              [(1, None, NULL), (2, None, NULL), (4, None, NULL), (5, None, NULL), (6, None, HANDLE), (7, None, HANDLE)]),
    "solve_rows": ([4, x, x, _params(), x, x, x, x, x],
                   [(0, -1, SIZE)] + [(3, p, c) for p, c in PARAM_FAULTS] +
                   [(1, None, NULL), (2, None, NULL), (4, None, NULL), (5, None, NULL), (6, None, HANDLE),
                    (7, None, HANDLE), (8, None, HANDLE)]),
    "solve_scatter": ([4, x, x, _params(), 2, (ctypes.c_void_p * 2)(8, 8), (ctypes.c_void_p * 2)(8, 8), 8, 4, x, x],
                      [(0, -1, SIZE), (4, 0, SIZE), (4, 17, SIZE), (7, -1, SIZE), (7, 7, SIZE), (8, -1, SIZE),
                       (8, 5, SIZE)] + [(3, p, c) for p, c in PARAM_FAULTS] +
                      [(1, None, NULL), (2, None, NULL), (5, None, NULL), (6, None, NULL),
                       (5, (ctypes.c_void_p * 2)(8, None), NULL), (6, (ctypes.c_void_p * 2)(None, 8), NULL),
                       (9, None, HANDLE), (10, None, HANDLE)]),
    "best_of": ([4, 2, x, x, x, x, x, x],
                [(0, -1, SIZE), (1, 0, SIZE)] + [(i, None, NULL) for i in range(2, 7)] + [(7, None, HANDLE)]),
    "project_edges": ([4, 3, x, x, x, x, _params(), x, x, x],
                      [(0, -1, SIZE), (1, -1, SIZE)] + [(6, p, c) for p, c in PARAM_FAULTS] +
                      [(i, None, NULL) for i in (2, 3, 4, 5, 7, 8)] + [(9, None, HANDLE)]),
    "collision": ([4, x, x, x], [(0, -1, SIZE), (1, None, NULL), (3, None, NULL), (2, None, HANDLE)]),
    "collision_sel": ([4, 2, x, x, x, x],
                      [(0, -1, SIZE), (1, -1, SIZE), (2, None, NULL), (3, None, NULL), (5, None, NULL),
                       (4, None, HANDLE)]),
    "clearance": ([4, x, x, 0.04, x],
                  [(0, -1, SIZE), (3, -1.0, PARAM), (3, math.nan, PARAM), (1, None, NULL), (4, None, NULL),
                   (2, None, HANDLE)]),
    "obstacle_distance": ([4, x, x, 2.0, x],
                          [(0, -1, SIZE), (3, 0.0, PARAM), (3, -1.0, PARAM), (3, math.nan, PARAM), (1, None, NULL),
                           (4, None, NULL), (2, None, HANDLE)]),
    "cube_collision": ([4, x, x], [(0, -1, SIZE), (1, None, NULL), (2, None, NULL)]),
    "solve_success": ([4, x, x, _params(), x, x, x, x, x, x],
                      [(0, -1, SIZE)] + [(3, p, c) for p, c in PARAM_FAULTS] +
                      [(i, None, NULL) for i in (1, 2, 4, 5, 6, 7, 8, 9)]),
    # n_points = 4096 with 15 free control points of dimension 15 needs more shared memory than a block gets
    "bezier_fit": ([4, 100, 15, 21] + [x] * 9,
                   [(0, -1, SIZE), (1, 0, SIZE), (2, 0, SIZE), (3, 6, SIZE), (1, 4096, SIZE)] +
                   [(i, None, NULL) for i in range(4, 13)]),
}


@pytest.mark.parametrize("sfx", ["f32", "f64"])
@pytest.mark.parametrize("entry", sorted(ENTRIES))
def test_entry_checks_its_arguments_before_the_handle(entry, sfx):
    from gik_b200 import _cabi
    f = getattr(_cabi.lib(), f"gik_{entry}_{sfx}")
    ok, faults = ENTRIES[entry]
    assert f(None, *ok, None) == HANDLE
    for i, value, code in faults:
        args = list(ok)
        args[i] = value
        assert f(None, *args, None) == code, (entry, i, value)


def test_report_helpers_check_their_arguments_before_the_handle():
    from gik_b200 import _cabi
    lib = _cabi.lib()
    b, t = ctypes.c_int32(), ctypes.c_int32()
    dims = lib.gik_solve_launch_dims
    assert dims(None, 4, 1024, ctypes.byref(b), ctypes.byref(t)) == HANDLE
    assert dims(None, 4, -1, ctypes.byref(b), ctypes.byref(t)) == SIZE
    assert dims(None, 2, 1024, ctypes.byref(b), ctypes.byref(t)) == PARAM
    assert dims(None, 8, 1024, None, ctypes.byref(t)) == NULL
    assert dims(None, 8, 1024, ctypes.byref(b), None) == NULL
    count = ctypes.c_int64(-1)
    assert lib.gik_launch_count(None, ctypes.byref(count)) == HANDLE
    assert lib.gik_launch_count(None, None) == NULL
    assert count.value == -1
