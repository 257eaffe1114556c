"""The C-ABI library builds, loads and exports every symbol include/gik.h declares (no compute calls: CPU only)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def _declared():
    src = open(os.path.join(ROOT, "include", "gik.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gik_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    from gik_b200 import _cabi
    _cabi.build()
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    names = _declared()
    assert len(names) >= 19
    for n in names:
        assert hasattr(lib, n), f"{n} declared in gik.h but not exported"
    assert sorted(_cabi.EXPORTS) == names


def test_struct_layouts_match_header():
    from gik_b200 import _cabi
    from gik_b200.model import GikTable
    assert ctypes.sizeof(_cabi.GikParams) == 32
    # nq + parent + axis (int32) are followed by doubles: 4 + 2*128 = 260 -> padded to 264
    assert GikTable.joint_R.offset == 264
    assert ctypes.sizeof(GikTable) == 264 + 8 * 32 * (9 + 3 + 1 + 1) + 8 + 8 * 2 * (9 + 3 + 9 + 3)


def test_struct_sizes_match_the_c_header(tmp_path):
    # compile sizeof() of every ABI struct from include/gik.h with the C compiler and compare with the ctypes mirrors
    import shutil
    import subprocess
    from gik_b200 import _cabi
    from gik_b200.model import GikTable
    from gik_b200.scene import GikGeom, GikScene
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "gik.h"\nint main(void){printf("%zu %zu %zu %zu\\n", sizeof(gik_table_t), '
                   'sizeof(gik_params_t), sizeof(gik_geom_t), sizeof(gik_scene_t));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    sizes = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [ctypes.sizeof(GikTable), ctypes.sizeof(_cabi.GikParams), ctypes.sizeof(GikGeom), ctypes.sizeof(GikScene)]


def test_error_codes_without_gpu():
    from gik_b200 import _cabi
    lib = _cabi.lib()
    assert lib.gik_strerror(0) == b"ok"
    assert b"null" in lib.gik_strerror(-1)
    assert lib.gik_flops_per_iter() == 3117
    assert lib.gik_bytes_per_solve(4) == 181 and lib.gik_bytes_per_solve(8) == 357
    h = ctypes.c_void_p()
    assert lib.gik_create(None, 0, ctypes.byref(h)) == -1              # GIK_E_NULL
    assert lib.gik_destroy(None) == -6                                 # GIK_E_HANDLE
    p = _cabi.GikParams()
    lib.gik_default_params(ctypes.byref(p))
    assert (p.eps, p.dt, p.damping, p.max_iters, p.flags) == (1e-3, 1e-2, 0.0, 1000, 0)
    x = ctypes.c_void_p(8)                                             # never dereferenced
    assert lib.gik_solve_f32(None, 1, x, x, ctypes.byref(p), x, x, None, None, None) == -6
    assert lib.gik_solve_f32(None, 1, None, None, None, None, None, None, None, None) == -1   # no params: checked first


def test_create_rejects_bad_tables_before_touching_cuda(table):
    import copy
    from gik_b200 import _cabi
    lib = _cabi.lib()
    h = ctypes.c_void_p()
    t = copy.deepcopy(table)
    t.axis = t.axis.copy(); t.axis[4] = 0                              # arm axis pattern broken
    assert lib.gik_create(ctypes.byref(t.to_c()), 0, ctypes.byref(h)) == -4    # GIK_E_TOPOLOGY
    t = copy.deepcopy(table)
    t.parent = t.parent.copy(); t.parent[3] = 5                        # parent listed after child
    assert lib.gik_create(ctypes.byref(t.to_c()), 0, ctypes.byref(h)) == -3    # GIK_E_MODEL


def test_product_fails_loudly_without_gpu():
    import torch
    import gik_b200
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gik_b200.GraspIK()
    with pytest.raises(RuntimeError):
        gik_b200.computeqgrasppose(None, [0.0] * 15, None, [0.33, -0.3, 0.93])
