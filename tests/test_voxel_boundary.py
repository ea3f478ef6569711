"""CPU-side checks of the voxel downsampling boundary: the header's declarations of icp_gpu_voxel_downsample[_dev] compile from C, and
the ctypes bindings use the parameter lists the header declares."""
import os
import re
import subprocess
import tempfile

import pytest

from icp_variants_b200 import capi

NEW = ("icp_gpu_voxel_downsample", "icp_gpu_voxel_downsample_dev")
PARAMS = "icp_gpu_ctx*, int32_t, const float*, const float*, const uint8_t*, const int64_t*, float, int, float*, float*, uint8_t*, int64_t*"


def declaration(name):
    with open(capi.HEADER_PATH) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def c_kind(param):
    if "*" in param:
        return "ptr"
    return {"int32_t": "i32", "int64_t": "i64", "float": "C.c_float", "int": "C.c_int"}[param.split()[0]]


def test_declarations_match_the_bindings():
    assert set(NEW) <= set(capi.declared_symbols())
    want = ["ptr", "i32"] + ["ptr"] * 4 + ["C.c_float", "C.c_int"] + ["ptr"] * 4
    src = open(capi.__file__).read()
    for name in NEW:
        assert [c_kind(p) for p in declaration(name)] == want, name
        m = re.search(r'"' + name + r'": \(C\.c_int, \[([^\]]*)\]\)', src)
        assert m, name
        args = [a.strip() for a in m.group(1).split(",")]
        assert ["ptr" if a in ("vp", "pf") else a for a in args] == want, name


def test_header_compiles_from_c():
    cc = os.environ.get("CC", "cc")
    code = ('#include "icp_gpu.h"\n'
            f"int (*f)({PARAMS}) = icp_gpu_voxel_downsample;\n"
            f"int (*g)({PARAMS}) = icp_gpu_voxel_downsample_dev;\n"
            "int role_only = ICP_GPU_CLOUD_ONLY;\n")
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "t.c")
        with open(path, "w") as f:
            f.write(code)
        try:
            r = subprocess.run([cc, "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.dirname(capi.HEADER_PATH), path],
                               stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        except FileNotFoundError:
            pytest.skip(f"no C compiler ({cc})")
        assert r.returncode == 0, r.stdout
