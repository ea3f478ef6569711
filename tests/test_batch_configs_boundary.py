"""CPU-side checks of the per-configuration batch boundary: the header declares icp_gpu_iterations_bound and
icp_gpu_estimate_pose_batch_configs[_dev] with the parameter lists the ctypes bindings use, and icp_gpu_iterations_bound
follows the multi-resolution schedule of ICPOptimizer.h:503-525 (restated below) wherever the library can be loaded."""
import ctypes as C
import re

import pytest

from icp_variants_b200 import capi

NEW = ("icp_gpu_iterations_bound", "icp_gpu_estimate_pose_batch_configs", "icp_gpu_estimate_pose_batch_configs_dev")


def declaration(name):
    with open(capi.HEADER_PATH) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def c_kind(param):
    """Parameter text -> the ctypes type capi binds it with."""
    if "icp_gpu_config" in param:
        return "config"
    if "*" in param:
        return "ptr"
    return {"int32_t": "i32", "int64_t": "i64"}[param.split()[0]]


def test_declarations_match_the_bindings():
    assert set(NEW) <= set(capi.declared_symbols())
    assert [c_kind(p) for p in declaration("icp_gpu_iterations_bound")] == ["config", "i64"]
    want = ["ptr", "i32", "config", "i32"] + ["ptr"] * 12 + ["i32"]
    assert [c_kind(p) for p in declaration("icp_gpu_estimate_pose_batch_configs")] == want
    assert [c_kind(p) for p in declaration("icp_gpu_estimate_pose_batch_configs_dev")] == want
    src = open(capi.__file__).read()
    for name in NEW:
        m = re.search(r'"' + name + r'": \(C\.c_int, \[([^\]]*)\]\)', src)
        assert m, name
        args = [a.strip() for a in m.group(1).split(",")]
        kinds = ["config" if "Config" in a else "ptr" if a in ("vp", "pf") else a for a in args]
        assert kinds == [c_kind(p) for p in declaration(name)], name


def schedule_bound(n_iterations, multires, n):
    """ICPOptimizer.h:503-525: halve the size until it drops below 100, doubling the coarsest stride; one iteration per level
    above stride 1, the rest at stride 1 (:634-655)."""
    if not multires:
        return n_iterations
    res, size = 1.0, n
    while True:
        size = int(size / 2.0)
        if size < 100:
            break
        res *= 2.0
    levels, s = 1, int(res)
    while s > 1:
        s //= 2
        levels += 1
    return max(n_iterations, levels)


def test_iterations_bound_follows_the_schedule():
    try:
        capi.lib()
    except Exception as e:       # the library is not built here
        pytest.skip(f"libicp_gpu.so not loadable: {e}")
    for it in (0, 1, 3, 20):
        for mr in (0, 1):
            c = capi.default_config(); c.n_iterations, c.multires = it, mr
            got = [capi.lib().icp_gpu_iterations_bound(C.byref(c), n) for n in range(0, 100001)]
            want = [schedule_bound(it, mr, n) for n in range(0, 100001)]
            assert got == want, (it, mr)
    c = capi.default_config()
    assert capi.lib().icp_gpu_iterations_bound(None, 10) == capi.E_ARG
    assert capi.lib().icp_gpu_iterations_bound(C.byref(c), -1) == capi.E_ARG
