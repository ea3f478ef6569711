"""ctypes binding of the icp_gpu_* C ABI (include/icp_gpu.h, built into lib/libicp_gpu.so).

This is the only way Python reaches the device path; there is NO CPU fallback: loading fails
loudly when the library has not been built, and creating a context fails when no B200-class
device is usable.  numpy arrays cross the boundary as plain pointers (packed float[3N] points /
normals, uint8[4N] colours, float[16] column-major poses -- the reference's
std::vector<Vector3f>/Vector4uc/Matrix4f storage).
"""
from __future__ import annotations

import ctypes as C
import os
import re
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", os.environ.get("ICP_GPU_LIB_NAME", "libicp_gpu.so"))   # the variable: A/B runs of build variants (profiles/)
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "icp_gpu.h")

OK, E_CUDA, E_ARG, E_STATE, E_NO_MATCHES, E_NUMERIC, E_PEER = 0, -1, -2, -3, -4, -5, -6
MAX_PARTIALS = 32
MAX_PEERS, PEER_HANDLE_BYTES = 8, 64
BATCH_MAX_TARGET = 8192


class IcpGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"icp_gpu error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    """icp_gpu_config -- one field per ICPOptimizer setter (ICPOptimizer.h:41-95)."""
    _fields_ = [("metric", C.c_int32), ("minimizer", C.c_int32), ("matching", C.c_int32), ("selection", C.c_int32),
                ("proba", C.c_double), ("seed", C.c_uint32), ("selection_rng", C.c_int32), ("weighting", C.c_int32),
                ("rejection", C.c_int32), ("max_distance_sq", C.c_float), ("color_icp", C.c_int32), ("multires", C.c_int32),
                ("pyramid_mode", C.c_int32), ("n_iterations", C.c_int32), ("lm_max_iterations", C.c_int32),
                ("nn_algorithm", C.c_int32), ("use_graph", C.c_int32), ("collect_stats", C.c_int32),
                ("weight_max_distance_sq", C.c_float), ("early_stop_rotation", C.c_float), ("early_stop_translation", C.c_float),
                ("reserved_", C.c_int32)]


class Timings(C.Structure):
    _fields_ = [("selection_ms", C.c_double), ("matching_ms", C.c_double), ("weighting_ms", C.c_double),
                ("rejection_ms", C.c_double), ("solver_ms", C.c_double), ("index_ms", C.c_double), ("total_ms", C.c_double),
                ("n_iterations", C.c_int32), ("n_match_launches", C.c_int32), ("n_solver_launches", C.c_int32), ("reserved_", C.c_int32),
                ("search_prep_ms", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("n_queries", C.c_uint64), ("n_matched", C.c_uint64), ("n_distance_evals", C.c_uint64),
                ("n_nodes_visited", C.c_uint64), ("n_kernel_launches", C.c_uint64), ("reduce_profile_ns", C.c_uint64 * 6)]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    csrc = os.path.join(_HERE, "csrc")
    args = ["make", "-C", csrc, "-j8"] + (["-B"] if force else [])
    r = subprocess.run(args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("building libicp_gpu.so failed")
    return LIB_PATH


def declared_symbols() -> list[str]:
    """Every function include/icp_gpu.h declares."""
    with open(HEADER_PATH) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(icp_gpu_[a-z0-9_]+)\s*\(", text)))


_lib = None


def lib():
    """The loaded C-ABI library.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback for the icp_gpu_* path)")
        L = C.CDLL(LIB_PATH)
        vp, i32, i64, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32
        pf = C.c_void_p
        sig = {
            "icp_gpu_abi_version": (C.c_int, []),
            "icp_gpu_device_count": (C.c_int, []),
            "icp_gpu_create": (C.c_int, [C.POINTER(vp), C.c_int]),
            "icp_gpu_destroy": (C.c_int, [vp]),
            "icp_gpu_last_error": (C.c_char_p, [vp]),
            "icp_gpu_set_stream": (C.c_int, [vp, vp]),
            "icp_gpu_synchronize": (C.c_int, [vp]),
            "icp_gpu_default_config": (None, [C.POINTER(Config)]),
            "icp_gpu_set_config": (C.c_int, [vp, C.POINTER(Config)]),
            "icp_gpu_get_config": (C.c_int, [vp, C.POINTER(Config)]),
            "icp_gpu_set_camera": (C.c_int, [vp, pf, u32, u32]),
            "icp_gpu_set_target": (C.c_int, [vp, pf, pf, pf, i64]),
            "icp_gpu_set_source": (C.c_int, [vp, pf, pf, pf, i64]),
            "icp_gpu_set_target_dev": (C.c_int, [vp, pf, pf, pf, i64]),
            "icp_gpu_set_source_dev": (C.c_int, [vp, pf, pf, pf, i64]),
            "icp_gpu_query_matches": (C.c_int, [vp, pf, pf, i64, pf, pf]),
            "icp_gpu_estimate_pose": (C.c_int, [vp, pf, pf, C.POINTER(i32), C.POINTER(Timings)]),
            "icp_gpu_max_iterations": (C.c_int, [vp]),
            "icp_gpu_estimate_pose_async": (C.c_int, [vp, pf]),
            "icp_gpu_estimate_pose_finish": (C.c_int, [vp, pf, pf, C.POINTER(i32)]),
            "icp_gpu_estimate_pose_batch": (C.c_int, [vp, i32, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf]),
            "icp_gpu_estimate_pose_batch_dev": (C.c_int, [vp, i32, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf]),
            "icp_gpu_iterations_bound": (C.c_int, [C.POINTER(Config), i64]),
            "icp_gpu_estimate_pose_batch_configs": (C.c_int, [vp, i32, C.POINTER(Config), i32, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, i32]),
            "icp_gpu_estimate_pose_batch_configs_dev": (C.c_int, [vp, i32, C.POINTER(Config), i32, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, i32]),
            "icp_gpu_estimate_pose_multistart": (C.c_int, [vp, i32, pf, pf, pf, pf, pf, pf, pf, pf, pf]),
            "icp_gpu_estimate_pose_multistart_dev": (C.c_int, [vp, i32, pf, pf, pf, pf, pf, pf, pf, pf, pf]),
            "icp_gpu_estimate_pose_batch_indexed": (C.c_int, [vp, i32, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, i32, pf, pf]),
            "icp_gpu_estimate_pose_batch_indexed_dev": (C.c_int, [vp, i32, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, pf, i32, pf, pf]),
            "icp_gpu_get_stats": (C.c_int, [vp, C.POINTER(Stats)]),
            "icp_gpu_measure_fp32_peak": (C.c_int, [vp, i32, C.POINTER(C.c_double)]),
            "icp_gpu_alignment_error": (C.c_int, [vp, pf, pf, C.POINTER(C.c_double)]),
            "icp_gpu_transform_points": (C.c_int, [vp, pf, pf, i64, pf]),
            "icp_gpu_transform_normals": (C.c_int, [vp, pf, pf, i64, pf]),
            "icp_gpu_apply_weights": (C.c_int, [vp, i32, C.c_float, pf, pf, pf, i64, pf, pf, pf, i64, pf, pf]),
            "icp_gpu_solve_linear": (C.c_int, [vp, i32, pf, pf, pf, pf, pf, i64, pf]),
            "icp_gpu_cloud_from_depth": (C.c_int, [vp, pf, pf, pf, pf, u32, u32, C.c_int, u32, C.c_float, C.c_int, pf, pf, pf, C.POINTER(i64)]),
            "icp_gpu_target_normals": (C.c_int, [vp, i32, pf, pf, pf]),
            "icp_gpu_voxel_downsample": (C.c_int, [vp, i32, pf, pf, pf, pf, C.c_float, C.c_int, pf, pf, pf, pf]),
            "icp_gpu_voxel_downsample_dev": (C.c_int, [vp, i32, pf, pf, pf, pf, C.c_float, C.c_int, pf, pf, pf, pf]),
            "icp_gpu_set_correspondences": (C.c_int, [vp, pf, pf, i64]),
            "icp_gpu_set_correspondences_pose": (C.c_int, [vp, pf]),
            "icp_gpu_convergence_errors": (C.c_int, [vp, pf, pf, i32, C.POINTER(i32)]),
            "icp_gpu_iteration_phases": (C.c_int, [vp]),
            "icp_gpu_iteration_begin": (C.c_int, [vp, pf]),
            "icp_gpu_iteration_local": (C.c_int, [vp, C.c_int, pf, C.POINTER(i32)]),
            "icp_gpu_iteration_apply": (C.c_int, [vp, C.c_int, pf, i32]),
            "icp_gpu_iteration_end": (C.c_int, [vp, pf]),
            "icp_gpu_iteration_local_dev": (C.c_int, [vp, C.c_int, C.POINTER(vp), C.POINTER(i32)]),
            "icp_gpu_iteration_apply_dev": (C.c_int, [vp, C.c_int]),
            "icp_gpu_peer_export": (C.c_int, [vp, pf]),
            "icp_gpu_peer_attach": (C.c_int, [vp, i32, i32, pf]),
            "icp_gpu_peer_address": (C.c_int, [vp, C.POINTER(vp)]),
            "icp_gpu_peer_attach_ptrs": (C.c_int, [vp, i32, i32, C.POINTER(vp)]),
            "icp_gpu_peer_detach": (C.c_int, [vp]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def default_config() -> Config:
    c = Config()
    lib().icp_gpu_default_config(C.byref(c))
    return c


def iterations_bound(cfg: Config, n_source: int) -> int:
    """The number of iterations estimate_pose runs at most for cfg and a source of n_source points (n_iterations, or
    max(n_iterations, pyramid levels) with multires)."""
    rc = int(lib().icp_gpu_iterations_bound(C.byref(cfg), int(n_source)))
    if rc < 0:
        raise IcpGpuError(rc, f"iterations_bound: n_source {n_source}")
    return rc


def _config_table(configs, config_index, B):
    """Sequence of Config -> (ctypes Config array, int32 [B] config_index)."""
    configs = list(configs)
    table = (Config * max(len(configs), 1))(*configs)
    ci = np.ascontiguousarray(config_index, dtype=np.int32)
    if ci.shape != (B,):
        raise ValueError(f"config_index: expected [{B}] indices, got {ci.shape}")
    return table, len(configs), ci


def best_start(inliers, rmse) -> int:
    """The start with the most inliers; ties go to the lower RMSE (NaN last), then to the lower index.  -1 for no start."""
    inl = np.asarray(inliers, np.int64)
    if len(inl) == 0:
        return -1
    r = np.asarray(rmse, np.float64)
    r = np.where(np.isnan(r), np.inf, r)
    return int(np.lexsort((np.arange(len(inl)), r, -inl))[0])


def pose_to_c(pose) -> np.ndarray:
    """4x4 (row-major numpy) -> float[16] column-major (Eigen::Matrix4f::data())."""
    return np.ascontiguousarray(np.asarray(pose, dtype=np.float32).T.reshape(16))


def pose_from_c(v) -> np.ndarray:
    return np.asarray(v, dtype=np.float32).reshape(4, 4).T.copy()


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a, cols):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] != cols:
        raise ValueError(f"expected [N,{cols}] float32, got {a.shape}")
    return a


def _u8(a):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.ndim != 2 or a.shape[1] != 4:
        raise ValueError(f"expected [N,4] uint8, got {a.shape}")
    return a


def _concat_clouds(clouds):
    """Sequence of synth.Cloud / [N,3] arrays -> (points [N,3], normals [N,3] or None, offsets [B+1] int64)."""
    pts = [_f32(getattr(c, "points", c), 3) for c in clouds]
    nrm = [getattr(c, "normals", None) for c in clouds]
    off = np.zeros(len(pts) + 1, np.int64)
    off[1:] = np.cumsum([len(p) for p in pts])
    xyz = np.concatenate(pts) if pts else np.zeros((0, 3), np.float32)
    if all(n is None for n in nrm):
        return xyz, None, off
    n3 = np.concatenate([np.zeros((len(p), 3), np.float32) if n is None else _f32(n, 3) for p, n in zip(pts, nrm)]) if pts else None
    if n3 is not None and len(n3) != len(xyz):
        raise ValueError("every cloud needs one normal per point")
    return xyz, n3, off


def _concat_clouds_rgba(clouds):
    """_concat_clouds plus the colours: (points, normals or None, colours [N,4] uint8 or None, offsets)."""
    xyz, n3, off = _concat_clouds(clouds)
    cols = [getattr(c, "colors", None) for c in clouds]
    if all(c is None for c in cols):
        return xyz, n3, None, off
    rgba = np.concatenate([np.zeros((off[b + 1] - off[b], 4), np.uint8) if c is None else _u8(c) for b, c in enumerate(cols)])
    if len(rgba) != len(xyz):
        raise ValueError("every cloud needs one colour per point")
    return xyz, n3, rgba, off


def _batch_poses(poses, B):
    """[B,4,4] row-major (None = identity) -> [B,16] column-major."""
    if poses is None:
        return np.tile(np.eye(4, dtype=np.float32).reshape(16), (B, 1))
    p = np.asarray(poses, np.float32)
    if p.shape != (B, 4, 4):
        raise ValueError(f"expected [{B},4,4] poses, got {p.shape}")
    return np.ascontiguousarray(p.transpose(0, 2, 1).reshape(B, 16))


class Context:
    """One icp_gpu_ctx: one device, one stream, device-resident clouds and loop state."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        rc = lib().icp_gpu_create(C.byref(self._h), device)
        if rc != OK:
            self._h = None
            raise IcpGpuError(rc, f"icp_gpu_create(device={device}) failed: no usable sm_100-class CUDA device (no CPU fallback)")
        self.device = device
        self.n_source = 0

    def close(self):
        if getattr(self, "_h", None):
            lib().icp_gpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc != OK:
            raise IcpGpuError(rc, lib().icp_gpu_last_error(self._h).decode())

    # -- configuration
    def set_config(self, cfg: Config):
        self._check(lib().icp_gpu_set_config(self._h, C.byref(cfg)))

    def get_config(self) -> Config:
        c = Config()
        self._check(lib().icp_gpu_get_config(self._h, C.byref(c)))
        return c

    def set_camera(self, K, width, height):
        k = np.ascontiguousarray(np.asarray(K, dtype=np.float32).T.reshape(9))   # column-major Matrix3f
        self._check(lib().icp_gpu_set_camera(self._h, _ptr(k), int(width), int(height)))

    def set_stream(self, cuda_stream: int | None):
        self._check(lib().icp_gpu_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def synchronize(self):
        self._check(lib().icp_gpu_synchronize(self._h))

    # -- clouds
    def set_target(self, xyz, nrm=None, rgba=None):
        xyz, nrm, rgba = _f32(xyz, 3), _f32(nrm, 3), _u8(rgba)
        self._check(lib().icp_gpu_set_target(self._h, _ptr(xyz), _ptr(nrm), _ptr(rgba), len(xyz)))

    def set_source(self, xyz, nrm=None, rgba=None):
        xyz, nrm, rgba = _f32(xyz, 3), _f32(nrm, 3), _u8(rgba)
        self._check(lib().icp_gpu_set_source(self._h, _ptr(xyz), _ptr(nrm), _ptr(rgba), len(xyz)))
        self.n_source = len(xyz)

    def set_target_dev(self, xyz_ptr: int, nrm_ptr: int | None, rgba_ptr: int | None, n: int):
        self._check(lib().icp_gpu_set_target_dev(self._h, C.c_void_p(xyz_ptr), C.c_void_p(nrm_ptr or 0), C.c_void_p(rgba_ptr or 0), n))

    def set_source_dev(self, xyz_ptr: int, nrm_ptr: int | None, rgba_ptr: int | None, n: int):
        self._check(lib().icp_gpu_set_source_dev(self._h, C.c_void_p(xyz_ptr), C.c_void_p(nrm_ptr or 0), C.c_void_p(rgba_ptr or 0), n))
        self.n_source = n

    # -- stages 2-4 at a given pose
    def query_matches(self, pose, sel_idx=None):
        sel = None if sel_idx is None else np.ascontiguousarray(sel_idx, dtype=np.int32)
        n = self.n_source if sel is None else len(sel)
        idx = np.empty(n, np.int32)
        w = np.empty(n, np.float32)
        p = pose_to_c(pose)
        self._check(lib().icp_gpu_query_matches(self._h, _ptr(p), _ptr(sel), n, _ptr(idx), _ptr(w)))
        return idx, w

    # -- the loop
    def max_iterations(self) -> int:
        return int(lib().icp_gpu_max_iterations(self._h))

    def estimate_pose(self, init_pose=None, want_history=True, timings: bool = False):
        """Returns (pose 4x4, history [iters,4,4] or None, n_iterations[, Timings])."""
        p = pose_to_c(np.eye(4, dtype=np.float32) if init_pose is None else init_pose).copy()
        cap = max(self.max_iterations(), 1)
        hist = np.zeros((cap, 16), np.float32) if want_history else None
        n_it = C.c_int32(0)
        tm = Timings() if timings else None
        rc = lib().icp_gpu_estimate_pose(self._h, _ptr(p), _ptr(hist), C.byref(n_it), C.byref(tm) if timings else None)
        if rc != OK:
            err = IcpGpuError(rc, lib().icp_gpu_last_error(self._h).decode())
            err.pose = pose_from_c(p)
            err.n_iterations = n_it.value
            raise err
        h = None
        if want_history:
            h = np.stack([pose_from_c(hist[i]) for i in range(n_it.value)]) if n_it.value else np.zeros((0, 4, 4), np.float32)
        out = (pose_from_c(p), h, n_it.value)
        return out + (tm,) if timings else out

    def estimate_pose_async(self, init_pose=None):
        p = pose_to_c(np.eye(4, dtype=np.float32) if init_pose is None else init_pose)
        self._check(lib().icp_gpu_estimate_pose_async(self._h, _ptr(p)))

    def estimate_pose_finish(self):
        p = np.empty(16, np.float32)
        n_it = C.c_int32(0)
        self._check(lib().icp_gpu_estimate_pose_finish(self._h, _ptr(p), None, C.byref(n_it)))
        return pose_from_c(p), n_it.value

    # -- many small registrations in one launch (one thread block per pair)
    def estimate_pose_batch(self, sources, targets, init_poses=None, want_history=False):
        """B independent registrations with the context's configuration.  sources / targets: sequences of synth.Cloud or
        [N,3] point arrays (no normals = zero normals); init_poses: [B,4,4] or None (identity).  Returns (poses [B,4,4],
        n_iterations [B], status [B] (OK / E_NO_MATCHES / E_NUMERIC per pair)[, history [B, n_iterations, 4, 4], rows past
        a pair's last iteration 0]).  A pair whose target has more than BATCH_MAX_TARGET points is refused (E_ARG)."""
        if len(sources) != len(targets):
            raise ValueError(f"{len(sources)} sources, {len(targets)} targets")
        B = len(sources)
        sp, sn, so = _concat_clouds(sources)
        tp, tn, to = _concat_clouds(targets)
        pin = _batch_poses(init_poses, B)
        pout = np.zeros((B, 16), np.float32)
        n_it = np.zeros(B, np.int32)
        status = np.zeros(B, np.int32)
        n_cap = self.get_config().n_iterations
        hist = np.zeros((B, n_cap, 16), np.float32) if want_history else None
        self._check(lib().icp_gpu_estimate_pose_batch(self._h, B, _ptr(sp), _ptr(sn), _ptr(so), _ptr(tp), _ptr(tn), _ptr(to), _ptr(pin), _ptr(pout),
                                                      _ptr(n_it), _ptr(status), _ptr(hist)))
        out = (pout.reshape(B, 4, 4).transpose(0, 2, 1).copy(), n_it, status)
        return out + (hist.reshape(B, n_cap, 4, 4).transpose(0, 1, 3, 2).copy(),) if want_history else out

    def estimate_pose_batch_dev(self, src_xyz, src_off, tgt_xyz, tgt_off, src_nrm=None, tgt_nrm=None, init_poses=None, want_history=False):
        """The same on CUDA torch tensors of the context's device, without a host round trip of the clouds: concatenated
        points / normals [N,3] float32, offsets [B+1] int64, init_poses [B,4,4] float32 (None = identity).  Returns CUDA
        tensors (poses [B,4,4], n_iterations [B] int32, status [B] int32[, history [B, n_iterations, 4, 4]]).  Work queued on
        the current torch stream is waited for; the results are complete when the call returns."""
        import torch
        dev = torch.device("cuda", self.device)

        def run(sp, sn, so, tp, tn, to, pin, pout, n_it, status, p):
            hist = torch.empty((len(so) - 1, self.get_config().n_iterations, 4, 4), dtype=torch.float32, device=dev) if want_history else None
            self._check(lib().icp_gpu_estimate_pose_batch_dev(self._h, len(so) - 1, p(sp), p(sn), p(so), p(tp), p(tn), p(to), p(pin), p(pout), p(n_it),
                                                              p(status), p(hist)))
            return hist

        return self._batch_dev(run, src_xyz, src_off, tgt_xyz, tgt_off, src_nrm, tgt_nrm, init_poses)

    def _batch_dev(self, run, src_xyz, src_off, tgt_xyz, tgt_off, src_nrm, tgt_nrm, init_poses):
        """Checks and lays out the torch operands of the _dev batch forms; run(...) makes the call and returns the history or None."""
        import torch
        dev = torch.device("cuda", self.device)

        def arr(x, name, cols):
            if x is None:
                return None
            if not (isinstance(x, torch.Tensor) and x.device == dev and x.dtype == torch.float32 and x.dim() == 2 and x.shape[1] == cols):
                raise ValueError(f"{name}: expected a float32 [N,{cols}] tensor on {dev}")
            return x.contiguous()

        def offs(x, name):
            if not (isinstance(x, torch.Tensor) and x.device == dev and x.dtype == torch.int64 and x.dim() == 1 and len(x) >= 1):
                raise ValueError(f"{name}: expected an int64 [B+1] tensor on {dev}")
            return x.contiguous()

        sp, tp = arr(src_xyz, "src_xyz", 3), arr(tgt_xyz, "tgt_xyz", 3)
        sn, tn = arr(src_nrm, "src_nrm", 3), arr(tgt_nrm, "tgt_nrm", 3)
        so, to = offs(src_off, "src_off"), offs(tgt_off, "tgt_off")
        if len(so) != len(to):
            raise ValueError(f"{len(so) - 1} source pairs, {len(to) - 1} target pairs")
        for x, n, name in ((sn, len(sp), "src_nrm"), (tn, len(tp), "tgt_nrm")):
            if x is not None and len(x) != n:
                raise ValueError(f"{name}: {len(x)} rows for {n} points")
        ends = torch.stack([so[-1], to[-1]]).tolist()
        if ends != [len(sp), len(tp)]:
            raise IcpGpuError(E_ARG, f"batch: the offsets end at {ends[0]} / {ends[1]}, the clouds hold {len(sp)} / {len(tp)} points")
        B = len(so) - 1
        if init_poses is None:
            pin = torch.eye(4, dtype=torch.float32, device=dev).expand(B, 4, 4)
        else:
            pin = init_poses
            if not (isinstance(pin, torch.Tensor) and pin.device == dev and pin.dtype == torch.float32 and tuple(pin.shape) == (B, 4, 4)):
                raise ValueError(f"init_poses: expected a float32 [{B},4,4] tensor on {dev}")
        pin = pin.transpose(1, 2).contiguous()               # column-major per pose (Eigen::Matrix4f::data())
        pout = torch.empty((B, 4, 4), dtype=torch.float32, device=dev)
        n_it = torch.empty(B, dtype=torch.int32, device=dev)
        status = torch.empty(B, dtype=torch.int32, device=dev)

        def p(x):
            return None if x is None else C.c_void_p(x.data_ptr())

        torch.cuda.current_stream(dev).synchronize()
        hist = run(sp, sn, so, tp, tn, to, pin, pout, n_it, status, p)
        out = (pout.transpose(1, 2).contiguous(), n_it, status)
        return out + (hist.transpose(2, 3).contiguous(),) if hist is not None else out

    def estimate_pose_batch_configs(self, configs, config_index, sources, targets, init_poses=None, want_history=False):
        """B independent registrations, pair b with configs[config_index[b]] (the context's own configuration is not used).
        Clouds and poses as estimate_pose_batch.  Returns (poses [B,4,4], n_iterations [B], status [B][, history [B, R, 4, 4]]),
        R = the largest iterations_bound of the batch's pairs, rows past a pair's last iteration 0."""
        if len(sources) != len(targets):
            raise ValueError(f"{len(sources)} sources, {len(targets)} targets")
        B = len(sources)
        table, n_cfg, ci = _config_table(configs, config_index, B)
        sp, sn, so = _concat_clouds(sources)
        tp, tn, to = _concat_clouds(targets)
        pin = _batch_poses(init_poses, B)
        pout = np.zeros((B, 16), np.float32)
        n_it = np.zeros(B, np.int32)
        status = np.zeros(B, np.int32)
        rows = 0
        if want_history:
            rows = max([iterations_bound(table[int(k)], so[b + 1] - so[b]) for b, k in enumerate(ci) if 0 <= k < n_cfg] + [0])
        hist = np.zeros((B, rows, 16), np.float32) if want_history else None
        self._check(lib().icp_gpu_estimate_pose_batch_configs(self._h, n_cfg, table, B, _ptr(ci), _ptr(sp), _ptr(sn), _ptr(so), _ptr(tp), _ptr(tn),
                                                              _ptr(to), _ptr(pin), _ptr(pout), _ptr(n_it), _ptr(status), _ptr(hist) if rows else None,
                                                              rows))
        out = (pout.reshape(B, 4, 4).transpose(0, 2, 1).copy(), n_it, status)
        return out + (hist.reshape(B, rows, 4, 4).transpose(0, 1, 3, 2).copy(),) if want_history else out

    def estimate_pose_batch_configs_dev(self, configs, config_index, src_xyz, src_off, tgt_xyz, tgt_off, src_nrm=None, tgt_nrm=None,
                                        init_poses=None, want_history=False):
        """The same on CUDA torch tensors of the context's device, shaped as estimate_pose_batch_dev's; config_index: an int32 [B]
        tensor on the device, configs: a sequence of Config (host).  Returns CUDA tensors (poses [B,4,4], n_iterations [B],
        status [B][, history [B, R, 4, 4]])."""
        import torch
        dev = torch.device("cuda", self.device)
        B = len(src_off) - 1
        if not (isinstance(config_index, torch.Tensor) and config_index.device == dev and config_index.dtype == torch.int32
                and tuple(config_index.shape) == (B,)):
            raise ValueError(f"config_index: expected an int32 [{B}] tensor on {dev}")
        table, n_cfg, _ = _config_table(configs, np.zeros(B, np.int32), B)
        ci = config_index.contiguous()
        rows = 0
        if want_history:
            ns = (src_off[1:] - src_off[:-1]).tolist()
            rows = max([iterations_bound(table[int(k)], n) for k, n in zip(ci.tolist(), ns) if 0 <= k < n_cfg] + [0])

        def run(sp, sn, so, tp, tn, to, pin, pout, n_it, status, p):
            hist = torch.zeros((B, rows, 4, 4), dtype=torch.float32, device=dev) if want_history else None
            self._check(lib().icp_gpu_estimate_pose_batch_configs_dev(self._h, n_cfg, table, B, p(ci), p(sp), p(sn), p(so), p(tp), p(tn), p(to),
                                                                      p(pin), p(pout), p(n_it), p(status), p(hist) if rows else None, rows))
            return hist

        return self._batch_dev(run, src_xyz, src_off, tgt_xyz, tgt_off, src_nrm, tgt_nrm, init_poses)

    # -- many starts of the context's own pair in one launch
    def estimate_pose_multistart(self, init_poses, want_history=False, want_matches=False):
        """K registrations of the context's source against its target from the initial poses init_poses [K,4,4], each scored at
        its final pose.  Returns a dict: poses [K,4,4], n_iterations [K], status [K] (OK / E_NO_MATCHES / E_NUMERIC per start),
        inliers [K] int64, rmse [K] float64 (NaN without an inlier), best (the start with the most inliers, ties to the lower RMSE,
        then the lower index; -1 when K = 0), and with want_history history [K, max_iterations, 4, 4] (rows past a start's last
        iteration 0), with want_matches match_idx / match_w [K, n_source] (query_matches at each final pose)."""
        p = np.asarray(init_poses, np.float32)
        if p.ndim != 3 or p.shape[1:] != (4, 4):
            raise ValueError(f"init_poses: expected [K,4,4], got {p.shape}")
        K, n = len(p), self.n_source
        pin = np.ascontiguousarray(p.transpose(0, 2, 1).reshape(K, 16))
        pout = np.zeros((K, 16), np.float32)
        n_it = np.zeros(K, np.int32)
        status = np.zeros(K, np.int32)
        inl = np.zeros(K, np.int64)
        rmse = np.zeros(K, np.float64)
        rows = max(self.max_iterations(), 0)
        hist = np.zeros((K, max(rows, 1), 16), np.float32) if want_history else None
        midx = np.zeros((K, max(n, 1)), np.int32) if want_matches else None
        mw = np.zeros((K, max(n, 1)), np.float32) if want_matches else None
        self._check(lib().icp_gpu_estimate_pose_multistart(self._h, K, _ptr(pin), _ptr(pout), _ptr(n_it), _ptr(status), _ptr(inl), _ptr(rmse),
                                                           _ptr(hist), _ptr(midx), _ptr(mw)))
        out = {"poses": pout.reshape(K, 4, 4).transpose(0, 2, 1).copy(), "n_iterations": n_it, "status": status, "inliers": inl,
               "rmse": rmse, "best": best_start(inl, rmse)}
        if want_history:
            out["history"] = hist[:, :rows].reshape(K, rows, 4, 4).transpose(0, 1, 3, 2).copy()
        if want_matches:
            out["match_idx"], out["match_w"] = midx[:, :n].copy(), mw[:, :n].copy()
        return out

    def estimate_pose_multistart_dev(self, init_poses, want_history=False, want_matches=False):
        """The same on CUDA torch tensors of the context's device: init_poses a float32 [K,4,4] tensor; the dict's arrays are CUDA
        tensors (best a Python int).  Work queued on the current torch stream is waited for; the results are complete when the
        call returns."""
        import torch
        dev = torch.device("cuda", self.device)
        if not (isinstance(init_poses, torch.Tensor) and init_poses.device == dev and init_poses.dtype == torch.float32
                and init_poses.dim() == 3 and tuple(init_poses.shape[1:]) == (4, 4)):
            raise ValueError(f"init_poses: expected a float32 [K,4,4] tensor on {dev}")
        K, n = init_poses.shape[0], self.n_source
        pin = init_poses.transpose(1, 2).contiguous()         # column-major per pose (Eigen::Matrix4f::data())
        pout = torch.empty((K, 4, 4), dtype=torch.float32, device=dev)
        n_it = torch.empty(K, dtype=torch.int32, device=dev)
        status = torch.empty(K, dtype=torch.int32, device=dev)
        inl = torch.empty(K, dtype=torch.int64, device=dev)
        rmse = torch.empty(K, dtype=torch.float64, device=dev)
        rows = max(self.max_iterations(), 0)
        hist = torch.zeros((K, max(rows, 1), 4, 4), dtype=torch.float32, device=dev) if want_history else None
        midx = torch.empty((K, max(n, 1)), dtype=torch.int32, device=dev) if want_matches else None
        mw = torch.empty((K, max(n, 1)), dtype=torch.float32, device=dev) if want_matches else None

        def p(x):
            return None if x is None else C.c_void_p(x.data_ptr())

        torch.cuda.current_stream(dev).synchronize()
        self._check(lib().icp_gpu_estimate_pose_multistart_dev(self._h, K, p(pin), p(pout), p(n_it), p(status), p(inl), p(rmse), p(hist),
                                                               p(midx), p(mw)))
        out = {"poses": pout.transpose(1, 2).contiguous(), "n_iterations": n_it, "status": status, "inliers": inl, "rmse": rmse,
               "best": best_start(inl.cpu().numpy(), rmse.cpu().numpy())}
        if want_history:
            out["history"] = hist[:, :rows].transpose(2, 3).contiguous()
        if want_matches:
            out["match_idx"], out["match_w"] = midx[:, :n], mw[:, :n]
        return out

    # -- many pairs of any size, each against its own index, in one launch
    def estimate_pose_batch_indexed(self, sources, targets, init_poses=None, want_history=False, want_matches=False):
        """B independent registrations with the context's configuration, every target indexed in the call, pairs of any size.
        sources / targets: sequences of synth.Cloud (points, optional normals and colours) or [N,3] point arrays; init_poses:
        [B,4,4] or None (identity).  Returns the dict of estimate_pose_multistart with one row per pair: poses, n_iterations,
        status, inliers, rmse, best, and with want_history history [B, R, 4, 4] (R = the largest iterations_bound of the batch's
        sources, rows past a pair's last iteration 0), with want_matches match_idx / match_w: one array per pair (query_matches at
        its final pose).  The context's own clouds and state are left as they are."""
        if len(sources) != len(targets):
            raise ValueError(f"{len(sources)} sources, {len(targets)} targets")
        B = len(sources)
        sp, sn, sc, so = _concat_clouds_rgba(sources)
        tp, tn, tc, to = _concat_clouds_rgba(targets)
        pin = _batch_poses(init_poses, B)
        pout = np.zeros((B, 16), np.float32)
        n_it = np.zeros(B, np.int32)
        status = np.zeros(B, np.int32)
        inl = np.zeros(B, np.int64)
        rmse = np.zeros(B, np.float64)
        cfg = self.get_config()
        rows = max([iterations_bound(cfg, so[b + 1] - so[b]) for b in range(B)] + [0]) if want_history else 0
        hist = np.zeros((B, max(rows, 1), 16), np.float32) if want_history else None
        ns = int(so[-1])
        midx = np.zeros(max(ns, 1), np.int32) if want_matches else None
        mw = np.zeros(max(ns, 1), np.float32) if want_matches else None
        self._check(lib().icp_gpu_estimate_pose_batch_indexed(self._h, B, _ptr(sp), _ptr(sn), _ptr(sc), _ptr(so), _ptr(tp), _ptr(tn), _ptr(tc), _ptr(to),
                                                              _ptr(pin), _ptr(pout), _ptr(n_it), _ptr(status), _ptr(inl), _ptr(rmse), _ptr(hist), rows,
                                                              _ptr(midx), _ptr(mw)))
        out = {"poses": pout.reshape(B, 4, 4).transpose(0, 2, 1).copy(), "n_iterations": n_it, "status": status, "inliers": inl,
               "rmse": rmse, "best": best_start(inl, rmse)}
        if want_history:
            out["history"] = hist[:, :rows].reshape(B, rows, 4, 4).transpose(0, 1, 3, 2).copy()
        if want_matches:
            out["match_idx"] = [midx[so[b]:so[b + 1]].copy() for b in range(B)]
            out["match_w"] = [mw[so[b]:so[b + 1]].copy() for b in range(B)]
        return out

    def estimate_pose_batch_indexed_dev(self, src_xyz, src_off, tgt_xyz, tgt_off, src_nrm=None, tgt_nrm=None, src_rgba=None, tgt_rgba=None,
                                        init_poses=None, want_history=False, want_matches=False):
        """The same on CUDA torch tensors of the context's device: concatenated points / normals [N,3] float32, colours [N,4] uint8,
        offsets [B+1] int64, init_poses [B,4,4] float32 (None = identity).  Returns the dict with CUDA tensors (best a Python int);
        match_idx / match_w are [sum n_src] tensors in each pair's original order, pair b's at src_off[b].  Work queued on the
        current torch stream is waited for; the results are complete when the call returns."""
        import torch
        dev = torch.device("cuda", self.device)

        def rgba(x, name, n):
            if x is None:
                return None
            if not (isinstance(x, torch.Tensor) and x.device == dev and x.dtype == torch.uint8 and tuple(x.shape) == (n, 4)):
                raise ValueError(f"{name}: expected a uint8 [{n},4] tensor on {dev}")
            return x.contiguous()

        sc, tc = rgba(src_rgba, "src_rgba", len(src_xyz)), rgba(tgt_rgba, "tgt_rgba", len(tgt_xyz))
        cfg = self.get_config()
        res = {}

        def run(sp, sn, so, tp, tn, to, pin, pout, n_it, status, p):
            B = len(so) - 1
            ns = int(so[-1]) if B > 0 else 0
            inl = torch.empty(B, dtype=torch.int64, device=dev)
            rmse = torch.empty(B, dtype=torch.float64, device=dev)
            rows = 0
            if want_history:
                rows = max([iterations_bound(cfg, n) for n in (so[1:] - so[:-1]).tolist()] + [0])
            hist = torch.zeros((B, max(rows, 1), 4, 4), dtype=torch.float32, device=dev) if want_history else None
            midx = torch.empty(max(ns, 1), dtype=torch.int32, device=dev) if want_matches else None
            mw = torch.empty(max(ns, 1), dtype=torch.float32, device=dev) if want_matches else None
            self._check(lib().icp_gpu_estimate_pose_batch_indexed_dev(self._h, B, p(sp), p(sn), p(sc), p(so), p(tp), p(tn), p(tc), p(to), p(pin), p(pout),
                                                                      p(n_it), p(status), p(inl), p(rmse), p(hist), rows, p(midx), p(mw)))
            res.update(inliers=inl, rmse=rmse, best=best_start(inl.cpu().numpy(), rmse.cpu().numpy()))
            if want_matches:
                res.update(match_idx=midx[:ns], match_w=mw[:ns])
            return hist[:, :rows] if want_history else None

        out = self._batch_dev(run, src_xyz, src_off, tgt_xyz, tgt_off, src_nrm, tgt_nrm, init_poses)
        res.update(poses=out[0], n_iterations=out[1], status=out[2])
        if want_history:
            res["history"] = out[3]
        return res

    def cloud_from_depth(self, depth, rgbx, K, extrinsics=None, keep_original_size=False, downsample=1, max_distance=0.1,
                         role: int = 2, download: bool = True):
        """PointCloud(depthMap, colorFrame, ...) (PointCloud.h:78-165) on the device.  role 0: the cloud becomes the
        target (buildIndex), 1: the source, 2: only returned.  Returns (points, normals, colours) or the point count."""
        depth = np.ascontiguousarray(depth, np.float32); h, w = depth.shape
        col = None if rgbx is None else np.ascontiguousarray(rgbx, np.uint8).reshape(-1)
        if col is not None and col.size < h * w + 3:
            raise ValueError("rgbx must hold the RGBX frame (4*w*h bytes)")
        Kc = np.ascontiguousarray(np.asarray(K, np.float32).T.reshape(9))
        Ec = None if extrinsics is None else pose_to_c(extrinsics)
        cap = (h * w + downsample - 1) // downsample if downsample > 0 else h * w
        n = C.c_int64(0)
        if download:
            po = np.empty((cap, 3), np.float32); no = np.empty((cap, 3), np.float32); co = np.empty((cap, 4), np.uint8)
        else:
            po = no = co = None
        self._check(lib().icp_gpu_cloud_from_depth(self._h, _ptr(depth), _ptr(col), _ptr(Kc), _ptr(Ec), w, h, int(keep_original_size),
                                                   int(downsample), float(max_distance), int(role), _ptr(po), _ptr(no), _ptr(co), C.byref(n)))
        if not download:
            return n.value
        return po[:n.value].copy(), no[:n.value].copy(), co[:n.value].copy()

    def voxel_downsample(self, xyz, voxel_size, nrm=None, rgba=None, role: int = 2):
        """Voxel-grid filter of one cloud on the device (icp_gpu_voxel_downsample): one centroid per occupied voxel of edge
        voxel_size.  role 0: the result becomes the target (indexed), 1: the source, 2: only returned.  Returns (points [M,3],
        normals [M,3] or None, colours [M,4] uint8 or None)."""
        xyz, nrm, rgba = _f32(xyz, 3), _f32(nrm, 3), _u8(rgba)
        for x, name in ((nrm, "nrm"), (rgba, "rgba")):
            if x is not None and len(x) != len(xyz):
                raise ValueError(f"{name}: {len(x)} rows for {len(xyz)} points")
        off = np.array([0, len(xyz)], np.int64)
        out = self._voxel_host(xyz, nrm, rgba, off, voxel_size, role)
        if role == 1:
            self.n_source = len(out[0])
        return out[:3]

    def voxel_downsample_batch(self, clouds, voxel_size):
        """The filter of many clouds in one call (synth.Cloud or [N,3] arrays, optional normals and colours): a list of clouds
        (points, normals or None, colours or None), in the order given."""
        xyz, n3, c4, off = _concat_clouds_rgba(clouds)
        po, no, co, oo = self._voxel_host(xyz, n3, c4, off, voxel_size, 2)
        return [(po[oo[b]:oo[b + 1]], None if no is None else no[oo[b]:oo[b + 1]], None if co is None else co[oo[b]:oo[b + 1]])
                for b in range(len(off) - 1)]

    def _voxel_host(self, xyz, nrm, rgba, off, voxel_size, role):
        cap = max(int(off[-1]), 1)
        po = np.empty((cap, 3), np.float32)
        no = np.empty((cap, 3), np.float32) if nrm is not None else None
        co = np.empty((cap, 4), np.uint8) if rgba is not None else None
        oo = np.zeros(len(off), np.int64)
        self._check(lib().icp_gpu_voxel_downsample(self._h, len(off) - 1, _ptr(xyz), _ptr(nrm), _ptr(rgba), _ptr(off), float(voxel_size), int(role),
                                                   _ptr(po), _ptr(no), _ptr(co), _ptr(oo)))
        m = int(oo[-1])
        return po[:m].copy(), None if no is None else no[:m].copy(), None if co is None else co[:m].copy(), oo

    def voxel_downsample_dev(self, xyz, off, voxel_size, nrm=None, rgba=None, role: int = 2):
        """The filter on CUDA torch tensors of the context's device: concatenated points / normals [N,3] float32, colours [N,4] uint8,
        offsets [B+1] int64.  Returns (points [M,3], normals or None, colours or None, offsets [B+1] int64), CUDA tensors, cloud b's
        voxels at [off_out[b], off_out[b+1]).  Work queued on the current torch stream is waited for; the results are complete when
        the call returns."""
        import torch
        dev = torch.device("cuda", self.device)

        def arr(x, name, dtype, cols):
            if x is None:
                return None
            if not (isinstance(x, torch.Tensor) and x.device == dev and x.dtype == dtype and x.dim() == 2 and x.shape[1] == cols):
                raise ValueError(f"{name}: expected a {dtype} [N,{cols}] tensor on {dev}")
            return x.contiguous()

        xyz, nrm, rgba = arr(xyz, "xyz", torch.float32, 3), arr(nrm, "nrm", torch.float32, 3), arr(rgba, "rgba", torch.uint8, 4)
        if not (isinstance(off, torch.Tensor) and off.device == dev and off.dtype == torch.int64 and off.dim() == 1 and len(off) >= 1):
            raise ValueError(f"off: expected an int64 [B+1] tensor on {dev}")
        off = off.contiguous()
        for x, name in ((nrm, "nrm"), (rgba, "rgba")):
            if x is not None and len(x) != len(xyz):
                raise ValueError(f"{name}: {len(x)} rows for {len(xyz)} points")
        cap = max(len(xyz), 1)
        po = torch.empty((cap, 3), dtype=torch.float32, device=dev)
        no = torch.empty((cap, 3), dtype=torch.float32, device=dev) if nrm is not None else None
        co = torch.empty((cap, 4), dtype=torch.uint8, device=dev) if rgba is not None else None
        oo = torch.zeros(len(off), dtype=torch.int64, device=dev)

        def p(x):
            return None if x is None else C.c_void_p(x.data_ptr())

        torch.cuda.current_stream(dev).synchronize()
        self._check(lib().icp_gpu_voxel_downsample_dev(self._h, len(off) - 1, p(xyz), p(nrm), p(rgba), p(off), float(voxel_size), int(role),
                                                       p(po), p(no), p(co), p(oo)))
        m = int(oo[-1]) if len(off) > 1 else 0
        if role == 1:
            self.n_source = m
        return po[:m], None if no is None else no[:m], None if co is None else co[:m], oo

    def target_normals(self, k: int = 5, viewpoint=None, n: int | None = None, curvature: bool = False):
        """PointCloud(pcl cloud) (PointCloud.h:41-76): k-NN PCA normals of the resident target (n = its size); they also
        replace the target's normals on the device.  Returns normals [n,3] (and curvature [n])."""
        if n is None:
            raise ValueError("pass n = number of target points")
        vp = None if viewpoint is None else np.ascontiguousarray(viewpoint, np.float32)
        nrm = np.empty((n, 3), np.float32); cur = np.empty(n, np.float32) if curvature else None
        self._check(lib().icp_gpu_target_normals(self._h, int(k), _ptr(vp), _ptr(nrm), _ptr(cur)))
        return (nrm, cur) if curvature else nrm

    def set_correspondences(self, src_xyz, ref_xyz):
        s = _f32(src_xyz, 3); r = _f32(ref_xyz, 3)
        assert len(s) == len(r)
        self._check(lib().icp_gpu_set_correspondences(self._h, _ptr(s), _ptr(r), len(s)))

    def set_correspondences_pose(self, gt_pose):
        """Every point of the resident source against itself under a ground-truth pose (main.cpp:300-307)."""
        self._check(lib().icp_gpu_set_correspondences_pose(self._h, _ptr(pose_to_c(gt_pose))))

    def alignment_error(self, pose, benchmark: bool = False):
        """(rmse, benchmark error | None) of one pose over the correspondences set before (ConvergenceMeasure.h:50-66, :104-151)."""
        r = np.zeros(1, np.float32); b = C.c_double(0.0)
        self._check(lib().icp_gpu_alignment_error(self._h, _ptr(pose_to_c(pose)), _ptr(r), C.byref(b) if benchmark else None))
        return float(r[0]), (float(b.value) if benchmark else None)

    def convergence_errors(self, benchmark: bool = False):
        """(rmse per iteration, benchmark error per iteration | None) of the last registration, computed on the device."""
        cap = self.max_iterations()
        rm = np.zeros(cap, np.float32); be = np.zeros(cap, np.float64) if benchmark else None
        n = C.c_int32(0)
        self._check(lib().icp_gpu_convergence_errors(self._h, _ptr(rm), _ptr(be), cap, C.byref(n)))
        return rm[:n.value].copy(), (be[:n.value].copy() if benchmark else None)

    # -- the reference API's value-level operations (utils.h, weighting.h, ProcrustesAligner.h / the linear solvers)
    def transform_points(self, pose, xyz):
        p = _f32(xyz, 3); out = np.empty_like(p)
        self._check(lib().icp_gpu_transform_points(self._h, _ptr(pose_to_c(pose)), _ptr(p), len(p), _ptr(out)))
        return out

    def transform_normals(self, pose, nrm):
        p = _f32(nrm, 3); out = np.empty_like(p)
        self._check(lib().icp_gpu_transform_normals(self._h, _ptr(pose_to_c(pose)), _ptr(p), len(p), _ptr(out)))
        return out

    def apply_weights(self, weighting, max_distance_sq, src_xyz, src_nrm, src_rgba, tgt_xyz, tgt_nrm, tgt_rgba, idx, weight):
        sp, tp = _f32(src_xyz, 3), _f32(tgt_xyz, 3)
        sn = None if src_nrm is None else _f32(src_nrm, 3); tn = None if tgt_nrm is None else _f32(tgt_nrm, 3)
        sc = None if src_rgba is None else np.ascontiguousarray(src_rgba, np.uint8); tc = None if tgt_rgba is None else np.ascontiguousarray(tgt_rgba, np.uint8)
        i = np.ascontiguousarray(idx, np.int32); w = np.ascontiguousarray(weight, np.float32).copy()
        self._check(lib().icp_gpu_apply_weights(self._h, int(weighting), float(max_distance_sq), _ptr(sp), _ptr(sn), _ptr(sc), len(sp), _ptr(tp), _ptr(tn),
                                                _ptr(tc), len(tp), _ptr(i), _ptr(w)))
        return w

    def solve_linear(self, metric, src_xyz, tgt_xyz, src_nrm=None, tgt_nrm=None, weights=None):
        s, t = _f32(src_xyz, 3), _f32(tgt_xyz, 3)
        assert len(s) == len(t)
        sn = None if src_nrm is None else _f32(src_nrm, 3); tn = None if tgt_nrm is None else _f32(tgt_nrm, 3)
        w = None if weights is None else np.ascontiguousarray(weights, np.float32)
        out = np.empty(16, np.float32)
        self._check(lib().icp_gpu_solve_linear(self._h, int(metric), _ptr(s), _ptr(sn), _ptr(t), _ptr(tn), _ptr(w), len(s), _ptr(out)))
        return pose_from_c(out)

    def measure_fp32_peak(self, mode: int = 0) -> float:
        """Measured non-tensor FP32 throughput of the device in TFLOP/s: mode 0 FFMA, 1 FMUL+FADD pairs."""
        t = C.c_double(0.0)
        self._check(lib().icp_gpu_measure_fp32_peak(self._h, int(mode), C.byref(t)))
        return float(t.value)

    def stats(self) -> Stats:
        s = Stats()
        self._check(lib().icp_gpu_get_stats(self._h, C.byref(s)))
        return s

    # -- point-sharded iteration (one context per rank)
    def iteration_phases(self) -> int:
        return int(lib().icp_gpu_iteration_phases(self._h))

    def iteration_begin(self, pose):
        p = pose_to_c(pose)
        self._check(lib().icp_gpu_iteration_begin(self._h, _ptr(p)))

    def iteration_local(self, phase: int) -> np.ndarray:
        out = np.zeros(MAX_PARTIALS, np.float64)
        n = C.c_int32(0)
        self._check(lib().icp_gpu_iteration_local(self._h, phase, _ptr(out), C.byref(n)))
        return out[:n.value].copy()

    def iteration_local_dev(self, phase: int):
        """Returns (device address of the partial-sum row, number of values)."""
        p = C.c_void_p()
        n = C.c_int32(0)
        self._check(lib().icp_gpu_iteration_local_dev(self._h, phase, C.byref(p), C.byref(n)))
        return p.value, n.value

    def iteration_apply(self, phase: int, reduced):
        r = np.ascontiguousarray(reduced, dtype=np.float64)
        self._check(lib().icp_gpu_iteration_apply(self._h, phase, _ptr(r), len(r)))

    def iteration_apply_dev(self, phase: int):
        self._check(lib().icp_gpu_iteration_apply_dev(self._h, phase))

    def iteration_end(self):
        p = np.empty(16, np.float32)
        self._check(lib().icp_gpu_iteration_end(self._h, _ptr(p)))
        return pose_from_c(p)

    # -- point-sharded registration with the exchange inside the reduction kernel (peer memory)
    def peer_export(self) -> bytes:
        """(Re)creates this context's mailbox; returns its 64-byte CUDA IPC handle for the other ranks."""
        h = C.create_string_buffer(PEER_HANDLE_BYTES)
        self._check(lib().icp_gpu_peer_export(self._h, h))
        return h.raw

    def peer_attach(self, rank: int, world: int, handles):
        """handles: the `world` handles in rank order (this rank's own entry is ignored)."""
        blob = b"".join(bytes(h) for h in handles)
        if len(blob) != world * PEER_HANDLE_BYTES:
            raise ValueError(f"expected {world} handles of {PEER_HANDLE_BYTES} bytes")
        self._check(lib().icp_gpu_peer_attach(self._h, rank, world, C.c_char_p(blob)))

    def peer_address(self) -> int:
        """(Re)creates this context's mailbox; returns its device address (contexts of one process)."""
        p = C.c_void_p()
        self._check(lib().icp_gpu_peer_address(self._h, C.byref(p)))
        return int(p.value)

    def peer_attach_ptrs(self, rank: int, world: int, addresses):
        arr = (C.c_void_p * world)(*[C.c_void_p(int(a)) for a in addresses])
        self._check(lib().icp_gpu_peer_attach_ptrs(self._h, rank, world, arr))

    def peer_detach(self):
        self._check(lib().icp_gpu_peer_detach(self._h))
