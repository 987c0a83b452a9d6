"""svn_icp_b200 -- B200-native SVN-ICP registration inner loop.

Python host-side mirror of the reference's registration-class interface (svnicp::SVNICP,
reference svn-icp/include/core/SVNICP.h:29-80, SVGDICP.h:64-211) over the C ABI in
include/svnicp_b200.h.  Same method names, argument meaning and call order
(add_cloud -> set_initial_mean -> stein_align -> getters, OdometryPipeline.cpp:582-607).

All compute happens in libsvnicp_b200.so (hand-written sm_100a CUDA).  There is no CPU fallback: if
the library is missing or no B200 is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SVNICP_B200_LIB: load another build of the same library (tests use it for the -DSVN_DEBUG_BOUNDS build); never a fallback
LIB_PATH = os.environ.get("SVNICP_B200_LIB") or os.path.join(_HERE, "lib", "libsvnicp_b200.so")

ALIGN_SUCCESS = 1  # SteinICPState, SVGDICP.h:59-62
NO_OPTIMIZER = 2
CLASS_SVNICP = 0
CLASS_SVGDICP = 1
MAX_PARTICLES = 65535  # SVNICP_MAX_PARTICLES

# svnicp_get_median_paths: how an iteration's bandwidth median was found (include/svnicp_b200.h)
MEDIAN_NONE, MEDIAN_SORT, MEDIAN_FAST, MEDIAN_RADIX, MEDIAN_OVERFLOW = -1, 0, 1, 2, 3


class SvnIcpError(RuntimeError):
    pass


class _CParams(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("use_minibatch", C.c_int32), ("batch_size", C.c_int32), ("lr", C.c_double),
                ("max_dist", C.c_double), ("normalize_cloud", C.c_int32), ("optimizer", C.c_char * 16),
                ("check_early_stop", C.c_int32), ("convergence_steps", C.c_int32), ("convergence_threshold", C.c_double),
                ("KNN_count", C.c_int32), ("SVN_full_grad", C.c_int32), ("use_weight_mean", C.c_int32),
                ("grid_cell", C.c_double), ("debug_corr", C.c_int32), ("flags", C.c_int32), ("gn_stages", C.c_int32),
                ("gn_smem_kb", C.c_int32)]


# svnicp_params.flags (include/svnicp_b200.h): A/B switches read once at construction
FLAG_NO_PARTICLE_SORT = 1
FLAG_FILTER_FULL = 2
FLAG_NCCL_GATHER = 8
FLAG_REUSE_STATS = 16
FLAG_DEBUG_SYNC = 32
FLAG_WATCHDOG = 64
FLAG_NO_GRAPH = 128
FLAG_FORCE_GRAPH = 256


@dataclasses.dataclass
class SteinICPParam:
    """SteinICPParam (SVGDICP.h:41-57), same field names and defaults."""
    iterations: int = 50
    use_minibatch: bool = False
    batch_size: int = 50
    lr: float = 0.02
    max_dist: float = 1.0
    normalize_cloud: bool = True
    optimizer: str = "Adam"
    check_early_stop: bool = False
    convergence_steps: int = 5
    convergence_threshold: float = 1e-5
    KNN_count: int = 100
    SVN_full_grad: bool = True
    # extensions
    grid_cell: float = 0.0
    debug_corr: bool = False
    flags: int = 0
    gn_stages: int = 0
    gn_smem_kb: int = 0


@dataclasses.dataclass
class ParticleWeightOpt:
    """ParticleWeightOpt (SVNICP.h:25-27)."""
    use_weight_mean: bool = False


_lib = None

EXPORTS = [
    "svnicp_abi_version", "svnicp_default_params", "svnicp_create", "svnicp_destroy", "svnicp_last_error", "svnicp_set_stream",
    "svnicp_nccl_unique_id", "svnicp_init_sharding", "svnicp_add_cloud", "svnicp_set_initial_mean", "svnicp_align",
    "svnicp_get_transformation", "svnicp_get_distribution", "svnicp_get_cov_matrix", "svnicp_get_particles",
    "svnicp_get_particle_weight", "svnicp_get_particle_history", "svnicp_get_runtime", "svnicp_set_k", "svnicp_set_threshold",
    "svnicp_initialize_particles", "svnicp_initialize_particles_gaussian", "svnicp_iterations_done", "svnicp_get_candidates",
    "svnicp_get_source_f32", "svnicp_get_correspondences", "svnicp_get_gn_system", "svnicp_get_stein", "svnicp_get_prune_stats",
    "svnicp_get_median_paths", "svnicp_get_timing", "svnicp_get_slice", "svnicp_get_launch_count", "svnicp_set_profiling", "svnicp_get_phase_times",
    "svnicp_get_scan_info", "svnicp_get_tail_stamps", "svnicp_evaluate",
    "svnicp_map_create", "svnicp_map_destroy", "svnicp_map_last_error", "svnicp_map_clear", "svnicp_map_add_cloud", "svnicp_map_get",
    "svnicp_map_download", "svnicp_map_size", "svnicp_map_evaluate", "svnicp_map_export", "svnicp_map_import",
    "svnicp_pre_create", "svnicp_pre_destroy", "svnicp_pre_last_error", "svnicp_pre_crop", "svnicp_pre_downsample_uniform",
    "svnicp_pre_to_f64", "svnicp_pre_download", "svnicp_pre_deskew", "svnicp_pose_compose",
    "svnicp_batch_create", "svnicp_batch_destroy", "svnicp_batch_last_error", "svnicp_batch_size", "svnicp_batch_stream", "svnicp_batch_align",
]


def load_library() -> C.CDLL:
    """dlopen the product library; raise loudly when it was not built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SvnIcpError(f"{LIB_PATH} not found: build it with `python -m svn_icp_b200.build` "
                              "(there is no CPU or PyTorch fallback for this path)")
        lib = C.CDLL(LIB_PATH)
        lib.svnicp_last_error.restype = C.c_char_p
        lib.svnicp_last_error.argtypes = [C.c_void_p]
        for name in EXPORTS:
            fn = getattr(lib, name)
            if name not in ("svnicp_last_error", "svnicp_destroy", "svnicp_default_params", "svnicp_map_last_error", "svnicp_map_destroy",
                            "svnicp_pre_last_error", "svnicp_pre_destroy", "svnicp_batch_destroy", "svnicp_batch_last_error", "svnicp_batch_stream"):
                fn.restype = C.c_int
        lib.svnicp_pre_destroy.restype = None
        lib.svnicp_pre_destroy.argtypes = [C.c_void_p]
        lib.svnicp_pre_last_error.restype = C.c_char_p
        lib.svnicp_pre_last_error.argtypes = [C.c_void_p]
        lib.svnicp_destroy.restype = None
        lib.svnicp_destroy.argtypes = [C.c_void_p]
        lib.svnicp_map_destroy.restype = None
        lib.svnicp_map_destroy.argtypes = [C.c_void_p]
        lib.svnicp_map_last_error.restype = C.c_char_p
        lib.svnicp_map_last_error.argtypes = [C.c_void_p]
        lib.svnicp_default_params.restype = None
        lib.svnicp_batch_destroy.restype = None
        lib.svnicp_batch_last_error.restype = C.c_char_p
        lib.svnicp_batch_stream.restype = C.c_void_p
        V, I, L, D = C.c_void_p, C.c_int, C.c_int64, C.c_double
        for name, at in _ARGTYPES(V, I, L, D).items():
            getattr(lib, name).argtypes = at
        _lib = lib
    return _lib


def _ARGTYPES(V, I, L, D):
    """argtypes of every export of include/svnicp_b200.h (pointers as void*): ctypes then converts Python ints itself and
    rejects a wrong argument count instead of passing garbage."""
    return {
        "svnicp_abi_version": [], "svnicp_default_params": [V], "svnicp_create": [V, V, I, V, I, I], "svnicp_set_stream": [V, V],
        "svnicp_nccl_unique_id": [V], "svnicp_init_sharding": [V, V, I, I], "svnicp_add_cloud": [V, V, L, I, V, L, I, V],
        "svnicp_set_initial_mean": [V, V, V], "svnicp_align": [V], "svnicp_get_transformation": [V, V],
        "svnicp_get_distribution": [V, V], "svnicp_get_cov_matrix": [V, V], "svnicp_get_particles": [V, V],
        "svnicp_get_particle_weight": [V, V], "svnicp_get_particle_history": [V, V, V], "svnicp_get_runtime": [V, V],
        "svnicp_set_k": [V, I], "svnicp_set_threshold": [V, D], "svnicp_initialize_particles": [I, V, V, C.c_uint64, V],
        "svnicp_initialize_particles_gaussian": [I, V, C.c_uint64, V], "svnicp_iterations_done": [V, V],
        "svnicp_get_candidates": [V, V, V], "svnicp_get_source_f32": [V, V], "svnicp_get_correspondences": [V, V, V, V],
        "svnicp_get_gn_system": [V, V, V, V], "svnicp_get_stein": [V, V, V], "svnicp_get_prune_stats": [V, V, V],
        "svnicp_get_median_paths": [V, V, V],
        "svnicp_get_timing": [V, V], "svnicp_get_slice": [V, V, V], "svnicp_get_launch_count": [V, V],
        "svnicp_get_tail_stamps": [V, V], "svnicp_set_profiling": [V, I], "svnicp_get_phase_times": [V, V], "svnicp_get_scan_info": [V, V],
        "svnicp_evaluate": [V, I, V, V, V, V, V, V],
        "svnicp_map_create": [V, D, D, I, L, I], "svnicp_map_clear": [V], "svnicp_map_add_cloud": [V, V, L, I, I, V, V],
        "svnicp_map_get": [V, V, D, V, V], "svnicp_map_download": [V, V, L], "svnicp_map_size": [V, V, V],
        "svnicp_map_evaluate": [V, V, L, I, I, V, V, I, V, D, V, V, V, V, V], "svnicp_map_export": [V, V, V, V, L, L, I],
        "svnicp_map_import": [V, V, V, V, L, L, I],
        "svnicp_pre_create": [V, L, I], "svnicp_pre_crop": [V, V, L, I, D, D, V, V, V],
        "svnicp_pre_downsample_uniform": [V, V, L, I, D, V, V], "svnicp_pre_to_f64": [V, V, L, V], "svnicp_pre_download": [V, V, L, V],
        "svnicp_pre_deskew": [V, V, L, I, V, I, I, V, V, V, V, V, V], "svnicp_pose_compose": [V, V, V, V, V],
        "svnicp_batch_create": [V, V, I, I, V, I], "svnicp_batch_destroy": [V], "svnicp_batch_last_error": [V], "svnicp_batch_size": [V],
        "svnicp_batch_stream": [V, I], "svnicp_batch_align": [V, V],
        "svnicp_destroy": [V], "svnicp_last_error": [V], "svnicp_map_destroy": [V], "svnicp_map_last_error": [V],
        "svnicp_pre_destroy": [V], "svnicp_pre_last_error": [V],
    }


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def initialize_particles(particle_count: int, ub, lb, seed: int = 0) -> np.ndarray:
    """initialize_particles (ICPUtils.cpp:45-58) -> [6, P]."""
    out = np.zeros((6, particle_count))
    rc = load_library().svnicp_initialize_particles(C.c_int(particle_count), _p(_f64(ub)), _p(_f64(lb)), C.c_uint64(seed), _p(out))
    if rc:
        raise SvnIcpError("initialize_particles: invalid argument")
    return out


def initialize_particles_gaussian(particle_count: int, cov_diag, seed: int = 0) -> np.ndarray:
    """initialize_particles_gaussian (ICPUtils.cpp:60-75) -> [6, P]."""
    out = np.zeros((6, particle_count))
    rc = load_library().svnicp_initialize_particles_gaussian(C.c_int(particle_count), _p(_f64(cov_diag)), C.c_uint64(seed), _p(out))
    if rc:
        raise SvnIcpError("initialize_particles_gaussian: invalid argument")
    return out


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = load_library().svnicp_nccl_unique_id(buf)
    if rc:
        raise SvnIcpError("ncclGetUniqueId failed: " + (load_library().svnicp_last_error(None) or b"").decode())
    return buf.raw


def _c_params(lib, param: SteinICPParam, opt: ParticleWeightOpt | None = None) -> _CParams:
    cp = _CParams()
    lib.svnicp_default_params(C.byref(cp))
    for f in ("iterations", "batch_size", "convergence_steps", "KNN_count", "flags", "gn_stages", "gn_smem_kb"):
        setattr(cp, f, int(getattr(param, f)))
    for f in ("use_minibatch", "normalize_cloud", "check_early_stop", "SVN_full_grad", "debug_corr"):
        setattr(cp, f, int(bool(getattr(param, f))))
    for f in ("lr", "max_dist", "convergence_threshold", "grid_cell"):
        setattr(cp, f, float(getattr(param, f)))
    cp.optimizer = param.optimizer.encode()[:15]
    cp.use_weight_mean = int(bool(opt.use_weight_mean)) if opt else 0
    return cp


class SVNICP:
    """Drop-in for svnicp::SVNICP.  init_pose: [6, P] (or the reference's [6, P, 1])."""

    class_type = CLASS_SVNICP

    def __init__(self, param: SteinICPParam, init_pose, opt: ParticleWeightOpt | None = None, device: int = -1):
        self._lib = load_library()
        self._h = C.c_void_p()
        init_pose = _f64(init_pose).reshape(6, -1)
        self.particle_size = init_pose.shape[1]
        self.param = dataclasses.replace(param)
        cp = _c_params(self._lib, param, opt)
        rc = self._lib.svnicp_create(C.byref(self._h), C.byref(cp), C.c_int(self.particle_size), _p(init_pose),
                                     C.c_int(self.class_type), C.c_int(device))
        if rc != 0:
            self._h = C.c_void_p()
            raise SvnIcpError(f"svnicp_create failed ({rc}): " + (self._lib.svnicp_last_error(None) or b"").decode())
        self.n_s = 0

    # -- plumbing ---------------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc < 0:
            raise SvnIcpError(f"{what} failed ({rc}): " + (self._lib.svnicp_last_error(self._h) or b"").decode())
        return rc

    @classmethod
    def _borrowed(cls, lib, handle: int, param: SteinICPParam, particle_size: int):
        """A view of a handle owned by someone else (SVNICPBatch): same methods, close() does not destroy it."""
        self = cls.__new__(cls)
        self._lib, self._h, self._owned = lib, C.c_void_p(handle), False
        self.param, self.particle_size, self.n_s = dataclasses.replace(param), particle_size, 0
        return self

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            if getattr(self, "_owned", True):
                self._lib.svnicp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int):
        self._check(self._lib.svnicp_set_stream(self._h, C.c_void_p(cuda_stream)), "set_stream")

    def init_sharding(self, unique_id: bytes, rank: int, n_ranks: int):
        self._check(self._lib.svnicp_init_sharding(self._h, C.c_char_p(unique_id), C.c_int(rank), C.c_int(n_ranks)), "init_sharding")

    # -- the reference interface ------------------------------------------------------------------
    def _init_pose(self, init_pose):
        """[6, P] float64, P checked: the C side reads exactly 6*P doubles (the count is fixed at construction, SVNICP.cpp:42,167)."""
        init_pose = _f64(init_pose).reshape(6, -1)
        if init_pose.shape[1] != self.particle_size:
            raise SvnIcpError("add_cloud: particle count is fixed at construction (SVNICP.cpp:42,167)")
        return init_pose

    def add_cloud(self, source, target, init_pose):
        """SVGDICP::add_cloud (SVGDICP.cpp:46-62).  source/target: host arrays [N,3] float64."""
        source, target = _f64(source), _f64(target)
        init_pose = self._init_pose(init_pose)
        self.n_s = len(source)
        self._check(self._lib.svnicp_add_cloud(self._h, _p(source), C.c_int64(len(source)), C.c_int(0), _p(target),
                                               C.c_int64(len(target)), C.c_int(0), _p(init_pose)), "add_cloud")

    def add_cloud_device(self, source_ptr: int, n_s: int, target_ptr: int, n_t: int, init_pose):
        """Same, with the clouds already resident in HBM (float64 [N,3] device pointers), as in the reference where
        the caller uploads (OdometryPipeline.cpp:574,581)."""
        init_pose = self._init_pose(init_pose)
        self.n_s = n_s
        self._check(self._lib.svnicp_add_cloud(self._h, C.c_void_p(source_ptr), C.c_int64(n_s), C.c_int(1), C.c_void_p(target_ptr),
                                               C.c_int64(n_t), C.c_int(1), _p(init_pose)), "add_cloud")

    def add_cloud_pinned(self, source_ptr: int, n_s: int, target_ptr: int, n_t: int, init_pose):
        """Same, host pointers given as integers (e.g. pinned torch tensors' data_ptr())."""
        init_pose = self._init_pose(init_pose)
        self.n_s = n_s
        self._check(self._lib.svnicp_add_cloud(self._h, C.c_void_p(source_ptr), C.c_int64(n_s), C.c_int(0), C.c_void_p(target_ptr),
                                               C.c_int64(n_t), C.c_int(0), _p(init_pose)), "add_cloud")

    def set_initial_mean(self, R0, t0):
        """SVGDICP::set_initial_mean (SVGDICP.h:102-110): rotation matrix [3,3] and translation [3] of the guess."""
        self._check(self._lib.svnicp_set_initial_mean(self._h, _p(_f64(R0).reshape(9)), _p(_f64(t0).reshape(3))), "set_initial_mean")

    def stein_align(self) -> int:
        """SVNICP::stein_align (SVNICP.cpp:41-114) -> SteinICPState."""
        return self._check(self._lib.svnicp_align(self._h), "stein_align")

    def get_transformation(self) -> np.ndarray:
        out = np.zeros(6)
        self._check(self._lib.svnicp_get_transformation(self._h, _p(out)), "get_transformation")
        return out

    def get_distribution(self) -> np.ndarray:
        out = np.zeros(6)
        self._check(self._lib.svnicp_get_distribution(self._h, _p(out)), "get_distribution")
        return out

    def get_cov_matrix(self) -> np.ndarray:
        out = np.zeros(36)
        self._check(self._lib.svnicp_get_cov_matrix(self._h, _p(out)), "get_cov_matrix")
        return out

    def get_particles(self) -> np.ndarray:
        """6P doubles, component-major [6][P] (SVGDICP.cpp:515-520)."""
        out = np.zeros(6 * self.particle_size)
        self._check(self._lib.svnicp_get_particles(self._h, _p(out)), "get_particles")
        return out

    def get_particle_weight(self) -> np.ndarray:
        out = np.zeros(self.particle_size)
        self._check(self._lib.svnicp_get_particle_weight(self._h, _p(out)), "get_particle_weight")
        return out

    def get_particle_history(self) -> np.ndarray:
        """[iterations, 6P] float32 (SVGDICP.cpp:526-534)."""
        I = self.param.iterations
        out = np.zeros((max(I, 1), 6 * self.particle_size), dtype=np.float32)
        rows = C.c_int32(0)
        self._check(self._lib.svnicp_get_particle_history(self._h, _p(out), C.byref(rows)), "get_particle_history")
        return out[:I]

    def get_runtime(self) -> np.ndarray:
        out = np.zeros(3)
        self._check(self._lib.svnicp_get_runtime(self._h, _p(out)), "get_runtime")
        return out

    def set_k(self, k: int):
        self._check(self._lib.svnicp_set_k(self._h, C.c_int(k)), "set_k")
        self.param.KNN_count = k

    def set_threshold(self, max_dist: float):
        self._check(self._lib.svnicp_set_threshold(self._h, C.c_double(max_dist)), "set_threshold")

    def evaluate(self, poses, want_system: bool = True, want_mask: bool = False, want_idx: bool = False) -> dict:
        """Registration objective of the last scan at caller-given poses (svnicp_evaluate; no reference counterpart).
        poses: (6,) or (6, M) in the particle convention of the class, relative to the scan's initial mean (get_transformation()
        and zeros are valid).  Returns numpy arrays: inliers [M] int64, fitness [M] (inlier fraction), rmse [M] (metres);
        with want_system H [M, 6, 6], b [M, 6] (the Gauss-Newton system of svnicp_get_gn_system's layout); with want_mask
        mask [M, N_s] uint8; with want_idx (handle created with debug_corr) idx [M, N_s] int32 global map indices.
        A (6,) input drops the leading M axis.  Changes no state of the handle."""
        x = np.asarray(poses, dtype=np.float64)
        single = x.ndim == 1
        x = np.ascontiguousarray(x.reshape(6, -1))
        M = x.shape[1]
        stats = np.zeros((M, 3))
        H = np.zeros((M, 6, 6)) if want_system else None
        b = np.zeros((M, 6)) if want_system else None
        mask = np.zeros((M, self.n_s), dtype=np.uint8) if want_mask else None
        idx = np.zeros((M, self.n_s), dtype=np.int32) if want_idx else None
        self._check(self._lib.svnicp_evaluate(self._h, C.c_int(M), _p(x), _p(stats), _p(H), _p(b), _p(mask), _p(idx)), "evaluate")
        out = dict(inliers=stats[:, 0].astype(np.int64), fitness=stats[:, 1].copy(), rmse=stats[:, 2].copy())
        for k, v in (("H", H), ("b", b), ("mask", mask), ("idx", idx)):
            if v is not None:
                out[k] = v
        return {k: v[0] for k, v in out.items()} if single else out

    # -- parity / debug taps ----------------------------------------------------------------------
    def iterations_done(self) -> int:
        v = C.c_int32(0)
        self._check(self._lib.svnicp_iterations_done(self._h, C.byref(v)), "iterations_done")
        return v.value

    def slice(self):
        lo, hi = C.c_int32(0), C.c_int32(0)
        self._check(self._lib.svnicp_get_slice(self._h, C.byref(lo), C.byref(hi)), "get_slice")
        return lo.value, hi.value

    def get_candidates(self, want_rel=False):
        K = self.param.KNN_count
        idx = np.zeros((self.n_s, K), dtype=np.int32)
        rel = np.zeros((self.n_s, K, 3), dtype=np.float32) if want_rel else None
        self._check(self._lib.svnicp_get_candidates(self._h, _p(idx), _p(rel)), "get_candidates")
        return (idx, rel) if want_rel else idx

    def get_source_f32(self):
        out = np.zeros((self.n_s, 3), dtype=np.float32)
        self._check(self._lib.svnicp_get_source_f32(self._h, _p(out)), "get_source_f32")
        return out

    def get_correspondences(self):
        lo, hi = self.slice()
        xf = np.zeros((hi - lo, 12), dtype=np.float32)
        idx = np.zeros((hi - lo, self.n_s), dtype=np.int32)
        mask = np.zeros((hi - lo, self.n_s), dtype=np.uint8)
        self._check(self._lib.svnicp_get_correspondences(self._h, _p(xf), _p(idx), _p(mask)), "get_correspondences")
        return xf, idx, mask

    def get_gn_system(self):
        P = self.particle_size
        H, b, x = np.zeros((P, 6, 6)), np.zeros((P, 6)), np.zeros((P, 6))
        self._check(self._lib.svnicp_get_gn_system(self._h, _p(H), _p(b), _p(x)), "get_gn_system")
        return H, b, x

    def get_stein(self):
        lo, hi = self.slice()
        d = np.zeros((hi - lo, 6))
        h = C.c_double(0)
        self._check(self._lib.svnicp_get_stein(self._h, _p(d), C.byref(h)), "get_stein")
        return d, h.value

    def get_prune_stats(self):
        out = np.zeros(max(self.param.iterations, 1))
        rows = C.c_int32(0)
        self._check(self._lib.svnicp_get_prune_stats(self._h, _p(out), C.byref(rows)), "get_prune_stats")
        return out[:self.param.iterations]

    def get_median_paths(self):
        """[iterations] int32: how each iteration's bandwidth median was found (MEDIAN_* codes; -1 none)."""
        out = np.full(max(self.param.iterations, 1), -1, dtype=np.int32)
        rows = C.c_int32(0)
        self._check(self._lib.svnicp_get_median_paths(self._h, _p(out), C.byref(rows)), "get_median_paths")
        return out[:self.param.iterations]

    def get_timing(self):
        out = np.zeros(4)
        self._check(self._lib.svnicp_get_timing(self._h, _p(out)), "get_timing")
        return dict(setup_ms=out[0], iterations_ms=out[1], epilogue_ms=out[2], total_ms=out[3])

    def set_profiling(self, on: bool):
        self._check(self._lib.svnicp_set_profiling(self._h, C.c_int(int(on))), "set_profiling")

    def get_phase_times(self):
        out = np.zeros(8)
        self._check(self._lib.svnicp_get_phase_times(self._h, _p(out)), "get_phase_times")
        names = ["prep_ms", "filter_ms", "gn_ms", "finalize_ms", "gather_ms", "stein_ms", "setup_ms", "iterations"]
        return dict(zip(names, out.tolist()))

    def get_scan_info(self):
        out = np.zeros(8, dtype=np.int64)
        self._check(self._lib.svnicp_get_scan_info(self._h, _p(out)), "get_scan_info")
        names = ["n_s", "n_t", "K", "knn_fallback_queries", "TB", "n_slices", "n_pgroups", "iterations_enqueued"]
        return dict(zip(names, out.tolist()))

    def get_tail_stamps(self):
        out = np.zeros(8)
        self._check(self._lib.svnicp_get_tail_stamps(self._h, _p(out)), "get_tail_stamps")
        return out

    def launch_count(self) -> int:
        v = C.c_int64(0)
        self._check(self._lib.svnicp_get_launch_count(self._h, C.byref(v)), "get_launch_count")
        return v.value


NO_OPTIMIZER = 2  # SteinICPState, SVGDICP.h:59-62


class SVGDICP(SVNICP):
    """Drop-in for svnicp::SVGDICP (SVGDICP.h:64-211, the `class_type: SVGDICP` branch of OdometryPipeline.cpp:282-288):
    Euler-angle particles, first-order gradient, RBF SVGD step, Adam / RMSprop / SGD / Adagrad update.  Same interface
    and device pipeline as SVNICP (in the reference SVNICP derives from SVGDICP; here the two share one handle type and
    differ by class_type).  stein_align returns NO_OPTIMIZER (2) for an unknown optimizer name, like the reference.
    Note the reference quirk kept here: the particle set given to the CONSTRUCTOR is what iteration 0 of the first
    scan evaluates the kernel on (add_cloud does not refresh pose_particles_, SVGDICP.cpp:46-62)."""

    class_type = CLASS_SVGDICP

    def __init__(self, param: SteinICPParam, init_pose, device: int = -1):
        super().__init__(param, init_pose, None, device)


def pose_compose(R0, t0, mean6):
    """ICP-mode updater (OdometryPipeline.cpp:37-45, ICPUtils.cpp:84-98): initial_guess * Pose3(Expmap(mean[3:6]), mean[0:3])."""
    R, t = np.zeros((3, 3)), np.zeros(3)
    rc = load_library().svnicp_pose_compose(_p(_f64(R0).reshape(9)), _p(_f64(t0).reshape(3)), _p(_f64(mean6).reshape(6)), _p(R), _p(t))
    if rc:
        raise SvnIcpError("pose_compose: invalid argument")
    return R, t


class SVNICPBatch:
    """Throughput mode (BASELINE.json configs[3]): S independent SVN-ICP streams on one GPU.  `streams[s]` is an SVNICP
    bound to stream s (add_cloud / set_initial_mean / getters as usual); `stein_align()` runs the scans of all streams
    interleaved so they overlap on the GPU and returns the per-stream SteinICPState list."""

    def __init__(self, param: SteinICPParam, init_poses, device: int = -1):
        self._lib = load_library()
        self._b = C.c_void_p()
        ip = _f64(init_poses)
        assert ip.ndim == 3 and ip.shape[1] == 6, "init_poses: [S, 6, P]"
        S, _, P = ip.shape
        cp = _c_params(self._lib, param)
        rc = self._lib.svnicp_batch_create(C.byref(self._b), C.byref(cp), C.c_int(S), C.c_int(P), _p(ip), C.c_int(device))
        if rc != 0:
            self._b = C.c_void_p()
            raise SvnIcpError(f"svnicp_batch_create failed ({rc}): " + (self._lib.svnicp_last_error(None) or b"").decode())
        self.streams = [SVNICP._borrowed(self._lib, self._lib.svnicp_batch_stream(self._b, C.c_int(s)), param, P) for s in range(S)]

    def stein_align(self):
        states = (C.c_int32 * len(self.streams))()
        rc = self._lib.svnicp_batch_align(self._b, states)
        if rc < 0:
            raise SvnIcpError(f"batch stein_align failed ({rc}): " + (self._lib.svnicp_batch_last_error(self._b) or b"").decode())
        return list(states)

    def close(self):
        if getattr(self, "_b", None) and self._b.value:
            for s in self.streams:
                s.close()
            self._lib.svnicp_batch_destroy(self._b)
            self._b = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


MAP_SNAPSHOT_MAGIC = b"SVNMAP01"
MAP_SNAPSHOT_VERSION = 1
_SNAP_HEADER = np.dtype([("magic", "S8"), ("version", "<u4"), ("max_pointscount", "<u4"), ("voxel_size", "<f8"), ("max_range", "<f8"),
                         ("n_voxels", "<i8"), ("n_points", "<i8")])  # 48 bytes, then voxels, counts and xyz, raw


@dataclasses.dataclass
class MapSnapshot:
    """A local map's content in canonical form (svnicp_map_export): voxels [V, 3] int32 in ascending (vx, vy, vz), counts [V]
    int32, points [sum(counts), 3] float32 (each voxel's points in stored order, the voxels in order), and the map parameters."""
    voxel_size: float
    max_range: float
    max_pointscount: int
    voxels: np.ndarray
    counts: np.ndarray
    points: np.ndarray


def write_map_snapshot(path: str, snap: MapSnapshot) -> None:
    """The snapshot file shared with the C++ mirror (svnicp::write_map_snapshot): little-endian header `SVNMAP01`, u32 version 1,
    u32 max_pointscount, f64 voxel_size, f64 max_range, i64 V, i64 Npts; then voxels int32 [V][3], counts int32 [V], xyz float32
    [Npts][3]."""
    vox = np.ascontiguousarray(snap.voxels, dtype="<i4").reshape(-1, 3)
    cnt = np.ascontiguousarray(snap.counts, dtype="<i4").reshape(-1)
    pts = np.ascontiguousarray(snap.points, dtype="<f4").reshape(-1, 3)
    if len(cnt) != len(vox):
        raise SvnIcpError("write_map_snapshot: voxels and counts differ in length")
    h = np.array([(MAP_SNAPSHOT_MAGIC, MAP_SNAPSHOT_VERSION, snap.max_pointscount, snap.voxel_size, snap.max_range, len(vox), len(pts))],
                 dtype=_SNAP_HEADER)
    with open(path, "wb") as f:
        for a in (h, vox, cnt, pts):
            f.write(a.tobytes())


def read_map_snapshot(path: str) -> MapSnapshot:
    """Read a snapshot file; rejects a wrong magic or version and a length that does not match the sizes."""
    with open(path, "rb") as f:
        data = f.read()
    if len(data) < _SNAP_HEADER.itemsize:
        raise SvnIcpError(f"{path}: not a map snapshot (shorter than its header)")
    h = np.frombuffer(data, dtype=_SNAP_HEADER, count=1)[0]
    if h["magic"] != MAP_SNAPSHOT_MAGIC:
        raise SvnIcpError(f"{path}: not a map snapshot (magic)")
    if h["version"] != MAP_SNAPSHOT_VERSION:
        raise SvnIcpError(f"{path}: map snapshot version {h['version']}, this reader knows {MAP_SNAPSHOT_VERSION}")
    V, N = int(h["n_voxels"]), int(h["n_points"])
    if V < 0 or N < 0 or len(data) != _SNAP_HEADER.itemsize + 16 * V + 12 * N:
        raise SvnIcpError(f"{path}: map snapshot length {len(data)} does not match V = {V}, Npts = {N}")
    o = _SNAP_HEADER.itemsize
    vox = np.frombuffer(data, dtype="<i4", count=3 * V, offset=o).reshape(V, 3).astype(np.int32)
    cnt = np.frombuffer(data, dtype="<i4", count=V, offset=o + 12 * V).astype(np.int32)
    pts = np.frombuffer(data, dtype="<f4", count=3 * N, offset=o + 16 * V).reshape(N, 3).astype(np.float32)
    return MapSnapshot(float(h["voxel_size"]), float(h["max_range"]), int(h["max_pointscount"]), vox, cnt, pts)


class VoxelHashMap:
    """Drop-in for svnicp::VoxelHashMap (VoxelHashMap.h:28-72, VoxelHashMap.cpp:22-101), device resident: the local map the
    node keeps between scans (OdometryPipeline.cpp:577-581, :630).  Same method names; poses are (R [3,3], t [3])."""

    def __init__(self, voxel_size: float = 1.0, max_range: float = 80.0, max_pointscount: int = 20, capacity_voxels: int = 1 << 19,
                 device: int = -1):
        self._lib = load_library()
        self._m = C.c_void_p()
        self.voxel_size_, self.max_range_, self.max_pointscount_ = voxel_size, max_range, max_pointscount
        rc = self._lib.svnicp_map_create(C.byref(self._m), C.c_double(voxel_size), C.c_double(max_range), C.c_int(max_pointscount),
                                         C.c_int64(capacity_voxels), C.c_int(device))
        if rc != 0:
            self._m = C.c_void_p()
            raise SvnIcpError(f"svnicp_map_create failed ({rc}): " + (self._lib.svnicp_map_last_error(None) or b"").decode())

    def _check(self, rc, what):
        if rc < 0:
            raise SvnIcpError(f"{what} failed ({rc}): " + (self._lib.svnicp_map_last_error(self._m) or b"").decode())
        return rc

    def close(self):
        if getattr(self, "_m", None) and self._m.value:
            self._lib.svnicp_map_destroy(self._m)
            self._m = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def Clear(self):
        self._check(self._lib.svnicp_map_clear(self._m), "Clear")

    def Size(self) -> int:
        v = C.c_int64(0)
        self._check(self._lib.svnicp_map_size(self._m, C.byref(v), None), "Size")
        return v.value

    def PointCount(self) -> int:
        v = C.c_int64(0)
        self._check(self._lib.svnicp_map_size(self._m, None, C.byref(v)), "Size")
        return v.value

    def Empty(self) -> bool:
        return self.Size() == 0

    def AddPointCloud(self, new_cloud, R, t):
        """VoxelHashMap::AddPointCloud (VoxelHashMap.cpp:22-43).  new_cloud: [N,3] float32 (pcl::PointXYZ) or float64, host."""
        a = np.asarray(new_cloud)
        f64 = a.dtype != np.float32
        a = np.ascontiguousarray(a, dtype=np.float64 if f64 else np.float32)
        self._check(self._lib.svnicp_map_add_cloud(self._m, _p(a), C.c_int64(len(a)), C.c_int(int(f64)), C.c_int(0),
                                                   _p(_f64(R).reshape(9)), _p(_f64(t).reshape(3))), "AddPointCloud")

    def AddPointCloudDevice(self, ptr: int, n: int, f64: bool, R, t):
        self._check(self._lib.svnicp_map_add_cloud(self._m, C.c_void_p(ptr), C.c_int64(n), C.c_int(int(f64)), C.c_int(1),
                                                   _p(_f64(R).reshape(9)), _p(_f64(t).reshape(3))), "AddPointCloud")

    def GetMapDevice(self, position=None, max_range: float = 0.0):
        """GetMap() / GetMap(pose, max_range) (VoxelHashMap.cpp:45-63) -> (device pointer to [n,3] float64, n): feed it to
        SVNICP.add_cloud_device as the target."""
        ptr = C.c_void_p()
        n = C.c_int64(0)
        pos = _p(_f64(position).reshape(3)) if position is not None else None
        self._check(self._lib.svnicp_map_get(self._m, pos, C.c_double(max_range), C.byref(ptr), C.byref(n)), "GetMap")
        return ptr.value, n.value

    def GetMap(self, position=None, max_range: float = 0.0) -> np.ndarray:
        """Same, copied to the host: [n,3] float64 (values are float32-representable, like pcl::PointXYZ)."""
        _, n = self.GetMapDevice(position, max_range)
        out = np.zeros((n, 3))
        self._check(self._lib.svnicp_map_download(self._m, _p(out), C.c_int64(n)), "GetMap")
        return out

    def Evaluate(self, source, R0, t0, poses, max_dist: float, want_system: bool = True, want_mask: bool = False,
                 want_nearest: bool = False) -> dict:
        """Registration objective of a scan at caller-given poses against this map (svnicp_map_evaluate; no reference
        counterpart).  source: [n,3] float32 or float64 sensor-frame points, host.  poses: (6,) or (6, M) x = [t ; omega]
        relative to T0 = (R0, t0) as the SVN-ICP particles (T_world = T0 * (Exp(omega), t); zeros score T0 itself).  Each point's
        exact nearest map point with d^2 < max_dist (max_dist as in the registration, squared metres).  Returns the dict of
        SVNICP.evaluate: inliers [M] int64, fitness [M], rmse [M] (metres); with want_system H [M, 6, 6], b [M, 6]; with want_mask
        mask [M, n] uint8; with want_nearest nearest [M, n, 3] float32 (zeros where there is none).  A (6,) pose drops the M axis.
        Changes no state of the map."""
        a = np.asarray(source)
        f64 = a.dtype != np.float32
        a = np.ascontiguousarray(a, dtype=np.float64 if f64 else np.float32).reshape(-1, 3)
        return self._evaluate(_p(a), len(a), f64, False, R0, t0, poses, max_dist, want_system, want_mask, want_nearest)

    def EvaluateDevice(self, ptr: int, n: int, f64: bool, R0, t0, poses, max_dist: float, want_system: bool = True,
                       want_mask: bool = False, want_nearest: bool = False) -> dict:
        """Evaluate for a device cloud: ptr to [n,3] float32 (f64 = False, e.g. a ScanPreprocessor output) or float64."""
        return self._evaluate(C.c_void_p(ptr), n, f64, True, R0, t0, poses, max_dist, want_system, want_mask, want_nearest)

    def _evaluate(self, src, n, f64, on_device, R0, t0, poses, max_dist, want_system, want_mask, want_nearest):
        x = np.asarray(poses, dtype=np.float64)
        single = x.ndim == 1
        x = np.ascontiguousarray(x.reshape(6, -1))
        M = x.shape[1]
        stats = np.zeros((M, 3))
        H = np.zeros((M, 6, 6)) if want_system else None
        b = np.zeros((M, 6)) if want_system else None
        mask = np.zeros((M, n), dtype=np.uint8) if want_mask else None
        near = np.zeros((M, n, 3), dtype=np.float32) if want_nearest else None
        self._check(self._lib.svnicp_map_evaluate(self._m, src, C.c_int64(n), C.c_int(int(f64)), C.c_int(int(on_device)),
                                                  _p(_f64(R0).reshape(9)), _p(_f64(t0).reshape(3)), C.c_int(M), _p(x),
                                                  C.c_double(max_dist), _p(stats), _p(H), _p(b), _p(mask), _p(near)), "Evaluate")
        out = dict(inliers=stats[:, 0].astype(np.int64), fitness=stats[:, 1].copy(), rmse=stats[:, 2].copy())
        for k, v in (("H", H), ("b", b), ("mask", mask), ("nearest", near)):
            if v is not None:
                out[k] = v
        return {k: v[0] for k, v in out.items()} if single else out

    # -- snapshots (svnicp_map_export / svnicp_map_import; no reference counterpart) --------------
    def Export(self) -> MapSnapshot:
        """The map's content in canonical form: the same bytes for the same content, whatever the slot layout or history."""
        V, N = self.Size(), self.PointCount()
        vox, cnt, pts = np.zeros((V, 3), dtype=np.int32), np.zeros(V, dtype=np.int32), np.zeros((N, 3), dtype=np.float32)
        self._check(self._lib.svnicp_map_export(self._m, _p(vox), _p(cnt), _p(pts), C.c_int64(V), C.c_int64(N), C.c_int(0)), "Export")
        return MapSnapshot(self.voxel_size_, self.max_range_, self.max_pointscount_, vox, cnt, pts)

    def ExportDevice(self, voxels_ptr: int, counts_ptr: int, xyz_ptr: int):
        """Export into device memory on the map's GPU: int32 [Size(), 3], int32 [Size()], float32 [PointCount(), 3]."""
        self._check(self._lib.svnicp_map_export(self._m, C.c_void_p(voxels_ptr), C.c_void_p(counts_ptr), C.c_void_p(xyz_ptr),
                                                C.c_int64(self.Size()), C.c_int64(self.PointCount()), C.c_int(1)), "Export")

    def Import(self, snapshot: MapSnapshot):
        """Replace the content by a snapshot (no transform, no RemoveFarPointCloud).  The snapshot's voxel_size, max_range and
        max_pointscount must be the map's.  All or nothing: on an error the map is unchanged."""
        mine = (self.voxel_size_, self.max_range_, self.max_pointscount_)
        theirs = (snapshot.voxel_size, snapshot.max_range, snapshot.max_pointscount)
        if tuple(map(float, mine)) != tuple(map(float, theirs)):
            raise SvnIcpError(f"Import: snapshot of a map with (voxel_size, max_range, max_pointscount) = {theirs}, this map has {mine}")
        vox = np.ascontiguousarray(snapshot.voxels, dtype=np.int32).reshape(-1, 3)
        cnt = np.ascontiguousarray(snapshot.counts, dtype=np.int32).reshape(-1)
        pts = np.ascontiguousarray(snapshot.points, dtype=np.float32).reshape(-1, 3)
        if len(cnt) != len(vox):
            raise SvnIcpError("Import: voxels and counts differ in length")
        self._check(self._lib.svnicp_map_import(self._m, _p(vox), _p(cnt), _p(pts), C.c_int64(len(vox)), C.c_int64(len(pts)), C.c_int(0)),
                    "Import")

    def ImportDevice(self, voxels_ptr: int, counts_ptr: int, xyz_ptr: int, n_voxels: int, n_points: int):
        """Import from device memory on the map's GPU (layout of ExportDevice).  Only the ABI's checks apply: counts and membership."""
        self._check(self._lib.svnicp_map_import(self._m, C.c_void_p(voxels_ptr), C.c_void_p(counts_ptr), C.c_void_p(xyz_ptr),
                                                C.c_int64(n_voxels), C.c_int64(n_points), C.c_int(1)), "Import")

    def Save(self, path: str):
        write_map_snapshot(path, self.Export())

    @classmethod
    def Load(cls, path: str, capacity_voxels: int | None = None, device: int = -1) -> "VoxelHashMap":
        """A new map with the file's parameters, a capacity of at least its voxel count, and its content."""
        snap = read_map_snapshot(path)
        cap = max(capacity_voxels if capacity_voxels is not None else 1 << 19, len(snap.counts), 1)
        m = cls(snap.voxel_size, snap.max_range, snap.max_pointscount, capacity_voxels=cap, device=device)
        m.Import(snap)
        return m


class ScanPreprocessor:
    """The node's scan pre-processing on the device (OdometryPipeline.cpp:555-560): `crop_pointcloud` (:692-704) and
    `downsample_uniform` (:684-690, pcl::UniformSampling).  Methods return (device pointer to [n,3] float32, n); feed one to the
    next method with on_device=True, to VoxelHashMap.AddPointCloudDevice, or through `to_f64` to SVNICP.add_cloud_device."""

    def __init__(self, max_points: int, device: int = -1):
        self._lib = load_library()
        self._p = C.c_void_p()
        self.scan_max_range_ = 0.0  # the reference's running maximum of the SQUARED norm (OdometryPipeline.cpp:699)
        rc = self._lib.svnicp_pre_create(C.byref(self._p), C.c_int64(max_points), C.c_int(device))
        if rc != 0:
            self._p = C.c_void_p()
            raise SvnIcpError(f"svnicp_pre_create failed ({rc}): " + (self._lib.svnicp_pre_last_error(None) or b"").decode())

    def _check(self, rc, what):
        if rc < 0:
            raise SvnIcpError(f"{what} failed ({rc}): " + (self._lib.svnicp_pre_last_error(self._p) or b"").decode())
        return rc

    def close(self):
        if getattr(self, "_p", None) and self._p.value:
            self._lib.svnicp_pre_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _src(cloud, n, on_device):
        if on_device:
            return C.c_void_p(cloud), int(n), None
        a = np.ascontiguousarray(cloud, dtype=np.float32)
        return _p(a), len(a), a

    def crop_pointcloud(self, cloud, min_range: float, max_range: float, n: int = 0, on_device: bool = False):
        src, n, keep = self._src(cloud, n, on_device)
        ptr, n_out, mx = C.c_void_p(), C.c_int64(0), C.c_double(0)
        self._check(self._lib.svnicp_pre_crop(self._p, src, C.c_int64(n), C.c_int(int(on_device)), C.c_double(min_range), C.c_double(max_range),
                                              C.byref(ptr), C.byref(n_out), C.byref(mx)), "crop_pointcloud")
        if mx.value > self.scan_max_range_:
            self.scan_max_range_ = mx.value
        return ptr.value, n_out.value

    def downsample_uniform(self, cloud, voxel_size: float, n: int = 0, on_device: bool = False):
        src, n, keep = self._src(cloud, n, on_device)
        ptr, n_out = C.c_void_p(), C.c_int64(0)
        self._check(self._lib.svnicp_pre_downsample_uniform(self._p, src, C.c_int64(n), C.c_int(int(on_device)), C.c_double(voxel_size),
                                                            C.byref(ptr), C.byref(n_out)), "downsample_uniform")
        return ptr.value, n_out.value

    def deskew_pointcloud(self, cloud, stamps, start_pose, finish_pose, n: int = 0, on_device: bool = False, kitti: bool = False):
        """OdometryPipeline::deskew_pointcloud (:357-447).  stamps: [n] per-point time stamps (host array; None with kitti=True);
        start_pose / finish_pose: (R [3,3], t [3]) = the two newest poses of the node's pose buffer.  Returns (device ptr, n, moved)."""
        src, n, keep = self._src(cloud, n, on_device)
        st = np.ascontiguousarray(stamps, dtype=np.float64) if stamps is not None else None
        ptr, moved = C.c_void_p(), C.c_int32(0)
        (Rs, ts), (Rf, tf) = start_pose, finish_pose
        self._check(self._lib.svnicp_pre_deskew(self._p, src, C.c_int64(n), C.c_int(int(on_device)), _p(st), C.c_int(0), C.c_int(int(kitti)),
                                                _p(_f64(Rs).reshape(9)), _p(_f64(ts).reshape(3)), _p(_f64(Rf).reshape(9)), _p(_f64(tf).reshape(3)),
                                                C.byref(ptr), C.byref(moved)), "deskew_pointcloud")
        return ptr.value, n, bool(moved.value)

    def to_f64(self, ptr: int, n: int) -> int:
        out = C.c_void_p()
        self._check(self._lib.svnicp_pre_to_f64(self._p, C.c_void_p(ptr), C.c_int64(n), C.byref(out)), "to_f64")
        return out.value

    def download(self, ptr: int, n: int) -> np.ndarray:
        out = np.zeros((n, 3), dtype=np.float32)
        self._check(self._lib.svnicp_pre_download(self._p, C.c_void_p(ptr), C.c_int64(n), _p(out)), "download")
        return out
