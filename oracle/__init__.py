"""ctypes front-ends for the CPU checkers.  TEST INFRASTRUCTURE ONLY.

* `Oracle`    -> oracle/liboracle.so   (plain-C fp64 restatement, svn_oracle.c)
* `Reference` -> oracle/_ref/libsvnicp_ref.so (the reference's own sources, CPU device swap)

Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference) import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_dp = C.POINTER(C.c_double)


class Params(C.Structure):
    _fields_ = [("iterations", C.c_int), ("lr", C.c_double), ("max_dist", C.c_double),
                ("check_early_stop", C.c_int), ("convergence_threshold", C.c_double),
                ("knn_count", C.c_int), ("svn_full_grad", C.c_int)]


def make_params(iterations=30, lr=1.0, max_dist=3.0, check_early_stop=False, convergence_threshold=5e-4,
                knn_count=100, svn_full_grad=True) -> Params:
    return Params(int(iterations), float(lr), float(max_dist), int(bool(check_early_stop)),
                  float(convergence_threshold), int(knn_count), int(bool(svn_full_grad)))


class Dumps(C.Structure):
    _fields_ = [("corr_idx", C.c_void_p), ("corr_mask", C.c_void_p), ("H", C.c_void_p), ("b", C.c_void_p),
                ("delta", C.c_void_p), ("x_before", C.c_void_p), ("x_after", C.c_void_p), ("bandwidth", C.c_void_p)]


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def build(force: bool = False) -> str:
    so = os.path.join(HERE, "liboracle.so")
    srcs = [os.path.join(HERE, f) for f in ("svn_oracle.c", "svgd_oracle.c", "voxelmap_oracle.c", "preprocess_oracle.c")]
    if force or not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["make", "-C", HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
    return so


class Oracle:
    def __init__(self):
        self.lib = C.CDLL(build())
        self.lib.oracle_rbf_kernel.restype = C.c_double
        self.lib.oracle_num_threads.restype = C.c_int

    def num_threads(self):
        return self.lib.oracle_num_threads()

    def set_num_threads(self, n):
        self.lib.oracle_set_num_threads(int(n))

    def so3_exp(self, r):
        R = np.zeros(9)
        Jl = np.zeros(9)
        with np.errstate(all="ignore"):
            self.lib.oracle_so3_exp(_ptr(_f64(r)), _ptr(R), _ptr(Jl))
        return R.reshape(3, 3), Jl.reshape(3, 3)

    def so3_log(self, R):
        w = np.zeros(3)
        self.lib.oracle_so3_log(_ptr(_f64(R).reshape(-1)), _ptr(w))
        return w

    def transform_q0(self, src, R0, t0):
        src = _f64(src)
        q0 = np.empty_like(src)
        self.lib.oracle_transform_q0(_ptr(src), C.c_int64(len(src)), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(q0))
        return q0

    def knn_mink(self, q, tgt, K):
        q, tgt = _f64(q), _f64(tgt)
        idx = np.zeros((len(q), K), dtype=np.int64)
        dist = np.zeros((len(q), K), dtype=np.float64)
        self.lib.oracle_knn_mink(_ptr(q), C.c_int64(len(q)), _ptr(tgt), C.c_int64(len(tgt)), C.c_int(K), _ptr(idx), _ptr(dist))
        return idx, dist

    def gn(self, R, t, R0, t0, src, tgt, cand_idx, max_dist, want_corr=False):
        R, t, src, tgt = _f64(R), _f64(t), _f64(src), _f64(tgt)
        P = len(R)
        cand_idx = np.ascontiguousarray(cand_idx, dtype=np.int64)
        K = cand_idx.shape[1]
        H = np.zeros((P, 6, 6))
        b = np.zeros((P, 6))
        ci = np.zeros((P, len(src)), dtype=np.int32) if want_corr else None
        cm = np.zeros((P, len(src)), dtype=np.uint8) if want_corr else None
        self.lib.oracle_gn(_ptr(R), _ptr(t), C.c_int(P), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(src), C.c_int64(len(src)),
                           _ptr(tgt), _ptr(cand_idx), C.c_int(K), C.c_double(max_dist), _ptr(H), _ptr(b), _ptr(ci), _ptr(cm))
        return (H, b, ci, cm) if want_corr else (H, b)

    def stein_step(self, x, H, b, full=True, lr=1.0):
        x, H, b = _f64(x), _f64(H), _f64(b)
        P = len(x)
        d = np.zeros((P, 6))
        h = C.c_double(0)
        self.lib.oracle_stein_step(_ptr(x), _ptr(H), _ptr(b), C.c_int(P), C.c_int(int(full)), C.c_double(lr), _ptr(d), C.byref(h))
        return d, h.value

    def pair_median_kernel_order(self, x):
        """(median, nearest distinct entry below, nearest above) of the P^2 pairwise squared distances of x [P, 6], rounded
        as the k_head_* kernels round them (oracle_pair_median_kernel_order)."""
        x = _f64(x)
        out = np.zeros(3)
        self.lib.oracle_pair_median_kernel_order(_ptr(x), C.c_int(len(x)), _ptr(out))
        return tuple(out.tolist())

    def pose_update(self, R, t, delta):
        R, t, delta = _f64(R).copy(), _f64(t).copy(), _f64(delta)
        with np.errstate(all="ignore"):
            self.lib.oracle_pose_update(_ptr(R), _ptr(t), _ptr(delta), C.c_int(len(R)))
        return R, t

    # ---- kernel-arithmetic mode (fp32 operation order of the CUDA kernels) ----
    def cand_sorted(self, q0, tgt, K):
        q0, tgt = _f64(q0), _f64(tgt)
        idx = np.zeros((len(q0), K), dtype=np.int32)
        rel = np.zeros((len(q0), K, 3), dtype=np.float32)
        self.lib.oracle_cand_sorted(_ptr(q0), C.c_int64(len(q0)), _ptr(tgt), C.c_int64(len(tgt)), C.c_int(K), _ptr(idx), _ptr(rel))
        return idx, rel

    def source_f32(self, src, R0):
        src = _f64(src)
        sp = np.zeros((len(src), 3), dtype=np.float32)
        self.lib.oracle_source_f32(_ptr(src), C.c_int64(len(src)), _ptr(_f64(R0)), _ptr(sp))
        return sp

    def transforms_f32(self, R, t, R0):
        R, t = _f64(R), _f64(t)
        xf = np.zeros((len(R), 12), dtype=np.float32)
        self.lib.oracle_transforms_f32(_ptr(R), _ptr(t), C.c_int(len(R)), _ptr(_f64(R0)), _ptr(xf))
        return xf

    def corr_f32(self, xf, sp, rel, cidx, max_dist):
        xf = np.ascontiguousarray(xf, dtype=np.float32)
        sp = np.ascontiguousarray(sp, dtype=np.float32)
        rel = np.ascontiguousarray(rel, dtype=np.float32)
        cidx = np.ascontiguousarray(cidx, dtype=np.int32)
        P, ns, K = len(xf), len(sp), cidx.shape[1]
        idx = np.zeros((P, ns), dtype=np.int32)
        mask = np.zeros((P, ns), dtype=np.uint8)
        self.lib.oracle_corr_f32(_ptr(xf), C.c_int(P), _ptr(sp), C.c_int64(ns), _ptr(rel), _ptr(cidx), C.c_int(K),
                                 C.c_double(max_dist), _ptr(idx), _ptr(mask))
        return idx, mask

    def gn_given_corr(self, R, t, R0, t0, src, tgt, corr_idx, corr_mask, max_dist):
        R, t, src, tgt = _f64(R), _f64(t), _f64(src), _f64(tgt)
        P = len(R)
        corr_idx = np.ascontiguousarray(corr_idx, dtype=np.int32)
        corr_mask = np.ascontiguousarray(corr_mask, dtype=np.uint8)
        H = np.zeros((P, 6, 6))
        b = np.zeros((P, 6))
        self.lib.oracle_gn_given_corr(_ptr(R), _ptr(t), C.c_int(P), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(src), C.c_int64(len(src)),
                                      _ptr(tgt), _ptr(corr_idx), _ptr(corr_mask), C.c_double(max_dist), _ptr(H), _ptr(b))
        return H, b

    def rbf_kernel(self, x):
        x = _f64(x)
        P = len(x)
        K = np.zeros((P, P))
        h = self.lib.oracle_rbf_kernel(_ptr(x), C.c_int(P), _ptr(K))
        return K, h

    def align(self, prm: Params, src, tgt, init_pose, R0, t0, dumps=()):
        """Whole scan.  dumps: subset of Dumps field names to record."""
        src, tgt, init_pose = _f64(src), _f64(tgt), _f64(init_pose)
        P, I, ns = init_pose.shape[1], prm.iterations, len(src)
        out = dict(particles=np.zeros((6, P)), mean=np.zeros(6), var=np.zeros(6), cov=np.zeros((6, 6)),
                   weights=np.zeros(P), history=np.zeros((I, 6, P), dtype=np.float32),
                   cand_idx=np.zeros((ns, prm.knn_count), dtype=np.int64))
        shapes = dict(corr_idx=((I, P, ns), np.int32), corr_mask=((I, P, ns), np.uint8), H=((I, P, 6, 6), np.float64),
                      b=((I, P, 6), np.float64), delta=((I, P, 6), np.float64), x_before=((I, P, 6), np.float64),
                      x_after=((I, P, 6), np.float64), bandwidth=((I,), np.float64))
        d = Dumps()
        for name in dumps:
            shp, dt = shapes[name]
            out[name] = np.zeros(shp, dtype=dt)
            setattr(d, name, out[name].ctypes.data)
        it = C.c_int(0)
        state = self.lib.oracle_align(C.byref(prm), _ptr(src), C.c_int64(ns), _ptr(tgt), C.c_int64(len(tgt)), _ptr(init_pose),
                                      C.c_int(P), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(out["particles"]), _ptr(out["mean"]),
                                      _ptr(out["var"]), _ptr(out["cov"]), _ptr(out["weights"]), _ptr(out["history"]),
                                      C.byref(it), _ptr(out["cand_idx"]), C.byref(d))
        out["state"] = state
        out["iters_done"] = it.value
        return out


    # ---- SVGD-ICP class (svgd_oracle.c) ----
    def svgd_align(self, prm: "SvgdParams", src, tgt, prev_pose, init_pose, R0, t0, dumps=()):
        src, tgt, init_pose, prev_pose = _f64(src), _f64(tgt), _f64(init_pose), _f64(prev_pose)
        P, I, ns = init_pose.shape[1], prm.iterations, len(src)
        out = dict(particles=np.zeros((6, P)), mean=np.zeros(6), var=np.zeros(6), cov=np.zeros((6, 6)),
                   weights=np.zeros(P), history=np.zeros((I, 6, P), dtype=np.float32))
        shapes = dict(grad=((I, P, 6), np.float64), stein=((I, P, 6), np.float64), bandwidth=((I,), np.float64),
                      x_after=((I, P, 6), np.float64), corr_idx=((I, P, ns), np.int32), corr_mask=((I, P, ns), np.uint8))
        d = SvgdDumps()
        for name in dumps:
            shp, dt = shapes[name]
            out[name] = np.zeros(shp, dtype=dt)
            setattr(d, name, out[name].ctypes.data)
        it = C.c_int(0)
        with np.errstate(all="ignore"):
            out["state"] = self.lib.oracle_svgd_align(
                C.byref(prm), _ptr(src), C.c_int64(ns), _ptr(tgt), C.c_int64(len(tgt)), _ptr(prev_pose), _ptr(init_pose),
                C.c_int(P), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(out["particles"]), _ptr(out["mean"]), _ptr(out["var"]),
                _ptr(out["cov"]), _ptr(out["weights"]), _ptr(out["history"]), C.byref(it), C.byref(d))
        out["iters_done"] = it.value
        return out

    def svgd_grad(self, poses, R0, t0, src, tgt, cand_idx, max_dist):
        poses, src, tgt = _f64(poses), _f64(src), _f64(tgt)
        cand_idx = np.ascontiguousarray(cand_idx, dtype=np.int64)
        g = np.zeros((len(poses), 6))
        self.lib.oracle_svgd_grad(_ptr(poses), C.c_int(len(poses)), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(src), C.c_int64(len(src)),
                                  _ptr(tgt), _ptr(cand_idx), C.c_int(cand_idx.shape[1]), C.c_double(max_dist), _ptr(g))
        return g

    def svgd_grad_given_corr(self, poses, R0, t0, src, tgt, corr_idx, corr_mask, max_dist):
        poses, src, tgt = _f64(poses), _f64(src), _f64(tgt)
        corr_idx = np.ascontiguousarray(corr_idx, dtype=np.int32)
        corr_mask = np.ascontiguousarray(corr_mask, dtype=np.uint8)
        g = np.zeros((len(poses), 6))
        self.lib.oracle_svgd_grad_given_corr(_ptr(poses), C.c_int(len(poses)), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(src),
                                             C.c_int64(len(src)), _ptr(tgt), _ptr(corr_idx), _ptr(corr_mask),
                                             C.c_double(max_dist), _ptr(g))
        return g

    def svgd_corr(self, poses, R0, t0, src, tgt, cand_idx, max_dist):
        poses, src, tgt = _f64(poses), _f64(src), _f64(tgt)
        cand_idx = np.ascontiguousarray(cand_idx, dtype=np.int64)
        idx = np.zeros((len(poses), len(src)), dtype=np.int32)
        mask = np.zeros((len(poses), len(src)), dtype=np.uint8)
        self.lib.oracle_svgd_corr(_ptr(poses), C.c_int(len(poses)), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(src), C.c_int64(len(src)),
                                  _ptr(tgt), _ptr(cand_idx), C.c_int(cand_idx.shape[1]), C.c_double(max_dist), _ptr(idx), _ptr(mask))
        return idx, mask

    def svgd_step(self, x, g):
        x, g = _f64(x), _f64(g)
        out = np.zeros_like(x)
        h = C.c_double(0)
        self.lib.oracle_svgd_step(_ptr(x), _ptr(g), C.c_int(len(x)), _ptr(out), C.byref(h))
        return out, h.value

    def opt_step(self, optimizer: str, lr, step, x, grad, state):
        """torch::optim step (SVGDICP.cpp:142-170 options) on flat arrays, in place: x [n], grad [n], state [n][2]."""
        assert x.dtype == np.float64 and state.dtype == np.float64 and x.flags.c_contiguous and state.flags.c_contiguous
        g = _f64(grad).reshape(-1)
        self.lib.oracle_opt_step_array(C.c_int(OPTIMIZERS[optimizer]), C.c_double(lr), C.c_int(step), _ptr(x), _ptr(g), _ptr(state),
                                       C.c_int64(x.size))

    def euler_R(self, r, p, y):
        R = np.zeros(9)
        self.lib.oracle_euler_R(C.c_double(r), C.c_double(p), C.c_double(y), _ptr(R))
        return R.reshape(3, 3)


OPTIMIZERS = {"Adam": 0, "RMSprop": 1, "SGD": 2, "Adagrad": 3}


class SvgdParams(C.Structure):
    _fields_ = [("iterations", C.c_int), ("lr", C.c_double), ("max_dist", C.c_double),
                ("check_early_stop", C.c_int), ("convergence_threshold", C.c_double),
                ("knn_count", C.c_int), ("optimizer", C.c_int)]


def make_svgd_params(iterations=30, lr=0.03, max_dist=3.0, check_early_stop=False, convergence_threshold=5e-4,
                     knn_count=100, optimizer="Adam") -> SvgdParams:
    return SvgdParams(int(iterations), float(lr), float(max_dist), int(bool(check_early_stop)),
                      float(convergence_threshold), int(knn_count), OPTIMIZERS.get(optimizer, -1))


class SvgdDumps(C.Structure):
    _fields_ = [("grad", C.c_void_p), ("stein", C.c_void_p), ("bandwidth", C.c_void_p), ("x_after", C.c_void_p),
                ("corr_idx", C.c_void_p), ("corr_mask", C.c_void_p)]


class VoxelMapOracle:
    """Sequential restatement of svnicp::VoxelHashMap (voxelmap_oracle.c)."""

    def __init__(self, voxel_size=1.0, max_range=80.0, max_pointscount=20):
        self.lib = C.CDLL(build())
        self.lib.oracle_vmap_create.restype = C.c_void_p
        self.lib.oracle_vmap_get.restype = C.c_int64
        self.lib.oracle_vmap_size.restype = C.c_int64
        self.m = C.c_void_p(self.lib.oracle_vmap_create(C.c_double(voxel_size), C.c_double(max_range), C.c_int(max_pointscount)))

    def __del__(self):
        try:
            self.lib.oracle_vmap_destroy(self.m)
        except Exception:
            pass

    def AddPointCloud(self, cloud, R, t):
        a = np.asarray(cloud)
        f64 = a.dtype != np.float32
        a = np.ascontiguousarray(a, dtype=np.float64 if f64 else np.float32)
        self.lib.oracle_vmap_add(self.m, _ptr(a), C.c_int64(len(a)), C.c_int(int(f64)), _ptr(_f64(R).reshape(9)), _ptr(_f64(t).reshape(3)))

    def GetMap(self, position=None, max_range=0.0):
        pos = _ptr(_f64(position).reshape(3)) if position is not None else None
        n = self.lib.oracle_vmap_get(self.m, pos, C.c_double(max_range), None)
        out = np.zeros((n, 3))
        self.lib.oracle_vmap_get(self.m, pos, C.c_double(max_range), _ptr(out))
        return out

    def Size(self):
        return self.lib.oracle_vmap_size(self.m)

    def Clear(self):
        self.lib.oracle_vmap_clear(self.m)


class PreprocessOracle:
    """Sequential restatement of the node's crop + pcl::UniformSampling (preprocess_oracle.c; down-sampling parity unpinned)."""

    def __init__(self):
        self.lib = C.CDLL(build())
        self.lib.oracle_crop.restype = C.c_int64
        self.lib.oracle_downsample_uniform.restype = C.c_int64

    def crop(self, cloud, min_range, max_range):
        a = np.ascontiguousarray(cloud, dtype=np.float32)
        out = np.zeros_like(a)
        mx = C.c_double(0)
        n = self.lib.oracle_crop(_ptr(a), C.c_int64(len(a)), C.c_double(min_range), C.c_double(max_range), _ptr(out), C.byref(mx))
        return out[:n].copy(), mx.value

    def downsample_uniform(self, cloud, radius):
        a = np.ascontiguousarray(cloud, dtype=np.float32)
        out = np.zeros_like(a)
        n = self.lib.oracle_downsample_uniform(_ptr(a), C.c_int64(len(a)), C.c_double(radius), _ptr(out))
        return out[:n].copy()

    # ---- de-skewing (OdometryPipeline.cpp:357-447; GTSAM 4.2 closed forms restated, pinned against scipy expm/logm) ----
    def pose3_expmap(self, xi):
        R, t = np.zeros((3, 3)), np.zeros(3)
        self.lib.oracle_pose3_expmap(_ptr(_f64(xi)), _ptr(R), _ptr(t))
        return R, t

    def pose3_logmap(self, R, t):
        xi = np.zeros(6)
        self.lib.oracle_pose3_logmap(_ptr(_f64(R)), _ptr(_f64(t)), _ptr(xi))
        return xi

    def deskew(self, cloud, stamps, start_pose, finish_pose, kitti=False):
        a = np.ascontiguousarray(cloud, dtype=np.float32)
        st = _f64(stamps) if stamps is not None else None
        out = np.zeros_like(a)
        (Rs, ts), (Rf, tf) = start_pose, finish_pose
        moved = self.lib.oracle_deskew(_ptr(a), _ptr(st), C.c_int64(len(a)), C.c_int(int(kitti)), _ptr(_f64(Rs)), _ptr(_f64(ts)),
                                       _ptr(_f64(Rf)), _ptr(_f64(tf)), _ptr(out))
        return out, bool(moved)


class ReferenceMap:
    """The reference's own svnicp::VoxelHashMap (oracle/_ref/libvmap_ref.so: VoxelHashMap.cpp compiled unmodified over
    stand-in PCL / Eigen / tsl types).  float32 clouds only (pcl::PointXYZI)."""

    def __init__(self, voxel_size=1.0, max_range=80.0, max_pointscount=20):
        self.lib = C.CDLL(os.path.join(HERE, "_ref", "libvmap_ref.so"))
        self.lib.ref_vmap_create.restype = C.c_void_p
        self.lib.ref_vmap_get.restype = C.c_int64
        self.lib.ref_vmap_size.restype = C.c_int64
        self.m = C.c_void_p(self.lib.ref_vmap_create(C.c_double(voxel_size), C.c_double(max_range), C.c_int(max_pointscount)))

    def __del__(self):
        try:
            self.lib.ref_vmap_destroy(self.m)
        except Exception:
            pass

    def AddPointCloud(self, cloud, R, t):
        a = np.ascontiguousarray(cloud, dtype=np.float32)
        self.lib.ref_vmap_add(self.m, _ptr(a), C.c_int64(len(a)), _ptr(_f64(R).reshape(9)), _ptr(_f64(t).reshape(3)))

    def GetMap(self, position=None, max_range=0.0):
        pos = _ptr(_f64(position).reshape(3)) if position is not None else None
        n = self.lib.ref_vmap_get(self.m, pos, C.c_double(max_range), None)
        out = np.zeros((n, 3))
        self.lib.ref_vmap_get(self.m, pos, C.c_double(max_range), _ptr(out))
        return out

    def Size(self):
        return self.lib.ref_vmap_size(self.m)


def ref_available() -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", "libsvnicp_ref.so"))


def ref_cuda_available() -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", "libsvnicp_ref_cuda.so"))


class Reference:
    """The reference's own registration classes (CPU device swap).  One (P, threshold) per PROCESS
    (function-static tensors, SVNICP.cpp:42,167) -- run each configuration in a fresh subprocess.
    cuda=True loads oracle/_ref/libsvnicp_ref_cuda.so instead (oracle/build_ref_cuda.sh): the same sources WITHOUT the
    device swap plus the reference's vendored knn.cu, i.e. the reference as it runs on a GPU (bench comparator only)."""

    def __init__(self, cuda: bool = False):
        import torch  # noqa: F401  (libtorch must be loaded first)
        if cuda:
            torch.zeros(1).cuda()  # CUDA context + libtorch_cuda loaded before the reference library
        self.lib = C.CDLL(os.path.join(HERE, "_ref", "libsvnicp_ref_cuda.so" if cuda else "libsvnicp_ref.so"))
        self.lib.ref_num_threads.restype = C.c_int

    def num_threads(self):
        return self.lib.ref_num_threads()

    def set_num_threads(self, n):
        self.lib.ref_set_num_threads(int(n))

    def scan(self, prm: Params, src, tgt, init_pose, R0, t0):
        src, tgt, init_pose = _f64(src), _f64(tgt), _f64(init_pose)
        P, I = init_pose.shape[1], prm.iterations
        out = dict(particles=np.zeros((6, P)), mean=np.zeros(6), var=np.zeros(6), cov=np.zeros((6, 6)),
                   weights=np.zeros(P), history=np.zeros((I, 6, P), dtype=np.float32), seconds=np.zeros(3))
        out["state"] = self.lib.ref_scan(C.byref(prm), _ptr(src), C.c_int64(len(src)), _ptr(tgt), C.c_int64(len(tgt)),
                                         _ptr(init_pose), C.c_int(P), _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(out["particles"]),
                                         _ptr(out["mean"]), _ptr(out["var"]), _ptr(out["cov"]), _ptr(out["weights"]),
                                         _ptr(out["history"]), _ptr(out["seconds"]))
        return out

    def svgd_scan(self, prm: Params, optimizer: str, src, tgt, ctor_pose, init_pose, R0, t0, init_pose2=None):
        """SVGDICP class: ctor(ctor_pose) -> add_cloud(init_pose) -> align [-> add_cloud(init_pose2) -> align]."""
        src, tgt, init_pose, ctor_pose = _f64(src), _f64(tgt), _f64(init_pose), _f64(ctor_pose)
        ip2 = _f64(init_pose2) if init_pose2 is not None else None
        P, I = init_pose.shape[1], prm.iterations
        out = dict(particles=np.zeros((6, P)), mean=np.zeros(6), var=np.zeros(6), cov=np.zeros((6, 6)),
                   weights=np.zeros(P), history=np.zeros((I, 6, P), dtype=np.float32), runtime=np.zeros(3))
        out["state"] = self.lib.ref_svgd_scan(C.byref(prm), optimizer.encode(), _ptr(src), C.c_int64(len(src)), _ptr(tgt),
                                              C.c_int64(len(tgt)), _ptr(ctor_pose), _ptr(init_pose), _ptr(ip2), C.c_int(P),
                                              _ptr(_f64(R0)), _ptr(_f64(t0)), _ptr(out["particles"]), _ptr(out["mean"]),
                                              _ptr(out["var"]), _ptr(out["cov"]), _ptr(out["weights"]), _ptr(out["history"]),
                                              _ptr(out["runtime"]))
        return out

    def scan_steps(self, prm: Params, src, tgt, init_pose, R0, t0, steps, want=("x_after", "H", "b", "tgt_paired", "cand_idx")):
        src, tgt, init_pose = _f64(src), _f64(tgt), _f64(init_pose)
        P, ns = init_pose.shape[1], len(src)
        shapes = dict(x_after=((steps, 6, P), np.float64), H=((steps, P, 6, 6), np.float64), b=((steps, P, 6), np.float64),
                      tgt_paired=((steps, P, ns, 3), np.float64), src_tr=((steps, P, ns, 3), np.float64),
                      cand_idx=((ns, prm.knn_count), np.int64))
        out = {k: np.zeros(*shapes[k]) for k in want}
        out.update(particles=np.zeros((6, P)), mean=np.zeros(6), var=np.zeros(6), cov=np.zeros((6, 6)))
        g = lambda k: _ptr(out.get(k))
        out["state"] = self.lib.ref_scan_steps(C.byref(prm), _ptr(src), C.c_int64(ns), _ptr(tgt), C.c_int64(len(tgt)),
                                               _ptr(init_pose), C.c_int(P), _ptr(_f64(R0)), _ptr(_f64(t0)), C.c_int(steps),
                                               g("x_after"), g("H"), g("b"), g("tgt_paired"), g("src_tr"), g("cand_idx"),
                                               _ptr(out["particles"]), _ptr(out["mean"]), _ptr(out["var"]), _ptr(out["cov"]))
        return out
