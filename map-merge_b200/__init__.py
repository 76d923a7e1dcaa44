"""map-merge_b200 — host-side Python binding of libmm3d.so (ctypes over include/mm3d.h).

The product is the shared library (CUDA kernels for sm_100a behind a C ABI) and
the C++ shim in include/map_merge_3d/.  This module is the thin binding the
tests and bench.py drive it through; it never computes anything itself and it
has no CPU fallback: if libmm3d.so is missing or no CUDA device is usable every
call raises.

Because the directory name carries a hyphen the package is imported through
``mm3d_pkg.load()`` at the repository root (importlib by path).
"""
from __future__ import annotations

import ctypes as C
import weakref
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmm3d.so")

f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_longlong)
f64p = C.POINTER(C.c_double)
u64p = C.POINTER(C.c_uint64)

DESC = dict(PFH=0, PFHRGB=1, FPFH=2, RSD=3, SHOT=4, SC3D=5)
KEYPOINT = dict(SIFT=0, HARRIS=1)
METHOD = dict(MATCHING=0, SAC_IA=1)
STAGES = ["downsampling", "removing outliers", "normals computation", "keypoints detection", "descriptors computation",
          "finding correspondences", "initial alignment", "ICP alignment", "scoring", "graph"]

# every symbol include/mm3d.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "mm3d_params_default", "mm3d_create", "mm3d_destroy", "mm3d_last_error", "mm3d_free", "mm3d_kernel_launches",
    "mm3d_estimate_maps_transforms", "mm3d_compose_maps", "mm3d_downsample", "mm3d_remove_outliers", "mm3d_normals",
    "mm3d_keypoints", "mm3d_descriptors", "mm3d_match", "mm3d_ransac", "mm3d_icp", "mm3d_score", "mm3d_global_transforms",
    "mm3d_maps_upload", "mm3d_maps_free", "mm3d_features_compute", "mm3d_features_count", "mm3d_features_sizes",
    "mm3d_features_export_dev", "mm3d_features_import_dev", "mm3d_features_export_host", "mm3d_features_free",
    "mm3d_register_pairs", "mm3d_estimate_resident", "mm3d_profile_begin", "mm3d_profile_end", "mm3d_sac_ia", "mm3d_knn_stats", "mm3d_compose_shard_begin", "mm3d_compose_shard_size",
    "mm3d_compose_shard_histogram", "mm3d_compose_shard_partition", "mm3d_compose_shard_points", "mm3d_shard_free", "mm3d_downsample_dev",
    "mm3d_knn", "mm3d_knn_tc_audit", "mm3d_create_multi", "mm3d_device_count", "mm3d_comm_id", "mm3d_comm_create", "mm3d_comm_destroy", "mm3d_comm_rank", "mm3d_comm_size",
    "mm3d_dist_block", "mm3d_dist_plan", "mm3d_estimate_maps_transforms_dist", "mm3d_estimate_resident_dist", "mm3d_compose_maps_dist",
    "mm3d_compose_resident_dist", "mm3d_estimate_maps_transforms_layout", "mm3d_compose_maps_layout", "mm3d_maps_upload_layout",
    "mm3d_mapset_create", "mm3d_mapset_update", "mm3d_mapset_size", "mm3d_mapset_estimate", "mm3d_mapset_compose", "mm3d_mapset_free",
]
COMM_ID_BYTES = 128


class Params(C.Structure):
    """mm3d_params == map_merge_3d::MapMergingParams (include/map_merge_3d/map_merging.h:28-44)."""
    _fields_ = [
        ("resolution", C.c_double), ("descriptor_radius", C.c_double), ("outliers_min_neighbours", C.c_int32),
        ("normal_radius", C.c_double), ("keypoint_type", C.c_int32), ("keypoint_threshold", C.c_double),
        ("descriptor_type", C.c_int32), ("estimation_method", C.c_int32), ("refine_transform", C.c_int32),
        ("inlier_threshold", C.c_double), ("max_correspondence_distance", C.c_double), ("max_iterations", C.c_int32),
        ("matching_k", C.c_uint64), ("transform_epsilon", C.c_double), ("confidence_threshold", C.c_double),
        ("output_resolution", C.c_double),
    ]


class Layout(C.Structure):
    """mm3d_layout: byte offsets of x, y, z and rgba inside records of point_step bytes (include/mm3d.h).  record_template
    (outputs only): point_step bytes every output record starts from, or None for zeros."""
    _fields_ = [("point_step", C.c_uint32), ("offset_x", C.c_int32), ("offset_y", C.c_int32), ("offset_z", C.c_int32),
                ("offset_rgba", C.c_int32), ("record_template", C.c_void_p)]

    def __init__(self, point_step, offset_x, offset_y, offset_z, offset_rgba, record_template=None):
        super().__init__(point_step, offset_x, offset_y, offset_z, offset_rgba, None)
        if record_template is not None:
            self._template = (C.c_uint8 * len(record_template)).from_buffer_copy(bytes(record_template))  # kept alive with the layout
            self.record_template = C.addressof(self._template)

    @property
    def template_bytes(self) -> bytes:
        return bytes(self._template) if self.record_template else bytes(self.point_step)


PACKED = Layout(16, 0, 4, 8, 12)
# pcl::PointXYZRGB: x y z, data[3] = 1.0f, rgba, three padding floats; a default-constructed point is (0, 0, 0, 1) with a = 255
PCL_XYZRGB = Layout(32, 0, 4, 8, 16, np.array([0.0, 0.0, 0.0, 1.0], np.float32).tobytes() +
                    np.array([0xff000000, 0, 0, 0], np.uint32).tobytes())


class MM3DError(RuntimeError):
    pass


def build(verbose: bool = False) -> None:
    """Compile libmm3d.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-C", _HERE, "-j8", "all"], stdout=None if verbose else subprocess.DEVNULL)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MM3DError(f"{LIB_PATH} is missing: run __graft_entry__.build() (there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.mm3d_last_error.restype = C.c_char_p
        L.mm3d_last_error.argtypes = [C.c_void_p]
        L.mm3d_kernel_launches.restype = C.c_longlong
        L.mm3d_kernel_launches.argtypes = [C.c_void_p]
        L.mm3d_free.argtypes = [C.c_void_p]
        L.mm3d_destroy.argtypes = [C.c_void_p]
        L.mm3d_maps_free.argtypes = [C.c_void_p]
        L.mm3d_features_free.argtypes = [C.c_void_p]
        L.mm3d_features_count.argtypes = [C.c_void_p]
        L.mm3d_shard_free.argtypes = [C.c_void_p]
        L.mm3d_compose_shard_size.argtypes = [C.c_void_p, u64p]
        L.mm3d_comm_destroy.argtypes = [C.c_void_p]
        L.mm3d_device_count.argtypes = [C.c_void_p]
        L.mm3d_mapset_size.argtypes = [C.c_void_p]
        L.mm3d_mapset_free.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def default_params(**kw) -> Params:
    p = Params()
    lib().mm3d_params_default(C.byref(p))
    for k, v in kw.items():
        if k == "descriptor_type" and isinstance(v, str):
            v = DESC[v]
        if k == "keypoint_type" and isinstance(v, str):
            v = KEYPOINT[v]
        if k == "estimation_method" and isinstance(v, str):
            v = METHOD[v]
        setattr(p, k, v)
    return p


def _f(a, cols=None):
    a = np.ascontiguousarray(a, np.float32)
    if cols is not None and a.size:
        a = a.reshape(-1, cols)
    return a, a.ctypes.data_as(f32p)


def _T_in(T):
    return np.ascontiguousarray(np.asarray(T, np.float32).reshape(4, 4).T)


def _T_out(buf):
    return np.asarray(buf, np.float32).reshape(4, 4).T.copy()


class Context:
    """One mm3d_ctx: a device plus a stream.  ``stream`` is a raw cudaStream_t (int) or None."""

    def __init__(self, device: int = 0, stream: int | None = None, devices=None):
        """devices: a list of CUDA ordinals (or "all") -> mm3d_create_multi: the high-level calls use all of them."""
        self.L = lib()
        self.h = C.c_void_p()
        if devices is not None:
            devs = [] if devices == "all" else [int(d) for d in devices]
            arr = (C.c_int * max(len(devs), 1))(*devs)
            rc = self.L.mm3d_create_multi(C.byref(self.h), arr if devs else None, len(devs))
            if rc != 0:
                raise MM3DError(f"mm3d_create_multi failed ({rc}) for devices {devices}; libmm3d has no CPU fallback")
            return
        rc = self.L.mm3d_create(C.byref(self.h), int(device), C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise MM3DError(f"mm3d_create failed ({rc}): no usable CUDA device {device}; libmm3d has no CPU fallback")

    @property
    def device_count(self) -> int:
        return int(self.L.mm3d_device_count(self.h))

    def close(self):
        if self.h:
            self.L.mm3d_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, ok=(0,)):
        if rc not in ok:
            raise MM3DError(f"mm3d error {rc}: {self.L.mm3d_last_error(self.h).decode()}")
        return rc

    def _take(self, ptr, n, dtype, shape=None):
        n = int(n)
        nbytes = n * np.dtype(dtype).itemsize
        if n and nbytes >= (1 << 20):
            # large outputs (composed maps) are adopted, not copied: the array keeps the library's buffer alive and
            # mm3d_free runs when the last view of it goes away
            addr = C.cast(ptr, C.c_void_p).value
            buf = (C.c_uint8 * nbytes).from_address(addr)
            weakref.finalize(buf, self.L.mm3d_free, C.c_void_p(addr))
            arr = np.frombuffer(buf, dtype)
            return arr.reshape(shape) if shape is not None else arr
        if n == 0:
            arr = np.zeros(0, dtype)
        else:
            arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(nbytes,)).view(dtype).copy()
        if ptr:
            self.L.mm3d_free(C.cast(ptr, C.c_void_p))
        return arr.reshape(shape) if shape is not None else arr

    @property
    def launches(self) -> int:
        return int(self.L.mm3d_kernel_launches(self.h))

    def knn_stats(self):
        out = (C.c_uint64 * 3)()
        self._check(self.L.mm3d_knn_stats(self.h, out))
        return dict(rows=int(out[0]), overflow_rows=int(out[1]), candidates=int(out[2]))  # rows, early flushes, exact evaluations

    def profile_begin(self):
        self._check(self.L.mm3d_profile_begin(self.h))

    def profile_end(self):
        import json
        s = C.c_char_p()
        self._check(self.L.mm3d_profile_end(self.h, C.byref(s)))
        out = json.loads(s.value.decode())
        return out

    # ---- low-level interface ------------------------------------------------
    def downsample(self, pts, resolution):
        a, ap = _f(pts, 4)
        out = f32p(); n = C.c_uint64()
        self._check(self.L.mm3d_downsample(self.h, ap, C.c_uint64(len(a)), C.c_double(resolution), C.byref(out), C.byref(n)))
        return self._take(out, n.value * 4, np.float32, (-1, 4))

    def remove_outliers(self, pts, radius, min_nb, index_leaf=0.0, with_counts=False):
        a, ap = _f(pts, 4)
        out = f32p(); n = C.c_uint64()
        counts = np.zeros(len(a), np.int32)
        self._check(self.L.mm3d_remove_outliers(self.h, ap, C.c_uint64(len(a)), C.c_double(radius), int(min_nb), C.c_double(index_leaf),
                                                C.byref(out), C.byref(n), counts.ctypes.data_as(i32p) if with_counts else None))
        r = self._take(out, n.value * 4, np.float32, (-1, 4))
        return (r, counts) if with_counts else r

    def normals(self, pts, radius, index_leaf=0.0):
        a, ap = _f(pts, 4)
        out = f32p()
        self._check(self.L.mm3d_normals(self.h, ap, C.c_uint64(len(a)), C.c_double(radius), C.c_double(index_leaf), C.byref(out)))
        return self._take(out, len(a) * 4, np.float32, (-1, 4))

    def keypoints(self, pts, normals=None, type="SIFT", threshold=5.0, radius=0.6, resolution=0.1, debug=False):
        a, ap = _f(pts, 4)
        nm, nmp = _f(normals if normals is not None else np.zeros((0, 4)), 4)
        kp = f32p(); nk = C.c_uint64(); dog = f32p(); nd = C.c_uint64()
        self._check(self.L.mm3d_keypoints(self.h, ap, C.c_uint64(len(a)), nmp if len(nm) else None, KEYPOINT[type], C.c_double(threshold),
                                          C.c_double(radius), C.c_double(resolution), C.byref(kp), C.byref(nk),
                                          C.byref(dog) if debug else None, C.byref(nd) if debug else None))
        r = self._take(kp, nk.value * 4, np.float32, (-1, 4))
        if debug:
            return r, self._take(dog, nd.value, np.float32, (-1, 5) if type == "SIFT" else None)  # SIFT: octave-0 DoG; HARRIS: response
        return r

    def descriptors(self, pts, normals, kp, type="FPFH", radius=0.8, index_leaf=0.0, debug=False):
        a, ap = _f(pts, 4); nm, nmp = _f(normals, 4); k, kpp = _f(kp, 4)
        ko = f32p(); nko = C.c_uint64(); desc = f32p(); dim = C.c_int(); sp = f32p()
        self._check(self.L.mm3d_descriptors(self.h, ap, C.c_uint64(len(a)), nmp, kpp, C.c_uint64(len(k)), DESC[type], C.c_double(radius),
                                            C.c_double(index_leaf), C.byref(ko), C.byref(nko), C.byref(desc), C.byref(dim),
                                            C.byref(sp) if debug else None))
        kout = self._take(ko, nko.value * 4, np.float32, (-1, 4))
        d = self._take(desc, nko.value * dim.value, np.float32, (-1, dim.value))
        if debug:  # FPFH: SPFH signatures (n x 33); SHOT: local reference frames (K' x 9)
            if type == "SHOT":
                return kout, d, self._take(sp, nko.value * 9, np.float32, (-1, 9))
            return kout, d, self._take(sp, len(a) * 33, np.float32, (-1, 33))
        return kout, d

    def match(self, ds, dt, k=5):
        a, ap = _f(ds); b, bp = _f(dt)
        dim = a.shape[1] if a.ndim == 2 and a.size else (b.shape[1] if b.ndim == 2 and b.size else 33)
        pairs = i32p(); dist = f32p(); nc = C.c_uint64()
        self._check(self.L.mm3d_match(self.h, ap, C.c_uint64(len(a)), bp, C.c_uint64(len(b)), dim, C.c_uint64(k), C.byref(pairs),
                                      C.byref(dist), C.byref(nc)))
        return self._take(pairs, nc.value * 2, np.int32, (-1, 2)), self._take(dist, nc.value, np.float32)

    def knn(self, a, b, k=5):
        """(idx int32[na, k], dist float32[na, k]): per row of a, its k nearest rows of b by (squared L2, index)."""
        a, ap = _f(a); b, bp = _f(b)
        dim = a.shape[1] if a.ndim == 2 and a.size else (b.shape[1] if b.ndim == 2 and b.size else 33)
        idx = np.full((max(len(a), 1), int(k)), -1, np.int32); dist = np.zeros((max(len(a), 1), int(k)), np.float32)
        self._check(self.L.mm3d_knn(self.h, ap, C.c_uint64(len(a)), bp, C.c_uint64(len(b)), dim, C.c_uint64(int(k)), idx.ctypes.data_as(i32p),
                                    dist.ctypes.data_as(f32p)))
        return idx[:len(a)], dist[:len(a)]

    def knn_tc_audit(self, a, b, k=5):
        """The tensor-core k-NN on one problem plus what its filter saw: dict(idx, dist, acc[na, nb], norm_a, norm_b, err_store)."""
        a, ap = _f(a); b, bp = _f(b)
        na, nb = len(a), len(b)
        idx = np.zeros((na, k), np.int32); dist = np.zeros((na, k), np.float32)
        acc = np.zeros((na, nb), np.float32); n_a = np.zeros(na, np.float32); n_b = np.zeros(nb, np.float32); es = C.c_float()
        self._check(self.L.mm3d_knn_tc_audit(self.h, ap, C.c_uint64(na), bp, C.c_uint64(nb), a.shape[1], C.c_uint64(k), idx.ctypes.data_as(i32p),
                                             dist.ctypes.data_as(f32p), acc.ctypes.data_as(f32p), n_a.ctypes.data_as(f32p),
                                             n_b.ctypes.data_as(f32p), C.byref(es)))
        return dict(idx=idx, dist=dist, acc=acc, norm_a=n_a, norm_b=n_b, err_store=float(es.value))

    def ransac(self, kps, kpt, pairs, inlier_threshold):
        s, sp = _f(kps, 4); t, tp = _f(kpt, 4)
        pr = np.ascontiguousarray(pairs, np.int32)
        T = np.zeros(16, np.float32); inl = i32p(); ni = C.c_uint64(); dbg = (C.c_int32 * 2)(); dd = C.c_double(); bm = np.zeros(16, np.float32)
        self._check(self.L.mm3d_ransac(self.h, sp, C.c_uint64(len(s)), tp, C.c_uint64(len(t)), pr.ctypes.data_as(i32p), C.c_uint64(len(pr)),
                                       C.c_double(inlier_threshold), T.ctypes.data_as(f32p), C.byref(inl), C.byref(ni), dbg, C.byref(dd),
                                       bm.ctypes.data_as(f32p)))
        i = self._take(inl, ni.value, np.int32)
        return _T_out(T), i, dict(iterations=dbg[0], best_count=dbg[1], sample_dist_thresh=dd.value, best_model=_T_out(bm))

    def sac_ia(self, kps, ds, kpt, dt, min_sample_distance, max_corr_dist, max_iterations, rand_calls=0):
        s, sp = _f(kps, 4); t, tp = _f(kpt, 4); a, ap = _f(ds); b, bp = _f(dt)
        dim = a.shape[1] if a.ndim == 2 and a.size else 33
        T = np.zeros(16, np.float32); rc = C.c_uint64(rand_calls); err = f32p(); ne = C.c_uint64()
        self._check(self.L.mm3d_sac_ia(self.h, sp, C.c_uint64(len(s)), ap, tp, C.c_uint64(len(t)), bp, dim, C.c_double(min_sample_distance),
                                       C.c_double(max_corr_dist), int(max_iterations), C.byref(rc), T.ctypes.data_as(f32p), C.byref(err),
                                       C.byref(ne)))
        e = self._take(err, ne.value, np.float32)
        return _T_out(T), dict(rand_calls=rc.value, errors=e)

    def icp(self, src, tgt, T0, max_dist, max_it, eps, index_leaf=0.0, outlier_threshold=0.5):
        s, sp = _f(src, 4); t, tp = _f(tgt, 4)
        T0c = _T_in(T0)
        T = np.zeros(16, np.float32); dbg = (C.c_int32 * 2)(); sums = i64p(); ns = C.c_uint64()
        self._check(self.L.mm3d_icp(self.h, sp, C.c_uint64(len(s)), tp, C.c_uint64(len(t)), T0c.ctypes.data_as(f32p), C.c_double(max_dist),
                                    C.c_double(outlier_threshold), int(max_it), C.c_double(eps), C.c_double(index_leaf),
                                    T.ctypes.data_as(f32p), dbg, C.byref(sums), C.byref(ns)))
        sm = self._take(sums, ns.value * 17, np.int64, (-1, 17))
        return _T_out(T), dict(iterations=dbg[0], converged=dbg[1], sums=sm)

    def score(self, src, tgt, T, max_distance, index_leaf=0.0):
        s, sp = _f(src, 4); t, tp = _f(tgt, 4)
        Tc = _T_in(T)
        out = C.c_double()
        self._check(self.L.mm3d_score(self.h, sp, C.c_uint64(len(s)), tp, C.c_uint64(len(t)), Tc.ctypes.data_as(f32p), C.c_double(max_distance),
                                      C.c_double(index_leaf), C.byref(out)))
        return out.value

    # ---- high-level interface -----------------------------------------------
    @staticmethod
    def _cloud_args(clouds):
        m = len(clouds)
        arrs = [np.ascontiguousarray(c, np.float32).reshape(-1, 4) if c is not None else None for c in clouds]
        ptrs = (f32p * max(m, 1))(*[(a.ctypes.data_as(f32p) if a is not None and len(a) else f32p()) for a in arrs])
        ns = (C.c_uint64 * max(m, 1))(*[(len(a) if a is not None else 0) for a in arrs])
        return arrs, ptrs, ns

    @staticmethod
    def _record_args(clouds, layout: Layout):
        """clouds: C-contiguous uint8 arrays of shape (n, layout.point_step), or None for an empty map."""
        m = len(clouds)
        arrs = []
        for c in clouds:
            if c is not None:
                c = np.asarray(c)
                if c.dtype != np.uint8 or c.ndim != 2 or c.shape[1] != layout.point_step or not c.flags.c_contiguous:
                    raise ValueError(f"records must be a C-contiguous uint8 array of shape (n, {layout.point_step}), got {c.dtype} {c.shape}")
            arrs.append(c)
        ptrs = (C.c_void_p * max(m, 1))(*[(a.ctypes.data if a is not None and len(a) else None) for a in arrs])
        ns = (C.c_uint64 * max(m, 1))(*[(len(a) if a is not None else 0) for a in arrs])
        return arrs, ptrs, ns

    def estimate_maps_transforms_layout(self, clouds, layout: Layout, params: Params):
        """estimate_maps_transforms on records in `layout` (converted on the GPU)."""
        arrs, ptrs, ns = self._record_args(clouds, layout)
        m = len(clouds)
        out = np.zeros((max(m, 1), 16), np.float32); no = C.c_int()
        self._check(self.L.mm3d_estimate_maps_transforms_layout(self.h, m, ptrs, ns, C.byref(layout), C.byref(params), out.ctypes.data_as(f32p),
                                                                C.byref(no)))
        return out[:no.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()

    def compose_maps_layout(self, clouds, transforms, resolution, in_layout: Layout, out_layout: Layout):
        """compose_maps on records in `in_layout`; returns uint8[n, out_layout.point_step] records (None for no maps)."""
        arrs, ptrs, ns = self._record_args(clouds, in_layout)
        T = np.asarray(transforms, np.float32).reshape(-1, 4, 4)
        Tc = np.ascontiguousarray(T.transpose(0, 2, 1)) if len(T) else np.zeros((1, 16), np.float32)
        out = C.c_void_p(); n = C.c_uint64()
        rc = self.L.mm3d_compose_maps_layout(self.h, len(clouds), ptrs, ns, C.byref(in_layout), len(T), Tc.ctypes.data_as(f32p),
                                             C.c_double(resolution), C.byref(out_layout), C.byref(out), C.byref(n))
        if rc == 1:
            return None
        self._check(rc)
        return self._take(out, n.value * out_layout.point_step, np.uint8, (-1, out_layout.point_step))

    def maps_upload_layout(self, clouds, layout: Layout):
        arrs, ptrs, ns = self._record_args(clouds, layout)
        h = C.c_void_p()
        self._check(self.L.mm3d_maps_upload_layout(self.h, len(clouds), ptrs, ns, C.byref(layout), C.byref(h)))
        return Maps(self, h, len(clouds))

    def estimate_maps_transforms(self, clouds, params: Params):
        arrs, ptrs, ns = self._cloud_args(clouds)
        m = len(clouds)
        out = np.zeros((max(m, 1), 16), np.float32); no = C.c_int()
        self._check(self.L.mm3d_estimate_maps_transforms(self.h, m, ptrs, ns, C.byref(params), out.ctypes.data_as(f32p), C.byref(no)))
        return out[:no.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()

    def compose_maps(self, clouds, transforms, resolution):
        arrs, ptrs, ns = self._cloud_args(clouds)
        T = np.asarray(transforms, np.float32).reshape(-1, 4, 4)
        Tc = np.ascontiguousarray(T.transpose(0, 2, 1)) if len(T) else np.zeros((1, 16), np.float32)
        out = f32p(); n = C.c_uint64()
        rc = self.L.mm3d_compose_maps(self.h, len(clouds), ptrs, ns, len(T), Tc.ctypes.data_as(f32p), C.c_double(resolution), C.byref(out),
                                      C.byref(n))
        if rc == 1:
            return None
        if rc == -3:
            raise MM3DError("composeMaps: clouds and transforms size must be the same.")
        self._check(rc)
        return self._take(out, n.value * 4, np.float32, (-1, 4))

    # ---- multi-GPU interface (one process per GPU) -------------------------------
    def comm_create(self, rank: int, world: int, comm_id: bytes) -> "Comm":
        h = C.c_void_p()
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(bytes(comm_id)[:COMM_ID_BYTES].ljust(COMM_ID_BYTES, b"\0"))
        self._check(self.L.mm3d_comm_create(self.h, int(rank), int(world), buf, C.byref(h)))
        return Comm(self, h, rank, world)

    def estimate_maps_transforms_dist(self, comm, clouds, params: Params):
        """clouds: ALL maps of the job (entries outside this rank's block may be None)."""
        arrs, ptrs, ns = self._cloud_args(clouds)
        m = len(clouds)
        out = np.zeros((max(m, 1), 16), np.float32); no = C.c_int()
        self._check(self.L.mm3d_estimate_maps_transforms_dist(self.h, comm.h if comm else None, m, ptrs, ns, C.byref(params),
                                                              out.ctypes.data_as(f32p), C.byref(no)))
        return out[:no.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()

    def estimate_resident_dist(self, comm, n_maps: int, local_maps: "Maps", params: Params, phases=False):
        out = np.zeros((max(n_maps, 1), 16), np.float32); no = C.c_int(); ph = np.zeros(5, np.float32)
        self._check(self.L.mm3d_estimate_resident_dist(self.h, comm.h if comm else None, int(n_maps), local_maps.h, C.byref(params),
                                                       out.ctypes.data_as(f32p), C.byref(no), ph.ctypes.data_as(f32p) if phases else None))
        T = out[:no.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()
        return (T, dict(zip(DIST_PHASES, ph.tolist()))) if phases else T

    def compose_maps_dist(self, comm, clouds_local, transforms_local, resolution):
        arrs, ptrs, ns = self._cloud_args(clouds_local)
        T = np.asarray(transforms_local, np.float32).reshape(-1, 4, 4)
        Tc = np.ascontiguousarray(T.transpose(0, 2, 1)) if len(T) else np.zeros((1, 16), np.float32)
        out = f32p(); n = C.c_uint64()
        rc = self.L.mm3d_compose_maps_dist(self.h, comm.h if comm else None, len(clouds_local), ptrs, ns, len(T), Tc.ctypes.data_as(f32p),
                                           C.c_double(resolution), C.byref(out), C.byref(n))
        if rc == -3:
            raise MM3DError("composeMaps: clouds and transforms size must be the same.")
        self._check(rc)
        return self._take(out, n.value * 4, np.float32, (-1, 4))

    def compose_resident_dist(self, comm, local_maps: "Maps", transforms_local, resolution):
        T = np.asarray(transforms_local, np.float32).reshape(-1, 4, 4)
        Tc = np.ascontiguousarray(T.transpose(0, 2, 1)) if len(T) else np.zeros((1, 16), np.float32)
        out = f32p(); n = C.c_uint64()
        rc = self.L.mm3d_compose_resident_dist(self.h, comm.h if comm else None, local_maps.h, len(T), Tc.ctypes.data_as(f32p),
                                               C.c_double(resolution), C.byref(out), C.byref(n))
        if rc == -3:
            raise MM3DError("composeMaps: clouds and transforms size must be the same.")
        self._check(rc)
        return self._take(out, n.value * 4, np.float32, (-1, 4))

    # ---- composeMaps sharded over ranks ----------------------------------------
    def compose_shard_begin(self, clouds, transforms):
        arrs, ptrs, ns = self._cloud_args(clouds)
        T = np.asarray(transforms, np.float32).reshape(-1, 4, 4)
        Tc = np.ascontiguousarray(T.transpose(0, 2, 1)) if len(T) else np.zeros((1, 16), np.float32)
        bbox = np.zeros(6, np.float32); h = C.c_void_p()
        self._check(self.L.mm3d_compose_shard_begin(self.h, len(clouds), ptrs, ns, len(T), Tc.ctypes.data_as(f32p), bbox.ctypes.data_as(f32p),
                                                    C.byref(h)))
        n = C.c_uint64()
        self.L.mm3d_compose_shard_size(h, C.byref(n))
        return bbox, h, int(n.value)

    def compose_shard_histogram(self, shard, global_bbox, resolution, n_buckets=4096):
        gb = np.ascontiguousarray(global_bbox, np.float32); hist = np.zeros(n_buckets, np.uint64)
        rc = self._check(self.L.mm3d_compose_shard_histogram(self.h, shard, gb.ctypes.data_as(f32p), C.c_double(resolution), int(n_buckets),
                                                             hist.ctypes.data_as(u64p)), ok=(0, 1))
        return None if rc == 1 else hist

    def compose_shard_partition(self, shard, global_bbox, resolution, splitters, out_dev_ptr, n_buckets=4096):
        gb = np.ascontiguousarray(global_bbox, np.float32); sp = np.ascontiguousarray(splitters, np.int32)
        n_ranks = len(sp) - 1
        counts = np.zeros(n_ranks, np.uint64)
        self._check(self.L.mm3d_compose_shard_partition(self.h, shard, gb.ctypes.data_as(f32p), C.c_double(resolution), int(n_buckets), n_ranks,
                                                        sp.ctypes.data_as(i32p), counts.ctypes.data_as(u64p), C.c_void_p(int(out_dev_ptr))))
        return counts.astype(np.int64)

    def compose_shard_points(self, shard):
        out = f32p(); no = C.c_uint64()
        self._check(self.L.mm3d_compose_shard_points(self.h, shard, C.byref(out), C.byref(no)))
        return self._take(out, no.value * 4, np.float32, (-1, 4))

    def shard_free(self, shard):
        self.L.mm3d_shard_free(shard)

    def downsample_dev(self, dev_ptr, n, resolution):
        out = f32p(); no = C.c_uint64()
        self._check(self.L.mm3d_downsample_dev(self.h, C.c_void_p(int(dev_ptr)), C.c_uint64(int(n)), C.c_double(resolution), C.byref(out), C.byref(no)))
        return self._take(out, no.value * 4, np.float32, (-1, 4))

    # ---- resident interface ---------------------------------------------------
    def maps_upload(self, clouds):
        arrs, ptrs, ns = self._cloud_args(clouds)
        h = C.c_void_p()
        self._check(self.L.mm3d_maps_upload(self.h, len(clouds), ptrs, ns, C.byref(h)))
        return Maps(self, h, len(clouds))

    def estimate_resident(self, maps: "Maps", params: Params, stage_times=False):
        out = np.zeros((max(maps.n, 1), 16), np.float32); no = C.c_int(); st = np.zeros(10, np.float32)
        self._check(self.L.mm3d_estimate_resident(self.h, maps.h, C.byref(params), out.ctypes.data_as(f32p), C.byref(no),
                                                  st.ctypes.data_as(f32p) if stage_times else None))
        T = out[:no.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()
        return (T, dict(zip(STAGES, st.tolist()))) if stage_times else T

    def mapset(self) -> "MapSet":
        """An empty map set on this context (mm3d_mapset_create): resident maps that re-estimate only what changed."""
        h = C.c_void_p()
        self._check(self.L.mm3d_mapset_create(self.h, C.byref(h)))
        return MapSet(self, h)

    def features_compute(self, maps: "Maps", first: int, count: int, params: Params):
        h = C.c_void_p()
        self._check(self.L.mm3d_features_compute(self.h, maps.h, int(first), int(count), C.byref(params), C.byref(h)))
        return Features(self, h)

    def features_import_dev(self, n_points, point_ptrs, n_keypoints, kp_ptrs, desc_ptrs, dim=33):
        m = len(n_points)
        npt = (C.c_int32 * m)(*[int(x) for x in n_points]); nk = (C.c_int32 * m)(*[int(x) for x in n_keypoints])
        pp = (C.c_void_p * m)(*[C.c_void_p(int(x)) for x in point_ptrs])
        kp = (C.c_void_p * m)(*[C.c_void_p(int(x)) for x in kp_ptrs])
        dp = (C.c_void_p * m)(*[C.c_void_p(int(x)) for x in desc_ptrs])
        h = C.c_void_p()
        self._check(self.L.mm3d_features_import_dev(self.h, m, npt, pp, nk, kp, dp, int(dim), C.byref(h)))
        return Features(self, h)

    def register_pairs(self, feats: "Features", ij, params: Params):
        ij = np.ascontiguousarray(ij, np.int32).reshape(-1, 2)
        P = len(ij)
        T = np.zeros((max(P, 1), 16), np.float32); conf = np.zeros(max(P, 1), np.float64); stats = np.zeros((max(P, 1), 4), np.int32)
        self._check(self.L.mm3d_register_pairs(self.h, feats.h, P, ij.ctypes.data_as(i32p), C.byref(params), T.ctypes.data_as(f32p),
                                               conf.ctypes.data_as(f64p), stats.ctypes.data_as(i32p)))
        return T[:P].reshape(-1, 4, 4).transpose(0, 2, 1).copy(), conf[:P].copy(), stats[:P].copy()


DIST_PHASES = ["features", "feature exchange", "pair registration", "result exchange", "graph"]


def comm_id() -> bytes:
    """rank 0: an ncclUniqueId to hand to every rank (mm3d_comm_id)."""
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    rc = lib().mm3d_comm_id(buf)
    if rc != 0:
        raise MM3DError(f"mm3d_comm_id failed ({rc}): NCCL is not available")
    return bytes(buf)


def dist_block(rank: int, world: int, n_maps: int):
    first = C.c_int(); count = C.c_int()
    if lib().mm3d_dist_block(int(rank), int(world), int(n_maps), C.byref(first), C.byref(count)) != 0:
        raise MM3DError("mm3d_dist_block: bad arguments")
    return first.value, count.value


def dist_plan(n_points, n_keypoints, dim: int, world: int):
    """(pairs int32[n, 2], owner int32[n]): the row-major pair list and the rank that registers each pair."""
    npt = np.ascontiguousarray(n_points, np.int32); nk = np.ascontiguousarray(n_keypoints, np.int32)
    m = len(npt)
    cap = max(m * (m - 1) // 2, 1)
    pairs = np.zeros((cap, 2), np.int32); owner = np.zeros(cap, np.int32); n = C.c_int()
    if lib().mm3d_dist_plan(m, npt.ctypes.data_as(i32p), nk.ctypes.data_as(i32p), int(dim), int(world), pairs.ctypes.data_as(i32p),
                            owner.ctypes.data_as(i32p), C.byref(n)) != 0:
        raise MM3DError("mm3d_dist_plan: bad arguments")
    return pairs[:n.value].copy(), owner[:n.value].copy()


class Comm:
    def __init__(self, ctx, h, rank, world):
        self.ctx, self.h, self.rank, self.world = ctx, h, rank, world

    def free(self):
        if self.h:
            self.ctx.L.mm3d_comm_destroy(self.h)
            self.h = C.c_void_p()


def global_transforms(st, transforms, conf, thr, debug=False):
    """computeGlobalTransforms on the host (no device needed)."""
    L = lib()
    st = np.ascontiguousarray(st, np.int32).reshape(-1, 2)
    conf = np.ascontiguousarray(conf, np.float64)
    n = len(st)
    Tc = np.ascontiguousarray(np.asarray(transforms, np.float32).reshape(-1, 4, 4).transpose(0, 2, 1)) if n else np.zeros((1, 16), np.float32)
    nodes = int(st.max()) + 1 if n else 0
    out = np.zeros((max(nodes, 1), 16), np.float32); no = C.c_int(); ref = C.c_int()
    # capacities per include/mm3d.h: tree edges (listed from both ends) < 2 x nodes, centres <= nodes (every isolated node below the max index is a centre)
    inc = np.zeros(max(n, 1), np.int32); te = np.zeros((2 * nodes + 2, 2), np.int32); nte = C.c_int(); cen = np.zeros(nodes + 1, np.int32); nc = C.c_int()
    rc = L.mm3d_global_transforms(n, st.ctypes.data_as(i32p), Tc.ctypes.data_as(f32p), conf.ctypes.data_as(f64p), C.c_double(thr),
                                  out.ctypes.data_as(f32p), C.byref(no), C.byref(ref), inc.ctypes.data_as(i32p), te.ctypes.data_as(i32p),
                                  C.byref(nte), cen.ctypes.data_as(i32p), C.byref(nc))
    if rc != 0:
        raise MM3DError(f"mm3d_global_transforms failed ({rc})")
    T = out[:no.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()
    if debug:
        return T, ref.value, inc[:n].copy(), te[:nte.value].copy(), cen[:nc.value].copy()
    return T, ref.value


class Maps:
    def __init__(self, ctx: Context, h, n):
        self.ctx, self.h, self.n = ctx, h, n

    def free(self):
        if self.h:
            self.ctx.L.mm3d_maps_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Features:
    def __init__(self, ctx: Context, h):
        self.ctx, self.h = ctx, h
        self.n = int(ctx.L.mm3d_features_count(h))

    def sizes(self):
        npt = np.zeros(max(self.n, 1), np.int32); nk = np.zeros(max(self.n, 1), np.int32); dim = C.c_int32()
        self.ctx.L.mm3d_features_sizes(self.h, npt.ctypes.data_as(i32p), nk.ctypes.data_as(i32p), C.byref(dim))
        return npt[:self.n].copy(), nk[:self.n].copy(), dim.value

    def export_host(self, m):
        npt, nk, dim = self.sizes()
        pts = np.zeros((npt[m], 4), np.float32); kp = np.zeros((nk[m], 4), np.float32); desc = np.zeros((nk[m], dim), np.float32)
        self.ctx._check(self.ctx.L.mm3d_features_export_host(self.ctx.h, self.h, int(m), pts.ctypes.data_as(f32p), kp.ctypes.data_as(f32p),
                                                             desc.ctypes.data_as(f32p)))
        return pts, kp, desc

    def export_dev(self, m, pts_ptr, kp_ptr, desc_ptr):
        self.ctx._check(self.ctx.L.mm3d_features_export_dev(self.ctx.h, self.h, int(m), C.c_void_p(int(pts_ptr)), C.c_void_p(int(kp_ptr)),
                                                            C.c_void_p(int(desc_ptr))))

    def free(self):
        if self.h:
            self.ctx.L.mm3d_features_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class MapSet:
    """mm3d_mapset: one slot per robot; each keeps its cloud, features and pair results on the device between calls.
    estimate() and compose() return bit for bit what estimate_maps_transforms and compose_maps_layout return on the slots'
    current clouds in slot order."""

    def __init__(self, ctx: Context, h):
        self.ctx, self.h = ctx, h

    def __len__(self):
        return int(self.ctx.L.mm3d_mapset_size(self.h))

    def update(self, clouds: dict, layout: Layout | None = None) -> list:
        """clouds = {slot: cloud or None}: float32[n, 4] points, or uint8[n, layout.point_step] records when a layout is
        given.  Returns, per entry in the dict's order, whether the slot's cloud changed (bit for bit)."""
        slots = [int(k) for k in clouds]
        values = list(clouds.values())
        if layout is None:
            arrs, ptrs, ns = self.ctx._cloud_args(values)
            layout = PACKED
        else:
            arrs, ptrs, ns = self.ctx._record_args(values, layout)
        n = len(slots)
        sl = (C.c_int32 * max(n, 1))(*slots)
        changed = (C.c_int32 * max(n, 1))()
        self.ctx._check(self.ctx.L.mm3d_mapset_update(self.ctx.h, self.h, n, sl, ptrs, ns, C.byref(layout), changed))
        return [bool(changed[i]) for i in range(n)]

    def estimate(self, params: Params, work: bool = False):
        """Transforms as estimate_maps_transforms returns them; work=True also returns [maps whose features were computed,
        pairs registered, pairs reused]."""
        m = len(self)
        out = np.zeros((max(m, 1), 16), np.float32); no = C.c_int(); w = (C.c_int32 * 3)()
        self.ctx._check(self.ctx.L.mm3d_mapset_estimate(self.ctx.h, self.h, C.byref(params), out.ctypes.data_as(f32p), C.byref(no), w))
        T = out[:no.value].reshape(-1, 4, 4).transpose(0, 2, 1).copy()
        return (T, [int(x) for x in w]) if work else T

    def compose(self, transforms, resolution, out_layout: Layout | None = None):
        """compose_maps over the slots: float32[n, 4] points, or uint8[n, out_layout.point_step] records when out_layout is
        given; None for a set without slots."""
        T = np.asarray(transforms, np.float32).reshape(-1, 4, 4)
        Tc = np.ascontiguousarray(T.transpose(0, 2, 1)) if len(T) else np.zeros((1, 16), np.float32)
        layout = PACKED if out_layout is None else out_layout
        out = C.c_void_p(); n = C.c_uint64()
        rc = self.ctx.L.mm3d_mapset_compose(self.ctx.h, self.h, len(T), Tc.ctypes.data_as(f32p), C.c_double(resolution), C.byref(layout),
                                            C.byref(out), C.byref(n))
        if rc == 1:
            return None
        self.ctx._check(rc)
        if out_layout is None:
            return self.ctx._take(out, n.value * 4, np.float32, (-1, 4))
        return self.ctx._take(out, n.value * layout.point_step, np.uint8, (-1, layout.point_step))

    def free(self):
        if self.h:
            self.ctx.L.mm3d_mapset_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
