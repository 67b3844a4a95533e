"""ctypes binding of the C ABI in include/ilsm.h plus a thin host-side mirror of the reference call sites.

The product path is libilsm_cuda.so; this module only marshals numpy / torch buffers into it.  There is no CPU
fallback: if the shared library is missing or no CUDA device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build

ILSM_OK = 0
ILSM_ERR_NOT_ENOUGH_MAP = -4
CONVERGENCE, NO_CONVERGENCE, FAILURE = 0, 1, 2
MAX_OUTER = 8


class IlsmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ilsm error {code}: {msg}")
        self.code = code


class RegOpts(C.Structure):
    _fields_ = [("outer_iterations", C.c_int32), ("max_num_iterations", C.c_int32), ("huber_a", C.c_double),
                ("knn_gate_sq", C.c_float), ("reserved0", C.c_float), ("line_eig_ratio", C.c_double),
                ("plane_tol", C.c_double), ("min_corner_map", C.c_int32), ("min_surf_map", C.c_int32)]


class SolveSummary(C.Structure):
    _fields_ = [("termination", C.c_int32), ("iterations", C.c_int32), ("num_successful_steps", C.c_int32),
                ("num_unsuccessful_steps", C.c_int32), ("num_edge_factors", C.c_int32),
                ("num_plane_factors", C.c_int32), ("num_evaluations", C.c_int32), ("reserved", C.c_int32),
                ("initial_cost", C.c_double), ("final_cost", C.c_double)]


class RegReport(C.Structure):
    _fields_ = [("passes", C.c_int32), ("reserved", C.c_int32), ("pass_", SolveSummary * MAX_OUTER)]


class FeatureCounts(C.Structure):
    _fields_ = [("n_cloud", C.c_int32), ("n_sharp", C.c_int32), ("n_less_sharp", C.c_int32), ("n_flat", C.c_int32),
                ("n_less_flat", C.c_int32), ("flags", C.c_int32), ("ring_start", C.c_int32 * 64),
                ("ring_end", C.c_int32 * 64)]


class Features(C.Structure):
    _fields_ = [("cloud_xyzi", C.c_void_p), ("curvature", C.c_void_p), ("label", C.c_void_p), ("src_index", C.c_void_p),
                ("sharp_idx", C.c_void_p), ("less_sharp_idx", C.c_void_p), ("flat_idx", C.c_void_p),
                ("less_flat_xyzi", C.c_void_p), ("counts", FeatureCounts)]


class CubeMapStats(C.Structure):
    _fields_ = [("n_map_corner", C.c_int32), ("n_map_surf", C.c_int32), ("n_stack_corner", C.c_int32),
                ("n_stack_surf", C.c_int32), ("ran_optimization", C.c_int32), ("n_valid", C.c_int32),
                ("cen", C.c_int32 * 3), ("flags", C.c_int32)]


class SlamStats(C.Structure):
    _fields_ = [("n_cloud", C.c_int32), ("n_sharp", C.c_int32), ("n_less_sharp", C.c_int32), ("n_flat", C.c_int32),
                ("n_less_flat", C.c_int32), ("ran_odometry", C.c_int32), ("odometry", RegReport), ("mapping", RegReport),
                ("cubemap", CubeMapStats)]


class Pc2Layout(C.Structure):
    """ilsm_pc2_layout: where x / y / z / intensity sit inside one point of a sensor_msgs/PointCloud2 blob."""
    _fields_ = [("point_step", C.c_int32), ("off_x", C.c_int32), ("off_y", C.c_int32), ("off_z", C.c_int32),
                ("off_intensity", C.c_int32), ("intensity_datatype", C.c_int32), ("is_bigendian", C.c_int32),
                ("reserved", C.c_int32)]


class GroundOpts(C.Structure):
    _fields_ = [("z_min", C.c_double), ("z_max", C.c_double), ("distance_threshold", C.c_double), ("probability", C.c_double),
                ("max_iterations", C.c_int32), ("seed", C.c_int32), ("band", C.c_double), ("max_angle_deg", C.c_double)]


class GroundInfo(C.Structure):
    _fields_ = [("n_band", C.c_int32), ("best_hypothesis", C.c_int32), ("n_best_inliers", C.c_int32), ("iterations", C.c_int32),
                ("accepted", C.c_int32), ("reserved", C.c_int32)]


class MapOptStats(C.Structure):
    _fields_ = [("ground", GroundInfo), ("ground_coeff", C.c_float * 4), ("n_ground", C.c_int32), ("n_plane_in", C.c_int32),
                ("n_query", C.c_int32), ("ran_optimization", C.c_int32), ("converged", C.c_int32), ("map_size", C.c_int32),
                ("solve", SolveSummary), ("q_key", C.c_double * 4), ("t_key", C.c_double * 3), ("reserved", C.c_double)]


class IcpOpts(C.Structure):
    """ilsm_icp_opts (pcl::IterativeClosestPoint's settings); IcpOpts() holds PCL 1.10's defaults."""
    _fields_ = [("max_correspondence_distance", C.c_double), ("max_iterations", C.c_int32), ("pad", C.c_int32),
                ("transformation_epsilon", C.c_double), ("transformation_rotation_epsilon", C.c_double),
                ("euclidean_fitness_epsilon", C.c_double), ("fitness_max_range", C.c_double)]

    def __init__(self, **kw):
        super().__init__()
        load_library().ilsm_icp_opts_default(C.byref(self))
        for k, v in kw.items():
            setattr(self, k, v)


ICP_NOT_CONVERGED, ICP_ITERATIONS, ICP_TRANSFORM, ICP_ABS_MSE, ICP_REL_MSE, ICP_NO_CORRESPONDENCES = range(6)


class IcpResult(C.Structure):
    """ilsm_icp_result: final transformation (source -> target), getFitnessScore, convergence state."""
    _fields_ = [("q_xyzw", C.c_double * 4), ("t", C.c_double * 3), ("fitness", C.c_double), ("mse", C.c_double),
                ("iterations", C.c_int32), ("state", C.c_int32), ("converged", C.c_int32), ("n_correspondences", C.c_int32)]

    @property
    def q(self):
        return np.array(self.q_xyzw[:], np.float64)

    @property
    def tv(self):
        return np.array(self.t[:], np.float64)


DMATCH_DTYPE = np.dtype([("queryIdx", "<i4"), ("trainIdx", "<i4"), ("imgIdx", "<i4"), ("distance", "<f4")])
FACTOR_DTYPE = np.dtype([("type", "<i4"), ("src", "<i4"), ("p", "<f8", 3), ("a", "<f8", 3), ("b", "<f8", 3)])

_lib = None


def pc2_layout_ouster() -> Pc2Layout:
    lay = Pc2Layout()
    load_library().ilsm_pc2_layout_ouster(C.byref(lay))
    return lay


def load_library(path: str | None = None):
    """dlopen libilsm_cuda.so (built in-tree by _build.build()).  Raises if it is absent: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or _build.LIB
    if not os.path.exists(path):
        raise IlsmError(-100, f"{path} not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    vp, i32, f32, f64 = C.c_void_p, C.c_int, C.c_float, C.c_double
    sig = {
        "ilsm_abi_version": (i32, []),
        "ilsm_last_error": (C.c_char_p, []),
        "ilsm_create": (i32, [i32, C.POINTER(vp)]),
        "ilsm_destroy": (None, [vp]),
        "ilsm_sync": (i32, [vp]),
        "ilsm_stream": (vp, [vp]),
        "ilsm_set_async": (i32, [vp, i32]),
        "ilsm_map_create": (i32, [vp, C.POINTER(vp)]),
        "ilsm_map_destroy": (None, [vp]),
        "ilsm_map_size": (i32, [vp]),
        "ilsm_map_build": (i32, [vp, vp, i32, i32, f32]),
        "ilsm_map_build_dev": (i32, [vp, vp, i32, i32, f32]),
        "ilsm_map_join": (i32, [vp]),
        "ilsm_knn": (i32, [vp, vp, i32, i32, i32, f32, vp, vp]),
        "ilsm_map_insert": (i32, [vp, vp, i32, i32, i32, f32]),
        "ilsm_map_points": (i32, [vp, vp, i32, C.POINTER(i32)]),
        "ilsm_knn_dev": (i32, [vp, vp, i32, i32, i32, f32, vp, vp]),
        "ilsm_reg_opts_default": (None, [C.POINTER(RegOpts)]),
        "ilsm_register": (i32, [vp, vp, vp, vp, i32, vp, i32, i32, vp, vp, C.POINTER(RegOpts), C.POINTER(RegReport)]),
        "ilsm_register_dev": (i32, [vp, vp, vp, vp, i32, vp, i32, i32, vp, C.POINTER(RegOpts), vp]),
        "ilsm_associate": (i32, [vp, vp, vp, vp, i32, vp, i32, i32, vp, vp, C.POINTER(RegOpts), vp, vp, vp]),
        "ilsm_project": (i32, [vp, vp, i32, i32, i32, vp, vp, vp]),
        "ilsm_project_dev": (i32, [vp, vp, i32, i32, i32, vp, vp, vp]),
        "ilsm_extract_features": (i32, [vp, vp, i32, i32, f32, C.POINTER(Features)]),
        "ilsm_voxelgrid": (i32, [vp, vp, i32, i32, f32, vp, C.POINTER(i32)]),
        "ilsm_map_build_pair_dev": (i32, [vp, vp, i32, vp, vp, i32, i32, C.c_float]),
        "ilsm_register_frame": (i32, [vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, C.c_float, vp, vp, vp, vp, vp]),
        "ilsm_register_frame_dev": (i32, [vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, C.c_float, vp, vp]),
        "ilsm_sc_create": (i32, [vp, C.POINTER(vp)]),
        "ilsm_sc_destroy": (None, [vp]),
        "ilsm_sc_size": (i32, [vp]),
        "ilsm_sc_make": (i32, [vp, vp, i32, i32, vp]),
        "ilsm_sc_add": (i32, [vp, vp, i32]),
        "ilsm_sc_add_dev": (i32, [vp, vp, i32]),
        "ilsm_sc_query_topk": (i32, [vp, vp, i32, i32, i32, vp, vp, vp]),
        "ilsm_sc_query_topk_dev": (i32, [vp, vp, i32, i32, i32, vp, vp, vp]),
        "ilsm_sc_merge_topk_dev": (i32, [vp, vp, i32, i32, vp]),
        "ilsm_sc_merge_topk": (i32, [vp, vp, vp, i32, i32, vp, vp, vp]),
        "ilsm_sc_query_candidates": (i32, [vp, vp, i32, i32, vp, vp, vp, vp]),
        "ilsm_sc_query_topk_batch": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp]),
        "ilsm_sc_query_topk_batch_dev": (i32, [vp, vp, i32, i32, i32, i32, vp]),
        "ilsm_sc_prefilter_debug": (i32, [vp, vp, i32, i32, vp, vp]),
        "ilsm_sc_nccl_unique_id": (i32, [vp]),
        "ilsm_sc_init_nccl_rank": (i32, [vp, vp, i32, i32]),
        "ilsm_sc_init_nccl": (i32, [vp, vp, i32, i32]),
        "ilsm_sc_nccl_version": (i32, [vp]),
        "ilsm_sc_query_topk_sharded": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp]),
        "ilsm_sc_query_topk_sharded_dev": (i32, [vp, vp, i32, i32, i32, i32, vp]),
        "ilsm_odometry": (i32, [vp, vp, vp, vp, i32, vp, i32, i32, vp, vp, C.POINTER(RegOpts), C.POINTER(RegReport), vp]),
        "ilsm_cubemap_create": (i32, [vp, f32, f32, i32, C.POINTER(vp)]),
        "ilsm_cubemap_destroy": (None, [vp]),
        "ilsm_cubemap_insert_world": (i32, [vp, vp, i32, vp, i32, i32, vp]),
        "ilsm_cubemap_frame": (i32, [vp, vp, i32, vp, i32, i32, vp, vp, vp, vp, C.POINTER(RegOpts), C.POINTER(RegReport),
                                     C.POINTER(CubeMapStats)]),
        "ilsm_cubemap_cube": (i32, [vp, i32, i32, vp, i32, C.POINTER(i32)]),
        "ilsm_slam_create": (i32, [vp, f32, f32, f32, i32, C.POINTER(vp)]),
        "ilsm_slam_create_mapopt": (i32, [vp, f32, f32, f32, C.POINTER(vp)]),
        "ilsm_slam_destroy": (None, [vp]),
        "ilsm_slam_cubemap": (vp, [vp]),
        "ilsm_slam_frame": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, vp, C.POINTER(SlamStats)]),
        "ilsm_slam_create_async": (i32, [vp, f32, f32, f32, i32, C.POINTER(vp)]),
        "ilsm_slam_frame_async": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, vp, C.POINTER(i32), C.POINTER(SlamStats)]),
        "ilsm_pc2_layout_pcl_xyzi": (None, [C.POINTER(Pc2Layout)]),
        "ilsm_pc2_pack": (i32, [vp, vp, i32, C.POINTER(Pc2Layout), vp]),
        "ilsm_pc2_pack_dev": (i32, [vp, vp, i32, C.POINTER(Pc2Layout), vp]),
        "ilsm_slam_create_staged": (i32, [vp, f32, f32, f32, i32, C.POINTER(vp)]),
        "ilsm_slam_frame_staged": (i32, [vp, vp, i32, i32, i32, vp, vp, C.POINTER(i32), vp, vp, C.POINTER(i32), C.POINTER(SlamStats)]),
        "ilsm_slam_host_phases": (i32, [vp, vp]),
        "ilsm_slam_flush": (i32, [vp, vp, vp, C.POINTER(i32), C.POINTER(SlamStats)]),
        "ilsm_slam_frame_pc2": (i32, [vp, vp, i32, C.POINTER(Pc2Layout), i32, vp, vp, vp, vp, C.POINTER(SlamStats)]),
        "ilsm_pc2_layout_ouster": (None, [C.POINTER(Pc2Layout)]),
        "ilsm_host_register": (i32, [vp, C.c_size_t]),
        "ilsm_host_unregister": (i32, [vp]),
        "ilsm_pc2_unpack": (i32, [vp, vp, i32, C.POINTER(Pc2Layout), vp]),
        "ilsm_pc2_unpack_dev": (i32, [vp, vp, i32, C.POINTER(Pc2Layout), vp]),
        "ilsm_ground_opts_default": (None, [C.POINTER(GroundOpts)]),
        "ilsm_ground_create": (i32, [vp, C.POINTER(vp)]),
        "ilsm_ground_destroy": (None, [vp]),
        "ilsm_ground_extract": (i32, [vp, vp, i32, i32, C.POINTER(GroundOpts), vp, i32, C.POINTER(i32), vp, C.POINTER(GroundInfo)]),
        "ilsm_mapopt_create": (i32, [vp, f32, f32, C.POINTER(vp)]),
        "ilsm_mapopt_destroy": (None, [vp]),
        "ilsm_mapopt_map_size": (i32, [vp]),
        "ilsm_mapopt_map_points": (i32, [vp, vp, i32, C.POINTER(i32)]),
        "ilsm_mapopt_frame": (i32, [vp, vp, i32, i32, vp, i32, i32, vp, vp, vp, vp, C.POINTER(GroundOpts), C.POINTER(MapOptStats)]),
        "ilsm_orb_match": (i32, [vp, vp, i32, vp, i32, i32, i32, f64, vp, C.POINTER(i32), vp, C.POINTER(i32)]),
        "ilsm_align_points": (i32, [vp, vp, vp, i32, i32, vp, vp, i32, f64, C.POINTER(SolveSummary)]),
        "ilsm_associate_dev": (i32, [vp, vp, vp, vp, i32, vp, i32, i32, vp, C.POINTER(RegOpts)]),
        "ilsm_launch_count": (C.c_longlong, []),
        "ilsm_debug_live_bytes": (None, [C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
        "ilsm_eval_normal_eq": (i32, [vp, vp, vp, f64, C.POINTER(f64), vp, vp]),
        "ilsm_eval_normal_eq_dev": (i32, [vp, vp, f64, vp]),
        "ilsm_solve_dev": (i32, [vp, vp, i32, f64]),
        "ilsm_solve": (i32, [vp, vp, vp, i32, f64, C.POINTER(SolveSummary)]),
        "ilsm_icp_opts_default": (None, [C.POINTER(IcpOpts)]),
        "ilsm_icp_align_batch": (i32, [vp, vp, i32, vp, vp, i32, vp, C.POINTER(IcpOpts), vp]),
        "ilsm_icp_align_batch_dev": (i32, [vp, vp, i32, vp, vp, i32, vp, C.POINTER(IcpOpts), vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def launch_count() -> int:
    return int(load_library().ilsm_launch_count())


def live_bytes() -> tuple[int, int]:
    """(device, pinned) bytes the library's buffers hold, all handles of the process together.  Makes no CUDA call."""
    dev, pin = C.c_longlong(0), C.c_longlong(0)
    load_library().ilsm_debug_live_bytes(C.byref(dev), C.byref(pin))
    return dev.value, pin.value


def _check(rc):
    if rc != ILSM_OK:
        raise IlsmError(rc, load_library().ilsm_last_error().decode(errors="replace"))


def _cloud(a):
    """float32 C-contiguous (n, >=3) array -> (array, n, stride_bytes)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("point cloud must be (n, >=3) float32")
    return a, a.shape[0], a.strides[0] if a.shape[0] else 4 * a.shape[1]


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def default_opts(**kw) -> RegOpts:
    o = RegOpts()
    load_library().ilsm_reg_opts_default(C.byref(o))
    for k, v in kw.items():
        setattr(o, k, v)
    return o


class Context:
    """One ilsm_ctx: a CUDA stream, scratch and the device-resident LM state."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        h = C.c_void_p()
        _check(self._lib.ilsm_create(device, C.byref(h)))
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ilsm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream_ptr(self) -> int:
        return int(self._lib.ilsm_stream(self._h) or 0)

    def sync(self):
        _check(self._lib.ilsm_sync(self._h))

    def set_async(self, on: bool = True):
        """Host-pointer map builds stop blocking (see ilsm_set_async in include/ilsm.h)."""
        _check(self._lib.ilsm_set_async(self._h, 1 if on else 0))

    def new_map(self) -> "LocalMap":
        return LocalMap(self)

    # -- laserMapping.cpp:640-861 / mapOptimization.cpp:377-450 -----------------------------------
    def register(self, map_corner, map_surf, corner, surf, q, t, opts: RegOpts | None = None):
        c, nc, sc = _cloud(corner)
        s, ns, ss = _cloud(surf)
        if nc and ns and sc != ss:
            raise ValueError("corner and surf stacks must share a stride")
        stride = sc if nc else ss
        qq = np.array(q, np.float64)
        tt = np.array(t, np.float64)
        rep = RegReport()
        rc = self._lib.ilsm_register(self._h, map_corner._h, map_surf._h, _ptr(c), nc, _ptr(s), ns, stride, _ptr(qq),
                                     _ptr(tt), C.byref(opts) if opts is not None else None, C.byref(rep))
        _check(rc)
        return qq, tt, rep

    def register_dev(self, map_corner, map_surf, d_corner_ptr, nc, d_surf_ptr, ns, stride, d_pose_ptr,
                     opts: RegOpts | None = None, d_report_ptr=None):
        _check(self._lib.ilsm_register_dev(self._h, map_corner._h, map_surf._h, d_corner_ptr, nc, d_surf_ptr, ns, stride,
                                           d_pose_ptr, C.byref(opts) if opts is not None else None, d_report_ptr))

    # -- ImageHandler::cloud_handler (image_handler.h_ouster:103-140) ----------------------------
    def cloud_handler(self, cloud, H=64, W=1024):
        a, n, stride = _cloud(cloud)
        if n != H * W:
            raise ValueError("cloud must be organised H*W")
        rng = np.empty((H, W), np.uint8)
        inten = np.empty((H, W), np.uint8)
        track = np.empty((H * W, 4), np.float32)
        _check(self._lib.ilsm_project(self._h, _ptr(a), H, W, stride, _ptr(rng), _ptr(inten), _ptr(track)))
        return rng, inten, track

    # -- pcl::fromROSMsg (scanRegistration.cpp:235, image_handler.h_ouster:44,106) ------------------
    def pc2_pack(self, cloud, layout: "Pc2Layout | None" = None):
        """(n, 4) packed xyzi -> the `data` blob of a sensor_msgs/PointCloud2 (uint8, n * point_step); default layout =
        pcl::toROSMsg of pcl::PointXYZI."""
        a = np.ascontiguousarray(np.asarray(cloud, np.float32)[:, :4])
        if layout is None:
            layout = Pc2Layout()
            self._lib.ilsm_pc2_layout_pcl_xyzi(C.byref(layout))
        out = np.empty(len(a) * layout.point_step, np.uint8)
        _check(self._lib.ilsm_pc2_pack(self._h, _ptr(a), len(a), C.byref(layout), _ptr(out)))
        return out

    def pc2_unpack(self, blob, layout: "Pc2Layout"):
        """sensor_msgs/PointCloud2 `data` blob -> (n, 4) packed xyzi float32."""
        b = np.ascontiguousarray(blob, np.uint8).reshape(-1)
        n = b.size // layout.point_step if layout.point_step > 0 else 0
        out = np.zeros((n, 4), np.float32)
        _check(self._lib.ilsm_pc2_unpack(self._h, _ptr(b), n, C.byref(layout), _ptr(out)))
        return out

    def project_dev(self, d_cloud_ptr, H, W, stride, d_range_ptr, d_inten_ptr, d_track_ptr):
        _check(self._lib.ilsm_project_dev(self._h, d_cloud_ptr, H, W, stride, d_range_ptr, d_inten_ptr, d_track_ptr))

    # -- laserCloudHandler numeric body (scanRegistration.cpp:235-589) ---------------------------
    def extract_features(self, cloud, min_range=0.3):
        a, n, stride = _cloud(cloud)
        cl = np.zeros((max(n, 1), 4), np.float32)
        curv = np.zeros(max(n, 1), np.float32)
        label = np.zeros(max(n, 1), np.int32)
        src = np.zeros(max(n, 1), np.int32)
        sharp = np.zeros(max(n, 1), np.int32)
        lsharp = np.zeros(max(n, 1), np.int32)
        flat = np.zeros(max(n, 1), np.int32)
        lflat = np.zeros((max(n, 1), 4), np.float32)
        f = Features(cl.ctypes.data, curv.ctypes.data, label.ctypes.data, src.ctypes.data, sharp.ctypes.data,
                     lsharp.ctypes.data, flat.ctypes.data, lflat.ctypes.data)
        _check(self._lib.ilsm_extract_features(self._h, _ptr(a), n, stride, min_range, C.byref(f)))
        k = f.counts
        N = k.n_cloud
        return dict(cloud=cl[:N], curvature=curv[:N], label=label[:N], src_index=src[:N], sharp_idx=sharp[:k.n_sharp],
                    less_sharp_idx=lsharp[:k.n_less_sharp], flat_idx=flat[:k.n_flat], less_flat=lflat[:k.n_less_flat],
                    ring_start=np.array(k.ring_start[:]), ring_end=np.array(k.ring_end[:]))

    # -- pcl::VoxelGrid::filter -------------------------------------------------------------------
    def voxelgrid(self, cloud, leaf):
        a, n, stride = _cloud(cloud)
        if stride < 16:
            raise ValueError("voxelgrid needs xyzi points (stride >= 16)")
        out = np.empty((max(n, 1), 4), np.float32)
        m = C.c_int(0)
        _check(self._lib.ilsm_voxelgrid(self._h, _ptr(a), n, stride, leaf, _ptr(out), C.byref(m)))
        return out[:m.value].copy()

    # -- laserOdometry.cpp:417-711 ----------------------------------------------------------------
    def odometry(self, last_corner_map, last_surf_map, sharp, flat, q, t, opts: RegOpts | None = None,
                 factors_only=False):
        sh, nsh, s1 = _cloud(sharp)
        fl, nfl, s2 = _cloud(flat)
        stride = s1 if nsh else s2
        qq = np.array(q, np.float64)
        tt = np.array(t, np.float64)
        rep = RegReport()
        fac = np.zeros(nsh + nfl, FACTOR_DTYPE) if factors_only else None
        _check(self._lib.ilsm_odometry(self._h, last_corner_map._h, last_surf_map._h, _ptr(sh), nsh, _ptr(fl), nfl,
                                       stride, _ptr(qq), _ptr(tt), C.byref(opts) if opts is not None else None,
                                       C.byref(rep), _ptr(fac) if factors_only else None))
        return fac if factors_only else (qq, tt, rep)

    # -- cv::BFMatcher(NORM_HAMMING, crossCheck).match + sort + best fraction (intensity_feature_tracker.cpp:631-648) --
    def orb_match(self, cur_desc, prev_desc, cross_check=True, keep_fraction=0.3):
        a = np.ascontiguousarray(cur_desc, np.uint8).reshape(-1, 32)
        b = np.ascontiguousarray(prev_desc, np.uint8).reshape(-1, 32)
        m = np.zeros(max(len(a), 1), DMATCH_DTYPE)
        g = np.zeros(max(len(a), 1), DMATCH_DTYPE)
        nm, ng = C.c_int(0), C.c_int(0)
        _check(self._lib.ilsm_orb_match(self._h, _ptr(a), len(a), _ptr(b), len(b), 32, 1 if cross_check else 0,
                                        float(keep_fraction), _ptr(m), C.byref(nm), _ptr(g), C.byref(ng)))
        return m[:nm.value], g[:ng.value]

    # -- feature_tracker::p2p_calculateRandT (intensity_feature_tracker.cpp:880-928) ---------------
    def align_points(self, src_xyz, dst_xyz, q=(0, 0, 0, 1), t=(0, 0, 0), max_num_iterations=20, huber_a=0.1):
        s = np.ascontiguousarray(np.asarray(src_xyz, np.float32)[:, :3])
        d = np.ascontiguousarray(np.asarray(dst_xyz, np.float32)[:, :3])
        if len(s) != len(d):
            raise ValueError("src and dst must pair up")
        qq, tt = np.array(q, np.float64), np.array(t, np.float64)
        sm = SolveSummary()
        _check(self._lib.ilsm_align_points(self._h, _ptr(s), _ptr(d), len(s), 12, _ptr(qq), _ptr(tt), max_num_iterations,
                                           huber_a, C.byref(sm)))
        return qq, tt, sm

    def register_frame(self, map_corner, map_surf, cloud, q, t, min_range=0.3, line_res=0.4, plane_res=0.8, opts: RegOpts | None = None):
        """Front end -> stacks -> registration of one organised frame against prebuilt maps (ilsm_register_frame).
        Returns (q, t, report, (n_less_sharp, n_less_flat, n_corner_stack, n_surf_stack))."""
        a, n, stride = _cloud(cloud)
        qq, tt = np.array(q, np.float64), np.array(t, np.float64)
        rep = RegReport()
        sizes = np.zeros(4, np.int32)
        _check(self._lib.ilsm_register_frame(self._h, map_corner._h, map_surf._h, _ptr(a), n, stride, min_range, line_res, plane_res,
                                             _ptr(qq), _ptr(tt), C.byref(opts) if opts is not None else None, C.byref(rep), _ptr(sizes)))
        return qq, tt, rep, tuple(int(v) for v in sizes)

    def register_frame_dev(self, map_corner, map_surf, d_cloud_ptr, n, stride, d_pose_ptr, min_range=0.3, line_res=0.4, plane_res=0.8,
                           opts: RegOpts | None = None):
        _check(self._lib.ilsm_register_frame_dev(self._h, map_corner._h, map_surf._h, d_cloud_ptr, n, stride, min_range, line_res,
                                                 plane_res, d_pose_ptr, C.byref(opts) if opts is not None else None))

    def associate_dev(self, map_corner, map_surf, d_corner_ptr, nc, d_surf_ptr, ns, stride, d_pose_ptr,
                      opts: RegOpts | None = None):
        _check(self._lib.ilsm_associate_dev(self._h, map_corner._h, map_surf._h, d_corner_ptr, nc, d_surf_ptr, ns,
                                            stride, d_pose_ptr, C.byref(opts) if opts is not None else None))

    def associate(self, map_corner, map_surf, corner, surf, q, t, opts: RegOpts | None = None, want_knn=False):
        c, nc, sc = _cloud(corner)
        s, ns, ss = _cloud(surf)
        stride = sc if nc else ss
        qq = np.array(q, np.float64)
        tt = np.array(t, np.float64)
        fac = np.zeros(nc + ns, FACTOR_DTYPE)
        idx = np.zeros((nc + ns, 5), np.int32) if want_knn else None
        d2 = np.zeros((nc + ns, 5), np.float32) if want_knn else None
        _check(self._lib.ilsm_associate(self._h, map_corner._h, map_surf._h, _ptr(c), nc, _ptr(s), ns, stride, _ptr(qq),
                                        _ptr(tt), C.byref(opts) if opts is not None else None, _ptr(fac),
                                        _ptr(idx) if want_knn else None, _ptr(d2) if want_knn else None))
        return (fac, idx, d2) if want_knn else fac

    def eval_normal_eq(self, q, t, huber_a=0.1):
        qq = np.array(q, np.float64)
        tt = np.array(t, np.float64)
        cost = C.c_double()
        H = np.zeros((6, 6))
        g = np.zeros(6)
        _check(self._lib.ilsm_eval_normal_eq(self._h, _ptr(qq), _ptr(tt), huber_a, C.byref(cost), _ptr(H), _ptr(g)))
        return cost.value, H, g

    def eval_normal_eq_dev(self, d_pose_ptr, d_out32_ptr, huber_a=0.1):
        _check(self._lib.ilsm_eval_normal_eq_dev(self._h, d_pose_ptr, huber_a, d_out32_ptr))

    def solve_dev(self, d_pose_in_ptr, max_num_iterations=4, huber_a=0.1):
        _check(self._lib.ilsm_solve_dev(self._h, d_pose_in_ptr, max_num_iterations, huber_a))

    def solve(self, q, t, max_num_iterations=4, huber_a=0.1):
        qq = np.array(q, np.float64)
        tt = np.array(t, np.float64)
        s = SolveSummary()
        _check(self._lib.ilsm_solve(self._h, _ptr(qq), _ptr(tt), max_num_iterations, huber_a, C.byref(s)))
        return qq, tt, s


    # -- loopClosureThread's pcl::IterativeClosestPoint (intensity_feature_tracker.cpp:195-393) ------
    def icp_align(self, target: "LocalMap", source, q=(0.0, 0.0, 0.0, 1.0), t=(0.0, 0.0, 0.0), **opts) -> IcpResult:
        """align(output, guess) of `source` ((n, >=3) points) to `target`, plus getFitnessScore; opts: IcpOpts fields."""
        return self.icp_align_batch([target], [source], [(q, t)], **opts)[0]

    def icp_align_batch(self, targets, sources, guesses=None, **opts) -> list:
        """One launch for every (target, source) pair; guesses: None (identity) or one (q_xyzw, t) per pair.  Returns a
        list of IcpResult."""
        n = len(targets)
        if len(sources) != n or (guesses is not None and len(guesses) != n):
            raise ValueError("one source (and guess) per target")
        pts = [np.asarray(s, np.float32)[:, :3] for s in sources]
        offs = np.zeros(n + 1, np.int32)
        offs[1:] = np.cumsum([len(p) for p in pts])
        src = np.ascontiguousarray(np.concatenate(pts) if n else np.zeros((0, 3), np.float32))
        g = None
        if guesses is not None:
            g = np.ascontiguousarray([np.concatenate([np.asarray(q, np.float64), np.asarray(t, np.float64)])
                                      for q, t in guesses], np.float64).reshape(n, 7)
        hs = (C.c_void_p * max(n, 1))(*[m._h.value for m in targets])
        res = (IcpResult * max(n, 1))()
        o = IcpOpts(**opts)
        _check(self._lib.ilsm_icp_align_batch(self._h, hs, n, _ptr(src), _ptr(offs), 12, _ptr(g) if g is not None else None,
                                              C.byref(o), res))
        return [res[i] for i in range(n)]


class LocalMap:
    """ilsm_map: the voxel-hashed local map.  Mirrors pcl::KdTreeFLANN (setInputCloud / nearestKSearch) and
    ikd-Tree (Build / Nearest_Search) as used by the reference."""

    def __init__(self, ctx: Context):
        self._ctx = ctx
        self._lib = ctx._lib
        h = C.c_void_p()
        _check(self._lib.ilsm_map_create(ctx._h, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self._ctx, "_h", None):
            self._lib.ilsm_map_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self._lib.ilsm_map_size(self._h))

    # kdtree->setInputCloud(cloud) / ikdtree->Build(points)
    def set_input_cloud(self, cloud, cell: float = 0.0):
        a, n, stride = _cloud(cloud)
        _check(self._lib.ilsm_map_build(self._h, _ptr(a), n, stride, cell))
        return self

    build = set_input_cloud

    def build_dev(self, d_ptr: int, n: int, stride: int, cell: float = 0.0):
        _check(self._lib.ilsm_map_build_dev(self._h, d_ptr, n, stride, cell))
        return self

    def build_pair_dev(self, d_ptr: int, n: int, other: "LocalMap", d_ptr_other: int, n_other: int, stride: int, cell: float = 0.0):
        """This map and `other` (the corner and surf structures of a frame) built by one set of three launches."""
        _check(self._lib.ilsm_map_build_pair_dev(self._h, d_ptr, n, other._h, d_ptr_other, n_other, stride, cell))
        return self

    def join(self):
        _check(self._lib.ilsm_map_join(self._h))
        return self

    # ikdtree->Add_Points(points, downsample_on)  (mapOptimization.cpp:475; ikd_Tree.cpp:570-640)
    def add_points(self, cloud, downsample=True, downsample_size=0.4):
        a, n, stride = _cloud(cloud)
        _check(self._lib.ilsm_map_insert(self._h, _ptr(a), n, stride, 1 if downsample else 0, downsample_size))
        return self

    # ikdtree->flatten(...)
    def points(self):
        n = C.c_int(0)
        _check(self._lib.ilsm_map_points(self._h, None, 0, C.byref(n)))
        out = np.empty((max(n.value, 1), 4), np.float32)
        _check(self._lib.ilsm_map_points(self._h, _ptr(out), n.value, C.byref(n)))
        return out[:n.value]

    # kdtree->nearestKSearch(point, k, idx, d2) / ikdtree->Nearest_Search(point, k, pts, d2)
    def nearest_k_search(self, queries, k: int = 5, max_dist: float = 0.0):
        q, nq, stride = _cloud(queries)
        idx = np.empty((nq, k), np.int32)
        d2 = np.empty((nq, k), np.float32)
        _check(self._lib.ilsm_knn(self._h, _ptr(q), nq, stride, k, max_dist, _ptr(idx), _ptr(d2)))
        return idx, d2

    def knn_dev(self, d_q_ptr: int, nq: int, stride: int, k: int, max_dist: float, d_idx_ptr: int, d_d2_ptr: int):
        _check(self._lib.ilsm_knn_dev(self._h, d_q_ptr, nq, stride, k, max_dist, d_idx_ptr, d_d2_ptr))


def merge_topk(dist, ids, shifts, k):
    """Deterministic merge of gathered per-shard top-k lists (host code of the library, no GPU needed)."""
    d = np.ascontiguousarray(dist, np.float64).ravel()
    i = np.ascontiguousarray(ids, np.int32).ravel()
    s = np.ascontiguousarray(shifts, np.int32).ravel()
    od, oi, os_ = np.zeros(k), np.zeros(k, np.int32), np.zeros(k, np.int32)
    _check(load_library().ilsm_sc_merge_topk(_ptr(d), _ptr(i), _ptr(s), len(d), k, _ptr(od), _ptr(oi), _ptr(os_)))
    return od, oi, os_


class ScanContextDb:
    """ilsm_sc: mirrors SCManager (makeScancontext / makeAndSaveScancontextAndKeys / detectLoopClosureID candidate
    scoring).  One instance holds one shard of the keyframe database."""
    NUM_EXCLUDE_RECENT = 50  # Scancontext.h:86
    SC_DIST_THRES = 0.13     # Scancontext.h:91

    def __init__(self, ctx: Context):
        self._ctx = ctx
        self._lib = ctx._lib
        h = C.c_void_p()
        _check(self._lib.ilsm_sc_create(ctx._h, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self._ctx, "_h", None):
            self._lib.ilsm_sc_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self._lib.ilsm_sc_size(self._h))

    def make_scancontext(self, points):
        a, n, stride = _cloud(points)
        d = np.empty((20, 60), np.float32)
        _check(self._lib.ilsm_sc_make(self._h, _ptr(a), n, stride, _ptr(d)))
        return d

    def add(self, descs):
        d = np.ascontiguousarray(descs, np.float32).reshape(-1, 1200)
        _check(self._lib.ilsm_sc_add(self._h, _ptr(d), len(d)))

    def add_dev(self, d_ptr, count):
        _check(self._lib.ilsm_sc_add_dev(self._h, d_ptr, count))

    def query_topk(self, desc, k=10, n_search=-1, id_offset=0):
        q = np.ascontiguousarray(desc, np.float32).reshape(1200)
        dist, ids, sh = np.zeros(k), np.zeros(k, np.int32), np.zeros(k, np.int32)
        _check(self._lib.ilsm_sc_query_topk(self._h, _ptr(q), n_search, id_offset, k, _ptr(dist), _ptr(ids), _ptr(sh)))
        return dist, ids, sh

    def query_topk_dev(self, d_desc_ptr, k, n_search, id_offset, d_dist_ptr, d_id_ptr, d_shift_ptr):
        _check(self._lib.ilsm_sc_query_topk_dev(self._h, d_desc_ptr, n_search, id_offset, k, d_dist_ptr, d_id_ptr,
                                                d_shift_ptr))


    NUM_CANDIDATES_FROM_TREE = 10  # Scancontext.h:87
    TREE_MAKING_PERIOD = 50        # Scancontext.h:95

    def query_candidates(self, desc, num_candidates=10, n_search=-1):
        """The reference's candidate search: ring-key nearest neighbours, then distanceBtnScanContext for those only.
        Returns (ids, float key distances, distances, shifts) in candidate order."""
        q = np.ascontiguousarray(desc, np.float32).reshape(1200)
        k = num_candidates
        ids, kd2 = np.zeros(k, np.int32), np.zeros(k, np.float32)
        dist, sh = np.zeros(k), np.zeros(k, np.int32)
        _check(self._lib.ilsm_sc_query_candidates(self._h, _ptr(q), n_search, k, _ptr(ids), _ptr(kd2), _ptr(dist), _ptr(sh)))
        return ids, kd2, dist, sh

    def detect_loop_closure_id(self, desc, n_search=-1, exhaustive=False):
        """SCManager::detectLoopClosureID (Scancontext.cpp:283-344) for a query descriptor against entries [0, n_search):
        (loop id or -1, min distance, aligning shift, nearest id).  exhaustive=True scores every entry instead of the
        10 ring-key candidates (superset; may differ from the reference)."""
        best, arg, align = 10000000.0, 0, 0
        if exhaustive:
            d, i, s = self.query_topk(desc, 1, n_search)
            if i[0] >= 0:
                best, arg, align = float(d[0]), int(i[0]), int(s[0])
        else:
            ids, _, dist, sh = self.query_candidates(desc, self.NUM_CANDIDATES_FROM_TREE, n_search)
            for ci, cd, cs in zip(ids, dist, sh):
                if ci >= 0 and cd < best:
                    best, arg, align = float(cd), int(ci), int(cs)
        return (arg if best < self.SC_DIST_THRES else -1), best, align, arg

    def query_topk_batch(self, descs, k=10, n_search=-1, id_offset=0):
        q = np.ascontiguousarray(descs, np.float32).reshape(-1, 1200)
        B = len(q)
        dist, ids, sh = np.zeros((B, k)), np.zeros((B, k), np.int32), np.zeros((B, k), np.int32)
        _check(self._lib.ilsm_sc_query_topk_batch(self._h, _ptr(q), B, n_search, id_offset, k, _ptr(dist), _ptr(ids), _ptr(sh)))
        return dist, ids, sh

    def prefilter_debug(self, descs, n_search=-1):
        """The tensor-core prefilter alone: (approximate distances (B, n), aligned shifts (B, n)); -1 = flagged pair."""
        q = np.ascontiguousarray(descs, np.float32).reshape(-1, 1200)
        n = len(self) if n_search < 0 else n_search
        D = np.zeros((len(q), n), np.float32)
        S = np.zeros((len(q), n), np.uint8)
        _check(self._lib.ilsm_sc_prefilter_debug(self._h, _ptr(q), len(q), n, _ptr(D), _ptr(S)))
        return D, S

    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _check(load_library().ilsm_sc_nccl_unique_id(buf))
        return buf.raw

    @staticmethod
    def nccl_version() -> int:
        v = C.c_int(0)
        _check(load_library().ilsm_sc_nccl_version(C.byref(v)))
        return v.value

    def init_nccl_rank(self, unique_id: bytes, n_ranks: int, rank: int):
        """Collective: every rank of the sharded database calls it with rank 0's unique id."""
        assert len(unique_id) == 128
        _check(self._lib.ilsm_sc_init_nccl_rank(self._h, C.c_char_p(unique_id), n_ranks, rank))

    def query_topk_sharded(self, descs, k=10, n_search=-1, id_offset=0):
        """Collective: local scoring -> one NCCL all-gather for the batch -> identical merge; every rank gets the global top-k."""
        q = np.ascontiguousarray(descs, np.float32).reshape(-1, 1200)
        B = len(q)
        dist, ids, sh = np.zeros((B, k)), np.zeros((B, k), np.int32), np.zeros((B, k), np.int32)
        _check(self._lib.ilsm_sc_query_topk_sharded(self._h, _ptr(q), B, n_search, id_offset, k, _ptr(dist), _ptr(ids), _ptr(sh)))
        return dist, ids, sh

    def query_topk_sharded_dev(self, d_desc_ptr, n_queries, k, n_search, id_offset, d_packed_out_ptr):
        _check(self._lib.ilsm_sc_query_topk_sharded_dev(self._h, d_desc_ptr, n_queries, n_search, id_offset, k, d_packed_out_ptr))

    def query_packed_dev(self, d_desc_ptr, k, n_search, id_offset, d_packed_ptr):
        """Local top-k written in the packed all-gather layout (k f64 dist | k i32 id | k i32 shift)."""
        self.query_topk_dev(d_desc_ptr, k, n_search, id_offset, d_packed_ptr, d_packed_ptr + 8 * k, d_packed_ptr + 12 * k)

    def merge_packed_dev(self, d_gathered_ptr, shards, k, d_out_packed_ptr):
        _check(self._lib.ilsm_sc_merge_topk_dev(self._h, d_gathered_ptr, shards, k, d_out_packed_ptr))


class CubeMap:
    """ilsm_cubemap: the device-resident rolling 21x21x11 cube map of laserMapping.cpp and one process() iteration per
    frame() call (transformAssociateToMap -> roll -> gather -> stack VoxelGrid -> guarded registration ->
    transformUpdate -> insertion -> per-cube VoxelGrid)."""

    def __init__(self, ctx: Context, line_res: float = 0.4, plane_res: float = 0.8, cube_capacity: int = 0):
        self._ctx = ctx
        self._lib = ctx._lib
        h = C.c_void_p()
        _check(self._lib.ilsm_cubemap_create(ctx._h, line_res, plane_res, cube_capacity, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self._ctx, "_h", None):
            self._lib.ilsm_cubemap_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _x4(a):
        a = np.asarray(a, np.float32)
        if a.ndim == 2 and a.shape[1] == 4 and a.flags.c_contiguous:
            return a
        out = np.zeros((len(a), 4), np.float32)
        out[:, :min(4, a.shape[1])] = a[:, :4]
        return out

    def insert_world(self, corner, surf, centre):
        c, s = self._x4(corner), self._x4(surf)
        ctr = np.ascontiguousarray(centre, np.float64)
        _check(self._lib.ilsm_cubemap_insert_world(self._h, _ptr(c), len(c), _ptr(s), len(s), 16, _ptr(ctr)))

    def frame(self, corner_last, surf_last, q_wodom, t_wodom, opts: RegOpts | None = None):
        c, s = self._x4(corner_last), self._x4(surf_last)
        qo, to = np.array(q_wodom, np.float64), np.array(t_wodom, np.float64)
        qw, tw = np.zeros(4), np.zeros(3)
        rep, st = RegReport(), CubeMapStats()
        _check(self._lib.ilsm_cubemap_frame(self._h, _ptr(c), len(c), _ptr(s), len(s), 16, _ptr(qo), _ptr(to), _ptr(qw),
                                            _ptr(tw), C.byref(opts) if opts is not None else None, C.byref(rep), C.byref(st)))
        return qw, tw, rep, st

    @staticmethod
    def _cube_of(lib, h, which, index):
        n = C.c_int(0)
        _check(lib.ilsm_cubemap_cube(h, which, index, None, 0, C.byref(n)))
        out = np.empty((max(n.value, 1), 4), np.float32)
        _check(lib.ilsm_cubemap_cube(h, which, index, _ptr(out), n.value, C.byref(n)))
        return out[:n.value]

    def cube(self, which: int, index: int):
        return self._cube_of(self._lib, self._h, which, index)


class Slam:
    """ilsm_slam: scanRegistration -> laserOdometry -> laserMapping for one frame per call, inter-node clouds resident on
    the GPU.  frame() returns (q_odom, t_odom, q_map, t_map, stats)."""

    def __init__(self, ctx: Context, line_res: float = 0.4, plane_res: float = 0.8, min_range: float = 0.3,
                 cube_capacity: int = 0, mapping: str = "laserMapping", voxel_leaf: float = 0.8, downsample_size: float = 0.4,
                 pipelined: bool = False, staged: bool = False):
        self._ctx = ctx
        self._lib = ctx._lib
        h = C.c_void_p()
        self.pipelined = bool(pipelined)
        self.staged = bool(staged)
        self._held = []
        if mapping == "laserMapping" and staged:
            _check(self._lib.ilsm_slam_create_staged(ctx._h, line_res, plane_res, min_range, cube_capacity, C.byref(h)))
        elif mapping == "laserMapping" and pipelined:
            _check(self._lib.ilsm_slam_create_async(ctx._h, line_res, plane_res, min_range, cube_capacity, C.byref(h)))
        elif mapping == "laserMapping":
            _check(self._lib.ilsm_slam_create(ctx._h, line_res, plane_res, min_range, cube_capacity, C.byref(h)))
        elif mapping == "mapOptimization":
            _check(self._lib.ilsm_slam_create_mapopt(ctx._h, voxel_leaf, downsample_size, min_range, C.byref(h)))
        else:
            raise ValueError("mapping must be 'laserMapping' or 'mapOptimization'")
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self._ctx, "_h", None):
            self._lib.ilsm_slam_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def cubemap(self) -> "CubeMap":
        """Non-owning view of the pipeline's cube map."""
        cm = CubeMap.__new__(CubeMap)
        cm._ctx, cm._lib = self._ctx, self._lib
        cm._h = None
        cm._view = C.c_void_p(self._lib.ilsm_slam_cubemap(self._h))
        cm.cube = lambda which, index, _cm=cm: CubeMap._cube_of(_cm._lib, _cm._view, which, index)
        return cm

    def frame(self, cloud, use_aloam: bool = True):
        a, n, stride = _cloud(cloud)
        qo, to, qm, tm = np.zeros(4), np.zeros(3), np.zeros(4), np.zeros(3)
        st = SlamStats()
        _check(self._lib.ilsm_slam_frame(self._h, _ptr(a), n, stride, 1 if use_aloam else 0, _ptr(qo), _ptr(to), _ptr(qm),
                                         _ptr(tm), C.byref(st)))
        return qo, to, qm, tm, st

    def frame_async(self, cloud, use_aloam: bool = True):
        """Pipelined mode (ilsm_slam_create_async): returns (q_odom, t_odom) of THIS frame and (q_map, t_map) of the PREVIOUS
        frame (None, None on the first call) while this frame's mapping keeps running on the GPU."""
        a, n, stride = _cloud(cloud)
        qo, to, qm, tm = np.zeros(4), np.zeros(3), np.zeros(4), np.zeros(3)
        st, have = SlamStats(), C.c_int32(0)
        _check(self._lib.ilsm_slam_frame_async(self._h, _ptr(a), n, stride, 1 if use_aloam else 0, _ptr(qo), _ptr(to), _ptr(qm),
                                               _ptr(tm), C.byref(have), C.byref(st)))
        return (qo, to, qm, tm, st) if have.value else (qo, to, None, None, st)

    def frame_staged(self, cloud=None, use_aloam: bool = True):
        """Staged mode (ilsm_slam_create_staged): pushes `cloud` (None: drain step) and returns
        (odom_frame, q_odom, t_odom, map_frame, q_map, t_map, stats); a frame index of -1 means "none in this call".  The
        odometry pose is that of the frame pushed one call earlier, the mapped pose that of the frame two calls earlier."""
        if cloud is None:
            a, n, stride = None, -1, 16
        else:
            a, n, stride = _cloud(cloud)
        qo, to, qm, tm = np.zeros(4), np.zeros(3), np.zeros(4), np.zeros(3)
        fo, fm = C.c_int32(-1), C.c_int32(-1)
        st = SlamStats()
        _check(self._lib.ilsm_slam_frame_staged(self._h, _ptr(a) if a is not None else None, n, stride, 1 if use_aloam else 0,
                                                _ptr(qo), _ptr(to), C.byref(fo), _ptr(qm), _ptr(tm), C.byref(fm), C.byref(st)))
        self._held = [self._held[-1] if self._held else None, a]  # the front-end stage reads `a` until the next call returns
        return fo.value, qo, to, fm.value, qm, tm, st

    def host_phases(self):
        """Host seconds per phase since the last call (see ilsm_slam_host_phases)."""
        out = np.zeros(8)
        _check(self._lib.ilsm_slam_host_phases(self._h, _ptr(out)))
        return out

    def flush(self):
        """Mapped pose of the last frame handed to frame_async (None, None when nothing is in flight)."""
        qm, tm = np.zeros(4), np.zeros(3)
        st, have = SlamStats(), C.c_int32(0)
        _check(self._lib.ilsm_slam_flush(self._h, _ptr(qm), _ptr(tm), C.byref(have), C.byref(st)))
        return (qm, tm, st) if have.value else (None, None, st)

    def frame_pc2(self, blob, layout: "Pc2Layout", use_aloam: bool = True):
        """One frame handed over as the sensor_msgs/PointCloud2 `data` blob (uint8, n_points * point_step bytes)."""
        b = np.ascontiguousarray(blob, np.uint8).reshape(-1)
        n = b.size // layout.point_step
        qo, to, qm, tm = np.zeros(4), np.zeros(3), np.zeros(4), np.zeros(3)
        st = SlamStats()
        _check(self._lib.ilsm_slam_frame_pc2(self._h, _ptr(b), n, C.byref(layout), 1 if use_aloam else 0, _ptr(qo), _ptr(to),
                                             _ptr(qm), _ptr(tm), C.byref(st)))
        return qo, to, qm, tm, st


class GroundExtractor:
    """ilsm_ground: ImageHandler::groundPlaneExtraction (image_handler.h_ouster:41-100)."""

    def __init__(self, ctx: Context):
        self._ctx = ctx
        self._lib = ctx._lib
        h = C.c_void_p()
        _check(self._lib.ilsm_ground_create(ctx._h, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self._ctx, "_h", None):
            self._lib.ilsm_ground_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def extract(self, cloud, **kw):
        a, n, stride = _cloud(cloud)
        o = GroundOpts()
        self._lib.ilsm_ground_opts_default(C.byref(o))
        for k, v in kw.items():
            setattr(o, k, v)
        out = np.zeros((max(n, 1), 4), np.float32)
        n_out = C.c_int(0)
        co = np.zeros(4, np.float32)
        info = GroundInfo()
        _check(self._lib.ilsm_ground_extract(self._h, _ptr(a), n, stride, C.byref(o), _ptr(out), n, C.byref(n_out), _ptr(co),
                                             C.byref(info)))
        return out[:n_out.value, :3].copy(), co, info


class MapOptimization:
    """ilsm_mapopt: mapOptimization::mapOptimizationCallback (the mapping node spot.launch starts), one frame per call."""

    def __init__(self, ctx: Context, voxel_leaf: float = 0.8, downsample_size: float = 0.4):
        self._ctx = ctx
        self._lib = ctx._lib
        h = C.c_void_p()
        _check(self._lib.ilsm_mapopt_create(ctx._h, voxel_leaf, downsample_size, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self._ctx, "_h", None):
            self._lib.ilsm_mapopt_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self._lib.ilsm_mapopt_map_size(self._h))

    def map_points(self):
        n = C.c_int(0)
        _check(self._lib.ilsm_mapopt_map_points(self._h, None, 0, C.byref(n)))
        out = np.empty((max(n.value, 1), 4), np.float32)
        _check(self._lib.ilsm_mapopt_map_points(self._h, _ptr(out), n.value, C.byref(n)))
        return out[:n.value, :3].copy()

    def frame(self, cloud, plane_cloud, q_wodom, t_wodom, **ground_kw):
        a, n, stride = _cloud(cloud)
        p, npl, pstride = _cloud(plane_cloud)
        qo, to = np.array(q_wodom, np.float64), np.array(t_wodom, np.float64)
        qw, tw = np.zeros(4), np.zeros(3)
        go = GroundOpts()
        self._lib.ilsm_ground_opts_default(C.byref(go))
        for k, v in ground_kw.items():
            setattr(go, k, v)
        st = MapOptStats()
        _check(self._lib.ilsm_mapopt_frame(self._h, _ptr(a), n, stride, _ptr(p), npl, pstride, _ptr(qo), _ptr(to), _ptr(qw), _ptr(tw),
                                           C.byref(go), C.byref(st)))
        return qw, tw, st
