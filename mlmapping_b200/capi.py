"""ctypes binding of the C ABI (include/mlmap_b200.h) and a thin Python mirror of the reference's
``class mlmap`` (reference include/mlmap.h:105-139): same method names, argument meaning and
sentinel returns, batched over numpy arrays.  Nothing here computes map values; every call goes to
the CUDA library and raises ``MlmError`` if that library or a B200 is missing."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
_LIB_PATH = Path(os.environ["MLM_LIB_PATH"]) if os.environ.get("MLM_LIB_PATH") else _PKG / "lib" / "libmlmap_b200.so"  # override: A/B builds

MLM_OK = 0
ERR_NAMES = {
    1: "MLM_ERR_INVALID_ARG",
    2: "MLM_ERR_INVALID_CONFIG",
    3: "MLM_ERR_CUDA",
    4: "MLM_ERR_POOL_EXHAUSTED",
    5: "MLM_ERR_CAPACITY",
    6: "MLM_ERR_UNSUPPORTED",
    7: "MLM_ERR_NO_DEVICE",
}
FREE, OCCUPIED, UNKNOWN = 1, 0, -1  # reference include/mlmap.h:109-114


class MlmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


class MlmConfig(C.Structure):
    """mirror of ``mlm_config`` (field order and padding must match include/mlmap_b200.h)"""

    _fields_ = [
        ("am_d_rho", C.c_double),
        ("am_d_phi_deg", C.c_double),
        ("am_d_z", C.c_double),
        ("am_n_rho", C.c_int32),
        ("am_n_z_below", C.c_int32),
        ("am_n_z_over", C.c_int32),
        ("use_raycasting", C.c_int32),
        ("_pad0", C.c_int32),
        ("depth_noise_coe", C.c_double),
        ("subbox_d_xyz", C.c_double),
        ("subbox_n", C.c_int32),
        ("log_odds_min", C.c_float),
        ("log_odds_max", C.c_float),
        ("log_odds_hit", C.c_float),
        ("log_odds_miss", C.c_float),
        ("log_odds_occupied_sh", C.c_float),
        ("use_exploration_frontiers", C.c_int32),
        ("_pad1", C.c_int32),
        ("cam_cx", C.c_float),
        ("cam_cy", C.c_float),
        ("cam_fx", C.c_float),
        ("cam_fy", C.c_float),
        ("T_bs", C.c_double * 7),
        ("inflate_n", C.c_int32),
        ("inflate_global_n", C.c_int32),
        ("apply_inflate", C.c_int32),
        ("_pad2", C.c_int32),
        ("inflate_height", C.c_double),
        ("sample_cnt", C.c_int32),
        ("max_points", C.c_int32),
        ("pool_submaps", C.c_int32),
        ("_pad3", C.c_int32),
    ]

    def copy(self) -> "MlmConfig":
        c = MlmConfig()
        C.memmove(C.byref(c), C.byref(self), C.sizeof(MlmConfig))
        return c


class FrameStats(C.Structure):
    _fields_ = [
        ("n_points", C.c_int32),
        ("n_inside", C.c_int32),
        ("n_cast", C.c_int32),
        ("n_hit_cells", C.c_int32),
        ("n_miss_cells", C.c_int32),
        ("n_touched_voxels", C.c_int32),
        ("n_new_submaps", C.c_int32),
        ("hit_bucket_count", C.c_int32),
        ("ordering_slow_path", C.c_int32),
        ("status", C.c_int32),
        ("ram_expand_cnt", C.c_int64),
        ("obs_cnt", C.c_int64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


SHARD_BLOB_BYTES = 128  # MLM_SHARD_BLOB_BYTES


class ShardExchange(C.Structure):
    """mirror of mlm_shard_exchange (include/mlmap_b200.h)"""
    _fields_ = [("world", C.c_int32), ("n_hit_total", C.c_int32), ("n_hit_local", C.c_int32), ("records_received", C.c_int32),
                ("records_from_self", C.c_int32), ("rehash_path", C.c_int32), ("wait_ns", C.c_int64), ("arena_bytes", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


RAY_INFLATED, RAY_INVALID = 1, -2  # MLM_RAY_INFLATED, MLM_RAY_INVALID


class RayHit(C.Structure):
    """mirror of mlm_ray_hit (include/mlmap_b200.h): one record of mlm_cast_rays"""
    _fields_ = [("status", C.c_int32), ("cell", C.c_int32 * 3), ("n_free", C.c_int32), ("n_unknown", C.c_int32),
                ("t", C.c_double)]


# the same record as a numpy dtype: MLMap.cast_rays returns arrays of it
RAY_HIT_DTYPE = np.dtype([("status", "<i4"), ("cell", "<i4", (3,)), ("n_free", "<i4"), ("n_unknown", "<i4"), ("t", "<f8")])

ESDF_INFLATED = 1  # MLM_ESDF_INFLATED
FRONTIER_CONN6 = 1  # MLM_FRONTIER_CONN6
# mlm_frontier_cluster (include/mlmap_b200.h): one record of mlm_frontier_clusters, 64 bytes
FRONTIER_CLUSTER_DTYPE = np.dtype([("n_cells", "<i4"), ("key", "<i4", (3,)), ("lo", "<i4", (3,)), ("hi", "<i4", (3,)),
                                   ("centroid", "<f8", (3,))])

VIEW_FRONTIER, VIEW_INFLATED, VIEW_INVALID = 1, 2, -2  # MLM_VIEW_FRONTIER, MLM_VIEW_INFLATED, MLM_VIEW_INVALID
REACH_INFLATED, REACH_UNKNOWN = 1, 2  # MLM_REACH_INFLATED, MLM_REACH_UNKNOWN


class ViewSensor(C.Structure):
    """mirror of mlm_view_sensor (include/mlmap_b200.h): a pinhole depth sensor, the project_depth model"""
    _fields_ = [("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double), ("cols", C.c_int32),
                ("rows", C.c_int32), ("min_depth", C.c_double), ("max_depth", C.c_double)]


# mlm_view_gain_record (include/mlmap_b200.h): one record of mlm_view_gain, 16 bytes
VIEW_GAIN_DTYPE = np.dtype([("status", "<i4"), ("n_target", "<i4"), ("n_visible", "<i4"), ("_pad", "<i4")])


# every symbol include/mlmap_b200.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "mlm_default_config", "mlm_create", "mlm_destroy", "mlm_last_error", "mlm_abi_version",
    "mlm_integrate_depth_u16", "mlm_integrate_depth_u16_device", "mlm_integrate_points_f64",
    "mlm_integrate_points_f64_device", "mlm_set_free_in_bound", "mlm_inflate_map",
    "mlm_get_occupancy", "mlm_get_occupancy_inflate", "mlm_get_inflate_occupancy", "mlm_get_odd",
    "mlm_get_odd_grad", "mlm_get_occupancy_device", "mlm_get_odd_device", "mlm_get_odd_grad_device",
    "mlm_sync", "mlm_timer_start", "mlm_timer_stop_ms", "mlm_device_alloc", "mlm_device_free",
    "mlm_copy_to_device", "mlm_copy_to_host", "mlm_flush_l2", "mlm_kernel_launch_count",
    "mlm_last_frame_hits", "mlm_last_frame_misses", "mlm_export_map_count", "mlm_export_map",
    "mlm_debug_log10f", "mlm_set_profiling", "mlm_last_frame_kernel_ms", "mlm_sizeof_config",
    "mlm_sizeof_frame_stats", "mlm_debug_phase_cycles", "mlm_host_alloc", "mlm_host_free", "mlm_srand", "mlm_debug_rand", "mlm_export_frontier", 
    "mlm_awareness_input_pc_pose_f64", "mlm_awareness_input_depth_u16", "mlm_local_input_pc_pose_direct", "mlm_set_sm_budget",
    "mlm_frame_submit_depth_u16_device", "mlm_frame_submit_points_f64_device", "mlm_frame_finish", "mlm_get_odd_at", "mlm_get_odd_at_device",
    "mlm_shard_open", "mlm_shard_connect", "mlm_shard_submit_points_f64", "mlm_shard_submit_points_f64_device", "mlm_shard_submit_points_slice_f64", "mlm_shard_finish",
    "mlm_shard_integrate_points_f64", "mlm_shard_last_exchange", "mlm_shard_last_kernel_ms", "mlm_shard_close", "mlm_dirty_count", "mlm_dirty_export", "mlm_dirty_import",
    "mlm_replica_open", "mlm_replica_connect", "mlm_replica_publish", "mlm_replica_apply", "mlm_replica_close",
    "mlm_export_cloud", "mlm_export_cloud_device", "mlm_export_odds_slice",
    "mlm_checkpoint_size", "mlm_checkpoint_save", "mlm_checkpoint_restore", "mlm_compensate_pose",
    "mlm_export_cloud", "mlm_export_cloud_device", "mlm_export_odds_slice",
    "mlm_cast_rays", "mlm_cast_rays_device", "mlm_sizeof_ray_hit",
    "mlm_esdf_build", "mlm_esdf_distance", "mlm_esdf_distance_device", "mlm_esdf_export", "mlm_esdf_export_device",
    "mlm_frontier_clusters", "mlm_frontier_clusters_device", "mlm_sizeof_frontier_cluster",
    "mlm_view_gain", "mlm_view_gain_device", "mlm_sizeof_view_gain",
    "mlm_reach_build", "mlm_reach_cost", "mlm_reach_cost_device", "mlm_reach_paths", "mlm_reach_paths_device",
    "mlm_reach_export", "mlm_reach_export_device", "mlm_reach_matrix", "mlm_reach_matrix_device",
]
FRAME_KERNELS = ["k_project", "k_column", "k_fuse"]

_lib = None


def library_path() -> Path:
    return _LIB_PATH


def build_library(verbose: bool = False) -> Path:
    """compile csrc/ for sm_100a with nvcc (works without a GPU)"""
    script = _PKG / "csrc" / "build.sh"
    res = subprocess.run(["sh", str(script)], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-8000:])
    if res.returncode != 0:
        raise RuntimeError("nvcc build of libmlmap_b200.so failed")
    return _LIB_PATH


def load_library() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise MlmError(7, f"{_LIB_PATH} is missing: build it with mlmapping_b200.build_library() "
                          "(python -c 'import __graft_entry__ as g; g.build()'); there is no CPU fallback")
    lib = C.CDLL(str(_LIB_PATH))
    vp, dp, ip, fp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_float)
    sz = C.c_size_t
    sig = {
        "mlm_default_config": ([C.POINTER(MlmConfig)], C.c_int),
        "mlm_create": ([C.POINTER(MlmConfig), C.c_int, C.POINTER(vp)], C.c_int),
        "mlm_destroy": ([vp], C.c_int),
        "mlm_last_error": ([], C.c_char_p),
        "mlm_abi_version": ([], C.c_int),
        "mlm_sizeof_config": ([], C.c_size_t),
        "mlm_sizeof_frame_stats": ([], C.c_size_t),
        "mlm_integrate_depth_u16": ([vp, vp, C.c_int, C.c_int, sz, dp, C.POINTER(FrameStats)], C.c_int),
        "mlm_integrate_depth_u16_device": ([vp, vp, C.c_int, C.c_int, dp, C.POINTER(FrameStats)], C.c_int),
        "mlm_integrate_points_f64": ([vp, vp, C.c_int, dp, C.POINTER(FrameStats)], C.c_int),
        "mlm_integrate_points_f64_device": ([vp, vp, C.c_int, dp, C.POINTER(FrameStats)], C.c_int),
        "mlm_set_free_in_bound": ([vp, dp, dp], C.c_int),
        "mlm_inflate_map": ([vp, dp], C.c_int),
        "mlm_get_occupancy": ([vp, vp, sz, vp], C.c_int),
        "mlm_get_occupancy_inflate": ([vp, vp, sz, C.c_float, vp], C.c_int),
        "mlm_get_inflate_occupancy": ([vp, vp, sz, vp], C.c_int),
        "mlm_get_odd": ([vp, vp, sz, vp], C.c_int),
        "mlm_get_odd_grad": ([vp, vp, sz, sz, vp], C.c_int),
        "mlm_get_occupancy_device": ([vp, vp, sz, vp], C.c_int),
        "mlm_get_odd_device": ([vp, vp, sz, vp], C.c_int),
        "mlm_get_odd_grad_device": ([vp, vp, sz, sz, vp], C.c_int),
        "mlm_cast_rays": ([vp, vp, vp, sz, C.c_int, vp], C.c_int),
        "mlm_cast_rays_device": ([vp, vp, vp, sz, C.c_int, vp], C.c_int),
        "mlm_sizeof_ray_hit": ([], C.c_size_t),
        "mlm_esdf_build": ([vp, dp, dp, C.c_double, C.c_int], C.c_int),
        "mlm_esdf_distance": ([vp, vp, sz, vp, vp], C.c_int),
        "mlm_esdf_distance_device": ([vp, vp, sz, vp, vp], C.c_int),
        "mlm_esdf_export": ([vp, vp, sz, ip, ip], C.c_int),
        "mlm_esdf_export_device": ([vp, vp, sz, ip, ip], C.c_int),
        "mlm_frontier_clusters": ([vp, dp, dp, C.c_int32, C.c_int, vp, sz, C.POINTER(sz), vp, vp, sz, C.POINTER(sz)], C.c_int),
        "mlm_frontier_clusters_device": ([vp, dp, dp, C.c_int32, C.c_int, vp, sz, C.POINTER(sz), vp, vp, sz, C.POINTER(sz)],
                                         C.c_int),
        "mlm_sizeof_frontier_cluster": ([], C.c_size_t),
        "mlm_view_gain": ([vp, vp, sz, C.POINTER(ViewSensor), vp, C.c_int, vp], C.c_int),
        "mlm_view_gain_device": ([vp, vp, sz, C.POINTER(ViewSensor), vp, C.c_int, vp], C.c_int),
        "mlm_sizeof_view_gain": ([], C.c_size_t),
        "mlm_reach_build": ([vp, dp, dp, vp, sz, C.c_double, C.c_int, ip], C.c_int),
        "mlm_reach_cost": ([vp, vp, sz, vp], C.c_int),
        "mlm_reach_cost_device": ([vp, vp, sz, vp], C.c_int),
        "mlm_reach_paths": ([vp, vp, sz, sz, vp, vp], C.c_int),
        "mlm_reach_paths_device": ([vp, vp, sz, sz, vp, vp], C.c_int),
        "mlm_reach_export": ([vp, vp, sz, ip, ip], C.c_int),
        "mlm_reach_export_device": ([vp, vp, sz, ip, ip], C.c_int),
        "mlm_reach_matrix": ([vp, dp, dp, vp, sz, vp, sz, C.c_double, C.c_int, vp], C.c_int),
        "mlm_reach_matrix_device": ([vp, dp, dp, vp, sz, vp, sz, C.c_double, C.c_int, vp], C.c_int),
        "mlm_sync": ([vp], C.c_int),
        "mlm_timer_start": ([vp], C.c_int),
        "mlm_timer_stop_ms": ([vp, fp], C.c_int),
        "mlm_device_alloc": ([vp, sz, C.POINTER(vp)], C.c_int),
        "mlm_device_free": ([vp, vp], C.c_int),
        "mlm_host_alloc": ([vp, sz, C.POINTER(vp)], C.c_int),
        "mlm_host_free": ([vp, vp], C.c_int),
        "mlm_copy_to_device": ([vp, vp, vp, sz], C.c_int),
        "mlm_copy_to_host": ([vp, vp, vp, sz], C.c_int),
        "mlm_flush_l2": ([vp], C.c_int),
        "mlm_kernel_launch_count": ([vp, C.POINTER(C.c_int64)], C.c_int),
        "mlm_last_frame_hits": ([vp, vp, vp, sz, C.POINTER(sz)], C.c_int),
        "mlm_last_frame_misses": ([vp, vp, sz, C.POINTER(sz)], C.c_int),
        "mlm_export_map_count": ([vp, C.POINTER(sz)], C.c_int),
        "mlm_export_map": ([vp, sz, vp, vp, vp, vp, vp, C.POINTER(sz)], C.c_int),
        "mlm_export_frontier": ([vp, sz, vp, vp, C.POINTER(sz)], C.c_int),
        "mlm_export_cloud": ([vp, C.c_int, vp, sz, C.POINTER(sz)], C.c_int),
        "mlm_export_cloud_device": ([vp, C.c_int, vp, sz, C.POINTER(sz)], C.c_int),
        "mlm_export_odds_slice": ([vp, C.c_double, vp, sz, C.POINTER(sz)], C.c_int),
        "mlm_checkpoint_size": ([vp, C.POINTER(sz)], C.c_int),
        "mlm_checkpoint_save": ([vp, vp, sz, C.POINTER(sz)], C.c_int),
        "mlm_checkpoint_restore": ([vp, vp, sz], C.c_int),
        "mlm_compensate_pose": ([dp, dp, dp, dp, C.c_double, C.c_double, C.c_double, dp], C.c_int),
        "mlm_awareness_input_pc_pose_f64": ([vp, vp, C.c_int, dp, C.POINTER(FrameStats)], C.c_int),
        "mlm_awareness_input_depth_u16": ([vp, vp, C.c_int, C.c_int, sz, dp, C.POINTER(FrameStats)], C.c_int),
        "mlm_local_input_pc_pose_direct": ([vp, C.POINTER(FrameStats)], C.c_int),
        "mlm_set_sm_budget": ([vp, C.c_int], C.c_int),
        "mlm_frame_submit_depth_u16_device": ([vp, vp, C.c_int, C.c_int, dp], C.c_int),
        "mlm_frame_submit_points_f64_device": ([vp, vp, C.c_int, dp], C.c_int),
        "mlm_frame_finish": ([vp, C.POINTER(FrameStats)], C.c_int),
        "mlm_get_odd_at": ([vp, vp, vp, sz, vp], C.c_int),
        "mlm_get_odd_at_device": ([vp, vp, vp, sz, vp], C.c_int),
        "mlm_shard_open": ([vp, C.c_int, C.c_int, vp], C.c_int),
        "mlm_shard_connect": ([vp, vp], C.c_int),
        "mlm_shard_submit_points_f64": ([vp, vp, C.c_int, dp], C.c_int),
        "mlm_shard_submit_points_f64_device": ([vp, vp, C.c_int, dp], C.c_int),
        "mlm_shard_submit_points_slice_f64": ([vp, vp, C.c_int, C.c_int, C.c_int, dp], C.c_int),
        "mlm_shard_finish": ([vp, C.POINTER(FrameStats)], C.c_int),
        "mlm_shard_integrate_points_f64": ([vp, vp, C.c_int, dp, C.POINTER(FrameStats)], C.c_int),
        "mlm_shard_last_exchange": ([vp, C.POINTER(ShardExchange)], C.c_int),
        "mlm_shard_close": ([vp], C.c_int),
        "mlm_shard_last_kernel_ms": ([vp, fp], C.c_int),
        "mlm_dirty_count": ([vp, ip, C.POINTER(sz)], C.c_int),
        "mlm_dirty_export": ([vp, vp, C.c_int32], C.c_int),
        "mlm_dirty_import": ([vp, vp, C.c_int32], C.c_int),
        "mlm_replica_open": ([vp, C.c_int, C.c_int, C.c_int, vp], C.c_int),
        "mlm_replica_connect": ([vp, vp], C.c_int),
        "mlm_replica_publish": ([vp, C.POINTER(C.c_int32)], C.c_int),
        "mlm_replica_apply": ([vp, C.POINTER(C.c_int32)], C.c_int),
        "mlm_replica_close": ([vp], C.c_int),
        "mlm_debug_log10f": ([vp, vp, sz, vp], C.c_int),
        "mlm_debug_phase_cycles": ([vp, vp, sz], C.c_int),
        "mlm_srand": ([vp, C.c_uint], C.c_int),
        "mlm_debug_rand": ([vp, vp, sz], C.c_int),
        "mlm_set_profiling": ([vp, C.c_int], C.c_int),
        "mlm_last_frame_kernel_ms": ([vp, fp], C.c_int),
    }
    for name, (args, ret) in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = ret
    if (lib.mlm_sizeof_config() != C.sizeof(MlmConfig) or lib.mlm_sizeof_frame_stats() != C.sizeof(FrameStats)
            or not lib.mlm_sizeof_ray_hit() == C.sizeof(RayHit) == RAY_HIT_DTYPE.itemsize
            or lib.mlm_sizeof_frontier_cluster() != FRONTIER_CLUSTER_DTYPE.itemsize
            or lib.mlm_sizeof_view_gain() != VIEW_GAIN_DTYPE.itemsize):
        raise MlmError(1, "ctypes struct layout does not match include/mlmap_b200.h")
    _lib = lib
    return lib


def default_config() -> MlmConfig:
    """the live reference configuration, launch/config/config_sim.yaml (filled by the C library)"""
    cfg = MlmConfig()
    rc = load_library().mlm_default_config(C.byref(cfg))
    if rc != MLM_OK:
        raise MlmError(rc, "mlm_default_config")
    return cfg


def _base_config() -> MlmConfig:
    """SURVEY §8d common parameters (config_sim.yaml:20-24,42,51-55) without needing the library"""
    c = MlmConfig()
    c.use_raycasting = 1
    c.subbox_n = 10
    c.log_odds_min, c.log_odds_max = -2.0, 4.2
    c.log_odds_hit, c.log_odds_miss, c.log_odds_occupied_sh = 0.7, -0.9, 3.0
    c.use_exploration_frontiers = 0
    c.T_bs[:] = [0.12, 0.0, 0.0, 0.5, -0.5, 0.5, -0.5]
    c.inflate_n, c.inflate_global_n, c.apply_inflate, c.inflate_height = 2, 2, 1, 0.1
    c.sample_cnt = 0
    return c


def config_cfg_a() -> MlmConfig:
    """CFG-A (BASELINE configs 1 & 2): D435i-like 640x480 @ 0.1 m (SURVEY §8d)"""
    c = _base_config()
    c.am_d_rho, c.am_d_phi_deg, c.am_d_z = 0.1, 1.0, 0.1
    c.am_n_rho, c.am_n_z_below, c.am_n_z_over = 65, 20, 20
    c.depth_noise_coe = 0.00375
    c.subbox_d_xyz = 0.1
    c.cam_cx, c.cam_cy, c.cam_fx, c.cam_fy = 320.0, 240.0, 347.99755859375, 347.99755859375
    c.max_points = 640 * 480
    c.pool_submaps = 16384
    return c


def config_cfg_b() -> MlmConfig:
    """CFG-B (BASELINE config 3): L515-like 1024x768 @ 0.05 m (synthetic, SURVEY §8d)"""
    c = _base_config()
    c.am_d_rho, c.am_d_phi_deg, c.am_d_z = 0.05, 1.0, 0.05
    c.am_n_rho, c.am_n_z_below, c.am_n_z_over = 180, 40, 40
    c.depth_noise_coe = 0.001
    c.subbox_d_xyz = 0.05
    c.cam_cx, c.cam_cy, c.cam_fx, c.cam_fy = 512.0, 384.0, 731.0, 731.0
    c.max_points = 1024 * 768
    c.pool_submaps = 131072
    return c


def config_cfg_c() -> MlmConfig:
    """CFG-C (BASELINE config 4): 128-beam LiDAR, 0.2 m voxels, 50 m range (synthetic, SURVEY §8d)"""
    c = _base_config()
    c.am_d_rho, c.am_d_phi_deg, c.am_d_z = 0.2, 1.0, 0.2
    c.am_n_rho, c.am_n_z_below, c.am_n_z_over = 250, 100, 100
    c.depth_noise_coe = 1e-4
    c.subbox_d_xyz = 0.2
    c.T_bs[:] = [0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0]
    c.cam_cx, c.cam_cy, c.cam_fx, c.cam_fy = 0.0, 0.0, 1.0, 1.0
    c.max_points = 128 * 2048
    c.pool_submaps = 65536
    return c


def _pose7(T_wb) -> "C.Array":
    a = np.ascontiguousarray(np.asarray(T_wb, dtype=np.float64).reshape(7))
    return (C.c_double * 7)(*a.tolist())


def compensate_pose(pos, quat_wxyz, lin_vel, ang_vel, gap_odom_s, gap_imu_s, latency_s) -> np.ndarray:
    """pose forwarded to the image stamp as in depth_odom_input_callback (src/mlmap.cpp:470-498): pose7 for integrate_*"""
    lib = load_library()
    a = [(C.c_double * len(v))(*[float(x) for x in v]) for v in (pos, quat_wxyz, lin_vel, ang_vel)]
    out = (C.c_double * 7)()
    rc = lib.mlm_compensate_pose(a[0], a[1], a[2], a[3], float(gap_odom_s), float(gap_imu_s), float(latency_s), out)
    if rc != MLM_OK:
        raise MlmError(rc, "mlm_compensate_pose")
    return np.array(out[:], dtype=np.float64)


class MLMap:
    """Host-side mirror of the reference's ``class mlmap`` (include/mlmap.h:105-139) over the C ABI.

    ``init_map(ros::NodeHandle&)`` becomes the constructor taking an ``MlmConfig``;
    ``project_depth()+update_map()`` become ``integrate_depth`` (full-frame mode); the inline
    queries are batched: positions are ``(n,3)`` float64 arrays."""

    FREE, OCCUPIED, UNKNOWN = FREE, OCCUPIED, UNKNOWN

    def __init__(self, cfg: MlmConfig, device: int = 0):
        self._lib = load_library()
        self.cfg = cfg.copy()
        self._h = C.c_void_p()
        rc = self._lib.mlm_create(C.byref(self.cfg), device, C.byref(self._h))
        if rc != MLM_OK:
            raise MlmError(rc, self._lib.mlm_last_error().decode())
        self.device = device
        self.has_data = False
        self.map_updated = False
        self.cells = self.cfg.subbox_n ** 3

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.mlm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != MLM_OK:
            raise MlmError(rc, self._lib.mlm_last_error().decode())

    # ---- per-frame update ------------------------------------------------------------------
    def integrate_depth(self, img_u16: np.ndarray, T_wb) -> FrameStats:
        """project_depth() + update_map() (reference src/mlmap.cpp:311-349,382-386)"""
        img = np.asarray(img_u16)
        assert img.dtype == np.uint16 and img.ndim == 2
        if img.strides[1] != 2:
            img = np.ascontiguousarray(img)
        st = FrameStats()
        # the binding itself is on the end-to-end path: a reused pose buffer instead of fresh ctypes objects
        self._check(self._lib.mlm_integrate_depth_u16(self._h, img.ctypes.data, img.shape[0], img.shape[1],
                                                      img.strides[0], self._pose(T_wb), C.byref(st)))
        self.has_data = self.map_updated = True
        return st

    def integrate_depth_ptr(self, host_ptr: int, rows: int, cols: int, stride_bytes: int, T_wb) -> FrameStats:
        """mlm_integrate_depth_u16 on a raw host address (what a C/C++ caller passes): no numpy work on the call path"""
        st = FrameStats()
        self._check(self._lib.mlm_integrate_depth_u16(self._h, host_ptr, rows, cols, stride_bytes, self._pose(T_wb), C.byref(st)))
        self.has_data = self.map_updated = True
        return st

    def _pose(self, T_wb):
        buf = self.__dict__.get("_pose_buf")
        if buf is None:
            buf = self._pose_buf = (C.c_double * 7)()
            self._pose_np = np.frombuffer(buf, dtype=np.float64)
        self._pose_np[:] = T_wb
        return buf

    def integrate_depth_device(self, d_img: int, rows: int, cols: int, T_wb) -> FrameStats:
        st = FrameStats()
        self._check(self._lib.mlm_integrate_depth_u16_device(self._h, d_img, rows, cols, self._pose(T_wb), C.byref(st)))
        return st

    def integrate_points(self, xyz: np.ndarray, T_wb) -> FrameStats:
        """awareness_map->input_pc_pose + local_map->input_pc_pose_direct (src/mlmap.cpp:382-386)"""
        pts = np.ascontiguousarray(np.asarray(xyz, dtype=np.float64).reshape(-1, 3))
        st = FrameStats()
        self._check(self._lib.mlm_integrate_points_f64(self._h, pts.ctypes.data, pts.shape[0], _pose7(T_wb), C.byref(st)))
        self.has_data = self.map_updated = True
        return st

    # ---- the two layer entry points of update_map (awareness_map->input_pc_pose, local_map->input_pc_pose_direct) ----
    def awareness_input_pc_pose(self, xyz: np.ndarray, T_wb) -> FrameStats:
        pts = np.ascontiguousarray(np.asarray(xyz, dtype=np.float64).reshape(-1, 3))
        st = FrameStats()
        self._check(self._lib.mlm_awareness_input_pc_pose_f64(self._h, pts.ctypes.data, pts.shape[0], _pose7(T_wb), C.byref(st)))
        return st

    def awareness_input_depth(self, img: np.ndarray, T_wb) -> FrameStats:
        img = np.ascontiguousarray(img, dtype=np.uint16)
        st = FrameStats()
        self._check(self._lib.mlm_awareness_input_depth_u16(self._h, img.ctypes.data, img.shape[0], img.shape[1], img.strides[0],
                                                            _pose7(T_wb), C.byref(st)))
        return st

    def local_input_pc_pose_direct(self) -> FrameStats:
        st = FrameStats()
        self._check(self._lib.mlm_local_input_pc_pose_direct(self._h, C.byref(st)))
        self.has_data = self.map_updated = True
        return st

    # ---- asynchronous frames (several maps of one process on one GPU) ----
    def set_sm_budget(self, n_sms: int):
        self._check(self._lib.mlm_set_sm_budget(self._h, n_sms))

    def submit_depth_device(self, d_img: int, rows: int, cols: int, T_wb):
        self._check(self._lib.mlm_frame_submit_depth_u16_device(self._h, d_img, rows, cols, self._pose(T_wb)))

    def submit_points_device(self, d_xyz: int, n: int, T_wb):
        self._check(self._lib.mlm_frame_submit_points_f64_device(self._h, d_xyz, n, self._pose(T_wb)))

    def finish_frame(self) -> FrameStats:
        st = FrameStats()
        self._check(self._lib.mlm_frame_finish(self._h, C.byref(st)))
        return st

    def getOdd_at(self, glb3, sub) -> np.ndarray:
        """getOdd(const Vec3I &glb_id, size_t subbox_id), include/mlmap.h:128"""
        g = np.ascontiguousarray(np.asarray(glb3, dtype=np.int32).reshape(-1, 3))
        sb = np.ascontiguousarray(np.asarray(sub, dtype=np.int32).reshape(-1))
        out = np.empty(g.shape[0], dtype=np.float32)
        self._check(self._lib.mlm_get_odd_at(self._h, g.ctypes.data, sb.ctypes.data, g.shape[0], out.ctypes.data))
        return out

    def integrate_points_device(self, d_xyz: int, n: int, T_wb) -> FrameStats:
        st = FrameStats()
        self._check(self._lib.mlm_integrate_points_f64_device(self._h, d_xyz, n, self._pose(T_wb), C.byref(st)))
        return st

    def setFree_map_in_bound(self, box_min, box_max):
        mn = (C.c_double * 3)(*[float(v) for v in box_min])
        mx = (C.c_double * 3)(*[float(v) for v in box_max])
        self._check(self._lib.mlm_set_free_in_bound(self._h, mn, mx))

    def inflate_map(self, ct_pos):
        p = (C.c_double * 3)(*[float(v) for v in ct_pos])
        self._check(self._lib.mlm_inflate_map(self._h, p))

    # ---- queries ---------------------------------------------------------------------------------
    @staticmethod
    def _pos(pos_w):
        return np.ascontiguousarray(np.asarray(pos_w, dtype=np.float64).reshape(-1, 3))

    def getOccupancy(self, pos_w, inflate: float | None = None) -> np.ndarray:
        p = self._pos(pos_w)
        out = np.empty(p.shape[0], dtype=np.int32)
        if inflate is None:
            self._check(self._lib.mlm_get_occupancy(self._h, p.ctypes.data, p.shape[0], out.ctypes.data))
        else:
            self._check(self._lib.mlm_get_occupancy_inflate(self._h, p.ctypes.data, p.shape[0], float(inflate),
                                                            out.ctypes.data))
        return out

    def getInflateOccupancy(self, pos_w) -> np.ndarray:
        p = self._pos(pos_w)
        out = np.empty(p.shape[0], dtype=np.int32)
        self._check(self._lib.mlm_get_inflate_occupancy(self._h, p.ctypes.data, p.shape[0], out.ctypes.data))
        return out

    def getOdd(self, pos_w) -> np.ndarray:
        p = self._pos(pos_w)
        out = np.empty(p.shape[0], dtype=np.float32)
        self._check(self._lib.mlm_get_odd(self._h, p.ctypes.data, p.shape[0], out.ctypes.data))
        return out

    def getOddGrad(self, pos_w, max_iter: int = 5) -> np.ndarray:
        p = self._pos(pos_w)
        out = np.empty((p.shape[0], 3), dtype=np.float64)
        self._check(self._lib.mlm_get_odd_grad(self._h, p.ctypes.data, p.shape[0], max_iter, out.ctypes.data))
        return out

    # ---- batched ray casting (no reference counterpart; spec in include/mlmap_b200.h) ----------------
    def cast_rays(self, from_, to, inflated: bool = False) -> np.ndarray:
        """segments from_[i] -> to[i] ((n,3) world coordinates) walked cell by cell up to the first blocking cell:
        a structured array of RAY_HIT_DTYPE (status OCCUPIED / FREE / RAY_INVALID, stop cell, free and unknown cells
        crossed, t of the stop cell).  inflated: cells of the inflation layer block too."""
        a, b = self._pos(from_), self._pos(to)
        if a.shape != b.shape:
            raise ValueError(f"from_ and to differ in shape: {a.shape} vs {b.shape}")
        out = np.empty(a.shape[0], dtype=RAY_HIT_DTYPE)
        self._check(self._lib.mlm_cast_rays(self._h, a.ctypes.data, b.ctypes.data, a.shape[0],
                                            RAY_INFLATED if inflated else 0, out.ctypes.data))
        return out

    def cast_rays_device(self, d_from: int, d_to: int, n: int, d_out: int, inflated: bool = False):
        """the same on device memory (n x 3 doubles each, n 32-byte records); only enqueues on the handle's stream"""
        self._check(self._lib.mlm_cast_rays_device(self._h, d_from, d_to, n, RAY_INFLATED if inflated else 0, d_out))

    # ---- signed distance field over a box (no reference counterpart; spec in include/mlmap_b200.h) ------
    def build_esdf(self, box_min, box_max, max_dist: float, inflated: bool = False):
        """exact Euclidean distance transform of the box's blocking cells (occupied; with inflated also the inflation
        layer), clamped to max_dist; a snapshot of the map until the next build.  Only enqueues."""
        a = (C.c_double * 3)(*[float(v) for v in np.asarray(box_min, dtype=np.float64).reshape(3)])
        b = (C.c_double * 3)(*[float(v) for v in np.asarray(box_max, dtype=np.float64).reshape(3)])
        self._check(self._lib.mlm_esdf_build(self._h, a, b, float(max_dist), ESDF_INFLATED if inflated else 0))

    def esdf_distance(self, pos_w):
        """(dist[n], grad[n, 3]): trilinear distance and its gradient at (n,3) world points; NaN and a zero gradient
        outside the box"""
        p = self._pos(pos_w)
        dist = np.empty(p.shape[0], dtype=np.float64)
        grad = np.empty((p.shape[0], 3), dtype=np.float64)
        self._check(self._lib.mlm_esdf_distance(self._h, p.ctypes.data, p.shape[0], dist.ctypes.data, grad.ctypes.data))
        return dist, grad

    def esdf_distance_device(self, d_pos: int, n: int, d_dist: int, d_grad: int = 0):
        """the same on device memory (n x 3 doubles in, n doubles and optionally n x 3 doubles out); only enqueues"""
        self._check(self._lib.mlm_esdf_distance_device(self._h, d_pos, n, d_dist, d_grad or None))

    def export_esdf(self):
        """(grid[N_z, N_y, N_x] float32, lo[3] int32): the cell values of the last build"""
        lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
        self._check(self._lib.mlm_esdf_export(self._h, None, 0, lo, dims))
        out = np.empty((dims[2], dims[1], dims[0]), dtype=np.float32)
        self._check(self._lib.mlm_esdf_export(self._h, out.ctypes.data, out.size, lo, dims))
        return out, np.array(lo[:], dtype=np.int32)

    def export_esdf_device(self, d_out: int, cap: int):
        """the grid into device memory of cap floats (only enqueues): (lo[3], dims[3] = N_x, N_y, N_z)"""
        lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
        self._check(self._lib.mlm_esdf_export_device(self._h, d_out or None, cap, lo, dims))
        return np.array(lo[:], dtype=np.int32), np.array(dims[:], dtype=np.int32)

    # ---- frontier clustering (no reference counterpart; spec in include/mlmap_b200.h) -------------------------
    @staticmethod
    def _frontier_box(box_min, box_max):
        if (box_min is None) != (box_max is None):
            raise ValueError("box_min and box_max go together")
        if box_min is None:
            return None, None
        return tuple((C.c_double * 3)(*[float(v) for v in np.asarray(b, dtype=np.float64).reshape(3)]) for b in (box_min, box_max))

    def frontier_clusters(self, box_min=None, box_max=None, min_cells: int = 1, conn6: bool = False, labels: bool = False):
        """connected components of the frontier sets (26-connected, or 6 with conn6), optionally inside a box: the
        clusters with >= min_cells cells as FRONTIER_CLUSTER_DTYPE records sorted by key (z, y, x); with labels also
        (cells[m, 3] int32, cluster_of[m] int32), every cell of a kept cluster with its cluster index"""
        a, b = self._frontier_box(box_min, box_max)
        flags = FRONTIER_CONN6 if conn6 else 0
        cap, cell_cap = self.__dict__.get("_fc_cap", 256), (self.__dict__.get("_fc_cell_cap", 4096) if labels else 0)
        n, m = C.c_size_t(), C.c_size_t()
        while True:
            out = np.empty(cap, dtype=FRONTIER_CLUSTER_DTYPE)
            cells = np.empty((cell_cap, 3), dtype=np.int32)
            of = np.empty(cell_cap, dtype=np.int32)
            self._check(self._lib.mlm_frontier_clusters(self._h, a, b, int(min_cells), flags, out.ctypes.data, cap,
                                                        C.byref(n), cells.ctypes.data if labels else None,
                                                        of.ctypes.data if labels else None, cell_cap, C.byref(m)))
            if n.value <= cap and (not labels or m.value <= cell_cap):
                break
            cap, cell_cap = max(cap, n.value), (max(cell_cap, m.value) if labels else 0)  # too small: size and retry
        self._fc_cap = cap
        if labels:
            self._fc_cell_cap = cell_cap
            return out[:n.value].copy(), cells[:m.value].copy(), of[:m.value].copy()
        return out[:n.value].copy()

    def frontier_clusters_device(self, d_out: int, cap: int, d_cells3: int = 0, d_cluster_of: int = 0, cell_cap: int = 0,
                                 box_min=None, box_max=None, min_cells: int = 1, conn6: bool = False):
        """the same into device memory (cap 64-byte records; cell_cap cells and labels): (clusters, labelled cells)"""
        a, b = self._frontier_box(box_min, box_max)
        n, m = C.c_size_t(), C.c_size_t()
        self._check(self._lib.mlm_frontier_clusters_device(self._h, a, b, int(min_cells), FRONTIER_CONN6 if conn6 else 0,
                                                           d_out or None, cap, C.byref(n), d_cells3 or None,
                                                           d_cluster_of or None, cell_cap, C.byref(m)))
        return n.value, m.value

    # ---- candidate-view gain (no reference counterpart; spec in include/mlmap_b200.h) --------------------------
    @staticmethod
    def _view_flags(frontier: bool, inflated: bool) -> int:
        return (VIEW_FRONTIER if frontier else 0) | (VIEW_INFLATED if inflated else 0)

    def view_gain(self, poses, sensor: ViewSensor, boxes=None, frontier: bool = False, inflated: bool = False) -> np.ndarray:
        """per body pose ((n, 7) tx ty tz qw qx qy qz, as the frames take them) the target cells in the frustum of a depth
        sensor mounted at T_bs (unknown cells, or with frontier the frontier-set cells) and how many of them it sees
        through free cells (inflated: the inflation layer blocks too): VIEW_GAIN_DTYPE records (status 0 or
        VIEW_INVALID, n_target, n_visible).  boxes: (n, 6) int32 inclusive cells lo[3], hi[3] that bound each view."""
        p = np.ascontiguousarray(np.asarray(poses, dtype=np.float64).reshape(-1, 7))
        b = None
        if boxes is not None:
            b = np.ascontiguousarray(np.asarray(boxes, dtype=np.int32).reshape(-1, 6))
            if b.shape[0] != p.shape[0]:
                raise ValueError(f"{p.shape[0]} poses but {b.shape[0]} boxes")
        out = np.zeros(p.shape[0], dtype=VIEW_GAIN_DTYPE)
        self._check(self._lib.mlm_view_gain(self._h, p.ctypes.data, p.shape[0], C.byref(sensor),
                                            None if b is None else b.ctypes.data, self._view_flags(frontier, inflated),
                                            out.ctypes.data))
        return out

    def view_gain_device(self, d_poses: int, n: int, sensor: ViewSensor, d_out: int, d_boxes: int = 0,
                         frontier: bool = False, inflated: bool = False):
        """the same on device memory (n x 7 doubles, n x 6 int32 boxes or 0, n 16-byte records); only enqueues"""
        self._check(self._lib.mlm_view_gain_device(self._h, d_poses, n, C.byref(sensor), d_boxes or None,
                                                   self._view_flags(frontier, inflated), d_out))

    # ---- reachability field over a box (no reference counterpart; spec in include/mlmap_b200.h) ---------------
    def build_reach(self, box_min, box_max, starts, max_dist: float, inflated: bool = False, unknown: bool = False) -> int:
        """exact 26-connected shortest-path costs from the cells of `starts` ((n,3) world points) through the box's free
        cells (inflated: not the inflation layer; unknown: unknown cells too), moves never cutting a corner, up to
        max_dist; a snapshot of the map until the next build.  Returns the number of distinct source cells."""
        a = (C.c_double * 3)(*[float(v) for v in np.asarray(box_min, dtype=np.float64).reshape(3)])
        b = (C.c_double * 3)(*[float(v) for v in np.asarray(box_max, dtype=np.float64).reshape(3)])
        s = self._pos(starts)
        n = C.c_int32()
        flags = (REACH_INFLATED if inflated else 0) | (REACH_UNKNOWN if unknown else 0)
        self._check(self._lib.mlm_reach_build(self._h, a, b, s.ctypes.data, s.shape[0], float(max_dist), flags, C.byref(n)))
        return n.value

    def reach_cost(self, pos_w) -> np.ndarray:
        """path cost in metres at (n,3) world points: +inf where unreachable, NaN outside the box"""
        p = self._pos(pos_w)
        out = np.empty(p.shape[0], dtype=np.float64)
        self._check(self._lib.mlm_reach_cost(self._h, p.ctypes.data, p.shape[0], out.ctypes.data))
        return out

    def reach_cost_device(self, d_pos: int, n: int, d_out: int):
        """the same on device memory (n x 3 doubles in, n doubles out); only enqueues"""
        self._check(self._lib.mlm_reach_cost_device(self._h, d_pos, n, d_out))

    def reach_paths(self, goals, max_cells: int):
        """shortest paths from each goal back to a source: (cells[n, max_cells, 3] int32, goal first, len[n] int32 = the
        full length, which may exceed max_cells; -1 unreachable, -2 outside the box)"""
        g = self._pos(goals)
        n = g.shape[0]
        cells = np.zeros((n, max_cells, 3), dtype=np.int32)
        ln = np.empty(n, dtype=np.int32)
        self._check(self._lib.mlm_reach_paths(self._h, g.ctypes.data, n, max_cells, cells.ctypes.data, ln.ctypes.data))
        return cells, ln

    def reach_paths_device(self, d_goals: int, n: int, max_cells: int, d_cells3: int, d_len: int):
        """the same on device memory (n x 3 doubles, n * max_cells * 3 and n int32); only enqueues"""
        self._check(self._lib.mlm_reach_paths_device(self._h, d_goals, n, max_cells, d_cells3 or None, d_len))

    def export_reach(self):
        """(grid[N_z, N_y, N_x] int32, lo[3] int32): the costs of the last build, -1 where unreachable"""
        lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
        self._check(self._lib.mlm_reach_export(self._h, None, 0, lo, dims))
        out = np.empty((dims[2], dims[1], dims[0]), dtype=np.int32)
        self._check(self._lib.mlm_reach_export(self._h, out.ctypes.data, out.size, lo, dims))
        return out, np.array(lo[:], dtype=np.int32)

    def export_reach_device(self, d_out: int, cap: int):
        """the grid into device memory of cap int32 (only enqueues): (lo[3], dims[3] = N_x, N_y, N_z)"""
        lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
        self._check(self._lib.mlm_reach_export_device(self._h, d_out or None, cap, lo, dims))
        return np.array(lo[:], dtype=np.int32), np.array(dims[:], dtype=np.int32)

    # ---- path-cost matrix over a box (no reference counterpart; spec in include/mlmap_b200.h) --------------------
    @staticmethod
    def _box3(box_min, box_max):
        return tuple((C.c_double * 3)(*[float(v) for v in np.asarray(b, dtype=np.float64).reshape(3)])
                     for b in (box_min, box_max))

    def reach_matrix(self, box_min, box_max, starts, goals, max_dist: float, inflated: bool = False,
                     unknown: bool = False) -> np.ndarray:
        """(n_starts, n_goals) path costs in metres: row i is reach_cost(goals) after build_reach(box_min, box_max,
        [starts[i]], max_dist, inflated, unknown) (+inf unreachable, NaN outside the box); the last build_reach field
        is left as it is"""
        a, b = self._box3(box_min, box_max)
        s, g = self._pos(starts), self._pos(goals)
        out = np.empty((s.shape[0], g.shape[0]), dtype=np.float64)
        flags = (REACH_INFLATED if inflated else 0) | (REACH_UNKNOWN if unknown else 0)
        self._check(self._lib.mlm_reach_matrix(self._h, a, b, s.ctypes.data, s.shape[0], g.ctypes.data, g.shape[0],
                                               float(max_dist), flags, out.ctypes.data))
        return out

    def reach_matrix_device(self, box_min, box_max, d_starts: int, n_starts: int, d_goals: int, n_goals: int,
                            max_dist: float, d_out: int, inflated: bool = False, unknown: bool = False):
        """the same on device memory (n_starts x 3 and n_goals x 3 doubles in, n_starts x n_goals doubles out); only
        enqueues"""
        a, b = self._box3(box_min, box_max)
        flags = (REACH_INFLATED if inflated else 0) | (REACH_UNKNOWN if unknown else 0)
        self._check(self._lib.mlm_reach_matrix_device(self._h, a, b, d_starts or None, n_starts, d_goals or None,
                                                      n_goals, float(max_dist), flags, d_out or None))

    # ---- stream / timing -------------------------------------------------------------------------
    def sync(self):
        self._check(self._lib.mlm_sync(self._h))

    def timer_start(self):
        self._check(self._lib.mlm_timer_start(self._h))

    def timer_stop_ms(self) -> float:
        ms = C.c_float()
        self._check(self._lib.mlm_timer_stop_ms(self._h, C.byref(ms)))
        return ms.value

    def flush_l2(self):
        self._check(self._lib.mlm_flush_l2(self._h))

    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._check(self._lib.mlm_device_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, ptr: int):
        self._check(self._lib.mlm_device_free(self._h, ptr))

    def pinned_array(self, shape, dtype) -> np.ndarray:
        """numpy view of page-locked host memory (never freed before the handle is closed)"""
        dt = np.dtype(dtype)
        n = int(np.prod(shape)) * dt.itemsize
        p = C.c_void_p()
        self._check(self._lib.mlm_host_alloc(self._h, max(n, 16), C.byref(p)))
        buf = (C.c_char * n).from_address(p.value)
        return np.frombuffer(buf, dtype=dt).reshape(shape)

    def to_device(self, arr: np.ndarray) -> int:
        a = np.ascontiguousarray(arr)
        p = self.device_alloc(max(a.nbytes, 16))
        self._check(self._lib.mlm_copy_to_device(self._h, p, a.ctypes.data, a.nbytes))
        return p

    def to_host(self, ptr: int, shape, dtype) -> np.ndarray:
        out = np.empty(shape, dtype=dtype)
        self._check(self._lib.mlm_copy_to_host(self._h, out.ctypes.data, ptr, out.nbytes))
        return out

    def set_profiling(self, enable: bool = True):
        self._check(self._lib.mlm_set_profiling(self._h, 1 if enable else 0))

    def last_frame_kernel_ms(self) -> dict:
        ms = (C.c_float * len(FRAME_KERNELS))()
        self._check(self._lib.mlm_last_frame_kernel_ms(self._h, ms))
        return dict(zip(FRAME_KERNELS, [float(v) for v in ms]))

    def debug_phase_cycles(self) -> np.ndarray:
        n = 2 * int(360 / self.cfg.am_d_phi_deg) + 256  # work columns (up to two half columns per phi) + per-CTA rows of k_frame
        out = np.zeros((n, 16), dtype=np.int64)
        self._check(self._lib.mlm_debug_phase_cycles(self._h, out.ctypes.data, out.size))
        return out

    def srand(self, seed: int):
        self._check(self._lib.mlm_srand(self._h, seed))

    def kernel_launch_count(self) -> int:
        v = C.c_int64()
        self._check(self._lib.mlm_kernel_launch_count(self._h, C.byref(v)))
        return v.value

    # ---- device-resident queries (enqueue only) ---------------------------------------------------
    def getOccupancy_device(self, d_pos: int, n: int, d_out: int):
        self._check(self._lib.mlm_get_occupancy_device(self._h, d_pos, n, d_out))

    def getOdd_device(self, d_pos: int, n: int, d_out: int):
        self._check(self._lib.mlm_get_odd_device(self._h, d_pos, n, d_out))

    def getOddGrad_device(self, d_pos: int, n: int, d_out: int, max_iter: int = 5):
        self._check(self._lib.mlm_get_odd_grad_device(self._h, d_pos, n, max_iter, d_out))

    # ---- parity / debug exports --------------------------------------------------------------------
    def last_frame_hits(self):
        """(keys[n,3] int32 (rho,phi,z), p[n] float32) in the reference's hash-map iteration order"""
        n = C.c_size_t()
        self._check(self._lib.mlm_last_frame_hits(self._h, None, None, 0, C.byref(n)))
        keys = np.empty((n.value, 3), dtype=np.int32)
        p = np.empty(n.value, dtype=np.float32)
        if n.value:
            self._check(self._lib.mlm_last_frame_hits(self._h, keys.ctypes.data, p.ctypes.data, n.value, C.byref(n)))
        return keys, p

    def last_frame_misses(self) -> np.ndarray:
        n = C.c_size_t()
        self._check(self._lib.mlm_last_frame_misses(self._h, None, 0, C.byref(n)))
        idx = np.empty(n.value, dtype=np.uint64)
        if n.value:
            self._check(self._lib.mlm_last_frame_misses(self._h, idx.ctypes.data, n.value, C.byref(n)))
        return idx

    def checkpoint(self) -> bytes:
        """byte image of the whole map (see include/mlmap_b200.h, checkpoint / restore)"""
        n = C.c_size_t()
        self._check(self._lib.mlm_checkpoint_size(self._h, C.byref(n)))
        buf = (C.c_ubyte * n.value)()
        self._check(self._lib.mlm_checkpoint_save(self._h, buf, n.value, C.byref(n)))
        return bytes(buf[:n.value])

    def restore(self, image: bytes):
        """replace this handle's map by a checkpoint taken with the same map configuration"""
        buf = (C.c_ubyte * len(image)).from_buffer_copy(image)
        self._check(self._lib.mlm_checkpoint_restore(self._h, buf, len(image)))

    CLOUD_INFLATED, CLOUD_OCCUPIED, CLOUD_FRONTIER = 0, 1, 2

    def export_cloud(self, kind: int = 0) -> np.ndarray:
        """[n,4] float32 points x,y,z,1 (pcl::PointXYZ layout) of the cells the reference's map / frontier topics
        carry (rviz_vis.cpp:267-327); compacted on the device, order unspecified"""
        n = C.c_size_t()
        self._check(self._lib.mlm_export_cloud(self._h, kind, None, 0, C.byref(n)))
        out = np.zeros((n.value, 4), dtype=np.float32)
        if n.value:
            self._check(self._lib.mlm_export_cloud(self._h, kind, out.ctypes.data, n.value, C.byref(n)))
            assert n.value == out.shape[0]
        return out

    def export_cloud_device(self, kind: int, d_ptr: int, cap: int) -> int:
        """same compaction into caller device memory (cap float4 points); returns the number of points in the map"""
        n = C.c_size_t()
        self._check(self._lib.mlm_export_cloud_device(self._h, kind, d_ptr, cap, C.byref(n)))
        return n.value

    def export_odds_slice(self, height: float) -> np.ndarray:
        """[n,4] float32 x,y,z,odd of the cells at `height` (mlmap::visualize_odds, mlmap.cpp:200-284)"""
        n = C.c_size_t()
        self._check(self._lib.mlm_export_odds_slice(self._h, float(height), None, 0, C.byref(n)))
        out = np.zeros((n.value, 4), dtype=np.float32)
        if n.value:
            self._check(self._lib.mlm_export_odds_slice(self._h, float(height), out.ctypes.data, n.value, C.byref(n)))
        return out

    def export_map(self):
        """dict with glb[n,3], collapsed[n], occupancy[n,cells] (S1), inflate[n,cells], log_odds[n,cells],
        sorted by glb index"""
        n = C.c_size_t()
        self._check(self._lib.mlm_export_map_count(self._h, C.byref(n)))
        cap = n.value
        glb = np.zeros((cap, 3), dtype=np.int32)
        col = np.zeros(cap, dtype=np.uint8)
        occ = np.zeros((cap, self.cells), dtype="S1")
        inf = np.zeros((cap, self.cells), dtype="S1")
        lo = np.zeros((cap, self.cells), dtype=np.float32)
        if cap:
            self._check(self._lib.mlm_export_map(self._h, cap, glb.ctypes.data, col.ctypes.data, occ.ctypes.data,
                                                 inf.ctypes.data, lo.ctypes.data, C.byref(n)))
            assert n.value == cap, (n.value, cap)
        order = np.lexsort((glb[:, 2], glb[:, 1], glb[:, 0]))
        out = {"glb": glb[order], "collapsed": col[order], "occupancy": occ[order], "inflate": inf[order],
               "log_odds": lo[order]}
        if self.cfg.use_exploration_frontiers:
            fw = (self.cells + 31) // 32
            g2 = np.zeros((cap, 3), dtype=np.int32)
            words = np.zeros((cap, fw), dtype=np.uint32)
            if cap:
                self._check(self._lib.mlm_export_frontier(self._h, cap, g2.ctypes.data, words.ctypes.data, C.byref(n)))
            o2 = np.lexsort((g2[:, 2], g2[:, 1], g2[:, 0]))
            assert np.array_equal(g2[o2], out["glb"])
            # same byte layout as the oracle's export: bit c of the little-endian bitmask, cells/8 bytes per subbox
            out["frontier"] = words[o2].view(np.uint8)[:, :(self.cells + 7) // 8].copy()
        return out

    def debug_log10f(self, x: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(x, dtype=np.float32)
        out = np.empty_like(a)
        self._check(self._lib.mlm_debug_log10f(self._h, a.ctypes.data, a.size, out.ctypes.data))
        return out
