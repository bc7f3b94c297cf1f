"""Named points of the configuration space that mlm_create accepts, each derived from a preset by changing only the
fields its name states and aimed at one edge of the kernels' index arithmetic (tests/test_config_space_gpu.py runs
them against the oracle, tests/test_config_space_host.py checks the table itself).  Also the host's derived constants
that decide which kernel branches a configuration reaches: K(rho), maxK and the half-column split."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from mlmapping_b200 import config_cfg_a, config_cfg_c, default_config, scenes
from oracle_binding import k_reach, update_hits_ok

MAX_PHI = 4096           # kMaxPhi


def n_phi(cfg) -> int:
    return int(360 / cfg.am_d_phi_deg)


def split_of(cfg) -> int:
    """the half-column split rule of mlm_create: 0 means whole phi columns are the work items"""
    k = k_reach(cfg)
    r = np.arange(cfg.am_n_rho)
    nz = cfg.am_n_z_below + cfg.am_n_z_over + 1
    if ((k > 0) & (2 * k >= r)).any():
        return 0
    if cfg.am_n_z_below < 1 or cfg.am_n_z_below >= nz - 1 or cfg.am_n_rho >= 4096 or 2 * n_phi(cfg) > MAX_PHI:
        return 0
    return 1


def largest_noise_coe(cfg) -> float:
    """the largest depth_noise_coe (to 1e-12 relative) that keeps update_hits_ok(cfg)"""
    c = cfg.copy()
    lo, hi = 0.0, 1.0
    while True:
        c.depth_noise_coe = hi
        if not update_hits_ok(c):
            break
        lo, hi = hi, 2 * hi
    while hi - lo > 1e-12 * hi:
        c.depth_noise_coe = mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if update_hits_ok(c) else (lo, mid)
    return lo


def _quat_mul(a, b):
    w1, x1, y1, z1 = a
    w2, x2, y2, z2 = b
    return np.array([w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2, w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                     w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2, w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2])


def tilted_T_bs(base):
    """base T_bs rotated by 11 degrees about the (1, 2, 3) axis and moved by (0.07, -0.045, 0.13) m"""
    axis = np.array([1.0, 2.0, 3.0]) / np.sqrt(14.0)
    a = np.deg2rad(11.0)
    q = _quat_mul(np.asarray(base[3:7], dtype=np.float64), np.r_[np.cos(a / 2), np.sin(a / 2) * axis])
    q /= np.linalg.norm(q)
    return [base[0] + 0.07, base[1] - 0.045, base[2] + 0.13, *q.tolist()]


@dataclass
class Case:
    name: str
    make: object                  # () -> MlmConfig
    scene: str = "depth"          # "depth": 320 x 240 corridor frames; "lidar": 32 x 512 scans
    frames: int = 3
    stride: int = 10              # trajectory steps between frames
    y_offset: float = 0.0
    rows: int = 240
    cols: int = 320
    edge: str = ""
    pool_from_oracle: bool = False   # pool_submaps from the oracle's final subbox count (+ slack), for n <= 3


def _a(**kw):
    def make():
        c = config_cfg_a()
        for k, v in kw.items():
            setattr(c, k, v)
        return c
    return make


def _lidar(**kw):
    """CFG-C at 24 m range, z within +-6 m (the small LiDAR configuration of the GPU tests)"""
    def make():
        c = config_cfg_c()
        c.am_n_rho, c.am_n_z_below, c.am_n_z_over = 120, 30, 30
        c.max_points = 32 * 512
        c.pool_submaps = 8192
        for k, v in kw.items():
            setattr(c, k, v)
        return c
    return make


def _noise_wide(n_rho=None):
    def make():
        c = config_cfg_a()
        if n_rho is not None:
            c.am_n_rho = n_rho
        c.depth_noise_coe = largest_noise_coe(c)
        return c
    return make


def _camera():
    c = config_cfg_a()
    c.cam_cx, c.cam_cy, c.cam_fx, c.cam_fy = 131.25, 151.75, 301.5, 377.125
    c.T_bs[:] = tilted_T_bs(list(c.T_bs))
    return c


def _fine_cells():
    c = config_cfg_a()
    c.am_d_rho = c.am_d_z = 0.05
    c.am_d_phi_deg = 0.25
    c.am_n_rho, c.am_n_z_below, c.am_n_z_over = 100, 40, 40
    c.subbox_d_xyz = 0.2
    return c


CASES = [
    Case("default_yaml", default_config, rows=360, cols=640, frames=4, stride=7, edge="the shipped configuration"),
    Case("n2", _a(subbox_n=2), pool_from_oracle=True, edge="8 cells per subbox; getOddGrad walks over several subboxes"),
    Case("n3", _a(subbox_n=3), pool_from_oracle=True, edge="LSG nearly as large as the LVG"),
    Case("n7", _a(subbox_n=7), edge="cells = 343: padded cell stride, partial last frontier word"),
    Case("n16", _a(subbox_n=16, pool_submaps=512), edge="front_words = 128"),
    Case("n64", _a(subbox_n=64, pool_submaps=64), edge="front_words = 8192"),
    Case("phi5", _lidar(am_d_phi_deg=5.0), scene="lidar", edge="5 degree sector borders"),
    Case("phi7", _lidar(am_d_phi_deg=7.0), scene="lidar", edge="nPhi = 51: partial last sector"),
    Case("phi0_125", _lidar(am_d_phi_deg=0.125), scene="lidar", edge="nPhi = 2880 > 2048: whole columns"),
    Case("phi360", _lidar(am_d_phi_deg=360.0), scene="lidar", edge="nPhi = 1"),
    Case("no_raycast", _a(use_raycasting=0), edge="no ray walks, empty miss sets"),
    Case("below0", _a(am_n_z_below=0), edge="sensor row at the bottom of the grid, whole columns"),
    Case("over0", _a(am_n_z_over=0), edge="sensor row at the top of the grid, whole columns"),
    Case("noise_wide", _noise_wide(), edge="maxK = 10: 21 contributions per point"),
    Case("noise_wide_short", _noise_wide(n_rho=20), edge="2 K(rho) >= rho: whole columns"),
    Case("fine_cells", _fine_cells, edge="more than 16 hits per voxel"),
    Case("coarse_cells_0.03", _a(subbox_d_xyz=0.03), edge="voxels finer than the awareness cells, inexact 1/d"),
    Case("coarse_cells_0.25", _a(subbox_d_xyz=0.25), edge="voxels coarser than the awareness cells"),
    Case("nrho_words_31", _a(am_n_rho=31), edge="one bitmap word per row, one bit spare"),
    Case("nrho_words_32", _a(am_n_rho=32), edge="one full bitmap word per row"),
    Case("nrho_words_33", _a(am_n_rho=33), edge="two bitmap words per row"),
    Case("camera", _camera, edge="off-centre principal point, fx != fy, tilted and shifted T_bs"),
    Case("log_odds", _a(log_odds_min=-3.5, log_odds_max=2.5, log_odds_occupied_sh=2.4375, log_odds_hit=0.55,
                        log_odds_miss=-0.35), frames=6, stride=3, edge="asymmetric clamp, threshold just below the max"),
    Case("inflate_n0", _a(inflate_n=0), edge="inflation by 0 cells"),
    Case("inflate_n1", _a(inflate_n=1), edge="inflation by 1 cell"),
    Case("inflate_n3", _a(inflate_n=3), edge="inflation by 3 cells"),
    Case("no_apply_inflate", _a(apply_inflate=0), edge="inflate_map without the height rule"),
    Case("explore_n7", _a(subbox_n=7, use_exploration_frontiers=1), frames=10, edge="frontier words of 343 cells"),
    Case("explore_n16", _a(subbox_n=16, use_exploration_frontiers=1, pool_submaps=1024), frames=10,
         edge="128 frontier words per subbox"),
    Case("far_origin", _a(), y_offset=-5000.0, edge="negative cell coordinates far from 0"),
]
BY_NAME = {c.name: c for c in CASES}


def frames(case, cfg):
    """(kind, data, pose) of the case's input frames, kind "depth" or "points"""
    out = []
    for k in range(case.frames):
        if case.scene == "lidar":
            pose = scenes.lidar_loop_pose(3 * k)
            out.append(("points", scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512, max_range=25.0), pose))
        else:
            pose = scenes.corridor_trajectory_pose(case.stride * k, y_offset=case.y_offset)
            img = scenes.corridor_depth_frame(cfg, pose, rows=case.rows, cols=case.cols, frame_idx=k, y_offset=case.y_offset)
            out.append(("depth", img, pose))
    return out


def integrate(m, kind, data, pose):
    return m.integrate_depth(data, pose) if kind == "depth" else m.integrate_points(data, pose)


def config_of(case, oracle_cls=None):
    """the case's configuration; for pool_from_oracle cases the pool is sized from a run of the oracle"""
    cfg = case.make()
    if case.pool_from_oracle:
        from oracle_binding import Oracle
        orc = (oracle_cls or Oracle)(cfg)
        for kind, data, pose in frames(case, cfg):
            integrate(orc, kind, data, pose)
        cfg.pool_submaps = 2 * int(orc.export_map()["glb"].shape[0]) + 64
        orc.close()
    return cfg


def hits_per_voxel(cfg, keys, pose):
    """voxel of every hit cell (rho, phi, z) of a frame (centre of the awareness cell in the awareness frame, which is
    the body position with the world's axes), counted per voxel.  A numpy recomputation, not the kernel's own voxel
    assignment: a count above 16 shows that such voxels occur in the frame, not that the fusion's list-walk branch ran
    (a voxel on a cell border may fall on the other side here)."""
    d_phi = cfg.am_d_phi_deg * np.pi / 180
    z_min = -(cfg.am_n_z_below * cfg.am_d_z) - 0.5 * cfg.am_d_z
    rho = cfg.am_d_rho / 2 + keys[:, 0] * cfg.am_d_rho
    phi = d_phi / 2 + keys[:, 1] * d_phi
    z = z_min + cfg.am_d_z / 2 + keys[:, 2] * cfg.am_d_z
    p = np.c_[rho * np.cos(phi), rho * np.sin(phi), z] + np.asarray(pose[:3])
    vox = np.floor(p / cfg.subbox_d_xyz).astype(np.int64)
    _, counts = np.unique(vox, axis=0, return_counts=True)
    return counts
