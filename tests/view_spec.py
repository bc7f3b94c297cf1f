"""The candidate-view-gain spec of include/mlmap_b200.h ("candidate-view gain") restated in plain Python / numpy, apart
from both the C++ oracle and the kernels: the pose algebra written out, every cell of a cube around the origin that holds
the whole frustum brute-forced (not the AABB the oracle and the kernels share), and the line of sight from
raycast_spec.walk.  Python floats and numpy's element-wise float64 operations are IEEE doubles without fused
multiply-add, so the records agree bit for bit.  Also: a writer of checkpoint images with arbitrary cell states, inflation
bytes, collapsed subboxes and frontier sets, candidate views around frontier clusters, and the sensors of the tests.
TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from mlmapping_b200.capi import VIEW_GAIN_DTYPE, VIEW_INVALID, ViewSensor
from frontier_spec import CkptHeader, decode_frontier, fnv1a64
from raycast_spec import MapStates, cell_of, walk


# ---- pose algebra (the frame path's Sophus / Eigen subset, in its order of evaluation) ----------------------------
def q_normalized(q):
    w, x, y, z = q
    n2 = (x * x + z * z) + (y * y + w * w)
    if not n2 > 0:
        return q
    n = math.sqrt(n2)
    return (w / n, x / n, y / n, z / n)


def q_mul(a, b):
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    x = (aw * bx + ay * bz) - (az * by - ax * bw)
    y = (aw * by + ay * bw) + (az * bx - ax * bz)
    z = (aw * bz - ay * bx) + (az * bw + ax * by)
    w = (aw * bw - ay * by) - (az * bz + ax * bx)
    return (w, x, y, z)


def rotate(q, v):
    """Eigen _transformVector; v may hold numpy arrays (element-wise, same order)"""
    w, x, y, z = q
    uvx = y * v[2] - z * v[1]
    uvy = z * v[0] - x * v[2]
    uvz = x * v[1] - y * v[0]
    uvx = uvx + uvx
    uvy = uvy + uvy
    uvz = uvz + uvz
    cx = y * uvz - z * uvy
    cy = z * uvx - x * uvz
    cz = x * uvy - y * uvx
    return (v[0] + w * uvx + cx, v[1] + w * uvy + cy, v[2] + w * uvz + cz)


def pose_from7(p):
    return q_normalized((p[3], p[4], p[5], p[6])), (p[0], p[1], p[2])


def compose(a, b):
    rt = rotate(a[0], b[1])
    return q_normalized(q_mul(a[0], b[0])), tuple(a[1][k] + rt[k] for k in range(3))


def inverse(a):
    w, x, y, z = a[0]
    q = q_normalized((w, -x, -y, -z))
    return q, rotate(q, tuple(t * -1. for t in a[1]))


def transform(T, v):
    r = rotate(T[0], v)
    return tuple(r[k] + T[1][k] for k in range(3))


# ---- the spec -----------------------------------------------------------------------------------------------------
def half_extents(S):
    hx = max(abs((-0.5 - S.cx) / S.fx), abs((float(S.cols) - 0.5 - S.cx) / S.fx))
    hy = max(abs((-0.5 - S.cy) / S.fy), abs((float(S.rows) - 0.5 - S.cy) / S.fy))
    return hx, hy


def in_frustum(S, p):
    """rule 3 on sensor coordinates (numpy arrays)"""
    with np.errstate(divide="ignore", invalid="ignore"):
        u = (p[0] / p[2]) * S.fx + S.cx
        v = (p[1] / p[2]) * S.fy + S.cy
    return ((p[2] >= S.min_depth) & (p[2] <= S.max_depth) & (u >= -0.5) & (u < float(S.cols) - 0.5) & (v >= -0.5)
            & (v < float(S.rows) - 0.5))


def view_cells(pose7, S, d, T_bs7, box=None):
    """(origin, cell(o), cells in view as an (m, 3) int64 array, sorted (z, y, x)), or None for an invalid view"""
    p = [float(v) for v in pose7]
    if not all(math.isfinite(v) for v in p):
        return None
    n2 = (p[4] * p[4] + p[6] * p[6]) + (p[5] * p[5] + p[3] * p[3])
    if not (n2 > 0 and math.isfinite(n2)):
        return None
    Tws = compose(pose_from7(p), pose_from7([float(v) for v in T_bs7]))
    Tsw = inverse(Tws)
    o = Tws[1]
    co = [cell_of(v, d) for v in o]
    if None in co:
        return None
    if box is not None and any(box[k] > box[3 + k] for k in range(3)):
        return None
    hx, hy = half_extents(S)
    K = int(math.ceil(S.max_depth * math.sqrt(1.0 + hx * hx + hy * hy) / d)) + 2
    g = np.indices((2 * K + 1,) * 3).reshape(3, -1)[::-1].T - K + np.array(co)  # x fastest
    if box is not None:
        g = g[((g >= np.array(box[:3])) & (g <= np.array(box[3:]))).all(1)]
    x = tuple((g[:, k].astype(np.float64) + 0.5) * d for k in range(3))
    keep = in_frustum(S, transform(Tsw, x))
    return o, tuple(co), g[keep]


def gain(states: MapStates, frontier_cells, poses, S, d, T_bs7, boxes=None, frontier=False, inflated=False):
    """VIEW_GAIN_DTYPE records of every pose; frontier_cells: the set of frontier cells (tuples) for frontier targets"""
    out = np.zeros(len(poses), dtype=VIEW_GAIN_DTYPE)
    for i, pose in enumerate(np.asarray(poses, dtype=np.float64).reshape(-1, 7)):
        r = view_cells(pose, S, d, T_bs7, None if boxes is None else [int(v) for v in boxes[i]])
        if r is None:
            out[i] = (VIEW_INVALID, 0, 0, 0)
            continue
        o, co, cells = r
        nt = nv = 0
        for c in map(tuple, cells.tolist()):
            if frontier:
                if c not in frontier_cells:
                    continue
            elif states(c)[0] in (b"f", b"o"):
                continue
            nt += 1
            x = [(float(c[k]) + 0.5) * d for k in range(3)]
            _, stop, _, _, _, path = walk(list(o), x, d, states, inflated)
            if tuple(stop) == c and all(states(q)[0] == b"f" for q in path[:-1]):
                nv += 1
        out[i] = (0, nt, nv, 0)
    return out


def frontier_set(ex, n):
    return set(map(tuple, decode_frontier(ex, n).tolist()))


# ---- sensors and candidate views ----------------------------------------------------------------------------------
def sensor(fx=347.99755859375, cx=320.0, cy=240.0, cols=640, rows=480, min_depth=0.1, max_depth=1.0, fy=None):
    """the CFG-A camera by default (640 x 480, fx 348)"""
    return ViewSensor(fx, fx if fy is None else fy, cx, cy, cols, rows, min_depth, max_depth)


def look_at(pos, target, T_bs7):
    """pose7 of the body such that the sensor at T_bs looks from pos towards target (optical axis z, image x level)"""
    from scipy.spatial.transform import Rotation
    z = np.asarray(target, dtype=np.float64) - np.asarray(pos, dtype=np.float64)
    z /= np.linalg.norm(z)
    up = np.array([0.0, 0.0, 1.0])
    x = np.cross(z, up)
    if np.linalg.norm(x) < 1e-9:
        x = np.array([1.0, 0.0, 0.0])
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    R_ws = Rotation.from_matrix(np.stack([x, y, z], 1))
    q = T_bs7[3:]
    R_bs = Rotation.from_quat([q[1], q[2], q[3], q[0]])
    xyzw = (R_ws * R_bs.inv()).as_quat()
    return np.array([*pos, xyzw[3], xyzw[0], xyzw[1], xyzw[2]], dtype=np.float64)


def candidates_around(centroids, T_bs7, seed, per_cluster=8, r_lo=1.0, r_hi=3.0):
    """FUEL-style candidates: on rings of radius r_lo..r_hi around each centroid, at its height +- 0.3 m, looking at it;
    returns (poses (m, 7), index of the cluster of each)"""
    rs = np.random.RandomState(seed)
    poses, of = [], []
    for j, c in enumerate(np.asarray(centroids, dtype=np.float64).reshape(-1, 3)):
        for _ in range(per_cluster):
            r, a = rs.uniform(r_lo, r_hi), rs.uniform(0.0, 2 * np.pi)
            pos = c + np.array([r * np.cos(a), r * np.sin(a), rs.uniform(-0.3, 0.3)])
            poses.append(look_at(pos, c, T_bs7))
            of.append(j)
    return np.array(poses).reshape(-1, 7), np.array(of, dtype=np.int64)


# ---- checkpoint images of arbitrary maps --------------------------------------------------------------------------
def write_map_checkpoint(template: bytes, cfg, ex) -> bytes:
    """a checkpoint image with the template's header (a fresh exploration handle's) and one record per subbox of the
    export-like dict ex: occupancy and inflation bytes per cell, collapsed flags (element 0 kept), frontier bytes, and
    the log-odds of ex["log_odds"] when it has them (else 0).  n_records, n_submaps and the checksum are fixed."""
    hd = CkptHeader.from_buffer_copy(template[:C.sizeof(CkptHeader)])
    n = cfg.subbox_n
    cells, fw = n ** 3, (n ** 3 + 31) // 32
    rb = (32 + cells * 6 + fw * 4 + 15) & ~15
    assert hd.header_bytes == C.sizeof(CkptHeader) and hd.rec_bytes == rb and hd.explore == 1
    glb = np.asarray(ex["glb"], dtype=np.int32).reshape(-1, 3)
    m = glb.shape[0]
    col = np.asarray(ex["collapsed"], dtype=bool)
    occ = np.asarray(ex["occupancy"]).view(np.uint8).reshape(m, cells)
    inf = np.asarray(ex["inflate"]).view(np.uint8).reshape(m, cells)
    lo = np.zeros((m, cells), np.float32) if "log_odds" not in ex else np.asarray(ex["log_odds"], np.float32)
    assert lo.shape == (m, cells), lo.shape
    recs = np.zeros((m, rb), dtype=np.uint8)
    head = np.zeros(m, dtype=[("g", "<i4", (3,)), ("flags", "<i4"), ("col_lo", "<f4"), ("col_occ", "u1"),
                              ("col_inf", "u1"), ("pad", "S10")])
    head["g"] = glb
    head["flags"] = col.astype(np.int32)
    head["col_lo"], head["col_occ"], head["col_inf"] = lo[:, 0], occ[:, 0], inf[:, 0]
    recs[:, :32] = head.view(np.uint8).reshape(m, 32)
    full = ~col
    recs[full, 32:32 + 4 * cells] = lo[full].astype("<f4").view(np.uint8).reshape(-1, 4 * cells)
    recs[full, 32 + 4 * cells:32 + 5 * cells] = occ[full]
    recs[full, 32 + 5 * cells:32 + 6 * cells] = inf[full]
    fr = np.zeros((m, 4 * fw), dtype=np.uint8)
    fr[:, :np.asarray(ex["frontier"]).shape[1]] = ex["frontier"]
    recs[full, 32 + 6 * cells:32 + 6 * cells + 4 * fw] = fr[full]
    body = recs.tobytes()
    hd.n_records = hd.n_submaps = m
    hd.checksum = fnv1a64(body)
    return bytes(hd) + body


def crafted_map(cells_state: dict, n, inflated=(), frontier=(), collapsed: dict | None = None):
    """an export-like dict from {cell: b'f' / b'o' / b'u'} (every other cell of a listed subbox unknown), inflation 'o'
    on the cells of `inflated`, frontier bits on `frontier`, and collapsed subboxes {glb: state byte}"""
    keys = {tuple(int(v) // n for v in c) for c in list(cells_state) + list(inflated) + list(frontier)}
    keys |= set(collapsed or {})
    glb = sorted(keys)
    row = {g: i for i, g in enumerate(glb)}
    m, cells = len(glb), n ** 3
    occ = np.full((m, cells), b"u", dtype="S1")
    inf = np.full((m, cells), b"u", dtype="S1")
    fr = np.zeros((m, (cells + 7) // 8), dtype=np.uint8)
    col = np.zeros(m, dtype=np.uint8)

    def at(c):
        g = tuple(int(v) // n for v in c)
        loc = [int(c[k]) - g[k] * n for k in range(3)]
        return row[g], (loc[2] * n + loc[1]) * n + loc[0]

    for c, s in cells_state.items():
        i, sub = at(c)
        occ[i, sub] = s
    for c in inflated:
        i, sub = at(c)
        inf[i, sub] = b"o"
    for c in frontier:
        i, sub = at(c)
        fr[i, sub // 8] |= np.uint8(1 << (sub % 8))
    for g, s in (collapsed or {}).items():
        i = row[g]
        col[i] = 1
        occ[i, :] = s
        inf[i, :] = b"u"
        fr[i, :] = 0
    return {"glb": np.array(glb, dtype=np.int32).reshape(-1, 3), "collapsed": col, "occupancy": occ, "inflate": inf,
            "frontier": fr}
