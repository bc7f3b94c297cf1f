"""The reachability field (mlm_reach_*) restated in numpy / scipy from the spec in include/mlmap_b200.h: the move graph
of rule 4 built vectorised with the corner rule, costs from scipy.sparse.csgraph.dijkstra with the integer weights (exact
in float64 below 2^53), the path rule 7, and a checker for paths.  Class grids are [N_z, N_y, N_x] with 0 free,
1 blocking, 2 unknown (the ray spec's rule 3)."""
import itertools

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import dijkstra

from esdf_spec import box_of, cells_of

FREE, BLOCKING, UNKNOWN = 0, 1, 2
# the 26 offsets (dx, dy, dz) in the path rule's order: lexicographic in (dz, dy, dx), z slowest
OFFSETS = [(dx, dy, dz) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if (dx, dy, dz) != (0, 0, 0)]


def weight(d):
    return (0, 1000, 1414, 1732)[sum(1 for v in d if v)]


def passable(cls, sources, unknown=False):
    """T or S (rules 2 and 3) as a boolean grid; sources are box-relative (x, y, z) cells inside the box"""
    p = (cls == FREE) | ((cls == UNKNOWN) if unknown else False)
    for x, y, z in sources:
        p[z, y, x] = True
    return p


def _shift(a, d, fill=False):
    """b[c] = a[c + d] (fill outside), d = (dx, dy, dz)"""
    out = np.full_like(a, fill)
    src, dst = [], []
    for k, n in zip((2, 1, 0), a.shape):
        v = d[k]
        src.append(slice(max(v, 0), n + min(v, 0)))
        dst.append(slice(max(-v, 0), n + min(-v, 0)))
    out[tuple(dst)] = a[tuple(src)]
    return out


def allowed_moves(pas, d):
    """rule 4, vectorised: ok[a] = every cell a + d' with d'_k in {0, d_k} is passable"""
    ok = pas.copy()
    for sel in itertools.product(*[(0, v) if v else (0,) for v in d]):
        ok &= _shift(pas, sel)
    return ok


def field(cls, sources, K, unknown=False):
    """rule 5 on a class grid: int64 costs, -1 unreachable (scipy's Dijkstra over the move graph)"""
    src = [tuple(int(v) for v in s) for s in np.asarray(sources).reshape(-1, 3)
           if all(0 <= s[k] < cls.shape[2 - k] for k in range(3))]
    src = sorted(set(src))
    out = np.full(cls.shape, -1, dtype=np.int64)
    if not src:
        return out
    pas = passable(cls, src, unknown)
    n = cls.size
    idx = np.arange(n).reshape(cls.shape)
    rows, cols, ws = [], [], []
    for d in OFFSETS:
        ok = allowed_moves(pas, d)
        a = idx[ok]
        rows.append(a)
        cols.append(_shift(idx, d, -1)[ok])
        ws.append(np.full(a.size, float(weight(d))))
    g = coo_matrix((np.concatenate(ws), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n)).tocsr()
    s_idx = [idx[z, y, x] for x, y, z in src]
    dist = dijkstra(g, indices=s_idx, min_only=True, limit=float(K) + 0.5)
    fin = np.isfinite(dist) & (dist <= K)
    out.reshape(-1)[fin] = np.rint(dist[fin]).astype(np.int64)
    return out


def path(cost, cls, sources, cell, unknown=False, max_steps=None):
    """rule 7 from the box-relative goal cell: the cells goal first, or -1 when it is unreachable"""
    pas = passable(cls, sources, unknown)
    shape = cost.shape
    x, y, z = cell
    if cost[z, y, x] < 0:
        return -1
    out = [(x, y, z)]
    while cost[z, y, x] > 0:
        for d in OFFSETS:
            p = (x + d[0], y + d[1], z + d[2])
            if not all(0 <= p[k] < shape[2 - k] for k in range(3)) or cost[p[2], p[1], p[0]] < 0:
                continue
            if not _move_ok(pas, p, (-d[0], -d[1], -d[2])):
                continue
            if cost[p[2], p[1], p[0]] + weight(d) == cost[z, y, x]:
                x, y, z = p
                out.append(p)
                break
        else:
            raise AssertionError(("no predecessor", (x, y, z)))
    return out


def _move_ok(pas, a, d):
    for sel in itertools.product(*[(0, v) if v else (0,) for v in d]):
        q = (a[0] + sel[0], a[1] + sel[1], a[2] + sel[2])
        if not all(0 <= q[k] < pas.shape[2 - k] for k in range(3)) or not pas[q[2], q[1], q[0]]:
            return False
    return True


def check_path(cells, cost, cls, sources, unknown=False):
    """every step is an allowed move whose weight is exactly the drop in cost, the path ends at a source, and every step
    takes the first offset in the spec's order that qualifies"""
    pas = passable(cls, sources, unknown)
    src = {tuple(int(v) for v in s) for s in sources}
    cells = [tuple(int(v) for v in c) for c in cells]
    assert cost[cells[0][2], cells[0][1], cells[0][0]] >= 0
    for a, b in zip(cells, cells[1:]):
        d = (b[0] - a[0], b[1] - a[1], b[2] - a[2])
        assert d in OFFSETS and _move_ok(pas, b, (-d[0], -d[1], -d[2])), (a, b)
        assert cost[b[2], b[1], b[0]] + weight(d) == cost[a[2], a[1], a[0]], (a, b)
        for e in OFFSETS[:OFFSETS.index(d)]:
            p = (a[0] + e[0], a[1] + e[1], a[2] + e[2])
            if all(0 <= p[k] < cost.shape[2 - k] for k in range(3)) and cost[p[2], p[1], p[0]] >= 0:
                assert not (_move_ok(pas, p, (-e[0], -e[1], -e[2])) and
                            cost[p[2], p[1], p[0]] + weight(e) == cost[a[2], a[1], a[0]]), ("earlier offset", a, e)
    last = cells[-1]
    assert cost[last[2], last[1], last[0]] == 0 and last in src
    assert len(cells) <= cost[cells[0][2], cells[0][1], cells[0][0]] // 1000 + 1


def budget(max_dist, d):
    """rule 5's K"""
    return int(np.floor((max_dist / d) * 1000.0))


def box_classes(exported, subbox_n, d, box_min, box_max, inflated=False):
    """rules 1-2 over an exported map: (lo, dims, classes[N_z, N_y, N_x])"""
    n = subbox_n
    lo, dims = box_of(box_min, box_max, d)
    hi = lo + dims - 1
    cls = np.full((dims[2], dims[1], dims[0]), UNKNOWN, dtype=np.int8)
    rows = {tuple(int(v) for v in g): i for i, g in enumerate(exported["glb"])}
    g0, g1 = np.floor_divide(lo, n), np.floor_divide(hi, n)
    for gz in range(g0[2], g1[2] + 1):
        for gy in range(g0[1], g1[1] + 1):
            for gx in range(g0[0], g1[0] + 1):
                i = rows.get((gx, gy, gz))
                if i is None:
                    continue
                g = np.array([gx, gy, gz])
                a, b = np.maximum(lo, g * n), np.minimum(hi, g * n + n - 1)
                dst = tuple(slice(a[k] - lo[k], b[k] - lo[k] + 1) for k in (2, 1, 0))
                if exported["collapsed"][i]:
                    s = exported["occupancy"][i, 0]
                    cls[dst] = BLOCKING if s == b"o" else (FREE if s == b"f" else UNKNOWN)
                    continue
                src = tuple(slice(a[k] - g[k] * n, b[k] - g[k] * n + 1) for k in (2, 1, 0))
                occ = exported["occupancy"][i].reshape(n, n, n)[src]
                blk = occ == b"o"
                if inflated:
                    blk = blk | (exported["inflate"][i].reshape(n, n, n)[src] == b"o")
                cls[dst] = np.where(blk, BLOCKING, np.where(occ == b"f", FREE, UNKNOWN))
    return lo, dims, cls


def source_cells(starts, lo, dims, d):
    """rule 3: the distinct box-relative source cells of world points"""
    valid, c = cells_of(np.asarray(starts, dtype=np.float64).reshape(-1, 3), d)
    ok = valid.all(1) & ((c >= lo) & (c - lo < dims)).all(1)
    return sorted({tuple(int(v) for v in r) for r in (c[ok] - lo)})


def cost_query(field_, lo, d, pos):
    """rule 6"""
    pos = np.asarray(pos, dtype=np.float64).reshape(-1, 3)
    dims = np.array(field_.shape[::-1])
    valid, c = cells_of(pos, d)
    inside = (valid & (c >= lo) & (c - lo < dims)).all(1)
    r = np.where(inside[:, None], c - lo, 0)
    v = field_[r[:, 2], r[:, 1], r[:, 0]]
    with np.errstate(invalid="ignore"):
        out = np.where(v < 0, np.inf, (v.astype(np.float64) / 1000.0) * d)
    return np.where(inside, out, np.nan)
