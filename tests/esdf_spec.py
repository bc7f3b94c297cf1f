"""The signed distance field (mlm_esdf_*) restated in plain numpy from the spec in include/mlmap_b200.h, and the query
point sets the ESDF tests share.  Squared distances come from brute force on small boxes and from
scipy.ndimage.distance_transform_edt on larger ones (its distances are square roots of exact integer sums, so
round(d ** 2) gives them back).  numpy float64 never fuses a multiply with an add, so rule 5 evaluated here in the stated
order gives the CUDA kernel's and the C++ oracle's results bit for bit."""
import numpy as np
from scipy import ndimage

LIMIT = 2.0 ** 30


def cells_of(p, d):
    """(valid, cell) of each coordinate: rule 1 of the ray spec, (int)floor(p / d) unless non-finite or |p / d| >= 2^30"""
    q = np.asarray(p, dtype=np.float64) / d
    valid = np.abs(q) < LIMIT
    return valid, np.floor(np.where(valid, q, 0.0)).astype(np.int64)


def box_of(box_min, box_max, d):
    """(lo[3], dims[3]) of rule 1"""
    v0, lo = cells_of(box_min, d)
    v1, hi = cells_of(box_max, d)
    assert v0.all() and v1.all()
    return lo, hi - lo + 1


def box_blocking(exported, subbox_n, d, box_min, box_max, inflated=False):
    """rule 2 over an exported map (MLMap.export_map / Oracle.export_map): (lo, dims, blocking[N_z, N_y, N_x])"""
    n = subbox_n
    lo, dims = box_of(box_min, box_max, d)
    hi = lo + dims - 1
    blk = np.zeros((dims[2], dims[1], dims[0]), dtype=bool)
    rows = {tuple(int(v) for v in g): i for i, g in enumerate(exported["glb"])}
    g0, g1 = np.floor_divide(lo, n), np.floor_divide(hi, n)
    for gz in range(g0[2], g1[2] + 1):
        for gy in range(g0[1], g1[1] + 1):
            for gx in range(g0[0], g1[0] + 1):
                i = rows.get((gx, gy, gz))
                if i is None:
                    continue                                    # absent: unknown, not blocking
                g = np.array([gx, gy, gz])
                a, b = np.maximum(lo, g * n), np.minimum(hi, g * n + n - 1)
                dst = tuple(slice(a[k] - lo[k], b[k] - lo[k] + 1) for k in (2, 1, 0))
                if exported["collapsed"][i]:
                    blk[dst] = exported["occupancy"][i, 0] == b"o"   # element 0; never blocks by inflation
                    continue
                src = tuple(slice(a[k] - g[k] * n, b[k] - g[k] * n + 1) for k in (2, 1, 0))
                occ = exported["occupancy"][i].reshape(n, n, n)[src] == b"o"
                if inflated:
                    occ = occ | (exported["inflate"][i].reshape(n, n, n)[src] == b"o")
                blk[dst] = occ
    return lo, dims, blk


def brute_force(blk):
    """(D+, D-) by comparing every pair of cells; -1 for an empty set"""
    zz, yy, xx = np.nonzero(np.ones_like(blk))
    c = np.stack([xx, yy, zz], 1).astype(np.int64)
    flat = blk.reshape(-1)
    out = []
    for sel in (flat, ~flat):
        if not sel.any():
            out.append(np.full(blk.shape, -1, dtype=np.int64))
            continue
        t = c[sel]
        d2 = ((c[:, None, :] - t[None, :, :]) ** 2).sum(-1)
        out.append(d2.min(1).reshape(blk.shape))
    return out[0], out[1]


def scipy_squared(blk):
    """(D+, D-) from scipy's exact Euclidean transform; -1 for an empty set"""
    out = []
    for target in (blk, ~blk):
        if not target.any():
            out.append(np.full(blk.shape, -1, dtype=np.int64))
            continue
        dist = ndimage.distance_transform_edt(~target)   # distance of every cell to the nearest target cell
        out.append(np.rint(dist * dist).astype(np.int64))
    return out[0], out[1]


def cell_values(blk, dplus, dminus, d, max_dist):
    """rule 4 (an empty set, -1 here, counts as beyond max_dist)"""
    def clamped(d2):
        r = np.sqrt(np.where(d2 < 0, 0, d2).astype(np.float64)) * d
        return np.where(d2 < 0, max_dist, np.minimum(r, max_dist))
    return np.where(blk, d - clamped(dminus), clamped(dplus))


def query(val, lo, d, pos):
    """rule 5 over the values val[N_z, N_y, N_x] of the box starting at lo: (dist[n], grad[n, 3])"""
    pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 3)
    dims = np.array([val.shape[2], val.shape[1], val.shape[0]])
    valid, c = cells_of(pos, d)
    inside = (valid & (c >= lo) & (c - lo < dims)).all(1)
    with np.errstate(invalid="ignore"):
        q = pos / d - 0.5
    i = np.floor(np.where(inside[:, None], q, 0.0)).astype(np.int64)
    w = q - i.astype(np.float64)
    u = 1.0 - w
    i0 = np.clip(i - lo, 0, dims - 1)
    i1 = np.clip(i - lo + 1, 0, dims - 1)
    ii = (i0, i1)

    def v(x, y, z):
        return val[ii[z][:, 2], ii[y][:, 1], ii[x][:, 0]]
    with np.errstate(invalid="ignore"):
        e = {(y, z): v(0, y, z) * u[:, 0] + v(1, y, z) * w[:, 0] for y in (0, 1) for z in (0, 1)}
        f0 = e[0, 0] * u[:, 1] + e[1, 0] * w[:, 1]
        f1 = e[0, 1] * u[:, 1] + e[1, 1] * w[:, 1]
        dist = f0 * u[:, 2] + f1 * w[:, 2]
        g = {(y, z): v(1, y, z) - v(0, y, z) for y in (0, 1) for z in (0, 1)}
        gx = ((((g[0, 0] * u[:, 1]) * u[:, 2] + (g[0, 1] * u[:, 1]) * w[:, 2]) + (g[1, 0] * w[:, 1]) * u[:, 2])
              + (g[1, 1] * w[:, 1]) * w[:, 2]) / d
        gy = ((e[1, 0] - e[0, 0]) * u[:, 2] + (e[1, 1] - e[0, 1]) * w[:, 2]) / d
        gz = (f1 - f0) / d
    grad = np.stack([gx, gy, gz], 1)
    dist = np.where(inside, dist, np.nan)
    grad = np.where(inside[:, None], grad, 0.0)
    return dist, grad


def query_points(lo, dims, d, n_random, seed):
    """random points inside and around the box (a cell beyond each face), points on cell centres and on the box faces,
    each also nudged by one ulp either way, and non-finite / out-of-range points"""
    rs = np.random.RandomState(seed)
    lo_w, hi_w = lo * d, (lo + dims) * d
    pad = 2.0 * d
    P = [rs.uniform(lo_w - pad, hi_w + pad, (n_random, 3))]
    k = max(n_random // 8, 16)
    c = rs.randint(lo, lo + dims, (k, 3)).astype(np.float64)
    centres = (c + 0.5) * d
    faces = rs.uniform(lo_w, hi_w, (k, 3))
    ax = rs.randint(0, 3, k)
    side = rs.randint(0, 2, k)
    faces[np.arange(k), ax] = np.where(side == 1, hi_w[ax], lo_w[ax])
    half = rs.uniform(lo_w, hi_w, (k, 3))                       # in the outer half cell of a face
    half[np.arange(k), ax] = np.where(side == 1, hi_w[ax] - rs.uniform(0, 0.5, k) * d, lo_w[ax] + rs.uniform(0, 0.5, k) * d)
    for base in (centres, faces):
        P += [base, np.nextafter(base, np.inf), np.nextafter(base, -np.inf)]
    P.append(half)
    nan, inf = float("nan"), float("inf")
    P.append(np.array([[nan, 0, 0], [0, inf, 0], [0, 0, -inf], [LIMIT * d, 0, 0], [0, -LIMIT * d, 0]]))
    return np.ascontiguousarray(np.concatenate(P))


def same_bits(a, b):
    """equal bit for bit (NaN only equal to the same NaN)"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def first_difference(a, b):
    """(flat index, a, b, count) of the first bit difference, or None"""
    a, b = np.ascontiguousarray(a).reshape(-1), np.ascontiguousarray(b).reshape(-1)
    ia = a.view(np.uint64 if a.itemsize == 8 else np.uint32)
    ib = b.view(np.uint64 if b.itemsize == 8 else np.uint32)
    diff = np.nonzero(ia != ib)[0]
    return None if diff.size == 0 else (int(diff[0]), a[diff[0]], b[diff[0]], int(diff.size))
