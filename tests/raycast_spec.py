"""Ray casting (mlm_cast_rays) restated in plain Python from the spec in include/mlmap_b200.h, and the segment sets the
ray tests share.  Python floats are IEEE doubles and Python never fuses a multiply with an add, so this walk gives the
same records as the CUDA kernel and the C++ oracle bit for bit."""
import math

import numpy as np

from mlmapping_b200.capi import RAY_HIT_DTYPE, RAY_INVALID

FREE, OCCUPIED = 1, 0


def cell_of(p, d):
    """(int)floor(p / d), or None for a non-finite p or |p / d| >= 2^30"""
    q = p / d
    if not abs(q) < 2.0 ** 30:
        return None
    return int(math.floor(q))


class MapStates:
    """cell states of an exported map (MLMap.export_map / Oracle.export_map), looked up the way getOccupancy /
    getInflateOccupancy answer"""

    def __init__(self, exported, subbox_n):
        self.n = subbox_n
        self.row = {tuple(int(v) for v in g): i for i, g in enumerate(exported["glb"])}
        self.collapsed = exported["collapsed"]
        self.occ = exported["occupancy"]
        self.inf = exported["inflate"]

    def __call__(self, c):
        """(state byte, inflation byte) of global cell c; b'u' for an absent subbox, and a collapsed subbox's element 0
        with no inflation"""
        n = self.n
        g = (c[0] // n, c[1] // n, c[2] // n)
        i = self.row.get(g)
        if i is None:
            return b"u", b"u"
        if self.collapsed[i]:
            return self.occ[i, 0], b"u"
        sub = ((c[2] - g[2] * n) * n + (c[1] - g[1] * n)) * n + (c[0] - g[0] * n)
        return self.occ[i, sub], self.inf[i, sub]


def walk(f, t, d, states, inflated=False):
    """one segment: (status, stop cell, n_free, n_unknown, t, visited cells)"""
    c = [cell_of(v, d) for v in f]
    e = [cell_of(v, d) for v in t]
    if None in c or None in e:
        return RAY_INVALID, (0, 0, 0), 0, 0, 0.0, []
    rem = [abs(e[k] - c[k]) for k in range(3)]
    if sum(rem) > 2 ** 20:
        return RAY_INVALID, (0, 0, 0), 0, 0, 0.0, []
    s = [(e[k] > c[k]) - (e[k] < c[k]) for k in range(3)]
    inv = [1.0 / (t[k] - f[k]) if rem[k] > 0 else 0.0 for k in range(3)]
    t_enter, n_free, n_unknown, path = 0.0, 0, 0, []
    while True:
        path.append(tuple(c))
        st, inf = states(c)
        if st == b"o" or (inflated and inf == b"o"):
            status = OCCUPIED
            break
        if st == b"f":
            n_free += 1
        else:
            n_unknown += 1
        if sum(rem) == 0:
            status = FREE
            break
        ax, tb = -1, 0.0
        for k in range(3):
            if rem[k] == 0:
                continue
            tk = (float(c[k] + (1 if s[k] > 0 else 0)) * d - f[k]) * inv[k]
            if ax < 0 or tk < tb:
                ax, tb = k, tk
        c[ax] += s[ax]
        rem[ax] -= 1
        t_enter = tb
    t_out = min(t_enter, 1.0) if t_enter > 0.0 else 0.0
    return status, tuple(c), n_free, n_unknown, t_out, path


def cast_rays(from_, to, d, states, inflated=False):
    """records of walk() for every segment as a RAY_HIT_DTYPE array, and the visited cells of each"""
    out = np.zeros(len(from_), dtype=RAY_HIT_DTYPE)
    paths = []
    for i, (f, t) in enumerate(zip(from_.tolist(), to.tolist())):
        st, cell, nf, nu, tt, path = walk(f, t, d, states, inflated)
        out[i] = (st, cell, nf, nu, tt)
        paths.append(path)
    return out, paths


def random_segments(n, lo, hi, seed, max_len, inflate=1.0):
    """starts from scenes.query_positions, uniformly random directions, lengths uniform in [0, max_len)"""
    from mlmapping_b200 import scenes
    a = scenes.query_positions(n, lo, hi, seed=seed, inflate=inflate)
    rs = np.random.RandomState(seed + 1)
    v = rs.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    return a, a + v * rs.uniform(0.0, max_len, (n, 1))


def edge_segments(exported, subbox_n, d, seed, n_each=100):
    """the edge cases of the spec: from == to, axis-parallel segments, endpoints on cell borders and lattice points
    (k*d and k*d +- 1 ulp), negative coordinates, segments longer than a subbox, starts inside occupied cells, segments
    entirely in unknown space, non-finite endpoints and over-long segments (INVALID)"""
    rs = np.random.RandomState(seed)
    glb = exported["glb"]
    lo, hi = glb.min(0) * subbox_n * d, (glb.max(0) + 1) * subbox_n * d
    F, T = [], []

    def add(a, b):
        F.append(np.asarray(a, dtype=np.float64).reshape(-1, 3))
        T.append(np.asarray(b, dtype=np.float64).reshape(-1, 3))

    p = rs.uniform(lo, hi, (n_each, 3))
    add(p, p)                                                   # from == to
    for k in range(3):                                          # axis-parallel, both directions
        p = rs.uniform(lo, hi, (n_each, 3))
        q = p.copy()
        q[:, k] += rs.uniform(-4.0, 4.0, n_each)
        add(p, q)
    # lattice points and cell borders: k*d, nudged by one ulp up or down per coordinate
    kk = rs.randint(np.floor(lo / d).astype(np.int64), np.ceil(hi / d).astype(np.int64), (4 * n_each, 3)).astype(np.float64) * d
    nudge = rs.randint(-1, 2, kk.shape)
    kk = np.where(nudge > 0, np.nextafter(kk, np.inf), np.where(nudge < 0, np.nextafter(kk, -np.inf), kk))
    add(kk[0::2], kk[1::2])
    p = rs.uniform(lo, hi, (n_each, 3))                         # one endpoint on a lattice point, the other inside
    add(np.floor(p / d) * d, rs.uniform(lo, hi, (n_each, 3)))
    p = -rs.uniform(0.01, 3.0, (n_each, 3))                     # negative coordinates
    add(p, p + rs.uniform(-2.0, 2.0, (n_each, 3)))
    p = rs.uniform(lo, hi, (n_each, 3))                         # longer than a subbox
    v = rs.normal(size=(n_each, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    add(p, p + v * rs.uniform(1.5 * subbox_n * d, 8.0, (n_each, 1)))
    occ_rows, occ_cells = np.nonzero((exported["occupancy"] == b"o") & (exported["collapsed"][:, None] == 0))
    if occ_rows.size:                                           # starts inside occupied cells
        pick = rs.randint(0, occ_rows.size, n_each)
        sub = occ_cells[pick]
        loc = np.stack([sub % subbox_n, (sub // subbox_n) % subbox_n, sub // (subbox_n * subbox_n)], 1)
        p = (glb[occ_rows[pick]] * subbox_n + loc + rs.uniform(0.05, 0.95, (n_each, 3))) * d
        add(p, p + rs.uniform(-1.0, 1.0, (n_each, 3)))
    p = rs.uniform(-40.0, -30.0, (n_each, 3))                   # entirely in unknown space
    add(p, p + rs.uniform(-3.0, 3.0, (n_each, 3)))
    nan, inf = float("nan"), float("inf")
    big = 2.0 ** 30 * d
    bad = [[nan, 0, 0], [0, inf, 0], [0, 0, -inf], [big, 0, 0], [0, -big, 0], [0, 0, 2 * big]]
    for b in bad:                                               # INVALID: non-finite / out of range, either end
        add([1.0, 0.5, 1.0], b)
        add(b, [1.0, 0.5, 1.0])
    long_ = (2 ** 20 + 1) * d                                   # INVALID: more than 2^20 cells
    add([0.05, 0.05, 0.05], [0.05 + long_, 0.05, 0.05])
    return np.ascontiguousarray(np.concatenate(F)), np.ascontiguousarray(np.concatenate(T))


def records_equal(a, b):
    """every field bit for bit (t compared as its 64-bit pattern)"""
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def first_difference(a, b):
    """(index, record a, record b, number of differing records) of the first mismatch, or None"""
    ra = np.ascontiguousarray(a).view(np.uint8).reshape(len(a), -1)
    rb = np.ascontiguousarray(b).view(np.uint8).reshape(len(b), -1)
    diff = np.nonzero((ra != rb).any(axis=1))[0]
    return None if diff.size == 0 else (int(diff[0]), a[diff[0]], b[diff[0]], int(diff.size))
