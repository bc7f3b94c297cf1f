"""getOdd and getOddGrad of the reference (include/mlmap.h:40, 213-295) restated in plain Python over crafted log-odds
maps, apart from both the C++ oracle and the kernels; a decoder that tells which of the 6 * max_iter candidate cells a
returned pseudo-gradient points at; and the host scan of the float log-odds domain that the kernels' shortcuts rest on.
The odd goes through math.pow, which is glibc's pow like the reference's (numpy's vectorised power is not: it may
differ from glibc in the last bit).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import math
import time

import numpy as np

# subbox_neighbors row order (src/map_local.cpp:78-120): +z, -z, +y, -y, +x, -x as (axis, step)
DIRS = ((2, 1), (2, -1), (1, 1), (1, -1), (0, 1), (0, -1))
K_TIE = np.float32(1e-2)      # k_get_odd_grad's near-tie window in log-odds
K_NEAR_ONE = np.float32(5.5)  # above it k_get_odd_grad checks every earlier direction
GLB_LIMIT = 1 << 20           # subbox indices live in [-2^20, 2^20)


def unit(d) -> np.ndarray:
    """the cell step of probe direction d"""
    e = np.zeros(3, np.int64)
    e[DIRS[d][0]] = DIRS[d][1]
    return e


def odd(lo) -> np.float32:
    """logit_inv (mlmap.h:40): pow(10, x) / (1 + pow(10, x)) in double, returned as float (NaN once 10^x overflows)"""
    try:
        y = math.pow(10.0, float(lo))
    except OverflowError:
        y = math.inf
    return np.float32(y / (1.0 + y)) if y != math.inf else np.float32(math.nan)


def odds(lo) -> np.ndarray:
    return np.array([odd(v) for v in np.asarray(lo, np.float32).ravel()], np.float32).reshape(np.shape(lo))


def same_floats(a, b) -> bool:
    """bit for bit, except that any two NaNs agree (their payloads are the platform's)"""
    a, b = np.asarray(a), np.asarray(b)
    u = a.view(np.uint32 if a.dtype == np.float32 else np.uint64)
    v = b.view(np.uint32 if b.dtype == np.float32 else np.uint64)
    return a.shape == b.shape and bool(((u == v) | (np.isnan(a) & np.isnan(b))).all())


class LogOddsMap:
    """subboxes {glb: float32 log-odds per cell}, and collapsed subboxes {glb: float32 element 0}; cells of subboxes
    that set() allocates hold `background`"""

    def __init__(self, n: int, d_sub: float, background=0.0):
        self.n, self.d_sub, self.background = n, d_sub, np.float32(background)
        self.d_glb = d_sub * n              # map_local.cpp: map_dxyz_obv_sub * subbox_nxyz
        self.d_half = d_sub * 0.5
        self.full: dict[tuple, np.ndarray] = {}
        self.collapsed: dict[tuple, np.float32] = {}

    # ---- building -----------------------------------------------------------------------------------------------
    def split(self, cell):
        g = tuple(int(c) // self.n for c in cell)
        loc = [int(cell[a]) - g[a] * self.n for a in range(3)]
        return g, (loc[2] * self.n + loc[1]) * self.n + loc[0]

    def fill(self, g, value):
        g = tuple(int(v) for v in g)
        self.collapsed.pop(g, None)
        self.full[g] = np.full(self.n ** 3, value, np.float32)

    def collapse(self, g, value):
        g = tuple(int(v) for v in g)
        self.full.pop(g, None)
        self.collapsed[g] = np.float32(value)

    def set(self, cell, value):
        """the log-odds of a cell of a full subbox (allocated with the background if absent)"""
        g, sub = self.split(cell)
        assert g not in self.collapsed, g
        if g not in self.full:
            self.fill(g, self.background)
        self.full[g][sub] = np.float32(value)

    @classmethod
    def from_export(cls, ex, n, d_sub):
        m = cls(n, d_sub)
        for g, c, lo in zip(map(tuple, ex["glb"].tolist()), ex["collapsed"], ex["log_odds"]):
            if c:
                m.collapse(g, lo[0])
            else:
                m.full[g] = np.asarray(lo, np.float32).copy()
        return m

    def export(self) -> dict:
        """an export_map-like dict (glb, collapsed, occupancy, inflate, frontier, log_odds), subboxes sorted"""
        keys = sorted(list(self.full) + list(self.collapsed))
        m, cells = len(keys), self.n ** 3
        lo = np.zeros((m, cells), np.float32)
        col = np.zeros(m, np.uint8)
        for i, g in enumerate(keys):
            if g in self.full:
                lo[i] = self.full[g]
            else:
                col[i], lo[i, 0] = 1, self.collapsed[g]
        occ = np.full((m, cells), b"u", dtype="S1")
        return {"glb": np.array(keys, np.int32).reshape(-1, 3), "collapsed": col, "occupancy": occ,
                "inflate": occ.copy(), "frontier": np.zeros((m, (cells + 7) // 8), np.uint8), "log_odds": lo}

    # ---- the reference's reads ----------------------------------------------------------------------------------
    def lo_at(self, g, sub):
        """(stored, log-odds) of cell sub of subbox g: log_odds[0] of a collapsed subbox, nothing for an absent one"""
        if g in self.full:
            return True, self.full[g][sub]
        if g in self.collapsed:
            return True, self.collapsed[g]
        return False, np.float32(0.0)

    def odd_at(self, g, sub) -> np.float32:
        """getOdd(glb, sub) (mlmap.h:227-235): 0.5 for an absent subbox"""
        stored, lo = self.lo_at(tuple(g), sub)
        return odd(lo) if stored else np.float32(0.5)

    def locate(self, p):
        """get_global_idx (map_local.h:148-173): the subbox by floor(p / d_glb), the cell by floor(p / d_sub) - g * n;
        a cell index outside the subbox is a missing key of subbox_cell_id_table, which answers 0"""
        g = tuple(math.floor(float(p[a]) / self.d_glb) for a in range(3))
        loc = [math.floor(float(p[a]) / self.d_sub) - g[a] * self.n for a in range(3)]
        if not all(0 <= v < self.n for v in loc):
            return g, 0
        return g, (loc[2] * self.n + loc[1]) * self.n + loc[0]

    def get_odd(self, p) -> np.float32:
        return self.odd_at(*self.locate(p))

    def step(self, g, sub, d):
        """subbox_neighbors row d of cell sub: one cell along DIRS[d], into the next subbox at a border"""
        n = self.n
        c = [sub % n, (sub // n) % n, sub // (n * n)]
        g = list(g)
        axis, s = DIRS[d]
        c[axis] += s
        if c[axis] >= n:
            g[axis], c[axis] = g[axis] + 1, 0
        elif c[axis] < 0:
            g[axis], c[axis] = g[axis] - 1, n - 1
        return tuple(g), (c[2] * n + c[1]) * n + c[0]

    def centre(self, g, sub):
        """subbox_id2xyz_glb_vec (map_local.h:208-213)"""
        n = self.n
        c = (sub % n, (sub // n) % n, sub // (n * n))
        return tuple(float(g[a]) * self.d_glb + float(c[a]) * self.d_sub + self.d_half for a in range(3))

    def grad(self, p, max_iter=5):
        """getOddGrad (mlmap.h:237-295): the six probes step along DIRS; within a round each probe whose odd is strictly
        below the running minimum (which starts at the origin's odd) becomes the winner; a round with a winner ends the
        search.  Returns (vector, winner or None, rounds): winner = (round k from 1, direction, glb, sub); rounds = the
        float odds of every round visited, [ori_odd] first"""
        g0, sub0 = self.locate(p)
        ori = mn = self.odd_at(g0, sub0)
        pos = [(g0, sub0)] * 6
        win, rounds = None, [[ori]]
        for k in range(1, max_iter + 1):
            row = []
            for d in range(6):
                pos[d] = self.step(*pos[d], d)
                t = self.odd_at(*pos[d])
                row.append(t)
                if t < mn:
                    mn, win = t, (k, d) + pos[d]
            rounds.append(row)
            if win:
                break
        if not win:
            return (0.0, 0.0, 0.0), None, rounds
        s = float(np.float32(ori - mn))   # float - float, then Vec3 * float in double
        c = self.centre(win[2], win[3])
        return tuple((c[a] - float(p[a])) * s for a in range(3)), win, rounds

    def round_lo(self, p, k):
        """the six log-odds of round k (0.0 where the subbox is absent)"""
        g, sub = self.locate(p)
        out = []
        for d in range(6):
            q = (g, sub)
            for _ in range(k):
                q = self.step(*q, d)
            out.append(self.lo_at(*q)[1])
        return np.array(out, np.float32)


def decode(m: LogOddsMap, p, vec, max_iter):
    """(round, direction) of the candidate cell a returned getOddGrad vector points at, None for the zero vector: the
    one candidate c with (centre(c) - p) * s == vec bit for bit for a positive float s.  Fails when no candidate or
    more than one fits (a query point on a cell centre makes the candidates of one axis parallel)"""
    vec = tuple(float(v) for v in vec)
    if vec == (0.0, 0.0, 0.0):
        return None
    g, sub = m.locate(p)
    hits = []
    for d in range(6):
        q = (g, sub)
        for k in range(1, max_iter + 1):
            q = m.step(*q, d)
            c = m.centre(*q)
            diff = [c[a] - float(p[a]) for a in range(3)]
            a = int(np.argmax(np.abs(diff)))
            s = float(np.float32(vec[a] / diff[a]))
            if s > 0 and all(diff[b] * s == vec[b] for b in range(3)):
                hits.append((k, d))
    assert len(hits) == 1, ("ambiguous or foreign gradient", p, vec, hits)
    return hits[0]


def kernel_rule_before_fix(lo0, lo_d):
    """the winner k_get_odd_grad chose in one round before the near-one check (kTie and lo_m < -30 only): the first
    lowest log-odds, or an earlier direction within kTie with the same float odd; -1 when no odd is strictly lower"""
    lo_d = np.asarray(lo_d, np.float32)
    m = int(np.argmin(lo_d))
    lo_m = lo_d[m]
    if not (lo_m < lo0 and odd(lo_m) < odd(lo0)):
        return -1
    for d in range(m):
        if (lo_d[d] - lo_m <= K_TIE or lo_m < np.float32(-30.0)) and lo_d[d] < lo0 and odd(lo_d[d]) == odd(lo_m):
            return d
    return m


def reference_rule(lo0, lo_d):
    """the reference's winner in one round: the first direction with the lowest float odd below the origin's, or -1"""
    o = odds(lo_d)
    m = int(np.argmin(o))
    return m if o[m] < odd(lo0) else -1


def _key(f):
    """an integer that orders floats like their values (-0.0 just below +0.0)"""
    b = int(np.float32(f).view(np.int32))
    return b if b >= 0 else -(b & 0x7FFFFFFF) - 1


def _from_key(k):
    return np.int32(k if k >= 0 else (-(k + 1)) | -0x80000000).view(np.float32)


def run_of(x):
    """(lowest, highest) float log-odds whose float odd equals x's: odd is monotone, so a binary search on the bits"""
    o, k = odd(x), _key(x)

    def edge(step):
        lo, hi = 0, 1
        while odd(_from_key(k + step * hi)) == o:
            lo, hi = hi, hi * 2
        while hi - lo > 1:
            mid = (lo + hi) // 2
            lo, hi = (mid, hi) if odd(_from_key(k + step * mid)) == o else (lo, mid)
        return _from_key(k + step * lo)

    return edge(-1), edge(1)


# ---- the float log-odds domain ------------------------------------------------------------------------------------
def _binade(e, sign):
    """the floats of sign * [2^e, 2^(e+1)), in ascending order"""
    a, b = np.float32(2.0 ** e).view(np.int32), np.float32(2.0 ** (e + 1)).view(np.int32)
    bits = np.arange(a, b, dtype=np.int32)
    return (bits.view(np.float32) if sign > 0 else -bits[::-1].view(np.float32))


def _odd_of(y):
    with np.errstate(over="ignore", invalid="ignore"):
        return (y / (1.0 + y)).astype(np.float32)


def scan_log_odds(lo_exp=-28, hi_exp=6, tie_from=-30.0):
    """Every float log-odds x with 2^lo_exp <= |x| <= 2^hi_exp, in ascending order, in chunks of one binade.

    (1) Stability of the float odd under an error of 10^x: the odd is computed from y = 10^x and from the doubles up
    to two ulps to either side.  numpy's power is within one ulp of the correctly rounded 10^x, so the window holds
    both doubles next to the exact value, which are the only results a 1-ulp exp10 or glibc's pow can return.  Values
    whose odd changes inside the window are checked again on those two doubles exactly (long-double pow); the ones that
    still differ are returned in `flips`.

    (2) The premise of k_get_odd_grad's near-tie window: among ascending x >= tie_from, the first x whose run of equal
    float odds reaches more than kTie above it (the float difference, as the kernel computes it).  Below that value a
    log-odds with the same odd as the round's minimum is within kTie of it.

    Returns {"count", "flips", "tie_threshold", "seconds"}."""
    t0 = time.perf_counter()
    chunks = [(e, -1) for e in range(hi_exp - 1, lo_exp - 1, -1)] + [(e, 1) for e in range(lo_exp, hi_exp)]
    count, flips = 0, []
    run_start, run_odd, threshold = None, None, None

    def runs(lo, r):
        nonlocal run_start, run_odd, threshold
        keep = lo >= np.float32(tie_from)
        lo, r = lo[keep], r[keep]
        if lo.size == 0 or threshold is not None:
            return
        new = np.ones(lo.size, bool)
        new[1:] = r[1:] != r[:-1]
        new[0] = run_odd is None or r[0] != run_odd
        starts = np.flatnonzero(new)
        first = np.where(new, np.arange(lo.size), 0)
        first = np.maximum.accumulate(first)
        start_lo = lo[first]
        if not new[0]:   # the open run of the previous chunk goes on
            start_lo[:starts[0] if starts.size else lo.size] = run_start
        wide = np.flatnonzero(lo - start_lo > K_TIE)
        if wide.size:
            threshold = start_lo[wide[0]]
            return
        run_start, run_odd = start_lo[-1], r[-1]

    for i, (e, sign) in enumerate(chunks):
        lo = _binade(e, sign)
        if e == hi_exp - 1 and sign > 0:
            lo = np.append(lo, np.float32(2.0 ** hi_exp))
        if e == hi_exp - 1 and sign < 0:
            lo = np.insert(lo, 0, np.float32(-(2.0 ** hi_exp)))
        count += lo.size
        x = lo.astype(np.float64)
        y = np.power(10.0, x)
        r = _odd_of(y)
        bad = np.zeros(lo.size, bool)
        up = dn = y
        for _ in range(2):
            up, dn = np.nextafter(up, np.inf), np.nextafter(dn, -np.inf)
            bad |= (_odd_of(up) != r) | (_odd_of(dn) != r)
        for v in lo[bad]:
            t = np.power(np.longdouble(10), np.longdouble(float(v)))
            a = np.float64(t)
            b = np.nextafter(a, np.inf) if np.longdouble(a) < t else (np.nextafter(a, -np.inf) if np.longdouble(a) > t else a)
            if _odd_of(np.array([a]))[0] != _odd_of(np.array([b]))[0]:
                flips.append(np.float32(v))
            else:
                r[lo == v] = _odd_of(np.array([a]))[0]
        runs(lo, r)
        if sign < 0 and e == lo_exp:
            # |x| < 2^lo_exp: the odd is 0.5 (10^x - 1 is below 2^-26.6, a quarter of which is under half an ulp of 0.5)
            runs(np.array([0.0], np.float32), np.array([0.5], np.float32))
    return {"count": count, "flips": flips, "tie_threshold": threshold, "seconds": time.perf_counter() - t0}
