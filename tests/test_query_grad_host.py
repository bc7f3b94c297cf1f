"""getOdd and getOddGrad without a device: the Python restatement (grad_spec) equals the oracle bit for bit on crafted
log-odds maps, and each crafted case reaches the edge it is named for; the checkpoint writer's images parse back with
their log-odds; and the scan of every float log-odds behind two shortcuts of the kernels: getOdd's exp10 (its 1-ulp
error never changes the float odd) and k_get_odd_grad's near-tie window (below 5.586 a log-odds with the same float
odd as the round's minimum is within kTie of it; above it the kernel checks every earlier direction)."""
import ctypes as C
from itertools import combinations

import numpy as np
import pytest

from frontier_spec import CkptHeader, fnv1a64, fresh_header, record_bytes
from grad_spec import (GLB_LIMIT, K_NEAR_ONE, K_TIE, LogOddsMap, decode, kernel_rule_before_fix, odd,
                       reference_rule, run_of, same_floats, scan_log_odds, unit)
from test_frontier_host import explore_cfg_a
from view_oracle import ViewOracle
from view_spec import write_map_checkpoint

SIZES = (2, 3, 10, 16)
OFF = np.array([0.37, 0.61, 0.29])   # query points off the cell centres: decode() is unambiguous there
F = np.float32


def cfg_n(n):
    cfg = explore_cfg_a()
    cfg.subbox_n, cfg.pool_submaps = n, 8192
    return cfg


def iters_of(n):
    """walks that cross 0 to 3 subbox borders"""
    return sorted({1, 5, n // 2 + 1, n + 1, 2 * n + 1, 3 * n + 1})


def point(cell, d):
    return (np.asarray(cell, np.float64) + OFF) * d


# ---- crafted cases ------------------------------------------------------------------------------------------------
class Case:
    """a crafted map and its queries (point, max_iter, tag); origins() places isolated origins on a grid whose spacing
    keeps every probe cell of one origin off the probe lines of the others"""

    def __init__(self, n, d, background=0.0):
        self.m = LogOddsMap(n, d, background)
        self.queries = []
        self.n, self.d = n, d

    def origins(self, specs, base=(0, 0, 0), spacing=None):
        """specs: dicts with lo0 (None: leave the origin cell alone), reach K, fill (the log-odds of every probe cell of
        rounds 1..K, None: leave them), cells {(k, d): log-odds}, iters, tag"""
        K = max(s["K"] for s in specs)
        spacing = spacing or 2 * K + 1
        w = int(np.ceil(len(specs) ** (1 / 3) - 1e-9))
        for j, s in enumerate(specs):
            o = np.array(base) + spacing * np.array([j % w, (j // w) % w, j // (w * w)])
            if s.get("fill") is not None:
                for k in range(1, s["K"] + 1):
                    for dd in range(6):
                        self.m.set(o + k * unit(dd), s["fill"])
            if s.get("lo0") is not None:
                self.m.set(o, s["lo0"])
            for (k, dd), v in s.get("cells", {}).items():
                self.m.set(o + k * unit(dd), v)
            for it in s["iters"]:
                self.queries.append((point(o, self.d), it, s.get("tag", "")))
        return self


def near_tie(n, d):
    """near-one ties: round k's lowest log-odds (a run start, 5.586 .. 7.2) in direction b, the highest log-odds with the
    same float odd (up to 0.2 higher) in direction a, the tie in an earlier and in a later direction; origins 5.9 .. 10"""
    specs = []
    for lm in (5.58623, 5.8, 6.3, 6.9, 7.2):
        start, end = run_of(F(lm))
        for a in range(6):
            for b in range(6):
                for k in ((1, 2) if a != b else ()):
                    lo0 = F(min(10.0, float(end) + 0.3 + 0.5 * a))
                    specs.append(dict(lo0=lo0, K=k, fill=lo0, cells={(k, b): start, (k, a): end}, iters=[k],
                                      tag=("earlier" if a < b else "later", float(lm), a, b)))
    return Case(n, d).origins(specs)


def resume(n, d):
    """round 1 holds a lower log-odds with the origin's float odd (not a winner: the search goes on); round 2 holds a
    lower odd, once with a near tie in an earlier direction; or no lower odd at all within reach"""
    specs = []
    for x in (0.3, 2.0, 4.0, 6.5, 7.2):
        start, end = run_of(F(x))
        low_s, low_e = run_of(np.nextafter(start, F(-np.inf)))
        for b in range(6):
            specs.append(dict(lo0=end, K=2, fill=end, cells={(1, b): start, (2, 5 - b): low_s}, iters=[2, 3],
                              tag=("resume", x, b)))
            specs.append(dict(lo0=end, K=2, fill=end, cells={(1, b): start, (2, 5): low_s, (2, b % 5): low_e},
                              iters=[2], tag=("resume-tie", x, b)))
        specs.append(dict(lo0=end, K=3, fill=start, iters=[3], tag=("never", x)))
    return Case(n, d).origins(specs)


def equal(n, d):
    """several directions with the same lowest log-odds (the first one wins); all six equal to the origin (no winner)"""
    specs = [dict(lo0=F(1.0), K=1, fill=F(1.0), cells={(1, dd): F(0.25) for dd in s}, iters=[1, 3], tag=("equal", s))
             for r in range(2, 7) for s in combinations(range(6), r)]
    specs.append(dict(lo0=F(1.0), K=1, fill=F(1.0), iters=[1], tag=("all-equal",)))
    specs.append(dict(lo0=F(-0.0), K=1, fill=F(0.0), iters=[1], tag=("signed-zeros",)))
    return Case(n, d).origins(specs)


def underflow(n, d):
    """log-odds below -30: denormal odds, and odds that underflow to 0 at any gap (the first direction wins)"""
    rs = np.random.RandomState(n)
    pool = F([-30.5, -31.5, -38.5, -41.0, -44.7, -44.9, -44.95, -45.1, -45.2, -46.0, -60.0, -1e4])
    specs = []
    for lo0 in F([-31.0, -40.0, -44.9, -46.0, -50.0]):
        specs.append(dict(lo0=lo0, K=1, cells={(1, 0): F(-45.2), (1, 5): F(-60.0)}, fill=lo0, iters=[1],
                          tag=("zero-odd-tie", float(lo0))))
        specs.append(dict(lo0=lo0, K=1, cells={(1, 1): F(-44.7), (1, 4): F(-45.1)}, fill=lo0, iters=[1],
                          tag=("denormal-tie", float(lo0))))
        for _ in range(6):
            specs.append(dict(lo0=lo0, K=2, fill=lo0, cells={(k, dd): rs.choice(pool) for k in (1, 2) for dd in range(6)},
                              iters=[1, 2], tag=("random", float(lo0))))
    return Case(n, d).origins(specs)


def zeros_and_absent(n, d):
    """log-odds +-0.0 (odd 0.5) next to absent subboxes (0.5 too): no winner there; a tiny negative log-odds whose odd is
    still 0.5; -2^-20 just below; an origin in an absent subbox with a lower cell across the border"""
    specs = []
    for lo0 in (F(0.0), F(-0.0)):
        for dd in range(6):
            specs.append(dict(lo0=lo0, K=1, iters=[1, n + 1], tag=("zero-border", dd)))
            specs.append(dict(lo0=lo0, K=3, cells={(1, dd): F(-1e-30), (2, dd): -lo0, (3, 5 - dd): F(-2.0 ** -20)},
                              iters=[3], tag=("zero-tiny", dd)))
            specs.append(dict(lo0=None, K=1, cells={(1, dd): F(-1.0)}, iters=[1], tag=("absent-origin", dd)))
    # origins on subbox corners, one subbox apart: their own subbox holds nothing unless a probe cell lands in it
    return Case(n, d).origins(specs, base=(n - 1, 0, n - 1), spacing=2 * n + 3)


def long_walks(n, d):
    """one lower cell at distance M on one probe line, nothing lower before it, the lines absent (odd 0.5 like the
    origin's 0.0) or stored; max_iter M (found), M - 1 (out of reach) and 3n+1; origins at every offset in the subbox"""
    specs = []
    for M in iters_of(n):
        for dd in range(6):
            for stored in (False, True):
                specs.append(dict(lo0=F(0.0), K=M, fill=F(0.0) if stored else None, cells={(M, dd): F(-0.5)},
                                  iters=sorted({M, max(M - 1, 1), 3 * n + 1}), tag=("walk", M, dd, stored)))
    return Case(n, d).origins(specs, spacing=2 * (3 * n + 1) + 1 + 1)


def collapsed(n, d):
    """collapsed neighbours (every cell reads element 0): lower, equal, a near tie; origins inside collapsed subboxes"""
    c = Case(n, d, background=1.0)
    c.m.fill((0, 0, 0), 1.0)
    start, end = run_of(F(6.3))
    for dd, v in enumerate(F([0.5, 1.0, end, 2.0, start, -0.0])):
        c.m.collapse(tuple(unit(dd)), v)
    for dd, v in enumerate(F([7.0, 7.0, 7.0, 7.0, 7.0, 7.0])):
        c.m.collapse(tuple(2 * unit(dd)), v)
    rs = np.random.RandomState(n)
    for it in (1, n // 2 + 1, n + 1, 2 * n + 1):
        for loc in [(0, 0, 0), (n - 1, n - 1, n - 1), (n // 2, n // 2, n // 2), (0, n - 1, n // 2)]:
            c.queries.append((point(loc, d), it, ("full", loc)))
        for dd in range(6):
            g = unit(dd) * (1 + rs.randint(2))
            c.queries.append((point(g * n + rs.randint(0, n, 3), d), it, ("in-collapsed", dd)))
    return c


def far_origin(n, d):
    """origins in the outermost subboxes, index 2^20 - 1, -(2^20 - 1) and -2^20, on both faces: the six neighbour
    subboxes are not all addressable there (the kernel's `inner` is false), the ones beyond the range are absent"""
    c = Case(n, d)
    for a in range(3):
        for j, G in enumerate((GLB_LIMIT - 1, -(GLB_LIMIT - 1), -GLB_LIMIT)):
            for loc_a in (0, n - 1):
                g = np.array([3 * j, 3 * a, 6 + 3 * loc_a // max(n - 1, 1)])
                g[a] = G
                for t in (-2, -1, 0, 1, 2):
                    h = g.copy()
                    h[a] += t
                    if -GLB_LIMIT <= h[a] < GLB_LIMIT:
                        c.m.fill(tuple(h), 1.0)
                loc = np.array([n // 2] * 3)
                loc[a] = loc_a
                cell = g * n + loc
                inner = cell.copy()
                inner[a] += -n - 1 if G > 0 else n + 1
                if -GLB_LIMIT <= inner[a] // n < GLB_LIMIT:
                    c.m.set(inner, 0.5)
                for it in (1, n + 1, 2 * n + 1):
                    c.queries.append((point(cell, d), it, ("far", a, G, loc_a)))
    return c


TIE_POOL = None


def tie_pool():
    """log-odds values where the two rules or the two sides could part: run starts and ends near odd 1, +-0, tiny
    negatives, underflow, equal values"""
    global TIE_POOL
    if TIE_POOL is None:
        v = [F(0.0), F(-0.0), F(-1e-30), F(-2.0 ** -20), F(1.0), F(-1.0), F(-45.2), F(-60.0), F(-44.9), F(8.0), F(10.0)]
        for x in (5.0, 5.58623, 5.7, 6.0, 6.4, 6.8, 7.3, 7.6):
            v += list(run_of(F(x)))
        TIE_POOL = np.array(v, np.float32)
    return TIE_POOL


def dense_random(n, d, negative=False):
    """a dense field of tie-prone values over a box of subboxes; off-centre random queries, or (negative) lattice
    points, the doubles next to them, 0.0 and -0.0, at negative coordinates"""
    rs = np.random.RandomState(100 + n + negative)
    c = Case(n, d)
    span = max(1, -(-12 // n))
    pool = tie_pool()
    box = range(-span, span) if not negative else range(-2 * span, 0)
    for gx in box:
        for gy in box:
            for gz in box:
                c.m.full[(gx, gy, gz)] = pool[rs.randint(0, pool.size, n ** 3)]
    lo, hi = box[0] * n, (box[-1] + 1) * n
    its = iters_of(n)
    if not negative:
        for _ in range(300):
            c.queries.append((point(rs.randint(lo, hi, 3), d), int(rs.choice(its)), ("random",)))
    else:
        for _ in range(150):
            p = rs.randint(lo, hi + 1, 3) * d
            for q in (p, np.nextafter(p, np.inf), np.nextafter(p, -np.inf)):
                c.queries.append((q, int(rs.choice(its)), ("lattice",)))
        for z in (0.0, -0.0):
            c.queries.append((np.array([z, z, z]), 5, ("zero",)))
            c.queries.append((np.array([lo * d, z, -z]), 5, ("zero",)))
    return c


def float_domain(n, d):
    """every stored value drawn from the whole finite float domain (uniform bits), with the edges of the odd spelled
    out: +-0, denormals, the log-odds where 10^x overflows a double (odd NaN on both sides), run starts and ends"""
    rs = np.random.RandomState(7 + n)
    special = F([0.0, -0.0, 1e-45, -1e-45, 2.0 ** -28, -(2.0 ** -28), 308.2547, 308.25472, 309.0, 3.4e38, -3.4e38,
                 -45.2, -44.9, 7.53, 7.54, 64.0, -64.0])
    c = Case(n, d)
    cells = n ** 3
    k = -(-4096 // cells)
    v = rs.randint(0, 2 ** 32, k * cells, dtype=np.uint64).astype(np.uint32).view(np.float32)
    v = np.where(np.isfinite(v), v, F(1.5))
    v[:special.size + tie_pool().size] = np.concatenate([special, tie_pool()])
    for i in range(k):
        c.m.full[(i, -i, 2 * i)] = v[i * cells:(i + 1) * cells].copy()
    for i in range(3):
        c.m.collapse((i, i, -5), special[i + 6])
    return c


CASES = {"near_tie": near_tie, "resume": resume, "equal": equal, "underflow": underflow,
         "zeros_and_absent": zeros_and_absent, "long_walks": long_walks, "collapsed": collapsed,
         "far_origin": far_origin, "dense_random": dense_random,
         "lattice_negative": lambda n, d: dense_random(n, d, negative=True), "float_domain": float_domain}
DECODABLE = {k for k in CASES if k not in ("lattice_negative",)}


def build(name, n):
    cfg = cfg_n(n)
    return cfg, CASES[name](n, cfg.subbox_d_xyz)


def stored_cells(ex, n):
    """every (glb, sub) a map stores: all cells of full subboxes, cells 0 and n^3 - 1 of collapsed ones"""
    glb, sub = [], []
    for g, col in zip(ex["glb"], ex["collapsed"]):
        s = np.array([0, n ** 3 - 1]) if col else np.arange(n ** 3)
        glb.append(np.repeat(g[None], s.size, 0))
        sub.append(s)
    return np.concatenate(glb).astype(np.int32), np.concatenate(sub).astype(np.int32)


def spec_results(c):
    """(odd (q,), vectors (q, 3), winners [(k, d) or None]) of every query, from the restatement"""
    o = np.array([c.m.get_odd(p) for p, _, _ in c.queries], np.float32)
    vec, win = [], []
    for p, it, _ in c.queries:
        v, w, _ = c.m.grad(p, it)
        vec.append(v)
        win.append(None if w is None else w[:2])
    return o, np.array(vec, np.float64).reshape(-1, 3), win


def oracle_results(orc, c):
    pts = np.array([p for p, _, _ in c.queries], np.float64)
    its = np.array([it for _, it, _ in c.queries])
    vec = np.zeros((len(pts), 3))
    for it in np.unique(its):
        sel = its == it
        vec[sel] = orc.getOddGrad(pts[sel], int(it))
    return orc.getOdd(pts), vec


# ---- edges: each case shows it reached the edge it is named for ------------------------------------------------------
def assert_edge(name, c, win):
    tags = [t for _, _, t in c.queries]
    if name == "near_tie":
        # with the tie in an earlier direction the reference's winner is NOT the (first) lowest log-odds direction,
        # and the rule without the near-one check would have picked the other one
        parted = 0
        for (p, it, t), w in zip(c.queries, win):
            kind, lm, a, b = t
            assert w == (it, a if kind == "earlier" else b), (t, w)
            lo0, lo_d = c.m.lo_at(*c.m.locate(p))[1], c.m.round_lo(p, it)
            assert reference_rule(lo0, lo_d) == w[1]
            parted += kernel_rule_before_fix(lo0, lo_d) != w[1]
        assert parted == sum(1 for t in tags if t[0] == "earlier"), parted
    elif name == "resume":
        for (p, it, t), w in zip(c.queries, win):
            if t[0] == "never":
                lo_d = c.m.round_lo(p, 1)
                assert w is None and (lo_d < c.m.lo_at(*c.m.locate(p))[1]).all()
            else:
                lo0 = c.m.lo_at(*c.m.locate(p))[1]
                r1 = c.m.round_lo(p, 1)
                assert r1.min() < lo0 and odd(r1.min()) == odd(lo0)   # lower log-odds, same odd: not a winner
                assert w is not None and w[0] == 2, (t, w)
                if t[0] == "resume-tie":
                    assert w[1] == t[2] % 5 and odd(c.m.round_lo(p, 2)[t[2] % 5]) == odd(c.m.round_lo(p, 2)[5])
    elif name == "equal":
        for (p, it, t), w in zip(c.queries, win):
            if t[0] == "equal" and it == 1:
                assert w == (1, t[1][0])
            elif t[0] != "equal":
                assert w is None, (t, w)
    elif name == "underflow":
        got = [w for (_, _, t), w in zip(c.queries, win) if t[0] == "zero-odd-tie" and w]
        assert got and all(w == (1, 0) for w in got)   # odd 0 at -45.2 (+z) and -60 (-x): the first wins
        assert any(w == (1, 1) for (_, _, t), w in zip(c.queries, win) if t[0] == "denormal-tie")
        assert odd(F(-44.7)) == odd(F(-45.1)) > 0 and odd(F(-45.1)) < np.finfo(np.float32).tiny
    elif name == "zeros_and_absent":
        for (p, it, t), w in zip(c.queries, win):
            if t[0] == "zero-border":
                assert w is None
            if t[0] == "zero-tiny":
                assert w is not None and w[0] == 3, (t, w)
            if t[0] == "absent-origin":
                assert w == (1, t[1]), (t, w)
        assert any(t[0] == "absent-origin" and c.m.locate(p)[0] not in c.m.full for p, _, t in c.queries)
    elif name == "long_walks":
        hops = set()
        for (p, it, t), w in zip(c.queries, win):
            _, M, dd, _ = t
            assert w == ((M, dd) if it >= M else None), (t, it, w)
            if w:
                g0, _ = c.m.locate(p)
                g1, _ = c.m.locate(np.asarray(p) + M * c.d * unit(dd))
                hops.add(int(np.abs(np.subtract(g1, g0)).sum()))
        assert hops >= {0, 1, 2, 3}, hops
    elif name == "collapsed":
        assert any(w is not None and c.m.locate(p)[0] in c.m.collapsed for (p, _, _), w in zip(c.queries, win))
        hit = 0
        for (p, it, t), w in zip(c.queries, win):
            if w is None:
                continue
            g, sub = c.m.locate(p)
            for _ in range(w[0]):
                g, sub = c.m.step(g, sub, w[1])
            hit += g in c.m.collapsed
        assert hit > 0
    elif name == "far_origin":
        gs = {c.m.locate(p)[0] for p, _, _ in c.queries}
        for G in (GLB_LIMIT - 1, -(GLB_LIMIT - 1), -GLB_LIMIT):
            assert any(G in g for g in gs)
        assert sum(w is not None for w in win) > len(win) // 2
    elif name in ("dense_random", "lattice_negative"):
        assert sum(w is not None for w in win) > len(win) // 3
    elif name == "float_domain":
        assert np.isnan(odd(F(309.0))) and odd(F(308.2547)) == 1.0


@pytest.fixture(scope="module")
def scan():
    r = scan_log_odds()
    print(f"\nfloat log-odds scan: {r['count']} values in {r['seconds']:.1f} s, {len(r['flips'])} flips, "
          f"tie threshold {float(r['tie_threshold'])!r}")
    return r


def test_exp10_error_never_changes_the_float_odd(scan):
    """every float 2^-28 <= |x| <= 64: the float odd is the same for both doubles next to 10^x, so a 1-ulp exp10 and
    glibc's pow give the same getOdd"""
    assert scan["count"] == 2 * (34 * 2 ** 23 + 1)
    assert scan["flips"] == [], scan["flips"][:20]


def test_near_tie_window_premise(scan):
    """the first log-odds >= -30 whose run of equal float odds reaches past kTie: the kernel's near-one bound sits below
    it, and the bound before it (none) is what the near-tie cases break"""
    T = scan["tie_threshold"]
    assert T == F(5.58623), repr(T)
    assert K_NEAR_ONE < T
    start, end = run_of(T)
    assert start == T and end - T > K_TIE
    s0, e0 = run_of(np.nextafter(T, F(-np.inf)))
    assert e0 - s0 <= K_TIE


def test_rules_part_above_the_threshold():
    """the worked case (origin 7.5, +z 7.0, -z 6.9): both neighbours' odds round to 1 - 2^-23, the reference takes +z,
    the rule without the near-one check -z; at every run start below the threshold the two rules agree"""
    lo0, row = F(7.5), F([7.0, 6.9, 9, 9, 9, 9])
    assert odd(F(7.0)) == odd(F(6.9)) == F(1 - 2.0 ** -23) and odd(lo0) == F(1 - 2.0 ** -24)
    assert reference_rule(lo0, row) == 0 and kernel_rule_before_fix(lo0, row) == 1
    for x in np.arange(4.0, 5.58, 0.05, dtype=np.float32):
        s, e = run_of(x)
        r = F([e, 9, 9, 9, 9, s])
        assert reference_rule(F(9.5), r) == kernel_rule_before_fix(F(9.5), r), x


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("name", sorted(CASES))
def test_spec_equals_the_oracle(name, n):
    cfg, c = build(name, n)
    ex = c.m.export()
    orc = ViewOracle(cfg)
    orc.set_map(ex)
    o_spec, v_spec, win = spec_results(c)
    o_orc, v_orc = oracle_results(orc, c)
    assert same_floats(o_spec, o_orc), name
    diff = np.flatnonzero((v_spec.view(np.uint64) != v_orc.view(np.uint64)).any(1))
    assert diff.size == 0, (name, c.queries[diff[0]] if diff.size else None)
    if name in DECODABLE:
        for (p, it, t), v, w in zip(c.queries, v_spec, win):
            assert decode(c.m, p, v, it) == w, (t, w)
    assert_edge(name, c, win)
    # every stored value read back through the cell-centre queries
    if name == "float_domain":
        glb, sub = stored_cells(ex, n)
        want = np.array([c.m.odd_at(tuple(g), s) for g, s in zip(glb.tolist(), sub.tolist())], np.float32)
        cen = np.array([c.m.centre(tuple(g), s) for g, s in zip(glb.tolist(), sub.tolist())])
        assert same_floats(orc.getOdd(cen), want)


def test_map_checkpoint_parses_back():
    """write_map_checkpoint's records: header, log-odds of full subboxes, col_lo of collapsed ones, states, frontier"""
    n = 3
    cfg = cfg_n(n)
    c = collapsed(n, cfg.subbox_d_xyz)
    ex = c.m.export()
    full = ex["collapsed"] == 0
    ex["log_odds"][full] = np.random.RandomState(1).uniform(-3, 9, (int(full.sum()), n ** 3)).astype(np.float32)
    i = int(np.flatnonzero(full)[0])
    ex["occupancy"][i, :5] = b"o"
    ex["frontier"][i, 0] = 0x5a
    image = write_map_checkpoint(fresh_header(cfg), cfg, ex)
    hd = CkptHeader.from_buffer_copy(image[:C.sizeof(CkptHeader)])
    rb, cells = record_bytes(n), n ** 3
    body = image[C.sizeof(CkptHeader):]
    m = ex["glb"].shape[0]
    assert hd.n_records == m and len(body) == m * rb and fnv1a64(body) == hd.checksum
    recs = np.frombuffer(body, np.uint8).reshape(m, rb)
    assert np.array_equal(recs[:, :12].copy().view("<i4"), ex["glb"])
    col = recs[:, 12:16].copy().view("<i4").ravel()
    assert np.array_equal(col, ex["collapsed"]) and col.sum() == 12
    col_lo = recs[:, 16:20].copy().view("<f4").ravel()
    lo = recs[:, 32:32 + 4 * cells].copy().view("<f4")
    full = col == 0
    assert np.array_equal(lo[full].view(np.uint32), ex["log_odds"][full].view(np.uint32))
    assert np.array_equal(col_lo.view(np.uint32), ex["log_odds"][:, 0].view(np.uint32))
    assert (lo[~full] == 0).all()
    assert np.array_equal(recs[full, 32 + 4 * cells:32 + 5 * cells], ex["occupancy"][full].view(np.uint8))
    assert recs[i, 32 + 6 * cells] == 0x5a
