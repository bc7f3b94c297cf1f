"""GPU: getOdd, getOdd_at and getOddGrad (k_get_odd, k_get_odd_at, k_get_odd_grad) bit for bit against the oracle and
the Python restatement on crafted log-odds maps restored from checkpoint images at subbox sizes 2, 3, 10 and 16, with
the winning candidate cell of every pseudo-gradient decoded and compared; and on a map built from frames whose
log-odds pass 5.8 (log_odds_max = 8), where near-one ties of the float odd occur."""
import numpy as np
import pytest

from grad_spec import LogOddsMap, decode, same_floats
from mlmapping_b200 import MLMap, config_cfg_a, scenes
from oracle_binding import Oracle
from test_query_grad_host import (CASES, DECODABLE, SIZES, cfg_n, iters_of, oracle_results, spec_results,
                                  stored_cells)
from view_oracle import ViewOracle
from view_spec import write_map_checkpoint

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=SIZES)
def handle(request):
    """an exploration handle at subbox size n and the header of its fresh checkpoint"""
    n = request.param
    cfg = cfg_n(n)
    gpu = MLMap(cfg)
    yield n, cfg, gpu, gpu.checkpoint()
    gpu.close()


def gpu_grad(gpu, pts, its):
    out = np.zeros((len(pts), 3))
    for it in np.unique(its):
        sel = its == it
        out[sel] = gpu.getOddGrad(pts[sel], int(it))
    return out


def first_difference(a, b):
    bad = np.flatnonzero((np.asarray(a).view(np.uint64) != np.asarray(b).view(np.uint64)).any(1))
    return None if bad.size == 0 else int(bad[0])


@pytest.mark.parametrize("name", sorted(CASES))
def test_crafted_map_bit_for_bit(handle, name):
    n, cfg, gpu, template = handle
    c = CASES[name](n, cfg.subbox_d_xyz)
    ex = c.m.export()
    gpu.restore(write_map_checkpoint(template, cfg, ex))
    back = gpu.export_map()
    assert np.array_equal(back["glb"], ex["glb"]) and np.array_equal(back["log_odds"].view(np.uint32),
                                                                     ex["log_odds"].view(np.uint32))
    orc = ViewOracle(cfg)
    orc.set_map(ex)
    pts = np.array([p for p, _, _ in c.queries], np.float64)
    its = np.array([it for _, it, _ in c.queries])
    o_spec, v_spec, win = spec_results(c)
    o_orc, v_orc = oracle_results(orc, c)
    assert same_floats(o_spec, o_orc) and first_difference(v_spec, v_orc) is None, name
    assert same_floats(gpu.getOdd(pts), o_orc), name
    v_gpu = gpu_grad(gpu, pts, its)
    i = first_difference(v_gpu, v_orc)
    if i is not None:
        p, it, tag = c.queries[i]
        got = decode(c.m, p, v_gpu[i], it) if name in DECODABLE else None
        raise AssertionError((name, n, tag, "max_iter", it, "gpu", v_gpu[i], got, "oracle", v_orc[i], win[i],
                              int((v_gpu.view(np.uint64) != v_orc.view(np.uint64)).any(1).sum()), "queries differ"))
    if name in DECODABLE:
        for (p, it, tag), v, w in zip(c.queries, v_gpu, win):
            assert decode(c.m, p, v, it) == w, (name, tag)
    # getOdd_at: every stored value of the float-domain map, a sample of the others
    glb, sub = stored_cells(ex, n)
    if name != "float_domain":
        sel = np.random.RandomState(n).choice(glb.shape[0], min(glb.shape[0], 20000), replace=False)
        glb, sub = glb[sel], sub[sel]
    want = np.array([c.m.odd_at(tuple(g), s) for g, s in zip(glb.tolist(), sub.tolist())], np.float32)
    assert same_floats(gpu.getOdd_at(glb, sub), want), name
    absent = [g for g in (glb[:200] + np.array([0, 0, 7])).tolist()
              if abs(g[2]) < 1 << 20 and tuple(g) not in c.m.full and tuple(g) not in c.m.collapsed]
    assert (gpu.getOdd_at(np.array(absent, np.int32).reshape(-1, 3), sub[:len(absent)]) == 0.5).all()


def test_frame_built_map_past_odd_one():
    """CFG-A with log_odds_max = 8: after eight corridor frames thousands of voxels hold log-odds above 5.8, where
    neighbours of different log-odds share a float odd; getOdd and getOddGrad at every walk length equal the oracle bit
    for bit, and a sample of the gradients the restatement and its decoded winner"""
    cfg = config_cfg_a()
    cfg.log_odds_max = 8.0
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(8):
        pose = scenes.corridor_trajectory_pose(5 * k)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    g, m = gpu.export_map(), orc.export_map()
    assert np.array_equal(g["glb"], m["glb"]) and np.array_equal(g["log_odds"].view(np.uint32), m["log_odds"].view(np.uint32))
    assert (m["log_odds"] > 5.8).sum() > 1000
    n, d = cfg.subbox_n, cfg.subbox_d_xyz
    # around the voxels past 5.8, off the cell centres, and anywhere in the map
    hot = np.argwhere(m["log_odds"] > 5.8)
    rs = np.random.RandomState(11)
    pick = hot[rs.choice(hot.shape[0], 20000)]
    sub = pick[:, 1]
    loc = np.stack([sub % n, (sub // n) % n, sub // (n * n)], 1)
    cells = m["glb"][pick[:, 0]].astype(np.int64) * n + loc + rs.randint(-2, 3, (20000, 3))
    pts = np.concatenate([(cells + rs.uniform(0.05, 0.95, (20000, 3))) * d,
                          scenes.query_positions(20000, m["glb"].min(0) * n * d, (m["glb"].max(0) + 1) * n * d, seed=3)])
    assert np.array_equal(gpu.getOdd(pts).view(np.uint32), orc.getOdd(pts).view(np.uint32))
    spec = LogOddsMap.from_export(m, n, d)
    for it in iters_of(n):
        vg, vo = gpu.getOddGrad(pts, it), orc.getOddGrad(pts, it)
        i = first_difference(vg, vo)
        assert i is None, (it, i, pts[i], vg[i], vo[i], spec.grad(pts[i], it)[1])
        for j in rs.choice(20000, 300, replace=False):   # (the points off the cell centres)
            v, w, _ = spec.grad(pts[j], it)
            assert np.array_equal(np.array(v), vg[j]) and decode(spec, pts[j], vg[j], it) == (None if w is None else w[:2])
