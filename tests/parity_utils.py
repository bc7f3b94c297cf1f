"""helpers shared by the parity tests: compare a CUDA map (mlmapping_b200.MLMap) with the CPU oracle"""
import numpy as np


def assert_frame_parity(gpu, orc, st_g, st_o, check_order=True, tag=""):
    """per-frame sets: bit-exact hit keys (in the reference's iteration order) + probabilities, miss set"""
    for f in ("n_points", "n_inside", "n_cast", "n_hit_cells", "n_miss_cells", "n_touched_voxels",
              "hit_bucket_count", "ram_expand_cnt", "obs_cnt"):
        assert getattr(st_g, f) == getattr(st_o, f), (tag, f, getattr(st_g, f), getattr(st_o, f))
    kg, pg = gpu.last_frame_hits()
    ko, po = orc.last_frame_hits()
    assert kg.shape == ko.shape, (tag, kg.shape, ko.shape)
    if check_order:
        assert np.array_equal(kg, ko), (tag, "hit key iteration order differs",
                                        int(np.argmax((kg != ko).any(axis=1))))
        assert np.array_equal(pg.view(np.uint32), po.view(np.uint32)), (tag, "hit probabilities differ")
    else:
        og = np.lexsort((kg[:, 2], kg[:, 1], kg[:, 0]))
        oo = np.lexsort((ko[:, 2], ko[:, 1], ko[:, 0]))
        assert np.array_equal(kg[og], ko[oo]), (tag, "hit key sets differ")
        assert np.array_equal(pg[og].view(np.uint32), po[oo].view(np.uint32)), (tag, "hit probabilities differ")
    mg = gpu.last_frame_misses()
    mo = orc.last_frame_misses()
    assert np.array_equal(mg, mo), (tag, "miss sets differ", mg.size, mo.size)


def assert_map_parity(gpu, orc, lo_tol=1e-6, tag=""):
    """whole map: same subbox set, bit-exact occupancy states, log-odds within lo_tol (reports exactness)"""
    g = gpu.export_map()
    o = orc.export_map()
    assert np.array_equal(g["glb"], o["glb"]), (tag, "allocated subbox sets differ", g["glb"].shape, o["glb"].shape)
    assert np.array_equal(g["collapsed"], o["collapsed"]), (tag, "collapsed flags differ")
    assert np.array_equal(g["occupancy"], o["occupancy"]), (
        tag, "occupancy states differ", int((g["occupancy"] != o["occupancy"]).sum()))
    assert np.array_equal(g["inflate"], o["inflate"]), (tag, "inflate states differ")
    if "frontier" in g:
        assert np.array_equal(g["frontier"], o["frontier"]), (
            tag, "frontier sets differ", int((np.unpackbits(g["frontier"]) != np.unpackbits(o["frontier"])).sum()))
    d = np.abs(g["log_odds"].astype(np.float64) - o["log_odds"].astype(np.float64))
    assert d.max(initial=0.0) <= lo_tol, (tag, "log-odds differ", float(d.max()))
    exact = np.array_equal(g["log_odds"].view(np.uint32), o["log_odds"].view(np.uint32))
    return {"subboxes": int(g["glb"].shape[0]), "log_odds_bit_exact": bool(exact), "max_abs_diff": float(d.max(initial=0.0))}


def _sorted_rows(a):
    a = np.ascontiguousarray(a)
    if a.shape[0] == 0:
        return a
    v = a.view(np.uint32).reshape(a.shape[0], -1)
    return a[np.lexsort(tuple(v[:, c] for c in range(v.shape[1] - 1, -1, -1)))]


def assert_cloud_parity(gpu, orc, kinds=(0, 1), heights=(0.75, 1.25), tag=""):
    """map clouds for consumers (rviz_vis.cpp:267-327, mlmap.cpp:200-284): same point SETS bit for bit (the order
    of the reference's clouds is its unordered_map iteration order, which no consumer can rely on); the slice's
    odd bit for bit like getOdd"""
    sizes = {}
    for kind in kinds:
        g, o = _sorted_rows(gpu.export_cloud(kind)), _sorted_rows(orc.export_cloud(kind))
        assert g.shape == o.shape, (tag, kind, g.shape, o.shape)
        assert np.array_equal(g.view(np.uint32), o.view(np.uint32)), (tag, "cloud", kind)
        sizes[kind] = g.shape[0]
    for hgt in heights:
        g, o = gpu.export_odds_slice(hgt), orc.export_odds_slice(hgt)
        assert g.shape == o.shape, (tag, "slice", hgt, g.shape, o.shape)
        gi = np.lexsort((g[:, 2], g[:, 1], g[:, 0]))
        oi = np.lexsort((o[:, 2], o[:, 1], o[:, 0]))
        g, o = g[gi], o[oi]
        assert np.array_equal(g[:, :3].view(np.uint32), o[:, :3].view(np.uint32)), (tag, "slice xyz", hgt)
        assert np.array_equal(g[:, 3].view(np.uint32), o[:, 3].view(np.uint32)), (tag, "slice odd", hgt)
        sizes[("slice", hgt)] = g.shape[0]
    return sizes
