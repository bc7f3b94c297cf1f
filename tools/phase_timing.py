"""per-column phase breakdown of k_column (needs a -DMLM_PHASE_TIMING build: sh csrc/build.sh -DMLM_PHASE_TIMING)"""
import sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
from mlmapping_b200 import MLMap, config_cfg_a, scenes
cfg = config_cfg_a()
m = MLMap(cfg)
for k in range(6):
    pose = scenes.corridor_trajectory_pose(100 + k)
    img = scenes.corridor_depth_frame(cfg, pose, frame_idx=100 + k)
    if "--flush" in sys.argv:
        m.flush_l2()
        m.sync()
    m.integrate_depth(img, pose)
c = m.debug_phase_cycles()
nc = c.shape[0] - 256
fr = c[nc:]
c = c[:nc]
act = c[:, 10] > 0
names = ["gather", "bound", "contrib", "radix", "fold||walks", "miss-stage"]
cc = np.concatenate([c[:, 15:16], c[:, :4], c[:, 6:8]], axis=1)
d = np.diff(cc, axis=1)[act]
tot = d.sum(1)
order = np.argsort(-tot)
print("columns", act.sum(), "cycles: total max", tot.max(), "mean", tot.mean())
print("phase", names)
print("mean  ", d.mean(0).astype(int))
print("max   ", d.max(0).astype(int))
# inside the overlapped phase (relative to its start, slot 3): fold half = heads, fold, hit staging; walk half = inside walks, outside walks
ca = c[act]
sub = np.stack([ca[:, 4] - ca[:, 3], ca[:, 5] - ca[:, 4], ca[:, 8] - ca[:, 5], ca[:, 9] - ca[:, 3], ca[:, 12] - ca[:, 9]], axis=1)
print("fold half [heads, fold, hit-stage] | walk half [inside walks, outside walks]")
print("mean  ", sub.mean(0).astype(int))
print("max   ", sub.max(0).astype(int))
for i in order[:6]:
    print("col", np.nonzero(act)[0][i], "n_c", ca[i, 10], "n_k", ca[i, 11], "tot", tot[i], d[i], "sub", sub[i])
t0 = ca[:, 13].min()
st, en = (ca[:, 13] - t0) / 1e3, (ca[:, 14] - t0) / 1e3
print("wall us: first start 0, last start %.1f, last end %.1f; starts>5us: %d" % (st.max(), en.max(), (st > 5).sum()))
print("per-item duration us: mean %.1f max %.1f sum %.0f" % ((en - st).mean(), (en - st).max(), (en - st).sum()))
late = np.argsort(-st)[:8]
print("latest starters (col, start, end, n_c, n_k):", [(int(np.nonzero(act)[0][i]), round(float(st[i]), 1), round(float(en[i]), 1), int(ca[i, 10]), int(ca[i, 11])) for i in late])
first = np.argsort(st)[:6]
print("first starters:", [(int(np.nonzero(act)[0][i]), round(float(st[i]), 1), round(float(en[i]), 1), int(ca[i, 10]), int(ca[i, 11])) for i in first])
fa = fr[fr[:, 0] > 0]
if len(fa):
    t0 = fa[:, 0].min()
    rel = (fa[:, :9] - t0) / 1e3
    names = ["start", "proj done", "bar1 out", "cols done", "bar2 out", "bar3 out", "end", "col prologue", "fuse ticket"]
    for i, n in enumerate(names):
        print(f"k_frame {n:10s}: min {rel[:, i].min():6.1f}  mean {rel[:, i].mean():6.1f}  max {rel[:, i].max():6.1f} us")
    # column prologue (bar1 out -> queue ready): odds / k_reach tables, per-column weights, merge of light columns, queue sort
    pro = np.stack([fa[:, 13] - fa[:, 2], fa[:, 14] - fa[:, 13], fa[:, 15] - fa[:, 14], fa[:, 7] - fa[:, 15]], axis=1) / 1e3
    print("col prologue us [tables, weights, merge, queue sort]: mean", pro.mean(0).round(2), "max", pro.max(0).round(2))
    ids = np.nonzero(fr[:, 0] > 0)[0]
    o = np.argsort(-rel[:, 8])
    print("fuse ticket times, slowest 12 (cta, bar2 out, ticket):", [(int(ids[i]), round(float(rel[i, 4]), 1), round(float(rel[i, 8]), 1)) for i in o[:12]])
    print("fuse ticket percentiles:", np.percentile(rel[:, 8], [0, 25, 50, 75, 90, 100]).round(1))
