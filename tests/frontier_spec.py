"""The frontier-clustering spec of include/mlmap_b200.h ("frontier clustering") restated in plain numpy / scipy, apart from
both the C++ oracle and the kernels: the frontier cells decoded from an export_map / export_frontier bitmask, labelled
with scipy.ndimage.label on their AABB grid (and, for small sets, a pure-Python union-find), and the records formed and
sorted as rules 3-4 say.  Also a writer of checkpoint images with arbitrary frontier sets (the record layout of
mlmapping_b200/csrc/shard_kernels.cuh), so that any frontier set can be put on the device through mlm_checkpoint_restore.
TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C

import numpy as np
from scipy import ndimage

from mlmapping_b200.capi import FRONTIER_CLUSTER_DTYPE, MlmConfig


def decode_frontier(ex, n):
    """(m, 3) int64 cells (x, y, z) of the frontier bitmasks of an export dict (bit c of the little-endian bytes = cell
    id c); collapsed subboxes hold none"""
    fr = np.asarray(ex["frontier"], dtype=np.uint8)
    if fr.shape[0] == 0:
        return np.zeros((0, 3), dtype=np.int64)
    bits = np.unpackbits(fr, axis=1, bitorder="little")[:, :n ** 3]
    bits[np.asarray(ex["collapsed"]) != 0] = 0
    r, ids = np.nonzero(bits)
    loc = np.stack([ids % n, (ids // n) % n, ids // (n * n)], 1)
    return np.asarray(ex["glb"], dtype=np.int64)[r] * n + loc


def box_cells(d, box_min, box_max):
    """rule 1 of the ray spec on both corners: (lo[3], hi[3]) int64"""
    lo = np.floor(np.asarray(box_min, dtype=np.float64) / d).astype(np.int64)
    hi = np.floor(np.asarray(box_max, dtype=np.float64) / d).astype(np.int64)
    return lo, hi


def label_scipy(cells, conn6=False):
    """component label (0..k-1, arbitrary numbering) of every cell, by scipy.ndimage.label on the AABB grid"""
    if cells.shape[0] == 0:
        return np.zeros(0, dtype=np.int64)
    lo = cells.min(0)
    g = np.zeros(tuple(cells.max(0) - lo + 1), dtype=bool)
    g[tuple((cells - lo).T)] = True
    lab, _ = ndimage.label(g, ndimage.generate_binary_structure(3, 1 if conn6 else 3))
    return lab[tuple((cells - lo).T)].astype(np.int64) - 1


def label_union_find(cells, conn6=False):
    """the same by a pure-Python union-find over a dict of cells (small sets only)"""
    index = {tuple(c): i for i, c in enumerate(cells.tolist())}
    parent = list(range(len(index)))

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    offs = [(dx, dy, dz) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)
            if (abs(dx) + abs(dy) + abs(dz) == 1) or (not conn6 and (dx, dy, dz) != (0, 0, 0))]
    for (x, y, z), i in index.items():
        for dx, dy, dz in offs:
            j = index.get((x + dx, y + dy, z + dz))
            if j is not None:
                a, b = find(i), find(j)
                if a != b:
                    parent[max(a, b)] = min(a, b)
    return np.array([find(i) for i in range(len(parent))], dtype=np.int64)


def clusters(cells, d, box=None, min_cells=1, conn6=False, labeller=label_scipy):
    """rules 1-5 on a cell set: (records as FRONTIER_CLUSTER_DTYPE, labelled cells (m, 3) int32, cluster index (m,)),
    the labelled cells sorted by (cluster index, z, y, x)"""
    cells = np.asarray(cells, dtype=np.int64).reshape(-1, 3)
    if box is not None:
        lo, hi = box
        cells = cells[((cells >= lo) & (cells <= hi)).all(1)]
    lab = labeller(cells, conn6)
    _, comp = np.unique(lab, return_inverse=True)
    k = int(comp.max()) + 1 if cells.shape[0] else 0
    order = np.lexsort((cells[:, 0], cells[:, 1], cells[:, 2], comp))  # by component, then (z, y, x)
    cells, comp = cells[order], comp[order]
    first = np.searchsorted(comp, np.arange(k))
    n_cells = np.bincount(comp, minlength=k)
    keep = n_cells >= min_cells
    keys = cells[first]
    rec = np.zeros(k, dtype=FRONTIER_CLUSTER_DTYPE)
    rec["n_cells"] = n_cells
    rec["key"] = keys
    for a in range(3):
        rec["lo"][:, a] = np.minimum.reduceat(cells[:, a], first) if k else 0
        rec["hi"][:, a] = np.maximum.reduceat(cells[:, a], first) if k else 0
        s = np.add.reduceat(cells[:, a], first) if k else np.zeros(0, np.int64)  # exact int64 sums
        rec["centroid"][:, a] = ((s.astype(np.float64) / n_cells.astype(np.float64)) + 0.5) * d
    kept = np.nonzero(keep)[0]
    kept = kept[np.lexsort((keys[kept, 0], keys[kept, 1], keys[kept, 2]))]
    index = np.full(k, -1, dtype=np.int64)
    index[kept] = np.arange(kept.size)
    sel = keep[comp]
    lab_cells, lab_of = cells[sel], index[comp[sel]]
    o = np.lexsort((lab_cells[:, 0], lab_cells[:, 1], lab_cells[:, 2], lab_of))
    return rec[kept], lab_cells[o].astype(np.int32), lab_of[o].astype(np.int32)


def sort_labels(cells, of):
    """labelled cells in the order clusters() gives them (the API leaves their order open)"""
    o = np.lexsort((cells[:, 0], cells[:, 1], cells[:, 2], of))
    return cells[o], of[o]


# ---- checkpoint images with arbitrary frontier sets ---------------------------------------------------------------
class CkptHeader(C.Structure):
    """CkptFileHeader of mlmapping_b200/csrc/mlmap_capi.cu"""
    _fields_ = [("magic", C.c_char * 8), ("version", C.c_uint32), ("header_bytes", C.c_uint32), ("cfg", MlmConfig),
                ("cells", C.c_int32), ("front_words", C.c_int32), ("explore", C.c_int32), ("rec_bytes", C.c_int32),
                ("n_records", C.c_uint64), ("bucket_count", C.c_uint32), ("bucket_count_miss", C.c_uint32),
                ("cum_ram_expand", C.c_int64), ("cum_obs", C.c_int64), ("n_submaps", C.c_int64),
                ("rng_r", C.c_int32 * 31), ("rng_f", C.c_int32), ("rng_b", C.c_int32), ("checksum", C.c_uint64)]


def record_bytes(n):
    cells, fw = n ** 3, (n ** 3 + 31) // 32
    return (32 + cells * 6 + fw * 4 + 15) & ~15


def fnv1a64(buf: bytes) -> int:
    """the checkpoint checksum: FNV-1a 64 over little-endian 8-byte words, then the tail bytes"""
    h, p, mask = 0xcbf29ce484222325, 0x100000001b3, (1 << 64) - 1
    words = np.frombuffer(buf[:len(buf) // 8 * 8], dtype="<u8").tolist()
    for w in words:
        h = ((h ^ w) * p) & mask
    for b in buf[len(buf) // 8 * 8:]:
        h = ((h ^ b) * p) & mask
    return h


def fresh_header(cfg) -> bytes:
    """the header a fresh exploration handle writes (bucket counts 1, counters 0) for images built without a device"""
    hd = CkptHeader()
    hd.magic, hd.version, hd.header_bytes = b"MLMCKPT1", 2, C.sizeof(CkptHeader)
    hd.cfg = cfg.copy()
    n = cfg.subbox_n
    hd.cells, hd.front_words, hd.explore, hd.rec_bytes = n ** 3, (n ** 3 + 31) // 32, 1, record_bytes(n)
    hd.bucket_count = hd.bucket_count_miss = 1
    return bytes(hd)


def frontier_words(cells, n):
    """cells (m, 3) -> (glb (s, 3) int32, words (s, front_words) uint32), one row per subbox that holds a cell"""
    cells = np.asarray(cells, dtype=np.int64).reshape(-1, 3)
    g = np.floor_divide(cells, n)
    loc = cells - g * n
    sub = (loc[:, 2] * n + loc[:, 1]) * n + loc[:, 0]
    glb, inv = np.unique(g, axis=0, return_inverse=True)
    fw = (n ** 3 + 31) // 32
    bits = np.zeros((glb.shape[0], fw * 32), dtype=np.uint8)
    bits[inv.reshape(-1), sub] = 1
    words = np.packbits(bits, axis=1, bitorder="little").view("<u4")
    return glb.astype(np.int32), words


def write_checkpoint(template: bytes, cfg, glb, words, collapsed=None) -> bytes:
    """a checkpoint image: the template's header (e.g. of a fresh exploration handle after one frame) with its records
    replaced by one per subbox glb[i]: all cells unknown, log-odds 0, frontier bitmask words[i] (collapsed[i]: a
    collapsed unknown subbox); n_records, n_submaps and the checksum fixed"""
    hd = CkptHeader.from_buffer_copy(template[:C.sizeof(CkptHeader)])
    n = cfg.subbox_n
    cells, rb = n ** 3, record_bytes(n)
    assert hd.header_bytes == C.sizeof(CkptHeader) and hd.rec_bytes == rb and hd.explore == 1
    glb = np.asarray(glb, dtype=np.int32).reshape(-1, 3)
    m = glb.shape[0]
    recs = np.zeros((m, rb), dtype=np.uint8)
    head = np.zeros(m, dtype=[("g", "<i4", (3,)), ("flags", "<i4"), ("col_lo", "<f4"), ("col_occ", "S1"),
                              ("col_inf", "S1"), ("pad", "S10")])
    head["g"] = glb
    col = np.zeros(m, bool) if collapsed is None else np.asarray(collapsed, bool)
    head["flags"] = col.astype(np.int32)
    head["col_occ"] = head["col_inf"] = b"u"
    recs[:, :32] = head.view(np.uint8).reshape(m, 32)
    full = ~col
    recs[full, 32 + 4 * cells:32 + 6 * cells] = ord("u")
    w = np.asarray(words, dtype="<u4").reshape(m, -1)
    recs[full, 32 + 6 * cells:32 + 6 * cells + 4 * w.shape[1]] = w[full].view(np.uint8).reshape(int(full.sum()), -1)
    body = recs.tobytes()
    hd.n_records = hd.n_submaps = m
    hd.checksum = fnv1a64(body)
    return bytes(hd) + body


def read_checkpoint(image: bytes, n):
    """the parser of write_checkpoint's images: (header, glb (m, 3), collapsed (m,), frontier words (m, front_words));
    raises AssertionError on a wrong size or checksum"""
    hd = CkptHeader.from_buffer_copy(image[:C.sizeof(CkptHeader)])
    rb, cells, fw = record_bytes(n), n ** 3, (n ** 3 + 31) // 32
    body = image[C.sizeof(CkptHeader):]
    assert hd.magic == b"MLMCKPT1" and hd.rec_bytes == rb and len(body) == hd.n_records * rb
    assert fnv1a64(body) == hd.checksum
    recs = np.frombuffer(body, dtype=np.uint8).reshape(-1, rb)
    glb = recs[:, :12].copy().view("<i4").reshape(-1, 3)
    col = recs[:, 12:16].copy().view("<i4").reshape(-1)
    words = recs[:, 32 + 6 * cells:32 + 6 * cells + 4 * fw].copy().view("<u4")
    return hd, glb, col, words


def export_of(glb, words, collapsed, n):
    """an export_map-like dict (glb, collapsed, frontier bytes) of the subboxes of a written image"""
    fr = np.asarray(words, dtype="<u4").view(np.uint8)[:, :(n ** 3 + 7) // 8]
    return {"glb": np.asarray(glb), "collapsed": np.asarray(collapsed, dtype=np.uint8), "frontier": fr}
