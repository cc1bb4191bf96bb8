import hashlib
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "T0_golden.npz")
REF_GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_ikdtree.npz")


class _Cfg:
    def __init__(self, a):
        self.laser_point_cov, self.img_point_cov, self.cell_size = float(a[0]), float(a[1]), float(a[2])


def load_golden():
    g = dict(np.load(GOLD))
    c = g["cam"]
    frame = {k: g[k] for k in ("map_xyz", "scan_body", "R_prop", "p_prop", "cov", "vel", "bg", "ba", "grav", "R_LI", "t_LI",
                               "Rcl", "Pcl", "image", "patch_pos", "patch_ref", "patch_level")}
    frame["cam"] = dict(width=int(c[0]), height=int(c[1]), fx=c[2], fy=c[3], cx=c[4], cy=c[5], d=tuple(c[6:11]))
    frame["cfg"] = _Cfg(g["cfg"])
    return frame, g


_ref_gold = None


def load_ref_golden():
    """What the reference's own ikd-Tree (include/ikd-Tree/ikd_Tree.cpp) computed on the cases below, and the CPU path
    built on it at the full sizes (tests/golden/make_golden_ref.py).  Large results are kept as SHA-256 digests."""
    global _ref_gold
    if _ref_gold is None:
        _ref_gold = dict(np.load(REF_GOLD))
    return _ref_gold


def digest(*arrays):
    """SHA-256 over dtype, shape and bytes of each array: equal digests <=> bit-identical arrays."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def rows_sorted(a):
    """Sorted view of an (n,3) float32 array as rows, for exact set comparison."""
    a = np.ascontiguousarray(a, np.float32)
    return np.sort(a.view(np.dtype((np.void, 12))).ravel())


def knn_queries(base, rng, n, sigma):
    return (base[rng.integers(0, len(base), n)] + rng.normal(0, sigma, (n, 3))).astype(np.float32)


def tie_lattice():
    """Map on a 0.25 m integer lattice and queries on lattice points and cell centres: exact float distance ties."""
    g = np.arange(-8, 9, dtype=np.float32) * 0.25
    lat = np.stack(np.meshgrid(g, g, g[:5], indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    rng = np.random.default_rng(3)
    lat = lat[rng.permutation(len(lat))]
    q = np.concatenate([lat[:400], lat[400:800] + np.float32(0.125), lat[800:1000] + np.array([0.125, 0, 0], np.float32)]).astype(np.float32)
    return lat, q


def world_scan(f):
    return ((f["R_true"] @ (f["R_LI"] @ f["scan_body"].T.astype(np.float64) + f["t_LI"][:, None])).T + f["p_true"]).astype(np.float32)


def add_points_case(f):
    """Three successive Add_Points batches (the second re-observes the same surfaces, the third is far-field clutter)
    and the kNN queries asked of the map afterwards."""
    rng = np.random.default_rng(3)
    new = world_scan(f)
    batches = [new, new + rng.normal(0, 0.02, new.shape).astype(np.float32),
               rng.uniform(f["map_xyz"].min(0), f["map_xyz"].max(0), (len(new) // 4, 3)).astype(np.float32)]
    return batches, knn_queries(new, rng, 2000, 0.1)


def delete_boxes_case(f):
    lo, hi = f["map_xyz"].min(0), f["map_xyz"].max(0)
    return np.array([[lo[0], lo[1], lo[2], lo[0] + 6, lo[1] + 40, hi[2] + 1],      # a slab along one wall
                     [0.0, 0.0, -1.0, 4.0, 4.0, 3.0],                              # a chunk in the middle
                     [hi[0] - 0.01, lo[1], lo[2], hi[0] + 1, hi[1] + 1, hi[2] + 1]], np.float32)
