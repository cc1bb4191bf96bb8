"""Inputs of the map-maintenance lifecycle cases (tests/golden/make_golden_map.py pins what the reference's ikd-Tree
returns on them; tests/test_gpu_map_lifecycle.py replays them on the device), plus plain numpy restatements of the rules
the cases are built around:

- lasermap_fov_segment (src/laserMapping.cpp:363-421): which boxes a moving sensor cuts out of the map,
- rebuild_grid's margin rule (fast-livo_b200/csrc/flb_capi.cu): the box the device kNN grid covers, which decides whether
  flb_map_add_points takes the incremental or the full path,
- KD_TREE::Add_Points(points, downsample = true) (ikd_Tree.cpp:382-457) point by point in float32, used to keep the
  voxel-boundary sets free of results that depend on the tree's traversal order.
"""
import numpy as np

from golden_util import digest, world_scan

F32 = np.float32

# ---- kNN grid box (rebuild_grid) ---------------------------------------------------------------------------------


def grid_box(map_lo, map_hi, cell_size):
    """The box the device kNN grid covers after it was built over a map with bounding box [map_lo, map_hi]: the box plus
    a margin of a whole number of cells, max(2 cells, 5 % of the extent), in float32 as rebuild_grid computes it."""
    cs = F32(cell_size)
    lo, hi = np.empty(3, F32), np.empty(3, F32)
    for k in range(3):
        ext = F32(F32(map_hi[k]) - F32(map_lo[k]))
        m = F32(cs * F32(np.ceil(F32(max(F32(2.0) * cs, F32(0.05) * ext) / cs))))
        lo[k] = F32(map_lo[k]) - m
        hi[k] = F32(map_hi[k]) + m
    return lo, hi


def takes_full_path(grid_lo, grid_hi, pts):
    """flb_map_add_points rebuilds everything (full path) when a new point lies outside the grid box."""
    return bool((pts.min(0) < grid_lo).any() or (pts.max(0) > grid_hi).any())


class GridBox:
    """Follows the device grid box over a sequence of calls: it is rebuilt over the live points by an upload, by every
    delete and by a full-path add, and left as it is by an incremental add."""

    def __init__(self, map_xyz, cell_size):
        self.cell = cell_size
        self.rebuilt(map_xyz)

    def rebuilt(self, live):
        self.lo, self.hi = grid_box(live.min(0), live.max(0), self.cell)

    def add(self, batch, live_after):
        """Whether adding `batch` takes the full path; `live_after` is the map it leaves."""
        full = takes_full_path(self.lo, self.hi, batch)
        if full:
            self.rebuilt(live_after)
        return full


# ---- the reference's Add_Points, point by point ----------------------------------------------------------------------


def voxel_box(p, ds):
    """Box and centre of the downsample voxel of p, in float32 as ikd_Tree.cpp:392-400 computes them."""
    ds = F32(ds)
    mn = (np.floor(F32(p) / ds).astype(F32) * ds).astype(F32)
    mx = (mn + ds).astype(F32)
    mid = (mn.astype(np.float64) + (mx - mn).astype(np.float64) / 2.0).astype(F32)
    return mn, mx, mid


def calc_dist(a, mid):
    d = (np.asarray(a, F32) - mid).astype(F32)
    return ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]).astype(F32)


def add_points_model(map_xyz, new_xyz, ds):
    """Add_Points(new, downsample = true) on a tree holding map_xyz.  Returns (points, ambiguous): `ambiguous` lists
    the new points whose result depends on the order in which the tree's box search returns points of equal distance
    to the voxel centre (the reference does not define it, so such inputs cannot be pinned)."""
    pts = [np.asarray(map_xyz, F32).reshape(-1, 3)]
    live = pts[0].copy()
    ambiguous = []
    for i, p in enumerate(np.asarray(new_xyz, F32)):
        mn, mx, mid = voxel_box(p, ds)
        inb = np.all((mn <= live) & (mx > live), axis=1)
        store = live[inb]
        dp = calc_dist(p, mid)
        result = p
        if len(store):
            d = calc_dist(store, mid)
            j = int(np.argmin(d))
            if d[j] < dp:
                result = store[j]
                ties = store[d == d[j]]
                if (ties != ties[0]).any():
                    ambiguous.append(i)
        if len(store) > 1 or result is p:
            live = np.concatenate([live[~inb], result[None, :]])
    return live, ambiguous


# ---- voxel-boundary sets -------------------------------------------------------------------------------------------

VOX_DS = (0.1, 0.15, 0.2, 0.3, 0.4, 0.5)
VOX_CENTRES = {"o": (0.0, 0.0, 0.0), "m50": (50.0, -50.0, 50.0), "m200": (-200.0, 200.0, -200.0)}
VOX_CELL = 0.6          # cell size of the handle the sets are replayed on (flb.Handle's default)


def _ulps(a, k):
    a = np.asarray(a, F32).copy()
    for _ in range(int(abs(k))):
        a = np.nextafter(a, F32(np.inf) if k > 0 else F32(-np.inf)).astype(F32)
    return a


def _lattice_points(rng, c, ds, n, span=3, interior=0.4):
    """n points on the k*ds lattice around voxel c moved by -2..2 ulps per axis, a share of them jittered into the
    voxel instead."""
    ds32 = F32(ds)
    out = np.empty((n, 3), F32)
    for i in range(n):
        k = c + rng.integers(-span, span + 1, 3)
        p = (k.astype(F32) * ds32).astype(F32)
        if rng.random() < interior:
            p = (p + rng.uniform(0.0, ds, 3).astype(F32)).astype(F32)
        else:
            p = np.array([_ulps(p[a], rng.integers(-2, 3)) for a in range(3)], F32)
        out[i] = p
    return out


def _mirror_ties(rng, pts, ds, n):
    """Points at exactly the same float distance from their voxel centre as a point of `pts` (reflections through the
    centre along some axes that survive the float rounding), in the same voxel."""
    out = []
    for q in pts[rng.permutation(len(pts))]:
        mn, mx, mid = voxel_box(q, ds)
        if not np.all((mn <= q) & (mx > q)):
            continue
        for axes in ((0,), (1,), (0, 2), (0, 1, 2)):
            r = q.copy()
            for a in axes:
                r[a] = F32(F32(2.0) * mid[a] - q[a])
            rmn, _, _ = voxel_box(r, ds)
            if (r != q).any() and (rmn == mn).all() and calc_dist(r, mid) == calc_dist(q, mid):
                out.append(r)
                break
        if len(out) == n:
            break
    return np.array(out, F32).reshape(-1, 3)


def vox_case(ds, centre, single=False):
    """One voxel-boundary set: (map, batch, sentinel).  `single`: a batch that only touches voxels holding exactly one
    existing point which is closer to the centre than every new point in it (Add_Points then changes nothing)."""
    seed = int(round(ds * 1000)) * 7919 + sum(ord(ch) for ch in centre) * 31 + (1 if single else 0)
    rng = np.random.default_rng(seed)
    c = np.round(np.array(VOX_CENTRES[centre]) / ds).astype(np.int64)
    ds32 = F32(ds)
    # two anchors well outside the lattice make the map box (and so the grid box) cover it
    anchors = np.array([(c - 6).astype(F32) * ds32 + F32(0.37) * ds32, (c + 6).astype(F32) * ds32 + F32(0.61) * ds32], F32)
    if single:
        ks = np.unique(c + rng.integers(-3, 4, (40, 3)), axis=0)[:24]
        near = (ks.astype(F32) * ds32 + F32(0.5) * ds32 + rng.uniform(-0.05, 0.05, ks.shape).astype(F32) * ds32).astype(F32)
        mp = np.concatenate([near, anchors])
        new = []
        for k, q in zip(ks, near):
            for _ in range(3):
                p = (k.astype(F32) * ds32 + rng.uniform(0.0, 1.0, 3).astype(F32) * ds32).astype(F32)
                new.append(p)
            new.append(np.array([_ulps(F32(k[a]) * ds32, 1) for a in range(3)], F32))   # a corner, still its own voxel
        new = np.array(new, F32)
        keep = []
        for p in new:
            mn, mx, mid = voxel_box(p, ds)
            inb = np.all((mn <= mp) & (mx > mp), axis=1)
            if inb.sum() == 1 and calc_dist(mp[inb][0], mid) < calc_dist(p, mid):
                keep.append(p)
        batch = np.array(keep, F32)
    else:
        mp = np.unique(_lattice_points(rng, c, ds, 60), axis=0)
        mp = np.concatenate([mp[rng.permutation(len(mp))], anchors])
        new = _lattice_points(rng, c, ds, 120)
        dup_map = mp[rng.choice(len(mp) - 2, 6, replace=False)]                 # exact copies of existing points
        dup_new = new[rng.choice(len(new), 6, replace=False)]                   # duplicates within the batch
        ties = np.concatenate([_mirror_ties(rng, mp[:-2], ds, 4), _mirror_ties(rng, new, ds, 4)])
        batch = np.concatenate([new, dup_map, dup_new, ties])
        batch = batch[rng.permutation(len(batch))]
    # drop what makes the reference's result depend on its traversal order (equal distances in one box search)
    for _ in range(len(batch) + len(mp)):
        _, amb = add_points_model(mp, batch, ds)
        if not amb:
            break
        batch = np.delete(batch, amb[0], axis=0)
    else:
        raise AssertionError("could not make the set unambiguous")
    glo, ghi = grid_box(mp.min(0), mp.max(0), VOX_CELL)
    assert not takes_full_path(glo, ghi, batch)
    sentinel = np.array([_ulps(ghi[0], 64), c[1] * ds32 + F32(0.5) * ds32, c[2] * ds32 + F32(0.5) * ds32], F32)
    return mp.astype(F32), batch.astype(F32), sentinel


def vox_names():
    names = [f"vox_{centre}_{ds}" for ds in VOX_DS for centre in VOX_CENTRES]
    names += [f"vox1_o_{ds}" for ds in VOX_DS]
    return names


def vox_case_by_name(name):
    kind, centre, ds = name.split("_")
    return vox_case(float(ds), centre, single=(kind == "vox1"))


# ---- moving sensor -------------------------------------------------------------------------------------------------

TRAJ_DS = (0.3, 0.2)
TRAJ_CELL = 0.6                     # C2's cell size
FOV = dict(cube_len=120.0, det_range=20.0, mov_threshold=1.5)
TRAJ_X = (0.0, 5.0, 15.0, 30.0, 45.0, 59.0, 73.0, 87.0, 101.0, 115.0, 129.0, 143.0, 157.0, 169.0, 150.0, 130.0, 115.0)
TRAJ_WINDOW = 20.0                  # half side of the square around the sensor a frame observes
TRAJ_N = 12000                      # points per frame
TRAJ_KNN_EVERY = 4
TRAJ_LIO_STEPS = (2, 4)             # after an incremental step and after a full one


class FovSegment:
    """lasermap_fov_segment (src/laserMapping.cpp:363-421) with fixed cube_len / DET_RANGE / MOV_THRESHOLD: the local
    map box follows the sensor, and the slabs it leaves behind are the boxes handed to Delete_Point_Boxes."""

    def __init__(self, cube_len, det_range, mov_threshold):
        self.cube_len, self.det, self.mov = cube_len, F32(det_range), F32(mov_threshold)
        self.lo = self.hi = None

    def step(self, pos):
        if self.lo is None:
            self.lo = np.array([pos[i] - self.cube_len / 2.0 for i in range(3)], F32)
            self.hi = np.array([pos[i] + self.cube_len / 2.0 for i in range(3)], F32)
            return np.zeros((0, 6), F32)
        thr = F32(self.mov * self.det)
        d0 = np.array([abs(pos[i] - float(self.lo[i])) for i in range(3)], F32)
        d1 = np.array([abs(pos[i] - float(self.hi[i])) for i in range(3)], F32)
        if not ((d0 <= thr) | (d1 <= thr)).any():
            return np.zeros((0, 6), F32)
        mov_dist = F32(max((self.cube_len - 2.0 * float(thr)) * 0.5 * 0.9, float(self.det * (self.mov - F32(1)))))
        nlo, nhi, boxes = self.lo.copy(), self.hi.copy(), []
        for i in range(3):
            blo, bhi = self.lo.copy(), self.hi.copy()
            if d0[i] <= thr:
                nlo[i] -= mov_dist
                nhi[i] -= mov_dist
                blo[i] = self.hi[i] - mov_dist
                boxes.append(np.concatenate([blo, bhi]))
            elif d1[i] <= thr:
                nlo[i] += mov_dist
                nhi[i] += mov_dist
                bhi[i] = self.lo[i] + mov_dist
                boxes.append(np.concatenate([blo, bhi]))
        self.lo, self.hi = nlo, nhi
        return np.array(boxes, F32).reshape(-1, 6)


def _surfaces(room_half, room_h):
    """(axis, value, lo2, hi2) rectangles: the C2 room's six faces and a corridor beyond its +x wall."""
    L, H = room_half, room_h
    x1 = L + 1.2 * 2 * L
    rects = [(2, 0.0, (-L, -L), (L, L)), (2, H, (-L, -L), (L, L)),
             (0, -L, (-L, 0.0), (L, H)), (0, L, (-L, 0.0), (L, H)),
             (1, -L, (-L, 0.0), (L, H)), (1, L, (-L, 0.0), (L, H)),
             (2, 0.0, (L, -6.0), (x1, 6.0)), (2, 4.0, (L, -6.0), (x1, 6.0)),
             (1, -6.0, (L, 0.0), (x1, 4.0)), (1, 6.0, (L, 0.0), (x1, 4.0)),
             (0, x1, (-6.0, 0.0), (6.0, 4.0))]
    return rects


def _observe(rng, rects, pos, w, n):
    """n points on the surfaces inside the square |x - px|, |y - py| <= w (sigma = 5 mm along the normal)."""
    clip = []
    for ax, val, lo2, hi2 in rects:
        o = [a for a in range(3) if a != ax]
        lo = np.array(lo2, float)
        hi = np.array(hi2, float)
        for j, a in enumerate(o):
            if a < 2:
                lo[j] = max(lo[j], pos[a] - w)
                hi[j] = min(hi[j], pos[a] + w)
        if ax < 2 and abs(val - pos[ax]) > w:
            continue
        if (hi > lo).all():
            clip.append((ax, val, lo, hi, float(np.prod(hi - lo))))
    area = np.array([c[4] for c in clip])
    cnt = np.floor(n * area / area.sum()).astype(int)
    cnt[np.argmax(cnt)] += n - cnt.sum()
    out = []
    for (ax, val, lo, hi, _), k in zip(clip, cnt):
        o = [a for a in range(3) if a != ax]
        p = np.empty((k, 3))
        p[:, ax] = val + rng.normal(0.0, 0.005, k)
        p[:, o] = rng.uniform(lo, hi, (k, 2))
        out.append(p)
    pts = np.concatenate(out)
    return pts[rng.permutation(len(pts))].astype(F32)


def traj_case(f):
    """A sensor walking out of the C2 room along +x, about 1.5 room sides into a corridor, and part of the way back.
    Per frame: (delete boxes, world points, kNN queries or None).  The first frames stay inside the mapped volume
    (incremental path), the walk out keeps seeing past the grid box (full path), and on the way back the sensor sees
    the part the deletes freed (full path after the box shrank)."""
    rng = np.random.default_rng(11)
    cfg = f["cfg"]
    area = 1.12 * cfg.n_map * cfg.pitch * cfg.pitch                  # the room side synth.make_frame chose
    L = max((-4 * cfg.room_h + np.sqrt(16 * cfg.room_h ** 2 + 8 * area)) / 4, 6.0) / 2
    rects = _surfaces(L, cfg.room_h)
    fov = FovSegment(**FOV)
    frames = []
    for i, x in enumerate(TRAJ_X):
        pos = (x, float(f["p_true"][1]), float(f["p_true"][2]))
        boxes = fov.step(pos)
        pts = _observe(rng, rects, pos, TRAJ_WINDOW, TRAJ_N)
        q = None
        if i % TRAJ_KNN_EVERY == TRAJ_KNN_EVERY - 1:
            near = pts[np.abs(pts[:, 0] - x) < 12.0]
            q = (near[rng.integers(0, len(near), 2000)] + rng.normal(0, 0.1, (2000, 3))).astype(F32)
        frames.append((boxes, pts, q))
    return frames


def delete_all_case(f):
    """Two boxes that together cover the whole map (Delete_Point_Boxes would empty it) and the batch added after."""
    lo, hi = f["map_xyz"].min(0), f["map_xyz"].max(0)
    mid = F32(0.5) * (lo[0] + hi[0])
    boxes = np.array([[lo[0] - 1, lo[1] - 1, lo[2] - 1, mid, hi[1] + 1, hi[2] + 1],
                      [mid, lo[1] - 1, lo[2] - 1, hi[0] + 1, hi[1] + 1, hi[2] + 1]], F32)
    return boxes, world_scan(f)


# ---- input digests ---------------------------------------------------------------------------------------------------


def traj_input_digest(frames):
    arrs = []
    for boxes, pts, q in frames:
        arrs += [boxes, pts] + ([q] if q is not None else [])
    return digest(*arrs)


def vox_input_digest(mp, batch, sentinel):
    return digest(mp, batch, sentinel)
