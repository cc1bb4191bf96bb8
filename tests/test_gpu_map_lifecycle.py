"""Map maintenance over a sequence of calls against the reference's own ikd-Tree (results pinned in
tests/golden/ref_map_maintenance.npz by tests/golden/make_golden_map.py, inputs built by tests/map_cases.py):

- a moving sensor (delete the boxes lasermap_fov_segment cuts, add the frame), through both paths of flb_map_add_points,
  with kNN, LIO and the nn_idx export checked on the maintained map;
- points within a few ulps of downsample-voxel boundaries, where float boxes of neighbouring voxels overlap or leave gaps;
- input strides, no-op calls, and a delete that would empty the map.

The last test runs without a GPU: the pinned inputs must still be what the builders make."""
import ctypes as C

import numpy as np
import pytest

import map_cases as mc
from conftest import bits
from golden_util import digest, rows_sorted, world_scan

GOLD_MAP = mc.__file__.replace("map_cases.py", "golden/ref_map_maintenance.npz")
STATE_RTOL = 1e-9          # as tests/test_gpu_parity.py

_gold = None


def gold():
    global _gold
    if _gold is None:
        _gold = dict(np.load(GOLD_MAP))
    return _gold


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def knn_check(h, q, n_ok, ok_digest, d2_digest):
    gi, gd = h.knn(q)
    m = h.map_download()
    ok = gd[:, 4] <= 5.0
    assert ok.sum() == n_ok and digest(ok) == ok_digest and digest(gd[ok]) == d2_digest
    d = (q[ok][:, None, :] - m[gi[ok]]).astype(np.float32)          # neighbour identity by coordinates
    rec = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    assert (bits(rec) == bits(gd[ok])).all()


def lio_check(flb, po, h, f, m):
    """flb_lio_update on the maintained map against the oracle built on the downloaded map, and the nn_idx export of a
    rematching pass indexing flb_map_download's order."""
    scan = f["scan_body"][::8]
    h.scan_upload(scan)
    lio = po.Lio(m, scan)
    xo, xpo = po.state_from_frame(f), po.state_from_frame(f)
    orep = lio.update(po.lio_params(f, 3), xo, xpo)
    xg, xpg = flb.capi.State18.from_frame(f), flb.capi.State18.from_frame(f)
    grep = h.lio_update(flb.capi.lio_params(f, 3), xg, xpg)
    assert (grep.passes, grep.knn_passes, grep.n_eff_last, grep.rows_total) == (orep.passes, orep.knn_passes, orep.n_eff_last, orep.rows_total)
    assert grep.n_eff_last > 1000
    assert rel(xg.vector(), xo.vector()) < STATE_RTOL
    assert rel(xg.P, xo.P) < 1e-7
    g = h.lio_pass(flb.capi.lio_params(f, 2), f["R_prop"], f["p_prop"], True)
    ok = g["nn_idx"][:, 4] >= 0
    assert ok.mean() > 0.5
    d = (g["world"][ok][:, None, :] - m[g["nn_idx"][ok]]).astype(np.float32)
    rec = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    assert (bits(rec) == bits(g["nn_d2"][ok])).all()


@pytest.fixture(scope="module")
def c2(flb):
    return flb.synth.make_frame("C2")


@pytest.mark.gpu
@pytest.mark.parametrize("persistent", [1, 0], ids=["persistent", "kernel-per-pass"])
@pytest.mark.parametrize("ds", mc.TRAJ_DS)
def test_trajectory_matches_reference_ikdtree(flb, po, c2, ds, persistent):
    g, key = gold(), f"traj_{ds}"
    frames = mc.traj_case(c2)
    assert mc.traj_input_digest(frames) == g[f"{key}_inputs"]
    h = flb.Handle(device=0, cell_size=c2["cfg"].cell_size, persistent=persistent)
    h.map_upload(c2["map_xyz"])
    grid = mc.GridBox(c2["map_xyz"], mc.TRAJ_CELL)
    knn_steps = list(g[f"{key}_knn_steps"])
    paths = []
    for i, (boxes, pts, q) in enumerate(frames):
        if len(boxes):
            h.map_delete_boxes(boxes)
            m = h.map_download()
            assert len(m) == g[f"{key}_counts_after_delete"][i]
            grid.rebuilt(m)
        h.map_add_points(pts, ds)
        m = h.map_download()
        assert len(m) == h.M == g[f"{key}_counts"][i], f"step {i}"
        assert digest(rows_sorted(m)) == g[f"{key}_set_digests"][i], f"step {i}"
        paths.append(grid.add(pts, m))
        if q is not None:
            j = knn_steps.index(i)
            knn_check(h, q, g[f"{key}_n_ok"][j], g[f"{key}_ok_digests"][j], g[f"{key}_d2_digests"][j])
        if i in mc.TRAJ_LIO_STEPS:
            lio_check(flb, po, h, c2, m)
    # the sequence exercises both paths of flb_map_add_points, as the fixture intends
    assert paths == list(g[f"{key}_full_path"])
    assert sum(paths) >= 2 and len(paths) - sum(paths) >= 2
    assert not paths[mc.TRAJ_LIO_STEPS[0]] and paths[mc.TRAJ_LIO_STEPS[1]]
    after_shrink = [i for i in range(1, len(frames)) if paths[i] and not paths[i - 1] and any(len(b) for b, _, _ in frames[:i])]
    assert after_shrink, "no full-path add after a delete shrank the box"
    h.close()


def _boxes_of(pts, ds):
    return [tuple(map(tuple, mc.voxel_box(p, ds)[:2])) for p in pts]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["incremental", "full"])
@pytest.mark.parametrize("name", mc.vox_names())
def test_voxel_boundaries_match_reference_ikdtree(flb, name, path):
    g = gold()
    ds = float(name.split("_")[2])
    mp, batch, sentinel = mc.vox_case_by_name(name)
    assert mc.vox_input_digest(mp, batch, sentinel) == g[f"{name}_inputs"]
    want = g[f"{name}_result"]
    if path == "full":
        batch = np.concatenate([batch, sentinel[None, :]])
        want = np.concatenate([want, sentinel[None, :]])
    h = flb.Handle(device=0, cell_size=mc.VOX_CELL)
    h.map_upload(mp)
    glo, ghi = mc.grid_box(mp.min(0), mp.max(0), mc.VOX_CELL)
    assert mc.takes_full_path(glo, ghi, batch) == (path == "full")
    h.map_add_points(batch, ds)
    got = h.map_download()
    h.close()
    a, b = set(map(bytes, rows_sorted(got))), set(map(bytes, rows_sorted(want)))
    if a != b or len(got) != len(want):
        only_dev = np.frombuffer(b"".join(sorted(a - b)), np.float32).reshape(-1, 3)
        only_ref = np.frombuffer(b"".join(sorted(b - a)), np.float32).reshape(-1, 3)
        lines = [f"{name} ({path}): device {len(got)} points, reference {len(want)}"]
        for tag, pts in (("only on the device", only_dev), ("only in the reference", only_ref)):
            for p, (mn, mx) in zip(pts, _boxes_of(pts, ds)):
                lines.append(f"  {tag}: {p.tolist()!r} float box [{mn!r}, {mx!r})")
        pytest.fail("\n".join(lines))


@pytest.mark.gpu
def test_add_points_strides_give_identical_maps(flb):
    f = flb.synth.make_frame("T1")
    batch = world_scan(f)
    out = []
    for stride in (3, 4, 12):
        wide = np.full((len(batch), stride), np.nan, np.float32)         # padding is never read
        wide[:, :3] = batch
        h = flb.Handle(device=0, cell_size=f["cfg"].cell_size)
        h.map_upload(f["map_xyz"])
        h.map_add_points(wide, 0.3)
        out.append(h.map_download())
        h.close()
    assert len(out[0]) == gold()["delete_all_add_count"]
    assert digest(rows_sorted(out[0])) == gold()["delete_all_add_set_digest"]
    for o in out[1:]:
        assert bits(o).shape == bits(out[0]).shape and (bits(o) == bits(out[0])).all()


@pytest.mark.gpu
def test_rejected_delete_and_noop_calls_leave_the_map_intact(flb):
    g = gold()
    f = flb.synth.make_frame("T1")
    boxes, batch = mc.delete_all_case(f)
    assert digest(boxes, batch) == g["delete_all_inputs"]
    assert g["delete_all_n_deleted"] == len(f["map_xyz"])            # the box set does cover the whole map
    h = flb.Handle(device=0, cell_size=f["cfg"].cell_size)
    h.map_upload(f["map_xyz"])
    q = (f["map_xyz"][np.random.default_rng(5).integers(0, len(f["map_xyz"]), 2000)] + np.float32(0.05)).astype(np.float32)
    m0, (i0, d0) = h.map_download(), h.knn(q)

    def unchanged():
        assert C.c_int(h.L.flb_map_size(h.h)).value == len(m0)
        assert (bits(h.map_download()) == bits(m0)).all()
        i1, d1 = h.knn(q)
        assert (i1 == i0).all() and (bits(d1) == bits(d0)).all()

    with pytest.raises(flb.FlbError) as e:
        h.map_delete_boxes(boxes)
    assert e.value.code == -4 and "empty map" in str(e.value)          # FLB_ERR_STATE
    unchanged()
    h.map_add_points(np.zeros((0, 3), np.float32), 0.3)
    unchanged()
    assert h.L.flb_map_delete_boxes(h.h, None, 0) == 0
    h.map_delete_boxes(np.zeros((0, 6), np.float32))
    unchanged()
    # the map still follows the reference after the refused delete
    h.map_add_points(batch, 0.3)
    m = h.map_download()
    assert len(m) == g["delete_all_add_count"] and digest(rows_sorted(m)) == g["delete_all_add_set_digest"]
    h.close()


def test_pinned_inputs_are_what_the_builders_make(flb):
    """No GPU: a change to a builder in tests/map_cases.py must not silently invalidate the pinned results."""
    g = gold()
    c2 = flb.synth.make_frame("C2")
    frames = mc.traj_case(c2)
    for ds in mc.TRAJ_DS:
        assert mc.traj_input_digest(frames) == g[f"traj_{ds}_inputs"]
    for name in mc.vox_names():
        assert mc.vox_input_digest(*mc.vox_case_by_name(name)) == g[f"{name}_inputs"], name
    t1 = flb.synth.make_frame("T1")
    assert digest(*mc.delete_all_case(t1)) == g["delete_all_inputs"]
