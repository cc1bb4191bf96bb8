"""Generate tests/golden/ref_map_maintenance.npz: what the reference's own ikd-Tree (include/ikd-Tree/ikd_Tree.cpp, built
into oracle/_ref/libikdtree_ref.so by oracle/Makefile where the reference sources are present) does over a sequence of
map maintenance calls, on the cases of tests/map_cases.py:

  traj_<ds>     a sensor walking out of the C2 room and part of the way back: per frame Delete_Point_Boxes with the boxes
                lasermap_fov_segment cuts, then Add_Points(frame, downsample = true); counts and set digests after every
                call, kNN of 2000 queries every 4th frame, and which path (full / incremental) the device takes per add.
  vox_* vox1_*  small sets on downsample-voxel boundaries (points within 2 ulps of k * ds), at three magnitudes of
                coordinates and six ds: the resulting point sets in full, so a failing test can show the points.
  delete_all    a box set covering the whole map, and the add that follows on the intact map.

Every case runs in a process of its own (each KD_TREE starts a thread that is never joined) and twice: the two runs must
agree digest for digest, so a result that depends on the tree's background rebuild would be caught here.  The digest of
every case's inputs is stored too, so the tests notice when a builder in tests/map_cases.py no longer makes the inputs
these results were computed from.  The archive is written with fixed timestamps: rerunning reproduces it byte for byte.
Run from the repo root:  python tests/golden/make_golden_map.py
"""
import io
import os
import subprocess
import sys
import tempfile
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import fastlivo_loader  # noqa: E402
import map_cases as mc  # noqa: E402
from golden_util import digest, rows_sorted  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_map_maintenance.npz")
CASES = [f"traj_{ds}" for ds in mc.TRAJ_DS] + mc.vox_names() + ["delete_all"]


def run_case(case):
    flb = fastlivo_loader.load()
    po = fastlivo_loader.oracle()
    out = {}
    if case.startswith("traj_"):
        ds = float(case.split("_")[1])
        f = flb.synth.make_frame("C2")
        frames = mc.traj_case(f)
        tree = po.IkdTreeRef(f["map_xyz"])
        grid = mc.GridBox(f["map_xyz"], mc.TRAJ_CELL)
        n_del, counts_del, counts, sets, full, knn_steps, n_ok, ok_d, d2_d = [], [], [], [], [], [], [], [], []
        for i, (boxes, pts, q) in enumerate(frames):
            n_del.append(tree.delete_boxes(boxes) if len(boxes) else 0)
            m = tree.points()
            counts_del.append(len(m))
            if len(boxes):
                grid.rebuilt(m)
            tree.add_points(pts, ds)
            m = tree.points()
            counts.append(len(m))
            sets.append(digest(rows_sorted(m)))
            full.append(grid.add(pts, m))
            if q is not None:
                ri, rd = tree.knn(q, nthreads=8)
                ok = rd[:, 4] <= 5.0
                knn_steps.append(i)
                n_ok.append(int(ok.sum()))
                ok_d.append(digest(ok))
                d2_d.append(digest(rd[ok]))
        out.update({f"{case}_inputs": np.array(mc.traj_input_digest(frames)), f"{case}_n_deleted": np.array(n_del),
                    f"{case}_counts_after_delete": np.array(counts_del), f"{case}_counts": np.array(counts),
                    f"{case}_set_digests": np.array(sets), f"{case}_full_path": np.array(full),
                    f"{case}_knn_steps": np.array(knn_steps), f"{case}_n_ok": np.array(n_ok),
                    f"{case}_ok_digests": np.array(ok_d), f"{case}_d2_digests": np.array(d2_d)})
    elif case.startswith("vox"):
        ds = float(case.split("_")[2])
        mp, batch, sentinel = mc.vox_case_by_name(case)
        res = []
        for b in (batch, np.concatenate([batch, sentinel[None, :]])):
            tree = po.IkdTreeRef(mp)
            tree.add_points(b, ds)
            res.append(rows_sorted(tree.points()).view(np.float32).reshape(-1, 3))
        # the sentinel sits in a voxel of its own: with it the result differs by exactly that point
        assert digest(res[1]) == digest(rows_sorted(np.concatenate([res[0], sentinel[None, :]])).view(np.float32).reshape(-1, 3))
        model, amb = mc.add_points_model(mp, batch, ds)
        assert not amb and digest(rows_sorted(model)) == digest(rows_sorted(res[0])), "the float32 model disagrees"
        out.update({f"{case}_inputs": np.array(mc.vox_input_digest(mp, batch, sentinel)), f"{case}_result": res[0]})
    elif case == "delete_all":
        f = flb.synth.make_frame("T1")
        boxes, batch = mc.delete_all_case(f)
        tree = po.IkdTreeRef(f["map_xyz"])
        tree.add_points(batch, 0.3)                     # the device refuses the delete and keeps its map: so does this
        m = tree.points()
        n_del = po.IkdTreeRef(f["map_xyz"]).delete_boxes(boxes)
        out.update({f"{case}_inputs": np.array(digest(boxes, batch)), f"{case}_n_deleted": np.array(n_del),
                    f"{case}_add_count": np.array(len(m)), f"{case}_add_set_digest": np.array(digest(rows_sorted(m)))})
    return out


def _run(case, tmp, tag):
    part = os.path.join(tmp, f"{case}.{tag}.npz")
    subprocess.check_call([sys.executable, os.path.abspath(__file__), "--case", case, part])
    return dict(np.load(part))


def save_npz_reproducible(path, arrays):
    """np.savez_compressed, but with fixed member timestamps and order, so equal arrays give an identical file."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED) as z:
        for k in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(arrays[k]), allow_pickle=False)
            info = zipfile.ZipInfo(k + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            info.external_attr = 0o644 << 16
            z.writestr(info, buf.getvalue())


def main():
    if fastlivo_loader.oracle().ref_lib() is None:
        sys.exit("oracle/_ref/libikdtree_ref.so is not built: it needs the reference sources (see oracle/Makefile)")
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for case in CASES:
            a, b = _run(case, tmp, "a"), _run(case, tmp, "b")
            assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a), f"{case}: the reference is not deterministic"
            out.update(a)
    save_npz_reproducible(OUT, out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    if len(sys.argv) == 4 and sys.argv[1] == "--case":
        np.savez(sys.argv[3], **run_case(sys.argv[2]))
        sys.stdout.flush()
        os._exit(0)          # skip the trees' destructors (they join a thread that never returns)
    main()
