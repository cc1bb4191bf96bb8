"""Generate tests/golden/ref_ikdtree.npz: what the reference's own ikd-Tree (include/ikd-Tree/ikd_Tree.cpp, built into
oracle/_ref/libikdtree_ref.so by oracle/Makefile where the reference sources are present) returns on the cases of
tests/golden_util.py, and the CPU path that uses it for kNN at the full sizes C1..C4.  The tests compare against this
file, so they run wherever the repository is checked out.  Run from the repo root:  python tests/golden/make_golden_ref.py

Each case runs in a process of its own: every KD_TREE starts a background thread that is never joined, and processes
holding several trees have crashed.  Results too large to store (whole point sets, kNN of a full scan, float distances) are kept as
SHA-256 digests of the exact bits (golden_util.digest), beside their sizes.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import fastlivo_loader  # noqa: E402
from golden_util import add_points_case, delete_boxes_case, digest, knn_queries, rows_sorted, tie_lattice  # noqa: E402

CASES = (["knn_T0", "knn_T1", "knn5000_T1", "ties", "frame_C1", "frame_C2", "frame_C3", "frame_C4", "scanknn_C2",
          "add_T0_0.3", "add_T1_0.3", "add_T1_0.5", "add_C2_0.3", "delete_T1", "ikfom_C2"])


def run_case(case):
    flb = fastlivo_loader.load()
    po = fastlivo_loader.oracle()
    if case == "ties":
        lat, q = tie_lattice()
        ri, rd = po.IkdTreeRef(lat).knn(q)
        return {"ties_idx": ri, "ties_d2": rd}
    kind, name = case.split("_")[:2]
    f = flb.synth.make_frame(name)
    out = {}
    if kind in ("knn", "knn5000"):
        n, seed, sigma = (3000, 1, 0.25) if kind == "knn" else (5000, 17, 0.3)
        q = knn_queries(f["map_xyz"], np.random.default_rng(seed), n, sigma)
        ri, rd = po.IkdTreeRef(f["map_xyz"]).knn(q, nthreads=4)
        assert 0 <= ri.min() and ri.max() < 65536
        out[f"{case}_idx"] = ri.astype(np.uint16)          # every query has 5 neighbours; the maps hold < 65536 points
        out[f"{case}_d2_digest"] = np.array(digest(rd))
    elif kind == "frame":
        cfg = f["cfg"]
        lio = po.Lio(f["map_xyz"], f["scan_body"], po.IkdTreeRef(f["map_xyz"]))
        x = po.state_from_frame(f)
        lrep = lio.update(po.lio_params(f, cfg.lio_passes - 1, nthreads=8, early_stop=False), x, x.copy())
        out[f"{case}_lio_report"] = np.array([lrep.passes, lrep.knn_passes, lrep.n_eff_last, lrep.rows_total])
        if cfg.n_patch:
            vio = po.Vio(f["image"], f["patch_pos"], f["patch_ref"], f["patch_level"], f["cam"])
            vrep = vio.update(po.vio_params(f, cfg.vio_passes, early_stop=False, force_all_passes=True), x, x.copy())
            out[f"{case}_vio_report"] = np.array([*vrep.passes, vrep.rows_total])
            out[f"{case}_vio_last_error"] = np.array(list(vrep.last_error), np.float32)
        out[f"{case}_state"] = x.vector()
        out[f"{case}_cov"] = x.P
    elif kind == "scanknn":
        o = po.Lio(f["map_xyz"], f["scan_body"]).run_pass(po.lio_params(f, 2), f["R_prop"], f["p_prop"], True)
        ri, rd = po.IkdTreeRef(f["map_xyz"]).knn(o["world"], nthreads=8)
        ok = rd[:, 4] <= 5.0
        out[f"{case}_world_digest"] = np.array(digest(o["world"]))
        out[f"{case}_ok_digest"] = np.array(digest(ok))
        out[f"{case}_digest"] = np.array(digest(ri[ok], rd[ok]))
        out[f"{case}_n_ok"] = np.array(int(ok.sum()))
    elif kind == "add":
        ds = float(case.split("_")[2])
        tree = po.IkdTreeRef(f["map_xyz"])
        batches, q = add_points_case(f)
        counts, sets = [], []
        for b in batches:
            tree.add_points(b, ds)
            pts = tree.points()
            counts.append(len(pts))
            sets.append(digest(rows_sorted(pts)))
        ri, rd = tree.knn(q, nthreads=8)
        ok = rd[:, 4] <= 5.0
        out[f"{case}_counts"] = np.array(counts)
        out[f"{case}_set_digests"] = np.array(sets)
        out[f"{case}_n_ok"] = np.array(int(ok.sum()))
        out[f"{case}_ok_digest"] = np.array(digest(ok))
        out[f"{case}_d2_digest"] = np.array(digest(rd[ok]))
    elif kind == "delete":
        tree = po.IkdTreeRef(f["map_xyz"])
        n_del = tree.delete_boxes(delete_boxes_case(f))
        pts = tree.points()
        out[f"{case}_n_deleted"] = np.array(n_del)
        out[f"{case}_count"] = np.array(len(pts))
        out[f"{case}_set_digest"] = np.array(digest(rows_sorted(pts)))
    elif kind == "ikfom":
        lio = po.Lio(f["map_xyz"], f["scan_body"], po.IkdTreeRef(f["map_xyz"]))
        x = po.state_ikfom_from_frame(f)
        rep = lio.update_ikfom(po.ikfom_params(f, 3, limit=0.001), x)
        out[f"{case}_report"] = np.array([rep.passes, rep.knn_passes, rep.n_eff_last, rep.rows_total, rep.converged_last])
        out[f"{case}_state"] = x.vector()
        out[f"{case}_cov"] = x.cov
    return out


def main():
    if fastlivo_loader.oracle().ref_lib() is None:
        sys.exit("oracle/_ref/libikdtree_ref.so is not built: it needs the reference sources (see oracle/Makefile)")
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for case in CASES:
            part = os.path.join(tmp, case + ".npz")
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "--case", case, part])
            out.update(np.load(part))
    path = os.path.join(ROOT, "tests", "golden", "ref_ikdtree.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) == 4 and sys.argv[1] == "--case":
        np.savez(sys.argv[3], **run_case(sys.argv[2]))
        sys.stdout.flush()
        os._exit(0)          # skip the trees' destructors (they join a thread that never returns)
    main()
