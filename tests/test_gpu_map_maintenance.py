"""GPU tier, SURVEY.md section 8 row f1: device-resident map maintenance against the reference's own ikd-Tree
(its results pinned in tests/golden/ref_ikdtree.npz by tests/golden/make_golden_ref.py): Add_Points(downsample = true)
(ikd_Tree.cpp:382-457) and Delete_Point_Boxes (:501-521)."""
import numpy as np
import pytest

from conftest import bits
from golden_util import add_points_case, delete_boxes_case, digest, load_ref_golden, rows_sorted

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,ds", [("T0", 0.3), ("T1", 0.3), ("T1", 0.5), ("C2", 0.3)])
def test_add_points_matches_reference_ikdtree(flb, name, ds):
    gold = load_ref_golden()
    key = f"add_{name}_{ds}"
    f = flb.synth.make_frame(name)
    h = flb.Handle(device=0, cell_size=f["cfg"].cell_size)
    h.map_upload(f["map_xyz"])
    batches, q = add_points_case(f)
    for b, n_ref, set_ref in zip(batches, gold[f"{key}_counts"], gold[f"{key}_set_digests"]):
        h.map_add_points(b, ds)
        got = h.map_download()
        assert len(got) == n_ref
        assert digest(rows_sorted(got)) == set_ref
    # the refreshed device grid answers kNN exactly like the refreshed reference tree
    gi, gd = h.knn(q)
    m = h.map_download()
    ok = gd[:, 4] <= 5.0
    assert ok.sum() == gold[f"{key}_n_ok"] > 1500
    assert digest(ok) == gold[f"{key}_ok_digest"]
    assert digest(gd[ok]) == gold[f"{key}_d2_digest"]
    # neighbour identity by coordinates (index spaces differ): distances recomputed from the returned neighbours
    got_nb = m[gi[ok]]
    d = (q[ok][:, None, :] - got_nb).astype(np.float32)
    rec = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    assert (bits(rec) == bits(gd[ok])).all()
    h.close()


def test_delete_boxes_matches_reference_ikdtree(flb, po):
    gold = load_ref_golden()
    f = flb.synth.make_frame("T1")
    h = flb.Handle(device=0)
    h.map_upload(f["map_xyz"])
    n_ref = int(gold["delete_T1_n_deleted"])
    h.map_delete_boxes(delete_boxes_case(f))
    got = h.map_download()
    assert n_ref > 100 and len(got) == gold["delete_T1_count"] == len(f["map_xyz"]) - n_ref
    assert digest(rows_sorted(got)) == gold["delete_T1_set_digest"]
    # LIO still runs on the pruned map and agrees with the oracle on the same point set
    h.scan_upload(f["scan_body"])
    lio = po.Lio(got, f["scan_body"])
    xo = po.state_from_frame(f)
    lio.update(po.lio_params(f, 3), xo, xo.copy())
    xg = flb.capi.State18.from_frame(f)
    h.lio_update(flb.capi.lio_params(f, 3), xg, xg.copy())
    assert np.abs(xg.vector() - xo.vector()).max() / np.abs(xo.vector()).max() < 1e-9
    h.close()


def test_map_maintenance_argument_errors(flb):
    h = flb.Handle(device=0)
    with pytest.raises(flb.FlbError) as e:
        h.map_add_points(np.zeros((3, 3), np.float32), 0.3)
    assert e.value.code == -4
    f = flb.synth.make_frame("T0")
    h.map_upload(f["map_xyz"])
    with pytest.raises(flb.FlbError) as e:
        h.map_add_points(np.full((3, 3), np.inf, np.float32), 0.3)
    assert e.value.code == -1
    with pytest.raises(flb.FlbError) as e:
        h.map_add_points(np.zeros((3, 3), np.float32), 0.0)
    assert e.value.code == -1
    h.close()
