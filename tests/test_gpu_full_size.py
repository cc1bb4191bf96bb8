"""GPU tier at BASELINE.json's full sizes (C1..C4): the whole frame against the CPU path (oracle +
the reference's ikd-Tree, its results pinned in tests/golden/ref_ikdtree.npz by tests/golden/make_golden_ref.py),
plus size-independent properties (sortedness, idempotence, symmetry)."""
import numpy as np
import pytest

from conftest import bits
from golden_util import digest, load_ref_golden

pytestmark = pytest.mark.gpu


def _frame_gpu(flb, h, f):
    cfg = f["cfg"]
    x = flb.capi.State18.from_frame(f)
    lrep = h.lio_update(flb.capi.lio_params(f, cfg.lio_passes - 1, early_stop=False), x, x.copy())
    vrep = None
    if cfg.n_patch:
        vrep = h.vio_update(flb.capi.vio_params(f, cfg.vio_passes, early_stop=False, force_all_passes=True), x, x.copy())
    return x, lrep, vrep


@pytest.mark.parametrize("name", ["C1", "C2", "C3", "C4"])
def test_full_size_frame_matches_cpu_path(flb, name):
    gold = load_ref_golden()
    key = f"frame_{name}"
    f = flb.synth.make_frame(name)
    cfg = f["cfg"]
    h = flb.Handle(device=0, cell_size=cfg.cell_size)
    h.load_frame(f)
    xg, lg, vg = _frame_gpu(flb, h, f)
    assert [lg.passes, lg.knn_passes, lg.n_eff_last, lg.rows_total] == list(gold[f"{key}_lio_report"])
    if vg is not None:
        assert [*vg.passes, vg.rows_total] == list(gold[f"{key}_vio_report"])
        np.testing.assert_allclose(list(vg.last_error), gold[f"{key}_vio_last_error"], rtol=1e-6)
    xo = gold[f"{key}_state"]
    rel = np.abs(xg.vector() - xo).max() / np.abs(xo).max()
    assert rel < 1e-9, rel                      # bar (north_star): 1e-5
    np.testing.assert_allclose(xg.P, gold[f"{key}_cov"], rtol=1e-6, atol=1e-14)
    # idempotence: the same update on the same inputs gives the same bits (deterministic reductions)
    xg2, _, _ = _frame_gpu(flb, h, f)
    assert (bits(xg2.vector()) == bits(xg.vector())).all() and (bits(xg2.P) == bits(xg.P)).all()
    # covariance stays symmetric and shrinks on the observed block
    P = xg.P
    np.testing.assert_allclose(P, P.T, atol=1e-10 * np.abs(P).max())
    assert np.all(np.diag(P)[:6] <= np.diag(f["cov"])[:6] * (1 + 1e-12))
    h.close()


def test_full_size_knn_and_pass_properties(flb, po):
    f = flb.synth.make_frame("C2")
    h = flb.Handle(device=0, cell_size=f["cfg"].cell_size)
    h.load_frame(f)
    prm = flb.capi.lio_params(f, 2)
    g = h.lio_pass(prm, f["R_prop"], f["p_prop"], True, width=12)
    ok = g["nn_idx"][:, 4] >= 0
    assert ok.mean() > 0.95
    d2 = g["nn_d2"][ok]
    assert (np.diff(d2, axis=1) >= 0).all() and (d2[:, 4] <= 5.0).all()          # sorted ascending, bounded
    # distances recomputed from the returned indices in float32, reference op order -> identical bits
    q = g["world"][ok][:, None, :]
    nb = f["map_xyz"][g["nn_idx"][ok]]
    d = (q - nb).astype(np.float32)
    rec = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    assert (bits(rec) == bits(d2)).all()
    # exactness against the reference's own ikd-Tree on the full scan (world points = the oracle's, bit for bit)
    gold = load_ref_golden()
    assert digest(g["world"]) == gold["scanknn_C2_world_digest"]
    assert ok.sum() == gold["scanknn_C2_n_ok"] and digest(ok) == gold["scanknn_C2_ok_digest"]
    assert digest(g["nn_idx"][ok].astype(np.int32), g["nn_d2"][ok].astype(np.float32)) == gold["scanknn_C2_digest"]
    # normal equations: symmetric, PSD, and consistent with the exported rows
    H = g["rows"]
    np.testing.assert_allclose(g["HTH"], H.T @ H, rtol=1e-10, atol=1e-9)
    np.testing.assert_allclose(g["HTh"], H.T @ g["meas"], rtol=1e-9, atol=1e-9)
    assert np.linalg.eigvalsh(g["HTH"]).min() > -1e-6
    # 6-wide layout is the permuted leading block of the 12-wide one
    g6 = h.lio_pass(prm, f["R_prop"], f["p_prop"], False, width=6)
    perm = [3, 4, 5, 0, 1, 2]
    np.testing.assert_allclose(g["HTH"][:6, :6][np.ix_(perm, perm)], g6["HTH"], rtol=1e-10)
    h.close()


def test_vio_pass_linearity_full_size(flb, po):
    """HTz is linear in the reference patches: z = I - P, so shifting every reference value by c shifts z by -c."""
    f = flb.synth.make_frame("C2")
    h = flb.Handle(device=0, cell_size=f["cfg"].cell_size)
    h.load_frame(f)
    prm = flb.capi.vio_params(f, 3)
    a = h.vio_pass(prm, f["R_prop"], f["p_prop"], 1)
    h.patches_upload(f["patch_pos"], f["patch_ref"] + np.float32(8.0), f["patch_level"])
    b = h.vio_pass(prm, f["R_prop"], f["p_prop"], 1)
    assert a["n_meas"] == b["n_meas"] == (len(f["patch_pos"]) - a["skipped"]) * 64
    np.testing.assert_allclose(b["z"], a["z"] - 8.0 * (np.abs(a["H_sub"]).sum(1) > 0), atol=1e-4)
    assert (bits(a["H_sub"]) == bits(b["H_sub"])).all()          # the Jacobian does not depend on the reference patch
    np.testing.assert_allclose(a["HTH6"], b["HTH6"], rtol=0, atol=0)
    h.close()
