"""CPU tier: the oracle itself, cross-checked in ways that do not depend on Eigen or on the
product (SURVEY.md §8c "Consequence / plan" (i)-(v))."""
import ctypes as C

import numpy as np
import pytest

from golden_util import digest, knn_queries, load_ref_golden


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("name", ["T0", "T1"])
def test_brute_knn_equals_reference_ikdtree(po, frames, name):
    """(i) our brute-force float32 kNN == the reference's own KD_TREE::Nearest_Search (its results on these queries
    are pinned in tests/golden/ref_ikdtree.npz)."""
    g = load_ref_golden()
    f = frames(name)
    q = knn_queries(f["map_xyz"], np.random.default_rng(1), 3000, 0.25)
    bi, bd = po.knn_brute(f["map_xyz"], q)
    assert (np.diff(bd, axis=1) > 0).all(), "fixture has distance ties"
    assert (bi == g[f"knn_{name}_idx"]).all()
    assert digest(bd) == g[f"knn_{name}_d2_digest"]


def test_plane_fit_vs_float64_least_squares(po, frames):
    """(ii) float32 QR plane vs float64 lstsq, within a conditioning-scaled bound."""
    f = frames("T1")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    o = lio.run_pass(po.lio_params(f, 3), f["R_prop"], f["p_prop"], True)
    rng = np.random.default_rng(2)
    checked = 0
    for i in rng.choice(len(o["nn_idx"]), 400, replace=False):
        if o["nn_idx"][i, 4] < 0:
            continue
        nb = f["map_xyz"][o["nn_idx"][i]].astype(np.float64)
        ok, pl = po.esti_plane(nb.astype(np.float32))
        x, *_ = np.linalg.lstsq(nb, -np.ones(5), rcond=None)
        n = np.linalg.norm(x)
        ref = np.concatenate([x / n, [1 / n]])
        cond = np.linalg.cond(nb)
        tol = 50 * cond * np.finfo(np.float32).eps
        assert np.abs(pl[:3] - ref[:3]).max() < tol
        assert abs(pl[3] - ref[3]) < tol * max(1.0, np.linalg.norm(nb, axis=1).max())
        checked += 1
    assert checked > 300


def test_lio_jacobian_vs_finite_differences(flb, po, frames):
    """(iii) H row = d(pd2)/d(delta) for R <- R Exp(d_rot), p <- p + d_pos (float64 FD)."""
    f = frames("T1")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    prm = po.lio_params(f, 3)
    R, p = f["R_prop"], f["p_prop"]
    o = lio.run_pass(prm, R, p, True)
    sel = o["sel_idx"][:200]
    pb = f["scan_body"][sel].astype(np.float64)
    pl = o["pabcd"][sel].astype(np.float64)

    def resid(Rm, pv):
        pw = (Rm @ (f["R_LI"] @ pb.T + f["t_LI"][:, None])).T + pv
        return (pl[:, :3] * pw).sum(1) + pl[:, 3]
    eps = 1e-6
    J = np.empty((len(sel), 6))
    for k in range(3):
        d = np.zeros(3)
        d[k] = eps
        J[:, k] = (resid(R @ flb.synth.exp_so3(d), p) - resid(R @ flb.synth.exp_so3(-d), p)) / (2 * eps)
        J[:, 3 + k] = (resid(R, p + d) - resid(R, p - d)) / (2 * eps)
    np.testing.assert_allclose(o["Hsub"][:200], J, rtol=1e-6, atol=1e-7)
    # measurement is -pd2 (src/laserMapping.cpp:1628)
    np.testing.assert_allclose(o["meas"][:200], -resid(R, p), atol=2e-5)


def test_ikfom_rows_contain_permuted_live_rows(po, frames):
    """(v) h_x = [n, A, B, C] (IKFoM) vs Hsub = [A, n] (live): same n and A."""
    f = frames("T1")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    o = lio.run_pass(po.lio_params(f, 3), f["R_prop"], f["p_prop"], True, rows12=True)
    np.testing.assert_allclose(o["h_x"][:, 0:3], o["Hsub"][:, 3:6], rtol=0, atol=0)
    np.testing.assert_allclose(o["h_x"][:, 3:6], o["Hsub"][:, 0:3], rtol=1e-12, atol=1e-15)
    perm = [3, 4, 5, 0, 1, 2]
    np.testing.assert_allclose(o["HTH12"][:6, :6][np.ix_(perm, perm)], o["HTH6"], rtol=1e-10)
    # C = R^T n has unit norm
    np.testing.assert_allclose(np.linalg.norm(o["h_x"][:, 9:12], axis=1), 1.0, atol=1e-6)


def test_ekf_step_equals_kalman_gain_form(flb, po, frames):
    """(iv) information form (src/laserMapping.cpp:1664-1672) == K = P H^T (H P H^T + sigma I)^-1."""
    f = frames("T0")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    prm = po.lio_params(f, 0, early_stop=False)       # T = 0: exactly one pass, then the covariance update
    x, xp = po.state_from_frame(f), po.state_from_frame(f)
    # make the prior differ from the linearisation point so `vec` is exercised
    xp.pos[0] += 0.01
    xp.rot[:] = (f["R_prop"] @ flb.synth.exp_so3(np.array([1e-3, -2e-3, 5e-4]))).ravel()
    o = lio.run_pass(prm, x.R, x.p, True)
    H = np.zeros((o["n"], 18))
    H[:, :6] = o["Hsub"]
    z = o["meas"]
    P = x.P
    sigma = prm.laser_point_cov
    K = P @ H.T @ np.linalg.inv(H @ P @ H.T + sigma * np.eye(o["n"]))
    vec = np.empty(18)
    po.lib().flo_state_boxminus(C.byref(xp), C.byref(x), _p(vec))
    sol = K @ (z - H @ vec) + vec
    P_new = (np.eye(18) - K @ H) @ P
    x_ref = x.copy()
    po.lib().flo_state_boxplus(C.byref(x_ref), _p(np.ascontiguousarray(sol)))
    rep = lio.update(prm, x, xp)
    assert rep.passes == 1
    np.testing.assert_allclose(x.vector(), x_ref.vector(), rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(x.P, P_new, rtol=1e-6, atol=1e-12)


def test_lio_update_control_flow(po, frames):
    """Pass / rematch schedule of SURVEY.md Appendix A with early stop disabled: T+1 passes, kNN on
    the first pass and after iterCount == T-2."""
    f = frames("T0")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    for T, passes, knn in [(0, 1, 1), (1, 2, 2), (2, 3, 2), (4, 5, 2)]:
        x = po.state_from_frame(f)
        rep = lio.update(po.lio_params(f, T, early_stop=False), x, x.copy())
        assert (rep.passes, rep.knn_passes) == (passes, knn), (T, rep.passes, rep.knn_passes)


def test_lio_update_converges_toward_truth(po, frames):
    f = frames("T1")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    x = po.state_from_frame(f)
    lio.update(po.lio_params(f, 4), x, x.copy())
    assert np.linalg.norm(x.p - f["p_true"]) < 0.5 * np.linalg.norm(f["p_prop"] - f["p_true"])
    ang = lambda R: np.linalg.norm(R - np.eye(3))
    assert ang(f["R_true"].T @ x.R) < 0.3 * ang(f["R_true"].T @ f["R_prop"])
    # covariance shrinks and stays symmetric positive
    P = x.P
    assert np.all(np.diag(P)[:6] < np.diag(f["cov"])[:6])
    np.testing.assert_allclose(P, P.T, atol=1e-12)


def test_vio_jacobian_vs_finite_differences(flb, po, frames):
    """(iii) photometric rows vs FD of the residual on a smooth image.  The analytic Jacobian uses a
    central-difference image gradient and ignores lens distortion, so agreement is ~percent-level."""
    f = dict(frames("T0"))
    h, w = f["image"].shape
    vv, uu = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    smooth = 128 + 50 * np.sin(uu / 37.0) * np.cos(vv / 29.0) + 40 * np.sin((uu + 2 * vv) / 53.0)
    img = np.clip(np.rint(smooth * 1.0), 0, 255).astype(np.uint8)
    vio = po.Vio(img, f["patch_pos"], f["patch_ref"], f["patch_level"], f["cam"])
    prm = po.vio_params(f, 3)
    R, p = f["R_true"], f["p_true"]
    level = 2          # coarse level: taps 4-8 px apart, quantisation noise of the uint8 image matters least
    o = vio.run_pass(prm, R, p, level)
    eps_r, eps_p = 2e-3, 2e-2

    def z_at(Rm, pv):
        return vio.run_pass(prm, Rm, pv, level)["z"]
    J = np.empty((len(o["z"]), 6))
    for k in range(3):
        d = np.zeros(3)
        d[k] = eps_r
        J[:, k] = (z_at(R @ flb.synth.exp_so3(d), p) - z_at(R @ flb.synth.exp_so3(-d), p)) / (2 * eps_r)
        d[k] = eps_p
        J[:, 3 + k] = (z_at(R, p + d) - z_at(R, p - d)) / (2 * eps_p)
    H = o["H_sub"]
    valid = np.abs(H).sum(1) > 0
    # compare column-wise in aggregate (per-pixel FD is noisy because of 8-bit quantisation)
    for c in range(6):
        a, b = H[valid, c], J[valid, c]
        corr = np.dot(a, b) / (np.linalg.norm(a) * np.linalg.norm(b))
        scale = np.dot(a, b) / np.dot(a, a)
        assert corr > 0.9, (c, corr)
        assert 0.8 < scale < 1.25, (c, scale)


def test_vio_update_reduces_photometric_error(po, frames):
    f = frames("T1")
    vio = po.Vio(f["image"], f["patch_pos"], f["patch_ref"], f["patch_level"], f["cam"])
    prm = po.vio_params(f, 4)
    e_prior = vio.run_pass(prm, f["R_prop"], f["p_prop"], 0)["error"]
    x = po.state_from_frame(f)
    rep = vio.update(prm, x, x.copy())
    e_post = vio.run_pass(prm, x.R, x.p, 0)["error"]
    assert rep.cov_updated == 1 and e_post < e_prior
    assert np.linalg.norm(x.p - f["p_true"]) < np.linalg.norm(f["p_prop"] - f["p_true"])


def test_vio_bounds_guard_and_empty(po, frames):
    """SURVEY.md §7 H5: patches whose tap footprint leaves the image are skipped and counted."""
    f = frames("T0")
    pos = f["patch_pos"].copy()
    vio = po.Vio(f["image"], pos, f["patch_ref"], f["patch_level"], f["cam"])
    prm = po.vio_params(f, 3)
    # rotate the camera away so every patch falls outside / behind
    Rbad = f["R_true"] @ np.array([[-1.0, 0, 0], [0, -1.0, 0], [0, 0, 1.0]])
    o = vio.run_pass(prm, Rbad, f["p_true"], 2)
    assert o["skipped"] == vio.Pn and o["n_meas"] == 0 and np.isnan(o["error"])
    assert not o["z"].any() and not o["H_sub"].any()
    # an update on such a frame must leave the state untouched (error is NaN -> reject branch)
    x = po.State18.make(Rbad, f["p_true"], cov=f["cov"])
    x0 = x.vector().copy()
    rep = vio.update(prm, x, x.copy())
    assert (x.vector() == x0).all() and rep.cov_updated == 0
    # zero patches: ComputeJ returns immediately (src/lidar_selection.cpp:969-970)
    v0 = po.Vio(f["image"], np.zeros((0, 3)), np.zeros((0, 192), np.float32), np.zeros(0, np.int32), f["cam"])
    x = po.state_from_frame(f)
    rep = v0.update(prm, x, x.copy())
    assert list(rep.passes) == [0, 0, 0]


def test_world2cam_distortion(po):
    cam = dict(width=640, height=512, fx=431.795259219, fy=431.550090267, cx=310.833037316, cy=266.985989326,
               d=(-0.0944205499243979, 0.0946727677776504, -0.00807970960613932, 8.07461209775283e-05, 0.0))
    # on the optical axis distortion vanishes
    np.testing.assert_allclose(po.world2cam(cam, [0, 0, 2.0]), [cam["cx"], cam["cy"]])
    px = po.world2cam(cam, [0.5, -0.3, 2.0])
    cam0 = dict(cam, d=(0, 0, 0, 0, 0))
    px0 = po.world2cam(cam0, [0.5, -0.3, 2.0])
    np.testing.assert_allclose(px0, [cam["fx"] * 0.25 + cam["cx"], cam["fy"] * -0.15 + cam["cy"]])
    assert 0.1 < np.linalg.norm(px - px0) < 5.0     # barrel distortion pulls the point inward by ~1 px
