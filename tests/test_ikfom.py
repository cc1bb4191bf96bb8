"""Row a8 (IKFoM-typed update, esekfom.hpp:1619-1928).  CPU tier: the oracle's manifold algebra
(round trips, consistency with the live 18-DoF path) and the product's device math compiled for the
host (bit-exact vs the oracle).  GPU tier: flb_lio_update_ikfom against the oracle."""
import ctypes as C

import numpy as np
import pytest

from conftest import bits
from golden_util import load_ref_golden


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _rand_state(po, f, rng):
    x = po.state_ikfom_from_frame(f)
    d = np.ascontiguousarray(rng.normal(size=23) * 0.05)
    po.lib().flo_ikfom_boxplus(C.byref(x), _p(d))
    return x


def test_oracle_boxplus_boxminus_round_trip(po, frames):
    f = frames("T0")
    rng = np.random.default_rng(0)
    L = po.lib()
    x = _rand_state(po, f, rng)
    for sc in (1e-9, 1e-5, 1e-2, 0.3):
        d = np.ascontiguousarray(rng.normal(size=23) * sc)
        y = x.copy()
        L.flo_ikfom_boxplus(C.byref(y), _p(d))
        r = np.zeros(23)
        L.flo_ikfom_boxminus(C.byref(y), C.byref(x), _p(r))
        np.testing.assert_allclose(r, d, rtol=1e-9, atol=1e-13)
        assert abs(np.linalg.norm(y.grav[:]) - 9.8090) < 1e-12          # stays on the sphere
        assert abs(np.linalg.norm(y.rot[:]) - 1) < 1e-12


def test_hostemu_manifold_math_bit_exact(hostemu, po, frames):
    f = frames("T0")
    rng = np.random.default_rng(1)
    L = po.lib()
    for sc in (0.0, 1e-12, 1e-6, 1e-2, 0.5):
        x = _rand_state(po, f, rng)
        y = _rand_state(po, f, rng)
        d = np.ascontiguousarray(rng.normal(size=23) * sc)
        xo = x.copy()
        L.flo_ikfom_boxplus(C.byref(xo), _p(d))
        xe = np.ascontiguousarray(x.vector())
        hostemu.emu_ikfom_boxplus(_p(xe), _p(d))
        assert (bits(xe) == bits(xo.vector())).all()
        ro, re = np.zeros(23), np.zeros(23)
        L.flo_ikfom_boxminus(C.byref(x), C.byref(y), _p(ro))
        hostemu.emu_ikfom_boxminus(_p(np.ascontiguousarray(x.vector())), _p(np.ascontiguousarray(y.vector())), _p(re))
        assert (bits(re) == bits(ro)).all()


def test_oracle_ikfom_update_consistent_with_live_path(po, frames):
    """Different filter (23-DoF, P re-projection) but the same measurements: with the extrinsic and gravity
    pinned by a tight prior the pose must agree with the live 18-DoF update to ~1e-4."""
    f = frames("T1")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    x = po.state_ikfom_from_frame(f)
    rep = lio.update_ikfom(po.ikfom_params(f, 4), x)
    x18 = po.state_from_frame(f)
    lio2 = po.Lio(f["map_xyz"], f["scan_body"])
    rep18 = lio2.update(po.lio_params(f, 4), x18, x18.copy())
    assert rep.passes == rep18.passes and rep.n_eff_last == rep18.n_eff_last
    assert np.linalg.norm(np.array(x.pos[:]) - x18.p) < 2e-4
    R = np.zeros(9)
    po.lib().flo_quat_to_R(_p(np.ascontiguousarray(x.rot[:])), _p(R))
    assert np.abs(R.reshape(3, 3) - x18.R).max() < 2e-4
    P = x.cov
    np.testing.assert_allclose(P, P.T, atol=1e-12)
    assert np.all(np.linalg.eigvalsh(P) > 0)
    assert np.all(np.diag(P)[:6] < np.diag(po.state_ikfom_from_frame(f).cov)[:6])


def test_oracle_ikfom_control_flow(po, frames):
    f = frames("T0")
    lio = po.Lio(f["map_xyz"], f["scan_body"])
    for T, passes in [(0, 1), (1, 2), (3, 4)]:
        x = po.state_ikfom_from_frame(f)
        rep = lio.update_ikfom(po.ikfom_params(f, T, limit=0.0), x)     # limit 0: never converges
        assert rep.passes == passes
        # kNN on the first pass and after i == maximum_iter - 2 (esekfom.hpp:1826-1829)
        assert rep.knn_passes == (1 if T == 0 else 2)


@pytest.mark.gpu
@pytest.mark.parametrize("name,T,limit", [("T0", 4, 0.001), ("T1", 4, 0.001), ("T1", 2, 0.0), ("T1", 10, 0.001), ("C2", 3, 0.001)])
def test_gpu_ikfom_update_parity(flb, po, name, T, limit):
    f = flb.synth.make_frame(name)
    if name == "C2":
        # at this size the CPU path takes its kNN from the reference's ikd-Tree: its result is pinned in
        # tests/golden/ref_ikdtree.npz (tests/golden/make_golden_ref.py, T = 3, limit = 0.001)
        gold = load_ref_golden()
        orep = tuple(int(v) for v in gold["ikfom_C2_report"])
        vo, co = gold["ikfom_C2_state"], gold["ikfom_C2_cov"]
    else:
        lio = po.Lio(f["map_xyz"], f["scan_body"])
        xo = po.state_ikfom_from_frame(f)
        r = lio.update_ikfom(po.ikfom_params(f, T, limit=limit), xo)
        orep = (r.passes, r.knn_passes, r.n_eff_last, r.rows_total, r.converged_last)
        vo, co = xo.vector(), xo.cov
    h = flb.Handle(device=0, cell_size=f["cfg"].cell_size)
    h.map_upload(f["map_xyz"])
    h.scan_upload(f["scan_body"])
    xg = flb.capi.StateIkfom()
    C.memmove(C.byref(xg), C.byref(po.state_ikfom_from_frame(f)), C.sizeof(xg))
    prm = flb.capi.IkfomParams()
    prm.laser_point_cov = f["cfg"].laser_point_cov
    prm.max_iteration = T
    prm.limit[:] = [limit] * 23
    grep = h.lio_update_ikfom(prm, xg)
    assert (grep.passes, grep.knn_passes, grep.n_eff_last, grep.rows_total, grep.converged_last) == orep
    vg = xg.vector()
    assert np.abs(vg - vo).max() / np.abs(vo).max() < 1e-9          # bar 1e-5
    # covariance: entries span 6 orders of magnitude; compare against the matrix scale
    assert np.abs(xg.cov - co).max() / np.abs(co).max() < 1e-6
    np.testing.assert_allclose(np.diag(xg.cov), np.diag(co), rtol=1e-6)
    h.close()
