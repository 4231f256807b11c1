"""GPU parity tests of the individual stages on frozen windows, through the C ABI.

Stage 1 (triangulation) must agree with the oracle BIT FOR BIT (positions, validity flags,
LM iteration counts).  Stages 2/4/5 are compared through basis-invariant quantities with the
tolerances of SURVEY Appendix C: gamma 1e-9 rel, gate booleans identical, delta_x and P
1e-9 relative (the BASELINE.json criterion)."""
import numpy as np
import pytest

from orcvio_b200 import api, synth
import helpers as H

pytestmark = pytest.mark.gpu


def _cam_poses(snap):
    N = snap["n_clones"]
    Rbc = snap["R_b2c"]
    cam_R = np.zeros((N, 9))
    cam_t = np.zeros((N, 3))
    for c in range(N):
        R = snap["clone_R"][c].reshape(3, 3)
        cam_R[c] = (R @ Rbc.T).ravel()
        cam_t[c] = snap["clone_p"][c] + R @ snap["t_c_b"]
    return cam_R, cam_t


@pytest.mark.parametrize("n_clones,n_feat,max_len,full", [(20, 300, 6, False), (30, 500, 6, False),
                                                           (12, 60, 6, True)])
def test_triangulation_bit_exact(n_clones, n_feat, max_len, full):
    snap = synth.stress_snapshot(n_clones, n_feat, max_len, seed=3, full_tracks=full)
    cam_R, cam_t = _cam_poses(snap)
    tri = dict(cost_threshold=1e-4, init_final_dist_threshold=50.0)   # make some features fail
    pos, st, it, cost = api.triangulate(cam_R, cam_t, snap["feat_off"], snap["obs_clone"], snap["obs_z"],
                                        -1.0, tri["cost_threshold"], tri["init_final_dist_threshold"])
    from oracle import feature as ofeat
    cfg = ofeat.default_opt_config()
    cfg.translation_threshold = -1.0
    cfg.cost_threshold = tri["cost_threshold"]
    cfg.init_final_dist_threshold = tri["init_final_dist_threshold"]
    fo = snap["feat_off"]
    n_valid = 0
    for f in range(n_feat):
        idx = range(fo[f], fo[f + 1])
        Rs = [[float(x) for x in cam_R[snap["obs_clone"][k]]] for k in idx]
        ts = [[float(x) for x in cam_t[snap["obs_clone"][k]]] for k in idx]
        zs = [(float(snap["obs_z"][k][0]), float(snap["obs_z"][k][1])) for k in idx]
        res = ofeat.triangulate(Rs, ts, zs, False, [0.0, 0.0, 0.0], cfg)
        assert bool(st[f] & 1) == res.valid, f"validity differs for feature {f}"
        assert (it[f][0], it[f][1]) == (res.n_outer, res.n_inner_total), f"LM iteration counts differ ({f})"
        assert cost[f] == res.total_cost, f"final cost differs bitwise ({f})"
        if res.valid:
            n_valid += 1
            assert tuple(pos[f]) == tuple(res.position), f"position differs bitwise ({f})"
    assert 0 < n_valid <= n_feat


@pytest.mark.parametrize("flags", [0, H.FL_LARVIO, H.FL_LEFT])
def test_measurement_jacobians(flags):
    snap = synth.stress_snapshot(20, 80, 6, seed=5)
    sigma2 = 1e-4
    vio = H.oracle_from_snapshot(snap, flags, sigma2, tri=dict(cost_threshold=1e3, init_final_dist_threshold=1e3))
    rng = np.random.default_rng(0)
    nf = len(snap["feat_off"]) - 1
    # plausible 3-D points: triangulate with the oracle, perturb a little
    pos = np.zeros((nf, 3))
    for f in range(nf):
        ft = vio.map_server[f]
        assert vio._initialize(ft, None)
        pos[f] = ft.position + rng.normal(0, 0.01, 3)
        ft.position = pos[f].copy()
    Hx, He, Hf, r = api.measurement_jacobians(snap["clone_R"], snap["clone_p"], snap["R_b2c"], snap["t_c_b"],
                                              pos, snap["feat_off"], snap["obs_clone"], snap["obs_z"], flags)
    fo = snap["feat_off"]
    for f in range(nf):
        for k in range(fo[f], fo[f + 1]):
            hx, he, hf, rr = vio.measurementJacobian_msckf(int(snap["obs_clone"][k]), vio.map_server[f])
            np.testing.assert_allclose(Hx[k], hx, rtol=1e-12, atol=1e-13)
            np.testing.assert_allclose(He[k], he, rtol=1e-12, atol=1e-13)
            np.testing.assert_allclose(Hf[k], hf, rtol=1e-12, atol=1e-13)
            np.testing.assert_allclose(r[k], rr, rtol=1e-12, atol=1e-13)


def _compare_update(snap, flags, sigma2, tri, out, ref):
    assert np.array_equal(out["status"] & 1, ref["status"] & 1), "triangulation validity differs"
    valid = (ref["status"] & 1) == 1
    np.testing.assert_array_equal(out["positions"][valid], ref["positions"][valid])
    g_ok = valid
    rel = np.abs(out["gamma"][g_ok] - ref["gamma"][g_ok]) / np.maximum(np.abs(ref["gamma"][g_ok]), 1e-300)
    assert rel.max() < 1e-9, f"gamma rel err {rel.max()}"
    assert np.array_equal(out["status"] & 2, ref["status"] & 2), "gate decisions differ"
    assert (ref["status"] & 2).sum() > 0
    # posterior
    dx_ref = ref["delta_x"]
    assert np.abs(out["delta_x"] - dx_ref).max() <= 1e-9 * np.abs(dx_ref).max()
    P_ref = ref["P"]
    assert np.abs(out["P"] - P_ref).max() <= 1e-9 * np.abs(P_ref).max()
    assert np.abs(out["P"] - out["P"].T).max() == 0.0


@pytest.mark.parametrize("flags,n_clones,n_feat,max_len,full", [
    (0, 20, 300, 6, False),
    (H.FL_LARVIO, 20, 60, 6, False),      # fewer rows than columns: no-compression case
    (H.FL_LEFT, 30, 800, 6, False),
    (0, 10, 40, 6, True),                 # long tracks (m = N): wide-window path
    (0, 30, 2000, 6, False),
])
def test_snapshot_update(flags, n_clones, n_feat, max_len, full):
    snap = synth.stress_snapshot(n_clones, n_feat, max_len, seed=11, full_tracks=full)
    sigma2 = 0.002 ** 2 * 4
    tri = dict(cost_threshold=1e-3, init_final_dist_threshold=100.0)
    out = api.snapshot_update(snap, flags=flags, noise_var=sigma2, translation_threshold=-1.0,
                              cost_threshold=tri["cost_threshold"],
                              init_final_dist_threshold=tri["init_final_dist_threshold"])
    ref = H.oracle_snapshot_update(snap, flags, sigma2, tri=dict(translation_threshold=-1.0, **tri))
    _compare_update(snap, flags, sigma2, tri, out, ref)
    # clone poses after the state increment
    vio = ref["vio"]
    for c in range(n_clones):
        np.testing.assert_allclose(out["clones"][c][:9].reshape(3, 3), vio.clones[c].orientation, atol=1e-12)
        np.testing.assert_allclose(out["clones"][c][9:], vio.clones[c].position, rtol=0, atol=1e-11)
