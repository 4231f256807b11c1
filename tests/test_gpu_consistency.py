"""GPU: filter consistency for the multi-trajectory batch.  The replay's per-frame state / covariance capture is exact and
changes nothing else; orcvio_trajectory_nees matches the NumPy restatement (tests/nees_oracle.py), is deterministic and
independent of how the samples are split; the Monte-Carlo path end to end."""
import numpy as np
import pytest

from oracle import mathutils as mu
import nees_oracle as tm
from orcvio_b200 import api, montecarlo as mc, synth
import helpers as H

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("config,ov", [("euroc", {}), ("unity", dict(if_ZUPT_valid=0))])
def test_capture_is_exact_and_non_intrusive(config, ov):
    ids = [0, 1, 2, 3]
    F = 40
    seqs = mc.make_sequences(config, ids, F, 120, ov, n_landmarks=3000)
    cfg = H.write_cfg(seqs[0]["cfg"])

    def batch():
        b = api.Batch(cfg, len(ids))
        for j, s in enumerate(seqs):
            it = s["init"]
            b.set_initial_state(j, it["t"], it["quat"], it["pos"], it["vel"], it["bg"], it["ba"])
        return b

    pack = mc.pack_replay(seqs, F)
    ba = batch()
    poses_a, ok_a = ba.replay(*pack)
    bb = batch()
    poses_b, ok_b, states, cov = bb.replay_states(*pack)
    np.testing.assert_array_equal(poses_b, poses_a)
    np.testing.assert_array_equal(ok_b, ok_a)
    assert np.all(ok_a == 1)
    assert bb.kernel_launches() == ba.kernel_launches() + F          # one k_capture_imu_cov per frame
    np.testing.assert_array_equal(states[..., 1:8], poses_a)
    # the same filters stepped frame by frame: the captured records are what Batch.state / Batch.cov read afterwards
    bc = batch()
    cursor = [0] * len(ids)
    for f in range(F):
        t_img, feats, feat_off, imu, imu_off = mc.pack_frame(seqs, f, cursor)
        used, pub = bc.process(t_img, feats, feat_off, imu, imu_off)
        for i in range(len(ids)):
            cursor[i] += int(used[i])
            np.testing.assert_array_equal(cov[i, f], bc.cov(i)[:15, :15])
            st = bc.state(i)
            assert states[i, f, 0] == st.time
            np.testing.assert_array_equal(states[i, f, 1:4], np.array(st.p))
            np.testing.assert_array_equal(states[i, f, 8:11], np.array(st.v))
            np.testing.assert_array_equal(states[i, f, 11:14], np.array(st.bg))
            np.testing.assert_array_equal(states[i, f, 14:17], np.array(st.ba))
            # (q is the quaternion of that R, already pinned bit for bit by poses_out; back to a matrix it is R up to the
            # rounding of the two conversions: a few ulps of a unit-norm entry)
            np.testing.assert_allclose(tm._q2R(states[i, f, 4:8]), np.array(st.R).reshape(3, 3), rtol=0, atol=4e-15)
    assert bc.kernel_launches() == ba.kernel_launches()             # replay = the frame loop, launch for launch
    # the NULL path of the new entry point is the plain replay
    bd = batch()
    poses_d, _, st_d, cv_d = bd.replay_states(*pack, states=False, cov=False)
    assert st_d is None and cv_d is None
    np.testing.assert_array_equal(poses_d, poses_a)
    assert bd.kernel_launches() == ba.kernel_launches()


def _random_inputs(rng, n, F, with_bad=True):
    scale = np.array([0.02] * 3 + [0.1] * 3 + [0.3] * 3 + [0.002] * 3 + [0.02] * 3)
    est = np.zeros((n, F, 17))
    gt = np.zeros((n, F, 17))
    cov = np.zeros((n, F, 15, 15))
    for i in range(n):
        for f in range(F):
            A = rng.normal(0, 1, (15, 15))
            P = (A @ A.T / 15 + np.eye(15)) * np.outer(scale, scale)
            cov[i, f] = P
            R = mu.so3_exp(rng.normal(0, 1.0, 3))
            est[i, f] = np.concatenate([[f * 0.05], rng.normal(0, 3, 3), synth._quat_xyzw(R), rng.normal(0, 1, 3),
                                        rng.normal(0, 0.01, 3), rng.normal(0, 0.05, 3)])
            dx = np.linalg.cholesky(P) @ rng.normal(0, 1, 15)
            g = est[i, f].copy()
            g[4:8] = synth._quat_xyzw(mu.so3_exp(dx[:3]) @ R)
            g[8:11] += dx[3:6]
            g[1:4] += dx[6:9]
            g[11:14] += dx[9:12]
            g[14:17] += dx[12:15]
            gt[i, f] = g
    # a rotation error near pi (the symmetric-part branch of the logarithm)
    gt[0, 0, 4:8] = synth._quat_xyzw(mu.so3_exp(np.array([0.3, -0.2, 3.0])) @ tm._q2R(est[0, 0, 4:8]))
    if with_bad:
        cov[1, 2, 4, 4] = -1.0                                  # not positive definite
        est[2, 3, 9] = np.inf
        cov[3, 1, 7, 2] = np.nan
    return est, gt, cov


def _assert_rows_close(a, b, rtol):
    assert np.array_equal(np.isnan(a), np.isnan(b))
    m = np.isfinite(b)
    np.testing.assert_allclose(a[m], b[m], rtol=rtol, atol=0)


def test_nees_kernel_matches_the_oracle():
    rng = np.random.default_rng(11)
    est, gt, cov = _random_inputs(rng, 37, 11)
    for flags in (0, 1, 2, 3):
        nees, summ = api.trajectory_nees(est, gt, cov, flags)
        ref, ref_s = tm.nees(est, gt, cov, flags)
        _assert_rows_close(nees, ref, 1e-10)
        assert np.isnan(nees[1, 2]).all() and np.isnan(nees[2, 3]).all() and np.isnan(nees[3, 1]).all()
        np.testing.assert_array_equal(summ[:, 8], ref_s[:, 8])
        _assert_rows_close(summ, ref_s, 1e-10)
    # the conventions differ: the left and right errors of the same pair are not the same vector
    assert not np.allclose(api.trajectory_nees(est, gt, cov, 0)[0][..., 0], api.trajectory_nees(est, gt, cov, 1)[0][..., 0])


def test_nees_is_deterministic_and_split_independent():
    rng = np.random.default_rng(12)
    n, F = 1024, 12
    e0, g0, c0 = _random_inputs(rng, 16, F, with_bad=False)
    reps = n // 16                                             # tile (cheap to generate) and perturb per trajectory
    est = np.tile(e0, (reps, 1, 1))
    gt = np.tile(g0, (reps, 1, 1))
    cov = np.tile(c0, (reps, 1, 1, 1))
    gt[:, :, 1:4] += rng.normal(0, 0.05, (n, F, 3))
    n1, s1 = api.trajectory_nees(est, gt, cov, 1)
    n2, s2 = api.trajectory_nees(est, gt, cov, 1)
    np.testing.assert_array_equal(n1, n2)
    np.testing.assert_array_equal(s1, s2)
    a, _ = api.trajectory_nees(est[:512], gt[:512], cov[:512], 1)
    b, _ = api.trajectory_nees(est[512:], gt[512:], cov[512:], 1)
    np.testing.assert_array_equal(np.concatenate([a, b]), n1)
    np.testing.assert_array_equal(api.nees_summary(np.concatenate([a, b])), s1)
    assert np.all(s1[:, 8] == n)


def test_run_replay_consistency_end_to_end():
    ids = list(range(16))
    seqs = mc.make_sequences("euroc", ids, 50, 120, {}, n_landmarks=3000, workers=4)
    cfg = H.write_cfg(seqs[0]["cfg"])
    rec, info = mc.run_replay(cfg, seqs, ids, n_threads=4, consistency=True)
    assert np.all(rec[:, 7] == 1.0)
    nees, summ = info["nees"], info["summary"]
    assert nees.shape == (16, 50, 8) and summ.shape == (50, 9)
    assert np.all(np.isfinite(nees)) and np.all(summ[:, 8] == 16)
    # truth at the estimates' own state times (an IMU stamp, not the image stamp)
    t_img = np.array([[t for t, _ in s["frames"][:50]] for s in seqs])
    assert np.all(np.abs(info["states"][:, :, 0] - t_img) < 0.05) and np.any(info["states"][:, :, 0] != t_img)
    ref, ref_s = tm.nees(info["states"], info["truth"], info["cov15"], api.nees_flags(seqs[0]["cfg"]))
    _assert_rows_close(nees, ref, 1e-10)
    _assert_rows_close(summ, ref_s, 1e-10)
    # the summary of the gathered rows (any world size) is the same bits
    np.testing.assert_array_equal(api.nees_summary(mc.gather_nees(nees, ids, 16, 0, 1)), summ)
    # and the default path is the plain replay
    rec0, info0 = mc.run_replay(cfg, seqs, ids, n_threads=4)
    np.testing.assert_array_equal(info0["poses"], info["poses"])
    assert info["kernel_launches"] == info0["kernel_launches"] + 50 * 4
