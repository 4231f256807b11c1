"""CPU tests of the filter-consistency surface: the NumPy NEES restatement (tests/nees_oracle.py) on known answers and
against the filter's own retraction, the chi-square bounds the ANEES is judged by, the truth records of the synthetic
sequences, the all_gather of the NEES rows (world size 2 over gloo), and the device entry point without a device."""
import math
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy import stats

from oracle import mathutils as mu
import nees_oracle as tm
from orcvio_b200 import api, montecarlo as mc, synth

BLOCKS = [(0, 3, [0, 1, 2]), (1, 3, [3, 4, 5]), (2, 3, [6, 7, 8]), (3, 6, [0, 1, 2, 6, 7, 8]),
          (4, 9, list(range(9))), (5, 15, list(range(15)))]      # (column, dof, indices in [theta, v, p, bg, ba])


def _state17(rng):
    R = mu.so3_exp(rng.normal(0, 1.0, 3))
    q = synth._quat_xyzw(R)
    return np.concatenate([[12.5], rng.normal(0, 3, 3), q, rng.normal(0, 1, 3), rng.normal(0, 0.01, 3),
                           rng.normal(0, 0.05, 3)])


def _retract(x17, dx, left):
    """incrementState_IMUCam (oracle/filter.py) on a state record: the estimate x17 moved by the error state dx."""
    R = tm._q2R(x17[4:8])
    Rt = mu.so3_exp(dx[0:3])
    Rn = Rt @ R if left else R @ Rt
    y = x17.copy()
    y[4:8] = synth._quat_xyzw(Rn)
    y[8:11] += dx[3:6]
    y[1:4] += dx[6:9]
    y[11:14] += dx[9:12]
    y[14:17] += dx[12:15]
    return y


def _spd(rng, scale):
    A = rng.normal(0, 1, (15, 15))
    return (A @ A.T / 15 + np.eye(15)) * np.outer(scale, scale)


SCALE = np.array([0.02] * 3 + [0.1] * 3 + [0.3] * 3 + [0.002] * 3 + [0.02] * 3)


def test_nees_known_answers():
    rng = np.random.default_rng(1)
    est = _state17(rng)
    sig = np.array([0.01, 0.02, 0.03, 0.1, 0.2, 0.3, 0.5, 0.6, 0.7, 1e-3, 2e-3, 3e-3, 0.01, 0.02, 0.03])
    P = np.diag(sig ** 2)
    d = rng.normal(0, 1, 15) * sig * 0.7
    gt = _retract(est, d, left=True)
    row = tm.nees_row(est, gt, P, left=True)
    r = d ** 2 / sig ** 2
    for col, dof, idx in BLOCKS:
        assert abs(row[col] - r[idx].sum()) <= 1e-10 * r[idx].sum()
    assert abs(row[6] - np.degrees(np.linalg.norm(d[:3]))) <= 1e-10
    assert abs(row[7] - np.linalg.norm(d[6:9])) <= 1e-12
    # a rotation error Exp(a) applied under either convention is recovered, also near pi (the symmetric-part branch)
    for a in (np.array([1e-9, -2e-9, 3e-10]), np.array([0.3, -0.2, 0.1]), np.array([1.5, 1.0, -1.2]),
              np.array([0.0, 0.0, 3.1]), np.array([1.7, -1.7, 1.7])):
        R_est = tm._q2R(est[4:8])
        for left in (True, False):
            R = mu.so3_exp(a) @ R_est if left else R_est @ mu.so3_exp(a)
            g = est.copy()
            g[4:8] = synth._quat_xyzw(R)
            # (the quaternion round trip of R costs ~1e-16 per entry: compare the error vector directly too)
            np.testing.assert_allclose(tm.so3_log(mu.so3_exp(a)), a, rtol=0, atol=1e-12)
            np.testing.assert_allclose(tm.error_state(est, g, left)[:3], a, rtol=0, atol=1e-12)


def test_round_trip_through_the_filter_retraction():
    rng = np.random.default_rng(2)
    for left in (True, False):
        for _ in range(20):
            est = _state17(rng)
            P = _spd(rng, SCALE)
            dx = np.linalg.cholesky(P) @ rng.normal(0, 1, 15)
            gt = _retract(est, dx, left)
            e = tm.error_state(est, gt, left)
            np.testing.assert_allclose(e, dx, rtol=0, atol=1e-12)
            row = tm.nees_row(est, gt, P, left)
            for col, dof, idx in BLOCKS:
                ref = dx[idx] @ np.linalg.solve(P[np.ix_(idx, idx)], dx[idx])
                assert abs(row[col] - ref) <= 1e-9 * max(ref, 1.0)


def test_nees_statistics_inside_chi2_bounds():
    rng = np.random.default_rng(3)
    n = 20000
    est = _state17(rng)
    P = _spd(rng, SCALE)
    L = np.linalg.cholesky(P)
    rows = np.zeros((n, 8))
    for k in range(n):
        left = bool(k & 1)
        dx = L @ rng.normal(0, 1, 15)
        rows[k] = tm.nees_row(est, _retract(est, dx, left), P, left)
    for col, dof, _ in BLOCKS:
        lo = stats.chi2.ppf(0.0005, n * dof) / n
        hi = stats.chi2.ppf(0.9995, n * dof) / n
        assert lo <= rows[:, col].mean() <= hi, (col, rows[:, col].mean(), lo, hi)


def test_oracle_nan_rows_and_summary():
    rng = np.random.default_rng(4)
    n, F = 5, 3
    est = np.stack([[_state17(rng) for _ in range(F)] for _ in range(n)])
    gt = est + 1e-3
    gt[..., 4:8] = est[..., 4:8]
    cov = np.stack([[_spd(rng, SCALE) for _ in range(F)] for _ in range(n)])
    cov[1, 0, 4, 4] = -1.0                                  # not positive definite
    gt[2, 1, 3] = np.inf
    rows, summ = tm.nees(est, gt, cov, 0)
    assert np.all(np.isnan(rows[1, 0])) and np.all(np.isnan(rows[2, 1]))
    assert np.isfinite(rows).sum() == (n * F - 2) * 8
    np.testing.assert_array_equal(summ[:, 8], [4, 4, 5])
    np.testing.assert_allclose(summ[2, :6], rows[:, 2, :6].mean(axis=0), rtol=1e-15)


@pytest.mark.parametrize("dof", [3, 6, 9, 15, 768, 3840, 15360])
def test_chi2_quantile_matches_scipy(dof):
    for p in (0.025, 0.975):
        ref = stats.chi2.ppf(p, dof)
        assert abs(api.chi2_quantile(p, dof) - ref) <= 1e-9 * ref
    if dof <= 15:                                          # the ANEES bounds of a block of this dof over 256 runs
        lo, hi = api.anees_bounds(256, dof)
        assert lo < dof < hi
        assert abs(lo - stats.chi2.ppf(0.025, 256 * dof) / 256) <= 1e-9 * lo
        assert abs(hi - stats.chi2.ppf(0.975, 256 * dof) / 256) <= 1e-9 * hi


def test_truth_states_reproduce_the_sequence_truth():
    for cfg, ov in (("euroc", {}), ("unity", dict(if_ZUPT_valid=0)), ("kitti_odom", {})):
        spec = synth.SynthSpec(config=cfg, seed=3, n_frames=6, feats_per_frame=20, n_landmarks=500, overrides=ov)
        seq = synth.make_sequence(spec)
        t = np.array([g[0] for g in seq["gt"]])
        tr = synth.truth_states(spec, t)
        for f, (tg, p, q) in enumerate(seq["gt"]):
            assert tr[f, 0] == tg
            np.testing.assert_array_equal(tr[f, 1:4], p)
            np.testing.assert_array_equal(tr[f, 4:8], q)
        np.testing.assert_array_equal(tr[:, 11:14], np.tile(spec.gyro_bias, (len(t), 1)))
        np.testing.assert_array_equal(tr[:, 14:17], np.tile(spec.acc_bias, (len(t), 1)))
        # truth velocity: the derivative of the truth position
        h = 1e-4
        pp = synth.truth_states(spec, t + h)[:, 1:4]
        pm = synth.truth_states(spec, t - h)[:, 1:4]
        np.testing.assert_allclose(tr[:, 8:11], (pp - pm) / (2 * h), rtol=0, atol=1e-5)
        # the sequence itself is what it was: a second generation gives the same arrays
        again = synth.make_sequence(spec)
        np.testing.assert_array_equal(again["imu"], seq["imu"])
        for (ta, fa), (tb, fb) in zip(again["frames"], seq["frames"]):
            assert ta == tb
            np.testing.assert_array_equal(fa, fb)


def test_sequences_unchanged_by_the_trajectory_helper():
    """make_sequence builds its trajectory through synth._trajectory, which draws nothing from the random stream: the
    generator's state after the IMU stream is what an untouched stream gives, and a known value of the stream pins it."""
    spec = synth.SynthSpec(config="unity", seed=5, n_frames=3, feats_per_frame=10, n_landmarks=300,
                           overrides=dict(if_ZUPT_valid=0))
    seq = synth.make_sequence(spec)
    base = synth.configs.make("unity", if_ZUPT_valid=0)
    traj = synth._trajectory(spec, base)
    rng = np.random.default_rng(1005)
    dt = 1.0 / float(base["imu_rate"])
    sg = spec.imu_noise_scale * float(base["noise_gyro"]) / math.sqrt(dt)
    sa = spec.imu_noise_scale * float(base["noise_acc"]) / math.sqrt(dt)
    for i in range(len(seq["imu"])):
        t = spec.t0 - 0.01 + i * dt
        _, _, _, w, f = traj.kinematics(t)
        np.testing.assert_array_equal(seq["imu"][i, 1:4], w + np.array(spec.gyro_bias) + rng.normal(0, sg, 3))
        np.testing.assert_array_equal(seq["imu"][i, 4:7], f + np.array(spec.acc_bias) + rng.normal(0, sa, 3))


def _worker(rank, world, port, n_traj, n_frames, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mine = mc.shard(n_traj, rank, world)
    rows = np.zeros((len(mine), n_frames, 8))
    for k, t in enumerate(mine):
        rows[k] = t + 0.01 * np.arange(n_frames * 8).reshape(n_frames, 8)
        if t == 3:
            rows[k, 1] = np.nan
    out = mc.gather_nees(rows, mine, n_traj, rank, world)
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_gather_nees_world2_gloo():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    n_traj, n_frames, world = 7, 5, 2
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_traj, n_frames, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    ref = np.stack([t + 0.01 * np.arange(n_frames * 8).reshape(n_frames, 8) for t in range(n_traj)])
    ref[3, 1] = np.nan
    for r in range(world):
        assert results[r].shape == (n_traj, n_frames, 8)
        np.testing.assert_array_equal(results[r], ref)
    single = mc.gather_nees(ref[[2, 0, 1, 3, 6, 4, 5]], [2, 0, 1, 3, 6, 4, 5], n_traj, 0, 1)
    np.testing.assert_array_equal(single, ref)


def test_trajectory_nees_without_a_device():
    L = api.lib()
    if L.orcvio_device_count() > 0:
        pytest.skip("a CUDA device is present")
    e = np.zeros((1, 1, 17))
    c = np.eye(15).reshape(1, 1, 225)
    out = np.zeros(8)
    s = np.zeros(9)
    rc = L.orcvio_trajectory_nees(api._dp(e), api._dp(e), api._dp(np.ascontiguousarray(c)), 1, 1, 0, api._dp(out),
                                  api._dp(s))
    assert rc == -1                                        # ORCVIO_ERR_NO_DEVICE: no CPU fallback
    assert L.orcvio_nees_summary(api._dp(np.zeros(8)), 1, 1, api._dp(s)) == -1
    with pytest.raises(RuntimeError):
        api.trajectory_nees(e, e, c.reshape(1, 1, 15, 15), 0)
