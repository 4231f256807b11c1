"""GPU: every device and pinned buffer of the library (csrc/devmem.h) is released again.

Each entry runs once to warm up; then, after every one of ten more rounds, the bytes the library holds
(orcvio_device_bytes_held) must be exactly what they were after the warm-up.  The stage-level entries build and drop a
filter per call, and the Frame and Batch handles are created and destroyed inside the round, so a buffer that a
destructor misses shows up here."""
import numpy as np
import pytest

from orcvio_b200 import api, montecarlo as mc, synth
import helpers as H

pytestmark = pytest.mark.gpu

ROUNDS = 10
NOISE_VAR = 1.6e-5
TRI = dict(cost_threshold=1e-3, init_final_dist_threshold=100.0)


@pytest.fixture(scope="module")
def snap():
    return synth.stress_snapshot(30, 4096, 6, seed=0)


@pytest.fixture(scope="module")
def euroc():
    """Hybrid MSCKF / EKF-SLAM filters with ZUPT (euroc.yaml as shipped), a few frames each."""
    ids = [0, 1]
    seqs = mc.make_sequences("euroc", ids, 8, 120, {}, n_landmarks=1500)
    assert seqs[0]["cfg"]["max_features_in_one_grid"] > 0 and seqs[0]["cfg"]["if_ZUPT_valid"] == 1
    return H.write_cfg(seqs[0]["cfg"]), seqs


def _cam_poses(snap):
    Rbc = snap["R_b2c"]
    cam_R = np.stack([(R.reshape(3, 3) @ Rbc.T).ravel() for R in snap["clone_R"]])
    cam_t = np.stack([p + R.reshape(3, 3) @ snap["t_c_b"] for R, p in zip(snap["clone_R"], snap["clone_p"])])
    return cam_R, cam_t


def _held_bytes_return_to_baseline(run):
    run()
    base = api.device_bytes_held()
    for k in range(ROUNDS):
        run()
        held = api.device_bytes_held()
        assert held == base, f"round {k}: (device, pinned) bytes held {held}, after the warm-up {base}"


def test_triangulate_with_iterations_and_cost(snap):
    cam_R, cam_t = _cam_poses(snap)

    def run():
        _, _, it, _ = api.triangulate(cam_R, cam_t, snap["feat_off"], snap["obs_clone"], snap["obs_z"], -1.0, **TRI)
        assert it.any()
    _held_bytes_return_to_baseline(run)


def test_measurement_jacobians_and_snapshot_update(snap):
    cam_R, cam_t = _cam_poses(snap)
    pos = api.triangulate(cam_R, cam_t, snap["feat_off"], snap["obs_clone"], snap["obs_z"], -1.0, **TRI)[0]

    def run():
        api.measurement_jacobians(snap["clone_R"], snap["clone_p"], snap["R_b2c"], snap["t_c_b"], pos,
                                  snap["feat_off"], snap["obs_clone"], snap["obs_z"])
        api.snapshot_update(snap, noise_var=NOISE_VAR, translation_threshold=-1.0, **TRI)
    _held_bytes_return_to_baseline(run)


def test_frame_load_graph_runs_update_destroy(snap):
    def run():
        fr = api.Frame(30, 0, NOISE_VAR, 0.95, -1.0, TRI["cost_threshold"], TRI["init_final_dist_threshold"])
        fr.load(snap)
        fr.run(3)                          # the third run onwards replays the captured graph
        assert fr.graph_replays() > 0
        fr.update(snap)
        del fr
    _held_bytes_return_to_baseline(run)


def test_hybrid_zupt_batch(euroc):
    cfg, seqs = euroc

    def run():
        b = api.Batch(cfg, len(seqs))
        for j, s in enumerate(seqs):
            it = s["init"]
            b.set_initial_state(j, it["t"], it["quat"], it["pos"], it["vel"], it["bg"], it["ba"])
        _, ok, _, _ = b.replay_states(*mc.pack_replay(seqs, 8))
        assert ok.all()
        del b
    _held_bytes_return_to_baseline(run)


def test_chol_probe():
    rng = np.random.default_rng(0)
    M = rng.normal(size=(40, 40))
    A = M @ M.T + 40 * np.eye(40)
    _held_bytes_return_to_baseline(lambda: api.chol_probe(A, rng.normal(size=(8, 40)), reps=1))
