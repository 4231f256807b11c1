"""GPU: the frame chain as bench.py times it.

Two paths of the frame update are not the one the other tests take:
- From the third orcvio_frame_run after a load, every run replays one CUDA graph of the resident chain (restore copies,
  both streams, the fork / join events, the PDL launches).  Inside the graph the triangulation epoch is a constant and
  the completion flags are cleared by a memset node.
- A phase with at least ORCVIO_TRI_OVERLAP_MIN (2400) candidates runs k_jac_gate candidate by candidate behind
  k_triangulate (epoch-stamped release flags, polls in the Jacobian kernel, the large-track kernel launched with PDL
  behind the small-track one).

Here the overlapped update is checked against the oracle with the bars of test_gpu_stages, graph replays against a
plain run bit for bit (Frame.fetch_last reads what a replay left on the device), the forced and the disabled overlap
against each other in child processes (the knobs are read once per process), and the frame handle's state after the
end-to-end call."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from orcvio_b200 import api, montecarlo as mc, synth
import helpers as H

pytestmark = pytest.mark.gpu

# the benchmark's settings (bench.py: NOISE_VAR, TRI, make_frame)
NOISE_VAR = 1.6e-5
TRI = dict(cost_threshold=1e-3, init_final_dist_threshold=100.0)
OVERLAP_MIN = 2400              # default of ORCVIO_TRI_OVERLAP_MIN (csrc/batch.cu, Batch::launch_phase)
KNOBS = ("ORCVIO_TRI_OVERLAP", "ORCVIO_TRI_OVERLAP_MIN")
OUT_KEYS = ("P", "delta_x", "status", "gamma", "clones")


def _frame(n_clones, flags=0):
    return api.Frame(n_clones, flags, NOISE_VAR, 0.95, -1.0, TRI["cost_threshold"], TRI["init_final_dist_threshold"])


def _snap(n_clones, n_feat, max_len=6, full=False, seed=0):
    return synth.stress_snapshot(n_clones, n_feat, max_len, seed=seed, full_tracks=full)


def _ref(snap, flags=0):
    return api.snapshot_update(snap, flags=flags, noise_var=NOISE_VAR, translation_threshold=-1.0, **TRI)


def _same(out, ref, what):
    for k in OUT_KEYS:
        assert np.array_equal(out[k], ref[k]), f"{what}: {k} differs"


def _no_knobs():
    set_ = [k for k in KNOBS if k in os.environ]
    if set_:
        pytest.skip(f"{', '.join(set_)} set in the environment: the overlap threshold is not the default one")


@pytest.mark.parametrize("flags,n_clones,n_feat,max_len,full", [
    (0, 30, 4096, 6, False),              # the benchmark's stress frame
    (0, 30, OVERLAP_MIN - 1, 6, False),   # one candidate below the threshold: grid-wide dependency
    (0, 30, OVERLAP_MIN, 6, False),       # at the threshold: per-candidate flags
    (0, 30, 2600, 12, False),             # small- and large-track Jacobian lists, both behind k_triangulate
    (0, 12, OVERLAP_MIN, 6, True),        # full tracks: the large-track list alone
    (H.FL_LEFT, 30, OVERLAP_MIN, 6, False),
    (H.FL_LARVIO, 30, OVERLAP_MIN, 6, False),
])
def test_overlapped_update_matches_oracle(flags, n_clones, n_feat, max_len, full):
    _no_knobs()
    snap = _snap(n_clones, n_feat, max_len, full)
    out = _ref(snap, flags)
    ref = H.oracle_snapshot_update(snap, flags, NOISE_VAR, tri=dict(translation_threshold=-1.0, **TRI))
    valid = (ref["status"] & 1) == 1
    assert np.array_equal(out["status"] & 1, ref["status"] & 1), "triangulation validity differs"
    np.testing.assert_array_equal(out["positions"][valid], ref["positions"][valid])
    rel = np.abs(out["gamma"][valid] - ref["gamma"][valid]) / np.maximum(np.abs(ref["gamma"][valid]), 1e-300)
    assert rel.max() < 1e-9, f"gamma rel err {rel.max()}"
    assert np.array_equal(out["status"] & 2, ref["status"] & 2), "gate decisions differ"
    assert (ref["status"] & 2).sum() > 0
    dx_ref, P_ref = ref["delta_x"], ref["P"]
    assert np.abs(out["delta_x"] - dx_ref).max() <= 1e-9 * np.abs(dx_ref).max()
    assert np.abs(out["P"] - P_ref).max() <= 1e-9 * np.abs(P_ref).max()
    assert np.abs(out["P"] - out["P"].T).max() == 0.0
    vio = ref["vio"]
    for c in range(n_clones):
        np.testing.assert_allclose(out["clones"][c][:9].reshape(3, 3), vio.clones[c].orientation, atol=1e-12)
        np.testing.assert_allclose(out["clones"][c][9:], vio.clones[c].position, rtol=0, atol=1e-11)


# small frames first, so that every capture after the first one follows a growth of the scratch buffers
REPLAY_FRAMES = [(12, 60, 6, True), (20, 40, 6, False), (30, 2000, 6, False), (30, 2600, 12, False),
                 (30, 4096, 6, False)]


def test_graph_replay_equals_plain_run():
    frames = {}
    handles = {}
    for (n, nf, m, full) in REPLAY_FRAMES:
        snap = _snap(n, nf, m, full)
        other = _snap(n, max(nf // 2, 8), m, full, seed=1)
        frames[(n, nf, m, full)] = (snap, _ref(snap), other, _ref(other))
    for key in REPLAY_FRAMES:
        n = key[0]
        snap, ref, other, ref_o = frames[key]
        fr = handles.setdefault(n, _frame(n))            # one handle per window size, reused by the larger frames
        what = f"{key}"

        def launches(fn):
            l0 = fr.kernel_launches()
            fn()
            return fr.kernel_launches() - l0

        fr.load(snap)
        with pytest.raises(RuntimeError):
            fr.fetch_last()                              # nothing ran since the load
        d3 = launches(lambda: fr.run(3))                 # two plain runs, then the capture and its first launch
        assert fr.graph_replays() >= 1, f"{what}: run(3) did not replay a graph"
        _same(fr.fetch_last(), ref, f"{what} run(3)")
        g0 = fr.graph_replays()
        d5 = launches(lambda: fr.run(5))                 # repeated replays
        assert fr.graph_replays() == g0 + 5
        _same(fr.fetch_last(), ref, f"{what} run(5)")
        _same(fr.fetch(), ref, f"{what} fetch")          # a plain run after replays (advances the epoch)
        _same(fr.fetch_last(), ref, f"{what} fetch_last after fetch")
        d1 = launches(lambda: fr.run(1))                 # a replay after a plain run
        assert fr.graph_replays() == g0 + 6
        _same(fr.fetch_last(), ref, f"{what} run(1) after fetch")
        d2 = launches(lambda: fr.run(2, stages=True))    # profiled: plain runs
        assert fr.graph_replays() == g0 + 6
        _same(fr.fetch_last(), ref, f"{what} profiled run(2)")
        assert d1 > 0 and d5 == 5 * d1 and d3 == 3 * d1 and d2 == 2 * d1, (what, d1, d2, d3, d5)
        fr.load(other)                                   # the graph is dropped with the work lists
        assert fr.graph_replays() == 0
        fr.run(4)
        assert fr.graph_replays() >= 1
        _same(fr.fetch_last(), ref_o, f"{what} other frame run(4)")
        fr.load(snap)
        fr.run(4)
        assert fr.graph_replays() >= 1
        _same(fr.fetch_last(), ref, f"{what} reloaded run(4)")


def test_forced_and_disabled_overlap_give_the_same_bits(tmp_path):
    """The overlap changes only how k_jac_gate waits for k_triangulate: every phase overlapped
    (ORCVIO_TRI_OVERLAP_MIN=1), none (ORCVIO_TRI_OVERLAP=0) and the default give identical outputs on frame updates,
    a graph replay and multi-trajectory replays (MSCKF, and hybrid + ZUPT with its speculative triangulation)."""
    unity = mc.make_sequences("unity", list(range(5)), 40, 60, dict(if_ZUPT_valid=0), n_landmarks=3000)
    euroc = mc.make_sequences("euroc", list(range(4)), 75, 120, {}, n_landmarks=3000, workers=4)
    work = dict(unity=(H.write_cfg(unity[0]["cfg"]), unity, list(range(5)), (1, 2)),
                euroc=(H.write_cfg(euroc[0]["cfg"]), euroc, list(range(4)), (1,)))
    pkl = tmp_path / "work.pkl"
    with open(pkl, "wb") as fh:
        pickle.dump(work, fh)
    child = os.path.join(os.path.dirname(os.path.abspath(__file__)), "timed_chain_child.py")
    base = {k: v for k, v in os.environ.items() if k not in KNOBS}
    runs = {}
    for name, knob in (("default", {}), ("forced", {"ORCVIO_TRI_OVERLAP_MIN": "1"}),
                       ("disabled", {"ORCVIO_TRI_OVERLAP": "0"})):
        out = tmp_path / f"{name}.npz"
        flags = ["-s"] if sys.flags.no_user_site else []
        p = subprocess.run([sys.executable, *flags, child, str(pkl), str(out)], env={**base, **knob},
                           capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, f"{name} child failed:\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}"
        runs[name] = dict(np.load(out))
    ref = runs["default"]
    assert int(ref["graph_replays"]) >= 1
    for name in ("forced", "disabled"):
        assert sorted(runs[name]) == sorted(ref)
        for k in ref:
            assert np.array_equal(runs[name][k], ref[k]), f"{name}: {k} differs from the default run"


@pytest.mark.parametrize("n_clones,n_feat", [(20, 300), (30, 4096)])
def test_update_leaves_no_resident_frame(n_clones, n_feat):
    """orcvio_frame_update keeps its work lists in the per-feature form, which the resident chain cannot run: run and
    fetch are refused until the next load, fetch_last returns what the update computed."""
    snap = _snap(n_clones, n_feat)
    ref = _ref(snap)
    fr = _frame(n_clones)
    inp = fr.prepare_inputs(snap)
    fr.load(snap)
    fr.run(3)
    for full_P in (True, False):
        out = {k: (v.copy() if hasattr(v, "copy") else v) for k, v in fr.update(inp, full_P=full_P).items()}
        assert fr.graph_replays() == 0
        with pytest.raises(RuntimeError, match="orcvio_frame_run failed: -2"):
            fr.run(1)
        with pytest.raises(RuntimeError, match="orcvio_frame_fetch failed: -2"):
            fr.fetch()
        last = fr.fetch_last()
        if full_P:
            _same(out, ref, "update")
        else:
            np.testing.assert_array_equal(out["P_lead9"], ref["P"][:9, :9])
        _same(last, ref, f"fetch_last after update (full_P={full_P})")
    fr.load(snap)
    fr.run(3)
    _same(fr.fetch_last(), ref, "run after a new load")
    _same(fr.fetch(), ref, "fetch after a new load")
