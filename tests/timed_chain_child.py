"""Child process of tests/test_gpu_timed_chain.py (not collected by pytest).

ORCVIO_TRI_OVERLAP and ORCVIO_TRI_OVERLAP_MIN are read once per process, so the test runs this script once per
setting of the two knobs and compares what each run writes:

    python timed_chain_child.py <workloads.pkl> <out.npz>

workloads.pkl holds the Monte-Carlo sequences (generated once by the parent).  The frame workloads are rebuilt here
from their seeds."""
import os
import pickle
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

from orcvio_b200 import api, montecarlo as mc, synth  # noqa: E402

NOISE_VAR = 1.6e-5
TRI = dict(cost_threshold=1e-3, init_final_dist_threshold=100.0)
# (n_clones, n_features, max_track_len, full_tracks): below and above the overlap threshold of the default setting
FRAMES = [(20, 300, 6, False), (12, 60, 6, True), (20, 200, 12, False), (30, 2600, 12, False)]
FRAME_KEYS = ("P", "delta_x", "status", "gamma", "positions", "clones")


def main(pkl, out_path):
    out = {}
    for (n, nf, m, full) in FRAMES:
        snap = synth.stress_snapshot(n, nf, m, seed=0, full_tracks=full)
        r = api.snapshot_update(snap, flags=0, noise_var=NOISE_VAR, translation_threshold=-1.0, **TRI)
        for k in FRAME_KEYS:
            out[f"snap_{n}_{nf}_{m}_{int(full)}_{k}"] = r[k]
    # the graph replay of a resident frame
    snap = synth.stress_snapshot(20, 300, 6, seed=0)
    fr = api.Frame(20, 0, NOISE_VAR, 0.95, -1.0, TRI["cost_threshold"], TRI["init_final_dist_threshold"])
    fr.load(snap)
    fr.run(3)
    out["graph_replays"] = np.array(fr.graph_replays())
    r = fr.fetch_last()
    for k in ("P", "delta_x", "status", "gamma", "clones"):
        out[f"graph_{k}"] = r[k]
    # multi-trajectory replays (MSCKF on unity.yaml, hybrid + ZUPT on euroc.yaml)
    with open(pkl, "rb") as fh:
        work = pickle.load(fh)
    for name, (cfg, seqs, ids, threads) in work.items():
        for t in threads:
            rec, info = mc.run_replay(cfg, seqs, ids, n_threads=t)
            out[f"{name}_t{t}_rec"] = rec
            out[f"{name}_t{t}_poses"] = info["poses"]
            out[f"{name}_t{t}_feature_updates"] = np.array(info["feature_updates"])
            out[f"{name}_t{t}_kernel_launches"] = np.array(info["kernel_launches"])
    np.savez(out_path, **out)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
