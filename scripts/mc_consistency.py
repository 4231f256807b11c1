"""Filter consistency of the multi-trajectory replay: NEES / ANEES of the IMU state over many synthetic runs.

    python scripts/mc_consistency.py [--traj 256] [--frames 200] [--timing-traj 1024] [--pairs 3] [--out PATH]

For euroc.yaml as shipped (hybrid MSCKF / EKF-SLAM + ZUPT), unity.yaml with if_ZUPT_valid: 0 and kitti_odom.yaml as
shipped, `--traj` trajectories x `--frames` frames replay through orcvio_batch_replay_states; the truth is evaluated at
every estimate's own state time and orcvio_trajectory_nees gives the NEES per run and frame and the ANEES per frame.
Recorded per config and block: the ANEES per frame, the fraction of frames whose ANEES lies inside the two-sided 95 %
chi-square bounds chi2_quantile(0.025 | 0.975, N dof) / N, and the RMS orientation / position errors.  Then, on the
`--timing-traj` x `--frames` EuRoC leg: the wall time of orcvio_trajectory_nees on those samples, and the replay
throughput without and with the covariance capture, alternated (`--pairs` pairs).  The GPU name and power limit are read
in the same run.  Output: profiles/r3_mc_consistency.json (or --out).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from orcvio_b200 import api, configs, montecarlo as mc  # noqa: E402

CASES = (
    ("euroc", {}, 3000, "euroc.yaml as shipped: hybrid MSCKF / EKF-SLAM, feature ZUPT"),
    ("unity", dict(if_ZUPT_valid=0), 3000, "unity.yaml with if_ZUPT_valid: 0"),
    ("kitti_odom", {}, 6000, "kitti_odom.yaml as shipped"),
)
KITTI_NOTE = ("The KITTI-shaped synthetic tracks carry 0.002 feature noise (pixel level) while kitti_odom.yaml makes the "
              "filter assume sigma = 1 (noise_feature: 1): the visual updates are weighted far below their accuracy, "
              "so the NEES of this config is far below its bound by construction.")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None


def _per_frame(x):
    """A per-frame series as stored in the record: 6 significant digits."""
    return [float(f"{v:.6g}") for v in np.asarray(x, dtype=float)]


def write_record(path, out):
    """JSON with one line per key down to the blocks of a case: lists (the per-frame series) and the record of a block
    stay on the line of their key."""
    def fmt(o, ind):
        if isinstance(o, dict) and ind < 3:
            pad = " " * (ind + 1)
            items = [f"{pad}{json.dumps(k)}: {fmt(v, ind + 1)}" for k, v in o.items()]
            return "{\n" + ",\n".join(items) + "\n" + " " * ind + "}"
        return json.dumps(o)
    with open(path, "w") as fh:
        fh.write(fmt(out, 0) + "\n")


def write_cfg(cfg):
    return configs.write_yaml(os.path.join(tempfile.mkdtemp(prefix="orcvio_mcc_"), "cfg.yaml"), cfg)


def consistency_case(name, ov, n_landmarks, n_traj, n_frames, feats, workers):
    ids = list(range(n_traj))
    t0 = time.perf_counter()
    seqs = mc.make_sequences(name, ids, n_frames, feats, ov, n_landmarks=n_landmarks, workers=workers)
    t_gen = time.perf_counter() - t0
    cfg = write_cfg(seqs[0]["cfg"])
    rec, info = mc.run_replay(cfg, seqs, ids, n_threads=min(workers, n_traj), consistency=True)
    summ = info["summary"]
    nees = info["nees"]
    valid = summ[:, 8]
    blocks = {}
    for b, (bn, dof) in enumerate(api.NEES_BLOCKS):
        lo = np.array([api.anees_bounds(int(n), dof)[0] if n > 0 else np.nan for n in valid])
        hi = np.array([api.anees_bounds(int(n), dof)[1] if n > 0 else np.nan for n in valid])
        a = summ[:, b]
        inside = (a >= lo) & (a <= hi)
        # (the bounds depend on the number of valid runs only: one pair when every frame has the same number)
        bounds = [float(lo[0]), float(hi[0])] if np.all(valid == valid[0]) else [_per_frame(lo), _per_frame(hi)]
        blocks[bn] = dict(dof=dof, anees_per_frame=_per_frame(a), bound95=bounds,
                          fraction_of_frames_inside_95=float(np.mean(inside)),
                          fraction_of_frames_above=float(np.mean(a > hi)), fraction_of_frames_below=float(np.mean(a < lo)),
                          anees_median_over_frames=float(np.nanmedian(a)),
                          anees_mean_last_half=float(np.nanmean(a[len(a) // 2:])))
    return dict(
        config=name, overrides=ov, trajectories=n_traj, frames=n_frames, features_per_frame=feats,
        n_landmarks=n_landmarks, sequence_generation_s=t_gen, replay_s=info["seconds"],
        all_published=bool(np.all(rec[:, 7] == 1.0)), nees_flags=api.nees_flags(seqs[0]["cfg"]),
        valid_trajectories_per_frame_min=int(valid.min()), nonfinite_nees_rows=int(np.sum(~np.isfinite(nees[..., 5]))),
        blocks=blocks,
        rms_orientation_deg_per_frame=_per_frame(summ[:, 6]),
        rms_position_m_per_frame=_per_frame(summ[:, 7]),
        rms_orientation_deg_last=float(summ[-1, 6]), rms_position_m_last=float(summ[-1, 7]),
        ate_m_mean=float(rec[:, 5].mean()))


def timing_leg(n_traj, n_frames, feats, workers, pairs):
    ids = list(range(n_traj))
    seqs = mc.make_sequences("euroc", ids, n_frames, feats, {}, n_landmarks=3000, workers=workers)
    cfg = write_cfg(seqs[0]["cfg"])
    nw = min(n_traj, 2 * workers)
    mc.run_replay(cfg, seqs[:nw], ids[:nw], n_threads=min(workers, nw))                     # warm-up, both paths
    mc.run_replay(cfg, seqs[:nw], ids[:nw], n_threads=min(workers, nw), consistency=True)
    plain, capture = [], []
    info_c = None
    for _ in range(pairs):
        _, info_p = mc.run_replay(cfg, seqs, ids, n_threads=workers)
        plain.append(info_p["seconds"])
        _, info_c = mc.run_replay(cfg, seqs, ids, n_threads=workers, consistency=True)
        capture.append(info_c["seconds"])
        assert np.array_equal(info_p["poses"], info_c["poses"])
    flags = api.nees_flags(seqs[0]["cfg"])
    api.trajectory_nees(info_c["states"][:8], info_c["truth"][:8], info_c["cov15"][:8], flags)       # warm-up
    t_nees = []
    for _ in range(5):
        t0 = time.perf_counter()
        api.trajectory_nees(info_c["states"], info_c["truth"], info_c["cov15"], flags)
        t_nees.append(time.perf_counter() - t0)
    fps_p = [n_traj * n_frames / s for s in plain]
    fps_c = [n_traj * n_frames / s for s in capture]
    return dict(
        trajectories=n_traj, frames=n_frames, features_per_frame=feats, host_threads=workers,
        replay_plain_s=plain, replay_capture_s=capture,
        trajectory_frames_per_sec_plain=fps_p, trajectory_frames_per_sec_capture=fps_c,
        capture_cost_pct_median=float(100.0 * (1.0 - np.median(fps_c) / np.median(fps_p))),
        capture_cost_pct_per_pair=[float(100.0 * (1.0 - c / p)) for p, c in zip(fps_p, fps_c)],
        trajectory_nees_wall_s=t_nees, trajectory_nees_wall_s_median=float(np.median(t_nees)),
        trajectory_nees_samples=n_traj * n_frames,
        timing=("replay: wall clock around the replay threads (mc.run_replay 'seconds'), plain and capture alternated; "
                "trajectory_nees: wall clock of the call on host arrays (allocation, host-to-device copies of "
                "17 + 17 + 225 doubles per sample, both kernels, copies back)"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--traj", type=int, default=256)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--feats", type=int, default=150)
    ap.add_argument("--timing-traj", type=int, default=1024)
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles",
                                                  "r3_mc_consistency.json"))
    args = ap.parse_args()
    if api.lib().orcvio_device_count() < 1:
        raise SystemExit("mc_consistency.py needs a CUDA device")
    workers = os.cpu_count() or 1
    out = dict(gpu=gpu_info(), host_cores=workers, kitti_note=KITTI_NOTE,
               definitions=("NEES of the IMU error state [theta, v, p, b_g, b_a] against the synthetic truth at each "
                            "estimate's state time; orientation error Log(R R_est^T) under use_larvio / left "
                            "perturbation, Log(R_est^T R) otherwise; ANEES = mean over the valid runs of a frame; "
                            "bounds = chi2_quantile(0.025 | 0.975, N dof) / N"),
               cases={})
    for name, ov, nl, desc in CASES:
        try:
            r = consistency_case(name, ov, nl, args.traj, args.frames, args.feats, workers)
            r["description"] = desc
        except Exception as e:       # one config failing still leaves the others recorded
            r = dict(description=desc, error=f"{type(e).__name__}: {e}")
        out["cases"][name] = r
        print(name, json.dumps({k: v for k, v in r.items() if not isinstance(v, (list, dict))}), flush=True)
        if "blocks" in r:
            print("  inside 95 %:", {b: round(v["fraction_of_frames_inside_95"], 3) for b, v in r["blocks"].items()},
                  "median ANEES:", {b: round(v["anees_median_over_frames"], 3) for b, v in r["blocks"].items()}, flush=True)
    out["timing"] = timing_leg(args.timing_traj, args.frames, args.feats, workers, args.pairs)
    print("timing", json.dumps({k: v for k, v in out["timing"].items() if k != "timing"}), flush=True)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    write_record(args.out, out)
    print("wrote", os.path.abspath(args.out))


if __name__ == "__main__":
    main()
