#!/usr/bin/env python
"""bench.py -- feature updates / s of the OrcVIO filter-update hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[3], "stress frame"): one frozen frame with a 30-clone window
(D = 202) and 4096 features, reference-faithful track lengths m in [3, 6] (`max_track_len: 6`
in every shipped yaml; SURVEY 8d case 4a).  One step = one pass of the hot path over the frame:
per-feature LM triangulation, measurement Jacobians + left-nullspace projection + chi-square
gate, QR compression of the stacked H, FP64 EKF gain + covariance update (stages 1,2,4,5 of
BASELINE.json's north_star).  metric = features that pass the gate and update the filter per
second; `us_per_frame` is the same time per frame.

  value : kernel chain on the HBM-resident frame, CUDA events on the launching stream, L2
          flushed between timed iterations.
  e2e   : orcvio_frame_update() through the C ABI with HOST buffers every step (host work-list
          build + H2D + kernels + D2H of P / delta_x / gate decisions inside the timed region).
  N > 1 : the path shards only across independent trajectories: every rank owns its own copy of
          the frame (the same seed on every rank: weak scaling means the same work per GPU -- with
          seed = rank the max over ranks measured the spread of the Levenberg-Marquardt tail between
          frames, 210 .. 239 us on ONE GPU, scripts/seed_spread.py), no data-path collective; NCCL
          gathers the per-rank counters.  Weak scaling; time = max over ranks.
  --impl reference : the CPU restatement of the reference algorithm (oracle/, dense like the
          reference) on the box's host cores, one independent frame per thread.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "feature_updates_per_sec"
UNIT = "features/s"
N_CLONES, N_FEATURES, MAX_TRACK = 30, 4096, 6
TARGET_FEATURES = 2000      # BASELINE.json north_star: "30-clone, 2000-feature frame runs under 200 us"
NOISE_VAR = 1.6e-5          # (2 x 0.002)^2: synthetic pixel noise of the KITTI-shaped generator
TRI = dict(cost_threshold=1e-3, init_final_dist_threshold=100.0)


def ncu_capture(kernel="k_syrk"):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes per launch) and the measured DMMA-pipe activity of one launch
    of `kernel`, read from the newest committed `ncu --set full` summary under profiles/ (scripts/ncu_summary.py)."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_summary.csv")))
    if not files:
        return None
    rows = list(csv.reader(open(files[-1])))
    hdr, units = rows[0], rows[1]
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for r in rows[2:]:
        if kernel in r[0]:
            def col(name):
                if name not in hdr:
                    return None, None
                i = hdr.index(name)
                return float(r[i]), units[i]
            rd, ru = col("dram__bytes_read.sum")
            wr, wu = col("dram__bytes_write.sum")
            pipe, _ = col("smsp__pipe_tensor_subpipe_dmma_cycles_active.avg.pct_of_peak_sustained_active")
            inst, _ = col("sm__inst_executed_pipe_tensor_subpipe_dmma.sum")
            us, _ = col("gpu__time_duration.sum")
            return dict(traffic=int(rd * scale.get(ru, 1.0) + wr * scale.get(wu, 1.0)) if rd is not None else None,
                        dmma_pipe_active_pct=pipe, dmma_instructions=inst, capture_us=us,
                        source=os.path.relpath(files[-1], ROOT))
    return None


WORKLOAD = f"stress frame: {N_CLONES}-clone window, {N_FEATURES} features, max_track_len {MAX_TRACK} (SURVEY 8d C4a)"


def make_frame(seed, n_feat=N_FEATURES):
    from orcvio_b200 import synth
    return synth.stress_snapshot(N_CLONES, n_feat, MAX_TRACK, seed=seed)


def dump_outputs(path, out):
    """What a caller of the frame update receives (posterior P, delta_x, per-feature status and gamma, updated clones),
    one float64 .npy per array, so that two builds can be compared output for output on the same seeded frame."""
    os.makedirs(path, exist_ok=True)
    for name in ("P", "delta_x", "status", "gamma", "clones"):
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(out[name], dtype=np.float64))


def algorithmic_bytes(snap, status, stage):
    """Compulsory HBM bytes of one launch of the dominant kernel (SURVEY 8d per-feature figures)."""
    fo = np.asarray(snap["feat_off"])
    m = np.diff(fo).astype(np.int64)
    N = int(snap["n_clones"])
    D = 22 + 6 * N
    r = 2 * m - 3
    c = 6 * m
    passed = (np.asarray(status) & 2) != 0
    per_frame = 8 * 24 * N + 8 * D * D            # clone records + covariance, read once
    if stage == "tri":
        return int((16 * m + 4 * m + 64 + 32 + 4).sum() + 8 * 24 * N)
    if stage == "jac_gate":
        # in: obs (16m) + clone idx (4m) + work record (64) + position (32);
        # out: gamma + status (12) and, for gated-in features, the compact r x (c+1) block
        return int((16 * m + 4 * m + 64 + 32 + 12).sum() + (8 * r * (c + 1))[passed].sum() + per_frame)
    if stage in ("qr_tiles", "qr_chain"):
        return int((8 * r * (c + 1))[passed].sum() + 8 * (6 * N) * (6 * N + 1))
    if stage == "update":
        return int(24 * D * D)
    return 0


def syrk_flops(snap, status):
    """Algorithmic flops of W = s^2 I + A^T A (k_syrk): one triangle of the (n+1) x (n+1) Gram
    matrix of the M gated rows of A = [H' L | r'], 2 flops per multiply-add  ->  M (n+1)(n+2).
    (The reference spends 2 M De^2 - 2/3 De^3 on the Householder QR of the same rows, SURVEY 8d.)"""
    m = np.diff(np.asarray(snap["feat_off"])).astype(np.int64)
    passed = (np.asarray(status) & 2) != 0
    M = int((2 * m - 3)[passed].sum())
    n1 = 6 * int(snap["n_clones"]) + 1
    return M * n1 * (n1 + 1), M


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
                for k, nm in enumerate(names):
                    if r[2 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=smax, reasons=sorted(reasons),
                    samples=len(sm))


def run_cpu_reference(n_threads, n_feat, repeats, seed0=0, variant="o3"):
    """Times the CPU restatement of the reference algorithm on `n_threads` independent frames
    (one per thread).  Returns (features gated in, seconds, kind).  variant "o3" = the -O3 / AVX2 + FMA build of the
    restatement (what a vectorised Release build of the reference's Eigen code would get; the default of both CPU legs,
    the favourable choice for the CPU), "" = the -O2 generic x86-64 build the parity tests use."""
    from oracle import cpu_ref
    if variant == "o3" and not os.path.exists(cpu_ref._SO_O3):
        variant = ""
    return cpu_ref.time_frames(N_CLONES, n_feat, MAX_TRACK, NOISE_VAR, TRI, n_threads, repeats, seed0, variant=variant)


CPU_BUILD = ("C++ restatement of the reference algorithm (kind: port), g++ -O3 -march=x86-64-v3 (AVX2 + FMA); the -O2 "
             "generic x86-64 build used by the parity tests is reported as value_o2_generic")


def reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_feat = args.ref_features
    # warm-up + timed steps, each step = one bounded sample (one frame per thread)
    for _ in range(max(args.warmup, 0)):
        run_cpu_reference(cores, min(n_feat, 512), 1)
    feats, secs = 0, 0.0
    for k in range(args.steps):
        f, s, kind = run_cpu_reference(cores, n_feat, 1, seed0=100 * k)
        feats += f
        secs += s
    value = feats / secs
    f2, s2, _ = run_cpu_reference(cores, n_feat, 1, seed0=7, variant="")
    sample = (f"{cores} independent frames per step (one per thread), each {N_CLONES} clones x {n_feat} features, "
              f"m in [3,{MAX_TRACK}]; dense per-feature H P H^T gate, Householder QR compression, dense EKF update")
    line = dict(metric=METRIC, value=value, unit=UNIT, impl="reference", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * secs / args.steps, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=WORKLOAD, sample=sample),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind=kind, sample=sample, build=CPU_BUILD,
                                  value_o2_generic=f2 / s2),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def _time_frame(api, torch, snap, n_clones, steps, warmup, l2_flush):
    """Device time (CUDA events, L2 flushed) and end-to-end wall time of one frozen frame."""
    fr = api.Frame(n_clones, 0, NOISE_VAR, 0.95, -1.0, TRI["cost_threshold"], TRI["init_final_dist_threshold"])
    inp = fr.prepare_inputs(snap)
    out = fr.update(inp)
    fr.load(snap)
    for _ in range(warmup):
        l2_flush()
        fr.run(1)
    us = 0.0
    for _ in range(steps):
        l2_flush()
        us += fr.run(1)
    for _ in range(3):
        fr.update(inp, out)
    t0 = time.perf_counter()
    for _ in range(steps):
        fr.update(inp, out)
    torch.cuda.synchronize()
    e2e = (time.perf_counter() - t0) / steps * 1e6
    m = np.diff(np.asarray(snap["feat_off"]))
    passed = (out["status"] & 2) != 0
    return dict(us_per_frame=us / steps, e2e_us_per_frame=e2e, features=int(len(m)), gated_in=int(passed.sum()),
                gated_rows=int((2 * m - 3)[passed].sum()), state_dim=22 + 6 * n_clones)


def _process_features_leg(api, configs_mod, synth, cfg_name, overrides, n_frames, feats, n_landmarks, skip):
    """Wall time of OrcVIO::processFeatures (propagation + augmentation + ZUPT test + both update chains + pruning),
    host buffers in, host state out, on a synthetic sequence of the given shape; the first `skip` frames (window
    filling up) are left out."""
    import tempfile
    seq = synth.make_sequence(synth.SynthSpec(config=cfg_name, seed=0, n_frames=n_frames, feats_per_frame=feats,
                                              overrides=overrides, n_landmarks=n_landmarks))
    path = os.path.join(tempfile.mkdtemp(prefix="orcvio_bench_"), "cfg.yaml")
    configs_mod.write_yaml(path, seq["cfg"])
    vio = api.OrcVIO(path)
    if not vio.initialize():
        return dict(error="initialize failed")
    k, times, n_states, cand = 0, [], 0, 0
    for fi, (t_img, f) in enumerate(seq["frames"]):
        k1 = k
        while k1 < len(seq["imu"]) and seq["imu"][k1][0] <= t_img + 0.02:
            k1 += 1
        vio.push_imu(seq["imu"][k:k1])
        k = k1
        t0 = time.perf_counter()
        ok = vio.processFeatures(t_img, f)
        dt = time.perf_counter() - t0
        if not ok:
            return dict(error=f"frame {fi} not published")
        if fi >= skip:
            times.append(dt)
            st = vio.frame_stats()
            cand += st.n_candidates_lost + st.n_candidates_prune
            n_states = max(n_states, len(vio.feature_states()[0]))
    st = vio.state()
    return dict(us_per_call_median=float(np.median(times)) * 1e6, us_per_call_mean=float(np.mean(times)) * 1e6,
                frames=len(times), features_per_frame=feats, clones=int(st.n_clones), state_dim=int(st.dim),
                candidates_per_frame=cand / max(len(times), 1), max_ekf_feature_states=int(n_states),
                config=f"{cfg_name}.yaml shape" + (f" with {overrides}" if overrides else " as shipped"))


def _object_leg(api, configs_mod, synth):
    """BASELINE configs[1]: Unity-shaped filter, one object (12 keypoints, 5 views) -- the stage-3 rows, their
    projection onto the window (constructObjectResidualJacobians) and the object update (removeLostObjects)."""
    import tempfile
    gold = os.path.join(ROOT, "tests", "golden", "one_car.npz")
    if not os.path.exists(gold):
        return dict(error="tests/golden/one_car.npz missing")
    g = np.load(gold)
    seq = synth.make_sequence(synth.SynthSpec(config="unity", seed=4, n_frames=26, feats_per_frame=100,
                                              overrides=dict(if_ZUPT_valid=0)))
    path = os.path.join(tempfile.mkdtemp(prefix="orcvio_bench_"), "cfg.yaml")
    configs_mod.write_yaml(path, seq["cfg"])
    vio = api.OrcVIO(path)
    if not vio.initialize():
        return dict(error="initialize failed")
    k = 0
    t_feat = []
    for (t_img, f) in seq["frames"]:
        k1 = k
        while k1 < len(seq["imu"]) and seq["imu"][k1][0] <= t_img + 0.02:
            k1 += 1
        vio.push_imu(seq["imu"][k:k1])
        k = k1
        t0 = time.perf_counter()
        vio.processFeatures(t_img, f)
        t_feat.append(time.perf_counter() - t0)
    poses, ids, times = vio.window()
    N = len(ids)
    T = np.array(seq["cfg"]["T_cam_imu"]).reshape(4, 4)
    Rbc = T[:3, :3]
    tcb = -Rbc.T @ T[:3, 3]
    frames, ts = [], []
    for c in [2, 4, 5, 7, N - 2]:
        R, p = poses[c][:9].reshape(3, 3), poses[c][9:]
        wTc = np.eye(4)
        wTc[:3, :3] = R @ Rbc.T
        wTc[:3, 3] = p + R @ tcb
        frames.append(wTc)
        ts.append(float(times[c]))
    frames = np.array(frames)
    kps = g["mean_shape"][0]
    shape = g["ellipsoid_shape"][0].ravel()
    wTo = np.eye(4)
    wTo[:3, 3] = frames[2][:3, 3] + frames[2][:3, :3] @ np.array([0.3, 0.1, 9.0])
    rng = np.random.default_rng(3)
    zs, zb = [], []
    for wTc in frames:
        pc = (np.linalg.inv(wTc) @ wTo @ np.hstack([kps, np.ones((len(kps), 1))]).T)[:3]
        uv = (pc[:2] / pc[2]).T
        zs.append(uv + rng.normal(0, 0.004, uv.shape))
        zb.append(np.array([uv[:, 0].min(), uv[:, 1].min(), uv[:, 0].max(), uv[:, 1].max()]) + rng.normal(0, 0.004, 4))
    zs, zb = np.array(zs), np.array(zb)
    P0 = vio.cov()
    reps, t_rows, t_con, t_upd, status = 10, 0.0, 0.0, 0.0, None
    for _ in range(reps):
        t0 = time.perf_counter()
        rows = api.object_residuals(frames, wTo, shape, kps, zs, zb, left=False, new_residual=True)
        t1 = time.perf_counter()
        flag, Hx, Hf, res = vio.constructObjectResidualJacobians(rows["fjac_cam"], ts, rows["fjac_obj"], rows["fvec"],
                                                                 rows["zs_num"], rows["cam_pose_se3"])
        t2 = time.perf_counter()
        status, gamma = vio.removeLostObjects(Hx, Hf, res)
        t3 = time.perf_counter()
        t_rows += t1 - t0
        t_con += t2 - t1
        t_upd += t3 - t2
    # the object state optimiser in front of stage 3 (ObjectFeatureInitializer): the reference's one_car sequence (47
    # frames x 12 keypoints) as a batch of 64 objects advanced in lock-step
    lm = {}
    try:
        xywh = g["zb"][:, 0, :]
        zb47 = np.column_stack([xywh[:, 0], xywh[:, 1], xywh[:, 0] + xywh[:, 2], xywh[:, 1] + xywh[:, 3]])
        init = api.ObjectFeatureInitializer(g["ellipsoid_shape"][-1].ravel(), g["mean_shape"][-1], [1.0, 3e-2, 1.0, 1.0])
        nobj = 64
        fl, zl, bl = [g["wTo"]] * nobj, [g["zs"]] * nobj, [zb47] * nobj
        init.single_object_initialization(fl, zl)
        t0 = time.perf_counter()
        ok, T0, _, _ = init.single_object_initialization(fl, zl)
        t1 = time.perf_counter()
        res = init.single_levenberg_marquardt(fl, zl, bl, T0, True, False)
        t2 = time.perf_counter()
        lm = dict(objects=nobj, frames_per_object=int(len(g["wTo"])), init_us_per_object=(t1 - t0) / nobj * 1e6,
                  lm_us_per_object=(t2 - t1) / nobj * 1e6, lm_rounds=int(res["rounds"]), lm_nfev=int(res["nfev"][0]),
                  lm_status=int(res["status"][0]), all_success=bool(np.all(res["success"])))
    except Exception as e:
        lm = dict(error=str(e))
    return dict(msckf_process_features_us_median=float(np.median(t_feat[10:])) * 1e6, object_rows_us=t_rows / reps * 1e6,
                object_optimiser=lm,
                construct_jacobians_us=t_con / reps * 1e6, remove_lost_objects_us=t_upd / reps * 1e6,
                object_rows=int(Hx.shape[0]), keypoints=int(len(kps)), views=int(len(frames)), clones=int(N),
                last_status=int(status), state_dim=int(P0.shape[0]),
                timing="wall clock around the C-ABI calls, host buffers in and out")


def extra_legs(api, torch, args, l2_flush):
    """SURVEY 8d: the other cases of the measurement row, rank 0 only, bounded (a few seconds each)."""
    from orcvio_b200 import synth, configs as configs_mod
    out = {}
    steps = max(10, min(args.steps, 50))
    try:
        # case 4b: every feature seen by all 30 clones (m = N = 30): M = 4096 x 57 = 233 k candidate rows.  The frame is
        # flop-bound by the GATE, not by the compression: gamma = r^T (H P H^T + s^2 I)^-1 r needs the 57 x 180 block of
        # every feature against the 180 x 180 window of P (2 r w^2 + 2 r^2 w = 4.9 Mflop per feature, 20 Gflop per frame,
        # plain DFMA), then the whitening A = H' L (2 M w n / 2, L lower triangular) and W = A^T A (M (n+1)(n+2)) on the
        # FP64 tensor cores
        snap = synth.stress_snapshot(N_CLONES, N_FEATURES, MAX_TRACK, seed=0, full_tracks=True)
        r = _time_frame(api, torch, snap, N_CLONES, max(5, steps // 5), 3, l2_flush)
        dfma, dmma = api.fp64_peak()
        m, w, n = N_CLONES, 6 * N_CLONES, 6 * N_CLONES
        rr = 2 * m - 3
        gate = r["features"] * (2.0 * rr * w * w + 2.0 * rr * rr * w)
        aform = r["gated_rows"] * 2.0 * w * n / 2
        syrk = r["gated_rows"] * (n + 1.0) * (n + 2.0)
        r["flop_bound_us"] = dict(gate_dfma=gate / (dfma * 1e12) * 1e6, aform_dmma=aform / (dmma * 1e12) * 1e6,
                                  syrk_dmma=syrk / (dmma * 1e12) * 1e6)
        r["flop_bound_us"]["total"] = sum(r["flop_bound_us"].values())
        r["frac_of_flop_bound"] = r["flop_bound_us"]["total"] / r["us_per_frame"]
        out["case_4b_full_tracks"] = r
    except Exception as e:
        out["case_4b_full_tracks"] = dict(error=str(e))
    for key, cfg, ncl, nf in (("C1_euroc_frame", "euroc", 20, 300), ("C3_kitti_frame", "kitti_odom", 30, 1000)):
        try:
            snap = synth.stress_snapshot(ncl, nf, MAX_TRACK, seed=0, config=cfg)
            out[key] = _time_frame(api, torch, snap, ncl, steps, 3, l2_flush)
        except Exception as e:
            out[key] = dict(error=str(e))
    try:
        out["C2_unity_object_update"] = _object_leg(api, configs_mod, synth)
    except Exception as e:
        out["C2_unity_object_update"] = dict(error=str(e))
    for key, cfg, ov, nfr, feats, nlm, skip in (
            ("process_features_euroc", "euroc", {}, 90, 300, 8000, 60),
            ("process_features_kitti", "kitti_odom", {}, 70, 1000, 30000, 45)):
        try:
            out[key] = _process_features_leg(api, configs_mod, synth, cfg, ov, nfr, feats, nlm, skip)
        except Exception as e:
            out[key] = dict(error=str(e))
    return out


def multi_trajectory_leg(api, torch, dist, args, rank, world, dev):
    """BASELINE configs[4]: `--mc-traj` independent EuRoC-shaped trajectories x `--mc-frames` frames, sharded over the
    ranks (trajectory t -> rank t mod world), no data-path collective: every rank replays its share through
    orcvio_batch_replay, split into one batch per host thread; NCCL gathers the per-trajectory records."""
    from orcvio_b200 import montecarlo as mc, configs as configs_mod
    import tempfile
    cores = os.cpu_count() or 1
    per_rank = max(1, cores // world)
    mine = mc.shard(args.mc_traj, rank, world)
    t0 = time.perf_counter()
    seqs = mc.make_sequences("euroc", mine, args.mc_frames, args.mc_feats, {}, n_landmarks=3000, workers=per_rank)
    t_gen = time.perf_counter() - t0
    path = os.path.join(tempfile.mkdtemp(prefix="orcvio_mc_"), "cfg.yaml")
    configs_mod.write_yaml(path, seqs[0]["cfg"])
    # warm-up: a small replay of the same shape (every kernel of the path, incl. the hybrid branch that only opens 5 s
    # into a sequence, is loaded and has run once before the timed replay)
    nw = min(len(seqs), 2 * per_rank)
    mc.run_replay(path, seqs[:nw], mine[:nw], n_threads=min(per_rank, nw))
    util = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    util.FIELDS = "utilization.gpu,clocks.sm"
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        util.start()
    rec, info = mc.run_replay(path, seqs, mine, n_threads=per_rank)
    torch.cuda.synchronize()
    busy = None
    if rank == 0 and util.proc:
        time.sleep(0.12)
        util.proc.terminate()
        vals = []
        for r in util.rows:
            try:
                vals.append(float(r[0]))
            except Exception:
                pass
        busy = float(np.mean(vals)) if vals else None
    secs = torch.tensor([info["seconds"]], dtype=torch.float64, device=dev)
    counts = torch.tensor([float(info["feature_updates"]), float(info["kernel_launches"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(secs, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    allrec = mc.gather_records(rec, args.mc_traj, rank, world, device=dev)
    s = secs.item()
    return dict(
        workload=f"Monte-Carlo replay: {args.mc_traj} independent euroc.yaml-shaped trajectories (hybrid MSCKF/EKF-SLAM + ZUPT as "
                 f"shipped) x {args.mc_frames} frames, ~{args.mc_feats} features per frame, trajectory t -> rank t mod {world}",
        n_gpus=world, trajectories=args.mc_traj, frames=args.mc_frames, host_threads_per_rank=per_rank, host_cores=cores,
        seconds=s, trajectory_frames_per_sec=args.mc_traj * args.mc_frames / s,
        feature_updates_per_sec=counts[0].item() / s, feature_updates=counts[0].item(), kernel_launches=counts[1].item(),
        all_published=bool(np.all(allrec[:, 7] == 1.0)), ate_m_mean=float(allrec[:, 5].mean()),
        ate_m_max=float(allrec[:, 5].max()), ate_checksum=float(np.sum(allrec[:, 5] * (1 + np.arange(len(allrec))))),
        gpu_utilization_pct_rank0=busy, sequence_generation_s_per_rank=t_gen, scaling="strong",
        warmup=f"one untimed replay of {nw} of the rank's trajectories",
        timing="wall clock around the replay threads of a rank (host bookkeeping + uploads + kernels + read-backs), "
               "barrier + synchronize on both sides, max over ranks; trajectory metrics by orcvio_trajectory_metrics on the device")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-features", type=int, default=N_FEATURES, help="features per frame of the CPU sample")
    ap.add_argument("--ref-repeats", type=int, default=6, help="frames per host thread in the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-flush", action="store_true", help="skip the L2 flush (profiling runs only)")
    ap.add_argument("--no-extra", action="store_true", help="skip the other SURVEY 8d cases (4b, C1-C3, processFeatures)")
    ap.add_argument("--no-mc", action="store_true", help="skip the multi-trajectory replay (BASELINE configs[4])")
    ap.add_argument("--mc-traj", type=int, default=1024)
    ap.add_argument("--mc-frames", type=int, default=200)
    ap.add_argument("--mc-feats", type=int, default=150)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed frame update computed in its last step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from orcvio_b200 import api

    if not torch.cuda.is_available() or api.lib().orcvio_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: orcvio_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    api.lib().orcvio_set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    snap = make_frame(seed=0)                          # the same work on every rank (see the module docstring)
    fr = api.Frame(N_CLONES, 0, NOISE_VAR, 0.95, -1.0, TRI["cost_threshold"], TRI["init_final_dist_threshold"])
    inp = fr.prepare_inputs(snap)
    out = fr.update(inp)                               # also the correctness anchor of this run
    n_pass = int(((out["status"] & 2) != 0).sum())
    n_valid = int(((out["status"] & 1) != 0).sum())
    fr.load(snap)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def l2_flush():
        if not args.no_flush:
            flush.zero_()
            torch.cuda.synchronize()

    # ---- value: HBM-resident frame, CUDA events around the kernel chain
    for _ in range(args.warmup):
        l2_flush()
        fr.run(1)
    _, stages = fr.run(5, stages=True)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = fr.kernel_launches()
    dev_us = 0.0
    for _ in range(args.steps):
        l2_flush()
        dev_us += fr.run(1)
    launches = fr.kernel_launches() - l0
    barrier()
    t_val = torch.tensor([dev_us * 1e-6], dtype=torch.float64, device=dev)
    if args.dump_outputs and rank == 0:
        # fetch() replays the chain once with the download queued; every run restores the frame's inputs first, so
        # this is exactly what the last timed step computed
        dump_outputs(args.dump_outputs, fr.fetch())

    # ---- e2e: host buffers through the C ABI, wall clock around synchronous calls
    for _ in range(args.warmup):
        fr.update(inp, out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fr.update(inp, out)
    torch.cuda.synchronize()
    t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    barrier()
    # the same call when the covariance stays on the device (pose / velocity covariance block back instead of all of P)
    for _ in range(args.warmup):
        fr.update(inp, out, full_P=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fr.update(inp, out, full_P=False)
    torch.cuda.synchronize()
    t_e2e_lite = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop() if rank == 0 else None

    # ---- the north star's target frame (30 clones, 2000 features, target < 200 us), rank 0 only: same chain, same
    # timing method (CUDA events on the launching stream, L2 flushed), reported beside the headline workload
    target = None
    if rank == 0:
        snap_t = make_frame(seed=0, n_feat=TARGET_FEATURES)
        fr_t = api.Frame(N_CLONES, 0, NOISE_VAR, 0.95, -1.0, TRI["cost_threshold"], TRI["init_final_dist_threshold"])
        out_t = fr_t.update(fr_t.prepare_inputs(snap_t))
        fr_t.load(snap_t)
        for _ in range(args.warmup):
            l2_flush()
            fr_t.run(1)
        us_t, n_t = 0.0, max(20, min(args.steps, 100))
        for _ in range(n_t):
            l2_flush()
            us_t += fr_t.run(1)
        _, st_t = fr_t.run(5, stages=True)
        target = dict(workload=f"{N_CLONES}-clone window, {TARGET_FEATURES} features, max_track_len {MAX_TRACK}",
                      us_per_frame=us_t / n_t, target_us=200.0, gated_in=int(((out_t["status"] & 2) != 0).sum()),
                      stage_us=dict(tri=round(st_t["tri"], 2), jac_gate=round(st_t["jac_gate"], 2),
                                    aform_incl_prior_wait=round(st_t["qr_tiles"], 2),
                                    syrk_plus_chol_w_solve=round(st_t["qr_chain"], 2),
                                    pinfo_increment=round(st_t["update"], 2), total=round(st_t["total"], 2)))
        del fr_t

    extras = None
    if rank == 0 and not args.no_extra:
        extras = extra_legs(api, torch, args, l2_flush)
    del flush
    mc_leg = None
    if not args.no_mc:
        try:
            mc_leg = multi_trajectory_leg(api, torch, dist, args, rank, world, dev)
        except Exception as e:
            mc_leg = dict(error=repr(e))
            if world > 1:
                raise

    counts = torch.tensor([float(n_pass), float(N_FEATURES)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_val, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    total_pass = counts[0].item()
    secs, secs_e2e = t_val.item(), t_e2e.item()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)" if peaks else "fallback 6650 GB/s"
        # stage split of the whitened-form path (api.Frame.STAGES keeps the generic names):
        #   qr_tiles = k_aform (+ wait for k_chol_prior), qr_chain = k_syrk + k_chol_w_solve, update = k_pinfo
        kt = fr.kernel_times()
        stage_named = dict(tri=stages["tri"], jac_gate=stages["jac_gate"], aform_incl_prior_wait=stages["qr_tiles"],
                           syrk=kt["syrk"], chol_w_solve=stages["qr_chain"] - kt["syrk"], pinfo_increment=stages["update"],
                           chol_prior_second_stream=kt["chol_prior"], total=stages["total"])
        # roofline kernel: k_syrk, the one kernel of the chain with GEMM-sized work (the FP64 tensor-core
        # compression GEMM of the north star); the other kernels are latency chains (DESIGN.md section 3)
        dfma_peak, dmma_peak = api.fp64_peak()
        cap = ncu_capture("k_syrk")
        flops, M_rows = syrk_flops(snap, out["status"])
        achieved = flops / (kt["syrk"] * 1e-6) / 1e12
        jac_bytes = algorithmic_bytes(snap, out["status"], "jac_gate")
        h2d = sum(inp[k].nbytes for k in ("clone_R", "clone_p", "Rbc", "tcb", "P", "feat_off", "obs_clone", "obs_z"))
        d2h = sum(out[k].nbytes for k in ("P", "delta_x", "status", "gamma", "clones"))
        line = dict(
            metric=METRIC, value=total_pass * args.steps / secs, unit=UNIT, n_gpus=world, steps=args.steps,
            warmup=args.warmup, ms_per_step=1e3 * secs / args.steps, higher_is_better=True, scaling="weak",
            vs_baseline=None, dtype="f64", data="synthetic",
            config=dict(workload=WORKLOAD, n_clones=N_CLONES, state_dim=22 + 6 * N_CLONES,
                        features_per_frame=N_FEATURES, triangulated_ok=n_valid, gated_in=n_pass,
                        frames_per_step_per_gpu=1, frame_seed=0,
                        sharding="independent frames (trajectories) per rank -- the same frame on every rank: fixed work "
                                 "per GPU --, no collective",
                        l2="flushed between timed iterations (256 MiB memset)" if not args.no_flush else "not flushed",
                        timing="CUDA events on the launching stream per iteration, max over ranks"),
            us_per_frame=1e6 * secs / args.steps,
            stage_us={k: round(v, 2) for k, v in stage_named.items()},
            stage_us_note="stage times come from a separate run with event records between the kernels (launched one by "
                          "one); the timed steps replay one CUDA graph of the whole chain, so their sum exceeds us_per_frame",
            e2e=dict(value=total_pass * args.steps / secs_e2e, unit=UNIT, h2d_bytes_per_step=int(h2d),
                     d2h_bytes_per_step=int(d2h), us_per_frame=1e6 * secs_e2e / args.steps,
                     pose_cov_only=dict(us_per_frame=1e6 * t_e2e_lite / args.steps,
                                        d2h_bytes_per_step=int(d2h - out["P"].nbytes + 81 * 8),
                                        note="orcvio_frame_update_pose_cov: the leading 9 x 9 block of P comes back "
                                             "instead of all of it (rank 0)")),
            gpu_launches=int(launches),
            roofline=dict(bound="tensor", kernel="k_syrk (W = s^2 I + A^T A: staircase-sparse split-K, cp.async operand pipeline, "
                                                 "mma.sync m8n8k4 f64, parallel slice reduction)", achieved=achieved,
                          peak=dmma_peak, unit="TFLOP/s", frac=achieved / dmma_peak, traffic=(cap or {}).get("traffic"),
                          ncu=cap,
                          algorithmic_flops=flops, gated_rows=M_rows, kernel_us=kt["syrk"],
                          peak_source="FP64 DMMA peak measured live on this GPU (orcvio_fp64_peak: mma.sync m8n8k4 "
                                      "micro-kernel; MEASURED_PEAKS.json carries only bf16 / HBM)",
                          fp64_dfma_peak=dfma_peak),
            roofline_hbm=dict(bound="hbm", kernel="k_jac_gate", achieved=jac_bytes / (stages["jac_gate"] * 1e-6) / 1e9,
                              peak=peak, unit="GB/s", frac=jac_bytes / (stages["jac_gate"] * 1e-6) / 1e9 / peak,
                              algorithmic_bytes=jac_bytes, kernel_us=stages["jac_gate"], peak_source=peak_src,
                              note="one frame's working set is L2-resident: latency-bound, not HBM-bound (SURVEY 8d)"),
            north_star_frame=target,
            other_cases=extras,
            multi_trajectory=mc_leg,
            clocks=clocks)
        if not args.no_cpu_baseline:
            try:
                cores = os.cpu_count() or 1
                f, s, kind = run_cpu_reference(cores, args.ref_features, args.ref_repeats)
                f2, s2, _ = run_cpu_reference(cores, args.ref_features, 1, seed0=7, variant="")
                line["cpu_baseline"] = dict(
                    value=f / s, unit=UNIT, cores=cores, kind=kind, build=CPU_BUILD, value_o2_generic=f2 / s2,
                    sample=f"{cores * args.ref_repeats} independent frames ({args.ref_repeats} per host thread), each "
                           f"{N_CLONES} clones x {args.ref_features} features, m in [3,{MAX_TRACK}]; "
                           f"{s * cores:.1f} core-seconds of CPU work")
            except Exception as e:       # the baseline is a reported number, never the product path
                line["cpu_baseline"] = dict(value=None, unit=UNIT, cores=0, kind="port", sample=f"failed: {e}")
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
