"""Multi-trajectory (Monte-Carlo / multi-sequence) replay: SURVEY 8e, BASELINE.json configs[4].

A filter is sequential frame to frame, so the path shards only across independent trajectories:
trajectory t goes to rank t mod world, every rank advances its trajectories in lock-step with
`orcvio_batch_*` (each kernel has a filter grid dimension), no collective touches the data path;
one all_gather of a fixed-size record per trajectory at the end (NCCL on the GPU box, gloo in the
CPU tests).  This module is host-side plumbing: sharding, input packing, record gathering.
"""
import numpy as np

from . import api, synth

RECORD = ("traj", "frames", "px", "py", "pz", "ate_m", "feature_updates", "ok")


def shard(n_traj, rank, world):
    """Trajectory indices owned by `rank` (round-robin: equal lengths -> balanced)."""
    return list(range(rank, n_traj, world))


def pack_frame(seqs, fi, imu_cursor):
    """Concatenate frame `fi` of every sequence into the CSR arrays orcvio_batch_process expects.
    imu_cursor[i] = first IMU sample of sequence i not yet consumed by the filter."""
    t_img = np.zeros(len(seqs))
    feats, feat_off, imus, imu_off = [], [0], [], [0]
    for i, s in enumerate(seqs):
        t, f = s["frames"][fi]
        t_img[i] = t
        feats.append(api.feats_array(f))
        feat_off.append(feat_off[-1] + len(f))
        imu = s["imu"]
        k0 = imu_cursor[i]
        k1 = k0
        while k1 < len(imu) and imu[k1][0] <= t + 0.02:
            k1 += 1
        imus.append(api.imu_array(imu[k0:k1]))
        imu_off.append(imu_off[-1] + (k1 - k0))
    return (t_img, np.concatenate(feats) if feats else np.zeros(0, dtype=api.FEAT_DTYPE),
            np.array(feat_off, dtype=np.int32), np.concatenate(imus), np.array(imu_off, dtype=np.int32))


def _make_one(args):
    config, t, n_frames, feats_per_frame, overrides, n_landmarks = args
    return synth.make_sequence(synth.SynthSpec(config=config, seed=int(t), n_frames=n_frames,
                                               feats_per_frame=feats_per_frame, overrides=overrides,
                                               n_landmarks=n_landmarks))


def make_sequences(config, traj_ids, n_frames, feats_per_frame, overrides, n_landmarks=3000, workers=1):
    """Synthetic sequences of the given trajectories (seed = trajectory id); `workers` > 1 spreads the (pure Python)
    generator over processes."""
    jobs = [(config, int(t), n_frames, feats_per_frame, overrides, n_landmarks) for t in traj_ids]
    if workers <= 1 or len(jobs) < 4:
        return [_make_one(j) for j in jobs]
    from concurrent.futures import ProcessPoolExecutor
    import multiprocessing as mp
    with ProcessPoolExecutor(max_workers=workers, mp_context=mp.get_context("fork")) as ex:
        return list(ex.map(_make_one, jobs, chunksize=max(1, len(jobs) // (4 * workers))))


def pack_replay(seqs, n_frames):
    """Arrays of a whole-sequence replay (api.Batch.replay) for the given sequences."""
    n = len(seqs)
    t_img = np.zeros((n, n_frames))
    feat_off = np.zeros((n, n_frames + 1), dtype=np.int32)
    feats, imus = [], []
    for i, s in enumerate(seqs):
        fr = s["frames"][:n_frames]
        t_img[i] = [t for t, _ in fr]
        feat_off[i, 1:] = np.cumsum([len(f) for _, f in fr])
        feats.append(api.feats_array(np.concatenate([f for _, f in fr]) if fr else np.zeros((0, 9))))
        imus.append(api.imu_array(s["imu"]))
    return t_img, feats, feat_off, imus


def gt_poses(seqs, n_frames):
    g = np.zeros((len(seqs), n_frames, 7))
    for i, s in enumerate(seqs):
        for f, (_, p, q) in enumerate(s["gt"][:n_frames]):
            g[i, f, :3] = p
            g[i, f, 3:] = q
    return g


def truth_states(seqs, states):
    """Ground truth of every sequence at its estimates' own state times (states[..., 0], an IMU stamp), in the layout of
    the state records: (n, F, 17)."""
    return np.stack([synth.truth_states(s["spec"], states[i, :, 0]) for i, s in enumerate(seqs)])


def run_replay(cfg_path, seqs, traj_ids, n_threads=1, consistency=False):
    """The local trajectories, split into `n_threads` batches that replay concurrently from as many host threads (the
    host bookkeeping of a filter is serial code: the batches are what spreads it over the cores, and their kernels
    overlap on the device).  Returns (records, dict(seconds, feature_updates, kernel_launches, poses)).

    consistency: replay through Batch.replay_states instead (the IMU state and the leading 15 x 15 covariance block after
    every frame, captured on the device) and add to the dict `states` (n, F, 17), `cov15` (n, F, 15, 15), `truth` (n, F,
    17, at the states' own times), `nees` (n, F, 8) and `summary` (F, 9) of api.trajectory_nees over these trajectories."""
    import threading
    import time
    n = len(seqs)
    n_frames = min(len(s["frames"]) for s in seqs)
    n_threads = max(1, min(n_threads, n))
    groups = [list(range(k, n, n_threads)) for k in range(n_threads)]
    batches, packs = [], []
    for g in groups:
        b = api.Batch(cfg_path, len(g))
        for j, i in enumerate(g):
            it = seqs[i]["init"]
            b.set_initial_state(j, it["t"], it["quat"], it["pos"], it["vel"], it["bg"], it["ba"])
        batches.append(b)
        packs.append(pack_replay([seqs[i] for i in g], n_frames))
    poses = np.zeros((n, n_frames, 7))
    ok = np.zeros(n)
    if consistency:
        states = np.zeros((n, n_frames, 17))
        cov15 = np.zeros((n, n_frames, 15, 15))
    errors = []

    def work(k):
        try:
            if consistency:
                p, o, st, cv = batches[k].replay_states(*packs[k])
                states[groups[k]] = st
                cov15[groups[k]] = cv
            else:
                p, o = batches[k].replay(*packs[k])
            poses[groups[k]] = p
            ok[groups[k]] = o
        except Exception as e:       # surfaced after the join
            errors.append(e)

    t0 = time.perf_counter()
    threads = [threading.Thread(target=work, args=(k,)) for k in range(n_threads)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    seconds = time.perf_counter() - t0
    if errors:
        raise errors[0]
    met = api.trajectory_metrics(poses, gt_poses(seqs, n_frames))      # on the device (System.cpp:885-943)
    rec = np.zeros((n, len(RECORD)))
    fu = sum(b.feature_updates() for b in batches)
    for i in range(n):
        rec[i] = [traj_ids[i], n_frames, *poses[i, -1, :3], met[i, 1], fu / max(n, 1), ok[i]]
    info = dict(seconds=seconds, feature_updates=fu, kernel_launches=sum(b.kernel_launches() for b in batches),
                poses=poses, metrics=met, n_frames=n_frames, n_batches=n_threads)
    if consistency:
        truth = truth_states(seqs, states)
        nees, summary = api.trajectory_nees(states, truth, cov15, api.nees_flags(seqs[0]["cfg"]))
        info.update(states=states, cov15=cov15, truth=truth, nees=nees, summary=summary)
    return rec, info


def run_local(cfg_path, seqs, traj_ids):
    """Advance the local trajectories in lock-step on the current device.  Returns the record
    matrix (len(seqs) x len(RECORD)) and the Batch (for timing / counters)."""
    n = len(seqs)
    b = api.Batch(cfg_path, n)
    for i, s in enumerate(seqs):
        it = s["init"]
        b.set_initial_state(i, it["t"], it["quat"], it["pos"], it["vel"], it["bg"], it["ba"])
    cursor = [0] * n
    n_frames = min(len(s["frames"]) for s in seqs)
    est = np.zeros((n, n_frames, 3))
    ok = np.ones(n)
    for fi in range(n_frames):
        t_img, feats, feat_off, imu, imu_off = pack_frame(seqs, fi, cursor)
        used, pub = b.process(t_img, feats, feat_off, imu, imu_off)
        for i in range(n):
            cursor[i] += int(used[i])
            ok[i] = min(ok[i], float(pub[i]))
            est[i, fi] = b.state(i).p[:]
    rec = np.zeros((n, len(RECORD)))
    for i, s in enumerate(seqs):
        gt = np.array([g[1] for g in s["gt"][:n_frames]])
        d = (est[i] - est[i, 0]) - (gt - gt[0])          # first-pose alignment (System.cpp:885-943)
        rec[i] = [traj_ids[i], n_frames, *est[i, -1], float(np.mean(np.linalg.norm(d, axis=1))), 0.0, ok[i]]
    rec[:, 6] = b.feature_updates() / max(n, 1)
    return rec, b


def gather_records(rec, n_traj, rank, world, device=None):
    """all_gather of the per-trajectory records; returns an (n_traj x len(RECORD)) matrix ordered
    by trajectory id on every rank.  Works on NCCL (device tensors) and gloo (CPU tensors)."""
    if world == 1:
        out = np.zeros((n_traj, len(RECORD)))
        out[rec[:, 0].astype(int)] = rec
        return out
    import torch
    import torch.distributed as dist
    per = (n_traj + world - 1) // world
    buf = torch.full((per, len(RECORD)), -1.0, dtype=torch.float64, device=device)
    if len(rec):
        buf[:len(rec)] = torch.as_tensor(rec, dtype=torch.float64, device=device)
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf)
    out = np.zeros((n_traj, len(RECORD)))
    for p in parts:
        a = p.cpu().numpy()
        a = a[a[:, 0] >= 0]
        out[a[:, 0].astype(int)] = a
    return out


def gather_nees(nees, traj_ids, n_traj, rank, world, device=None):
    """all_gather of the per-trajectory NEES rows (fixed size n_frames x 8 each, api.trajectory_nees); returns (n_traj,
    n_frames, 8) ordered by trajectory id on every rank.  The summary over all trajectories is then
    api.nees_summary(rows): the same rows in the same order, hence the same bits for every world size."""
    nees = np.asarray(nees, dtype=np.float64)
    n_frames = nees.shape[1]
    width = 1 + n_frames * 8
    rows = np.zeros((len(traj_ids), width))
    rows[:, 0] = traj_ids
    rows[:, 1:] = nees.reshape(len(traj_ids), -1)
    if world == 1:
        out = np.zeros((n_traj, width))
        out[rows[:, 0].astype(int)] = rows
        return out[:, 1:].reshape(n_traj, n_frames, 8)
    import torch
    import torch.distributed as dist
    per = (n_traj + world - 1) // world
    buf = torch.full((per, width), -1.0, dtype=torch.float64, device=device)
    if len(rows):
        buf[:len(rows)] = torch.as_tensor(rows, dtype=torch.float64, device=device)
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf)
    out = np.zeros((n_traj, width))
    for p in parts:
        a = p.cpu().numpy()
        a = a[a[:, 0] >= 0]
        out[a[:, 0].astype(int)] = a
    return out[:, 1:].reshape(n_traj, n_frames, 8)
