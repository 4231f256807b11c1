"""Deterministic synthetic front-end for the filter-update path.

Emits exactly the boundary types the reference filter consumes (SURVEY A.3):
IMU samples (t, gyro, acc) and per-image lists of MonoFeatureMeasurement
(id, u, v, u_init, v_init, u_vel, v_vel, u_init_vel, v_init_vel) in undistorted
normalised coordinates -- reference include/orcvio/feat/feature_msg.h:14-55 and
include/sensors/ImuData.hpp:16-39.  There is no network and no dataset in this
environment, so EuRoC-, KITTI- and Unity-*shaped* sequences are generated from an
analytic trajectory, a random landmark cloud and the noise levels of the named
config.  Seeds: numpy.random.default_rng(1000 + k).
"""
import math
from dataclasses import dataclass, field

import numpy as np

from . import configs

GRAVITY = np.array([0.0, 0.0, -9.81])


def _rot_zyx(yaw, pitch, roll):
    cy, sy = math.cos(yaw), math.sin(yaw)
    cp, sp = math.cos(pitch), math.sin(pitch)
    cr, sr = math.cos(roll), math.sin(roll)
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1.0]])
    Ry = np.array([[cp, 0, sp], [0, 1.0, 0], [-sp, 0, cp]])
    Rx = np.array([[1.0, 0, 0], [0, cr, -sr], [0, sr, cr]])
    return Rz @ Ry @ Rx


def _quat_xyzw(R):
    t = np.trace(R)
    if t > 0:
        s = math.sqrt(t + 1.0) * 2
        q = [(R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s, 0.25 * s]
    else:
        i = int(np.argmax(np.diag(R)))
        j, k = (i + 1) % 3, (i + 2) % 3
        s = math.sqrt(R[i, i] - R[j, j] - R[k, k] + 1.0) * 2
        q = [0.0] * 4
        q[i] = 0.25 * s
        q[j] = (R[j, i] + R[i, j]) / s
        q[k] = (R[k, i] + R[i, k]) / s
        q[3] = (R[k, j] - R[j, k]) / s
    q = np.array(q)
    return q / np.linalg.norm(q) * (1 if q[3] >= 0 else -1)


@dataclass
class Trajectory:
    """Analytic trajectory: position p(t) (world) and orientation R(t) (body->world).
    The orientation is defined through the camera (optical axis along the heading,
    image y pointing down) so that any T_cam_imu sees the landmark cloud."""
    kind: str = "euroc"
    speed: float = 1.0
    phase: float = 0.0
    amp: float = 1.0
    R_b2c: np.ndarray = None
    stops: tuple = ()                # (t_begin, t_end) intervals during which the platform stands still
    stop_ramp: float = 0.4           # seconds of smooth deceleration / acceleration around a stop

    def _warp(self, t):
        """Trajectory time tau(t): tau' = 1 outside the stops, 0 inside, C^2 ramps in between."""
        tau = t
        r = self.stop_ramp
        for (a, b) in self.stops:
            def ramp_int(x):         # integral of the smootherstep 6x^5-15x^4+10x^3 on [0, x]
                x = min(max(x, 0.0), 1.0)
                return x ** 6 - 3 * x ** 5 + 2.5 * x ** 4
            # bump(t) = s((t-a)/r) on [a, a+r], 1 on [a+r, b-r], 1 - s((t-(b-r))/r) on [b-r, b]
            up = r * ramp_int((t - a) / r)
            flat = min(max(t - (a + r), 0.0), max(b - r - (a + r), 0.0))
            x = min(max((t - (b - r)) / r, 0.0), 1.0)
            down = r * (x - ramp_int(x))
            tau -= up + flat + down
        return tau

    @staticmethod
    def _cam_frame(psi):
        c, s = math.cos(psi), math.sin(psi)
        return np.array([[s, 0.0, c], [-c, 0.0, s], [0.0, -1.0, 0.0]])   # columns x_c, y_c, z_c

    def pose(self, t):
        if self.stops:
            t = self._warp(t)
        if self.kind == "kitti":
            v0 = 10.0 * self.speed
            k = 0.05
            x = v0 * t
            y = v0 * 0.15 * (-math.cos(k * t + self.phase) + math.cos(self.phase)) / k
            z = 0.2 * math.sin(0.3 * t + self.phase)
            psi = math.atan2(0.15 * math.sin(k * t + self.phase), 1.0)
            wob = _rot_zyx(0.01 * math.sin(0.9 * t), 0.02 * math.sin(0.7 * t), 0.02 * math.cos(0.5 * t))
            p = np.array([x, y, z])
        else:
            w = 0.35 * self.speed
            a, b = 4.0 * self.amp, 3.0 * self.amp
            p = np.array([a * math.cos(w * t + self.phase), b * math.sin(w * t + self.phase),
                          1.0 + 0.5 * math.sin(2 * w * t)])
            psi = math.atan2(b * math.cos(w * t + self.phase), -a * math.sin(w * t + self.phase))
            psi += 0.3 * math.sin(0.5 * t)
            wob = _rot_zyx(0.05 * math.sin(0.9 * t), 0.08 * math.sin(0.7 * t + self.phase),
                           0.08 * math.cos(0.8 * t))
        R_c2w = self._cam_frame(psi) @ wob
        return p, R_c2w @ self.R_b2c

    def kinematics(self, t, h=1e-4):
        """(p, R, v, body angular rate, body specific force) by central differences."""
        p0, R0 = self.pose(t)
        pp, Rp = self.pose(t + h)
        pm, Rm = self.pose(t - h)
        v = (pp - pm) / (2 * h)
        acc = (pp - 2 * p0 + pm) / (h * h)
        Rd = (Rp - Rm) / (2 * h)
        Wx = R0.T @ Rd
        w = np.array([Wx[2, 1] - Wx[1, 2], Wx[0, 2] - Wx[2, 0], Wx[1, 0] - Wx[0, 1]]) / 2
        f = R0.T @ (acc - GRAVITY)
        return p0, R0, v, w, f


@dataclass
class SynthSpec:
    config: str = "euroc"            # which reference config the shapes/noise follow
    seed: int = 0
    n_frames: int = 60
    feats_per_frame: int = 300
    t0: float = 10.0
    img_offset: float = 0.001        # image stamps sit 1 ms after an IMU stamp -> dt != 0
    n_landmarks: int = 6000
    drop_prob: float = 0.03          # per-frame chance a track is lost early
    imu_noise_scale: float = 0.1     # true IMU noise = scale x the (inflated) config densities
    init_prob: float = 0.5           # chance a new track carries u_init/v_init
    gyro_bias: tuple = (0.002, -0.001, 0.0015)
    acc_bias: tuple = (0.02, 0.01, -0.015)
    overrides: dict = field(default_factory=dict)
    stops: tuple = ()                # stand-still intervals (ZUPT test sequences)
    feat_noise_scale: float = 1.0    # true pixel noise = scale x the noise the filter assumes (0: noise-free tracks)


def _extrinsics(cfg):
    T = np.array(cfg["T_cam_imu"], dtype=float).reshape(4, 4)
    R_b2c = T[:3, :3]                    # = R_imu_cam0 after the reference's double inverse
    t_c_b = -R_b2c.T @ T[:3, 3]          # camera origin in the body frame
    return R_b2c, t_c_b


def _trajectory(spec: SynthSpec, base):
    """The analytic trajectory of a sequence (depends on the seed, the config's extrinsics and the stops only; draws
    nothing from the random stream)."""
    k = spec.seed
    kind = "kitti" if spec.config == "kitti_odom" else "euroc"
    R_b2c, _ = _extrinsics(base)
    return Trajectory(kind=kind, speed=1.0 + 0.05 * ((k * 7) % 5), phase=0.37 * k,
                      amp=1.0 + 0.03 * (k % 4), R_b2c=R_b2c, stops=tuple(spec.stops))


def truth_states(spec: SynthSpec, times):
    """Ground truth of the sequence `spec` at arbitrary times, as (len(times), 17) records in the layout of the filter's
    state records: t, p (3), q xyzw (4), v (3), b_g (3), b_a (3) -- the biases are the spec's constant true biases.
    At an image stamp p and q are exactly the sequence's `gt` entry."""
    base = configs.make(spec.config, **spec.overrides)
    traj = _trajectory(spec, base)
    times = np.asarray(times, dtype=float).reshape(-1)
    out = np.zeros((len(times), 17))
    for i, t in enumerate(times):
        p, R, v, _, _ = traj.kinematics(float(t))
        out[i, 0] = t
        out[i, 1:4] = p
        out[i, 4:8] = _quat_xyzw(R)
        out[i, 8:11] = v
        out[i, 11:14] = spec.gyro_bias
        out[i, 14:17] = spec.acc_bias
    return out


def make_sequence(spec: SynthSpec):
    """Returns dict(cfg, imu (n,7), frames [(t, feats (k,9))], gt [(t,p,q)], init)."""
    k = spec.seed
    rng = np.random.default_rng(1000 + k)
    base = configs.make(spec.config, **spec.overrides)
    kind = "kitti" if spec.config == "kitti_odom" else "euroc"
    imu_rate = float(base["imu_rate"])
    img_dt = 1.0 / float(base["pub_frequency"])
    dt_imu = 1.0 / imu_rate
    R_b2c, t_c_b = _extrinsics(base)
    traj = _trajectory(spec, base)
    fx, fy = base["intrinsics"]["fx"], base["intrinsics"]["fy"]
    cx, cy = base["intrinsics"]["cx"], base["intrinsics"]["cy"]
    x_min, x_max = -cx / fx, (base["resolution_width"] - cx) / fx
    y_min, y_max = -cy / fy, (base["resolution_height"] - cy) / fy
    sig_f = float(base["noise_feature"])
    if spec.config == "kitti_odom":
        sig_f = 0.002                      # pixel-level noise; the filter still assumes sigma = 1
    sig_f *= spec.feat_noise_scale
    bg = np.array(spec.gyro_bias)
    ba = np.array(spec.acc_bias)

    t_end = spec.t0 + spec.n_frames * img_dt + 0.05
    n_imu = int(round((t_end - spec.t0 + 0.02) * imu_rate))
    imu = np.zeros((n_imu, 7))
    sg = spec.imu_noise_scale * float(base["noise_gyro"]) / math.sqrt(dt_imu)
    sa = spec.imu_noise_scale * float(base["noise_acc"]) / math.sqrt(dt_imu)
    for i in range(n_imu):
        t = spec.t0 - 0.01 + i * dt_imu
        _, _, _, w, f = traj.kinematics(t)
        imu[i, 0] = t
        imu[i, 1:4] = w + bg + rng.normal(0, sg, 3)
        imu[i, 4:7] = f + ba + rng.normal(0, sa, 3)

    # landmark cloud around the path
    if kind == "kitti":
        x0 = traj.pose(spec.t0)[0]
        x1 = traj.pose(t_end)[0]
        lm = np.column_stack([rng.uniform(x0[0] - 5, x1[0] + 70, spec.n_landmarks),
                              rng.uniform(min(x0[1], x1[1]) - 30, max(x0[1], x1[1]) + 30, spec.n_landmarks),
                              rng.uniform(-3, 8, spec.n_landmarks)])
        dmin, dmax = 5.0, 60.0
    else:
        lm = np.column_stack([rng.uniform(-12, 12, spec.n_landmarks),
                              rng.uniform(-12, 12, spec.n_landmarks),
                              rng.uniform(-4, 6, spec.n_landmarks)])
        dmin, dmax = 0.8, 18.0

    frames, gt = [], []
    tracked = {}          # landmark index -> (track id, prev u, prev v)
    next_id = 0
    prev_uv_all = None
    prev_t = None
    for fi in range(spec.n_frames):
        # image stamp: on the IMU grid + img_offset
        t_img = spec.t0 + round((fi + 1) * img_dt * imu_rate) * dt_imu + spec.img_offset
        p, R, _, _, _ = traj.kinematics(t_img)
        R_c2w = R @ R_b2c.T
        t_c_w = p + R @ t_c_b
        pc = (lm - t_c_w) @ R_c2w          # rows: R_c2w^T (lm - t)
        z = pc[:, 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            u = pc[:, 0] / z
            v = pc[:, 1] / z
        vis = (z > dmin) & (z < dmax) & (u > x_min) & (u < x_max) & (v > y_min) & (v < y_max)
        uv_noisy = np.column_stack([u, v]) + rng.normal(0, sig_f, (lm.shape[0], 2))
        frame_dt = (t_img - prev_t) if prev_t is not None else img_dt

        feats = []
        new_tracked = {}
        for li, (tid, pu, pv) in tracked.items():
            if not vis[li] or rng.random() < spec.drop_prob:
                continue
            cu, cv = uv_noisy[li]
            feats.append((tid, cu, cv, -1.0, -1.0, (cu - pu) / frame_dt, (cv - pv) / frame_dt, 0.0, 0.0))
            new_tracked[li] = (tid, cu, cv)
        room = spec.feats_per_frame - len(new_tracked)
        if room > 0:
            cand = np.flatnonzero(vis)
            cand = cand[~np.isin(cand, list(new_tracked.keys()))]
            rng.shuffle(cand)
            for li in cand[:room]:
                cu, cv = uv_noisy[li]
                tid = next_id
                next_id += 1
                if prev_uv_all is not None and prev_uv_all[1][li] and rng.random() < spec.init_prob:
                    iu, iv = prev_uv_all[0][li]
                    uvx, uvy = (cu - iu) / frame_dt, (cv - iv) / frame_dt
                    feats.append((tid, cu, cv, iu, iv, uvx, uvy, uvx, uvy))
                else:
                    feats.append((tid, cu, cv, -1.0, -1.0, 0.0, 0.0, 0.0, 0.0))
                new_tracked[li] = (tid, cu, cv)
        tracked = new_tracked
        prev_uv_all = (uv_noisy, vis)
        prev_t = t_img
        feats.sort(key=lambda f: f[0])
        frames.append((t_img, np.array(feats, dtype=float).reshape(-1, 9)))
        gt.append((t_img, p.copy(), _quat_xyzw(R)))

    p0, R0, v0, _, _ = traj.kinematics(spec.t0)
    init = dict(t=spec.t0, quat=_quat_xyzw(R0), pos=p0, vel=v0, bg=bg * 0.0, ba=ba * 0.0)
    cfg = configs.with_initial_state(base, init["t"], init["quat"], init["pos"], init["vel"],
                                     init["bg"], init["ba"])
    return dict(cfg=cfg, imu=imu, frames=frames, gt=gt, init=init, spec=spec)


def stress_snapshot(n_clones=30, n_features=2000, max_track_len=6, seed=0, full_tracks=False,
                    config="kitti_odom"):
    """Frozen-frame workload (BASELINE.json configs[3], SURVEY 8d case C4): a window of
    `n_clones` camera clones, `n_features` features each observed by m consecutive clones
    (m in [3, max_track_len], or m = n_clones when full_tracks), a plausible SPD covariance.

    Returns dict of flat arrays in the layout of the C ABI's snapshot entry points."""
    rng = np.random.default_rng(1000 + seed)
    base = configs.make(config)
    R_b2c, t_c_b = _extrinsics(base)
    traj = Trajectory(kind="kitti" if config == "kitti_odom" else "euroc", R_b2c=R_b2c)
    img_dt = 0.1
    N = n_clones
    clone_R = np.zeros((N, 9))
    clone_p = np.zeros((N, 3))
    cam_R = np.zeros((N, 3, 3))
    cam_t = np.zeros((N, 3))
    for i in range(N):
        p, R, _, _, _ = traj.kinematics(5.0 + i * img_dt)
        # small pose error so residuals are not pure noise-free
        clone_R[i] = R.ravel()
        clone_p[i] = p
        cam_R[i] = R @ R_b2c.T
        cam_t[i] = p + R @ t_c_b
    D = 22 + 6 * N
    A = rng.normal(0, 1, (D, D)) * 0.02
    P = A @ A.T * 0.05 + np.diag(np.concatenate([
        np.full(3, 4e-4), np.full(3, 0.05), np.full(3, 0.02), np.full(3, 4e-4), np.full(3, 0.01),
        np.zeros(7), np.tile(np.concatenate([np.full(3, 4e-4), np.full(3, 0.02)]), N)]))
    P[15:22, :] = 0.0
    P[:, 15:22] = 0.0
    sig = 0.002 if config == "kitti_odom" else float(base["noise_feature"])
    obs_clone, obs_z, feat_off = [], [], [0]
    for f in range(n_features):
        m = N if full_tracks else int(rng.integers(3, max_track_len + 1))
        s = int(rng.integers(0, N - m + 1))
        # a landmark in front of the middle camera of its track
        mid = s + m // 2
        depth = rng.uniform(6.0, 40.0)
        ray = np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.2, 0.2), 1.0]) * depth
        pw = cam_R[mid] @ ray + cam_t[mid]
        for c in range(s, s + m):
            pc = cam_R[c].T @ (pw - cam_t[c])
            obs_clone.append(c)
            obs_z.append(pc[:2] / pc[2] + rng.normal(0, sig, 2))
        feat_off.append(len(obs_clone))
    return dict(cfg=base, n_clones=N, clone_R=clone_R, clone_p=clone_p, P=P,
                R_b2c=R_b2c, t_c_b=t_c_b,
                feat_off=np.array(feat_off, dtype=np.int32),
                obs_clone=np.array(obs_clone, dtype=np.int32),
                obs_z=np.array(obs_z, dtype=float))
