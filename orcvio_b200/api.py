"""ctypes binding of liborcvio_b200.so: a host-side mirror of the reference's
`orcvio::OrcVIO` class (include/orcvio/orcvio.h:39-119) plus the batch and stage-level
entry points declared in include/orcvio_b200.h.

Everything numerical happens in the CUDA library; this module only marshals NumPy arrays.
If the library is missing it is built on import (nvcc); if it cannot be loaded the import
fails loudly -- there is no Python/NumPy fallback path.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBPATH = os.path.join(_HERE, "lib", "liborcvio_b200.so")


class OrcvioFeature(C.Structure):
    _fields_ = [("id", C.c_ulonglong), ("u", C.c_double), ("v", C.c_double),
                ("u_init", C.c_double), ("v_init", C.c_double),
                ("u_vel", C.c_double), ("v_vel", C.c_double),
                ("u_init_vel", C.c_double), ("v_init_vel", C.c_double)]


class OrcvioImu(C.Structure):
    _fields_ = [("t", C.c_double), ("gyro", C.c_double * 3), ("acc", C.c_double * 3)]


class OrcvioState(C.Structure):
    _fields_ = [("state_id", C.c_longlong), ("time", C.c_double), ("R", C.c_double * 9),
                ("p", C.c_double * 3), ("v", C.c_double * 3), ("bg", C.c_double * 3),
                ("ba", C.c_double * 3), ("P_pose", C.c_double * 36), ("P_vel", C.c_double * 9),
                ("n_clones", C.c_int), ("dim", C.c_int), ("n_map_features", C.c_int)]


class OrcvioFrameStats(C.Structure):
    _fields_ = [("n_candidates_lost", C.c_int), ("n_tri_invalid_lost", C.c_int),
                ("n_gate_pass_lost", C.c_int), ("n_candidates_prune", C.c_int),
                ("n_tri_invalid_prune", C.c_int), ("n_gate_pass_prune", C.c_int),
                ("n_removed_clones", C.c_int), ("removed_ids", C.c_longlong * 2), ("zupt", C.c_int),
                ("zupt_chi2", C.c_double), ("zupt_vnorm", C.c_double)]


FEAT_DTYPE = np.dtype([("id", "<u8"), ("u", "<f8"), ("v", "<f8"), ("u_init", "<f8"), ("v_init", "<f8"),
                       ("u_vel", "<f8"), ("v_vel", "<f8"), ("u_init_vel", "<f8"), ("v_init_vel", "<f8")])
IMU_DTYPE = np.dtype([("t", "<f8"), ("gyro", "<f8", 3), ("acc", "<f8", 3)])
assert FEAT_DTYPE.itemsize == C.sizeof(OrcvioFeature) and IMU_DTYPE.itemsize == C.sizeof(OrcvioImu)

_lib = None


def lib():
    """Load (building first if needed) the CUDA library.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("ORCVIO_LIB", _LIBPATH)     # (diagnostics: another build of the same library)
    if not os.path.exists(path):
        _build.build()
    L = C.CDLL(path)
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_void_p
    L.orcvio_create.restype = vp
    L.orcvio_create.argtypes = [C.c_char_p]
    L.orcvio_destroy.argtypes = [vp]
    L.orcvio_initialize.argtypes = [vp]
    L.orcvio_set_initial_state.argtypes = [vp, C.c_double, dp, dp, dp, dp, dp]
    L.orcvio_process_features.argtypes = [vp, C.c_double, vp, C.c_int, vp, ip]
    L.orcvio_get_state.argtypes = [vp, C.POINTER(OrcvioState)]
    L.orcvio_get_cov.argtypes = [vp, dp, C.c_int, ip]
    L.orcvio_set_cov.argtypes = [vp, dp, C.c_int]
    L.orcvio_get_window.argtypes = [vp, dp, C.POINTER(C.c_longlong), dp, C.c_int]
    L.orcvio_get_frame_stats.argtypes = [vp, C.POINTER(OrcvioFrameStats)]
    L.orcvio_get_map_points.argtypes = [vp, C.POINTER(C.c_longlong), dp, C.c_int]
    L.orcvio_get_candidate_log.argtypes = [vp, C.POINTER(C.c_longlong), ip, ip, dp, C.c_int]
    L.orcvio_get_feature_states.argtypes = [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), dp, dp, dp, C.c_int]
    L.orcvio_get_hybrid_log.argtypes = [vp, C.c_int, C.POINTER(C.c_longlong), ip, dp, C.c_int]
    L.orcvio_batch_create.restype = vp
    L.orcvio_batch_create.argtypes = [C.c_char_p, C.c_int]
    L.orcvio_batch_destroy.argtypes = [vp]
    L.orcvio_batch_set_initial_state.argtypes = [vp, C.c_int, C.c_double, dp, dp, dp, dp, dp]
    L.orcvio_batch_process.argtypes = [vp, dp, vp, ip, vp, ip, ip, ip]
    L.orcvio_batch_get_state.argtypes = [vp, C.c_int, C.POINTER(OrcvioState)]
    L.orcvio_batch_replay.argtypes = [vp, C.c_int, dp, vp, ip, vp, ip, C.c_double, dp, ip]
    L.orcvio_batch_replay_states.argtypes = [vp, C.c_int, dp, vp, ip, vp, ip, C.c_double, dp, ip, dp, dp]
    L.orcvio_trajectory_metrics.argtypes = [dp, dp, C.c_int, C.c_int, dp]
    L.orcvio_trajectory_nees.argtypes = [dp, dp, dp, C.c_int, C.c_int, C.c_int, dp, dp]
    L.orcvio_nees_summary.argtypes = [dp, C.c_int, C.c_int, dp]
    L.orcvio_get_tcw.argtypes = [vp, dp, dp]
    L.orcvio_set_pose_log.argtypes = [vp, C.c_char_p]
    L.orcvio_batch_get_cov.argtypes = [vp, C.c_int, dp, C.c_int, ip]
    L.orcvio_batch_get_frame_stats.argtypes = [vp, C.c_int, C.POINTER(OrcvioFrameStats)]
    L.orcvio_batch_feature_updates.restype = C.c_longlong
    L.orcvio_batch_feature_updates.argtypes = [vp]
    L.orcvio_batch_kernel_launches.restype = C.c_longlong
    L.orcvio_batch_kernel_launches.argtypes = [vp]
    L.orcvio_batch_set_profiling.argtypes = [vp, C.c_int]
    L.orcvio_batch_get_phase_times.argtypes = [vp, dp, C.POINTER(C.c_longlong)]
    L.orcvio_chi2_quantile.restype = C.c_double
    L.orcvio_chi2_quantile.argtypes = [C.c_double, C.c_int]
    L.orcvio_version.restype = C.c_char_p
    L.orcvio_set_device.argtypes = [C.c_int]
    L.orcvio_fp64_peak.argtypes = [dp, dp]
    L.orcvio_latency_probe.argtypes = [dp]
    L.orcvio_chol_probe.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp, C.POINTER(C.c_longlong), C.c_int,
                                    C.POINTER(C.c_float)]
    L.orcvio_triangulate.argtypes = [dp, dp, C.c_int, ip, ip, dp, C.c_int, C.c_double, C.c_double,
                                     C.c_double, dp, ip, ip, dp]
    L.orcvio_snapshot_update.argtypes = [dp, dp, C.c_int, dp, dp, dp, ip, ip, dp, C.c_int, C.c_int,
                                         C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                         dp, dp, ip, dp, dp, dp, C.POINTER(C.c_float), C.c_int]
    L.orcvio_measurement_jacobians.argtypes = [dp, dp, C.c_int, dp, dp, dp, ip, ip, dp, C.c_int, C.c_int,
                                               dp, dp, dp, dp]
    L.orcvio_object_residuals.argtypes = [dp, C.c_int, dp, dp, dp, C.c_int, dp, dp, C.c_int, dp, dp, dp,
                                          ip, dp, ip]
    L.orcvio_construct_object_jacobians.argtypes = [vp, dp, C.c_int, dp, C.c_int, dp, C.c_int, dp, ip, dp,
                                                    dp, dp, dp, ip]
    L.orcvio_remove_lost_objects.argtypes = [vp, dp, dp, dp, C.c_int, C.c_int, ip, dp]
    L.orcvio_set_state_cov.argtypes = [vp, C.c_int, C.c_int]
    L.orcvio_set_win_pose_timestamps.argtypes = [vp, dp, C.c_int]
    L.orcvio_fix_dcampose_dimupose_to_i.argtypes = [vp]
    L.orcvio_propagate.argtypes = [dp, dp, dp, dp, dp, vp, C.c_int, dp, C.c_int, C.c_int, dp]
    fpt = C.POINTER(C.c_float)
    L.orcvio_frame_create.restype = vp
    L.orcvio_frame_create.argtypes = [C.c_int, C.c_int] + [C.c_double] * 5
    L.orcvio_frame_destroy.argtypes = [vp]
    L.orcvio_frame_update.argtypes = [vp, dp, dp, C.c_int, dp, dp, dp, ip, ip, dp, C.c_int, dp, dp, ip, dp, dp]
    L.orcvio_frame_update_pose_cov.argtypes = [vp, dp, dp, C.c_int, dp, dp, dp, ip, ip, dp, C.c_int, dp, dp, ip, dp, dp]
    L.orcvio_frame_load.argtypes = [vp, dp, dp, C.c_int, dp, dp, dp, ip, ip, dp, C.c_int]
    L.orcvio_frame_run.argtypes = [vp, C.c_int, fpt, fpt]
    L.orcvio_frame_fetch.argtypes = [vp, dp, dp, ip, dp, dp]
    L.orcvio_frame_kernel_launches.restype = C.c_longlong
    L.orcvio_frame_kernel_launches.argtypes = [vp]
    L.orcvio_frame_host_times.argtypes = [vp, C.POINTER(C.c_float)]
    L.orcvio_frame_kernel_times.argtypes = [vp, C.POINTER(C.c_float)]
    _lib = L
    return L


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int)) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def feats_array(feats):
    """(k, 9) float array [id,u,v,u_init,v_init,u_vel,v_vel,u_init_vel,v_init_vel] -> struct array."""
    feats = np.asarray(feats, dtype=np.float64).reshape(-1, 9)
    out = np.zeros(feats.shape[0], dtype=FEAT_DTYPE)
    out["id"] = feats[:, 0].astype(np.uint64)
    for k, name in enumerate(FEAT_DTYPE.names[1:], start=1):
        out[name] = feats[:, k]
    return out


def imu_array(imu):
    """(n, 7) float array [t, w, a] -> struct array."""
    imu = np.asarray(imu, dtype=np.float64).reshape(-1, 7)
    out = np.zeros(imu.shape[0], dtype=IMU_DTYPE)
    out["t"] = imu[:, 0]
    out["gyro"] = imu[:, 1:4]
    out["acc"] = imu[:, 4:7]
    return out


class OrcVIO:
    """Mirror of orcvio::OrcVIO for the filter-update path (same method names)."""

    def __init__(self, config_file):
        self._L = lib()
        self._h = self._L.orcvio_create(str(config_file).encode())
        self._imu = np.zeros(0, dtype=IMU_DTYPE)     # the caller-owned imu_msg_buffer

    def __del__(self):
        try:
            if self._h:
                self._L.orcvio_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def initialize(self):
        return bool(self._L.orcvio_initialize(self._h))

    def set_initial_state(self, t, quat_xyzw, p, v, bg=(0, 0, 0), ba=(0, 0, 0)):
        a = [_f64(x) for x in (quat_xyzw, p, v, bg, ba)]
        return self._L.orcvio_set_initial_state(self._h, float(t), *[_dp(x) for x in a])

    def push_imu(self, imu):
        """Append samples to the IMU buffer (the reference's caller does imu_msg_buffer.push_back)."""
        self._imu = np.concatenate([self._imu, imu_array(imu)])

    def processFeatures(self, t_img, feats):
        f = feats if (isinstance(feats, np.ndarray) and feats.dtype == FEAT_DTYPE) else feats_array(feats)
        n = C.c_int(len(self._imu))
        buf = np.ascontiguousarray(self._imu)
        rc = self._L.orcvio_process_features(self._h, float(t_img), f.ctypes.data, len(f), buf.ctypes.data,
                                             C.byref(n))
        if rc < 0:
            raise RuntimeError(f"orcvio_process_features failed: {rc}")
        self._imu = buf[:n.value].copy()
        return bool(rc)

    def state(self):
        s = OrcvioState()
        rc = self._L.orcvio_get_state(self._h, C.byref(s))
        if rc != 0:
            raise RuntimeError(f"orcvio_get_state failed: {rc}")
        return s

    def cov(self):
        d = C.c_int(0)
        self._L.orcvio_get_cov(self._h, None, 0, C.byref(d))
        P = np.zeros((d.value, d.value))
        rc = self._L.orcvio_get_cov(self._h, _dp(P), P.size, C.byref(d))
        if rc != 0:
            raise RuntimeError(f"orcvio_get_cov failed: {rc}")
        return P

    def set_cov(self, P):
        P = _f64(P)
        return self._L.orcvio_set_cov(self._h, _dp(P), P.shape[0])

    def window(self):
        cap = 64
        poses = np.zeros((cap, 12))
        ids = np.zeros(cap, dtype=np.int64)
        times = np.zeros(cap)
        n = self._L.orcvio_get_window(self._h, _dp(poses), ids.ctypes.data_as(C.POINTER(C.c_longlong)),
                                      _dp(times), cap)
        return poses[:n], ids[:n], times[:n]

    def frame_stats(self):
        s = OrcvioFrameStats()
        self._L.orcvio_get_frame_stats(self._h, C.byref(s))
        return s

    def map_points(self, cap=65536):
        """getMSCKFMapPointPositions: (ids, xyz); xyz is NaN for features not yet initialised."""
        ids = np.zeros(cap, dtype=np.int64)
        xyz = np.zeros((cap, 3))
        n = self._L.orcvio_get_map_points(self._h, ids.ctypes.data_as(C.POINTER(C.c_longlong)), _dp(xyz), cap)
        return ids[:n], xyz[:n]

    def candidate_log(self, cap=65536):
        ids = np.zeros(cap, dtype=np.int64)
        ph = np.zeros(cap, dtype=np.int32)
        st = np.zeros(cap, dtype=np.int32)
        g = np.zeros(cap)
        n = self._L.orcvio_get_candidate_log(self._h, ids.ctypes.data_as(C.POINTER(C.c_longlong)), _ip(ph),
                                             _ip(st), _dp(g), cap)
        return ids[:n], ph[:n], st[:n], g[:n]

    def getTcw(self):
        """src/orcvio.cpp:2978-2988 -> (R camera->world 3x3, camera position)."""
        R = np.zeros(9)
        t = np.zeros(3)
        if self._L.orcvio_get_tcw(self._h, _dp(R), _dp(t)) != 0:
            raise RuntimeError("orcvio_get_tcw failed")
        return R.reshape(3, 3), t

    def set_pose_log(self, path):
        """The state_est_geo_feat.txt side effect of processFeatures (src/orcvio.cpp:422, 640-645)."""
        return self._L.orcvio_set_pose_log(self._h, None if path is None else str(path).encode())

    def feature_states(self, cap=256):
        """state_server.feature_states (hybrid mode) in state order:
        (ids, anchor state ids, inverse depths, obs_anchor (n, 2), world positions (n, 3))."""
        ll = C.POINTER(C.c_longlong)
        ids = np.zeros(cap, dtype=np.int64)
        anc = np.zeros(cap, dtype=np.int64)
        rho = np.zeros(cap)
        oa = np.zeros((cap, 2))
        xyz = np.zeros((cap, 3))
        n = self._L.orcvio_get_feature_states(self._h, ids.ctypes.data_as(ll), anc.ctypes.data_as(ll), _dp(rho),
                                              _dp(oa), _dp(xyz), cap)
        return ids[:n], anc[:n], rho[:n], oa[:n], xyz[:n]

    def getStableMapPointPositions(self):
        """src/orcvio.cpp:3046-3051 (the reference returns its whole `map_points` archive; the features of the state
        are the ones this path maintains)."""
        return self.feature_states()[4]

    def getActiveMapPointPositions(self):
        """src/orcvio.cpp:3053-3058."""
        return self.feature_states()[4]

    def hybrid_log(self, cap=4096):
        """EKF-SLAM branches of the last frame: dict(ekf_lost, ekf {id: (pass, gamma)}, new {id: (entered, gamma)},
        reanchored {id: (old anchor, new anchor)})."""
        ll = C.POINTER(C.c_longlong)
        out = {}
        for what, name in ((0, "ekf_lost"), (1, "ekf"), (2, "new"), (3, "reanchored")):
            ids = np.zeros(cap, dtype=np.int64)
            fl = np.zeros(cap, dtype=np.int32)
            g = np.zeros(cap)
            n = self._L.orcvio_get_hybrid_log(self._h, what, ids.ctypes.data_as(ll), _ip(fl), _dp(g), cap)
            if what == 0:
                out[name] = [int(i) for i in ids[:n]]
            elif what == 3:
                out[name] = {int(ids[3 * k]): (int(ids[3 * k + 1]), int(ids[3 * k + 2])) for k in range(n // 3)}
            else:
                out[name] = {int(i): (bool(f), float(x)) for i, f, x in zip(ids[:n], fl[:n], g[:n])}
        return out

    # -- object path (stage 3, filter side)
    def setStateCov(self, imu_dim, num_clone):
        self._dim_override = imu_dim + 6 * num_clone
        return self._L.orcvio_set_state_cov(self._h, imu_dim, num_clone)

    def setWinPoseTimestamps(self, ts):
        ts = _f64(ts)
        return self._L.orcvio_set_win_pose_timestamps(self._h, _dp(ts), len(ts))

    def fixDcamposeDimuposeToI(self):
        return self._L.orcvio_fix_dcampose_dimupose_to_i(self._h)

    def constructObjectResidualJacobians(self, jac_sensor, timestamps, Hf, res, zs_num, cam_pose_se3):
        jac = np.asfortranarray(jac_sensor, dtype=np.float64)
        Hf_ = np.asfortranarray(Hf, dtype=np.float64)
        res_ = _f64(res)
        ts = _f64(timestamps)
        zn = _i32(zs_num)
        se3 = np.asfortranarray(cam_pose_se3, dtype=np.float64)
        rows, odim = Hf_.shape
        d = C.c_int(0)
        self._L.orcvio_get_cov(self._h, None, 0, C.byref(d))
        if getattr(self, "_dim_override", None):
            d = C.c_int(self._dim_override)
        Hx_o = np.zeros((rows, d.value), order="F")
        Hf_o = np.zeros((rows, odim), order="F")
        res_o = np.zeros(rows)
        ro = C.c_int(0)
        flag = self._L.orcvio_construct_object_jacobians(
            self._h, _dp(jac), rows, _dp(ts), len(ts), _dp(Hf_), odim, _dp(res_), _ip(zn), _dp(se3),
            _dp(Hx_o), _dp(Hf_o), _dp(res_o), C.byref(ro))
        if flag < 0:
            raise RuntimeError(f"orcvio_construct_object_jacobians failed: {flag}")
        n = ro.value
        return bool(flag), Hx_o[:n], Hf_o[:n], res_o[:n]

    def removeLostObjects(self, Hx, Hf, res):
        Hx_ = np.asfortranarray(Hx, dtype=np.float64)
        Hf_ = np.asfortranarray(Hf, dtype=np.float64)
        res_ = _f64(res)
        st = C.c_int(0)
        g = C.c_double(0)
        rc = self._L.orcvio_remove_lost_objects(self._h, _dp(Hx_), _dp(Hf_), _dp(res_), Hx_.shape[0],
                                                Hf_.shape[1], C.byref(st), C.byref(g))
        if rc < 0:
            raise RuntimeError(f"orcvio_remove_lost_objects failed: {rc}")
        return st.value, g.value


class Batch:
    """n independent filters advanced in lock-step (multi-trajectory mode, SURVEY 8e)."""

    def __init__(self, config_file, n):
        self._L = lib()
        self.n = n
        self._h = self._L.orcvio_batch_create(str(config_file).encode(), n)
        if not self._h:
            raise RuntimeError("orcvio_batch_create failed (no CUDA device or unsupported config)")

    def __del__(self):
        try:
            if self._h:
                self._L.orcvio_batch_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def set_initial_state(self, i, t, quat_xyzw, p, v, bg=(0, 0, 0), ba=(0, 0, 0)):
        a = [_f64(x) for x in (quat_xyzw, p, v, bg, ba)]
        return self._L.orcvio_batch_set_initial_state(self._h, i, float(t), *[_dp(x) for x in a])

    def process(self, t_img, feats, feat_off, imu, imu_off):
        """feats / imu: struct arrays concatenated over filters, *_off CSR offsets (n+1)."""
        t_img = _f64(t_img)
        feat_off = _i32(feat_off)
        imu_off = _i32(imu_off)
        used = np.zeros(self.n, dtype=np.int32)
        pub = np.zeros(self.n, dtype=np.int32)
        rc = self._L.orcvio_batch_process(self._h, _dp(t_img), feats.ctypes.data, _ip(feat_off),
                                          imu.ctypes.data, _ip(imu_off), _ip(used), _ip(pub))
        if rc != 0:
            raise RuntimeError(f"orcvio_batch_process failed: {rc}")
        return used, pub

    def _replay_args(self, t_img, feats, feat_off, imus, imu_window):
        """(n, F, the inputs of orcvio_batch_replay[_states] up to imu_window); the arrays stay referenced by the tuple."""
        t_img = np.ascontiguousarray(t_img, dtype=np.float64)
        n, F = t_img.shape
        assert n == self.n
        feat_off = np.ascontiguousarray(feat_off, dtype=np.int32)
        fptr = (C.c_void_p * n)(*[f.ctypes.data for f in feats])
        iptr = (C.c_void_p * n)(*[m.ctypes.data for m in imus])
        n_imu = np.array([len(m) for m in imus], dtype=np.int32)
        return n, F, (F, _dp(t_img), fptr, _ip(feat_off), iptr, _ip(n_imu), float(imu_window))

    def replay(self, t_img, feats, feat_off, imus, imu_window=0.02):
        """Whole-sequence replay (orcvio_batch_replay).  t_img (n, F); feats: list of n struct arrays (all frames of a
        filter concatenated); feat_off (n, F + 1); imus: list of n struct arrays.  Returns (poses (n, F, 7), ok (n,)).
        The call releases the GIL: several batches replay concurrently from Python threads."""
        n, F, args = self._replay_args(t_img, feats, feat_off, imus, imu_window)
        poses = np.zeros((n, F, 7))
        ok = np.zeros(n, dtype=np.int32)
        rc = self._L.orcvio_batch_replay(self._h, *args, _dp(poses), _ip(ok))
        if rc != 0:
            raise RuntimeError(f"orcvio_batch_replay failed: {rc}")
        return poses, ok

    def replay_states(self, t_img, feats, feat_off, imus, imu_window=0.02, states=True, cov=True):
        """replay() that also records, after every frame, the IMU state (n, F, 17: t, p, q xyzw, v, bg, ba) and the
        leading 15 x 15 block of the covariance (n, F, 15, 15; error state [theta, v, p, b_g, b_a]), captured on the
        device (orcvio_batch_replay_states).  Returns (poses, ok, states, cov15); a record not asked for is None."""
        n, F, args = self._replay_args(t_img, feats, feat_off, imus, imu_window)
        poses = np.zeros((n, F, 7))
        ok = np.zeros(n, dtype=np.int32)
        st = np.zeros((n, F, 17)) if states else None
        cv = np.zeros((n, F, 15, 15)) if cov else None
        rc = self._L.orcvio_batch_replay_states(self._h, *args, _dp(poses), _ip(ok), _dp(st), _dp(cv))
        if rc != 0:
            raise RuntimeError(f"orcvio_batch_replay_states failed: {rc}")
        return poses, ok, st, cv

    def state(self, i):
        s = OrcvioState()
        self._L.orcvio_batch_get_state(self._h, i, C.byref(s))
        return s

    def cov(self, i):
        d = C.c_int(0)
        self._L.orcvio_batch_get_cov(self._h, i, None, 0, C.byref(d))
        P = np.zeros((d.value, d.value))
        self._L.orcvio_batch_get_cov(self._h, i, _dp(P), P.size, C.byref(d))
        return P

    def frame_stats(self, i):
        s = OrcvioFrameStats()
        self._L.orcvio_batch_get_frame_stats(self._h, i, C.byref(s))
        return s

    def feature_updates(self):
        return int(self._L.orcvio_batch_feature_updates(self._h))

    def kernel_launches(self):
        return int(self._L.orcvio_batch_kernel_launches(self._h))

    def set_profiling(self, on):
        self._L.orcvio_batch_set_profiling(self._h, int(on))

    def phase_times(self):
        ms = np.zeros(6)
        n = np.zeros(6, dtype=np.int64)
        self._L.orcvio_batch_get_phase_times(self._h, _dp(ms), n.ctypes.data_as(C.POINTER(C.c_longlong)))
        names = ["tri", "jac_gate", "qr_tiles", "qr_chain", "update", "propagate"]
        return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(names)}


class Frame:
    """Persistent frozen-frame updater (orcvio_frame_*): the 'stack -> compress -> update'
    chain of removeLostFeatures on one frame, reused for a stream of frames."""

    STAGES = ["tri", "jac_gate", "qr_tiles", "qr_chain", "update", "total"]

    def __init__(self, n_clones_cap=30, flags=0, noise_var=1.0, chi2_p=0.95, translation_threshold=-1.0,
                 cost_threshold=4.7673e-4, init_final_dist_threshold=5.0):
        self._L = lib()
        self._h = self._L.orcvio_frame_create(n_clones_cap, flags, noise_var, chi2_p, translation_threshold,
                                              cost_threshold, init_final_dist_threshold)
        if not self._h:
            raise RuntimeError("orcvio_frame_create failed (no CUDA device: there is no CPU fallback)")
        self._keep = None

    def __del__(self):
        try:
            if self._h:
                self._L.orcvio_frame_destroy(self._h)
                self._h = None
        except Exception:
            pass

    @staticmethod
    def _inputs(snap):
        N = int(snap["n_clones"])
        return dict(N=N, clone_R=_f64(snap["clone_R"]).reshape(N, 9), clone_p=_f64(snap["clone_p"]).reshape(N, 3),
                    Rbc=_f64(snap["R_b2c"]).reshape(9), tcb=_f64(snap["t_c_b"]).reshape(3),
                    P=np.asfortranarray(snap["P"], dtype=np.float64), feat_off=_i32(snap["feat_off"]),
                    obs_clone=_i32(snap["obs_clone"]), obs_z=_f64(snap["obs_z"]).reshape(-1, 2))

    def _outputs(self, N, nf):
        D = 22 + 6 * N
        return dict(P=np.zeros((D, D), order="F"), delta_x=np.zeros(D), status=np.zeros(nf, dtype=np.int32),
                    gamma=np.zeros(nf), clones=np.zeros((N, 12)))

    def prepare_inputs(self, snap):
        return self._inputs(snap)

    def update(self, inp, out=None, full_P=True):
        """Host buffers in -> host buffers out (the per-frame call of a host integration).  full_P=False: only the
        leading 9 x 9 block of the posterior comes back (out["P_lead9"]), orcvio_frame_update_pose_cov."""
        if not isinstance(inp, dict) or "Rbc" not in inp:
            inp = self._inputs(inp)
        nf = len(inp["feat_off"]) - 1
        if out is None:
            out = self._outputs(inp["N"], nf)
        if not full_P:
            if "P_lead9" not in out:
                out["P_lead9"] = np.zeros((9, 9))
            pi = inp.get("_ptrs")
            if pi is None:
                pi = inp["_ptrs"] = (_dp(inp["clone_R"]), _dp(inp["clone_p"]), inp["N"], _dp(inp["Rbc"]), _dp(inp["tcb"]),
                                     _dp(inp["P"]), _ip(inp["feat_off"]), _ip(inp["obs_clone"]), _dp(inp["obs_z"]), nf)
            pl = out.get("_ptrs_lite")
            if pl is None:
                pl = out["_ptrs_lite"] = (_dp(out["P_lead9"]), _dp(out["delta_x"]), _ip(out["status"]), _dp(out["gamma"]),
                                          _dp(out["clones"]))
            rc = self._L.orcvio_frame_update_pose_cov(self._h, *pi, *pl)
            if rc != 0:
                raise RuntimeError(f"orcvio_frame_update_pose_cov failed: {rc}")
            return out
        # the ctypes pointer objects are cached on the buffers' dicts: building 14 of them costs more than the
        # GPU spends on a stage of the frame
        pi = inp.get("_ptrs")
        if pi is None:
            pi = inp["_ptrs"] = (_dp(inp["clone_R"]), _dp(inp["clone_p"]), inp["N"], _dp(inp["Rbc"]), _dp(inp["tcb"]),
                                 _dp(inp["P"]), _ip(inp["feat_off"]), _ip(inp["obs_clone"]), _dp(inp["obs_z"]), nf)
        po = out.get("_ptrs")
        if po is None:
            po = out["_ptrs"] = (_dp(out["P"]), _dp(out["delta_x"]), _ip(out["status"]), _dp(out["gamma"]),
                                 _dp(out["clones"]))
        rc = self._L.orcvio_frame_update(self._h, *pi, *po)
        if rc != 0:
            raise RuntimeError(f"orcvio_frame_update failed: {rc}")
        return out

    def load(self, snap):
        inp = self._inputs(snap)
        self._keep = inp
        nf = len(inp["feat_off"]) - 1
        rc = self._L.orcvio_frame_load(
            self._h, _dp(inp["clone_R"]), _dp(inp["clone_p"]), inp["N"], _dp(inp["Rbc"]), _dp(inp["tcb"]),
            _dp(inp["P"]), _ip(inp["feat_off"]), _ip(inp["obs_clone"]), _dp(inp["obs_z"]), nf)
        if rc != 0:
            raise RuntimeError(f"orcvio_frame_load failed: {rc}")

    def run(self, repeat=1, stages=False):
        """Kernel chain on the resident frame; returns total device microseconds over `repeat`
        runs (and the mean per-stage microseconds when stages=True)."""
        tot = C.c_float(0)
        st = np.zeros(6, dtype=np.float32)
        rc = self._L.orcvio_frame_run(self._h, repeat, C.byref(tot),
                                      st.ctypes.data_as(C.POINTER(C.c_float)) if stages else None)
        if rc != 0:
            raise RuntimeError(f"orcvio_frame_run failed: {rc}")
        return (tot.value, dict(zip(self.STAGES, st.tolist()))) if stages else tot.value

    def fetch(self):
        inp = self._keep
        out = self._outputs(inp["N"], len(inp["feat_off"]) - 1)
        rc = self._L.orcvio_frame_fetch(self._h, _dp(out["P"]), _dp(out["delta_x"]), _ip(out["status"]),
                                        _dp(out["gamma"]), _dp(out["clones"]))
        if rc != 0:
            raise RuntimeError(f"orcvio_frame_fetch failed: {rc}")
        return out

    def kernel_launches(self):
        return int(self._L.orcvio_frame_kernel_launches(self._h))

    def host_times(self):
        """Wall-clock split (us) of the last update(): prepare, launch, wait+fetch, total."""
        us = (C.c_float * 4)()
        self._L.orcvio_frame_host_times(self._h, us)
        return dict(prepare=us[0], launch=us[1], wait_fetch=us[2], total=us[3])

    def kernel_times(self):
        """Device microseconds of k_syrk and k_chol_prior in the last run(stages=True)."""
        us = (C.c_float * 2)()
        self._L.orcvio_frame_kernel_times(self._h, us)
        return dict(syrk=us[0], chol_prior=us[1])


# ---------------------------------------------------------------- stage-level calls
def object_kabsch_init(mean_pts, world_pts, se2=False):
    """findTransform (+ poseSE32SE2) for a batch of objects: lists of (n_i, 3) arrays -> ((n_obj, 4, 4), ok)."""
    L = lib()
    L.orcvio_object_kabsch_init.argtypes = [C.POINTER(C.c_double)] * 2 + [C.POINTER(C.c_int), C.c_int, C.c_int,
                                                                        C.POINTER(C.c_double), C.POINTER(C.c_int)]
    off = np.zeros(len(mean_pts) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(m) for m in mean_pts])
    a = np.ascontiguousarray(np.concatenate([np.asarray(m, dtype=np.float64).reshape(-1, 3) for m in mean_pts]))
    b = np.ascontiguousarray(np.concatenate([np.asarray(w, dtype=np.float64).reshape(-1, 3) for w in world_pts]))
    assert a.shape == b.shape
    T = np.zeros((len(mean_pts), 4, 4))
    ok = np.zeros(len(mean_pts), dtype=np.int32)
    rc = L.orcvio_object_kabsch_init(_dp(a), _dp(b), _ip(off), len(mean_pts), int(bool(se2)), _dp(T), _ip(ok))
    if rc != 0:
        raise RuntimeError(f"orcvio_object_kabsch_init failed: {rc}")
    return T, ok


def _object_batch(frames_list, zs_list, zb_list=None):
    """Flattens per-object (T_i, 4, 4) / (T_i, K, 2) / (T_i, 4) arrays into the batch layout of the C ABI."""
    off = np.zeros(len(frames_list) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(f) for f in frames_list])
    frames = np.ascontiguousarray(np.concatenate([_f64(f).reshape(-1, 16) for f in frames_list]))
    K = np.asarray(zs_list[0]).shape[1]
    zs = np.ascontiguousarray(np.concatenate([_f64(z).reshape(-1, K, 2) for z in zs_list]))
    zb = None if zb_list is None else np.ascontiguousarray(np.concatenate([_f64(b).reshape(-1, 4) for b in zb_list]))
    return off, frames, zs, zb, K


class ObjectFeatureInitializer:
    """Mirror of orcvio::ObjectFeatureInitializer (include/orcvio/obj/ObjectFeatureInitializer.h) for a batch of objects
    of one class: same constructor arguments (mean ellipsoid shape, mean keypoints, residual weights; the camera
    intrinsics are the identity as everywhere in the reference) and the two methods the object branch calls."""

    def __init__(self, object_mean_shape, object_keypoints_mean, residual_weights=(1.0, 1.0, 1.0, 1.0)):
        self.mean_shape = _f64(object_mean_shape).reshape(3)
        self.kps_mean = _f64(object_keypoints_mean).reshape(-1, 3)
        self.weights = _f64(residual_weights).reshape(4)
        self.estimate_SE2_pose_flag = True       # hard-coded in the reference (ObjectFeatureInitializer.cpp:29)

    def single_object_initialization(self, frames_list, zs_list):
        """-> (ok (n_obj), wTq (n_obj, 4, 4), kp_world (n_obj, K, 3), kp_valid (n_obj, K))."""
        L = lib()
        off, frames, zs, _, K = _object_batch(frames_list, zs_list)
        assert K == len(self.kps_mean)
        n = len(frames_list)
        T = np.zeros((n, 4, 4))
        ok = np.zeros(n, dtype=np.int32)
        kw = np.zeros((n, K, 3))
        kv = np.zeros((n, K), dtype=np.int32)
        L.orcvio_object_init.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int,
                                         C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int),
                                         C.POINTER(C.c_double), C.POINTER(C.c_int)]
        rc = L.orcvio_object_init(n, _ip(off), _dp(frames), _dp(zs), K, _dp(self.kps_mean),
                                  int(self.estimate_SE2_pose_flag), _dp(T), _ip(ok), _dp(kw), _ip(kv))
        if rc != 0:
            raise RuntimeError(f"orcvio_object_init failed: {rc}")
        return ok, T, kw, kv

    def _lm_args(self, frames_list, zs_list, zb_list):
        off, frames, zs, zb, K = _object_batch(frames_list, zs_list, zb_list)
        assert K == len(self.kps_mean)
        return off, frames, zs, zb, K

    def single_levenberg_marquardt(self, frames_list, zs_list, zb_list, wTo_init, use_left_perturbation_flag=True,
                                   use_new_bbox_residual_flag=False):
        """-> dict(success, status, nfev, njev, fnorm, wTo, shape, kps, kps_world, rounds), arrays over the objects."""
        L = lib()
        off, frames, zs, zb, K = self._lm_args(frames_list, zs_list, zb_list)
        n = len(frames_list)
        w0 = np.ascontiguousarray(_f64(wTo_init).reshape(n, 16))
        out = dict(wTo=np.zeros((n, 4, 4)), shape=np.zeros((n, 3)), kps=np.zeros((n, K, 3)), kps_world=np.zeros((n, K, 3)),
                   status=np.zeros(n, dtype=np.int32), nfev=np.zeros(n, dtype=np.int32), njev=np.zeros(n, dtype=np.int32),
                   fnorm=np.zeros(n))
        rounds = C.c_int(0)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.orcvio_object_lm.argtypes = [C.c_int, ip, dp, dp, dp, C.c_int, dp, dp, dp, C.c_int, dp, dp, dp, dp, dp, ip, ip, ip,
                                       dp, ip]
        flags = (1 if use_left_perturbation_flag else 0) | (2 if use_new_bbox_residual_flag else 0)
        rc = L.orcvio_object_lm(n, _ip(off), _dp(frames), _dp(zs), _dp(zb), K, _dp(self.kps_mean), _dp(self.mean_shape),
                                _dp(self.weights), flags, _dp(w0), _dp(out["wTo"]), _dp(out["shape"]), _dp(out["kps"]),
                                _dp(out["kps_world"]), _ip(out["status"]), _ip(out["nfev"]), _ip(out["njev"]),
                                _dp(out["fnorm"]), C.byref(rounds))
        if rc != 0:
            raise RuntimeError(f"orcvio_object_lm failed: {rc}")
        out["rounds"] = rounds.value
        out["success"] = (out["status"] != 0) & (out["status"] != 5)
        return out

    def lm_eval(self, frames_list, zs_list, zb_list, states, use_left_perturbation_flag=True,
                use_new_bbox_residual_flag=False):
        """|f|, J^T f, J^T J of the ObjectLM model at `states` = list of (wTo, shape, kps)."""
        L = lib()
        off, frames, zs, zb, K = self._lm_args(frames_list, zs_list, zb_list)
        n = len(frames_list)
        nn = 9 + 3 * K
        xs = np.ascontiguousarray(np.stack([np.concatenate([_f64(w).reshape(16), _f64(s).reshape(3), _f64(k).reshape(3 * K)])
                                            for (w, s, k) in states]))
        out = np.zeros((n, 1 + nn + nn * nn))
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.orcvio_object_lm_eval.argtypes = [C.c_int, ip, dp, dp, dp, C.c_int, dp, dp, dp, C.c_int, dp, dp]
        flags = (1 if use_left_perturbation_flag else 0) | (2 if use_new_bbox_residual_flag else 0)
        rc = L.orcvio_object_lm_eval(n, _ip(off), _dp(frames), _dp(zs), _dp(zb), K, _dp(self.kps_mean), _dp(self.mean_shape),
                                     _dp(self.weights), flags, _dp(xs), _dp(out))
        if rc != 0:
            raise RuntimeError(f"orcvio_object_lm_eval failed: {rc}")
        return out[:, 0], out[:, 1:1 + nn], out[:, 1 + nn:].reshape(n, nn, nn)


def lm_known_answer(which):
    """The reference's Levenberg-Marquardt known-answer problems through the library's driver (no device needed)."""
    L = lib()
    x = np.zeros(4)
    st, nf, nj = C.c_int(0), C.c_int(0), C.c_int(0)
    fn = C.c_double(0)
    L.orcvio_lm_known_answer.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                         C.POINTER(C.c_int), C.POINTER(C.c_double)]
    rc = L.orcvio_lm_known_answer(which, _dp(x), C.byref(st), C.byref(nf), C.byref(nj), C.byref(fn))
    if rc != 0:
        raise RuntimeError(f"orcvio_lm_known_answer failed: {rc}")
    return dict(x=x[:{0: 3, 1: 1}.get(which, 2)], status=st.value, nfev=nf.value, njev=nj.value, fnorm=fn.value)


def trajectory_metrics(est_pose7, gt_pose7):
    """System::publishGroundtruth on the device for a batch of trajectories (orcvio_trajectory_metrics):
    (n, F, 7) poses (p, q xyzw) -> (n, 4): mean orientation error (deg), mean position error, position RMSE, final
    position error after first-pose alignment."""
    e = np.ascontiguousarray(est_pose7, dtype=np.float64)
    g = np.ascontiguousarray(gt_pose7, dtype=np.float64)
    assert e.shape == g.shape and e.ndim == 3 and e.shape[2] == 7
    out = np.zeros((e.shape[0], 4))
    rc = lib().orcvio_trajectory_metrics(_dp(e), _dp(g), e.shape[0], e.shape[1], _dp(out))
    if rc != 0:
        raise RuntimeError(f"orcvio_trajectory_metrics failed: {rc}")
    return out


NEES_BLOCKS = (("theta", 3), ("v", 3), ("p", 3), ("pose", 6), ("nav", 9), ("full", 15))


def nees_flags(cfg):
    """The orientation-error convention of a configuration: bit0 use_larvio_flag, bit1 use_left_perturbation_flag."""
    return (1 if int(cfg.get("use_larvio_flag", 0)) else 0) | (2 if int(cfg.get("use_left_perturbation_flag", 0)) else 0)


def trajectory_nees(est17, gt17, cov15, flags):
    """NEES of filter runs against their truth on the device (orcvio_trajectory_nees).  est17 / gt17 (n, F, 17) state
    records (t, p, q xyzw, v, bg, ba), cov15 (n, F, 15, 15), flags: bit0 use_larvio, bit1 use_left_perturbation.
    Returns (nees (n, F, 8): NEES theta, v, p, pose, nav, full, |dtheta| deg, |dp| m -- NaN rows where the block is not
    positive definite or an input is not finite;  summary (F, 9): per frame ANEES of the six blocks, RMS orientation error
    (deg), RMS position error (m), number of valid trajectories)."""
    e = np.ascontiguousarray(est17, dtype=np.float64)
    g = np.ascontiguousarray(gt17, dtype=np.float64)
    c = np.ascontiguousarray(cov15, dtype=np.float64)
    assert e.shape == g.shape and e.ndim == 3 and e.shape[2] == 17 and c.size == e.shape[0] * e.shape[1] * 225
    n, F = e.shape[:2]
    nees = np.zeros((n, F, 8))
    summ = np.zeros((F, 9))
    rc = lib().orcvio_trajectory_nees(_dp(e), _dp(g), _dp(c), n, F, int(flags), _dp(nees), _dp(summ))
    if rc != 0:
        raise RuntimeError(f"orcvio_trajectory_nees failed: {rc}")
    return nees, summ


def nees_summary(nees):
    """The per-frame summary of trajectory_nees from NEES rows alone (orcvio_nees_summary, the same kernel)."""
    r = np.ascontiguousarray(nees, dtype=np.float64)
    assert r.ndim == 3 and r.shape[2] == 8
    summ = np.zeros((r.shape[1], 9))
    rc = lib().orcvio_nees_summary(_dp(r), r.shape[0], r.shape[1], _dp(summ))
    if rc != 0:
        raise RuntimeError(f"orcvio_nees_summary failed: {rc}")
    return summ


def anees_bounds(n, dof, p=0.95):
    """Two-sided `p` bounds of the ANEES of a dof-dimensional block averaged over n runs:
    chi2_quantile((1 -+ p) / 2, n dof) / n."""
    a = (1.0 - p) / 2.0
    return chi2_quantile(a, n * dof) / n, chi2_quantile(1.0 - a, n * dof) / n


def trajectory_align_ate(est_pose7, gt_pose7, method="sim3"):
    """Umeyama alignment + absolute translation error (orcvio_trajectory_align_ate): (n, F, 7) -> dict(s (n), R (n, 3, 3),
    t (n, 3), mean (n), rmse (n))."""
    e = np.ascontiguousarray(est_pose7, dtype=np.float64)
    g = np.ascontiguousarray(gt_pose7, dtype=np.float64)
    assert e.shape == g.shape and e.ndim == 3 and e.shape[2] == 7
    out = np.zeros((e.shape[0], 15))
    f = lib().orcvio_trajectory_align_ate
    f.argtypes = [C.POINTER(C.c_double)] * 2 + [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    rc = f(_dp(e), _dp(g), e.shape[0], e.shape[1], {"sim3": 0, "se3": 1}[method], _dp(out))
    if rc != 0:
        raise RuntimeError(f"orcvio_trajectory_align_ate failed: {rc}")
    return dict(s=out[:, 0], R=out[:, 1:10].reshape(-1, 3, 3), t=out[:, 10:13], mean=out[:, 13], rmse=out[:, 14])


def kitti_relative_error(est_pose7, gt_pose7, lengths, scale=None):
    """The reference's KITTI-style relative error on the device (orcvio_kitti_relative_error): (n, F, 7) poses ->
    ((n, n_len, 4): samples, mean translation %, mean rotation deg / m, mean translation m;  (n,): TransError(%))."""
    e = np.ascontiguousarray(est_pose7, dtype=np.float64)
    g = np.ascontiguousarray(gt_pose7, dtype=np.float64)
    L = np.ascontiguousarray(lengths, dtype=np.float64)
    assert e.shape == g.shape and e.ndim == 3 and e.shape[2] == 7
    out = np.zeros((e.shape[0], len(L), 4))
    summ = np.zeros(e.shape[0])
    f = lib().orcvio_kitti_relative_error
    f.argtypes = [C.POINTER(C.c_double)] * 2 + [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int] + [C.POINTER(C.c_double)] * 3
    sc = None if scale is None else np.ascontiguousarray(scale, dtype=np.float64)
    rc = f(_dp(e), _dp(g), e.shape[0], e.shape[1], _dp(L), len(L), None if sc is None else _dp(sc), _dp(out), _dp(summ))
    if rc != 0:
        raise RuntimeError(f"orcvio_kitti_relative_error failed: {rc}")
    return out, summ


def object_residuals(frames_wTc, wTo, shape, kps, zs, zb, left=True, new_residual=False):
    """Stage 3 functor evaluation (O1-O4): returns dict(fvec, fjac_cam, fjac_obj, zs_num, cam_pose_se3)."""
    L = lib()
    frames = _f64(frames_wTc).reshape(-1, 16)
    T = frames.shape[0]
    kps = _f64(kps).reshape(-1, 3)
    K = kps.shape[0]
    zs = _f64(zs).reshape(T, K, 2)
    zb = _f64(zb).reshape(T, 4)
    wTo, shape = _f64(wTo).reshape(16), _f64(shape).reshape(3)
    cap = 2 * K * T + 4 * T
    odim = 9 + 3 * K
    fvec = np.zeros(cap)
    jc = np.zeros(cap * 6)
    jo = np.zeros(cap * odim)
    zn = np.zeros(T, dtype=np.int32)
    xi = np.zeros((6, T), order="F")
    rows = C.c_int(0)
    rc = L.orcvio_object_residuals(_dp(frames), T, _dp(wTo), _dp(shape), _dp(kps), K, _dp(zs), _dp(zb),
                                   (1 if left else 0) | (2 if new_residual else 0), _dp(fvec), _dp(jc), _dp(jo),
                                   _ip(zn), _dp(xi), C.byref(rows))
    if rc != 0:
        raise RuntimeError(f"orcvio_object_residuals failed: {rc}")
    r = rows.value
    return dict(fvec=fvec[:r].copy(), fjac_cam=jc[:r * 6].reshape(6, r).T.copy(),
                fjac_obj=jo[:r * odim].reshape(odim, r).T.copy(), zs_num=zn, cam_pose_se3=np.array(xi))


def propagate(R, v, p, t, bg, ba, gyro_old, acc_old, imu, P, flags, noise4):
    """Stage 6 stand-alone: (R, v, p, t, P) after the IMU samples `imu` ((n,7) rows [t, w, a])."""
    L = lib()
    st = np.zeros(16)
    st[:9] = _f64(R).reshape(9)
    st[9:12] = v
    st[12:15] = p
    st[15] = t
    Pm = np.ascontiguousarray(P, dtype=np.float64).copy()
    arr = imu_array(imu)
    rc = L.orcvio_propagate(_dp(st), _dp(_f64(bg)), _dp(_f64(ba)), _dp(_f64(gyro_old)), _dp(_f64(acc_old)),
                            arr.ctypes.data, len(arr), _dp(Pm), Pm.shape[0], flags, _dp(_f64(noise4)))
    if rc != 0:
        raise RuntimeError(f"orcvio_propagate failed: {rc}")
    return st[:9].reshape(3, 3).copy(), st[9:12].copy(), st[12:15].copy(), float(st[15]), Pm


def triangulate(cam_R, cam_t, feat_off, obs_clone, obs_z, translation_threshold=-1.0,
                cost_threshold=4.7673e-4, init_final_dist_threshold=5.0):
    L = lib()
    cam_R, cam_t, obs_z = _f64(cam_R).reshape(-1, 9), _f64(cam_t).reshape(-1, 3), _f64(obs_z).reshape(-1, 2)
    feat_off, obs_clone = _i32(feat_off), _i32(obs_clone)
    nf = len(feat_off) - 1
    pos = np.zeros((nf, 3))
    st = np.zeros(nf, dtype=np.int32)
    it = np.zeros((nf, 2), dtype=np.int32)
    cost = np.zeros(nf)
    rc = L.orcvio_triangulate(_dp(cam_R), _dp(cam_t), cam_R.shape[0], _ip(feat_off), _ip(obs_clone), _dp(obs_z),
                              nf, translation_threshold, cost_threshold, init_final_dist_threshold, _dp(pos),
                              _ip(st), _ip(it), _dp(cost))
    if rc != 0:
        raise RuntimeError(f"orcvio_triangulate failed: {rc}")
    return pos, st, it, cost


def snapshot_update(snap, flags=0, noise_var=None, chi2_p=0.95, translation_threshold=-1.0,
                    cost_threshold=4.7673e-4, init_final_dist_threshold=5.0, repeat=1):
    """snap: dict from synth.stress_snapshot (clone_R, clone_p, P, R_b2c, t_c_b, feat_off, ...)."""
    L = lib()
    N = int(snap["n_clones"])
    D = 22 + 6 * N
    clone_R, clone_p = _f64(snap["clone_R"]).reshape(N, 9), _f64(snap["clone_p"]).reshape(N, 3)
    Rbc, tcb = _f64(snap["R_b2c"]).reshape(9), _f64(snap["t_c_b"]).reshape(3)
    P = np.asfortranarray(snap["P"], dtype=np.float64)
    feat_off, obs_clone = _i32(snap["feat_off"]), _i32(snap["obs_clone"])
    obs_z = _f64(snap["obs_z"]).reshape(-1, 2)
    nf = len(feat_off) - 1
    out = dict(P=np.zeros((D, D), order="F"), delta_x=np.zeros(D), status=np.zeros(nf, dtype=np.int32),
               gamma=np.zeros(nf), positions=np.zeros((nf, 3)), clones=np.zeros((N, 12)),
               timings_us=np.zeros(8, dtype=np.float32))
    if noise_var is None:
        noise_var = float(snap["cfg"]["noise_feature"]) ** 2
    rc = L.orcvio_snapshot_update(
        _dp(clone_R), _dp(clone_p), N, _dp(Rbc), _dp(tcb), _dp(P), _ip(feat_off), _ip(obs_clone), _dp(obs_z),
        nf, flags, noise_var, chi2_p, translation_threshold, cost_threshold, init_final_dist_threshold,
        _dp(out["P"]), _dp(out["delta_x"]), _ip(out["status"]), _dp(out["gamma"]), _dp(out["positions"]),
        _dp(out["clones"]), out["timings_us"].ctypes.data_as(C.POINTER(C.c_float)), repeat)
    if rc != 0:
        raise RuntimeError(f"orcvio_snapshot_update failed: {rc}")
    return out


def measurement_jacobians(clone_R, clone_p, R_b2c, t_c_b, positions, feat_off, obs_clone, obs_z, flags=0):
    L = lib()
    clone_R, clone_p = _f64(clone_R).reshape(-1, 9), _f64(clone_p).reshape(-1, 3)
    positions, obs_z = _f64(positions).reshape(-1, 3), _f64(obs_z).reshape(-1, 2)
    feat_off, obs_clone = _i32(feat_off), _i32(obs_clone)
    Rbc, tcb = _f64(R_b2c).reshape(9), _f64(t_c_b).reshape(3)
    no = len(obs_clone)
    Hx, He, Hf, r = np.zeros((no, 2, 6)), np.zeros((no, 2, 6)), np.zeros((no, 2, 3)), np.zeros((no, 2))
    rc = L.orcvio_measurement_jacobians(_dp(clone_R), _dp(clone_p), clone_R.shape[0], _dp(Rbc), _dp(tcb),
                                        _dp(positions), _ip(feat_off), _ip(obs_clone), _dp(obs_z),
                                        len(feat_off) - 1, flags, _dp(Hx), _dp(He), _dp(Hf), _dp(r))
    if rc != 0:
        raise RuntimeError(f"orcvio_measurement_jacobians failed: {rc}")
    return Hx, He, Hf, r


def fp64_peak():
    """(DFMA TFLOP/s, DMMA TFLOP/s) measured on the current device."""
    a, b = C.c_double(0), C.c_double(0)
    rc = lib().orcvio_fp64_peak(C.byref(a), C.byref(b))
    if rc != 0:
        raise RuntimeError(f"orcvio_fp64_peak failed: {rc}")
    return a.value, b.value


def latency_probe():
    """Dependent-chain latencies (cycles): dict(dfma, sqrt, div, rsqrt, lds, syncthreads512, shfl64)."""
    out = np.zeros(7)
    rc = lib().orcvio_latency_probe(_dp(out))
    if rc != 0:
        raise RuntimeError(f"orcvio_latency_probe failed: {rc}")
    return dict(zip(["dfma", "sqrt", "div", "rsqrt", "lds", "syncthreads512", "shfl64"], out.tolist()))


def latency_probe1():
    """Single-warp dependent latencies (cycles)."""
    out = np.zeros(10)
    L = lib()
    L.orcvio_latency_probe1.argtypes = [C.POINTER(C.c_double)]
    L.orcvio_latency_probe1.restype = C.c_int
    rc = L.orcvio_latency_probe1(_dp(out))
    if rc != 0:
        raise RuntimeError(f"orcvio_latency_probe1 failed: {rc}")
    return dict(zip(["dfma", "dmma_dep", "dmma_x2", "dmma_x4", "dmma_x8", "shfl64", "lds128", "fence_cta", "rcp_approx"],
                    out.tolist()))


def chol_probe(A, X=None, reps=10):
    """Runs csrc/chol.cuh on one SPD matrix: returns (L, X C^-T, per-panel clock stamps, mean us)."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    m = A.shape[0]
    nx = 0 if X is None else X.shape[0]
    Xc = np.ascontiguousarray(X if X is not None else np.zeros((1, m)), dtype=np.float64)
    L = np.zeros((m, m))
    Xs = np.zeros_like(Xc)
    prof = np.zeros((64, 8), dtype=np.int64)
    us = C.c_float(0)
    rc = lib().orcvio_chol_probe(m, nx, _dp(A), _dp(Xc), _dp(L), _dp(Xs),
                                 prof.ctypes.data_as(C.POINTER(C.c_longlong)), int(reps), C.byref(us))
    if rc != 0:
        raise RuntimeError(f"orcvio_chol_probe failed: {rc}")
    return L, (Xs if X is not None else None), prof, us.value


def chi2_quantile(p, dof):
    return float(lib().orcvio_chi2_quantile(float(p), int(dof)))


def ekf_measurement_jacobians(clone_R, clone_p, R_b2c, t_c_b, anchor, inv_depth, f_an, positions, feat_off,
                              obs_clone, obs_z):
    """H1 (measurementJacobian_ekf_1didp, orcvio.cpp:1356-1478) per observation: H_f (n,2), H_a, H_x, H_e (n,2,6), r (n,2)."""
    L = lib()
    clone_R, clone_p = _f64(clone_R).reshape(-1, 9), _f64(clone_p).reshape(-1, 3)
    Rbc, tcb = _f64(R_b2c).reshape(9), _f64(t_c_b).reshape(3)
    anchor, feat_off, obs_clone = _i32(anchor), _i32(feat_off), _i32(obs_clone)
    rho, fan, pos, oz = _f64(inv_depth), _f64(f_an).reshape(-1, 2), _f64(positions).reshape(-1, 3), _f64(obs_z).reshape(-1, 2)
    no = len(obs_clone)
    out = dict(H_f=np.zeros((no, 2)), H_a=np.zeros((no, 2, 6)), H_x=np.zeros((no, 2, 6)), H_e=np.zeros((no, 2, 6)),
               r=np.zeros((no, 2)))
    L.orcvio_ekf_measurement_jacobians.restype = C.c_int
    L.orcvio_ekf_measurement_jacobians.argtypes = [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 9 + [C.c_int] + [C.c_void_p] * 5
    rc = L.orcvio_ekf_measurement_jacobians(
        clone_R.ctypes.data, clone_p.ctypes.data, clone_R.shape[0], Rbc.ctypes.data, tcb.ctypes.data, anchor.ctypes.data,
        rho.ctypes.data, fan.ctypes.data, pos.ctypes.data, feat_off.ctypes.data, obs_clone.ctypes.data, oz.ctypes.data,
        len(feat_off) - 1, out["H_f"].ctypes.data, out["H_a"].ctypes.data, out["H_x"].ctypes.data, out["H_e"].ctypes.data,
        out["r"].ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_measurement_jacobians failed: {rc}")
    return out


def ekf_feature_rows(clone_R, clone_p, R_b2c, t_c_b, anchor, inv_depth, f_an, positions, z_cur, P, noise_var, chi2_p=0.95):
    """H2 (featureJacobian_ekf, orcvio.cpp:1575-1651) + the dof-2 gate for the features of the state observed by the
    newest clone: H (2F, D), r (2F), gamma (F), pass (F)."""
    L = lib()
    clone_R, clone_p = _f64(clone_R).reshape(-1, 9), _f64(clone_p).reshape(-1, 3)
    Rbc, tcb = _f64(R_b2c).reshape(9), _f64(t_c_b).reshape(3)
    anchor = _i32(anchor)
    rho, fan, pos, z = _f64(inv_depth), _f64(f_an).reshape(-1, 2), _f64(positions).reshape(-1, 3), _f64(z_cur).reshape(-1, 2)
    F = len(anchor)
    Pm = np.ascontiguousarray(P, dtype=np.float64)
    D = Pm.shape[0]
    out = dict(H=np.zeros((2 * F, D)), r=np.zeros(2 * F), gamma=np.zeros(F), **{"pass": np.zeros(F, dtype=np.int32)})
    L.orcvio_ekf_feature_rows.restype = C.c_int
    L.orcvio_ekf_feature_rows.argtypes = ([C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 7 + [C.c_int, C.c_void_p, C.c_int,
                                          C.c_double, C.c_double] + [C.c_void_p] * 4)
    rc = L.orcvio_ekf_feature_rows(
        clone_R.ctypes.data, clone_p.ctypes.data, clone_R.shape[0], Rbc.ctypes.data, tcb.ctypes.data, anchor.ctypes.data,
        rho.ctypes.data, fan.ctypes.data, pos.ctypes.data, z.ctypes.data, F, Pm.ctypes.data, D, float(noise_var),
        float(chi2_p), out["H"].ctypes.data, out["r"].ctypes.data, out["gamma"].ctypes.data, out["pass"].ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_feature_rows failed: {rc}")
    return out


def ekf_update_feature_cov(P, clone_R, clone_p, R_b2c, t_c_b, feat_idx, old_idx, new_idx, p_w, inv_depth_new):
    """H4 (updateFeatureCov_1didp, orcvio.cpp:3611-3773): returns (P after the anchor change, Jacobian row)."""
    L = lib()
    clone_R, clone_p = _f64(clone_R).reshape(-1, 9), _f64(clone_p).reshape(-1, 3)
    Rbc, tcb, pw = _f64(R_b2c).reshape(9), _f64(t_c_b).reshape(3), _f64(p_w).reshape(3)
    Pm = np.array(P, dtype=np.float64, order="C")
    D = Pm.shape[0]
    J = np.zeros(D)
    L.orcvio_ekf_update_feature_cov.restype = C.c_int
    L.orcvio_ekf_update_feature_cov.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p]
    rc = L.orcvio_ekf_update_feature_cov(Pm.ctypes.data, D, clone_R.ctypes.data, clone_p.ctypes.data, clone_R.shape[0],
                                         Rbc.ctypes.data, tcb.ctypes.data, int(feat_idx), int(old_idx), int(new_idx),
                                         pw.ctypes.data, float(inv_depth_new), J.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_update_feature_cov failed: {rc}")
    return Pm, J


def ekf_remove_feature_cov(P, n_clones, feat_idx):
    """H4 (rmLostFeaturesCov, orcvio.cpp:3776-3828): P without the feature's row / column."""
    L = lib()
    Pm = np.ascontiguousarray(P, dtype=np.float64)
    D = Pm.shape[0]
    out = np.zeros((D - 1, D - 1))
    L.orcvio_ekf_remove_feature_cov.restype = C.c_int
    L.orcvio_ekf_remove_feature_cov.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
    rc = L.orcvio_ekf_remove_feature_cov(Pm.ctypes.data, D, int(n_clones), int(feat_idx), out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_remove_feature_cov failed: {rc}")
    return out


def ekf_new_feature_rows(clone_R, clone_p, R_b2c, t_c_b, anchor, inv_depth, f_an, positions, feat_off, obs_clone, obs_z, D):
    """H2 + H3 (featureJacobian_ekf_new + new-feature sparsification): H_1 (F, D), h_2 (F), r_1 (F), H_o (rows, D), r_o."""
    L = lib()
    clone_R, clone_p = _f64(clone_R).reshape(-1, 9), _f64(clone_p).reshape(-1, 3)
    Rbc, tcb = _f64(R_b2c).reshape(9), _f64(t_c_b).reshape(3)
    anchor, feat_off, obs_clone = _i32(anchor), _i32(feat_off), _i32(obs_clone)
    rho, fan, pos, oz = _f64(inv_depth), _f64(f_an).reshape(-1, 2), _f64(positions).reshape(-1, 3), _f64(obs_z).reshape(-1, 2)
    F = len(anchor)
    cap = 2 * len(obs_clone)
    out = dict(H_1=np.zeros((F, D)), h_2=np.zeros(F), r_1=np.zeros(F), H_o=np.zeros((cap, D)), r_o=np.zeros(cap))
    rows = C.c_int(0)
    L.orcvio_ekf_new_feature_rows.restype = C.c_int
    L.orcvio_ekf_new_feature_rows.argtypes = ([C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 9 + [C.c_int, C.c_int] +
                                              [C.c_void_p] * 5 + [C.POINTER(C.c_int)])
    rc = L.orcvio_ekf_new_feature_rows(
        clone_R.ctypes.data, clone_p.ctypes.data, clone_R.shape[0], Rbc.ctypes.data, tcb.ctypes.data, anchor.ctypes.data,
        rho.ctypes.data, fan.ctypes.data, pos.ctypes.data, feat_off.ctypes.data, obs_clone.ctypes.data, oz.ctypes.data,
        F, int(D), out["H_1"].ctypes.data, out["h_2"].ctypes.data, out["r_1"].ctypes.data, out["H_o"].ctypes.data,
        out["r_o"].ctypes.data, C.byref(rows))
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_new_feature_rows failed: {rc}")
    out["H_o"], out["r_o"] = out["H_o"][:rows.value], out["r_o"][:rows.value]
    return out


def ekf_delayed_init(P, dx_leg, H_1, h_2, r_1, noise_var):
    """The new-state part of measurementUpdate_hybrid: returns (dx_new, P_aug)."""
    L = lib()
    Pm = np.ascontiguousarray(P, dtype=np.float64)
    D = Pm.shape[0]
    dx, H1, h2, r1 = _f64(dx_leg), _f64(H_1).reshape(-1, D), _f64(h_2), _f64(r_1)
    F = len(h2)
    dx_new, P_aug = np.zeros(F), np.zeros((D + F, D + F))
    L.orcvio_ekf_delayed_init.restype = C.c_int
    L.orcvio_ekf_delayed_init.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_double, C.c_void_p, C.c_void_p]
    rc = L.orcvio_ekf_delayed_init(Pm.ctypes.data, D, dx.ctypes.data, H1.ctypes.data, h2.ctypes.data, r1.ctypes.data, F,
                                   float(noise_var), dx_new.ctypes.data, P_aug.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_delayed_init failed: {rc}")
    return dx_new, P_aug


def hybrid_update_dense(P, H, r, noise_var):
    """Legacy-state part of measurementUpdate_hybrid on a state with feature columns: returns (dx, P_posterior)."""
    L = lib()
    Pm = np.ascontiguousarray(P, dtype=np.float64)
    D = Pm.shape[0]
    Hm = np.ascontiguousarray(H, dtype=np.float64).reshape(-1, D)
    rv = _f64(r)
    dx, Po = np.zeros(D), np.zeros((D, D))
    L.orcvio_hybrid_update_dense.restype = C.c_int
    L.orcvio_hybrid_update_dense.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p,
                                             C.c_void_p]
    rc = L.orcvio_hybrid_update_dense(Pm.ctypes.data, D, Hm.ctypes.data, rv.ctypes.data, Hm.shape[0], float(noise_var),
                                      dx.ctypes.data, Po.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_hybrid_update_dense failed: {rc}")
    return dx, Po


def ekf_augment_cov(P, n_clones):
    """stateAugmentation's covariance step with a feature block behind the clones: (D+6) x (D+6)."""
    L = lib()
    Pm = np.ascontiguousarray(P, dtype=np.float64)
    D = Pm.shape[0]
    out = np.zeros((D + 6, D + 6))
    L.orcvio_ekf_augment_cov.restype = C.c_int
    L.orcvio_ekf_augment_cov.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    rc = L.orcvio_ekf_augment_cov(Pm.ctypes.data, D, int(n_clones), out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_augment_cov failed: {rc}")
    return out


def ekf_remove_clone_cov(P, n_clones, clone_idx):
    """Drop one clone's 6 rows / columns of P (pruneImuStateBuffer)."""
    L = lib()
    Pm = np.ascontiguousarray(P, dtype=np.float64)
    D = Pm.shape[0]
    out = np.zeros((D - 6, D - 6))
    L.orcvio_ekf_remove_clone_cov.restype = C.c_int
    L.orcvio_ekf_remove_clone_cov.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
    rc = L.orcvio_ekf_remove_clone_cov(Pm.ctypes.data, D, int(n_clones), int(clone_idx), out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orcvio_ekf_remove_clone_cov failed: {rc}")
    return out
