"""Filter configurations with the reference's `config/*.yaml` semantics.

The key set and the values are those read by OrcVIO::loadParameters
(reference src/orcvio.cpp:62-329) from config/euroc.yaml, config/unity.yaml and
config/kitti_odom.yaml (the table in SURVEY.md A.2).  They are kept here as Python
dictionaries and written out as OpenCV-YAML (`%YAML:1.0`, `!!opencv-matrix`) so that
both the product's C++ reader and cv2.FileStorage (oracle) parse the same file.
"""
import copy

_COMMON = dict(
    output_dir="/tmp/",
    if_FEJ=0, estimate_extrin=0, estimate_td=0, calib_imu_instrinsic=0,
    td=0.0, pub_frequency=10, sw_size=20, position_std_threshold=8.0,
    rotation_threshold=0.2618, translation_threshold=0.4, tracking_rate_threshold=0.5,
    least_observation_number=3, max_track_len=6, feature_translation_threshold=-1.0,
    initial_covariance_orientation=4e-4, initial_covariance_velocity=0.25,
    initial_covariance_position=1.0, initial_covariance_gyro_bias=4e-4,
    initial_covariance_acc_bias=0.01, initial_covariance_extrin_rot=3.0462e-8,
    initial_covariance_extrin_trans=9e-8, reset_fej_threshold=10.11,
    zupt_max_feature_dis=2e-3, zupt_noise_v=1e-2, zupt_noise_p=1e-2, zupt_noise_q=3.4e-2,
    static_duration=1.0, aug_grid_rows=5, aug_grid_cols=6, feature_idp_dim=1, use_schmidt=0,
    use_left_perturbation_flag=0, use_closed_form_cov_prop_flag=1,
    chi_square_threshold_feat=0.95, prediction_only_flag=0,
)

EUROC = dict(
    _COMMON,
    resolution_width=752, resolution_height=480,
    intrinsics=dict(fx=458.654, fy=457.296, cx=367.215, cy=248.375),
    T_cam_imu=[0.014865542981794, 0.999557249008346, -0.025774436697440, 0.065222909535531,
               -0.999880929698575, 0.014967213324719, 0.003756188357967, -0.020706385492719,
               0.004140296794224, 0.025715529947966, 0.999660727177902, -0.008054602460030,
               0, 0, 0, 1.0],
    noise_gyro=0.004, noise_acc=0.08, noise_gyro_bias=2e-6, noise_acc_bias=4e-5, noise_feature=0.008,
    if_ZUPT_valid=1, if_use_feature_zupt_flag=1, imu_rate=200, img_rate=20,
    max_features_in_one_grid=1, use_larvio_flag=1,
    feature_cost_threshold=4.7673e-04, init_final_dist_threshold=1e2,
    discard_large_update_flag=0, use_object_residual_update_cam_pose_flag=0, initial_use_gt=0,
)

UNITY = dict(
    _COMMON,
    resolution_width=640, resolution_height=480,
    intrinsics=dict(fx=260.99805320956386, fy=260.99805320956386, cx=320, cy=240),
    T_cam_imu=[0.0, -1.0, 0.0, 0.1,
               0.0, 0.0, -1.0, 0,
               1.0, 0.0, 0.0, -0.1,
               0.0, 0.0, 0.0, 1.0],
    noise_gyro=0.004, noise_acc=0.08, noise_gyro_bias=2e-6, noise_acc_bias=4e-5, noise_feature=0.008,
    if_ZUPT_valid=1, if_use_feature_zupt_flag=0, imu_rate=250, img_rate=30,
    max_features_in_one_grid=0, use_larvio_flag=0,
    feature_cost_threshold=4.7673e-04, init_final_dist_threshold=1e1,
    discard_large_update_flag=0, use_object_residual_update_cam_pose_flag=1, initial_use_gt=0,
)

KITTI_ODOM = dict(
    _COMMON,
    resolution_width=1242, resolution_height=375,
    intrinsics=dict(fx=721.5377, fy=721.5377, cx=609.5593, cy=172.8540),
    T_cam_imu=[9.98747206e-04, -9.99990382e-01, 4.25937849e-03, -3.14076870e-01,
               8.41690183e-03, -4.25082114e-03, -9.99955570e-01, 7.19452036e-01,
               9.99964049e-01, 1.03455328e-03, 8.41257521e-03, -1.08908294e+00,
               0, 0, 0, 1.0],
    noise_gyro=2.0e-5, noise_acc=3.0e-3, noise_gyro_bias=2.0e-4, noise_acc_bias=2.0e-3, noise_feature=1,
    if_ZUPT_valid=0, if_use_feature_zupt_flag=0, imu_rate=250, img_rate=10,
    max_features_in_one_grid=1, use_larvio_flag=0,
    feature_cost_threshold=1e3, init_final_dist_threshold=1e3,
    discard_large_update_flag=1, use_object_residual_update_cam_pose_flag=1, initial_use_gt=1,
    initial_state_time=0.91149066666667,
    initial_pos=[0, 0, 0], initial_ba=[0.0, 0.0, 0.0], initial_bg=[0.0, 0.0, 0.0],
    initial_quat=[-0.00047348, 0.00624186, -0.151103, 0.988498],
    initial_vel=[2.38645, -0.666818, 0.0784056],
)

BY_NAME = dict(euroc=EUROC, unity=UNITY, kitti_odom=KITTI_ODOM)

_MATRIX_SHAPES = dict(T_cam_imu=(4, 4), initial_pos=(3, 1), initial_ba=(3, 1), initial_bg=(3, 1),
                      initial_vel=(3, 1), initial_quat=(4, 1))


def make(name, **overrides):
    """Config dictionary `name` ('euroc' | 'unity' | 'kitti_odom') with overrides."""
    cfg = copy.deepcopy(BY_NAME[name])
    cfg.update(overrides)
    return cfg


def with_initial_state(cfg, t, quat_xyzw, pos, vel, bg=(0, 0, 0), ba=(0, 0, 0)):
    """initial_use_gt: 1 semantics (reference src/orcvio.cpp:123-146, 514-544)."""
    cfg = copy.deepcopy(cfg)
    cfg.update(initial_use_gt=1, initial_state_time=float(t),
               initial_quat=[float(x) for x in quat_xyzw], initial_pos=[float(x) for x in pos],
               initial_vel=[float(x) for x in vel], initial_bg=[float(x) for x in bg],
               initial_ba=[float(x) for x in ba])
    return cfg


def to_yaml(cfg):
    out = ["%YAML:1.0"]
    for k, v in cfg.items():
        if k in _MATRIX_SHAPES:
            r, c = _MATRIX_SHAPES[k]
            data = ", ".join(repr(float(x)) for x in v)
            out += [f"{k}: !!opencv-matrix", f"   rows: {r}", f"   cols: {c}", "   dt: d",
                    f"   data: [{data}]"]
        elif isinstance(v, dict):
            out.append(f"{k}:")
            out += [f"   {kk}: {vv!r}" for kk, vv in v.items()]
        elif isinstance(v, str):
            out.append(f'{k}: "{v}"')
        else:
            out.append(f"{k}: {v!r}")
    return "\n".join(out) + "\n"


def write_yaml(path, cfg):
    with open(path, "w") as fh:
        fh.write(to_yaml(cfg))
    return path
