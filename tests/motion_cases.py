"""SMPL pose sequences that exercise every branch of the expert-table math (uhc_b200/csrc/motion_fk.h, uhc_b200/motion_lib.py): used by the CPU
test of the header and the GPU test of uhc_load_clips_smpl."""
import os

import numpy as np
from scipy.spatial.transform import Rotation as sRot


def smooth_pose(T, rng, amp=0.4, width=72):
    """smooth random axis-angle rows: a few low-frequency sinusoids per column"""
    t = np.arange(T)[:, None] / 30.0
    pose = np.zeros((T, width))
    for _ in range(3):
        pose += rng.uniform(0, amp / 3, width) * np.sin(2 * np.pi * rng.uniform(0.1, 1.5, width) * t + rng.uniform(0, 2 * np.pi, width))
    pose[:, :3] += np.array([1.2092, 1.2092, 1.2092])        # upright in the Z-up world (tests/helpers.py)
    return pose


def smooth_trans(T, rng):
    t = np.arange(T)[:, None] / 30.0
    return np.array([0.3, -0.2, 0.0]) * t * rng.uniform(0.5, 1.5) + np.array([0.0, 0.0, 0.9]) + 0.02 * np.sin(2 * np.pi * t * rng.uniform(0.2, 1.0))


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def edge_clips(rng, golden_dir=None):
    """[(name, pose_aa, trans or None)]: golden inputs, random rotvecs (zero, below 1e-3, near pi), exact gimbal lock, root quaternions with
    w < 0 and root rotations crossing pi between frames, a root fast enough to hit the +-10 qvel clip, SMPL-H rows, no trans, 2 frames"""
    out = []
    if golden_dir is not None:
        for tag in ("sway", "kick"):
            z = np.load(os.path.join(golden_dir, f"expert_{tag}.npz"))
            out.append((f"golden_{tag}", z["pose_aa"].copy(), z["trans"].copy()))
    T = 40
    # random rotvecs of every size, including the zero rotvec, the small-angle series (< 1e-3) and angles just below pi
    p = rng.normal(0, 1.2, (T, 72))
    p[0] = 0.0
    p[1:6] = (_unit(rng, 5 * 24) * rng.uniform(0, 1e-3, (5 * 24, 1))).reshape(5, 72)
    p[6:10] = (_unit(rng, 4 * 24) * (np.pi - rng.uniform(1e-9, 1e-3, (4 * 24, 1)))).reshape(4, 72)
    p[10:12, 3:] = 1e-3 * _unit(rng, 2 * 23).reshape(2, 69)            # exactly at the series threshold
    out.append(("random_rotvec", p, smooth_trans(T, rng)))
    # gimbal lock: every joint at pitch +-pi/2 of its ZYX angles
    p = smooth_pose(T, rng)
    for t in range(T):
        e = np.stack([rng.uniform(-3, 3, 24), np.where(rng.uniform(size=24) < 0.5, np.pi / 2, -np.pi / 2), rng.uniform(-3, 3, 24)], 1)
        p[t, 3:] = sRot.from_euler("ZYX", e[1:]).as_rotvec().reshape(69)
    out.append(("gimbal_lock", p, smooth_trans(T, rng)))
    # root quaternion with w < 0 (rotation angle above pi), and a root angle sweeping through pi so consecutive stored quaternions flip sign
    p = smooth_pose(T, rng)
    ax = _unit(rng, 1)[0]
    p[:, :3] = ax * np.linspace(np.pi - 0.6, np.pi + 0.6, T)[:, None]
    out.append(("root_flip", p, smooth_trans(T, rng)))
    p = smooth_pose(T, rng)
    p[:, :3] = _unit(rng, T) * rng.uniform(np.pi + 0.1, 2 * np.pi - 0.1, (T, 1))
    out.append(("root_w_negative", p, smooth_trans(T, rng)))
    # a root moving 0.5 m and turning 0.6 rad per frame: linear and angular qvel beyond +-10
    p = smooth_pose(T, rng)
    p[:, :3] = np.array([0.0, 0.0, 1.0]) * (0.6 * np.arange(T))[:, None] % (2 * np.pi)
    tr = smooth_trans(T, rng)
    tr[:, 0] += 0.5 * np.arange(T)
    out.append(("fast_root", p, tr))
    out.append(("smplh_156", smooth_pose(T, rng, width=156), smooth_trans(T, rng)))
    out.append(("no_trans", smooth_pose(T, rng), None))
    out.append(("two_frames", smooth_pose(2, rng), smooth_trans(2, rng)))
    return out


def scaled_model(seed=5):
    from uhc_b200.model import HumanoidModel
    return HumanoidModel(scale=np.random.default_rng(seed).uniform(0.85, 1.15, 24))
