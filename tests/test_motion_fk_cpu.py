"""CPU: the expert-table math of uhc_load_clips_smpl (uhc_b200/csrc/motion_fk.h, compiled for the host with g++) against the host motion
library it restates, pack_expert(make_expert(...)) of uhc_b200/motion_lib.py, on inputs that reach every branch (tests/motion_cases.py)."""
import ctypes as C
import os
import subprocess
import warnings

import numpy as np
import pytest

from tests.motion_cases import edge_clips, scaled_model
from uhc_b200 import motion_lib as ML
from uhc_b200.engine import pack_expert
from uhc_b200.model import HumanoidModel

HERE = os.path.dirname(os.path.abspath(__file__))
# record columns held to 1e-12 (qpos, positions, quaternions) and to 1e-10 (finite differences: qvel, bangvel)
TIGHT = np.r_[0:76, 151:415, 487:576]
FD = np.r_[76:151, 415:487]


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("motion_fk") / "libmotion_fk_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so, os.path.join(HERE, "emu", "motion_fk_host.cpp")])
    return C.CDLL(so)


def header_table(lib, pose, trans, model):
    pose = np.ascontiguousarray(pose, dtype=np.float64)
    T, pd = pose.shape
    tr = None if trans is None else np.ascontiguousarray(np.asarray(trans, dtype=np.float64).reshape(T, 3))
    kin = np.ascontiguousarray(np.concatenate([model.offset, model.ipos], 1))
    par, ee = np.ascontiguousarray(model.parent, np.int32), np.ascontiguousarray(model.ee, np.int32)
    out = np.full((T, 576), np.nan)
    d = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    i = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
    lib.motion_fk_host(d(pose), C.c_int(T), C.c_int(pd), d(tr) if tr is not None else None, d(kin), i(par), i(ee), d(out))
    return out


def host_table(pose, trans, model):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # scipy's gimbal-lock warning
        return pack_expert(ML.make_expert(pose, trans, model))


def check(lib, pose, trans, model, name):
    got, ref = header_table(lib, pose, trans, model), host_table(pose, trans, model)
    assert np.isfinite(got).all(), name
    assert np.abs(got[:, TIGHT] - ref[:, TIGHT]).max() <= 1e-12, (name, np.unravel_index(np.abs(got[:, TIGHT] - ref[:, TIGHT]).argmax(), got[:, TIGHT].shape))
    assert np.abs(got[:, FD] - ref[:, FD]).max() <= 1e-10, (name, np.abs(got[:, FD] - ref[:, FD]).max())
    return got, ref


def test_body_permutation_and_root_offset(lib):
    m = HumanoidModel()
    out = np.zeros(24, np.int32)
    lib.motion_smpl_joint(out.ctypes.data_as(C.POINTER(C.c_int)))
    assert list(out) == [ML.SMPL_BONE_ORDER_NAMES.index(n) for n in m.body_names]
    # the kernel takes the root offset from body 0's offset of each variant
    for v in (m, scaled_model()):
        assert np.array_equal(v.offset[0], v.root_offset)


@pytest.mark.parametrize("variant", ["default", "scaled"])
def test_header_matches_host_motion_lib(lib, golden_dir, variant):
    model = HumanoidModel() if variant == "default" else scaled_model()
    seen = set()
    for name, pose, trans in edge_clips(np.random.default_rng(11), golden_dir):
        got, ref = check(lib, pose, trans, model, name)
        seen.add(name)
        if name == "fast_root":
            assert (np.abs(ref[:, 76:82]) == 10.0).any(axis=0)[[0, 5]].all(), "the root must hit the +-10 qvel clip linearly and angularly"
        if name == "two_frames":
            assert np.array_equal(got[0, 76:151], got[1, 76:151])
        assert (got[:, 574:] == 0).all()
    assert len(seen) == 10


def test_branches_are_reached():
    """the edge cases really take the branches they are named after"""
    from scipy.spatial.transform import Rotation as sRot
    cases = {n: (p, t) for n, p, t in edge_clips(np.random.default_rng(11))}
    p = cases["random_rotvec"][0].reshape(-1, 24, 3)
    ang = np.linalg.norm(p, axis=-1)
    assert (ang == 0).any() and ((ang > 0) & (ang < 1e-3)).any() and (ang > np.pi - 1e-3).any()
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        sRot.from_rotvec(cases["gimbal_lock"][0][:, 3:].reshape(-1, 3)).as_euler("ZYX")
    assert any("Gimbal lock" in str(x.message) for x in w)
    rq = sRot.from_rotvec(cases["root_w_negative"][0][:, :3]).as_quat()
    assert (rq[:, 3] < 0).all()
    q = ML.smpl_to_qpos(*cases["root_flip"])[:, 3:7]
    d = ML.qmul(q[1:], ML.qinv(q[:-1]))
    assert (d[:, 0] < 0).any(), "consecutive root quaternions on opposite hemispheres: the finite difference wraps past pi"
