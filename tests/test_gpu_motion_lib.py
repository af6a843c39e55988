"""GPU: expert tables built on the device from raw SMPL sequences (uhc_load_clips_smpl / uhc_get_clip_frames, include/uhc_motion.h;
Engine.load_smpl_clips; the drop-in's motion_lib: device) against the host motion library, pack_expert(make_expert(...))."""
import ctypes as C
import os
import warnings

import joblib
import numpy as np
import pytest

from tests.motion_cases import edge_clips, scaled_model, smooth_pose, smooth_trans

pytestmark = pytest.mark.gpu


def _clip_set(golden_dir, n=300, seed=3):
    """n clips of mixed length (2 .. 300 frames) with the edge cases of tests/motion_cases.py in front; per-clip body-shape variant 0 / 1"""
    rng = np.random.default_rng(seed)
    edge = [(p, t) for name, p, t in edge_clips(rng, golden_dir) if p.shape[1] == 72]
    lens = np.clip(np.round(np.exp(rng.normal(np.log(45.0), 0.9, n - len(edge)))), 2, 300).astype(int)
    clips = edge + [(smooth_pose(int(T), rng), smooth_trans(int(T), rng) if i % 7 else None) for i, T in enumerate(lens)]
    return [p for p, _ in clips], [t for _, t in clips], rng.integers(0, 2, n).astype(np.int32)


def _host_table(pose, trans, models, clip_models):
    from uhc_b200 import motion_lib as ML
    from uhc_b200.engine import pack_expert
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")          # scipy's gimbal-lock warning
        return np.concatenate([pack_expert(ML.make_expert(p, t, models[c])) for p, t, c in zip(pose, trans, clip_models)])


def _engine(precision, models, E=16, **cfg):
    from uhc_b200.engine import Engine
    return Engine(E, model=models[0], precision=precision, variants=models, **cfg)


@pytest.fixture(scope="module")
def table(golden_dir):
    from uhc_b200.model import HumanoidModel
    models = [HumanoidModel(), scaled_model()]
    pose, trans, cm = _clip_set(golden_dir)
    return models, pose, trans, cm, _host_table(pose, trans, models, cm)


def test_fp64_engine_matches_host_records(table):
    models, pose, trans, cm, ref = table
    eng = _engine(64, models)
    eng.load_smpl_clips(pose, trans, clip_models=cm)
    assert list(eng.clip_len) == [len(p) for p in pose]
    got = eng.get_clip_frames()
    assert got.shape == ref.shape
    err = np.abs(got - ref).max(0)
    assert err.max() <= 1e-10, (int(err.argmax()), float(err.max()))
    print(f"fp64: max |diff| {err.max():.3g}, bit-equal {np.mean(got == ref):.6f}")
    # SMPL-H rows (156 wide) and no trans at all
    rng = np.random.default_rng(8)
    ph = [smooth_pose(T, rng, width=156) for T in (2, 30, 77)]
    eng.load_smpl_clips(ph, None)
    ref_h = _host_table(ph, [None] * 3, models, [0, 0, 0])
    assert np.abs(eng.get_clip_frames() - ref_h).max() <= 1e-10
    eng.close()


def test_fp32_engine_within_one_ulp(table):
    models, pose, trans, cm, ref = table
    eng = _engine(32, models)
    eng.load_smpl_clips(pose, trans, clip_models=cm)
    got = eng.get_clip_frames().astype(np.float32)
    ref32 = ref.astype(np.float32)
    # within 1 fp32 ulp of float32(host).  Elements whose exact value is zero (e.g. the angular velocity of a joint that does not move)
    # come out of both fp64 paths as rounding residue of order 1e-16, different on each side because libm and CUDA round sin / cos / acos
    # differently; an fp32 ulp at that size is ~1e-23, so those elements are held to 1e-12 absolute, the agreement of the fp64 tables
    diff = np.abs(got.astype(np.float64) - ref32.astype(np.float64))
    ulp = np.spacing(np.abs(ref32)).astype(np.float64)
    bad = diff > np.maximum(ulp, 1e-12)
    assert not bad.any(), [(int(i) // 576, int(i) % 576, float(got.flat[i]), float(ref32.flat[i])) for i in np.flatnonzero(bad)[:10]]
    residue = (diff > ulp) & (np.abs(ref) < 1e-12)
    assert residue.sum() == (diff > ulp).sum(), "every element beyond 1 ulp is a rounding residue of zero"
    print(f"fp32: bit-equal fraction {np.mean(got == ref32):.8f} of {got.size} elements; {int(residue.sum())} residues of zero (|host| < 1e-12) "
          f"differ by more than 1 ulp, by at most {diff[residue].max() if residue.any() else 0.0:.3g}")
    eng.close()


def test_side_effects_match_load_clips(table):
    """every env record invalidated (a step without reset is counted as invalid), clip weights back to the default sampling rule"""
    import torch
    models, pose, trans, cm, ref = table
    n = 40
    E = 64
    eng = _engine(32, models, E=E, auto_reset=1, t_min=5, t_max=60)
    from uhc_b200 import motion_lib as ML
    eng.load_clips([ML.make_expert(p, t) for p, t in zip(pose[:n], trans[:n])])
    eng.reset(np.arange(E), clip=np.zeros(E, np.int32), start=0, length=2)
    act = torch.zeros(E, eng.act_dim, device="cuda", dtype=torch.float32)
    eng.step(act)
    inv0 = eng.counters["invalid_env_steps"]
    w = np.zeros(n, np.float32)
    w[3] = 1.0
    eng.set_clip_weights(w)                        # one-hot: every re-seeded episode would take clip 3
    eng.load_smpl_clips(pose[:n], trans[:n], clip_models=cm[:n])
    eng.step(act)
    assert eng.counters["invalid_env_steps"] == inv0 + E
    eng.reset(np.arange(E), clip=np.zeros(E, np.int32), start=0, length=2)
    seen = set()
    for _ in range(40):                            # the 2-frame episodes end at the first step and re-seed from the clip CDF
        eng.step(act)
        seen |= set(eng.get_states()["clip"].tolist())
    assert len(seen) > 5, seen                     # the default rule (len // t_max + 1 copies per clip), not the one-hot weights
    eng.close()


def test_bad_arguments_keep_the_old_table(table):
    import torch
    from uhc_b200.agent import BatchedAgent
    from uhc_b200.engine import EX_SIZE
    models, pose, trans, cm, ref = table
    n = 12
    ag = BatchedAgent(16, {"pose_aa": pose[:n], "trans": trans[:n]}, device=0, policy_hsize=(64, 32), value_hsize=(64, 32), model=models[0],
                      variants=models, clip_models=cm[:n])
    eng, lib = ag.engine, ag.engine.lib
    before = eng.get_clip_frames()
    ref_n = ref[:sum(len(p) for p in pose[:n])]
    assert (np.abs(before - ref_n) <= 1e-6 * np.maximum(1.0, np.abs(ref_n))).all()
    ev0 = ag.evaluate(0, n, False)
    P = np.ascontiguousarray(np.concatenate(pose[:4]))
    lens = np.array([len(p) for p in pose[:4]], np.int32)
    shp, cmod = np.zeros((4, 17)), np.zeros(4, np.int32)
    d = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    i = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))

    def call(nc=4, ln=lens, pd=72, pose_=P, tr=None, sh=shp, cmo=None):
        rc = lib.uhc_load_clips_smpl(eng.h, C.c_int(nc), i(ln), C.c_int(pd), d(pose_) if pose_ is not None else None, d(tr) if tr is not None else None,
                                     d(sh), i(cmo) if cmo is not None else None)
        return rc, lib.uhc_last_error().decode()
    short = lens.copy()
    short[2] = 1
    nan_pose = P.copy()
    nan_pose[17, 40] = np.nan
    inf_tr = np.zeros((len(P), 3))
    inf_tr[5, 2] = np.inf
    nan_shape = shp.copy()
    nan_shape[1, 3] = np.nan
    cases = {"nclips": dict(nc=0), "short": dict(ln=short), "pose_dim": dict(pd=69), "null_pose": dict(pose_=None), "clip_model": dict(cmo=np.array([0, 1, 2, 0], np.int32)),
             "nan_pose": dict(pose_=nan_pose), "inf_trans": dict(tr=inf_tr), "nan_shape": dict(sh=nan_shape)}
    for name, kw in cases.items():
        rc, msg = call(**kw)
        assert rc < 0 and msg.startswith("uhc_load_clips_smpl"), (name, rc, msg)
    assert call(cmo=cmod)[0] == 0 and np.isfinite(eng.get_clip_frames(0, int(lens.sum()))).all()     # the same call with good arguments is accepted
    eng.load_smpl_clips(pose[:n], trans[:n], clip_models=cm[:n])
    eng.reset(np.arange(16), clip=np.arange(16) % n)
    inv = eng.counters["invalid_env_steps"]
    for name, kw in cases.items():
        assert call(**kw)[0] < 0
    eng.step(torch.zeros(16, eng.act_dim, device="cuda", dtype=torch.float32))
    assert eng.counters["invalid_env_steps"] == inv, "a rejected call must not invalidate the env records"
    assert list(eng.clip_len) == [len(p) for p in pose[:n]]
    assert np.array_equal(eng.get_clip_frames(), before)
    with pytest.raises(RuntimeError):
        eng.get_clip_frames(int(eng.clip_len.sum()) - 1, 2)
    ev = ag.evaluate(0, n, False)
    for k in ("nframes", "last_t", "fail_any", "reward_sum", "clip_metrics"):
        assert np.array_equal(ev[k], ev0[k], equal_nan=True), k
    for a, b in zip(ev["frame_metrics"], ev0["frame_metrics"]):
        assert np.array_equal(a, b, equal_nan=True)
    assert before.shape[1] == EX_SIZE
    eng.close()


def _per_clip(cfg, epoch, names):
    out = {}
    for nm in names:
        src = os.path.join(cfg.output_dir, f"{epoch}_{nm}_coverage_full.pkl")
        out[nm] = joblib.load(src)
        os.remove(src)
    return out


def test_eval_policy_device_motion_lib_matches_host(tmp_path, monkeypatch):
    """eval_policy through the drop-in with motion_lib: device and with the default (host) on the same synthetic dataset and a second test
    loader (two table reloads per evaluation): the same success per clip, per-clip metrics within 0.01 mm"""
    import torch
    from tests.helpers import write_synthetic_pkl
    from tests.test_gpu_dropin import _cfg
    from uhc.agents import agent_dict
    res = {}
    for ml in ("host", "device"):
        (tmp_path / ml).mkdir()
        cfg = _cfg(tmp_path / ml, monkeypatch)
        cfg.data_specs["file_path"] = write_synthetic_pkl(str(tmp_path / "clips.pkl"), nclips=8, seed=4)
        cfg.data_specs["test_file_path"] = write_synthetic_pkl(str(tmp_path / "test_clips.pkl"), nclips=5, seed=7)
        if ml == "device":
            cfg.cfg_dict["motion_lib"] = "device"        # the extra key, as a yaml line `motion_lib: device` sets it
        ac = agent_dict[cfg.agent_name](cfg, torch.float32, torch.device("cuda", 0), training=True, checkpoint_epoch=0)
        assert len(ac.test_data_loaders) == 2
        if ml == "device":
            assert ac.data_loader._experts is None and ac.test_data_loaders[1]._experts is None, "device path: no host expert tables"
        names = [l.name for l in ac.test_data_loaders]
        ac.eval_policy(epoch=3, dump=True)
        res[ml] = _per_clip(cfg, 3, names)
        if ml == "device":
            assert ac.data_loader._experts is None and ac.test_data_loaders[1]._experts is None
            assert len(ac.agent.engine.clip_len) == ac.data_loader.get_len()
        ac.agent.engine.close()
        del ac
    for nm in res["host"]:
        h, g = res["host"][nm], res["device"][nm]
        assert list(h) == list(g)
        for k in h:
            assert np.array_equal(h[k]["succ"], g[k]["succ"]), (nm, k)
            for m in ("root_dist", "mpjpe", "mpjpe_g", "pa_mpjpe", "accel_dist", "vel_dist"):
                if m in h[k]:
                    assert abs(np.mean(h[k][m]) - np.mean(g[k][m])) <= 0.01, (nm, k, m, np.mean(h[k][m]), np.mean(g[k][m]))
