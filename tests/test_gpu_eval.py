"""GPU: policy evaluation on the device (uhc_evaluate / uhc_eval_metrics, include/uhc_eval.h; BatchedAgent.evaluate; AgentCopycat.eval_policy)
against the host loop it replaced, restated here as the reference implementation (host_eval_loop / host_eval_policy): lock-step batches
of E clips stepped until the longest ends, three device-to-host reads and a state gather per step, fail_safe through set_states, numpy
metrics (uhc_b200/metrics.py) per clip."""
import ctypes as C
import os
import shutil

import joblib
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
KEYS = ("qpos", "qvel", "wbpos", "wbquat", "bquat", "bangvel", "ee_wpos", "com")


# ---------------------------------------------------------------- the reference: the host loop eval_policy ran before uhc_evaluate
def host_eval_loop(agent, experts, n, fail_safe):
    """clips 0 .. n-1 of the loaded table, E at a time, each batch stepped until its longest clip ends.  Returns per clip: pred / pred_jpos /
    t (one row per recorded step), last_t, fail_any, rsum."""
    import torch
    from uhc_b200 import nn
    eng, E = agent.engine, agent.E
    out = []
    for c0 in range(0, n, E):
        ids = np.arange(min(E, n - c0), dtype=np.int32)
        clips = (c0 + ids).astype(np.int32)
        if len(ids) < E:                                   # idle envs: park them on clip c0 so every record is valid (their outputs are ignored)
            eng.reset(np.arange(len(ids), E, dtype=np.int32), np.full(E - len(ids), c0, np.int32), 0, None)
        obs = eng.reset(ids, clips, 0, None)
        lens = eng.clip_len[clips]
        alive = np.ones(len(ids), bool); fail_any = np.zeros(len(ids), bool)
        rsum = np.zeros(len(ids)); last_t = np.zeros(len(ids), np.int64)
        traj = [dict(pred=[], pred_jpos=[], t=[]) for _ in ids]
        det = torch.ones(E, dtype=torch.uint8, device=obs.device)
        for t in range(int(lens.max()) - 1):
            s = agent.running_state(obs, update=False)
            mean = agent.policy.forward_tc(s)
            a, _ = nn.gaussian_sample(mean, agent.log_std, 0, 0, det)
            obs, rew, ci, fail, end, pct = eng.step(a)
            f, e, r = fail.cpu().numpy()[ids] != 0, end.cpu().numpy()[ids] != 0, rew.cpu().numpy()[ids]
            live = np.nonzero(alive)[0]
            st = eng.get_states(ids[live])
            for j, i in enumerate(live):
                traj[i]["pred"].append(st["qpos"][j].copy()); traj[i]["pred_jpos"].append(st["xpos"][j].reshape(-1).copy()); traj[i]["t"].append(int(st["cur_t"][j]))
                last_t[i] = st["cur_t"][j]
            rsum[live] += r[live]
            failed = live[f[live]]
            fail_any[failed] = True
            if len(failed):
                if fail_safe:
                    tt = [min(int(last_t[i]), experts[clips[i]]["qpos"].shape[0] - 1) for i in failed]
                    eng.set_states(ids[failed], np.stack([experts[clips[i]]["qpos"][k] for i, k in zip(failed, tt)]),
                                   np.stack([experts[clips[i]]["qvel"][k] for i, k in zip(failed, tt)]))
                else:
                    alive[failed] = False
            alive[live[e[live]]] = False
            if not alive.any():
                break
        for i in ids:
            out.append(dict(pred=np.array(traj[i]["pred"]).reshape(-1, 76), pred_jpos=np.array(traj[i]["pred_jpos"]).reshape(-1, 72),
                            t=np.array(traj[i]["t"], dtype=np.int64), last_t=int(last_t[i]), fail_any=bool(fail_any[i]), rsum=float(rsum[i]), len=int(lens[i])))
    return out


def host_eval_policy(ac, epoch=0, dump=False):
    """AgentCopycat.eval_policy as it was before uhc_evaluate (host loop + numpy metrics per clip)"""
    import os.path as osp
    from uhc_b200.metrics import compute_metrics
    cfg = ac.cfg
    res_dicts = []
    eng = ac.agent.engine
    for loader in ac.test_data_loaders:
        n = loader.get_len()
        if loader is not ac.data_loader:
            eng.load_clips(loader.experts, loader.shapes)
        eng.set_cfg(**ac._env_cfg(test=True))
        res = {}
        for i, tr in enumerate(host_eval_loop(ac.agent, loader.experts, n, cfg.fail_safe)):
            k = loader.data_keys[i]
            ex = loader.experts[i]
            tt = np.minimum(tr["t"], ex["len"] - 1)
            percent = float(tr["last_t"]) / float(max(tr["len"] - 1, 1))
            r_i = {"pred": tr["pred"], "gt": np.asarray(ex["qpos"])[tt], "pred_jpos": tr["pred_jpos"], "gt_jpos": np.asarray(ex["wbpos"])[tt],
                   "percent": 1.0 if (percent >= 1.0 and not tr["fail_any"]) else min(percent, 0.999), "fail_safe": bool(tr["fail_any"] and cfg.fail_safe)}
            m = compute_metrics(r_i) if len(tt) >= 3 else {"succ": np.array([False])}
            m["succ"] = np.array([bool(m["succ"][0]) and not tr["fail_any"]])
            m["reward"] = np.float64(tr["rsum"]) / max(tr["len"] - 1, 1)
            m["percent"] = percent
            res[k] = m
            if k in ac.freq_dict:
                ac.freq_dict[k] = (ac.freq_dict[k] + [[1.0 if m["succ"][0] else min(percent, 0.999), 0]])[-ac.max_freq:]
        if loader is not ac.data_loader:
            eng.load_clips(ac.data_loader.experts, ac.data_loader.shapes)
        eng.set_cfg(**ac._env_cfg(test=False))
        ac.agent.obs = None
        names = ("succ", "reward", "mpjpe", "mpjpe_g", "pa_mpjpe", "accel_dist", "vel_dist", "root_dist")
        metrics = {m: float(np.mean([np.mean(r[m]) for r in res.values() if m in r])) if any(m in r for r in res.values()) else float("nan") for m in names}
        coverage = int(round(metrics["succ"] * n))
        metrics.update(mean_coverage=coverage / n, num_coverage=coverage, all_coverage=n)
        del metrics["succ"]
        res_dicts.append({f"coverage_{loader.name}": metrics})
        if dump:
            joblib.dump(res, osp.join(cfg.output_dir, f"{epoch}_{loader.name}_coverage_full.pkl"))
    ac._push_clip_weights()
    return res_dicts


# ---------------------------------------------------------------- fixtures
def eval_clip_set(golden_dir, nsyn=150, seed=0):
    """nsyn synthetic clips (kinds normal / sitting / airborne, lengths 2 .. 400) + the sway and kick goldens"""
    from uhc_b200.motion_lib import synthetic_clip
    rng = np.random.RandomState(seed)
    lens = np.concatenate([[2, 3, 4, 400], rng.randint(2, 401, nsyn - 4)])
    experts = [synthetic_clip(int(T), rng, kind=("normal", "sitting", "airborne")[i % 3]) for i, T in enumerate(lens)]
    shapes = [np.zeros(17) for _ in experts]
    for tag in ("sway", "kick"):
        z = np.load(os.path.join(golden_dir, f"expert_{tag}.npz"))
        experts.append({k: z[k] for k in KEYS})
        shapes.append(np.concatenate([z["beta"][0], [z["gender"][0]]]))
    for e in experts:
        e["len"] = len(e["qpos"])
    return experts, shapes


@pytest.fixture(scope="module")
def clip_set(golden_dir):
    return eval_clip_set(golden_dir)


def _agent(experts, shapes, actor, E=64, seed=3, **env_cfg):
    from uhc_b200.agent import BatchedAgent
    kw = dict(actor_type="mcp", num_primitive=4, composer_dim=(64, 32)) if actor == "mcp" else {}
    ag = BatchedAgent(E, experts, shapes, policy_hsize=(128, 64), value_hsize=(64,), seed=seed, log_std=-2.3, **kw, **env_cfg)
    ag.engine.set_cfg(auto_reset=0)
    # a seeded random normaliser: large normalised inputs make the untrained policy fail often
    st = ag.running_state.stats
    D = ag.obs_dim
    g = np.random.RandomState(seed)
    import torch
    st[0] = 2.0
    st[1:1 + D] = torch.as_tensor(g.normal(0, 0.05, D), device=st.device)
    st[1 + D:1 + 2 * D] = torch.as_tensor(g.uniform(0.001, 0.01, D), device=st.device)
    return ag


# ---------------------------------------------------------------- tests
def test_eval_metrics_kernel_matches_reference_golden(golden_dir):
    import torch
    from uhc_b200.engine import load_library
    from uhc_b200.agent import EVAL_METRICS
    L = load_library()
    L.uhc_eval_last_error.restype = C.c_char_p
    g = np.load(os.path.join(golden_dir, "metrics.npz"))
    ins = {k: np.concatenate([g[f"{t}.in.{k}"] for t in ("a", "b")]) for k in ("pred", "gt", "pred_jpos", "gt_jpos")}
    Ta = len(g["a.in.pred"])
    off = np.array([0, Ta, len(ins["pred"])], np.int32)
    d = {k: torch.as_tensor(v, device="cuda", dtype=torch.float64).contiguous() for k, v in ins.items()}
    fm = torch.full((len(ins["pred"]), 6), -1.0, device="cuda", dtype=torch.float64)
    cm = torch.full((2, 6), -1.0, device="cuda", dtype=torch.float64)
    offd = torch.as_tensor(off, device="cuda")
    p = lambda x: C.c_void_p(x.data_ptr())
    assert L.uhc_eval_metrics(p(d["pred"]), p(d["gt"]), p(d["pred_jpos"]), p(d["gt_jpos"]), p(offd), None, C.c_int(2), p(fm), p(cm), None) == 0, L.uhc_eval_last_error()
    torch.cuda.synchronize()
    fm, cm = fm.cpu().numpy(), cm.cpu().numpy()
    for ci, tag in enumerate(("a", "b")):
        rows = fm[off[ci]:off[ci + 1]]
        got = dict(zip(EVAL_METRICS, rows.T))
        got["vel_dist"], got["accel_dist"] = got["vel_dist"][1:], got["accel_dist"][2:]
        for j, k in enumerate(EVAL_METRICS):
            ref = g[f"{tag}.out.{k}"]
            assert got[k].shape == ref.shape
            assert np.abs(got[k] - ref).max() < 1e-8 * max(1.0, np.abs(ref).max()), (tag, k)
            assert abs(cm[ci, j] - ref.mean()) < 1e-8 * max(1.0, abs(ref.mean())), (tag, k)
    # bad arguments
    z = torch.zeros(1, device="cuda", dtype=torch.float64)
    assert L.uhc_eval_metrics(p(d["pred"]), p(d["gt"]), p(d["pred_jpos"]), p(d["gt_jpos"]), p(offd), None, C.c_int(0), p(z), p(z), None) < 0
    assert b"n <= 0" in L.uhc_eval_last_error()
    assert L.uhc_eval_metrics(None, p(d["gt"]), p(d["pred_jpos"]), p(d["gt_jpos"]), p(offd), None, C.c_int(2), p(z), p(z), None) < 0
    assert b"missing buffer" in L.uhc_eval_last_error()


@pytest.mark.parametrize("actor,fail_safe,n", [("gauss", True, None), ("gauss", False, None), ("mcp", True, None), ("mcp", False, None), ("gauss", True, 40)])
def test_evaluate_matches_host_loop(clip_set, actor, fail_safe, n):
    """more clips than env slots (E = 64, 152 clips) through the work queue against the lock-step host loop: per clip, recorded rows, cur_t,
    failure flags and trajectories bit for bit; rewards to 1e-6 relative; metrics to 1e-3 mm (device fp32 expert table vs fp64 host table)"""
    from uhc_b200.metrics import compute_metrics
    from uhc_b200.agent import EVAL_METRICS
    experts, shapes = clip_set
    n = n or len(experts)
    ag = _agent(experts, shapes, actor)
    ev = ag.evaluate(0, n, fail_safe, trajectories=True)
    if fail_safe:       # every clip runs to its end
        assert ev["steps"] >= int(max(e["len"] for e in experts[:n])) - 1
    host = host_eval_loop(ag, experts, n, fail_safe)
    assert ag.engine.counters["invalid_env_steps"] == 0
    nfail = 0
    for i, h in enumerate(host):
        T = len(h["t"])
        assert ev["nframes"][i] == T and ev["last_t"][i] == h["last_t"] and bool(ev["fail_any"][i]) == h["fail_any"], i
        assert np.array_equal(ev["frame_t"][i], h["t"]), i
        assert np.array_equal(ev["pred_qpos"][i], h["pred"].astype(np.float32)), (i, np.abs(ev["pred_qpos"][i] - h["pred"]).max())
        assert np.array_equal(ev["pred_jpos"][i], h["pred_jpos"].astype(np.float32)), i
        assert abs(ev["reward_sum"][i] - h["rsum"]) <= 1e-6 * max(1.0, abs(h["rsum"])), i
        nfail += h["fail_any"]
        L = h["len"]
        succ_h = T >= 3 and h["last_t"] >= L - 1 and not h["fail_any"]
        succ_d = ev["nframes"][i] >= 3 and ev["last_t"][i] / max(L - 1, 1) >= 1.0 and not ev["fail_any"][i]
        assert succ_h == succ_d
        if T >= 3:
            tt = np.minimum(h["t"], L - 1)
            m = compute_metrics({"pred": h["pred"], "gt": experts[i]["qpos"][tt], "pred_jpos": h["pred_jpos"], "gt_jpos": experts[i]["wbpos"][tt],
                                 "percent": 1.0, "fail_safe": False})
            fm = ev["frame_metrics"][i]
            for j, k in enumerate(EVAL_METRICS):
                got = fm[2:, j] if k == "accel_dist" else (fm[1:, j] if k == "vel_dist" else fm[:, j])
                assert got.shape == m[k].shape and np.abs(got - m[k]).max() < 1e-3, (i, k, np.abs(got - m[k]).max())
                assert abs(ev["clip_metrics"][i, j] - m[k].mean()) < 1e-3, (i, k)
        else:
            assert np.isnan(ev["clip_metrics"][i]).all()
    assert nfail >= len(host) // 4, "the random policy should fail often (%d of %d)" % (nfail, len(host))
    # a second evaluation on the same engine (cached graph, queue re-initialised) repeats the first
    ev2 = ag.evaluate(0, n, fail_safe)
    assert np.array_equal(ev2["nframes"], ev["nframes"]) and np.array_equal(ev2["reward_sum"], ev["reward_sum"])
    ag.engine.close()


def test_evaluate_rejects_bad_arguments(clip_set):
    import torch
    from uhc_b200.agent import UhcEvalBuf
    experts, shapes = clip_set
    ag = _agent(experts[:6], shapes[:6], "gauss", E=8)
    for clip0, n, msg in ((4, 5, "clip range"), (-1, 2, "clip range"), (0, 0, "clip range"), (0, -3, "clip range")):
        with pytest.raises(RuntimeError, match=msg):
            ag.evaluate(clip0, n, True)
    L = ag.engine.lib
    ag.evaluate(0, 2, True)       # a valid call sets the error-string restype
    lens = ag.engine.clip_len[:2]
    rows = int((lens - 1).sum())
    bufs = dict(pred_qpos=torch.zeros(rows, 76, device="cuda"), pred_jpos=torch.zeros(rows, 72, device="cuda"), frame_t=torch.zeros(rows, dtype=torch.int32, device="cuda"),
                frame_metrics=torch.zeros(rows, 6, dtype=torch.float64, device="cuda"), nframes=torch.zeros(2, dtype=torch.int32, device="cuda"),
                last_t=torch.zeros(2, dtype=torch.int32, device="cuda"), fail_any=torch.zeros(2, dtype=torch.int32, device="cuda"),
                reward_sum=torch.zeros(2, dtype=torch.float64, device="cuda"), clip_metrics=torch.zeros(2, 6, dtype=torch.float64, device="cuda"))

    def call(off, drop=None, cap=rows):
        b = UhcEvalBuf()
        fo = torch.as_tensor(np.asarray(off, np.int32), device="cuda")
        b.frame_off = fo.data_ptr()
        for k, v in bufs.items():
            setattr(b, k, None if k == drop else v.data_ptr())
        b.frame_cap = cap
        rc = L.uhc_evaluate(ag.engine.h, C.c_int(0), C.c_int(2), C.byref(ag._policy_struct()), C.c_void_p(ag.log_std.data_ptr()), C.c_void_p(ag.running_state.stats.data_ptr()),
                            C.c_float(5.0), C.c_int(1), C.byref(b), None)
        return rc, L.uhc_eval_last_error().decode()
    good = [0, int(lens[0] - 1), rows]
    assert call(good)[0] == 0
    rc, msg = call(good, drop="pred_jpos")
    assert rc < 0 and "missing buffer" in msg
    rc, msg = call([0, int(lens[0] - 2), rows - 1])
    assert rc < 0 and "frame_off" in msg and "needs" in msg
    rc, msg = call(good, cap=rows - 1)
    assert rc < 0 and "frame_cap" in msg
    torch.cuda.synchronize()
    ag.engine.close()


def test_eval_policy_matches_host_reference(tmp_path, monkeypatch):
    """AgentCopycat.eval_policy on the device against the host loop it replaced: returned dicts, the coverage dump and freq_dict, with a second
    test loader; then a training iteration runs with auto_reset restored"""
    import copy
    import torch
    from tests.helpers import write_synthetic_pkl
    from tests.test_gpu_dropin import _cfg
    from uhc.agents import agent_dict
    cfg = _cfg(tmp_path, monkeypatch)
    cfg.data_specs["test_file_path"] = write_synthetic_pkl(str(tmp_path / "sample_data" / "test_clips.pkl"), nclips=5, seed=7)
    ac = agent_dict[cfg.agent_name](cfg, torch.float32, torch.device("cuda", 0), training=True, checkpoint_epoch=0)
    assert len(ac.test_data_loaders) == 2
    ac.optimize_policy(0)
    f0 = copy.deepcopy(ac.freq_dict)
    ref = host_eval_policy(ac, epoch=5, dump=True)
    f_ref = copy.deepcopy(ac.freq_dict)
    names = [l.name for l in ac.test_data_loaders]
    for nm in names:
        shutil.move(os.path.join(cfg.output_dir, f"5_{nm}_coverage_full.pkl"), str(tmp_path / f"ref_{nm}.pkl"))
    ac.freq_dict = copy.deepcopy(f0)
    got = ac.eval_policy(epoch=5, dump=True)
    assert [list(d) for d in got] == [list(d) for d in ref]
    for dg, dr in zip(got, ref):
        for key in dr:
            assert list(dg[key]) == list(dr[key])
            for m, v in dr[key].items():
                if m in ("mean_coverage", "num_coverage", "all_coverage", "reward"):
                    assert dg[key][m] == v, (key, m)
                else:
                    assert abs(dg[key][m] - v) < 1e-3 or (np.isnan(v) and np.isnan(dg[key][m])), (key, m, dg[key][m], v)
    assert ac.freq_dict == f_ref
    for nm in names:
        rg = joblib.load(os.path.join(cfg.output_dir, f"5_{nm}_coverage_full.pkl"))
        rr = joblib.load(str(tmp_path / f"ref_{nm}.pkl"))
        assert list(rg) == list(rr)
        for k in rr:
            assert list(rg[k]) == list(rr[k]), k
            for m in rr[k]:
                a, b = np.asarray(rg[k][m]), np.asarray(rr[k][m])
                assert a.shape == b.shape and a.dtype == b.dtype, (k, m)
                if m in ("succ", "reward", "percent"):
                    assert np.array_equal(a, b), (k, m)
                else:
                    assert np.abs(a - b).max() < 1e-3, (k, m)
    assert ac.agent.obs is None and ac.agent.engine._cfg.auto_reset == 1
    assert len(ac.agent.engine.clip_len) == ac.data_loader.get_len()
    info = ac.optimize_policy(1)
    assert np.isfinite(info["log"]["avg_reward"]) and info["log"]["num_steps"] >= cfg.min_batch_size


def _fixed_buffers(rows, n):
    import torch
    d = "cuda"
    return dict(frame_off=torch.zeros(n + 1, dtype=torch.int32, device=d), pred_qpos=torch.zeros(rows, 76, device=d), pred_jpos=torch.zeros(rows, 72, device=d),
                frame_t=torch.zeros(rows, dtype=torch.int32, device=d), frame_metrics=torch.zeros(rows, 6, dtype=torch.float64, device=d),
                nframes=torch.zeros(n, dtype=torch.int32, device=d), last_t=torch.zeros(n, dtype=torch.int32, device=d), fail_any=torch.zeros(n, dtype=torch.int32, device=d),
                reward_sum=torch.zeros(n, dtype=torch.float64, device=d), clip_metrics=torch.zeros(n, 6, dtype=torch.float64, device=d))


def _evaluate_into(ag, bufs, n, fail_safe):
    """uhc_evaluate of clips 0 .. n-1 into caller buffers that stay the same from call to call (the route-B pattern)"""
    import torch
    from uhc_b200.agent import UhcEvalBuf
    L = ag.engine.lib
    L.uhc_eval_last_error.restype = C.c_char_p
    off = np.concatenate([[0], np.cumsum(ag.engine.clip_len[:n] - 1)]).astype(np.int32)
    bufs["frame_off"].copy_(torch.as_tensor(off))
    b = UhcEvalBuf()
    for k, v in bufs.items():
        setattr(b, k, v.data_ptr())
    b.frame_cap = bufs["pred_qpos"].shape[0]
    rc = L.uhc_evaluate(ag.engine.h, C.c_int(0), C.c_int(n), C.byref(ag._policy_struct()), C.c_void_p(ag.log_std.data_ptr()),
                        C.c_void_p(ag.running_state.stats.data_ptr()), C.c_float(ag.running_state.clip), C.c_int(int(fail_safe)), C.byref(b), None)
    assert rc == 0, L.uhc_eval_last_error()
    torch.cuda.synchronize()
    h = {k: v.cpu().numpy() for k, v in bufs.items()}
    return {k: h[k] for k in ("nframes", "last_t", "fail_any", "reward_sum")} | \
        {k: [h[k][off[i]:off[i] + h["nframes"][i]] for i in range(n)] for k in ("pred_qpos", "pred_jpos", "frame_t", "frame_metrics")}


def _assert_same_evaluation(a, b):
    for k in ("nframes", "last_t", "fail_any", "reward_sum"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("pred_qpos", "pred_jpos", "frame_t", "frame_metrics"):
        for i, (x, y) in enumerate(zip(a[k], b[k])):
            assert np.array_equal(x, y, equal_nan=True), (k, i)


def test_evaluate_sees_a_reloaded_table_and_a_new_configuration(clip_set):
    """the same caller buffers across calls: after uhc_load_clips of another table with the same clip count and a uhc_engine_set_cfg, the next
    uhc_evaluate must give what a fresh engine on that table and configuration gives"""
    experts, shapes = clip_set
    t1, t2 = list(range(0, 40)), list(range(40, 80))
    rows = int(max(sum(experts[i]["len"] - 1 for i in t1), sum(experts[i]["len"] - 1 for i in t2)))
    ag = _agent([experts[i] for i in t1], [shapes[i] for i in t1], "gauss", E=16)
    bufs = _fixed_buffers(rows, 40)
    first = _evaluate_into(ag, bufs, 40, True)
    ag.engine.load_clips([experts[i] for i in t2], [shapes[i] for i in t2])
    ag.engine.set_cfg(body_diff_thresh=0.3)
    again = _evaluate_into(ag, bufs, 40, True)
    fresh = _agent([experts[i] for i in t2], [shapes[i] for i in t2], "gauss", E=16)
    fresh.engine.set_cfg(body_diff_thresh=0.3)
    _assert_same_evaluation(again, _evaluate_into(fresh, _fixed_buffers(rows, 40), 40, True))
    assert not np.array_equal(first["reward_sum"], again["reward_sum"])
    ag.engine.close(); fresh.engine.close()


def test_evaluate_ignores_auto_reset_and_reactive_starts(clip_set):
    """auto_reset = 1 with reactive_v = 1 and reactive_rate = 1 (every training reset starts from the standing-neutral pose) must evaluate exactly
    like auto_reset = 0: the first clip of every slot as well as the clips it takes from the queue start from the clip's own frame 0"""
    experts, shapes = clip_set
    n = 60
    rows = int(sum(e["len"] - 1 for e in experts[:n]))
    ag = _agent(experts[:n], shapes[:n], "gauss", E=16, reactive_v=1, reactive_rate=1.0)
    bufs = _fixed_buffers(rows, n)
    ag.engine.set_cfg(auto_reset=1)
    with_reset = _evaluate_into(ag, bufs, n, True)
    ag.engine.set_cfg(auto_reset=0)
    _assert_same_evaluation(with_reset, _evaluate_into(ag, bufs, n, True))
    ag.engine.close()
