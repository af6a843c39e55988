#!/usr/bin/env python
"""Generate tests/golden/*.npz by executing the REFERENCE's own Python (see tools/ref_harness.py).

Runs only in the build container (needs /root/reference); the vectors it writes travel with the repo.
  expert_<clip>.npz     inputs pose_aa/trans/beta/gender  ->  smpl_to_qpose + Humanoid.qpos_fk outputs
                        (uhc/smpllib/smpl_mujoco.py:543-607, uhc/smpllib/torch_smpl_humanoid.py:155-261)
  env_<clip>_<act>.npz  HumanoidEnv.reset/step + world_rfc_implicit_reward traces on the oracle physics
                        (uhc/envs/humanoid_im.py, uhc/losses/reward_function.py:12-88)
  ppo_small.npz         PolicyGaussian / Value / estimate_advantages / AgentPPO.update_policy / ZFilter traces
                        (uhc/khrylib/rl/core/*, uhc/khrylib/rl/agents/agent_ppo.py, khrylib/utils/zfilter.py)
  math_doctest.npz      the known-answer constants in uhc/utils/transformation.py doctests
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ref_harness as H  # noqa: E402

OUT = os.path.join(H.ROOT, "tests", "golden")
EXPERT_KEYS = ["qpos", "qvel", "wbpos", "wbquat", "bquat", "body_com", "bangvel", "ee_wpos", "ee_pos", "com", "rlinv",
               "rlinv_local", "rangv"]


def gen_env(cfg, dl, key, tag, nframes, nsteps, act_mode, seed=1, mode="train", out_tag=None, save_expert=True, term_body=None, reward_only=False):
    from uhc.losses.reward_function import reward_func
    reward = reward_func[cfg.reward_id]                       # world_rfc_implicit (uhc_implicit_shape) / world_rfc_explicit (uhc_explicit)
    seq = dl.get_sample_from_key(key, full_sample=False, fr_start=0)
    seq = {k: (v[:nframes] if hasattr(v, "shape") and v.shape[:1] == (300,) or (hasattr(v, "shape") and len(v) > nframes) else v)
           for k, v in seq.items()}
    env = H.make_env(cfg, seq, mode=mode)
    env.seed(seed)
    ex = env.expert
    if term_body == "Head" and "head_height_lb" not in ex:      # the AMASS loader's expert carries height_lb only (torch_smpl_humanoid.py:250); uhc/utils/tools.py:95 defines the head bound
        ex["head_height_lb"] = ex["wbpos"].reshape(ex["wbpos"].shape[0], -1, 3)[:, env.get_head_idx(), 2].min()
    if save_expert:
        np.savez_compressed(os.path.join(OUT, f"expert_{tag}.npz"), pose_aa=seq["pose_aa"][:, :72].copy(),
                            trans=seq["trans"], beta=seq["beta"], gender=seq["gender"],
                            height_lb=ex["height_lb"], length=ex["len"], **{k: ex[k] for k in EXPERT_KEYS})
    rng = np.random.RandomState(seed)
    obs0 = env.reset()
    rec = {k: [] for k in ("action", "obs", "reward", "c_info", "fail", "end", "percent", "qpos", "qvel", "torque",
                           "body_diff", "xpos", "bquat", "prev_bquat", "ncon")}
    for t in range(nsteps):
        if act_mode == "zero":
            a = np.zeros(env.action_dim)
        else:
            a = rng.normal(0.0, 0.1, env.action_dim)
            if env.vf_dim == 6:
                a[69:75] *= 0.3
            else:                                             # explicit residual forces: 24 x (contact point 3, force 3, torque 3)
                vf = a[69:69 + env.vf_dim].reshape(-1, 9)
                vf[:, 3:] *= 0.05
        ob, _, done, info = env.step(a.copy())
        r, ci = reward(env, None, a, info)
        rec["action"].append(a); rec["obs"].append(ob); rec["reward"].append(r); rec["c_info"].append(ci)
        rec["fail"].append(bool(info["fail"])); rec["end"].append(bool(info["end"])); rec["percent"].append(info["percent"])
        rec["qpos"].append(env.data.qpos.copy()); rec["qvel"].append(env.data.qvel.copy())
        rec["torque"].append(np.array(env.curr_torque)); rec["body_diff"].append(env.calc_body_diff())
        rec["xpos"].append(env.data.body_xpos[1:].copy()); rec["bquat"].append(env.bquat.copy())
        rec["prev_bquat"].append(env.prev_bquat.copy()); rec["ncon"].append(env.data.ncon)
        if info["end"]:
            break
    extra = {"head_idx": env.get_head_idx(), "head_height_lb": ex["head_height_lb"]} if term_body == "Head" else {}
    if reward_only:     # same trajectory as the env_<tag>_<act_mode> golden: keep what the reward function returned
        np.savez_compressed(os.path.join(OUT, f"env_{out_tag}_{act_mode}.npz"), base=f"env_{tag}_{act_mode}.npz", reward_id=cfg.reward_id, reward=np.array(rec["reward"]),
                            c_info=np.array(rec["c_info"]), action=np.array(rec["action"]), reward_weights=np.array([cfg.reward_weights.get(k, d) for k, d in
                            (("w_p", 0.6), ("w_v", 0.1), ("w_e", 0.2), ("w_c", 0.1), ("w_vf", 0.0))]))
        print(out_tag, "mean r %.4f" % np.mean(rec["reward"]))
        return
    if term_body:       # same trajectory as the env_<tag>_<act_mode> golden (the actions do not depend on the flags): keep the flags and the heights they are decided on
        np.savez_compressed(os.path.join(OUT, f"env_{out_tag}_{act_mode}.npz"), base=f"env_{tag}_{act_mode}.npz", term_body=term_body, height_lb=ex["height_lb"],
                            fail=np.array(rec["fail"]), end=np.array(rec["end"]), percent=np.array(rec["percent"]), action=np.array(rec["action"]),
                            root_z=np.array(rec["qpos"])[:, 2], head_z=np.array(rec["xpos"])[:, env.get_head_idx(), 2], **extra)
        print(out_tag, "fail from step", int(np.argmax(rec["fail"])))
        return
    np.savez_compressed(os.path.join(OUT, f"env_{out_tag or tag}_{act_mode}.npz"), obs0=obs0, expert=f"expert_{tag}.npz", vf_dim=env.vf_dim, **extra,
                        **{k: np.array(v) for k, v in rec.items()})
    print(tag, act_mode, "steps", len(rec["reward"]), "fails", int(np.sum(rec["fail"])), "mean r %.4f" % np.mean(rec["reward"]),
          "max ncon", max(rec["ncon"]))


def gen_ppo():
    import torch
    from uhc.khrylib.models.mlp import MLP
    from uhc.khrylib.rl.core.policy_gaussian import PolicyGaussian
    from uhc.khrylib.rl.core.critic import Value
    from uhc.khrylib.rl.core.common import estimate_advantages
    from uhc.khrylib.rl.agents.agent_ppo import AgentPPO
    from uhc.khrylib.utils.zfilter import ZFilter

    torch.set_default_dtype(torch.float64)
    torch.manual_seed(1)
    rng = np.random.RandomState(1)
    S, A, N, hs = 657, 105, 384, [96, 64, 48]

    class Cfg:
        policy_hsize, policy_htype, fix_std, log_std = hs, "gelu", True, -2.3

    pol = PolicyGaussian(Cfg(), action_dim=A, state_dim=S)
    val = Value(MLP(S, hs, "gelu"))
    # obs normaliser trace
    zf = ZFilter((S,), clip=5)
    raw = rng.normal(0, 2.0, (40, S)) * rng.uniform(0.1, 3, S)
    zout = np.array([zf(x) for x in raw])
    states = rng.normal(0, 1, (N, S)).clip(-5, 5)
    st = torch.tensor(states)
    with torch.no_grad():
        mean = pol.forward(st).loc.numpy()
        actions_t = pol.select_action(st, False)
        logp = pol.get_log_prob(st, actions_t).numpy()
        values = val(st).numpy()
    actions = actions_t.numpy()
    rewards = rng.uniform(0, 1, N)
    masks = (rng.uniform(0, 1, N) > 0.05).astype(np.float64)
    masks[-1] = 0
    adv, ret = estimate_advantages(torch.tensor(rewards)[:, None], torch.tensor(masks)[:, None], torch.tensor(values), 0.95, 0.95)
    exps = (rng.uniform(0, 1, N) > 0.1).astype(np.float64)
    p0 = {k: v.detach().numpy().copy() for k, v in pol.state_dict().items()}
    v0 = {k: v.detach().numpy().copy() for k, v in val.state_dict().items()}

    agent = AgentPPO.__new__(AgentPPO)
    agent.policy_net, agent.value_net = pol, val
    agent.optimizer_policy = torch.optim.Adam(pol.parameters(), lr=5e-5)
    agent.optimizer_value = torch.optim.Adam(val.parameters(), lr=3e-4)
    agent.clip_epsilon, agent.opt_num_epochs, agent.use_mini_batch = 0.2, 3, False
    agent.policy_grad_clip = [(pol.parameters(), 40)]
    agent.update_modules = [pol, val]
    agent.value_opt_niter = 1
    agent.update_policy(st, actions_t, ret, adv, torch.tensor(exps))
    p1 = {k: v.detach().numpy().copy() for k, v in pol.state_dict().items()}
    v1 = {k: v.detach().numpy().copy() for k, v in val.state_dict().items()}
    out = dict(hsize=np.array(hs), states=states, actions=actions, mean=mean, logp=logp, values=values, rewards=rewards,
               masks=masks, advantages=adv.numpy(), returns=ret.numpy(), exps=exps, gamma=0.95, tau=0.95, clip_eps=0.2,
               epochs=3, policy_lr=5e-5, value_lr=3e-4, grad_clip=40.0, z_raw=raw, z_out=zout, z_mean=zf.rs.mean,
               z_std=zf.rs.std, z_n=zf.rs.n)
    for k, v in p0.items():
        out["p0." + k] = v
    for k, v in p1.items():
        out["p1." + k] = v
    for k, v in v0.items():
        out["v0." + k] = v
    for k, v in v1.items():
        out["v1." + k] = v
    np.savez_compressed(os.path.join(OUT, "ppo_small.npz"), **out)
    print("ppo_small: N", N, "adv mean/std", adv.mean().item(), adv.std().item())


def gen_mcp():
    """PolicyMCP (uhc/models/policy_mcp.py:9-37, the actor of config/release/uhc_implicit.yml) forward and AgentPPO.update_policy with it, in the
    reference's fp64 torch, at fixture size: 160 -> [128, 96] relu primitives x 4, composer 160 -> [48, 32] -> 4, 75 actions, N = 512 rows, 2 epochs."""
    import torch
    from uhc.khrylib.models.mlp import MLP
    from uhc.models.policy_mcp import PolicyMCP
    from uhc.khrylib.rl.core.critic import Value
    from uhc.khrylib.rl.agents.agent_ppo import AgentPPO
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(5)
    rng = np.random.RandomState(5)
    S, A, N, hs, P, cdim = 160, 75, 512, [128, 96], 4, [48, 32]

    class Cfg(dict):
        policy_hsize, policy_htype, fix_std, log_std, num_primitive = hs, "relu", True, -2.3, P
    pol = PolicyMCP(Cfg(composer_dim=cdim), action_dim=A, state_dim=S)
    val = Value(MLP(S, hs, "relu"))
    states = rng.normal(0, 1, (N, S)).clip(-5, 5)
    st = torch.tensor(states)
    with torch.no_grad():
        mean = pol.forward(st).loc.numpy()
        weight = pol.composer(st).numpy()
        actions_t = pol.select_action(st, False)
        logp = pol.get_log_prob(st, actions_t).numpy()
        values = val(st).numpy()
    ret = torch.tensor(values + rng.normal(0, 0.5, values.shape))
    adv = torch.tensor(rng.normal(0, 1, (N, 1)))
    exps = (rng.uniform(0, 1, N) > 0.1).astype(np.float64)
    p0 = {k: v.detach().numpy().copy() for k, v in pol.state_dict().items()}
    v0 = {k: v.detach().numpy().copy() for k, v in val.state_dict().items()}
    agent = AgentPPO.__new__(AgentPPO)
    agent.policy_net, agent.value_net = pol, val
    agent.optimizer_policy = torch.optim.Adam(pol.parameters(), lr=5e-5)
    agent.optimizer_value = torch.optim.Adam(val.parameters(), lr=3e-4)
    agent.clip_epsilon, agent.opt_num_epochs, agent.use_mini_batch = 0.2, 2, False
    agent.policy_grad_clip = [(pol.parameters(), 40)]
    agent.update_modules = [pol, val]
    agent.value_opt_niter = 1
    agent.update_policy(st, actions_t, ret, adv, torch.tensor(exps))
    with torch.no_grad():
        mean1 = pol.forward(st[:64]).loc.numpy()
    out = dict(hsize=np.array(hs), nprim=P, composer_dim=np.array(cdim), states=states.astype(np.float32), actions=actions_t.numpy(), mean=mean, weight=weight, logp=logp, values=values,
               returns=ret.numpy(), advantages=adv.numpy(), exps=exps, mean_after=mean1, epochs=2)
    # weights: p0 only for the layers (fp32 is enough to rebuild the fp64 init to 1e-8 relative); after the update the probe output and the head deltas
    for k, v in p0.items():
        out["p0." + k] = v.astype(np.float32)
    for k, v in v0.items():
        out["v0." + k] = v.astype(np.float32)
    p1 = pol.state_dict()
    for k, v in p1.items():
        out["p1." + k] = v.detach().numpy().astype(np.float32)
    for k, v in val.state_dict().items():
        out["v1." + k] = v.detach().numpy().astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "mcp_ppo.npz"), **out)
    print("mcp_ppo: mean abs", np.abs(mean).mean(), "weight row", weight[0])


def ppo_real_inputs(N=8192, S=657, A=105, hs=(2048, 1024, 512), seed=11):
    """Seeded inputs of the real-size PPO parity case, regenerated identically by tests/test_gpu_product_paths.py (numpy and torch CPU
    generators only): initial weights (nn.Linear rule, head x0.1 / bias 0), states, actions, returns, advantages, exps."""
    import torch
    g = torch.Generator().manual_seed(seed)
    dims = [S] + list(hs)

    def net(out_dim):
        Ws, bs = [], []
        d = dims + [out_dim]
        for i in range(len(d) - 1):
            k = 1.0 / np.sqrt(d[i])
            W = (torch.rand(d[i + 1], d[i], generator=g, dtype=torch.float64) * 2 - 1) * k
            b = (torch.rand(d[i + 1], generator=g, dtype=torch.float64) * 2 - 1) * k
            if i == len(d) - 2:
                W, b = W * 0.1, b * 0.0
            Ws.append(W.float().double()); bs.append(b.float().double())      # exactly representable in fp32
        return Ws, bs
    pol, val = net(A), net(1)
    rng = np.random.RandomState(seed)
    states = rng.normal(0, 1, (N, S)).clip(-5, 5).astype(np.float32).astype(np.float64)
    actions = rng.normal(0, 0.15, (N, A)).astype(np.float32).astype(np.float64)
    returns = rng.uniform(0, 8, N).astype(np.float32).astype(np.float64)
    adv = rng.normal(0, 1, N)
    adv = ((adv - adv.mean()) / adv.std()).astype(np.float32).astype(np.float64)
    exps = (rng.uniform(0, 1, N) > 0.1).astype(np.float64)
    probe = rng.normal(0, 1, (256, S)).clip(-5, 5).astype(np.float32).astype(np.float64)
    return pol, val, states, actions, returns, adv, exps, probe


def gen_ppo_real():
    """AgentPPO.update_policy (agent_ppo.py:16-51) at the production sizes 657-2048-1024-512-{105,1}, N = 8192, 3 epochs, fp64 on the CPU.
    The inputs are seeded (ppo_real_inputs); the golden keeps the policy / value outputs on a 256-row probe batch before and after the
    update and 4096 sampled entries of every parameter tensor after the update."""
    import torch
    from uhc.khrylib.models.mlp import MLP
    from uhc.khrylib.rl.core.policy_gaussian import PolicyGaussian
    from uhc.khrylib.rl.core.critic import Value
    from uhc.khrylib.rl.agents.agent_ppo import AgentPPO
    torch.set_default_dtype(torch.float64)
    torch.set_num_threads(os.cpu_count() or 1)
    (pW, pb), (vW, vb), states, actions, returns, adv, exps, probe = ppo_real_inputs()
    hs = [2048, 1024, 512]

    class Cfg:
        policy_hsize, policy_htype, fix_std, log_std = hs, "gelu", True, -2.3

    pol = PolicyGaussian(Cfg(), action_dim=105, state_dim=657)
    val = Value(MLP(657, hs, "gelu"))

    def load(net, Ws, bs, head):
        sd = net.state_dict()
        for i in range(3):
            sd[f"net.affine_layers.{i}.weight"] = Ws[i]; sd[f"net.affine_layers.{i}.bias"] = bs[i]
        sd[f"{head}.weight"], sd[f"{head}.bias"] = Ws[3], bs[3]
        net.load_state_dict(sd)
    load(pol, pW, pb, "action_mean"); load(val, vW, vb, "value_head")
    st, pr = torch.tensor(states), torch.tensor(probe)
    with torch.no_grad():
        mean0, v0 = pol.forward(pr).loc.numpy().copy(), val(pr).numpy().copy()
    agent = AgentPPO.__new__(AgentPPO)
    agent.policy_net, agent.value_net = pol, val
    agent.optimizer_policy = torch.optim.Adam(pol.parameters(), lr=5e-5)
    agent.optimizer_value = torch.optim.Adam(val.parameters(), lr=3e-4)
    agent.clip_epsilon, agent.opt_num_epochs, agent.use_mini_batch = 0.2, 3, False
    agent.policy_grad_clip = [(pol.parameters(), 40)]
    agent.update_modules = [pol, val]
    agent.value_opt_niter = 1
    agent.update_policy(st, torch.tensor(actions), torch.tensor(returns)[:, None], torch.tensor(adv)[:, None], torch.tensor(exps))
    with torch.no_grad():
        mean1, v1 = pol.forward(pr).loc.numpy().copy(), val(pr).numpy().copy()
    out = dict(N=8192, epochs=3, seed=11, mean0=mean0, v0=v0, mean1=mean1, v1=v1)
    rs = np.random.RandomState(5)
    for tag, net, W0, b0, head in (("p", pol, pW, pb, "action_mean"), ("v", val, vW, vb, "value_head")):
        sd = net.state_dict()
        for i in range(4):
            kw = f"net.affine_layers.{i}.weight" if i < 3 else f"{head}.weight"
            kb = f"net.affine_layers.{i}.bias" if i < 3 else f"{head}.bias"
            W1, b1 = sd[kw].numpy().reshape(-1), sd[kb].numpy().reshape(-1)
            idx = rs.randint(0, W1.size, 4096)
            out[f"{tag}.W{i}.idx"], out[f"{tag}.W{i}.new"], out[f"{tag}.W{i}.old"] = idx, W1[idx], W0[i].numpy().reshape(-1)[idx]
            out[f"{tag}.b{i}.new"], out[f"{tag}.b{i}.old"] = b1, b0[i].numpy()
    np.savez_compressed(os.path.join(OUT, "ppo_real.npz"), **out)
    print("ppo_real: |dmean| %.3e |dv| %.3e" % (np.abs(mean1 - mean0).mean(), np.abs(v1 - v0).mean()))


def gen_sampler(cfg):
    """DatasetAMASSSingle.sample_seq (dataset_amass_single.py:172-253) draw statistics on take5_test_small: (a) no success history
    (sample_keys rule), (b) the training loop's call with a success history (failure-weighted mixture)."""
    import random
    from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
    out = {}
    for tag, t_min, t_max in (("a", 15, 60), ("b", 15, 60)):
        cfg.data_specs["t_min"], cfg.data_specs["t_max"] = t_min, t_max
        dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
        keys = list(dl.data_keys)
        lens = np.array([dl.data["pose_aa"][k].shape[0] for k in keys])
        np.random.seed(3); random.seed(3)
        freq = None
        if tag == "b":   # synthetic per-clip success histories [success, fr_start] as agent_copycat.py:561 records them
            rs = np.random.RandomState(9)
            freq = {k: [[float(rs.uniform() < p), 0] for _ in range(30)] for k, p in zip(keys, np.linspace(0.1, 0.95, len(keys)))}
            out["freq_succ"] = np.array([[r[0] for r in freq[k]] for k in keys])
        n = 40000
        clip, start, length = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int64)
        for i in range(n):
            s = dl.sample_seq(freq_dict=freq, full_sample=False, sampling_temp=0.2, sampling_freq=0.5)
            clip[i], start[i], length[i] = keys.index(dl.curr_key), dl.fr_start, dl.fr_end - dl.fr_start
        out[f"{tag}.clip_hist"] = np.bincount(clip, minlength=len(keys))
        out[f"{tag}.start_mean"] = np.array([start[clip == c].mean() for c in range(len(keys))])
        out[f"{tag}.start_max"] = np.array([start[clip == c].max() for c in range(len(keys))])
        out[f"{tag}.len_ok"] = np.array(all(length[i] == min(t_max, lens[clip[i]] - start[i]) for i in range(n)))
        out["lens"], out["t_min"], out["t_max"], out["n"] = lens, t_min, t_max, n
        print("sampler", tag, out[f"{tag}.clip_hist"], out[f"{tag}.len_ok"])
    np.savez_compressed(os.path.join(OUT, "sampler_hist.npz"), **out)


def gen_metrics():
    """smpl_eval.compute_metrics / p_mpjpe (uhc/smpllib/smpl_eval.py:24-123) on seeded inputs."""
    from uhc.smpllib.smpl_eval import compute_metrics
    rng = np.random.RandomState(8)
    out = {}
    for tag, T in (("a", 40), ("b", 7)):
        gt = rng.normal(0, 0.3, (T, 76)); gt[:, 3:7] = rng.normal(size=(T, 4)); gt[:, 3:7] /= np.linalg.norm(gt[:, 3:7], axis=1, keepdims=True)
        pred = gt + rng.normal(0, 0.02, (T, 76)); pred[:, 3:7] /= np.linalg.norm(pred[:, 3:7], axis=1, keepdims=True)
        gj = rng.normal(0, 0.5, (T, 72)); pj = gj + rng.normal(0, 0.03, (T, 72))
        res = {"pred": pred, "gt": gt, "pred_jpos": pj, "gt_jpos": gj, "percent": 1.0 if tag == "a" else 0.6, "fail_safe": False}
        m = compute_metrics(res)
        for k, v in res.items():
            out[f"{tag}.in.{k}"] = np.asarray(v)
        for k, v in m.items():
            out[f"{tag}.out.{k}"] = np.asarray(v)
    np.savez_compressed(os.path.join(OUT, "metrics.npz"), **out)
    print("metrics golden:", {k: np.mean(v) for k, v in m.items()})


def gen_reactive(cfg, dl):
    """reset_model's reactive_v = 1 branch (humanoid_im.py:1255-1271, match_heading_and_pos :1312-1320) on the sway clip: reactive_rate = 1
    forces the standing-neutral start; the state / observation after env.reset() and three zero-action steps are recorded."""
    from uhc.losses.reward_function import world_rfc_implicit_reward
    key = "0-ACCAD_Male2General_c3d_A2- Sway_poses"
    seq = dl.get_sample_from_key(key, full_sample=False, fr_start=0)
    seq = {k: (v[:90] if hasattr(v, "shape") and len(v) > 90 else v) for k, v in seq.items()}
    cfg.reactive_v, cfg.reactive_rate = 1, 1.0
    env = H.make_env(cfg, seq, mode="train")
    env.seed(1)
    obs0 = env.reset()
    rec = dict(obs0=obs0, qpos0=env.data.qpos.copy(), qvel0=env.data.qvel.copy(), neutral_qpos=np.array(env.netural_data["qpos"]),
               neutral_qvel=np.array(env.netural_data["qvel"]), qpos=[], reward=[])
    for t in range(3):
        a = np.zeros(env.action_dim)
        ob, _, done, info = env.step(a)
        r, _ = world_rfc_implicit_reward(env, None, a, info)
        rec["qpos"].append(env.data.qpos.copy()); rec["reward"].append(r)
    cfg.reactive_v = 0
    np.savez_compressed(os.path.join(OUT, "reactive_sway.npz"), **{k: np.array(v) for k, v in rec.items()})
    print("reactive golden: z", rec["qpos0"][2], "joints == neutral", np.abs(rec["qpos0"][7:] - rec["neutral_qpos"][7:]).max())


def gen_math():
    from uhc.utils import transformation as T
    from uhc.utils import math_utils as MU
    rng = np.random.RandomState(3)
    qs = rng.normal(size=(16, 4))
    qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    vs = rng.normal(size=(16, 3))
    out = dict(
        q=qs, v=vs,
        about_axis=T.quaternion_about_axis(0.123, [1, 0, 0]),                     # transformation.py:350-351
        mul_doctest=T.quaternion_multiply([4, 1, -2, 3], [8, -5, 6, 7]),          # transformation.py:1481-1483
        euler_doctest=T.quaternion_from_euler(1, 2, 3, "ryxz"),                   # transformation.py:1237-1239
        mul=np.array([T.quaternion_multiply(qs[i], qs[(i + 1) % 16]) for i in range(16)]),
        inv=np.array([T.quaternion_inverse(q * 1.3) for q in qs]),
        euler_rzyx=np.array([T.quaternion_from_euler(v[0], v[1], v[2], "rzyx") for v in vs]),
        heading=np.array([MU.get_heading(q) for q in qs]),
        heading_q=np.array([MU.get_heading_q(q) for q in qs]),
        de_heading=np.array([MU.de_heading(q) for q in qs]),
        rot_from_quat=np.array([T.rotation_from_quaternion(q) for q in qs]),
        transform_vec=np.array([MU.transform_vec(v, q, "root") for v, q in zip(vs, qs)]),
        quat_mul_vec=np.array([MU.quat_mul_vec(q, v) for v, q in zip(vs, qs)]),
    )
    np.savez_compressed(os.path.join(OUT, "math_doctest.npz"), **out)
    print("math goldens ok", out["mul_doctest"])


# the configuration keys uhc.agents.agent_copycat.supported_variant reads, and the one the drop-in dispatches on
SUPPORTED_VARIANT_KEYS = ("agent_name", "obs_v", "actor_type", "reward_id", "fix_std", "residual_force", "obs_vel", "obs_coord", "obs_phase", "has_shape",
                         "env_term_body", "residual_force_mode", "residual_force_bodies", "residual_force_torque", "residual_force_bodies_num",
                         "residual_contact_only", "residual_contact_projection", "env_init_noise")


def gen_compat():
    """The drop-in boundary, recorded from the reference's own code for tests/test_checkpoint_compat.py, tests/test_shim_cpu.py and
    tests/test_gpu_dropin.py:
      reference_configs.json        the keys supported_variant reads, of every yaml under the reference's config/
      zfilter_roundtrip.npz         a running_state pickled by the reference's ZFilter (40 rows of x ~ RandomState(1).normal(0.5, 3, (40, 657))
                                    pushed one by one), and the reference's ZFilter applied to x[0] after loading this repo's pickle of the same statistics
      reference_script_imports.json what scripts/train_uhc.py and scripts/eval_uhc.py import from `uhc` / `mujoco_py` when they run with this
                                    repo's package on a machine without a CUDA device (they stop where AgentCopycat asks for one)"""
    import glob
    import json
    import shutil
    import subprocess
    import tempfile
    import yaml
    views = {}
    for f in sorted(glob.glob(os.path.join(H.REF, "config", "**", "*.yml"), recursive=True)):
        d = yaml.safe_load(open(f)) or {}
        views[os.path.relpath(f, os.path.join(H.REF, "config"))] = {k: d[k] for k in SUPPORTED_VARIANT_KEYS if k in d}
    json.dump(views, open(os.path.join(OUT, "reference_configs.json"), "w"), indent=0, sort_keys=True)

    work = tempfile.mkdtemp(prefix="uhc_compat_")
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    run = lambda code, path, cwd=work, **kw: subprocess.run([sys.executable, "-c", f"import sys; sys.path.insert(0, {path!r})\n" + code], cwd=cwd,
                                                           env=dict(env, **kw), check=True)
    xs = "import numpy as np, pickle\nx = np.random.RandomState(1).normal(0.5, 3.0, (40, 657))\n"
    run(xs + "from uhc.khrylib.utils.zfilter import ZFilter\n"
        "pickle.dump({'running_state': ZFilter.from_stats(40, x.mean(0), ((x - x.mean(0)) ** 2).sum(0), clip=5.0)}, open('ours.p', 'wb'))", H.ROOT)
    run(xs + f"from uhc.khrylib.utils import zfilter\nassert zfilter.__file__.startswith({H.REF!r})\n"
        "np.save('y.npy', pickle.load(open('ours.p', 'rb'))['running_state'](x[0], update=False))\n"
        "z = zfilter.ZFilter((657,), clip=5)\nfor r in x: z(r)\npickle.dump({'running_state': z}, open('ref.p', 'wb'))", H.REF)
    np.savez_compressed(os.path.join(OUT, "zfilter_roundtrip.npz"), y_ref_from_ours=np.load(os.path.join(work, "y.npy")),
                        ref_pickle=np.frombuffer(open(os.path.join(work, "ref.p"), "rb").read(), np.uint8))

    sys.path.insert(0, H.ROOT)
    from tests.helpers import write_synthetic_pkl
    for d in ("uhc", "uhc_b200", "mujoco_py"):
        os.symlink(os.path.join(H.ROOT, d), os.path.join(work, d))
    os.makedirs(os.path.join(work, "config"))
    base = yaml.safe_load(open(os.path.join(H.ROOT, "config", "uhc_b200_default.yml")))
    base["data_specs"]["file_path"] = write_synthetic_pkl(os.path.join(work, "sample_data", "clips.pkl"))
    yaml.safe_dump(base, open(os.path.join(work, "config", "refscript.yml"), "w"))
    imports = {}
    for script, argv in (("train_uhc.py", ["--cfg", "refscript", "--no_log"]), ("eval_uhc.py", ["--cfg", "refscript", "--epoch", "2", "--mode", "stats"])):
        path = os.path.join(H.REF, "scripts", script)
        code = (f"import builtins, json, runpy\nrec, imp = [], builtins.__import__\n"
                "def hook(name, g=None, l=None, fromlist=(), level=0):\n"
                f"    if (g or {{}}).get('__file__') == {path!r} and name.split('.')[0] in ('uhc', 'mujoco_py'):\n"
                "        rec.append([name, sorted(fromlist or ())])\n"
                "    return imp(name, g, l, fromlist, level)\n"
                f"builtins.__import__ = hook\nsys.argv = [{path!r}] + {argv!r}\n"
                f"try:\n    runpy.run_path({path!r}, run_name='__main__')\nexcept RuntimeError as e:\n    assert 'needs a CUDA device' in str(e), e\n"
                "json.dump(rec, open('imports.json', 'w'))")
        run(code, work, WANDB_MODE="disabled", CUDA_VISIBLE_DEVICES="")
        imports["scripts/" + script] = json.load(open(os.path.join(work, "imports.json")))
    json.dump(imports, open(os.path.join(OUT, "reference_script_imports.json"), "w"), indent=1)
    shutil.rmtree(work)
    print("compat goldens:", len(views), "configs;", imports)


def main():
    os.makedirs(OUT, exist_ok=True)
    if sys.argv[1:] == ["compat"]:            # needs the reference checkout, not the harness's stubs
        return gen_compat()
    H.install()
    what = sys.argv[1:] or ["math", "env", "ppo"]
    if "math" in what:
        gen_math()
    if "env" in what:
        cfg = H.make_cfg()
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
        gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 60, "zero")
        gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 60, "noise")
        gen_env(cfg, dl, "0-BioMotionLab_NTroje_rub008_0025_kicking1_poses", "kick", 70, 69, "noise")
    if "explicit" in what:       # config/release/uhc_explicit.yml: per-body residual forces through mj_applyFT, world_rfc_explicit reward
        cfg = H.make_cfg("uhc_explicit")
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
        gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 40, "noise", out_tag="sway_explicit", save_expert=False)
    if "implicit" in what:       # config/release/uhc_implicit.yml: obs_v 1 (784 dims, per-body COM blocks, no shape), no meta-PD (75-wide actions), joint gains from the yaml
        cfg = H.make_cfg("uhc_implicit")
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
        gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 40, "noise", out_tag="sway_implicit", save_expert=False)
    if "obsv3" in what:          # config/meta_pd/copycat_35.yml: obs_v 3 = five v2 blocks, ten frames apart (the yaml has no `skip` key) (humanoid_im.py:505-513); relu nets, meta-PD, implicit RFC
        cfg = H.make_cfg("copycat_35")
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
        gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 12, "noise", out_tag="sway_obsv3", save_expert=False)
    if "term" in what:           # cfg.env_term_body "root" / "Head" (humanoid_im.py:1223-1226): the episode fails when the root / the head drops 0.1 m below the clip's lowest
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        for tb in ("root", "Head"):
            cfg = H.make_cfg()
            cfg.env_term_body = tb
            dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
            gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 45, "noise", out_tag="sway_term" + tb.lower(), save_expert=False, term_body=tb)
    if "obsv56" in what:         # obs_v 5 / 6 (get_full_obs_v5 :505-594, get_full_obs_v6 :596-666) on the default implicit-RFC, shape-conditioned configuration
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        for v in (5, 6):
            cfg = H.make_cfg()
            cfg.obs_v = v
            dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
            gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 14, "noise", out_tag=f"sway_obsv{v}", save_expert=False)
    if "rewmul" in what:         # reward_id world_rfc_implicit_v1_mul (reward_function.py:174-250): the five terms of world_rfc_implicit multiplied instead of averaged
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        cfg = H.make_cfg()
        cfg.reward_id = "world_rfc_implicit_v1_mul"
        dl = DatasetAMASSSingle(cfg.data_specs, data_mode="train")
        gen_env(cfg, dl, "0-ACCAD_Male2General_c3d_A2- Sway_poses", "sway", 90, 30, "noise", out_tag="sway_rewmul", save_expert=False, reward_only=True)
    if "reactive" in what:
        cfg = H.make_cfg()
        from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
        gen_reactive(cfg, DatasetAMASSSingle(cfg.data_specs, data_mode="train"))
    if "ppo" in what:
        gen_ppo()
    if "mcp" in what:
        gen_mcp()
    if "ppo_real" in what:
        gen_ppo_real()
    if "metrics" in what:
        gen_metrics()
    if "sampler" in what:
        gen_sampler(H.make_cfg())


if __name__ == "__main__":
    main()
