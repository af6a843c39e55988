"""Batched rollout + PPO driver on the engine (SURVEY.md section 8a rows a11, a15-a17).

Replaces the reference's fork-per-iteration CPU workers (uhc/agents/agent_copycat.py:496-605, khrylib/rl/agents/agent.py:42-126)
by E device-resident environments stepped in lock-step: per control step one obs-normaliser pass, one policy forward
(tensor cores), one Gaussian sample, one fused physics/task kernel, and the transition lands in a time-major [T][E] buffer
in HBM.  Episode semantics follow Appendix C of SURVEY.md: an env that fails or reaches the end of its clip slice gets
mask 0 and is re-seeded with a freshly sampled (clip, start) slice (dataset_amass_single.py:172-253); rollouts cut mid-episode
are bootstrapped with V(s_T) (the reference never truncates, so this is the one semantic addition, documented in DESIGN.md).
Multi-GPU: envs are sharded, one process per GPU; the flat gradient tensor of each net is all-reduced once per optimisation step
(nn.GradComm, overlapped with the other net's backward); nothing else crosses GPUs.
"""
import ctypes as C
import time

import numpy as np

from . import nn
from .engine import Engine


class UhcRolloutBuf(C.Structure):
    """include/uhc_rollout.h UhcRolloutBuf"""
    _fields_ = [(k, C.c_void_p) for k in ("states", "actions", "rewards", "masks", "exps", "logp", "fails", "obs_cur", "ep_clip", "ep_pct")] + \
               [("T_cap", C.c_int), ("reserved", C.c_int)]


class UhcEvalBuf(C.Structure):
    """include/uhc_eval.h UhcEvalBuf"""
    _fields_ = [(k, C.c_void_p) for k in ("frame_off", "pred_qpos", "pred_jpos", "frame_t", "frame_metrics", "nframes", "last_t", "fail_any", "reward_sum",
                                         "clip_metrics")] + [("frame_cap", C.c_int), ("reserved", C.c_int)]


EVAL_METRICS = ("root_dist", "mpjpe", "mpjpe_g", "pa_mpjpe", "vel_dist", "accel_dist")      # frame_metrics / clip_metrics columns


def ewma(x, alpha=0.05):
    """uhc/utils/math_utils.py:25-29"""
    avg = float(x[0])
    for i in x[1:]:
        avg = alpha * float(i) + (1 - alpha) * avg
    return avg


def failure_weights(success_hist, sampling_temp=0.2, sampling_freq=0.5):
    """Per-clip sampling weights of the training loop (DatasetAMASSSingle.sample_seq with freq_dict, dataset_amass_single.py:183-186):
    with probability sampling_freq the clip is drawn from p ~ exp(-ewma(success history) / temp) (0 for an empty history), else
    uniformly over the clips.  success_hist: one list of 0/1 outcomes per clip (freq_dict[k][:, 0] == 1).  Returns the mixture
    weights w = sampling_freq * p + (1 - sampling_freq) / C for uhc_set_clip_weights."""
    s = np.array([ewma(np.asarray(h, dtype=np.float64) == 1) if len(h) > 0 else 0.0 for h in success_hist])
    p = np.exp(-s / sampling_temp)
    p = p / p.sum()
    return (sampling_freq * p + (1.0 - sampling_freq) / len(p)).astype(np.float32)


class ClipSampler:
    """DatasetAMASSSingle.sample_seq / get_sample_from_key (dataset_amass_single.py:172-253): uniform clip choice (or
    failure-weighted when freq stats are given), start ~ U[0, len - t_min), slice length min(t_max, len - start)."""

    def __init__(self, clip_lens, t_min=5, t_max=300, seed=0):
        self.lens, self.t_min, self.t_max = np.asarray(clip_lens), t_min, t_max
        self.rng = np.random.RandomState(seed)
        self.probs = None

    def set_failure_weights(self, success_ewma, temp=0.1):
        p = np.exp(-np.asarray(success_ewma) / temp)
        self.probs = p / p.sum()

    def sample(self, n, freq=0.5):
        if self.probs is not None:
            pick_w = self.rng.binomial(1, freq, n).astype(bool)
            clip = np.where(pick_w, self.rng.choice(len(self.lens), n, p=self.probs), self.rng.randint(0, len(self.lens), n))
        else:
            clip = self.rng.randint(0, len(self.lens), n)
        L = self.lens[clip]
        start = (self.rng.random_sample(n) * np.maximum(L - self.t_min, 1)).astype(np.int64)
        length = np.minimum(self.t_max if self.t_max > 0 else L, L - start)
        return clip.astype(np.int32), start.astype(np.int32), length.astype(np.int32)


class RolloutBuffer:
    def __init__(self, T, E, device, act_dim=105, obs_dim=657):
        import torch
        f = dict(device=device, dtype=torch.float32)
        self.T, self.E = T, E
        self.states = torch.empty(T, E, obs_dim, **f)
        self.actions = torch.empty(T, E, act_dim, **f)
        self.rewards, self.masks, self.exps, self.logp = (torch.empty(T, E, **f) for _ in range(4))
        self.last_obs = torch.empty(E, obs_dim, **f)
        self.last_alive = torch.empty(E, **f)
        self.fails = torch.zeros(T, E, device=device, dtype=torch.int32)
        self.ep_clip = torch.full((T, E), -1, device=device, dtype=torch.int32)      # clip of the episode that ended at (t, e), -1 = none
        self.ep_pct = torch.zeros(T, E, **f)                                         # its completed fraction (info["percent"])

    def c_struct(self, obs_cur):
        b = UhcRolloutBuf()
        for k in ("states", "actions", "rewards", "masks", "exps", "logp", "fails", "ep_clip", "ep_pct"):
            setattr(b, k, getattr(self, k).data_ptr())
        b.obs_cur, b.T_cap = obs_cur.data_ptr(), self.T
        return b

    # TrajBatch-compatible flat views (khrylib/rl/core/trajbatch.py)
    def flat(self, name):
        t = getattr(self, name)
        return t.reshape(self.T * self.E, *t.shape[2:])


class BatchedAgent:
    def __init__(self, num_envs, clips, shapes=None, device=0, seed=1, precision=32, policy_hsize=(2048, 1024, 512),
                 value_hsize=(2048, 1024, 512), htype="gelu", log_std=-2.3, policy_lr=5e-5, value_lr=3e-4, gamma=0.95, tau=0.95,
                 clip_epsilon=0.2, num_optim_epoch=10, grad_clip=40.0, t_min=5, t_max=300, noise_rate=1.0, rank=0, world=1,
                 grad_sync=None, model=None, update_tc=True, variants=None, clip_models=None, c_update=True, actor_type="gauss", num_primitive=8,
                 composer_dim=(300, 200), **env_cfg):
        import torch
        self.torch = torch
        self.dev = torch.device("cuda", device)
        torch.cuda.set_device(self.dev)
        self.E, self.seed, self.rank, self.world = num_envs, seed, rank, world
        self.auto_reset = bool(env_cfg.pop("auto_reset", True))
        self.engine = Engine(num_envs, model=model, device=device, precision=precision, variants=variants, auto_reset=int(self.auto_reset), t_min=t_min, t_max=t_max,
                             reset_seed=seed * 7919 + rank * 104729 + 1, **env_cfg)
        # clips: expert dicts (host motion library) or {"pose_aa": [...], "trans": [...]} raw SMPL sequences whose tables are built on the device;
        # clip_models: body-shape variant per clip (the reference rebuilds the robot per clip)
        if isinstance(clips, dict):
            self.engine.load_smpl_clips(clips["pose_aa"], clips.get("trans"), shapes, clip_models)
        else:
            self.engine.load_clips(clips, shapes, clip_models)
        self.sampler = ClipSampler(self.engine.clip_len, t_min, t_max, seed=seed * 9973 + rank)
        A = self.act_dim = self.engine.act_dim          # env.action_dim (humanoid_im.py:250): 69 + (6 | 216) + (30 if meta_pd)
        D = self.obs_dim = self.engine.obs_dim          # env.obs_dim: 657 (obs v2) or 784 (obs v1)
        assert actor_type in ("gauss", "mcp"), "actor_type: gauss (PolicyGaussian) | mcp (PolicyMCP)"
        self.actor_type = actor_type
        if actor_type == "mcp":        # policy_mcp.py:9-37 (config/release/uhc_implicit.yml): runs through uhc_rollout_mcp / uhc_ppo_trainer_create_mcp only
            assert c_update and update_tc and bool(env_cfg.get("auto_reset", True)), "the PolicyMCP actor runs on the C-side rollout / update paths"
            self.policy = nn.MCPNet(D, policy_hsize, A, htype, num_primitive=num_primitive, composer_dim=composer_dim, device=self.dev, seed=seed)
        else:
            self.policy = nn.MLPNet(D, policy_hsize, A, htype, device=self.dev, head_name="action_mean", seed=seed)
        self.value = nn.MLPNet(D, value_hsize, 1, htype, device=self.dev, head_name="value_head", seed=seed + 1)
        self.log_std = torch.full((A,), float(log_std), device=self.dev, dtype=torch.float32)
        self.running_state = nn.ZFilter(D, clip=5.0, device=self.dev)
        self.opt_p, self.opt_v = nn.Adam(self.policy.params(), policy_lr, net=self.policy), nn.Adam(self.value.params(), value_lr, net=self.value)
        self.comm = nn.GradComm(world)
        self.gamma, self.tau, self.clip_epsilon, self.epochs, self.grad_clip = gamma, tau, clip_epsilon, num_optim_epoch, grad_clip
        self.noise_rate, self.grad_sync, self.update_tc = noise_rate, grad_sync, update_tc
        self.c_update, self._ctrainer, self._nccl = c_update, None, None      # uhc_ppo_update (include/uhc_ppo.h): the update behind one C-ABI call
        self.global_step = 0
        self.obs = None
        self.ep_len = torch.zeros(num_envs, device=self.dev, dtype=torch.float32)
        self.ep_ret = torch.zeros(num_envs, device=self.dev, dtype=torch.float32)
        self.nn_launches = 0
        self._notdone = torch.zeros(num_envs, device=self.dev, dtype=torch.bool)

    # ---- env.reset for a subset with freshly sampled clip slices
    def reset_envs(self, ids=None):
        ids = np.arange(self.E, dtype=np.int32) if ids is None else np.asarray(ids, dtype=np.int32)
        clip, start, length = self.sampler.sample(len(ids))
        self.obs = self.engine.reset(ids, clip, start, length)
        return self.obs

    def policy_step(self, obs, update_filter=True, mean_action=None, use_tc=True, out_state=None, out_action=None, out_logp=None):
        """running_state -> policy -> sample.  Returns (normalised state, action, logp); the out_* tensors (rows of the rollout
        buffer) are written in place by the kernels."""
        s = self.running_state(obs, update=update_filter, out=out_state)
        mean = self.policy.forward_tc(s) if use_tc else self.policy.forward(s)
        a, lp = nn.gaussian_sample(mean, self.log_std, self.seed * 1000003 + self.rank, self.global_step, mean_action, out_action, out_logp)
        self.nn_launches += (3 if update_filter else 1) + (1 + len(self.policy.W) if use_tc else len(self.policy.W)) + 1
        return s, a, lp

    def step_once(self, buf, k, use_tc=True):
        """one lock-step control step of every env: normalise, policy, sample, physics+task kernel, buffer write, re-seed ended episodes."""
        t = self.torch
        mean_action = None
        if self.noise_rate < 1.0:
            mean_action = (t.rand(self.E, device=self.dev, dtype=t.float32) < (1.0 - self.noise_rate)).to(t.uint8)
        s, a, lp = self.policy_step(self.obs, True, mean_action, use_tc, buf.states[k], buf.actions[k], buf.logp[k])
        if mean_action is not None:
            buf.exps[k].copy_(1.0 - mean_action.float())
        elif not getattr(buf, "_exps_ones", False):
            buf.exps.fill_(1.0)
            buf._exps_ones = True
        obs, rew, cinfo, fail, end, pct = self.engine.step(a, reward_out=buf.rewards[k])
        done = (fail | end) != 0
        t.logical_not(done, out=self._notdone)
        buf.masks[k].copy_(self._notdone)
        self.global_step += 1
        buf.fails[k].copy_(fail)
        if self.auto_reset:
            return            # finished episodes were re-seeded inside the step kernel (no host round trip)
        ids = done.nonzero().flatten()
        if ids.numel():
            self.reset_envs(ids.cpu().numpy().astype(np.int32))

    def rollout(self, buf, T, row0=0, use_graph=True):
        """T control steps through the C-side loop (uhc_rollout, include/uhc_rollout.h): the same kernels as step_once, enqueued from C and
        replayed as one CUDA graph.  Needs auto_reset (finished episodes are re-seeded inside the step kernel)."""
        assert self.auto_reset, "uhc_rollout re-seeds finished episodes in the step kernel: build the agent with auto_reset=True"
        L = self.engine.lib
        if not getattr(self, "_ro_ready", False):
            L.uhc_rollout_last_error.restype = C.c_char_p
            self._ro_ready = True
        mcp = self.actor_type == "mcp"
        self._policy_struct()
        if getattr(self, "_ro_step", None) != self.global_step:
            L.uhc_rollout_set_step(self.engine.h, C.c_ulonglong(self.global_step))
        bs = buf.c_struct(self.obs)
        st = C.c_void_p(self.torch.cuda.current_stream(self.dev).cuda_stream)
        rc = (L.uhc_rollout_mcp if mcp else L.uhc_rollout)(self.engine.h, C.c_int(T), C.c_int(row0), C.byref(self._mlp_c), C.c_void_p(self.log_std.data_ptr()),
                           C.c_void_p(self.running_state.stats.data_ptr()), C.c_float(self.running_state.clip), C.c_int(1),
                           C.c_ulonglong(self.seed * 1000003 + self.rank), C.c_float(self.noise_rate), C.byref(bs), C.c_int(int(use_graph)), st)
        if rc != 0:
            raise RuntimeError("uhc_rollout: " + L.uhc_rollout_last_error().decode())
        self.global_step += T
        self._ro_step = self.global_step
        self.nn_launches += T * (L.uhc_rollout_launches_per_step(self.engine.h) - 1)      # the env-step launch is counted by the engine

    def _policy_struct(self):
        if self.policy._bf16 is None or getattr(self, "_mlp_c", None) is None:
            self._mlp_c = nn.mcp_struct(self.policy) if self.actor_type == "mcp" else nn.mlp_struct(self.policy)
        return self._mlp_c

    def evaluate(self, clip0, n, fail_safe, trajectories=False):
        """Deterministic evaluation of clips [clip0, clip0 + n) of the loaded table from frame 0 (uhc_evaluate, include/uhc_eval.h): a device
        work queue of clips over the env slots, fail_safe re-seating inside the step kernel, metrics on the device.  Uses the env records (the
        next sample() must reset them: set self.obs = None).  Returns numpy arrays per clip: nframes, last_t, fail_any, reward_sum,
        clip_metrics [n][6] (columns EVAL_METRICS, mm), frame_metrics (list of [nframes][6]), steps (control steps run); with trajectories
        also pred_qpos / pred_jpos / frame_t (lists of [nframes][...])."""
        t = self.torch
        L = self.engine.lib
        if not getattr(self, "_ev_ready", False):
            L.uhc_eval_last_error.restype = C.c_char_p
            self._ev_ready = True
        clip0, n = int(clip0), int(n)
        lens = np.asarray(self.engine.clip_len[max(clip0, 0):max(clip0 + n, 0)], np.int64)
        rows = np.maximum(lens - 1 + max(int(self.engine._cfg.trail_steps), 0), 0)
        off = np.zeros(max(n, 0) + 1, np.int32)
        off[1:len(rows) + 1] = np.cumsum(rows)
        off[len(rows) + 1:] = off[len(rows)]
        F, nn_ = max(int(off[-1]), 1), max(n, 1)
        d, i32, f64 = self.dev, t.int32, t.float64
        o = dict(frame_off=t.as_tensor(off, device=d), pred_qpos=t.empty(F, 76, device=d, dtype=t.float32), pred_jpos=t.empty(F, 72, device=d, dtype=t.float32), frame_t=t.empty(F, device=d, dtype=i32),
                 frame_metrics=t.empty(F, 6, device=d, dtype=f64), nframes=t.empty(nn_, device=d, dtype=i32), last_t=t.empty(nn_, device=d, dtype=i32),
                 fail_any=t.empty(nn_, device=d, dtype=i32), reward_sum=t.empty(nn_, device=d, dtype=f64), clip_metrics=t.empty(nn_, 6, device=d, dtype=f64))
        b = UhcEvalBuf()
        for k, v in o.items():
            setattr(b, k, v.data_ptr())
        b.frame_cap = int(off[-1])
        st = C.c_void_p(t.cuda.current_stream(self.dev).cuda_stream)
        fn = L.uhc_evaluate_mcp if self.actor_type == "mcp" else L.uhc_evaluate
        rc = fn(self.engine.h, C.c_int(clip0), C.c_int(n), C.byref(self._policy_struct()), C.c_void_p(self.log_std.data_ptr()),
                C.c_void_p(self.running_state.stats.data_ptr()), C.c_float(self.running_state.clip), C.c_int(int(bool(fail_safe))), C.byref(b), st)
        if rc != 0:
            raise RuntimeError("uhc_evaluate: " + L.uhc_eval_last_error().decode())
        steps = C.c_longlong(0)
        L.uhc_eval_last_steps(self.engine.h, C.byref(steps))
        h = {k: v.cpu().numpy() for k, v in o.items() if trajectories or k not in ("pred_qpos", "pred_jpos", "frame_t")}
        nf = h["nframes"][:n]
        out = dict(nframes=nf, last_t=h["last_t"][:n], fail_any=h["fail_any"][:n] != 0, reward_sum=h["reward_sum"][:n], clip_metrics=h["clip_metrics"][:n],
                   steps=int(steps.value))
        for k in ("frame_metrics",) + (("pred_qpos", "pred_jpos", "frame_t") if trajectories else ()):
            out[k] = [h[k][off[i]:off[i] + nf[i]] for i in range(n)]
        return out

    def sample(self, T, buf=None, use_tc=True, c_loop=None):
        """agent.sample(): T lock-step control steps of all envs.  Returns (buffer, log).  c_loop (default: whenever auto_reset is on):
        the loop runs behind the C ABI as one CUDA graph; otherwise the Python loop over step_once (identical kernels and results)."""
        t = self.torch
        if self.obs is None:
            self.reset_envs()
        buf = buf or RolloutBuffer(T, self.E, self.dev, self.act_dim, self.obs_dim)
        t0 = time.time()
        len0, ret0 = self.ep_len.clone(), self.ep_ret.clone()
        if c_loop is None:
            c_loop = self.auto_reset and use_tc
        if c_loop:
            self.rollout(buf, T)
        else:
            for k in range(T):
                self.step_once(buf, k, use_tc)
        buf.last_obs.copy_(self.obs)
        # episode statistics from the buffer (one sync at the end of the rollout): segment the [T][E] masks per env
        m, r = buf.masks[:T], buf.rewards[:T]
        done = m == 0
        n_eps = int(done.sum())
        run_len = t.zeros(self.E, device=self.dev, dtype=t.float32); run_ret = t.zeros(self.E, device=self.dev, dtype=t.float32)
        run_len += len0; run_ret += ret0
        tot_len = t.zeros((), device=self.dev, dtype=t.float32); tot_ret = t.zeros((), device=self.dev, dtype=t.float32)
        for k in range(T):
            run_len += 1; run_ret += r[k]
            d = done[k]
            tot_len += (run_len * d).sum(); tot_ret += (run_ret * d).sum()
            run_len *= ~d; run_ret *= ~d
        self.ep_len, self.ep_ret = run_len, run_ret
        n_fail = int(((buf.fails[:T] != 0) & done).sum())
        log = dict(num_steps=T * self.E, num_episodes=n_eps, avg_episode_len=float(tot_len) / max(n_eps, 1),
                   avg_episode_reward=float(tot_ret) / max(n_eps, 1), fail_rate=n_fail / max(n_eps, 1),
                   avg_reward=float(r.mean()), sample_time=time.time() - t0)
        return buf, log

    def update_params(self, buf):
        """AgentPG.update_params (agent_pg.py:39-56): V(s), GAE (+bootstrap), advantage normalisation, PPO epochs -- all on the
        tensor-core path.  Multi-GPU (envs sharded by rank): the ONLY collective is the all-reduce of the flat gradient tensors; the
        global-batch statistics the reference's full-batch semantics need (advantage sum / sum of squares / count, the number of
        selected rows, the ZFilter increments of every rank) ride in the tail of the first one (SURVEY.md section 8e)."""
        t = self.torch
        L = nn._lib()
        ev = [t.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        T, E = buf.T, buf.E
        N = T * E
        states = buf.flat("states")
        if not self.update_tc:               # fp32 SIMT parity path (single GPU)
            t0 = time.time()
            values = self.value.forward(states).reshape(T, E)
            last_v = self.value.forward(self.running_state(buf.last_obs, update=False)).reshape(E)
            adv, ret = nn.gae(buf.rewards, buf.masks, values, last_v, self.gamma, self.tau, normalize=True)
            losses = nn.ppo_update(self.policy, self.value, self.log_std, self.opt_p, self.opt_v, states, buf.flat("actions"), ret.reshape(-1),
                                   adv.reshape(-1), buf.flat("exps"), self.clip_epsilon, self.epochs, self.grad_clip, use_tc=False)
            t.cuda.synchronize()
            self._mlp_c = None
            return dict(update_time=time.time() - t0, surr_loss=float(losses[0]), value_loss=float(losses[1]))
        if self.c_update:
            return self._update_params_c(buf, ev)
        tp = getattr(self.policy, "_tc_trainer", None) or nn.TCTrainer(self.policy)
        tv = getattr(self.value, "_tc_trainer", None) or nn.TCTrainer(self.value)
        self.policy._tc_trainer, self.value._tc_trainer = tp, tv
        xb, xT = tp.prepare_input(states)
        tv.cache["xb"], tv.cache["xT"] = xb, xT
        v0, ctx0 = tv.forward(xb)                                                   # V(s): GAE input and epoch 0's value forward
        last_v = self.value.forward_tc(self.running_state(buf.last_obs, update=False)).reshape(E)
        adv, ret = nn.gae(buf.rewards, buf.masks, v0.reshape(T, E), last_v, self.gamma, self.tau, normalize=False)
        adv, ret, exps = adv.reshape(-1), ret.reshape(-1), buf.flat("exps")
        mom = t.zeros(2, device=self.dev, dtype=t.float64)
        nn._chk(L.uhc_adv_moments(nn._p(adv), C.c_long(N), nn._p(mom), nn._stream(adv)))
        cnt = (exps != 0).sum().to(t.float64).reshape(1)
        inv_count = t.zeros(1, device=self.dev, dtype=t.float32)
        after = None
        if self.world <= 1:
            nn._chk(L.uhc_adv_normalize(nn._p(adv), C.c_long(N), nn._p(mom), None, nn._stream(adv)))
            inv_count.copy_(1.0 / t.clamp(cnt, min=1.0))
        else:
            D = self.obs_dim
            zs = self.running_state.stats
            if getattr(self, "_z_sync", None) is None:                               # fresh agent: every rank starts from empty statistics
                self._z_sync = t.zeros_like(zs)                                      # additive form of the statistics every rank agreed on last
            d = t.cat([mom, t.full((1,), float(N), device=self.dev, dtype=t.float64), cnt, nn.zfilter_to_sums(zs, D) - self._z_sync])
            planes = nn.split_double(d)                                              # [5, nd] exact fixed-point digits (fp32)
            tail = self.value.gfull[self.value.nflat:]
            tail.zero_()
            nd = d.numel()
            assert planes.numel() <= tail.numel()
            tail[:planes.numel()].copy_(planes.reshape(-1))
            ntot = t.zeros(1, device=self.dev, dtype=t.float64)

            def after(tail_r):
                g = nn.join_double(tail_r[:nn.SPLIT_CHUNKS * nd].reshape(nn.SPLIT_CHUNKS, nd))   # summed over the ranks by the gradient all-reduce
                ntot.copy_(g[2:3])
                gm = g[0:2].contiguous()
                nn._chk(L.uhc_adv_normalize(nn._p(adv), C.c_long(N), nn._p(gm), nn._p(ntot), nn._stream(adv)))
                inv_count.copy_(1.0 / t.clamp(g[3:4], min=1.0))
                self._z_sync = self._z_sync + g[4:]
                zs.copy_(nn.zfilter_from_sums(self._z_sync, D))                     # every rank now holds the same running_state
        ev[1].record()
        losses = nn.ppo_epochs_tc(self.policy, self.value, self.log_std, self.opt_p, self.opt_v, xb, xT, buf.flat("actions"), ret, adv, exps,
                                  self.clip_epsilon, self.epochs, self.grad_clip, comm=self.comm, first_value=(v0, ctx0), after_first_reduce=after,
                                  inv_count_dev=inv_count, world=self.world)
        ev[2].record()
        t.cuda.synchronize()
        self._mlp_c = None
        out = dict(update_time=1e-3 * ev[0].elapsed_time(ev[2]), gae_ms=ev[0].elapsed_time(ev[1]), epochs_ms=ev[1].elapsed_time(ev[2]),
                   surr_loss=float(losses[0]), value_loss=float(losses[1]))
        if self.world > 1:
            out.update(allreduce_ms=self.comm.pop_ms(), allreduce_bytes=self.comm.bytes, allreduce_calls=self.comm.calls)
            self.comm.bytes = self.comm.calls = 0
        return out

    def _update_params_c(self, buf, ev):
        """the production update: ONE call of uhc_ppo_update (include/uhc_ppo.h) -- V(s) and V(s_T), GAE, global advantage normalisation, the
        epochs of both nets, Adam, and (world > 1) the gradient all-reduces on this job's ncclComm_t with the statistics tail."""
        t = self.torch
        T, E = buf.T, buf.E
        if self._ctrainer is None or self._ctrainer.max_rows < T * E or self._ctrainer.max_envs < E:
            if self._ctrainer is not None:
                self._ctrainer.close()
            self._ctrainer = nn.CPpoTrainer(self.policy, self.value, self.opt_p, self.opt_v, T * E, E, self.dev)
        zs = zsync = None
        if self.world > 1:
            if self._nccl is None:
                self._nccl = nn.make_nccl_comm(self.rank, self.world, self.dev)
            zs = self.running_state.stats
            if getattr(self, "_z_sync", None) is None:
                self._z_sync = t.zeros_like(zs)
            zsync = self._z_sync
        last_s = self.running_state(buf.last_obs, update=False)
        if getattr(self, "_losses", None) is None:
            self._losses = t.zeros(2, device=self.dev, dtype=t.float32)
        ev[1].record()
        self._ctrainer.update(buf.flat("states"), last_s, buf.flat("actions"), buf.rewards, buf.masks, buf.flat("exps"), self.log_std, T, E, self.gamma,
                              self.tau, self.clip_epsilon, self.epochs, self.grad_clip, self._losses, zfilter=zs, z_sync=zsync, comm=self._nccl, world=self.world)
        ev[2].record()
        t.cuda.synchronize()
        out = dict(update_time=1e-3 * ev[0].elapsed_time(ev[2]), gae_ms=0.0, epochs_ms=ev[1].elapsed_time(ev[2]),      # GAE runs inside the call
                   surr_loss=float(self._losses[0]), value_loss=float(self._losses[1]))
        if self.world > 1:
            ms, by, calls = self._ctrainer.comm_stats()
            out.update(allreduce_ms=ms, allreduce_bytes=by, allreduce_calls=calls)
        return out

    def optimize_policy(self, T):
        buf, log = self.sample(T)
        log.update(self.update_params(buf))
        return log

    # checkpoint in the reference's wire format (agent_copycat.py:190-201): policy_dict / value_dict / running_state
    def state_dicts(self):
        pd = self.policy.state_dict()
        pd["action_log_std"] = self.log_std.detach().cpu().reshape(1, -1)
        # `running_state` in the reference's wire format: a ZFilter object (agent_copycat.py:194-200 pickles the object itself and
        # load_checkpoint assigns it back, :249-260), filled from the device statistics
        from uhc.khrylib.utils.zfilter import ZFilter as HostZFilter
        st = self.running_state.stats.cpu().numpy()
        D = self.running_state.dim
        return {"policy_dict": pd, "value_dict": self.value.state_dict(),
                "running_state": HostZFilter.from_stats(st[0], st[1:1 + D], st[1 + D:], clip=self.running_state.clip)}

    def load_state_dicts(self, cp):
        t = self.torch
        self.policy.load_state_dict(cp["policy_dict"])
        self.value.load_state_dict(cp["value_dict"])
        if "action_log_std" in cp["policy_dict"]:
            self.log_std.copy_(t.as_tensor(np.asarray(cp["policy_dict"]["action_log_std"]), dtype=t.float32).reshape(-1))
        rs = cp.get("running_state")
        if rs is not None:
            if isinstance(rs, dict):          # round-1 checkpoints of this repo
                self.running_state.load(rs["n"], rs["mean"], rs["std"])
            else:                             # a pickled khrylib ZFilter (reference checkpoints and this repo's)
                self.running_state.load_sums(rs.rs._n, rs.rs._M, rs.rs._S)
            # a loaded normaliser is common to every rank: the cross-rank merge (update_params) only exchanges what is added from here on
            self._z_sync = nn.zfilter_to_sums(self.running_state.stats, self.running_state.dim).clone()


def make_nccl_grad_sync(world):
    """flatten -> one torch.distributed all_reduce(sum) -> unflatten, averaged over ranks (full-batch mean semantics)."""
    import torch
    import torch.distributed as dist

    def sync(grads):
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat.div_(world)
        out, o = [], 0
        for g in grads:
            n = g.numel()
            out.append(flat[o:o + n].view_as(g))
            o += n
        return out
    return sync
