"""AgentCopycat with the reference's surface (uhc/agents/agent_copycat.py:51-605) on the batched B200 engine.

  AgentCopycat(cfg, dtype, device, training=True, checkpoint_epoch=0)
  .optimize_policy(epoch)   per_epoch_update -> sample -> update_params -> checkpoint / eval every save_n_epochs -> log   (:326-352)
  .sample(min_batch_size)   -> (batch, log)      batch: states / actions / masks / rewards / exps (device resident, numpy on demand)
  .update_params(batch)     GAE + PPO epochs (khrylib agent_pg.py:39-56, agent_ppo.py:16-51)
  .eval_policy(epoch, dump) deterministic roll-out of every clip on the device (uhc_evaluate), coverage / error statistics (:354-494)
  .save_checkpoint / .load_checkpoint   pickle {"policy_dict", "value_dict", "running_state"} at models/iter_%04d.p        (:190-260)

Differences that are inherent to the batched design are listed in DESIGN.md (lock-step horizon with value bootstrap, batched
ZFilter merge, clip sampling without the per-clip failure history unless eval statistics are available).
"""
import logging
import math
import os
import os.path as osp
import pickle
import time
from collections import defaultdict

import joblib
import numpy as np

from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
from uhc.envs.humanoid_im import HumanoidEnv
from uhc.losses.reward_function import reward_func
from uhc_b200.agent import BatchedAgent, RolloutBuffer, make_nccl_grad_sync
from uhc_b200.model import HumanoidModel


class _Batch:
    """TrajBatch-compatible view (khrylib/rl/core/trajbatch.py:4-15) over the device rollout buffer."""

    def __init__(self, buf):
        self.buf = buf

    def __getattr__(self, name):
        if name in ("states", "actions", "rewards", "masks", "exps"):
            return self.buf.flat(name).cpu().numpy()
        raise AttributeError(name)


class _Log(dict):
    __getattr__ = dict.get


def supported_variant(cfg):
    """The reference configuration keys this engine implements; returns the residual-force mode ("implicit" | "explicit" | "none").  `cfg` needs `.get(key, default)`
    and the attributes obs_v, actor_type, reward_id, fix_std, residual_force (uhc/utils/config_utils/copycat_config.py).  Everything else raises an AssertionError
    naming the key: of the reference's 115 yaml files 86 pass (tests/test_shim_cpu.py counts them); the others use explicit residual forces with contact gating /
    projection / body subsets (10), the six-term world_rfc_implicit_v2 / _v3 rewards (8), obs_v 0 / 4 (6), a trained log_std (2), ..."""
    assert cfg.obs_v in (1, 2, 3, 5, 6) and cfg.actor_type in ("gauss", "mcp") and cfg.reward_id in reward_func, \
        "the B200 engine implements obs_v 1 | 2 | 3 | 5 | 6, the gauss and mcp actors, world_rfc_implicit (_v1_mul) / world_rfc_explicit (obs_v 0/4, reward v2/v3: SURVEY.md section 8f, next)"
    assert cfg.get("obs_vel", "full") == "full" and cfg.get("obs_coord", "root") == "root" and not cfg.get("obs_phase", False), "obs_vel full / obs_coord root / no phase only"
    if cfg.obs_v == 1:
        assert not cfg.get("has_shape", False), "obs_v 1 carries no shape vector (has_shape: false in config/release/uhc_implicit.yml)"
    # variants the batched engine does not implement must not be accepted silently (ADVICE r1)
    assert cfg.fix_std, "log_std is not a trained parameter in this engine (fix_std: true in every released config)"
    assert cfg.get("env_term_body", "body") in ("body", "root", "Head"), "env_term_body: 'body' (calc_body_diff), 'root' or 'Head' (humanoid_im.py:1223-1229)"
    rfc_mode = cfg.get("residual_force_mode", "implicit") if cfg.residual_force else "none"     # residual_force: false -> no residual-force dims (humanoid_im.py:231-243)
    assert rfc_mode in ("implicit", "explicit", "none"), "residual_force_mode: implicit | explicit"
    if rfc_mode == "explicit":      # the kernel restates the release settings of the explicit mode (config/release/uhc_explicit.yml)
        assert cfg.get("residual_force_bodies", "all") == "all" and cfg.get("residual_force_torque", True) and int(cfg.get("residual_force_bodies_num", 1)) == 1 \
            and not cfg.get("residual_contact_only", False) and not cfg.get("residual_contact_projection", False), \
            "explicit residual force: only residual_force_bodies = all, one point per body, torque on, no contact gating / projection"
    # the fused reward follows the residual-force mode (world_rfc_implicit :12-88 / world_rfc_explicit :253-341), as the released configs pair them
    assert cfg.reward_id in (("world_rfc_explicit",) if rfc_mode == "explicit" else ("world_rfc_implicit", "world_rfc_implicit_v1_mul")), "reward_id must match residual_force_mode"
    assert float(cfg.get("env_init_noise", 0.0)) == 0.0, "env_init_noise > 0 is not implemented"
    return rfc_mode


class AgentCopycat:
    def __init__(self, cfg, dtype, device, training=True, checkpoint_epoch=0):
        import torch
        self.cfg = self.cc_cfg = cfg
        self.dtype, self.device, self.training = dtype, device, training
        self.epoch, self.max_freq = 0, 50
        dev_index = device.index if getattr(device, "type", "cpu") == "cuda" and device.index is not None else int(getattr(cfg, "gpu_index", 0) or 0)
        if not torch.cuda.is_available():
            raise RuntimeError("the B200 engine needs a CUDA device (the reference's CPU sampling path is replaced, not kept as a fallback)")
        self.model_tables = HumanoidModel()
        # extra key motion_lib: "host" (expert tables from uhc_b200.motion_lib, packed and uploaded) | "device" (built on the GPU from the
        # raw SMPL sequences, Engine.load_smpl_clips)
        self.motion_lib = str(cfg.get("motion_lib", "host"))
        assert self.motion_lib in ("host", "device"), "motion_lib: host | device"
        # data (setup_data_loader :128-134)
        self.data_loader = DatasetAMASSSingle(cfg.data_specs, data_mode="train", model=self.model_tables, motion_lib=self.motion_lib)
        self.test_data_loaders = [self.data_loader]
        if len(cfg.data_specs.get("test_file_path", [])) > 0:
            self.test_data_loaders.append(DatasetAMASSSingle(cfg.data_specs, data_mode="test", model=self.model_tables, motion_lib=self.motion_lib))
        self.freq_dict = {k: [] for k in self.data_loader.data_keys}
        rw = cfg.reward_weights or {}
        w = [rw.get(k, d) for k, d in (("w_p", 0.6), ("w_v", 0.1), ("w_e", 0.2), ("w_c", 0.1), ("w_vf", 0.0))]
        kk = [rw.get(k, d) for k, d in (("k_p", 2), ("k_v", 0.005), ("k_e", 20), ("k_c", 1000), ("k_vf", 1))]
        self.num_envs = int(cfg.get("num_envs", 4096))
        self.horizon = max(2, int(math.ceil(cfg.min_batch_size / self.num_envs)))
        world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
        sync = None
        if world > 1:
            import torch.distributed as dist
            if not dist.is_initialized():
                dist.init_process_group("nccl")
            sync = make_nccl_grad_sync(world)
        rfc_mode = supported_variant(cfg)       # refuses (AssertionError) what the batched engine does not implement instead of accepting it silently (ADVICE r1)
        self.agent = BatchedAgent(
            self.num_envs, self.data_loader.smpl_clips() if self.motion_lib == "device" else self.data_loader.experts, self.data_loader.shapes, device=dev_index, seed=cfg.seed, policy_hsize=cfg.policy_hsize,
            value_hsize=cfg.value_hsize, htype=cfg.policy_htype, log_std=cfg.log_std, policy_lr=cfg.policy_lr, value_lr=cfg.value_lr,
            gamma=cfg.gamma, tau=cfg.tau, clip_epsilon=cfg.clip_epsilon, num_optim_epoch=cfg.num_optim_epoch, grad_clip=40.0,
            t_min=cfg.data_specs.get("t_min", 90), t_max=cfg.data_specs.get("t_max", -1), rank=rank, world=world, grad_sync=sync,
            model=self.model_tables, base_rot=cfg.data_specs.get("base_rot", [0.7071, 0.7071, 0.0, 0.0]), rfc_scale=cfg.residual_force_scale,
            rfc_lim=cfg.residual_force_lim, rfc_rate=0.0 if cfg.rfc_decay else 1.0, body_diff_thresh=cfg.get("body_diff_thresh", 0.5),
            meta_pd=int(cfg.meta_pd), env_episode_len=cfg.env_episode_len, trail_steps=cfg.env_expert_trail_steps, w=w, k=kk, rfc_mode=rfc_mode,
            obs_v=int(cfg.obs_v), fut_frames=int(cfg.get("fut_frames", 10)), fut_skip=int(cfg.get("skip", 10)),
            has_shape=bool(cfg.get("has_shape", False)) and bool(cfg.get("has_shape_obs", True)), actor_type=cfg.actor_type, num_primitive=int(cfg.get("num_primitive", 8)), composer_dim=tuple(cfg.get("composer_dim", [300, 200])),
            reactive_v=int(cfg.get("reactive_v", 0)), reactive_rate=float(cfg.get("reactive_rate", 0.3)),
            term_body=cfg.get("env_term_body", "body"), head_body=self.model_tables.body_names.index("Head"), reward_mul=cfg.reward_id == "world_rfc_implicit_v1_mul")
        self.policy_net, self.value_net, self.running_state = self.agent.policy, self.agent.value, self.agent.running_state
        self.state_dim, self.action_dim = self.agent.obs_dim, self.agent.act_dim
        self.expert_reward = reward_func[cfg.reward_id]
        self.env = None   # single-env facade, built lazily (eval_seq / visualisation code paths)
        self.logger = logging.getLogger(f"uhc_b200.{cfg.id}")
        if not self.logger.handlers:
            logging.basicConfig(level=logging.INFO, format="%(message)s")
        if checkpoint_epoch > 0:
            self.load_checkpoint(checkpoint_epoch)
            self.epoch = checkpoint_epoch

    # ---------------------------------------------------------------- schedules (:279-297)
    def per_epoch_update(self, epoch):
        cfg = self.cfg
        cfg.update_adaptive_params(epoch)
        self.agent.noise_rate = cfg.adp_noise_rate
        self.agent.opt_p.lr = cfg.adp_policy_lr
        if cfg.rfc_decay:
            rate = float(np.clip(1 - epoch / cfg.get("rfc_decay_max", 10000), 0, 1))
            self.agent.engine.set_cfg(rfc_rate=rate)
        if cfg.fix_std:
            self.agent.log_std.fill_(float(cfg.adp_log_std))

    # ---------------------------------------------------------------- sampling / update
    def sample(self, min_batch_size=None):
        T = self.horizon if min_batch_size is None else max(2, int(math.ceil(min_batch_size / self.num_envs)))
        buf, log = self.agent.sample(T)
        self._update_freq_dict(buf)
        log = _Log(log)
        log.update(avg_c_reward=log["avg_reward"], avg_episode_c_reward=log["avg_episode_reward"])
        return _Batch(buf), log

    def _update_freq_dict(self, buf):
        """per-clip success history from the episodes that ended in this rollout ([percent, fr_start] per episode, agent_copycat.py:561,
        590-603, capped at max_freq entries), then the device sampler's weights (dataset_amass_single.py:183-186)."""
        clip = buf.ep_clip.cpu().numpy().reshape(-1)
        pct = buf.ep_pct.cpu().numpy().reshape(-1)
        sel = clip >= 0
        keys = self.data_loader.data_keys
        for c, p in zip(clip[sel], pct[sel]):
            self.freq_dict[keys[c]].append([float(p), 0])
        self.freq_dict = {k: v[-self.max_freq:] for k, v in self.freq_dict.items()}
        self._push_clip_weights()

    def _push_clip_weights(self):
        from uhc_b200.agent import failure_weights
        cfg = self.cfg
        hist = [[r[0] for r in self.freq_dict[k]] for k in self.data_loader.data_keys]
        if any(len(h) for h in hist):
            self.agent.engine.set_clip_weights(failure_weights(hist, cfg.get("sampling_temp", 0.2), cfg.get("sampling_freq", 0.5)))

    def update_params(self, batch):
        return self.agent.update_params(batch.buf)["update_time"]

    def optimize_policy(self, epoch, save_model=True):
        cfg = self.cfg
        self.epoch = epoch
        t0 = time.time()
        self.per_epoch_update(epoch)
        batch, log = self.sample(cfg.min_batch_size)
        t1 = time.time()
        self.update_params(batch)
        t2 = time.time()
        info = {"log": log, "T_sample": t1 - t0, "T_update": t2 - t1, "T_total": t2 - t0}
        if save_model and (self.epoch + 1) % cfg.save_n_epochs == 0:
            self.save_checkpoint(epoch)
            info["log_eval"] = self.eval_policy(epoch)
        self.log_train(info)
        return info

    def log_train(self, info):
        log = info["log"]
        self.logger.info(f"{self.cfg.id} | {self.epoch:4d} | T_s {info['T_sample']:.2f} T_u {info['T_update']:.2f} | steps {log['num_steps']} "
                         f"({log['num_steps'] / max(info['T_sample'], 1e-9):.0f}/s) | eps_len {log['avg_episode_len']:.1f} | avg_r {log['avg_reward']:.4f} "
                         f"| eps_r {log['avg_episode_reward']:.2f} | fail {log['fail_rate']:.2f}")
        if not getattr(self.cfg, "no_log", True):
            try:
                import wandb
                wandb.log({"rewards": log["avg_reward"], "eps_len": log["avg_episode_len"], "avg_rwd": log["avg_episode_reward"]}, step=self.epoch)
                if "log_eval" in info:
                    [wandb.log(t, step=self.epoch) for t in info["log_eval"]]
            except Exception:
                pass

    # ---------------------------------------------------------------- evaluation (:354-494) on the device: BatchedAgent.evaluate
    def eval_policy(self, epoch=0, dump=False):
        """eval_policy / eval_seq (agent_copycat.py:354-494) for every clip: each clip is imitated from frame 0 with the deterministic policy
        (uhc_evaluate: a work queue of clips over the env slots, fail_safe re-seating a failed humanoid on the expert pose inside the step
        kernel, humanoid_im.py:902-905), and scored on the device with the reference's metrics (smpl_eval.compute_metrics: mpjpe / pa-mpjpe /
        accel / vel / root distance, restated in uhc_b200/metrics.py)."""
        from uhc_b200.agent import EVAL_METRICS
        cfg = self.cfg
        res_dicts = []
        eng = self.agent.engine
        for loader in self.test_data_loaders:
            n = loader.get_len()
            if loader is not self.data_loader:
                self._load_tables(loader)      # invalidates every env record: evaluate resets the slots it runs
            eng.set_cfg(**self._env_cfg(test=True))
            ev = self.agent.evaluate(0, n, bool(cfg.fail_safe))
            res = {}
            for i in range(n):
                k = loader.data_keys[i]
                L, fail_any = int(eng.clip_len[i]), bool(ev["fail_any"][i])
                percent = float(ev["last_t"][i]) / float(max(L - 1, 1))
                if ev["nframes"][i] >= 3:
                    fm = dict(zip(EVAL_METRICS, ev["frame_metrics"][i].T))
                    m = {"root_dist": fm["root_dist"], "mpjpe_g": fm["mpjpe_g"], "pa_mpjpe": fm["pa_mpjpe"], "mpjpe": fm["mpjpe"],
                         "accel_dist": fm["accel_dist"][2:], "vel_dist": fm["vel_dist"][1:]}
                    m["succ"] = np.array([percent >= 1.0 and not fail_any])
                else:
                    m = {"succ": np.array([False])}
                m["reward"] = ev["reward_sum"][i] / max(L - 1, 1)
                m["percent"] = percent
                res[k] = m
                if k in self.freq_dict:      # eval outcome feeds the failure-weighted sampler like a training episode ([percent, fr_start])
                    self.freq_dict[k] = (self.freq_dict[k] + [[1.0 if m["succ"][0] else min(percent, 0.999), 0]])[-self.max_freq:]
            if loader is not self.data_loader:
                self._load_tables(self.data_loader)
            eng.set_cfg(**self._env_cfg(test=False))
            self.agent.obs = None
            names = ("succ", "reward", "mpjpe", "mpjpe_g", "pa_mpjpe", "accel_dist", "vel_dist", "root_dist")
            metrics = {m: float(np.mean([np.mean(r[m]) for r in res.values() if m in r])) if any(m in r for r in res.values()) else float("nan") for m in names}
            coverage = int(round(metrics["succ"] * n))
            self.logger.info(f"Coverage {loader.name} of {coverage} out of {n} | " + " \t".join(f"{k}: {v:.3f}" for k, v in metrics.items()))
            metrics.update(mean_coverage=coverage / n, num_coverage=coverage, all_coverage=n)
            del metrics["succ"]
            res_dicts.append({f"coverage_{loader.name}": metrics})
            if dump:
                path = osp.join(cfg.output_dir, f"{epoch}_{loader.name}_coverage_full.pkl")
                joblib.dump(res, path)
        self._push_clip_weights()
        return res_dicts

    def _load_tables(self, loader):
        eng = self.agent.engine
        if self.motion_lib == "device":
            c = loader.smpl_clips()
            eng.load_smpl_clips(c["pose_aa"], c["trans"], loader.shapes)
        else:
            eng.load_clips(loader.experts, loader.shapes)

    def _env_cfg(self, test):
        cfg = self.cfg
        rw = cfg.reward_weights or {}
        return dict(base_rot=cfg.data_specs.get("base_rot", [0.7071, 0.7071, 0.0, 0.0]), rfc_scale=cfg.residual_force_scale, rfc_lim=cfg.residual_force_lim,
                    rfc_rate=0.0 if cfg.rfc_decay else 1.0, body_diff_thresh=cfg.get("body_diff_thresh_test" if test else "body_diff_thresh", 0.5),
                    meta_pd=int(cfg.meta_pd), env_episode_len=cfg.env_episode_len, trail_steps=cfg.env_expert_trail_steps, auto_reset=0 if test else 1,
                    rfc_mode=cfg.get("residual_force_mode", "implicit") if cfg.residual_force else "none", obs_v=int(cfg.obs_v),
                    fut_frames=int(cfg.get("fut_frames", 10)), fut_skip=int(cfg.get("skip", 10)),
                    has_shape=bool(cfg.get("has_shape", False)) and bool(cfg.get("has_shape_obs", True)),
                    term_body=cfg.get("env_term_body", "body"), head_body=self.model_tables.body_names.index("Head"), reward_mul=cfg.reward_id == "world_rfc_implicit_v1_mul",
                    w=[rw.get(k, d) for k, d in (("w_p", 0.6), ("w_v", 0.1), ("w_e", 0.2), ("w_c", 0.1), ("w_vf", 0.0))],
                    k=[rw.get(k, d) for k, d in (("k_p", 2), ("k_v", 0.005), ("k_e", 20), ("k_c", 1000), ("k_vf", 1))])

    def make_env(self, init_expert=None, mode="test"):
        """single-env facade (HumanoidEnv) for gym-style loops"""
        if init_expert is None:
            init_expert = self.data_loader.get_sample_from_key(self.data_loader.data_keys[0], full_sample=True)
        self.env = HumanoidEnv(self.cfg, init_expert, self.cfg.data_specs, mode=mode)
        return self.env

    # ---------------------------------------------------------------- checkpoints (:190-260)
    def save_checkpoint(self, epoch):
        """pickle {"policy_dict", "value_dict", "running_state": ZFilter} (agent_copycat.py:190-201).  Multi-GPU: every rank holds identical
        weights and running_state (uhc_b200/agent.py update_params), so rank 0 alone writes the file."""
        cfg = self.cfg
        path = "%s/iter_%04d.p" % (cfg.model_dir, epoch + 1)
        if int(os.environ.get("RANK", "0")) == 0:
            with open(path, "wb") as f:
                pickle.dump(self.agent.state_dicts(), f)
            joblib.dump(self.freq_dict, osp.join(cfg.result_dir, "freq_dict.pt"))
        return path

    def load_checkpoint(self, epoch):
        cfg = self.cfg
        path = "%s/iter_%04d.p" % (cfg.model_dir, epoch) if isinstance(epoch, int) else epoch
        self.logger.info("loading model from checkpoint: %s" % path)
        cp = pickle.load(open(path, "rb"))
        self.agent.load_state_dicts(cp)
        fd = osp.join(cfg.result_dir, "freq_dict.pt")
        if osp.exists(fd):
            self.freq_dict = joblib.load(fd)
