"""ctypes binding of libuhc_b200.so (include/uhc_b200.h) -- the batched humanoid-imitation engine.

PyTorch is plumbing here: it owns the device buffers handed to the C ABI and the CUDA stream.  There is NO CPU fallback:
if the CUDA library is missing or no GPU is visible this module raises.
"""
import ctypes as C
import os

import numpy as np

from .model import HumanoidModel, UhcModelHost

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.environ.get("UHC_B200_SO") or os.path.join(_HERE, "libuhc_b200.so")   # override: scratch builds of kernel variants
OBS_DIM, ACT_DIM, NQ, NV, NU, EX_SIZE = 657, 105, 76, 75, 69, 576
EXPERT_FIELDS = (("qpos", 76), ("qvel", 75), ("wbpos", 72), ("wbquat", 96), ("bquat", 96), ("bangvel", 72), ("ee_wpos", 15), ("com", 3))


class UhcEnvCfg(C.Structure):
    _fields_ = [("base_rot", C.c_double * 4), ("rfc_scale", C.c_double), ("rfc_lim", C.c_double), ("rfc_rate", C.c_double),
                ("body_diff_thresh", C.c_double), ("meta_pd", C.c_int), ("env_episode_len", C.c_int), ("trail_steps", C.c_int),
                ("newton_max_iter", C.c_int), ("w", C.c_double * 5), ("k", C.c_double * 5), ("newton_tol", C.c_double),
                ("auto_reset", C.c_int), ("t_min", C.c_int), ("t_max", C.c_int), ("reactive_v", C.c_int), ("reset_seed", C.c_ulonglong),
                ("reactive_rate", C.c_double), ("rfc_mode", C.c_int), ("vf_slot", C.c_int * 24), ("obs_v", C.c_int), ("fut_frames", C.c_int), ("fut_skip", C.c_int), ("no_shape", C.c_int), ("term_body", C.c_int), ("head_body", C.c_int), ("reward_mul", C.c_int)]


def make_cfg(precision=32, base_rot=(0.7071, 0.7071, 0.0, 0.0), rfc_scale=100.0, rfc_lim=100.0, rfc_rate=1.0, body_diff_thresh=0.5,
             meta_pd=1, env_episode_len=100000, trail_steps=0, w=(0.3, 0.1, 0.45, 0.1, 0.05), k=(2.0, 0.005, 5.0, 100.0, 1.0),
             newton_max_iter=None, newton_tol=None, auto_reset=0, t_min=5, t_max=300, reset_seed=1, reactive_v=0, reactive_rate=0.3,
             rfc_mode="implicit", vf_slot=None, obs_v=2, fut_frames=10, fut_skip=10, has_shape=True, term_body="body", head_body=13, reward_mul=False):
    """Defaults = config/release/uhc_implicit_shape.yml + copycat_config.py defaults of the reference."""
    c = UhcEnvCfg()
    c.base_rot = (C.c_double * 4)(*base_rot)
    c.rfc_scale, c.rfc_lim, c.rfc_rate, c.body_diff_thresh = rfc_scale, rfc_lim, rfc_rate, body_diff_thresh
    c.meta_pd, c.env_episode_len, c.trail_steps = int(meta_pd), int(env_episode_len), int(trail_steps)
    c.newton_max_iter = newton_max_iter or (20 if precision == 64 else 12)
    c.newton_tol = newton_tol or (1e-11 if precision == 64 else 1e-5)
    c.w, c.k = (C.c_double * 5)(*w), (C.c_double * 5)(*k)
    c.auto_reset, c.t_min, c.t_max, c.reset_seed = int(auto_reset), int(t_min), int(t_max), int(reset_seed)
    c.reactive_v, c.reactive_rate = int(reactive_v), float(reactive_rate)
    # cfg.residual_force_mode: "implicit" (6 action dims: root wrench) | "explicit" (24 x 9: contact point, force, torque per body, mj_applyFT)
    c.rfc_mode = 1 if rfc_mode in (1, "explicit") else (2 if rfc_mode in (2, "none", None, False) else 0)      # "none": cfg.residual_force false
    c.vf_slot = (C.c_int * 24)(*(list(vf_slot) if vf_slot is not None else range(24)))
    assert int(obs_v) in (1, 2, 3, 5, 6), "obs_v: 1 (get_full_obs_v1), 2 (get_full_obs_v2), 3 (get_full_obs_v3: fut_frames v2 blocks, skip frames apart), 5 / 6 (get_full_obs_v5 / v6)"
    c.obs_v, c.fut_frames, c.fut_skip, c.no_shape = int(obs_v), int(fut_frames), int(fut_skip), int(not has_shape)
    # cfg.env_term_body: "body" | "root" | "Head" (humanoid_im.py:1223-1229); head_body = model body of "Head" (13 in the SMPL humanoid)
    c.term_body = {"body": 0, "root": 1, "Head": 2, "head": 2, 0: 0, 1: 1, 2: 2}[term_body]
    c.head_body = int(head_body)
    c.reward_mul = int(bool(reward_mul))          # reward_id world_rfc_implicit_v1_mul
    return c


def obs_dim_of(cfg):
    """env.obs_dim: 657 (obs v2 with the shape vector) or 784 (obs v1)"""
    block = OBS_DIM - (17 if cfg.no_shape else 0)
    if cfg.obs_v in (5, 6):
        return (636 if cfg.obs_v == 5 else 384) + (0 if cfg.no_shape else 17)
    return 784 if cfg.obs_v == 1 else (block * (cfg.fut_frames if cfg.fut_frames > 0 else 10) if cfg.obs_v == 3 else block)


def act_dim_of(cfg):
    """env.action_dim (humanoid_im.py:250)"""
    return NU + {0: 6, 1: 216, 2: 0}[cfg.rfc_mode] + (30 if cfg.meta_pd else 0)


def pack_expert(ex):
    """expert dict -> [T][576] frame records (layout: include/uhc_b200.h UHC_EX_SIZE).  body_com (72, obs v1) starts where com (its first 3
    values: the root body's centre of mass) sits; an expert dict without body_com (obs v2 only) leaves the rest zero."""
    T = len(ex["qpos"])
    out = np.zeros((T, EX_SIZE))
    o = 0
    for k, n in EXPERT_FIELDS:
        out[:, o:o + n] = np.asarray(ex[k], dtype=np.float64).reshape(T, n)
        o += n
    if "body_com" in ex:
        bc = np.asarray(ex["body_com"], dtype=np.float64).reshape(T, 72)
        assert np.abs(bc[:, :3] - out[:, 502:505]).max() < 1e-9, "expert['com'] must be the root body's body_com"
        out[:, 502:574] = bc
    return out


_lib = None


def load_library():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise RuntimeError(f"{_SO} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback for the engine)")
        L = C.CDLL(_SO)
        L.uhc_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def _chk(rc):
    if rc != 0:
        raise RuntimeError("uhc_b200: " + load_library().uhc_last_error().decode())


def _ip(a):
    return np.ascontiguousarray(a, dtype=np.int32).ctypes.data_as(C.POINTER(C.c_int))


class Engine:
    """E environments on one GPU.  Mirrors HumanoidEnv.reset/step (+ the agent's custom_reward) for all envs at once."""

    def __init__(self, num_envs, model=None, device=0, precision=32, variants=None, **cfg):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("uhc_b200.Engine needs a CUDA device (no CPU fallback)")
        self.torch = torch
        self.lib = load_library()
        self.E, self.device, self.precision = int(num_envs), int(device), precision
        self.model = model or HumanoidModel()
        self.variants = variants
        self._ms = self.model.host_struct(variants)
        if cfg.get("rfc_mode") in (1, "explicit") and cfg.get("vf_slot") is None:
            cfg["vf_slot"] = self.model.vf_slot()                 # slot order of the reference: SMPL_BONE_ORDER_NAMES
        self._cfg_kw = dict(cfg)
        self._cfg = make_cfg(precision, **cfg)
        self.act_dim, self.obs_dim = act_dim_of(self._cfg), obs_dim_of(self._cfg)
        h = C.c_void_p()
        _chk(self.lib.uhc_engine_create(C.byref(self._ms), C.byref(self._cfg), C.c_int(self.E), C.c_int(self.device), C.c_int(precision), C.byref(h)))
        self.h = h
        dev = torch.device("cuda", self.device)
        f = dict(device=dev, dtype=torch.float32)
        self.obs = torch.zeros(self.E, self.obs_dim, **f)
        self.reward = torch.zeros(self.E, **f)
        self.cinfo = torch.zeros(self.E, 5, **f)
        self.percent = torch.zeros(self.E, **f)
        self.fail = torch.zeros(self.E, device=dev, dtype=torch.int32)
        self.end = torch.zeros(self.E, device=dev, dtype=torch.int32)
        self.clip_len = None
        if int(cfg.get("reactive_v", 0)) == 1:
            self.set_neutral_pose()

    def set_neutral_pose(self, qpos=None, qvel=None):
        """standing-neutral pose of the reactive starts; default = the bundled copy of the reference's sample_data/standing_neutral.pkl"""
        if qpos is None:
            z = np.load(os.path.join(_HERE, "assets", "standing_neutral.npz"))
            qpos, qvel = z["qpos"], z["qvel"]
        q, v = np.ascontiguousarray(qpos, np.float64), np.ascontiguousarray(qvel, np.float64)
        _chk(self.lib.uhc_set_neutral_pose(self.h, q.ctypes.data_as(C.POINTER(C.c_double)), v.ctypes.data_as(C.POINTER(C.c_double))))
        self.neutral = (q.copy(), v.copy())

    def close(self):
        if getattr(self, "h", None):
            self.lib.uhc_rollout_release(self.h)
            self.lib.uhc_eval_release(self.h)
            self.lib.uhc_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_cfg(self, **cfg):
        self._cfg_kw = dict(getattr(self, "_cfg_kw", {}), **cfg)
        self._cfg = make_cfg(self.precision, **self._cfg_kw)
        assert obs_dim_of(self._cfg) == self.obs_dim, "obs_v cannot change on a live engine (buffers are sized at creation)"
        self.act_dim = act_dim_of(self._cfg)
        _chk(self.lib.uhc_engine_set_cfg(self.h, C.byref(self._cfg)))

    def load_clips(self, experts, shapes=None, clip_models=None):
        """experts: list of dicts with the fields of Humanoid.qpos_fk (torch_smpl_humanoid.py:234-260); shapes: [C][17]."""
        lens = np.array([len(e["qpos"]) for e in experts], np.int32)
        frames = np.ascontiguousarray(np.concatenate([pack_expert(e) for e in experts]))
        shp = np.zeros((len(experts), 17)) if shapes is None else np.asarray(shapes, dtype=np.float64).reshape(len(experts), 17)
        shp = np.ascontiguousarray(shp)
        _chk(self.lib.uhc_load_clips(self.h, C.c_int(len(experts)), _ip(lens), frames.ctypes.data_as(C.POINTER(C.c_double)),
                                     shp.ctypes.data_as(C.POINTER(C.c_double))))
        self.clip_len = lens
        if clip_models is not None:
            _chk(self.lib.uhc_set_clip_models(self.h, C.c_int(len(experts)), _ip(clip_models)))

    def load_smpl_clips(self, pose_aa, trans, shapes=None, clip_models=None):
        """expert tables built on the device from raw SMPL sequences (uhc_load_clips_smpl, include/uhc_motion.h): the records
        make_expert + load_clips would give, without any host expert dict.  pose_aa: per-clip [T][72] or [T][156] axis-angle arrays (one width
        for all clips); trans: per-clip [T][3] arrays (a None entry, or trans None, = the default root height); shapes: [C][17]; clip_models:
        body-shape variant per clip."""
        pose = [np.asarray(p, dtype=np.float64) for p in pose_aa]
        n = len(pose)
        widths = {p.shape[1] for p in pose}
        if len(widths) != 1:
            raise ValueError(f"load_smpl_clips: every clip needs the same pose width, got {sorted(widths)}")
        lens = np.array([len(p) for p in pose], np.int32)
        tr = None
        if trans is not None and any(t is not None for t in trans):
            tr = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.float64).reshape(len(p), 3) if t is not None
                                                      else np.tile([0.0, 0.0, 0.91437225], (len(p), 1)) for p, t in zip(pose, trans)]))
        frames = np.ascontiguousarray(np.concatenate(pose))
        shp = np.ascontiguousarray(np.zeros((n, 17)) if shapes is None else np.asarray(shapes, dtype=np.float64).reshape(n, 17))
        cm = None if clip_models is None else np.ascontiguousarray(clip_models, dtype=np.int32)
        d = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        _chk(self.lib.uhc_load_clips_smpl(self.h, C.c_int(n), _ip(lens), C.c_int(widths.pop()), d(frames), d(tr) if tr is not None else None, d(shp),
                                          cm.ctypes.data_as(C.POINTER(C.c_int)) if cm is not None else None))
        self.clip_len = lens

    def get_clip_frames(self, frame0=0, nframes=None):
        """rows of the device clip table (all clips concatenated) as [n][576] doubles (uhc_get_clip_frames)"""
        n = int(self.clip_len.sum()) - frame0 if nframes is None else int(nframes)
        out = np.empty((n, EX_SIZE))
        _chk(self.lib.uhc_get_clip_frames(self.h, C.c_int(frame0), C.c_int(n), out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self, env_ids=None, clip=None, start=None, length=None, qpos=None, qvel=None):
        """env.reset() for the listed envs; returns the (whole) obs tensor [E,657] (rows of env_ids refreshed)."""
        t = self.torch
        ids = np.arange(self.E, dtype=np.int32) if env_ids is None else np.asarray(env_ids, dtype=np.int32)
        n = len(ids)
        clip = np.zeros(n, np.int32) if clip is None else np.broadcast_to(np.asarray(clip, np.int32), (n,))
        start = np.zeros(n, np.int32) if start is None else np.broadcast_to(np.asarray(start, np.int32), (n,))
        length = (self.clip_len[clip] - start) if length is None else np.broadcast_to(np.asarray(length, np.int32), (n,))
        qd = vd = None
        if qpos is not None:
            qd = t.as_tensor(np.asarray(qpos, np.float32).reshape(n, NQ)).to(self.obs.device).contiguous()
            vd = t.as_tensor(np.asarray(qvel, np.float32).reshape(n, NV)).to(self.obs.device).contiguous()
        _chk(self.lib.uhc_env_reset(self.h, C.c_int(n), _ip(ids), _ip(clip), _ip(start), _ip(length),
                                    C.c_void_p(qd.data_ptr() if qd is not None else None), C.c_void_p(vd.data_ptr() if vd is not None else None),
                                    C.c_void_p(self.obs.data_ptr()), self._stream()))
        return self.obs

    def step(self, actions, torque_out=None, reward_out=None):
        """env.step(a) + custom_reward for all envs.  actions: float32 cuda tensor [E,105].  Returns views of the engine's
        output tensors (obs, reward, cinfo, fail, end, percent)."""
        t = self.torch
        assert actions.is_cuda and actions.dtype == t.float32 and actions.is_contiguous() and tuple(actions.shape) == (self.E, self.act_dim)
        rew = self.reward if reward_out is None else reward_out
        _chk(self.lib.uhc_env_step(self.h, C.c_void_p(actions.data_ptr()), C.c_void_p(self.obs.data_ptr()), C.c_void_p(rew.data_ptr()),
                                   C.c_void_p(self.cinfo.data_ptr()), C.c_void_p(self.fail.data_ptr()), C.c_void_p(self.end.data_ptr()),
                                   C.c_void_p(self.percent.data_ptr()), C.c_void_p(torque_out.data_ptr() if torque_out is not None else None),
                                   self._stream()))
        return self.obs, rew, self.cinfo, self.fail, self.end, self.percent

    def step_host(self, actions, obs=None, reward=None, cinfo=None, fail=None, end=None, percent=None):
        """Host-buffer entry (H2D of actions and D2H of every requested output inside the call)."""
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.E, self.act_dim)
        obs = np.empty((self.E, self.obs_dim), np.float32) if obs is None else obs
        reward = np.empty(self.E, np.float32) if reward is None else reward
        cinfo = np.empty((self.E, 5), np.float32) if cinfo is None else cinfo
        fail = np.empty(self.E, np.int32) if fail is None else fail
        end = np.empty(self.E, np.int32) if end is None else end
        percent = np.empty(self.E, np.float32) if percent is None else percent
        p = lambda x: C.c_void_p(x.ctypes.data)
        _chk(self.lib.uhc_env_step_host(self.h, p(a), p(obs), p(reward), p(cinfo), p(fail), p(end), p(percent)))
        return obs, reward, cinfo, fail, end, percent

    def get_state(self, env=0):
        q, v, xp, bq, ist = np.zeros(NQ), np.zeros(NV), np.zeros(72), np.zeros(96), np.zeros(8, np.int32)
        d = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))
        _chk(self.lib.uhc_env_get_state(self.h, C.c_int(env), d(q), d(v), d(xp), d(bq), ist.ctypes.data_as(C.POINTER(C.c_int))))
        return dict(qpos=q, qvel=v, xpos=xp.reshape(24, 3), bquat=bq, cur_t=int(ist[0]), clip=int(ist[1]), start=int(ist[2]), len=int(ist[3]),
                    newton_iters=int(ist[6]), ncon=int(ist[7]))

    def get_states(self, env_ids=None):
        """state of many envs with one gather launch + one copy (evaluation / parity hook): dict of arrays [n, ...]."""
        ids = np.arange(self.E, dtype=np.int32) if env_ids is None else np.ascontiguousarray(env_ids, dtype=np.int32)
        n = len(ids)
        out, ist = np.zeros((n, 319)), np.zeros((n, 8), np.int32)
        _chk(self.lib.uhc_env_get_state_batch(self.h, C.c_int(n), _ip(ids), out.ctypes.data_as(C.POINTER(C.c_double)), ist.ctypes.data_as(C.POINTER(C.c_int))))
        return dict(qpos=out[:, :76], qvel=out[:, 76:151], xpos=out[:, 151:223].reshape(n, 24, 3), bquat=out[:, 223:319], cur_t=ist[:, 0], clip=ist[:, 1],
                    start=ist[:, 2], len=ist[:, 3], episode=ist[:, 4], flags=ist[:, 5], newton_iters=ist[:, 6], ncon=ist[:, 7])

    def set_state(self, env, qpos, qvel):
        self.set_states([env], np.asarray(qpos)[None], np.asarray(qvel)[None])

    def set_states(self, env_ids, qpos, qvel):
        """fail_safe for many envs at once (humanoid_im.py:902-905): one reset-with-override launch."""
        ids = np.ascontiguousarray(env_ids, dtype=np.int32)
        q = np.ascontiguousarray(qpos, np.float64).reshape(len(ids), NQ)
        v = np.ascontiguousarray(qvel, np.float64).reshape(len(ids), NV)
        _chk(self.lib.uhc_env_set_state_batch(self.h, C.c_int(len(ids)), _ip(ids), q.ctypes.data_as(C.POINTER(C.c_double)), v.ctypes.data_as(C.POINTER(C.c_double))))

    def set_clip_weights(self, weights=None):
        """sampling weights of the in-kernel re-seeding (None = the reference's sample_keys rule)."""
        if weights is None:
            _chk(self.lib.uhc_set_clip_weights(self.h, C.c_int(len(self.clip_len)), None))
        else:
            w = np.ascontiguousarray(weights, dtype=np.float32)
            _chk(self.lib.uhc_set_clip_weights(self.h, C.c_int(len(w)), w.ctypes.data_as(C.POINTER(C.c_float))))

    @property
    def counters(self):
        out = np.zeros(4, np.int32)
        _chk(self.lib.uhc_engine_counters(self.h, out.ctypes.data_as(C.POINTER(C.c_int))))
        return dict(contact_overflow_steps=int(out[0]), invalid_env_steps=int(out[1]))

    @property
    def kernel_launches(self):
        return self.lib.uhc_kernel_launches(self.h)
