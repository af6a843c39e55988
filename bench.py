#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched humanoid-imitation rollout (BASELINE.json metric) on N B200s.

A "step" is one lock-step control step of every environment: observation normaliser -> policy MLP forward (tcgen05) ->
Gaussian sample -> fused physics(15 substeps)+task kernel -> transition written to the HBM rollout buffer -> re-seeding of
finished episodes; the whole step is one call of the C-ABI loop (uhc_rollout) = one CUDA-graph launch.  Workload at N=1 = BASELINE.json configs[1]: 4096 SMPL-neutral humanoids imitating one AMASS-shaped clip,
policy rollout only.  N>1: weak scaling, 4096 envs per GPU, no data-path collective (the rollout has none).

  python bench.py --gpus 1 --steps 20 --warmup 3
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference          # the reference's CPU path: oracle port (fp64 C) on all host cores
  python bench.py --dump-outputs DIR         # also write what the last timed step computed, DIR/<name>.npy, to compare two builds
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
ENVS_PER_GPU = 4096
CLIP_FRAMES = 320                      # length of '0-ACCAD_Male2General_c3d_A2- Sway_poses', the clip configs[1] names
BYTES_PER_ENV_STEP = 6396              # algorithmic HBM bytes of the fused physics/task step, SURVEY.md section 8(d)
METRIC, UNIT = "env_steps_per_s", "env-steps/s"
DUMP_LIMIT = 64 << 20                  # bytes, all --dump-outputs arrays together


def make_clip(seed=1):
    from uhc_b200 import motion_lib
    ex = motion_lib.synthetic_clip(CLIP_FRAMES, np.random.default_rng(seed))
    shape = np.zeros(17)
    return ex, shape


def dump_outputs(path, arrays):
    """DIR/<name>.npy for each array (tensor or numpy; float64 kept, everything else as float32), at most DUMP_LIMIT bytes in all."""
    out = {}
    for k, v in arrays.items():
        a = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
        out[k] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------ CPU reference arm
REF_ENVS_PER_CORE = 32                 # bounded sample: every host process owns this many oracle envs; one "step" steps each of them once
_REF_POLICY = None


def _ref_policy():
    """The bench policy (same seeded initial weights as the GPU arm) evaluated the way the reference does: torch fp64 on the CPU
    (scripts/train_uhc.py:80-81 sets float64; khrylib/rl/core/policy_gaussian.py:26-31)."""
    global _REF_POLICY
    if _REF_POLICY is None:
        import torch
        from uhc_b200 import nn
        net = nn.MLPNet(657, (2048, 1024, 512), 105, "gelu", device="cpu", head_name="action_mean", seed=1)
        _REF_POLICY = ([w.double() for w in net.W], [b.double() for b in net.b])
    return _REF_POLICY


def _cpu_worker(args):
    """One host process: REF_ENVS_PER_CORE oracle envs; per step ZFilter -> policy MLP (fp64) -> Gaussian sample -> env.step + reward,
    finished episodes re-seeded (start ~ U[0, L - t_min)).  Runs `warmup` untimed and `steps` timed steps; returns the timed wall."""
    import torch
    seed, steps, warmup, nenv = args
    torch.set_num_threads(1)
    from oracle import oracle as O
    ex, shape = make_clip()
    rng = np.random.RandomState(seed)
    keys = ("qpos", "qvel", "wbpos", "wbquat", "bquat", "bangvel", "ee_wpos", "com")
    om = O.Model()

    def seeded():
        s = rng.randint(0, CLIP_FRAMES - 5)
        return {k: np.asarray(ex[k])[s:s + 300] for k in keys}
    envs = [O.Env(om, seeded(), shape) for _ in range(nenv)]
    obs = np.stack([e.reset() for e in envs])
    Ws, bs = _ref_policy()
    n, mean, S = 0.0, np.zeros(657), np.zeros(657)
    t0 = None
    for it in range(warmup + steps):
        if it == warmup:
            t0 = time.perf_counter()
        nb, mb = float(len(obs)), obs.mean(0)                       # ZFilter, batched Chan merge (zfilter.py:7-73), clip 5
        Sb = ((obs - mb) ** 2).sum(0)
        d = mb - mean
        tot = n + nb
        mean, S, n = mean + d * nb / tot, S + Sb + d * d * n * nb / tot, tot
        std = np.sqrt(S / (n - 1)) if n > 1 else np.abs(mean)
        h = torch.from_numpy(np.clip((obs - mean) / (std + 1e-8), -5, 5))
        for i, (W, b) in enumerate(zip(Ws, bs)):
            h = h @ W.T + b
            if i < len(Ws) - 1:
                h = torch.nn.functional.gelu(h)
        act = h.numpy() + np.exp(-2.3) * rng.standard_normal((len(obs), 105))
        for j, e in enumerate(envs):
            o, _, done, _ = e.step(act[j])
            if done:
                e.load_expert(seeded(), shape)
                o = e.reset()
            obs[j] = o
    return nenv * steps, time.perf_counter() - t0


def usable_cores():
    """host threads this process may actually use: min(os.cpu_count, scheduler affinity, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().split()[0])
                    n = min(n, max(1, q // period))
        except Exception:
            pass
    return max(1, n)


def cpu_baseline(steps=8, warmup=1, cores=None, envs_per_core=REF_ENVS_PER_CORE):
    """The reference's CPU path restated (oracle/uhc_oracle.c: PD + 15 substeps + obs + reward; the policy in torch fp64 as the
    reference runs it), one process per usable host core, on a bounded sample of the bench workload: cores x envs_per_core envs, `steps`
    lock-step control steps.  Returns throughput and the MEASURED wall time per step of that sample."""
    import multiprocessing as mp
    from oracle import oracle as O
    O.build()
    _ref_policy()
    cores = cores or usable_cores()
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(i + 1, steps, warmup, envs_per_core) for i in range(cores)])
    env_steps = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    return dict(value=env_steps / wall, unit=UNIT, cores=cores, kind="port", sample_envs=cores * envs_per_core, sample_steps=steps,
                ms_per_sample_step=1e3 * wall / steps,
                sample=f"{cores * envs_per_core} envs ({envs_per_core} per process, {cores} processes) x {steps} control steps of the same workload = {env_steps} env-steps "
                       f"in {wall:.2f} s: fp64 obs normaliser + 657-2048-1024-512-105 policy (torch fp64, same initial weights) + fp64 C restatement of the "
                       "MuJoCo+Python step (oracle/, NOT MuJoCo itself), episodes re-seeded on termination")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.time()
    cb = cpu_baseline(steps=args.steps, warmup=args.warmup)
    cfg = workload_config(args.gpus)
    cfg["reference_sample"] = (f"each reference step = one control step of {cb['sample_envs']} envs ({REF_ENVS_PER_CORE} per host process), a bounded sample of the "
                               f"{ENVS_PER_GPU * args.gpus}-env workload; ms_per_step is the measured wall time of that sample step")
    line = dict(impl="reference", metric=METRIC, value=cb["value"], unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=cb["ms_per_sample_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic", config=cfg, cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), wall_s=time.time() - t0)
    print(json.dumps(line))


def workload_config(n):
    return {"workload": f"{ENVS_PER_GPU} SMPL-neutral humanoids per GPU imitating one {CLIP_FRAMES}-frame AMASS-shaped clip, policy rollout only "
                        "(obs normaliser + 657-2048-1024-512-105 gelu policy + physics/task step), uhc_implicit_shape hyper-parameters",
            "envs_per_gpu": ENVS_PER_GPU, "global_envs": ENVS_PER_GPU * n, "parallelism": f"env-sharded x{n}, no data-path collective",
            "l2": "flushed (256 MiB write) between timed steps", "policy_gemm": "tcgen05 bf16 operands, fp32 accumulate",
            "physics": "fp32, 15 substeps/step, primal Newton contact solve"}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 20 ms from before the warm-up; stop(t0, t1) keeps the samples whose
    timestamp falls inside the timed region [t0, t1] (wall clock), or the nearest ones when the region is shorter than a sample."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self, t0=None, t1=None):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.p.terminate()
        self.p.wait()
        self.f.seek(0)
        import datetime
        rows = []
        for line in self.f.read().strip().splitlines():
            r = [x.strip() for x in line.split(",")]
            if len(r) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(r[1]), float(r[2]), float(r[3]), r[4:8]))
            except Exception:
                continue
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "samples": 0}
        sel = [r for r in rows if t0 is not None and t0 <= r[0] <= t1]
        where = "inside the timed region"
        if not sel:
            mid = 0.5 * ((t0 or rows[-1][0]) + (t1 or rows[-1][0]))
            sel = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            where = "nearest to the timed region (region shorter than the sampling period)"
        reasons = set()
        for r in sel:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median([r[1] for r in sel])), "sm_max_mhz": sel[0][2], "power_w_max": max(r[3] for r in sel),
                "samples": len(sel), "where": where, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    from uhc_b200.agent import BatchedAgent, RolloutBuffer
    ex, shape = make_clip()
    E, K, W = ENVS_PER_GPU, args.steps, max(args.warmup, 3)
    agent = BatchedAgent(E, [ex], [shape], device=local, seed=1, rank=rank, world=world)
    agent.reset_envs()
    L, h = agent.engine.lib, agent.engine.h
    R = max(1, min(K, 32))                               # buffer rows in use: one CUDA graph (and one pair of kernel events) per row
    buf = RolloutBuffer(R, E, agent.dev, agent.act_dim, agent.obs_dim)
    if L.uhc_rollout_time_env_step(h, C.c_int(R)) != 0:  # CUDA events around k_env_step, recorded on the launching stream inside the graph
        raise RuntimeError("uhc_rollout_time_env_step failed")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=agent.dev)
    clocks = ClockSampler(local) if rank == 0 else None
    for k in range(max(W, R)):                           # warm-up: every row's graph is captured and instantiated here, outside the timed region
        agent.rollout(buf, 1, k % R)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    l0, n0 = agent.engine.kernel_launches, agent.nn_launches
    per_step = L.uhc_rollout_launches_per_step(h)
    torch.cuda.synchronize()
    t_wall0 = time.time()
    for k in range(K):
        flush.fill_(k & 0xFF)                            # L2 flush, outside the timed region
        ev[k][0].record()
        agent.rollout(buf, 1, k % R)                     # ONE control step of all envs: uhc_rollout -> one CUDA-graph launch
        ev[k][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall1 = time.time()
    last = None
    if args.dump_outputs and rank == 0:                  # the last timed step's results, copied before the steps below overwrite them
        r = (K - 1) % R
        last = dict(next_obs=agent.obs, state=buf.states[r], action=buf.actions[r], logp=buf.logp[r], reward=buf.rewards[r], mask=buf.masks[r],
                    fail=buf.fails[r], obs_filter_stats=agent.running_state.stats)
        last = {k: v.cpu() for k, v in last.items()}
    clk = clocks.stop(t_wall0, t_wall1) if clocks else None
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    ms = C.c_float(0)
    kms, kern_src = [], "CUDA events around k_env_step recorded inside the timed graph replays (external event-record nodes on the launching stream)"
    for r in range(R):
        if L.uhc_rollout_env_step_ms(h, C.c_int(r), C.byref(ms)) != 0:
            kms = None
            break
        kms.append(ms.value)
    if kms is None:
        # fallback: the same steps launched as plain stream launches (identical kernels), events around k_env_step on that stream
        kern_src = "CUDA events around k_env_step in an extra pass of plain stream launches of the same step (graph event nodes unreadable on this driver)"
        kms = []
        for k in range(R):
            flush.fill_(k & 0xFF)
            agent.rollout(buf, 1, k % R, use_graph=False)
        torch.cuda.synchronize()
        for r in range(R):
            if L.uhc_rollout_env_step_ms(h, C.c_int(r), C.byref(ms)) != 0:
                L.uhc_rollout_last_error.restype = C.c_char_p
                raise RuntimeError("uhc_rollout_env_step_ms failed: " + L.uhc_rollout_last_error().decode())
            kms.append(ms.value)
    kern_ms = float(np.mean(kms))
    launches = per_step * K
    tt = torch.tensor([total_ms], device=agent.dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    value = E * world * K / (total_ms * 1e-3)

    # end to end through host buffers: the step's input (the observations) comes from pinned host memory, the step runs through the public
    # call (BatchedAgent.rollout -> uhc_rollout), and its results (next obs, actions, reward, mask, fail) are read back to the host; one sync per step
    Ke = K
    pin = lambda *shape, dtype=torch.float32: torch.empty(*shape, dtype=dtype).pin_memory()
    obs_h, act_h, rew_h, mask_h, fail_h = pin(E, 657), pin(E, 105), pin(E), pin(E), pin(E, dtype=torch.int32)
    obs_h.copy_(agent.obs)
    torch.cuda.synchronize()

    def e2e_step():
        agent.obs.copy_(obs_h, non_blocking=True)
        agent.rollout(buf, 1, 0)
        obs_h.copy_(agent.obs, non_blocking=True); act_h.copy_(buf.actions[0], non_blocking=True); rew_h.copy_(buf.rewards[0], non_blocking=True)
        mask_h.copy_(buf.masks[0], non_blocking=True); fail_h.copy_(buf.fails[0], non_blocking=True)
        torch.cuda.synchronize()
    for _ in range(3):
        e2e_step()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(Ke):
        e2e_step()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=agent.dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = E * world * Ke / float(te.item())
    counters = agent.engine.counters
    st = agent.engine.get_states()        # solver work of the last control step (what the step time is made of)
    counters.update(newton_iters_per_env_step=float(st["newton_iters"].mean()), newton_iters_max=int(st["newton_iters"].max()),
                    max_contacts_per_env_step_mean=float(st["ncon"].mean()))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = BYTES_PER_ENV_STEP * E / (kern_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r02_env_step_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("how")
        except Exception:
            pass
    cb = cpu_baseline(steps=6, warmup=1) if (world == 1 and not os.environ.get("UHC_BENCH_SKIP_CPU")) else None   # (skipped under ncu)
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=total_ms / K, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", config=workload_config(world),
                roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=traffic, traffic_source=traffic_src,
                              kernel="k_env_step<float>", kernel_ms=kern_ms, kernel_ms_source=kern_src, kernel_share_of_step=kern_ms / (total_ms / K),
                              peak_source="MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                              note="algorithmic bytes 6396 B/env-step (SURVEY 8d); the step is latency/issue bound, not HBM bound -- see DESIGN.md"),
                e2e=dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=E * 657 * 4, d2h_bytes_per_step=E * (657 + 105 + 1 + 1 + 1) * 4, steps=Ke,
                         path="pinned host obs -> device, BatchedAgent.rollout (uhc_rollout, 1 step), next obs / action / reward / mask / fail -> pinned host, one sync"),
                gpu_launches=launches, launches_per_step=per_step, step_driver="uhc_rollout: one CUDA-graph launch per control step",
                env_counters=counters, clocks=clk)
    if cb:
        line["cpu_baseline"] = cb
    if last:
        dump_outputs(args.dump_outputs, last)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ train workload (BASELINE configs 3-5)
TAKE5_LENS = (320, 375, 146, 236, 121, 170, 137, 69, 209, 189)     # clip lengths of sample_data/amass_copycat_take5_test_small.pkl
TRAIN_T, TRAIN_EPOCHS = 32, 10


def make_train_clips(world):
    """N = 1: BASELINE configs[2] -- ten AMASS-shaped clips with the lengths of take5_test_small, one body shape.
    N > 1: configs[3]/[4] -- 24 clips in the issue-class proportions of amass_copycat_occlusion_v2 (normal / sitting / airborne ~ 54 / 33 / 13 %,
    SURVEY.md section 8d) and three synthetic body-shape variants (limb scaling; the SMPL files are licence-gated)."""
    from uhc_b200 import motion_lib
    from uhc_b200.model import HumanoidModel, NB
    rng = np.random.default_rng(7)
    if world == 1:
        clips = [motion_lib.synthetic_clip(L, rng) for L in TAKE5_LENS]
        return clips, [np.zeros(17) for _ in clips], None, None, None
    kinds = ["normal"] * 13 + ["sitting"] * 8 + ["airborne"] * 3
    clips = [motion_lib.synthetic_clip(int(rng.integers(60, 300)), rng, kind=k) for k in kinds]
    base = HumanoidModel()
    variants = [base] + [HumanoidModel(scale=np.full(NB, sc)) for sc in (0.92, 1.08)]
    clip_models = [i % 3 for i in range(len(clips))]
    shapes = [np.concatenate([np.full(16, 0.1 * m), [0.0]]) for m in clip_models]
    return clips, shapes, base, variants, clip_models


def run_train(args):
    """`--workload train`: one "step" = one full PPO iteration on every GPU: T = 32 lock-step control steps of 4096 envs per GPU (uhc_rollout),
    V(s) + GAE + advantage normalisation, 10 epochs of (value step, clipped-surrogate policy step) on the tensor-core path, with the
    gradient all-reduce (the design's only collective) INSIDE the timed region."""
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    from uhc_b200.agent import BatchedAgent, RolloutBuffer
    clips, shapes, base, variants, clip_models = make_train_clips(world)
    E, K, W, T = ENVS_PER_GPU, args.steps, max(args.warmup, 3), TRAIN_T
    agent = BatchedAgent(E, clips, shapes, device=local, seed=1, rank=rank, world=world, model=base, variants=variants, clip_models=clip_models,
                         num_optim_epoch=TRAIN_EPOCHS, t_min=15, t_max=300)
    agent.reset_envs()
    buf = RolloutBuffer(T, E, agent.dev, agent.act_dim, agent.obs_dim)
    clocks = ClockSampler(local) if rank == 0 else None
    for _ in range(W):
        agent.sample(T, buf); agent.update_params(buf)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * K + 1)]
    phases = dict(gae_ms=0.0, epochs_ms=0.0, allreduce_ms=0.0, allreduce_bytes=0, allreduce_calls=0)
    def launches():       # env-step launches (engine) + the rollout's other kernels + the kernels uhc_ppo_update enqueued
        return agent.engine.kernel_launches + agent.nn_launches + (agent._ctrainer.kernel_launches if agent._ctrainer is not None else 0)
    l0 = launches()
    t_wall0 = time.time()
    ev[0].record()
    for k in range(K):
        agent.rollout(buf, T)
        buf.last_obs.copy_(agent.obs)
        ev[2 * k + 1].record()
        out = agent.update_params(buf)
        ev[2 * k + 2].record()
        for key in phases:
            phases[key] += out.get(key, 0)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall1 = time.time()
    if args.dump_outputs and rank == 0:                  # the parameters and observation statistics after the last iteration, and its losses
        dump_outputs(args.dump_outputs, dict(policy_params=agent.policy.flat, value_params=agent.value.flat, obs_filter_stats=agent.running_state.stats,
                                             losses=np.array([out["surr_loss"], out["value_loss"]], np.float32)))
    clk = clocks.stop(t_wall0, t_wall1) if clocks else None
    total_ms = ev[0].elapsed_time(ev[2 * K])
    sample_ms = sum(ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(K)) / K
    update_ms = sum(ev[2 * k + 1].elapsed_time(ev[2 * k + 2]) for k in range(K)) / K
    tt = torch.tensor([total_ms], device=agent.dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    value = E * world * T * K / (total_ms * 1e-3)
    # identical parameters and observation normaliser on every rank (the tail of the gradient all-reduce keeps them in lock-step)
    chk = torch.stack([agent.policy.flat.double().sum(), agent.value.flat.double().sum(), agent.running_state.stats.sum()])
    same = True
    if world > 1:
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same = bool(torch.equal(lo, hi))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    N = T * E
    npar = agent.policy.flat.numel() + agent.value.flat.numel()
    flops_update = TRAIN_EPOCHS * 6.0 * (sum(w.numel() for w in agent.policy.W) + sum(w.numel() for w in agent.value.W)) * N
    peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    ach = flops_update / (phases["epochs_ms"] / K * 1e-3) / 1e12
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=total_ms / K, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f32 physics / bf16 tensor-core operands, fp32 accumulate + fp32 master weights", data="synthetic",
                config={"workload": f"full PPO train loop, {E} envs per GPU x T={T} control steps per iteration (N = {N} transitions per GPU), GAE + {TRAIN_EPOCHS} full-batch epochs "
                                    "(value step + clipped-surrogate policy step, Adam), 657-2048-1024-512-{105,1} gelu nets, "
                                    + ("10 AMASS-shaped clips with the take5_test_small lengths (BASELINE configs[2])" if world == 1 else
                                       "24 synthetic clips in the occlusion_v2 class mix (normal/sitting/airborne), 3 body-shape variants (BASELINE configs[3]/[4] shapes)"),
                        "envs_per_gpu": E, "global_envs": E * world, "global_batch": N * world,
                        "parallelism": f"env-sharded x{world}; per optimisation step one all-reduce of each net's flat fp32 gradient tensor (NCCL), overlapped with the other net's backward; "
                                       "advantage / ZFilter statistics ride in its tail; nothing else crosses GPUs",
                        "l2": "not flushed: every iteration streams a 1.3 GB rollout buffer (inputs larger than L2)"},
                phases=dict(sample_ms=sample_ms, update_ms=update_ms, gae_ms=phases["gae_ms"] / K, epochs_ms=phases["epochs_ms"] / K,
                            allreduce_ms_per_iter=phases["allreduce_ms"] / K, allreduce_bytes_per_iter=phases["allreduce_bytes"] / K,
                            allreduce_calls_per_iter=phases["allreduce_calls"] / K,
                            allreduce_busbw_GBps=(phases["allreduce_bytes"] * 2 * (world - 1) / world / (phases["allreduce_ms"] * 1e-3) / 1e9) if phases["allreduce_ms"] > 0 else None),
                replicas_identical=same, parameters=npar,
                roofline=dict(bound="tensor", kernel="k_linear_tc2 (CTA-pair tcgen05 GEMMs: forward, dX with the activation backward fused, split-K dW of both nets)", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak, traffic=None,
                              peak_source="MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1400 TFLOP/s",
                              note="6 x parameters x N flop per epoch over the measured time of the 10 epochs (includes the loss, head activation-gradient, weight-transpose, Adam and bf16 weight-refresh kernels)"),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=16,
                         note="the training iteration has no host inputs (observations, rollout buffer and weights are device resident); the host reads back the two loss scalars"),
                gpu_launches=(launches() - l0), update_driver="uhc_ppo_update: one C-ABI call per iteration (V(s), GAE, epochs, Adam, gradient all-reduce on the job's ncclComm_t)",
                clocks=clk)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="rollout", choices=["rollout", "train"],
                    help="rollout (default, the headline: BASELINE configs[1]) or train (configs[2] at N=1, configs[3]/[4] shapes at N>1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's envs) as DIR/<name>.npy: float32 / float64, at most 64 MB; "
                         "the same arguments give the same inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "train":
        run_train(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
