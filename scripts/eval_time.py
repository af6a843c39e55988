"""Wall time of one AgentCopycat.eval_policy (eval_uhc.py --mode stats, every save_n_epochs of training): the host loop it replaced (restated
in tests/test_gpu_eval.py as host_eval_policy) against the device path (uhc_evaluate), alternated, two runs each.

Cases: E = 4096 env slots with 12 288 synthetic clips, and with the first 100 of them.  The clips are slices of 512 synthetic motions
(motion_lib.synthetic_clip, kinds normal / sitting / airborne in turn); their lengths are drawn from a log-normal distribution, median 45
frames, sigma 0.8, clipped to [8, 600] (right-skewed: a few long clips; an assumption, not AMASS statistics).  Policy: the production
sizes of config/uhc_b200_default.yml, untrained (seeded initial weights), fail_safe on.  Reported per evaluation: wall seconds, control steps
that had an active slot, mean fraction of env slots busy (recorded rows / (steps x E)).  Also the wall time of one training iteration
(optimize_policy at the same E, min_batch_size of the config) and from it the share of a save_n_epochs = 100 checkpoint interval that one
evaluation costs; with --parent-tree DIR (a built checkout of the parent commit) the rollout bench (bench.py --gpus 1 --steps 20 --warmup 3)
of the parent and of this tree, before and after the evaluation timing.

    python scripts/eval_time.py [OUT.json] [--parent-tree DIR]      (one JSON document to OUT.json and stdout)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import types

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)


class ClipLoader:
    """the part of DatasetAMASSSingle eval_policy reads"""

    def __init__(self, experts, shapes, name):
        self.experts, self.shapes, self.name = experts, shapes, name
        self.data_keys = [f"synthetic_{i}" for i in range(len(experts))]

    def get_len(self):
        return len(self.experts)


def clip_set(nclips, seed=0):
    from uhc_b200.motion_lib import synthetic_clip
    rng = np.random.RandomState(seed)
    lens = np.clip(np.round(np.exp(rng.normal(np.log(45.0), 0.8, nclips))), 8, 600).astype(int)
    base = [synthetic_clip(600, rng, kind=("normal", "sitting", "airborne")[i % 3]) for i in range(512)]
    keys = ("qpos", "qvel", "wbpos", "wbquat", "bquat", "bangvel", "ee_wpos", "com", "body_com")
    experts = []
    for i, T in enumerate(lens):
        b = base[i % len(base)]
        s = int(rng.randint(0, 600 - T + 1))
        e = {k: b[k][s:s + T] for k in keys}
        e["len"] = int(T)
        experts.append(e)
    return experts, [np.zeros(17) for _ in experts], lens


def make_agent(tmp, E):
    import torch
    import yaml
    from tests.helpers import write_synthetic_pkl
    from uhc.agents import agent_dict
    from uhc.utils.config_utils.copycat_config import Config
    os.chdir(tmp)
    base = yaml.safe_load(open(os.path.join(ROOT, "config", "uhc_b200_default.yml")))
    base.update(num_envs=E, no_log=True)
    base["data_specs"]["file_path"] = write_synthetic_pkl(os.path.join(tmp, "sample_data", "clips.pkl"))
    cfg = Config(cfg_id="eval_time", create_dirs=True, cfg_dict=base)
    cfg.update(types.SimpleNamespace(cfg="eval_time", render=False, test=False, num_threads=1, gpu_index=0, epoch=0, show_noise=False,
                                     resume=None, no_log=True, debug=False, full_eval=False))
    return agent_dict[cfg.agent_name](cfg, torch.float32, torch.device("cuda", 0), training=True, checkpoint_epoch=0)


def bench_leg(tree):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "3"], cwd=tree, capture_output=True, text=True)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    return json.loads(lines[-1])["value"] if r.returncode == 0 and lines else "failed (rc %d): %s" % (r.returncode, r.stderr[-300:])


def bench_legs(parent):
    if not parent:
        return None
    return {"parent": bench_leg(parent), "this": bench_leg(ROOT)}


def main():
    import torch
    from tests.test_gpu_eval import host_eval_loop, host_eval_policy
    import tests.test_gpu_eval as tge
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--parent-tree", default=None)
    args = ap.parse_args()
    out_path = os.path.abspath(args.out) if args.out else None      # make_agent changes the working directory
    parent = os.path.abspath(args.parent_tree) if args.parent_tree else None
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["clocks_max_sm_mhz"] = float(q[0]), float(q[1])
    except Exception as ex:      # the numbers are reported as not measured
        out["power_limit_w"] = out["clocks_max_sm_mhz"] = "not measured (%s)" % ex
    bench = {"before": bench_legs(parent)}
    E, N = 4096, 12288
    t0 = time.time()
    experts, shapes, lens = clip_set(N)
    out["clips"] = dict(n=N, length_distribution="round(exp(N(log 45, 0.8))) clipped to [8, 600]", mean_len=float(lens.mean()),
                        median_len=float(np.median(lens)), max_len=int(lens.max()), total_frames=int(lens.sum()), build_s=time.time() - t0)
    tmp = tempfile.mkdtemp(prefix="eval_time_")
    ac = make_agent(tmp, E)
    out["policy"] = "config/uhc_b200_default.yml: policy_hsize %s, untrained; fail_safe %s" % (list(ac.cfg.policy_hsize), bool(ac.cfg.fail_safe))
    ac.optimize_policy(0, save_model=False)                 # warm-up, then one training iteration's wall time (sample + update)
    torch.cuda.synchronize()
    t1 = time.time()
    for i in range(1, 4):
        ac.optimize_policy(i, save_model=False)
    torch.cuda.synchronize()
    iter_s = (time.time() - t1) / 3
    out["train_iteration"] = dict(E=E, min_batch_size=int(ac.cfg.min_batch_size), wall_s=iter_s)
    stats = {}

    # per-evaluation counters: steps and recorded rows of the host loop (a batch runs until its last live clip ends) / of uhc_evaluate
    def counted_host_loop(agent, ex, n, fail_safe):
        res = host_eval_loop(agent, ex, n, fail_safe)
        rows = np.array([len(r["t"]) for r in res])
        steps = sum(int(rows[c0:c0 + agent.E].max()) for c0 in range(0, n, agent.E))
        stats["last"] = (steps, int(rows.sum()))
        return res
    tge.host_eval_loop = counted_host_loop
    evaluate = ac.agent.evaluate

    def counted_evaluate(*a, **k):
        r = evaluate(*a, **k)
        stats["last"] = (r["steps"], int(r["nframes"].sum()))
        return r
    ac.agent.evaluate = counted_evaluate
    cases = []
    for n in (N, 100):
        loader = ClipLoader(experts[:n], shapes[:n], f"synthetic_{n}")
        ac.agent.engine.load_clips(loader.experts, loader.shapes)
        ac.data_loader, ac.test_data_loaders = loader, [loader]
        ac.freq_dict = {k: [] for k in loader.data_keys}
        runs = []
        for rep in range(2):
            for name, fn in (("host_loop", lambda: host_eval_policy(ac, 0, False)), ("device", lambda: ac.eval_policy(0, False))):
                torch.cuda.synchronize()
                t1 = time.time()
                res = fn()
                torch.cuda.synchronize()
                wall = time.time() - t1
                steps, rows = stats["last"]
                m = res[0][f"coverage_{loader.name}"]
                runs.append(dict(path=name, rep=rep, wall_s=wall, control_steps=steps, recorded_rows=rows, busy_slot_fraction=rows / float(steps * E),
                                 mean_coverage=m["mean_coverage"], mpjpe=m["mpjpe"]))
                print(json.dumps(runs[-1]), flush=True)
        cases.append(dict(E=E, n=n, runs=runs))
    out["cases"] = cases
    interval = 100 * iter_s
    out["summary"] = {f"n{c['n']}": {p: dict(wall_s=[r["wall_s"] for r in c["runs"] if r["path"] == p],
                                            share_of_100_iteration_interval=[r["wall_s"] / (interval + r["wall_s"]) for r in c["runs"] if r["path"] == p])
                                     for p in ("host_loop", "device")} for c in cases}
    out["summary"]["note"] = ("the first device run includes the first launches of the evaluation kernels; share = evaluation / (100 training "
                              "iterations + evaluation)")
    bench["after"] = bench_legs(parent)
    if parent:
        out["rollout_bench_env_steps_per_s"] = bench
    txt = json.dumps(out, indent=1)
    if out_path:
        with open(out_path, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
