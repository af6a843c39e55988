"""Wall time of turning a dataset into the engine's expert table: the host path (motion_lib.make_expert per clip in numpy fp64, then
Engine.load_clips: pack_expert into [frames][576] doubles, the float conversion loop and the upload of uhc_load_clips) against the device path
(Engine.load_smpl_clips: concatenate the raw rows, uhc_load_clips_smpl builds the records on the GPU).  Both on a precision-32 engine.

Inputs: synthetic smooth SMPL sequences, seeded (tests/motion_cases.py smooth_pose / smooth_trans: three sinusoids per axis-angle column,
upright root, slow root walk).  Sets: the 12 288 clip lengths of scripts/eval_time.py (round(exp(N(log 45, 0.8))) clipped to [8, 600]), and
32 long clips of 1 500 .. 3 000 frames.  Each path is warmed up on 64 clips first; the timed window is host clock around work that ends in a
device synchronise.  The host path runs once per set (it takes minutes), the device path three times.  In the same run both tables are read
back (uhc_get_clip_frames, in chunks) and compared: max |diff| and the fraction of bit-equal elements.  The GPU name and power limit are read
in the same run.

    python scripts/motion_lib_time.py [OUT.json]      (one JSON document to OUT.json and stdout)
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)


def clip_set(kind, seed=0):
    from tests.motion_cases import smooth_pose, smooth_trans
    rng = np.random.RandomState(seed)
    if kind == "eval_time_12288":
        lens = np.clip(np.round(np.exp(rng.normal(np.log(45.0), 0.8, 12288))), 8, 600).astype(int)
    else:
        lens = rng.randint(1500, 3001, 32)
    g = np.random.default_rng(seed)
    return [smooth_pose(int(T), g) for T in lens], [smooth_trans(int(T), g) for T in lens], lens


def host_path(eng, pose, trans):
    from uhc_b200 import motion_lib as ML
    t0 = time.time()
    experts = [ML.make_expert(p, t) for p, t in zip(pose, trans)]
    t1 = time.time()
    eng.load_clips(experts)
    eng.torch.cuda.synchronize()
    t2 = time.time()
    return dict(make_expert_s=t1 - t0, pack_and_load_clips_s=t2 - t1, total_s=t2 - t0)


def device_path(eng, pose, trans):
    t0 = time.time()
    eng.load_smpl_clips(pose, trans)
    eng.torch.cuda.synchronize()
    return dict(total_s=time.time() - t0)


def compare(a, b, total, chunk=65536):
    mx, eq = 0.0, 0
    for f0 in range(0, total, chunk):
        n = min(chunk, total - f0)
        x, y = a.get_clip_frames(f0, n), b.get_clip_frames(f0, n)
        mx = max(mx, float(np.abs(x - y).max()))
        eq += int((x == y).sum())
    return dict(max_abs_diff=mx, bit_equal_fraction=eq / float(total * 576), elements=total * 576)


def main():
    import torch
    from uhc_b200.engine import Engine
    out_path = os.path.abspath(sys.argv[1]) if len(sys.argv) > 1 else None
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["clocks_max_sm_mhz"] = float(q[0]), float(q[1])
    except Exception as ex:      # the numbers are reported as not measured
        out["power_limit_w"] = out["clocks_max_sm_mhz"] = "not measured (%s)" % ex
    host_eng, dev_eng = Engine(16, precision=32), Engine(16, precision=32)
    wp, wt, _ = clip_set("eval_time_12288", seed=1)
    host_path(host_eng, wp[:64], wt[:64])
    device_path(dev_eng, wp[:64], wt[:64])
    sets = []
    for kind in ("eval_time_12288", "long_32"):
        pose, trans, lens = clip_set(kind)
        s = dict(set=kind, clips=len(lens), total_frames=int(lens.sum()), mean_len=float(lens.mean()), max_len=int(lens.max()),
                 upload_bytes=dict(host_path=int(lens.sum()) * 576 * 4, device_path=int(lens.sum()) * (72 + 3) * 8))
        s["device"] = [device_path(dev_eng, pose, trans) for _ in range(3)]
        s["host"] = host_path(host_eng, pose, trans)
        s["device"].append(device_path(dev_eng, pose, trans))
        s["tables"] = compare(host_eng, dev_eng, int(lens.sum()))
        s["speedup_host_over_best_device"] = s["host"]["total_s"] / min(r["total_s"] for r in s["device"])
        print(json.dumps(s), flush=True)
        sets.append(s)
    out["sets"] = sets
    out["note"] = ("precision-32 engines; wall seconds, host clock around work ending in a device synchronise; the device path includes the "
                   "host concatenation of the rows and their upload; make_expert is single-threaded numpy on the GPU host's CPU")
    txt = json.dumps(out, indent=1)
    if out_path:
        with open(out_path, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
