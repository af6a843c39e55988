"""CPU: the metric stage of uhc_evaluate (uhc_b200/csrc/eval_metrics.h, compiled for the host with g++) against outputs of the reference's own
smpl_eval.compute_metrics (tests/golden/metrics.npz), within the tolerance tests/test_metrics.py holds uhc_b200.metrics to."""
import ctypes as C
import os
import subprocess

import numpy as np

from uhc_b200.agent import EVAL_METRICS

HERE = os.path.dirname(os.path.abspath(__file__))


def _lib(tmp_path):
    so = str(tmp_path / "libeval_metrics_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so, os.path.join(HERE, "emu", "eval_metrics_host.cpp")])
    return C.CDLL(so)


def frame_metrics_host(lib, pred, gt, pred_jpos, gt_jpos):
    a = [np.ascontiguousarray(x, dtype=np.float64) for x in (pred, gt, pred_jpos, gt_jpos)]
    T = len(a[0])
    out = np.full((T, 6), -1.0)
    p = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))
    lib.eval_metrics_host(p(a[0]), p(a[1]), p(a[2]), p(a[3]), C.c_int(T), p(out))
    return out


def test_eval_metric_header_matches_reference(tmp_path, golden_dir):
    lib = _lib(tmp_path)
    g = np.load(os.path.join(golden_dir, "metrics.npz"))
    for tag in ("a", "b"):
        fm = frame_metrics_host(lib, *(g[f"{tag}.in.{k}"] for k in ("pred", "gt", "pred_jpos", "gt_jpos")))
        T = len(fm)
        got = dict(zip(EVAL_METRICS, fm.T))
        got["vel_dist"], got["accel_dist"] = got["vel_dist"][1:], got["accel_dist"][2:]      # vel from the 2nd row on, accel from the 3rd
        assert np.isnan(fm[0, 4]) and np.isnan(fm[:2, 5]).all() and np.isfinite(fm[:, :4]).all()
        for k in EVAL_METRICS:
            ref = g[f"{tag}.out.{k}"]
            assert got[k].shape == ref.shape, (tag, k, got[k].shape, ref.shape)
            assert np.abs(got[k] - ref).max() < 1e-8 * max(1.0, np.abs(ref).max()), (tag, k, np.abs(got[k] - ref).max())
        # the drop-in's success rule on these rows: the clip end reached without failure (percent == 1, no fail_safe re-seat)
        succ = T >= 3 and float(g[f"{tag}.in.percent"]) == 1 and not bool(g[f"{tag}.in.fail_safe"])
        assert succ == bool(g[f"{tag}.out.succ"][0])


def test_procrustes_handles_reflections_and_degenerate_sets(tmp_path):
    """the 3x3 SVD path against numpy on random frames, a mirrored prediction (reflection fix) and a planar joint set (rank 2)"""
    from uhc_b200.metrics import compute_metrics
    lib = _lib(tmp_path)
    rng = np.random.RandomState(3)
    T = 6
    gq = np.zeros((T, 76)); gq[:, 3] = 1.0
    gj = rng.normal(0, 0.4, (T, 24, 3))
    cases = {"random": gj + rng.normal(0, 0.05, gj.shape), "mirrored": gj * np.array([-1.0, 1.0, 1.0]), "planar": gj * np.array([1.0, 1.0, 0.0])}
    for name, pj in cases.items():
        gjj = gj * np.array([1.0, 1.0, 0.0]) if name == "planar" else gj
        fm = frame_metrics_host(lib, gq, gq, pj.reshape(T, 72), gjj.reshape(T, 72))
        ref = compute_metrics({"pred": gq, "gt": gq, "pred_jpos": pj.reshape(T, 72), "gt_jpos": gjj.reshape(T, 72), "percent": 1.0, "fail_safe": False})
        assert np.abs(fm[:, 3] - ref["pa_mpjpe"]).max() < 1e-8 * max(1.0, np.abs(ref["pa_mpjpe"]).max()), (name, fm[:, 3], ref["pa_mpjpe"])
