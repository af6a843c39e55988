"""CPU: the checkpoint wire format (agent_copycat.py:190-201, :249-260).  `running_state` is a pickled
uhc.khrylib.utils.zfilter.ZFilter; a file written by this repo must load into the REFERENCE's class and a file written by the reference
must load here.  The cross-checks against the reference compare with what its own code wrote (tests/golden, tools/make_golden.py compat)."""
import io
import os
import pickle
import subprocess
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_host_zfilter_matches_running_statistics():
    from uhc.khrylib.utils.zfilter import ZFilter
    rng = np.random.RandomState(0)
    x = rng.normal(1.0, 2.0, (50, 6))
    z = ZFilter((6,), clip=5)
    ys = [z(r) for r in x[:10]]                          # per-sample pushes (the reference's use) ...
    z(x[10:])                                            # ... and one batch merge give the statistics of all 50 rows
    assert z.rs.n == 50 and np.allclose(z.rs.mean, x.mean(0)) and np.allclose(z.rs.var, x.var(0, ddof=1))
    assert np.allclose(ys[0], 0.0)                       # first sample: (x - x) / (|x| + eps)
    z2 = ZFilter.from_stats(50, x.mean(0), ((x - x.mean(0)) ** 2).sum(0), clip=5.0)
    assert np.allclose(z2(x[3], update=False), z(x[3], update=False))
    z3 = pickle.loads(pickle.dumps(z2))
    assert z3.rs._n == 50 and np.allclose(z3.rs._M, z2.rs._M) and np.allclose(z3.rs._S, z2.rs._S) and z3.clip == 5.0


class _ClassRecorder(pickle.Unpickler):
    """unpickles into this repo's classes and records the ones from `uhc` the file names"""
    def find_class(self, module, name):
        if module.split(".")[0] == "uhc":
            self.names.add((module, name))
        return super().find_class(module, name)


def _classes(data):
    u = _ClassRecorder(io.BytesIO(data))
    u.names = set()
    return u.load(), u.names


def _layout(o):
    """attribute names, recursively through the `uhc` objects"""
    return {k: _layout(v) if type(v).__module__.split(".")[0] == "uhc" else None for k, v in vars(o).items()}


def test_running_state_round_trips_through_the_reference_class(golden_dir):
    """tests/golden/zfilter_roundtrip.npz (tools/make_golden.py compat): a running_state pickled by the reference's own ZFilter, and what the
    reference's ZFilter computed after loading this repo's pickle of the same statistics.  Ours must name the same classes with the same
    attribute layout (so that it loads into the reference's), normalise as the reference did, and the reference's file must load here."""
    from uhc.khrylib.utils.zfilter import ZFilter
    g = np.load(os.path.join(golden_dir, "zfilter_roundtrip.npz"))
    x = np.random.RandomState(1).normal(0.5, 3.0, (40, 657))
    ours = ZFilter.from_stats(40, x.mean(0), ((x - x.mean(0)) ** 2).sum(0), clip=5.0)
    ours_back, ours_names = _classes(pickle.dumps({"running_state": ours}))
    theirs, their_names = _classes(g["ref_pickle"].tobytes())
    assert their_names == {("uhc.khrylib.utils.zfilter", "ZFilter"), ("uhc.khrylib.utils.zfilter", "RunningStat")} and ours_names == their_names
    theirs = theirs["running_state"]                                  # unpickles into this repo's stand-in (same module path)
    assert _layout(ours_back["running_state"]) == _layout(theirs)
    assert np.allclose(g["y_ref_from_ours"], ours(x[0], update=False))
    assert type(theirs).__module__ == "uhc.khrylib.utils.zfilter" and theirs.rs._n == 40
    assert np.allclose(theirs.rs._M, x.mean(0)) and np.allclose(theirs.rs._S, ((x - x.mean(0)) ** 2).sum(0))


def test_reference_train_script_file_reaches_the_agent_on_this_package(tmp_path, golden_dir):
    """What the reference's OWN scripts/train_uhc.py and scripts/eval_uhc.py import from `uhc` (tests/golden/reference_script_imports.json, recorded by
    running the unmodified script files against this package, tools/make_golden.py compat) resolves against a tree holding this repo's `uhc`
    package and config layout, put on sys.path as the scripts do (train_uhc.py:24 appends the cwd).  Without a GPU the script's sequence
    -- Config by id from the cwd, torch.set_default_dtype(float64), agent_dict[cfg.agent_name] -- must stop exactly where AgentCopycat asks for
    a CUDA device.  (With a GPU the same sequence trains: tests/test_gpu_dropin.py.)"""
    import yaml
    from tests.helpers import write_synthetic_pkl
    for d in ("uhc", "uhc_b200", "mujoco_py", "assets"):
        if os.path.exists(os.path.join(ROOT, d)):
            os.symlink(os.path.join(ROOT, d), tmp_path / d)
    os.makedirs(tmp_path / "config")
    base = yaml.safe_load(open(os.path.join(ROOT, "config", "uhc_b200_default.yml")))
    base.update(policy_hsize=[64], value_hsize=[64], min_batch_size=256, num_optim_epoch=1, num_envs=8, num_epoch=1)
    base["data_specs"]["file_path"] = write_synthetic_pkl(str(tmp_path / "sample_data" / "clips.pkl"))
    yaml.safe_dump(base, open(tmp_path / "config" / "refscript.yml", "w"))
    code = f"""
import importlib, json, os, sys
sys.path.append(os.getcwd())
for script, imports in json.load(open({os.path.join(golden_dir, "reference_script_imports.json")!r})).items():
    for module, names in imports:
        m = importlib.import_module(module)
        assert m.__file__.startswith(os.getcwd()), m.__file__
        for n in names:
            assert hasattr(m, n), (script, module, n)
import torch
from uhc.utils.config_utils.copycat_config import Config
from uhc.agents import agent_dict
cfg = Config(cfg_id="refscript", create_dirs=True)
assert cfg.get("num_envs") == 8 and os.path.isdir("results/motion_im/refscript/models")
torch.set_default_dtype(torch.float64)
agent_dict[cfg.agent_name](cfg, torch.float64, torch.device("cpu"), training=True, checkpoint_epoch=0)
"""
    env = dict({k: v for k, v in os.environ.items() if k != "PYTHONPATH"}, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "needs a CUDA device" in r.stderr, r.stderr[-3000:]
