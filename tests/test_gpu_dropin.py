"""GPU: the drop-in boundary end to end -- the statement sequence of the reference's scripts/train_uhc.py:49-97 and
scripts/eval_uhc.py:62-103 executed against this repo's `uhc` package."""
import os
import pickle
import types

import numpy as np
import pytest

from tests.helpers import write_synthetic_pkl

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _float64_default():
    """the reference's scripts run everything under torch.set_default_dtype(torch.float64) (scripts/train_uhc.py:80-81, eval_uhc.py:94-95):
    every implicit-dtype allocation of the drop-in package must survive that"""
    import torch
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(old)


def _cfg(tmp_path, monkeypatch, cfg_file="uhc_b200_default.yml"):
    import yaml
    monkeypatch.chdir(tmp_path)
    from uhc.utils.config_utils.copycat_config import Config
    base = yaml.safe_load(open(os.path.join(os.path.dirname(__file__), "..", "config", cfg_file)))
    base.update(policy_hsize=[128, 64], value_hsize=[128, 64], min_batch_size=1024, num_optim_epoch=2, num_envs=64, save_n_epochs=2, num_epoch=2)
    base["data_specs"]["file_path"] = write_synthetic_pkl(str(tmp_path / "sample_data" / "clips.pkl"))
    base["data_specs"]["t_max"] = 40
    cfg = Config(cfg_id="dropin_test", create_dirs=True, cfg_dict=base)
    cfg.update(types.SimpleNamespace(cfg="dropin_test", render=False, test=False, num_threads=30, gpu_index=0, epoch=0, show_noise=False,
                                     resume=None, no_log=True, debug=False, full_eval=False))
    return cfg


@pytest.mark.parametrize("cfg_file", ["uhc_b200_default.yml", "uhc_b200_explicit.yml", "uhc_b200_implicit.yml"])     # the three configs of config/release/
def test_train_script_sequence(tmp_path, monkeypatch, cfg_file):
    import torch
    from uhc.agents import agent_dict
    from uhc.utils.flags import flags
    cfg = _cfg(tmp_path, monkeypatch, cfg_file)
    flags.debug = False
    dtype = torch.float64
    device = torch.device("cuda", index=0)
    np.random.seed(cfg.seed)
    torch.manual_seed(cfg.seed)
    agent = agent_dict[cfg.agent_name](cfg, dtype, device, training=True, checkpoint_epoch=0)
    assert agent.action_dim == {"uhc_b200_default.yml": 105, "uhc_b200_explicit.yml": 315, "uhc_b200_implicit.yml": 75}[cfg_file]
    assert agent.state_dim == (784 if "implicit.yml" in cfg_file else 657)
    for i_iter in range(0, cfg.num_epoch):
        info = agent.optimize_policy(i_iter)
        assert info["log"]["num_steps"] >= cfg.min_batch_size and np.isfinite(info["log"]["avg_reward"])
    ck = os.path.join(cfg.model_dir, "iter_0002.p")          # (epoch + 1) % save_n_epochs == 0 -> agent_copycat.py:346-349
    assert os.path.exists(ck)
    cp = pickle.load(open(ck, "rb"))
    assert set(cp) == {"policy_dict", "value_dict", "running_state"}
    assert ("nets.0.0.affine_layers.0.weight" if "implicit.yml" in cfg_file else "net.affine_layers.0.weight") in cp["policy_dict"] and "value_head.bias" in cp["value_dict"]
    # eval_uhc.py --mode stats: resume from the checkpoint and evaluate every clip deterministically
    agent2 = agent_dict[cfg.agent_name](cfg, dtype, device, training=True, checkpoint_epoch=2)
    res = agent2.eval_policy(epoch=2, dump=True)
    m = res[0][f"coverage_{agent2.data_loader.name}"]
    assert 0.0 <= m["mean_coverage"] <= 1.0 and m["all_coverage"] == 3 and np.isfinite(m["mpjpe_g"])
    assert os.path.exists(os.path.join(cfg.output_dir, f"2_{agent2.data_loader.name}_coverage_full.pkl"))


def test_single_env_facade_matches_engine_and_oracle(tmp_path, monkeypatch, golden_dir):
    """HumanoidEnv.reset/step (numpy in / numpy out, float64) against the CPU oracle on a golden clip."""
    from oracle import oracle as O
    from uhc.envs.humanoid_im import HumanoidEnv
    from uhc.losses.reward_function import reward_func
    cfg = _cfg(tmp_path, monkeypatch)
    z = np.load(os.path.join(golden_dir, "expert_sway.npz"))
    pose = np.concatenate([z["pose_aa"][:, :66], np.zeros((len(z["pose_aa"]), 6))], 1)
    seq = {"pose_aa": pose, "trans": z["trans"], "beta": z["beta"], "gender": z["gender"], "seq_name": "sway"}
    env = HumanoidEnv(cfg, seq, cfg.data_specs, mode="train")
    obs = env.reset()
    assert obs.shape == (657,) and obs.dtype == np.float64 and env.action_space.shape == (105,)
    oe = O.Env(O.Model(), env.expert, np.concatenate([z["beta"][0], [z["gender"][0]]]))
    o0 = oe.reset()
    assert np.abs(o0 - obs).max() < 1e-4
    rng = np.random.RandomState(0)
    for t in range(5):
        a = rng.normal(0, 0.1, 105)
        ob, r, done, info = env.step(a)
        oo, ro, do, io = oe.step(a)
        cr, ci = reward_func["world_rfc_implicit"](env, None, a, info)
        assert r == 1.0 and done == do and info["fail"] == io["fail"] and abs(info["percent"] - io["percent"]) < 1e-6
        assert np.abs(ob - oo).max() < 2e-3 and abs(cr - ro) < 1e-3 and np.abs(ci - io["c_info"]).max() < 2e-3
        assert abs(env.calc_body_diff() - oe.body_diff()) < 1e-4
        # getters of the reference surface (humanoid_im.py:910-965, :1198): end effectors, Pelvis COM, previous body quats
        assert np.abs(env.get_com() - oe.d.xipos[:3]).max() < 1e-4
        ee = env.get_ee_pos(None).reshape(5, 3)
        assert np.abs(ee - oe.d.xpos.reshape(24, 3)[env.model_tables.ee]).max() < 1e-4
        assert env.get_ee_pos("heading").shape == (15,) and env.prev_bquat.shape == (96,)
        assert np.abs(env.data.qpos - oe.d.qpos).max() < 1e-4 and len(env.model.actuator_names) == 69
    env.fail_safe()
    assert np.abs(env.get_humanoid_qpos() - env.get_expert_qpos()).max() < 1e-6


def test_reference_script_files_run_against_this_package(tmp_path, golden_dir):
    """The reference's scripts/train_uhc.py, then scripts/eval_uhc.py --mode stats, as they run with cwd = a scratch copy of this repo's
    config/assets layout (`sys.path.append(os.getcwd())`, train_uhc.py:24, resolves `uhc` to this package): every name they import from `uhc`
    (tests/golden/reference_script_imports.json, recorded from the unmodified script files, tools/make_golden.py compat) resolves there, Config finds
    the yaml by id under the cwd, training writes the epoch-2 checkpoint under results/ and the evaluation (on the device the eval script passes,
    the CPU one, eval_uhc.py:84-90) resumes from it."""
    import subprocess
    import sys
    import yaml
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    for d in ("uhc", "uhc_b200", "mujoco_py", "assets"):
        if os.path.exists(os.path.join(root, d)):
            os.symlink(os.path.join(root, d), tmp_path / d)
    os.makedirs(tmp_path / "config")
    base = yaml.safe_load(open(os.path.join(root, "config", "uhc_b200_default.yml")))
    base.update(policy_hsize=[128, 64], value_hsize=[128, 64], min_batch_size=1024, num_optim_epoch=2, num_envs=64, save_n_epochs=2, num_epoch=2)
    base["data_specs"]["file_path"] = write_synthetic_pkl(str(tmp_path / "sample_data" / "clips.pkl"))
    base["data_specs"]["t_max"] = 40
    yaml.safe_dump(base, open(tmp_path / "config" / "refscript.yml", "w"))
    args = dict(cfg="refscript", test=False, num_threads=30, gpu_index=0, show_noise=False, resume=None, no_log=True, debug=False)
    code = f"""
import importlib, json, os, sys, types
sys.path.append(os.getcwd())
for script, imports in json.load(open({os.path.join(golden_dir, "reference_script_imports.json")!r})).items():
    for module, names in imports:
        m = importlib.import_module(module)
        assert m.__file__.startswith(os.getcwd()), m.__file__
        for n in names:
            assert hasattr(m, n), (script, module, n)
import numpy as np, torch
from uhc.utils.flags import flags
from uhc.utils.config_utils.copycat_config import Config
from uhc.agents import agent_dict
from uhc.agents.agent_copycat import AgentCopycat
cfg = Config(cfg_id="refscript", create_dirs=True)
cfg.update(types.SimpleNamespace(render=False, epoch=0, full_eval=False, **{args!r}))
flags.debug = False
torch.set_default_dtype(torch.float64)
torch.cuda.set_device(0)
np.random.seed(cfg.seed); torch.manual_seed(cfg.seed)
agent = agent_dict[cfg.agent_name](cfg, torch.float64, torch.device("cuda", index=0), training=True, checkpoint_epoch=0)
for i_iter in range(0, cfg.num_epoch):
    agent.optimize_policy(i_iter)
    torch.cuda.empty_cache()
print("training done!")
cfg = Config(cfg_id="refscript", create_dirs=False)
cfg.update(types.SimpleNamespace(epoch=2, data={str(tmp_path / "sample_data" / "clips.pkl")!r}, mode="stats", render=False, **{args!r}))
cfg.no_log = True
cfg.output = os.path.join("results/renderings/uhc/", cfg.id)
os.makedirs(cfg.output, exist_ok=True)
cfg.data_specs["file_path"] = cfg.data
cfg.data_specs.pop("test_file_path", None)
np.random.seed(cfg.seed); torch.manual_seed(cfg.seed)
AgentCopycat(cfg, torch.float64, torch.device("cpu"), training=True, checkpoint_epoch=2).eval_policy(epoch=2, dump=True)
"""
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    r = subprocess.run([sys.executable, "-c", code], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "training done!" in r.stdout, r.stderr[-3000:]
    assert os.path.exists(tmp_path / "results" / "motion_im" / "refscript" / "models" / "iter_0002.p")
