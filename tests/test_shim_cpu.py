"""CPU: the drop-in `uhc` package surface (SURVEY.md section 8b): Config defaults / schedules, dataset schema and sampling."""
import os

import numpy as np

from tests.helpers import write_synthetic_pkl


def test_config_defaults_and_schedules(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    from uhc.utils.config_utils.copycat_config import Config
    from uhc.utils.flags import flags
    cfg = Config(cfg_id="uhc_b200_default", create_dirs=False)
    assert cfg.policy_hsize == [2048, 1024, 512] and cfg.policy_htype == "gelu" and cfg.obs_v == 2 and cfg.meta_pd
    assert cfg.residual_force and cfg.residual_force_scale == 100 and cfg.residual_force_lim == 100.0       # copycat_config.py:106 default
    assert cfg.reward_id == "world_rfc_implicit" and cfg.env_term_body == "body" and cfg.fix_std and cfg.log_std == -2.3
    assert os.path.isdir(cfg.model_dir) and cfg.get("nonexistent", 7) == 7
    cfg.update_adaptive_params(10)
    assert cfg.adp_noise_rate == 1.0 and cfg.adp_policy_lr == 5e-5 and cfg.adp_log_std == -2.3

    import types
    cfg.update(types.SimpleNamespace(num_threads=3, no_log=True))
    assert cfg.num_threads == 3 and cfg.no_log is True
    flags.debug = True
    assert flags.debug


def test_adaptive_schedule_interpolates(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    from uhc.utils.config_utils.copycat_config import Config
    import yaml
    base = yaml.safe_load(open(os.path.join(os.path.dirname(__file__), "..", "config", "uhc_b200_default.yml")))
    base.update(adp_iter_cp=[0, 100], adp_noise_rate_cp=[1.0, 0.0], adp_policy_lr_cp=[5e-5, 1e-5])
    cfg = Config(cfg_id="x", cfg_dict=base)
    cfg.update_adaptive_params(50)
    assert abs(cfg.adp_noise_rate - 0.5) < 1e-12 and abs(cfg.adp_policy_lr - 3e-5) < 1e-12
    cfg.update_adaptive_params(500)
    assert cfg.adp_noise_rate == 0.0


def test_dataset_schema_and_sampling(tmp_path):
    from uhc.data_loaders.dataset_amass_single import DatasetAMASSSingle
    p = write_synthetic_pkl(str(tmp_path / "sample_data" / "clips.pkl"))
    ds = DatasetAMASSSingle({"file_path": p, "t_min": 5, "t_max": 60})
    assert ds.get_len() == 3 and len(ds.experts) == 3
    for ex, k in zip(ds.experts, ds.data_keys):
        T = ds.get_sample_len_from_key(k)
        assert ex["qpos"].shape == (T, 76) and ex["wbpos"].shape == (T, 72) and ex["bangvel"].shape == (T, 72)
    s = ds.sample_seq()
    assert s["pose_aa"].shape[0] <= 60 and s["beta"].shape[1] == 16 and s["seq_name"] in ds.data_keys
    full = ds.get_sample_from_key(ds.data_keys[1], full_sample=True)
    assert full["pose_aa"].shape[0] == ds.get_sample_len_from_key(ds.data_keys[1]) and full["gender"][0] == 1


def _cfg_view(d):
    """what supported_variant reads from a Config, built from a yaml dict with copycat_config.py's defaults"""
    import types
    return types.SimpleNamespace(get=d.get, obs_v=d.get("obs_v", 0), actor_type=d.get("actor_type", "gauss"), reward_id=d.get("reward_id", "quat"),
                                 fix_std=d.get("fix_std", False), residual_force=d.get("residual_force", False))


def test_supported_variant_accepts_the_shipped_configs_and_names_what_it_refuses():
    import glob
    import yaml
    from uhc.agents.agent_copycat import supported_variant
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "config")
    modes = {}
    for f in sorted(glob.glob(os.path.join(here, "*.yml"))):
        modes[os.path.basename(f)] = supported_variant(_cfg_view(yaml.safe_load(open(f))))
    assert modes["uhc_b200_default.yml"] == "implicit" and modes["uhc_b200_explicit.yml"] == "explicit" and modes["uhc_b200_implicit.yml"] == "implicit"
    base = yaml.safe_load(open(os.path.join(here, "uhc_b200_default.yml")))
    for key, val, word in (("obs_v", 4, "obs_v"), ("fix_std", False, "log_std"), ("env_term_body", "head", "env_term_body"), ("reward_id", "world_rfc_implicit_v2", "obs_v"),
                           ("env_init_noise", 0.1, "env_init_noise"), ("obs_coord", "heading", "obs_coord")):
        d = dict(base); d[key] = val
        try:
            supported_variant(_cfg_view(d))
        except AssertionError as e:
            assert word in str(e), (key, str(e))
        else:
            raise AssertionError(f"{key} = {val!r} must be refused")
    for key, val in (("obs_v", 5), ("obs_v", 6), ("env_term_body", "root"), ("env_term_body", "Head"), ("reward_id", "world_rfc_implicit_v1_mul"), ("actor_type", "mcp")):
        d = dict(base); d[key] = val
        assert supported_variant(_cfg_view(d)) == "implicit"


def test_reference_yaml_coverage(golden_dir):
    """how many of the reference's own config files the drop-in accepts (tests/golden/reference_configs.json: the keys supported_variant reads, of
    each yaml under the reference's config/, tools/make_golden.py compat); the count is what DESIGN.md section 5 quotes"""
    import json
    from uhc.agents.agent_copycat import supported_variant
    views = json.load(open(os.path.join(golden_dir, "reference_configs.json")))
    accepted = 0
    for d in views.values():
        if d.get("agent_name", "agent_copycat") != "agent_copycat":
            continue
        try:
            supported_variant(_cfg_view(d)); accepted += 1
        except AssertionError:
            pass
    assert len(views) == 115 and accepted == 86, (len(views), accepted)
