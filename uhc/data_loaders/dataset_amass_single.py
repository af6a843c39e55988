"""DatasetAMASSSingle of the reference (uhc/data_loaders/dataset_amass_single.py:27-253): same pickle schema
{key: {pose_aa, pose_6d, trans, beta, gender, ...}}, same filtering (len >= t_min + 1), same sampling rules; in addition it
precomputes the expert tables of every clip once (uhc_b200.motion_lib) instead of once per episode.  With motion_lib="device" the engine builds
the tables from the raw sequences (smpl_clips(), Engine.load_smpl_clips) and the host tables are computed only if `experts` is read."""
import random

import joblib
import numpy as np

from uhc_b200 import motion_lib


def _gender_code(g):
    g = g.item() if isinstance(g, np.ndarray) else g
    if isinstance(g, bytes):
        g = g.decode("utf-8")
    return {"neutral": 0, "male": 1, "female": 2}[g]


class DatasetAMASSSingle:
    def __init__(self, data_specs, data_mode="train", model=None, motion_lib="host"):
        np.random.seed(0)
        random.seed(0)
        self.data_root = data_specs["file_path"] if data_mode == "train" else data_specs["test_file_path"]
        self.data_specs = data_specs
        self.t_min, self.t_max = data_specs.get("t_min", 90), data_specs.get("t_max", -1)
        self.name = self.data_root.split("/")[-1]
        self.pickle_data = joblib.load(open(self.data_root, "rb"))
        self.data_mode = data_mode
        self.data, self.data_keys, self.sample_keys = {"pose_aa": {}, "trans": {}, "beta": {}, "gender": {}}, [], []
        for k, v in self.pickle_data.items():
            n = v["pose_aa"].shape[0]
            if n < self.t_min + 1:
                continue
            self.data["pose_aa"][k] = v["pose_aa"]
            self.data["trans"][k] = v["trans"] if v["trans"].shape[0] == n else v["qpos"][:, :3]
            beta = np.repeat(v["beta"][None], n, axis=0) if v["beta"].shape[0] != n else v["beta"]
            if beta.shape[1] != 16:
                beta = np.concatenate([beta, np.zeros((n, 16 - beta.shape[1]))], axis=1)
            self.data["beta"][k] = beta
            self.data["gender"][k] = np.repeat([_gender_code(v["gender"])], n, axis=0)
            self.data_keys.append(k)
            reps = n // self.t_max + 1 if self.t_max != -1 else 1
            self.sample_keys += [(k, [-1])] * reps
        self.seq_len = len(self.data_keys)
        self.curr_key = ""
        self.shapes = [np.concatenate([self.data["beta"][k][0], [self.data["gender"][k][0]]]) for k in self.data_keys]
        assert motion_lib in ("host", "device"), "motion_lib: host | device"
        self._model, self._experts = model, None
        if motion_lib == "host":
            self._experts = self._make_experts()

    def _make_experts(self):
        # expert tables of every clip, once (humanoid_im.py:182-215 does this per episode)
        return [motion_lib.make_expert(self.data["pose_aa"][k], self.data["trans"][k], self._model) for k in self.data_keys]

    @property
    def experts(self):
        if self._experts is None:
            self._experts = self._make_experts()
        return self._experts

    def smpl_clips(self):
        """the raw sequences of every clip in data_keys order, as BatchedAgent / Engine.load_smpl_clips take them"""
        return {"pose_aa": [self.data["pose_aa"][k] for k in self.data_keys], "trans": [self.data["trans"][k] for k in self.data_keys]}

    def get_len(self):
        return self.seq_len

    def get_sample_len_from_key(self, take_key):
        return self.data["pose_aa"][take_key].shape[0]

    def sample_seq(self, full_sample=False, freq_dict=None, sampling_temp=0.2, sampling_freq=0.5, precision_mode=False):
        self.curr_key = random.choice(self.sample_keys)[0]
        return self.get_sample_from_key(self.curr_key, full_sample=full_sample)

    def get_sample_from_key(self, take_key, full_sample=False, freq_dict=None, fr_start=-1, precision_mode=False, sampling_freq=0.75):
        self.curr_key = take_key
        n = self.data["pose_aa"][take_key].shape[0]
        if full_sample:
            fr_start, fr_end = 0, n
        else:
            if fr_start == -1:
                fr_start = np.random.randint(0, n - self.t_min)
            fr_end = fr_start + self.t_max if (fr_start + self.t_max < n and self.t_max != -1) else n
        self.fr_start, self.fr_end = fr_start, fr_end
        s = {k: self.data[k][take_key][fr_start:fr_end] for k in ("pose_aa", "trans", "beta", "gender")}
        s.update(seq_name=take_key, has_obj=False, num_obj=0, obj_pose=s["pose_aa"], clip_index=self.data_keys.index(take_key),
                 fr_start=fr_start)
        return s
