"""MyoSuite 1.2.3 envs/myo/reach_v0.py ``ReachEnvV0``, restated from memory ([3P-MEM], SURVEY.md). No file of the reference
builds on it: what the reach fixtures pin is this restatement, run over the fp64 oracle, not MyoSuite itself."""
import collections

import gym
import numpy as np

from myosuite.envs.myo.base_v0 import BaseV0


class ReachEnvV0(BaseV0):
    DEFAULT_OBS_KEYS = ["qpos", "qvel", "tip_pos", "reach_err"]
    DEFAULT_RWD_KEYS_AND_WEIGHTS = {"reach": 1.0, "bonus": 4.0, "penalty": 50}

    def __init__(self, model_path, obsd_model_path=None, seed=None, **kwargs):
        gym.utils.EzPickle.__init__(self, model_path, obsd_model_path, seed, **kwargs)
        super().__init__(model_path=model_path, obsd_model_path=obsd_model_path, seed=seed)
        self._setup(**kwargs)

    def _setup(self, target_reach_range, far_th=.35, obs_keys=DEFAULT_OBS_KEYS, weighted_reward_keys=DEFAULT_RWD_KEYS_AND_WEIGHTS,
               **kwargs):
        self.far_th = far_th
        self.target_reach_range = target_reach_range
        super()._setup(obs_keys=obs_keys, weighted_reward_keys=weighted_reward_keys, sites=self.target_reach_range.keys(), **kwargs)

    def get_obs_dict(self, sim):
        obs_dict = {}
        obs_dict["t"] = np.array([sim.data.time])
        obs_dict["qpos"] = sim.data.qpos[:].copy()
        obs_dict["qvel"] = sim.data.qvel[:].copy() * self.dt
        if sim.model.na > 0:
            obs_dict["act"] = sim.data.act[:].copy()
        obs_dict["tip_pos"] = np.array([])
        obs_dict["target_pos"] = np.array([])
        for isite in range(len(self.tip_sids)):
            obs_dict["tip_pos"] = np.append(obs_dict["tip_pos"], sim.data.site_xpos[self.tip_sids[isite]].copy())
            obs_dict["target_pos"] = np.append(obs_dict["target_pos"], sim.data.site_xpos[self.target_sids[isite]].copy())
        obs_dict["reach_err"] = np.array(obs_dict["target_pos"]) - np.array(obs_dict["tip_pos"])
        return obs_dict

    def get_reward_dict(self, obs_dict):
        reach_dist = np.linalg.norm(obs_dict["reach_err"], axis=-1)
        act_mag = np.linalg.norm(self.obs_dict["act"], axis=-1) / self.sim.model.na if self.sim.model.na != 0 else 0
        far_th = self.far_th * len(self.tip_sids) if np.squeeze(obs_dict["t"]) > 2 * self.dt else np.inf
        near_th = len(self.tip_sids) * .0125
        rwd_dict = collections.OrderedDict((
            ("reach", -1. * reach_dist),
            ("bonus", 1. * (reach_dist < 2 * near_th) + 1. * (reach_dist < near_th)),
            ("act_reg", -1. * act_mag),
            ("penalty", -1. * (reach_dist > far_th)),
            ("sparse", -1. * reach_dist),
            ("solved", reach_dist < near_th),
            ("done", reach_dist > far_th),
        ))
        rwd_dict["dense"] = np.sum([wt * rwd_dict[key] for key, wt in self.rwd_keys_wt.items()], axis=0)
        return rwd_dict

    def generate_target_pose(self):
        for site, span in self.target_reach_range.items():
            sid = self.sim.model.site_name2id(site + "_target")
            self.sim.model.site_pos[sid] = self.np_random.uniform(low=span[0], high=span[1])
        self.sim.forward()

    def reset(self):
        self.generate_target_pose()
        self.robot.sync_sims(self.sim, self.sim_obsd)
        return super().reset()
