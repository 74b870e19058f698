"""``MyoVecEnv``: thousands of worlds behind the SB3 ``VecEnv`` contract.

Replaces ``make_parallel_envs`` + ``SubprocVecEnv([...16 thunks])`` + ``Monitor``
(/root/reference/src/main_baoding.py:56-65,74) for the envs registered in
/root/reference/src/envs/__init__.py: one object, ``num_envs`` worlds stepped by one kernel launch,
auto-reset inside the step with ``terminal_observation`` / ``TimeLimit.truncated`` / ``episode`` infos
as the SubprocVecEnv worker and ``Monitor`` produce them.  ``VecNormalize``
(/root/reference/src/main_baoding.py:75) is the companion class below.

Two ways to call it:
* host arrays (``reset() / step_async(actions) / step_wait()``) - the SB3 signature, numpy in and out through
  pinned buffers;
* device tensors (``reset_device() / step_device(actions)``) - the same step without leaving the GPU, for a
  rollout whose policy also runs on the device.
"""
from __future__ import annotations

import time
from typing import Any, Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _capi
from .sim import BatchSim, Model


class Box:
    """Minimal ``gym.spaces.Box`` stand-in (gym is not a dependency): ``low``, ``high``, ``shape``, ``dtype``."""

    def __init__(self, low, high, shape, dtype=np.float32):
        self.low = np.full(shape, low, dtype=dtype)
        self.high = np.full(shape, high, dtype=dtype)
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)

    def sample(self, rng: Optional[np.random.Generator] = None):
        rng = rng or np.random.default_rng()
        return rng.uniform(self.low, self.high).astype(self.dtype)

    def __repr__(self):
        return f"Box({self.low.min()}, {self.high.max()}, {self.shape}, {self.dtype})"


class LazyInfos(Sequence):
    """``infos`` of one step. Dicts are built on access: 32k Python dicts per step would cost more than the
    physics. ``infos[i]`` carries the reward terms (``info.update(info["rwd_dict"])`` of
    /root/reference/src/envs/pose.py:103), ``solved``, and for finished episodes ``terminal_observation``,
    ``TimeLimit.truncated`` and Monitor's ``episode`` = {r, l, t}."""

    def __init__(self, keys, info, done, truncated, terminal_obs, ep_ret, ep_len, t0):
        self._keys, self._info, self._done, self._trunc = keys, info, done, truncated
        self._tobs, self._ret, self._len, self._t0 = terminal_obs, ep_ret, ep_len, t0

    def __len__(self):
        return len(self._done)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        row = self._info[i]
        rwd = {k: float(row[j]) for j, k in enumerate(self._keys) if k != "dense"}
        d: Dict[str, Any] = dict(rwd)
        d["rwd_dict"] = rwd
        d["rwd_dense"] = float(row[7])
        d["solved"] = bool(rwd["solved"])
        if self._done[i]:
            d["terminal_observation"] = self._tobs[i].copy()
            d["TimeLimit.truncated"] = bool(self._trunc[i])
            d["episode"] = {"r": float(self._ret[i]), "l": int(self._len[i]), "t": round(time.time() - self._t0, 6)}
        return d


BAODING_KEYS = ("pos_dist_1", "pos_dist_2", "act_reg", "alive", "sparse", "solved", "done")
POSE_KEYS = ("pose", "bonus", "penalty", "act_reg", "sparse", "solved", "done")
# CustomReorientEnv.get_reward_dict (/root/reference/src/envs/reorient.py:21-46); slot 7 is the dense reward in every task
REORIENT_KEYS = ("pos_dist", "rot_dist", "act_reg", "alive", "sparse", "solved", "done", "dense", "pos_dist_diff", "rot_dist_diff")
# MyoSuite ReachEnvV0.get_reward_dict [3P-MEM]
REACH_KEYS = ("reach", "bonus", "act_reg", "penalty", "sparse", "solved", "done")

# obs-dict entries of each task kind (get_obs_dict), numbered as the MYO_OBS_<KIND>_* ids of include/myo_b200.h: the keys `obs_keys`
# may list
OBS_KEYS = {
    _capi.TASK_BAODING: ("t", "hand_pos", "object1_pos", "object1_velp", "object2_pos", "object2_velp", "target1_pos", "target2_pos",
                         "target1_err", "target2_err", "act"),
    _capi.TASK_REORIENT: ("t", "hand_qpos", "hand_qvel", "obj_pos", "goal_pos", "pos_err", "obj_rot", "goal_rot", "rot_err", "act"),
    _capi.TASK_POSE: ("t", "qpos", "qvel", "act", "pose_err"),
    _capi.TASK_REACH: ("t", "qpos", "qvel", "act", "tip_pos", "target_pos", "reach_err"),
}
# DEFAULT_OBS_KEYS of BaodingEnvV1, ReorientEnvV0, PoseEnvV0 and ReachEnvV0 (MyoSuite 1.2.3): the layout of an env created without
# `obs_keys`, plus the "act" that BaseV0._setup appends for a model with activations
DEFAULT_OBS_KEYS = {
    _capi.TASK_BAODING: OBS_KEYS[_capi.TASK_BAODING][1:10],
    _capi.TASK_REORIENT: OBS_KEYS[_capi.TASK_REORIENT][1:9],
    _capi.TASK_POSE: ("qpos", "qvel", "pose_err"),
    _capi.TASK_REACH: ("qpos", "qvel", "tip_pos", "reach_err"),
}


class MyoVecEnv:
    """SB3 ``VecEnv``-shaped front end over ``BatchSim``."""

    def __init__(self, model: Model, cfg: _capi.TaskCfg, num_envs: int, device="cuda:0", seed: int = 0, lib=None):
        self.sim = BatchSim(model, num_envs, cfg, device=device, seed=seed)
        self.num_envs = int(num_envs)
        self.device = self.sim.device
        self.cfg = cfg
        self.observation_space = Box(-10.0, 10.0, (self.sim.nobs,), np.float32)
        self.action_space = Box(-1.0, 1.0, (self.sim.nu,), np.float32)
        keys = {_capi.TASK_BAODING: BAODING_KEYS, _capi.TASK_REORIENT: REORIENT_KEYS, _capi.TASK_REACH: REACH_KEYS,
                _capi.TASK_POSE: POSE_KEYS, _capi.TASK_NONE: POSE_KEYS}
        if cfg.kind not in keys:
            raise ValueError(f"no reward keys for task kind {cfg.kind}")
        self._keys = keys[cfg.kind]
        self.info_keys = tuple(self._keys)      # names of the columns of ``sim.info`` (the reward terms ``infos[i]`` carries)
        # the obs-dict entries the observation concatenates (None for a kind without keys)
        if cfg.n_obs_keys:
            self.obs_keys = tuple(OBS_KEYS[cfg.kind][cfg.obs_keys[i]] for i in range(cfg.n_obs_keys))
        elif cfg.kind in DEFAULT_OBS_KEYS:
            self.obs_keys = DEFAULT_OBS_KEYS[cfg.kind] + (("act",) if self.sim.na > 0 else ())
        else:
            self.obs_keys = None
        n, pin = self.num_envs, self.device.type == "cuda"
        self._h_act = torch.zeros(n, self.sim.nu, dtype=torch.float32, pin_memory=pin)
        self._h_obs = torch.zeros(n, self.sim.nobs, dtype=torch.float32, pin_memory=pin)
        self._h_tobs = torch.zeros(n, self.sim.nobs, dtype=torch.float32, pin_memory=pin)
        self._h_rew = torch.zeros(n, dtype=torch.float32, pin_memory=pin)
        self._h_done = torch.zeros(n, dtype=torch.uint8, pin_memory=pin)
        self._h_trunc = torch.zeros(n, dtype=torch.uint8, pin_memory=pin)
        self._h_info = torch.zeros(n, _capi.MYO_INFO_TERMS, dtype=torch.float32, pin_memory=pin)
        self._d_act = torch.zeros(n, self.sim.nu, dtype=torch.float32, device=self.device)
        # Monitor bookkeeping on the device: episode return / length
        self._ep_ret = torch.zeros(n, dtype=torch.float32, device=self.device)
        self._ep_len = torch.zeros(n, dtype=torch.int32, device=self.device)
        self._last_ret = torch.zeros(n, dtype=torch.float32, device=self.device)
        self._last_len = torch.zeros(n, dtype=torch.int32, device=self.device)
        self._t0 = time.time()
        self.h2d_bytes_per_step = self._h_act.numel() * 4
        self.d2h_bytes_per_step = (self._h_obs.numel() + self._h_rew.numel()) * 4 + self._h_done.numel()
        self._pending = False

    # -- device-resident API -------------------------------------------------------------------
    def reset_device(self) -> torch.Tensor:
        self._ep_ret.zero_(); self._ep_len.zero_()
        return self.sim.reset()

    def step_device(self, actions: torch.Tensor):
        """(obs, reward, done, truncated) as device tensors owned by the env (overwritten by the next step)."""
        return self.sim.step(actions)

    @property
    def terminal_obs(self) -> torch.Tensor:
        """Device tensor [n, obs_dim]: the last observation of the episode for worlds whose ``done`` is set this step
        (SB3's ``infos[i]["terminal_observation"]``)."""
        return self.sim.terminal_obs

    # -- SB3 VecEnv API --------------------------------------------------------------------------
    def reset(self) -> np.ndarray:
        obs = self.reset_device()
        self._h_obs.copy_(obs, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return self._h_obs.numpy().copy()

    def step_async(self, actions) -> None:
        a = torch.as_tensor(np.asarray(actions, dtype=np.float32))
        if tuple(a.shape) != (self.num_envs, self.sim.nu):
            raise ValueError(f"expected actions of shape {(self.num_envs, self.sim.nu)}, got {tuple(a.shape)}")
        self._h_act.copy_(a)
        self._d_act.copy_(self._h_act, non_blocking=True)
        obs, rew, done, trunc = self.sim.step(self._d_act)
        # Monitor: accumulate, latch the finished episodes' totals, clear
        self._ep_ret += rew
        self._ep_len += 1
        fin = done.bool()
        self._last_ret = torch.where(fin, self._ep_ret, self._last_ret)
        self._last_len = torch.where(fin, self._ep_len, self._last_len)
        self._ep_ret.masked_fill_(fin, 0.0)
        self._ep_len.masked_fill_(fin, 0)
        self._h_obs.copy_(obs, non_blocking=True)
        self._h_rew.copy_(rew, non_blocking=True)
        self._h_done.copy_(done, non_blocking=True)
        self._pending = True

    def step_wait(self, with_infos: bool = True):
        if not self._pending:
            raise RuntimeError("step_wait() without step_async()")
        self._pending = False
        infos: Any = None
        if with_infos:
            self._h_trunc.copy_(self.sim.truncated, non_blocking=True)
            self._h_info.copy_(self.sim.info, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        done = self._h_done.numpy().astype(bool)
        if with_infos:
            if done.any():
                self._h_tobs.copy_(self.sim.terminal_obs)
            infos = LazyInfos(self._keys, self._h_info.numpy().copy(), done, self._h_trunc.numpy().astype(bool), self._h_tobs.numpy().copy(),
                              self._last_ret.cpu().numpy(), self._last_len.cpu().numpy(), self._t0)
        return self._h_obs.numpy().copy(), self._h_rew.numpy().copy(), done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def get_attr(self, name: str, indices=None) -> List[Any]:
        n = self.num_envs if indices is None else len(list(indices))
        return [getattr(self, name)] * n

    def set_attr(self, name: str, value, indices=None) -> None:
        setattr(self, name, value)

    def env_method(self, method_name: str, *args, indices=None, **kwargs):
        return [getattr(self, method_name)(*args, **kwargs)]

    def seed(self, seed: Optional[int] = None):
        return [seed] * self.num_envs

    def close(self) -> None:
        self.sim.close()


class RunningMeanStd:
    """SB3 ``RunningMeanStd`` (Chan parallel-variance merge, initial count 1e-4), fp64 on the host."""

    def __init__(self, shape=(), epsilon: float = 1e-4):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = float(epsilon)

    def update_from_moments(self, batch_mean, batch_var, batch_count) -> None:
        delta = batch_mean - self.mean
        tot = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot
        m2 = self.var * self.count + batch_var * batch_count + np.square(delta) * self.count * batch_count / tot
        self.mean, self.var, self.count = new_mean, m2 / tot, tot

    def update(self, x: np.ndarray) -> None:
        self.update_from_moments(x.mean(axis=0), x.var(axis=0), x.shape[0])

    def update_distributed(self, x: np.ndarray, group=None) -> None:
        """Same update when the batch is sharded over ranks (worlds are sharded over GPUs, SURVEY.md 8e): the ranks
        all-reduce (count, sum, sum of squares) of their shards, so every rank applies the moments of the global batch
        and the statistics stay identical on all ranks. Falls back to ``update`` outside a process group."""
        import torch
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()):
            return self.update(x)
        x = np.asarray(x, np.float64).reshape(x.shape[0], -1)
        buf = torch.from_numpy(np.concatenate([[x.shape[0]], x.sum(0), np.square(x).sum(0)]))
        dist.all_reduce(buf, group=group)
        cnt = float(buf[0])
        d = x.shape[1]
        mean = buf[1:1 + d].numpy() / cnt
        var = buf[1 + d:].numpy() / cnt - np.square(mean)
        self.update_from_moments(mean.reshape(self.mean.shape), np.maximum(var, 0.0).reshape(self.var.shape), cnt)


def check_obs_width(obs_mean, nobs: int, path: str) -> None:
    """Observation statistics saved for one layout cannot normalise another (e.g. an env created with other ``obs_keys``)."""
    d = int(np.asarray(obs_mean).size)
    if d != int(nobs):
        raise ValueError(f"{path}: the saved observation statistics are {d} wide, the env's observations {int(nobs)}")


def rank_seed(base_seed: int, rank: int) -> int:
    """Seed of the worlds owned by ``rank``: world w of rank r draws from the stream (base + 1000 r, w, episode)."""
    return int(base_seed) + 1000 * int(rank)


class VecNormalize:
    """SB3 ``VecNormalize`` over a ``MyoVecEnv`` (host-array path): running obs / return moments,
    ``clip((x - mean) / sqrt(var + eps), +-clip)``, reward scaled by the std of the discounted return,
    ``terminal_observation`` normalised, ``returns[dones] = 0``  (SURVEY.md B.5;
    /root/reference/src/main_baoding.py:75, /root/reference/src/main_eval.py:65-67)."""

    def __init__(self, venv: MyoVecEnv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8):
        self.venv = venv
        self.num_envs = venv.num_envs
        self.observation_space, self.action_space = venv.observation_space, venv.action_space
        self.obs_rms = RunningMeanStd(venv.observation_space.shape)
        self.ret_rms = RunningMeanStd(())
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.returns = np.zeros(self.num_envs)
        self.old_obs = None
        self.old_reward = None

    @classmethod
    def from_moments(cls, venv, obs_mean, obs_var, obs_count, ret_mean=0.0, ret_var=1.0, ret_count=1e-4, **kw):
        """Rebuild from stored statistics (the content of an SB3 VecNormalize pickle such as the reference's env.pkl)."""
        v = cls(venv, **kw)
        v.obs_rms.mean, v.obs_rms.var, v.obs_rms.count = np.asarray(obs_mean, np.float64), np.asarray(obs_var, np.float64), float(obs_count)
        v.ret_rms.mean, v.ret_rms.var, v.ret_rms.count = float(ret_mean), float(ret_var), float(ret_count)
        return v

    @classmethod
    def load(cls, load_path: str, venv):
        """``VecNormalize.load(path, venv)`` on an SB3 pickle (e.g. the reference's ``env.pkl``)."""
        from . import checkpoint

        st = checkpoint.load_vecnormalize(load_path)
        check_obs_width(st["obs_mean"], venv.observation_space.shape[0], load_path)
        return cls.from_moments(venv, st["obs_mean"], st["obs_var"], st["obs_count"], st["ret_mean"], st["ret_var"], st["ret_count"],
                                training=st["training"], norm_obs=st["norm_obs"], norm_reward=st["norm_reward"], clip_obs=st["clip_obs"],
                                clip_reward=st["clip_reward"], gamma=st["gamma"], epsilon=st["epsilon"])

    def save(self, save_path: str) -> None:
        from . import checkpoint

        checkpoint.save_vecnormalize(save_path, dict(
            obs_mean=self.obs_rms.mean, obs_var=self.obs_rms.var, obs_count=self.obs_rms.count, ret_mean=self.ret_rms.mean, ret_var=self.ret_rms.var,
            ret_count=self.ret_rms.count, clip_obs=self.clip_obs, clip_reward=self.clip_reward, gamma=self.gamma, epsilon=self.epsilon,
            training=self.training, norm_obs=self.norm_obs, norm_reward=self.norm_reward), self.num_envs, self.action_space.shape[0])

    def normalize_obs(self, obs: np.ndarray) -> np.ndarray:
        if not self.norm_obs:
            return obs
        return np.clip((obs - self.obs_rms.mean) / np.sqrt(self.obs_rms.var + self.epsilon), -self.clip_obs, self.clip_obs).astype(np.float32)

    def normalize_reward(self, r: np.ndarray) -> np.ndarray:
        if not self.norm_reward:
            return r
        return np.clip(r / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward, self.clip_reward).astype(np.float32)

    def get_original_obs(self):
        return self.old_obs.copy()

    def get_original_reward(self):
        return self.old_reward.copy()

    def reset(self) -> np.ndarray:
        obs = self.venv.reset()
        self.old_obs = obs
        self.returns = np.zeros(self.num_envs)
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)

    def step_async(self, actions) -> None:
        self.venv.step_async(actions)

    def step_wait(self):
        obs, rews, dones, infos = self.venv.step_wait()
        self.old_obs, self.old_reward = obs, rews
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        if self.training:
            self.returns = self.returns * self.gamma + rews
            self.ret_rms.update(self.returns)
        out_r = self.normalize_reward(rews)
        norm_infos = _NormInfos(infos, self) if infos is not None else None
        self.returns[dones] = 0
        return self.normalize_obs(obs), out_r, dones, norm_infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self):
        self.venv.close()


class _NormInfos(Sequence):
    def __init__(self, infos, vn):
        self._infos, self._vn = infos, vn

    def __len__(self):
        return len(self._infos)

    def __getitem__(self, i):
        d = self._infos[i]
        if isinstance(d, dict) and "terminal_observation" in d:
            d["terminal_observation"] = self._vn.normalize_obs(d["terminal_observation"])
        return d
