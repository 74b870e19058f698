"""Ensemble and mixture-of-ensembles evaluation (/root/reference/src/eval_mixture_of_ensembles.py:125-345), batched over the
worlds of a ``MyoVecEnv`` and kept on the device.

The reference's final submission acts with the MEAN of the deterministic actions of several RecurrentPPO checkpoints, each fed
the observation normalised by ITS OWN ``VecNormalize`` statistics and carrying its own LSTM state (``eval_perf``, :235-262). A
task classifier (``models/classifier.py:160-174``: 234 -> 200 -> 100 -> 1 MLP on the scaled ``obs[29:47]`` of the first 13 steps of
an episode) decides after step 13 whether the episode is the HOLD task; if so the "hold" ensemble takes over with fresh LSTM
states (``SuperModel.process_before_action``, :178-196). Here every member is a ``RecurrentPolicy`` (tcgen05 kernel, obs
normalisation fused into its input load), all members run on all worlds every step, and per-world masks select which
ensemble's mean action a world takes; a member's LSTM state is zeroed for a world by raising its ``episode_start`` flag, which
is what ``state=None`` means in ``RecurrentPPO.predict``.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _capi, checkpoint
from .policy import RecurrentPolicy

N_OBS_PER_TRIAL = 13           # models/classifier.py:25
OBS_SLICE = (29, 47)           # eval_mixture_of_ensembles.py:176: ball positions / velocities / targets
DIMS_PER_OBS = OBS_SLICE[1] - OBS_SLICE[0]


class TaskClassifier:
    """``TaskClassifier`` + the ``StandardScaler`` saved next to it (``classifier.pt`` / ``scaler.pkl``): logits of
    "the episode is a rotation task" from the 13 x 18 window; ``predict`` returns 0 (hold) / 1 (rotate)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], scaler_mean=None, scaler_scale=None, device="cuda:0"):
        dev = torch.device(device)
        f = lambda k: torch.as_tensor(np.asarray(state_dict[k])).to(device=dev, dtype=torch.float32)
        self.w = [f("layer_1.weight"), f("layer_2.weight"), f("layer_out.weight")]
        self.b = [f("layer_1.bias"), f("layer_2.bias"), f("layer_out.bias")]
        d = self.w[0].shape[1]
        self.mean = torch.zeros(d, device=dev) if scaler_mean is None else torch.as_tensor(np.asarray(scaler_mean)).to(device=dev, dtype=torch.float32)
        self.scale = torch.ones(d, device=dev) if scaler_scale is None else torch.as_tensor(np.asarray(scaler_scale)).to(device=dev, dtype=torch.float32)
        self.device = dev

    @classmethod
    def load(cls, classifier_path: str, scaler_path: Optional[str] = None, device="cuda:0"):
        sd = torch.load(classifier_path, map_location="cpu", weights_only=True)
        mean = scale = None
        if scaler_path is not None:
            with open(scaler_path, "rb") as fh:
                sc = checkpoint._loads(fh.read())      # sklearn StandardScaler as an attribute bag (no sklearn import)
            mean, scale = sc.mean_, sc.scale_
        return cls(sd, mean, scale, device)

    @staticmethod
    def check_env(env) -> None:
        """The window is ``obs[29:47]`` of the default Baoding layout: refuse an env whose observation is laid out otherwise."""
        from .vec_env import DEFAULT_OBS_KEYS

        want = DEFAULT_OBS_KEYS[_capi.TASK_BAODING] + ("act",)
        if env.cfg.kind != _capi.TASK_BAODING or getattr(env, "obs_keys", want) != want:
            raise ValueError(f"the task classifier reads obs[{OBS_SLICE[0]}:{OBS_SLICE[1]}] of the default Baoding observation; this env's "
                             f"observation is {list(env.obs_keys) if getattr(env, 'obs_keys', None) else 'not a Baoding one'}")

    def logits(self, window: torch.Tensor) -> torch.Tensor:
        """``window``: [n, 13 * 18] raw observations, step-major as ``np.concatenate(obs_for_classifier)`` lays them out."""
        x = (window.to(self.device, torch.float32) - self.mean) / self.scale
        x = torch.relu(x @ self.w[0].T + self.b[0])
        x = torch.relu(x @ self.w[1].T + self.b[1])
        return (x @ self.w[2].T + self.b[2]).squeeze(-1)

    def predict(self, window: torch.Tensor) -> torch.Tensor:
        return torch.round(torch.sigmoid(self.logits(window))).to(torch.int64)


class Ensemble:
    """K policies, each with its own VecNormalize moments and LSTM states; ``act`` returns the mean deterministic action."""

    def __init__(self, policies: Sequence[RecurrentPolicy], norms: Sequence[Optional[Dict]]):
        if len(policies) != len(norms) or not policies:
            raise ValueError("one normaliser entry (or None) per policy")
        self.policies = list(policies)
        for p, nm in zip(self.policies, norms):
            if nm is not None:
                p.set_obs_norm(nm["obs_mean"], nm["obs_var"], float(nm.get("epsilon", 1e-8)), float(nm.get("clip_obs", 10.0)))
            else:
                p.set_obs_norm(None, None)
        self.states: List = []

    @classmethod
    def load(cls, model_paths: Sequence[str], vecnormalize_paths: Sequence[str], device="cuda:0", max_batch: int = 4096, precision="fp32"):
        """SB3 zips + ``VecNormalize`` pickles as the reference lists them (``PATH_TO_*_NET`` / ``PATH_TO_NORMALIZED_*_ENV``)."""
        pols, norms = [], []
        for mp, vp in zip(model_paths, vecnormalize_paths):
            ck = checkpoint.load_sb3_zip(mp)
            sd = ck["state_dict"]
            arch = checkpoint.architecture_of(sd)
            p = RecurrentPolicy(arch["obs_dim"], arch["act_dim"], arch["lstm_hidden"], arch["pi"], arch["vf"], max_batch=max_batch, device=device,
                                precision=precision)
            p.load_state_dict(sd)
            pols.append(p)
            norms.append(checkpoint.load_vecnormalize(vp) if vp else None)
        return cls(pols, norms)

    def initial_state(self, n: int) -> None:
        self.states = [p.initial_state(n) for p in self.policies]

    def act(self, obs: torch.Tensor, starts: torch.Tensor) -> torch.Tensor:
        if not self.states or self.states[0][0].shape[1] != obs.shape[0]:
            self.initial_state(obs.shape[0])
        acc = None
        for p, st in zip(self.policies, self.states):
            a, _, _, _ = p.forward(obs, st, starts, deterministic=True)
            acc = a.clone() if acc is None else acc.add_(a)
        return acc / float(len(self.policies))


class MixtureOfEnsembles:
    """``SuperModel`` + the action selection of ``eval_perf``: base ensemble until the classifier (after the 13th observation of
    an episode) says HOLD, then the hold ensemble with LSTM states that start at that step."""

    def __init__(self, base: Ensemble, hold: Ensemble, classifier: TaskClassifier):
        self.base, self.hold, self.classifier = base, hold, classifier
        self._n = 0

    def _alloc(self, n, dev):
        self._n = n
        self.timestep = torch.zeros(n, dtype=torch.int64, device=dev)
        self.window = torch.zeros(n, N_OBS_PER_TRIAL, DIMS_PER_OBS, dtype=torch.float32, device=dev)
        self.use_hold = torch.zeros(n, dtype=torch.bool, device=dev)
        self.current_task = torch.ones(n, dtype=torch.int64, device=dev)
        self.base.initial_state(n); self.hold.initial_state(n)

    def act(self, obs: torch.Tensor, starts: torch.Tensor) -> torch.Tensor:
        """``obs``: raw (un-normalised) observations [n, obs_dim]; ``starts``: episode-start flags of this step."""
        n, dev = obs.shape[0], obs.device
        if self._n != n:
            self._alloc(n, dev)
        st = starts.bool()
        # process_before_action
        self.use_hold &= ~st
        self.timestep.masked_fill_(st, 0)
        rec = self.timestep < N_OBS_PER_TRIAL
        slot = self.timestep.clamp(max=N_OBS_PER_TRIAL - 1)
        cur = self.window[torch.arange(n, device=dev), slot]
        self.window[torch.arange(n, device=dev), slot] = torch.where(rec[:, None], obs[:, OBS_SLICE[0]:OBS_SLICE[1]], cur)
        decide = self.timestep == N_OBS_PER_TRIAL - 1
        switched = torch.zeros_like(self.use_hold)
        if bool(decide.any()):
            task = self.classifier.predict(self.window.reshape(n, -1))
            self.current_task = torch.where(decide, task, self.current_task)
            switched = decide & (task == 0)
            self.use_hold |= switched
        self.timestep += 1
        a_base = self.base.act(obs, st)
        a_hold = self.hold.act(obs, st | switched)          # just_switched: the hold nets start from state None
        return torch.where(self.use_hold[:, None], a_hold, a_base)


def evaluate_mixture(model, env, n_episodes: int = 2000, max_steps: Optional[int] = None) -> Dict[str, float]:
    """``eval_perf``: episodes played back to back with the mixture's actions; mean length / reward with standard errors, mean
    effort (``|act| / na`` averaged per episode) and the classifier's error rate against the env's own task (``which_task`` of
    each world, clipped to hold / rotate). ``model``: ``MixtureOfEnsembles`` or ``Ensemble``; ``env``: ``MyoVecEnv`` (raw obs)."""
    if isinstance(model, MixtureOfEnsembles):
        TaskClassifier.check_env(env)
    n, dev = env.num_envs, env.device
    quota = max(1, math.ceil(n_episodes / n))
    obs = env.reset_device()
    starts = torch.ones(n, dtype=torch.uint8, device=dev)
    ep_ret = torch.zeros(n, dtype=torch.float64, device=dev); ep_eff = torch.zeros_like(ep_ret)
    ep_len = torch.zeros(n, dtype=torch.int64, device=dev); played = torch.zeros_like(ep_len)
    rets, lens, effs = [], [], []
    cls_n = cls_err = 0
    baoding = env.cfg.kind == _capi.TASK_BAODING
    horizon = int(env.cfg.max_episode_steps) if env.cfg.max_episode_steps > 0 else 1000
    limit = max_steps if max_steps is not None else quota * horizon + 1
    na = max(env.sim.na, 1)
    for _ in range(limit):
        live = played < quota
        if baoding and isinstance(model, MixtureOfEnsembles):
            truth = env.sim.get_task_state()[0][:, 2].clamp(0, 1).to(torch.int64)      # task of the episode being played
        actions = model.act(obs, starts)
        act_mag = torch.linalg.vector_norm(env.sim.get_state()[2].double(), dim=1) / na
        obs, rew, done, _ = env.step_device(actions.clamp(-1.0, 1.0))
        ep_ret += torch.where(live, rew.double(), torch.zeros_like(ep_ret))
        ep_eff += torch.where(live, act_mag, torch.zeros_like(ep_eff))
        ep_len += live.long()
        if baoding and isinstance(model, MixtureOfEnsembles):
            at13 = live & (ep_len == N_OBS_PER_TRIAL)
            cls_n += int(at13.sum()); cls_err += int((at13 & (model.current_task != truth)).sum())
        fin = done.bool() & live
        if bool(fin.any()):
            rets.append(ep_ret[fin].clone()); lens.append(ep_len[fin].clone()); effs.append((ep_eff[fin] / ep_len[fin].clamp(min=1)).clone())
            ep_ret.masked_fill_(fin, 0.0); ep_eff.masked_fill_(fin, 0.0); ep_len.masked_fill_(fin, 0)
            played += fin.long()
        starts = done
        if bool((played >= quota).all()):
            break
    cat = lambda xs: torch.cat(xs).double() if xs else torch.zeros(0, dtype=torch.float64, device=dev)
    r, l, e = cat(rets), cat(lens), cat(effs)
    k = max(int(r.numel()), 1)
    sem = lambda x: float(x.std(unbiased=False) / math.sqrt(k)) if x.numel() > 1 else 0.0
    mean = lambda x: float(x.mean()) if x.numel() else float("nan")
    return {"episodes": int(r.numel()), "mean_length": mean(l), "length_sem": sem(l), "mean_reward": mean(r), "reward_sem": sem(r),
            "mean_effort": mean(e), "effort_std": float(e.std(unbiased=False)) if e.numel() > 1 else 0.0,
            "classifier_inaccuracy": (cls_err / cls_n) if cls_n else float("nan"), "classified_episodes": cls_n}
