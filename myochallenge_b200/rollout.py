"""Device-resident rollout side of the PPO loop (SURVEY.md 8a rows a14, a17): VecNormalize's running moments and
reward scaling, sb3-contrib's RecurrentRolloutBuffer with GAE, and the rollout collection loop of
``RecurrentPPO.collect_rollouts`` - the part of /root/reference/src/train/trainer.py:67-71 that runs between two
policy updates - over a ``MyoVecEnv`` and a ``RecurrentPolicy`` without leaving HBM.

PyTorch provides the tensors and streams; the arithmetic is in libmyo_b200.so (csrc/myo_rollout.cu, the world and
policy kernels). Cross-rank: worlds are sharded, so the only exchange is the merge of the running moments
(``DeviceRunningMeanStd.sync``: all-gather of (count, mean, M2), 2 d + 1 doubles per rank, Chan merge in rank order).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _capi
from .vec_env import check_obs_width


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class DeviceRunningMeanStd:
    """SB3 ``RunningMeanStd`` with the state (mean[d], var[d], count; fp64) on the device."""

    def __init__(self, d: int, device, epsilon: float = 1e-4):
        self.d, self.device = int(d), torch.device(device)
        self.state = torch.zeros(2 * self.d + 1, dtype=torch.float64, device=self.device)
        self.state[self.d: 2 * self.d] = 1.0
        self.state[2 * self.d] = epsilon
        self.mean_f = torch.zeros(self.d, dtype=torch.float32, device=self.device)
        self.var_f = torch.ones(self.d, dtype=torch.float32, device=self.device)
        self._scratch = None
        self._L = _capi.lib()
        self.launch_count = 0

    def _scratch_for(self, n):
        need = self._L.myo_running_moments_scratch(int(n), self.d)
        if self._scratch is None or self._scratch.numel() < need:
            self._scratch = torch.empty(need, dtype=torch.float64, device=self.device)
        return self._scratch

    def update(self, x: torch.Tensor):
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
        assert (x.shape[-1] == self.d) if x.dim() > 1 else (self.d == 1)
        n = x.shape[0]
        s = self._scratch_for(n)
        _capi.check(self._L, self._L.myo_running_moments_update(_p(self.state), _p(x), n, self.d, _p(s), _p(self.mean_f), _p(self.var_f), _stream_ptr(self.device)))
        self.launch_count += 3

    def load(self, mean, var, count):
        self.state[: self.d] = torch.as_tensor(np.asarray(mean, np.float64).reshape(-1), device=self.device)
        self.state[self.d: 2 * self.d] = torch.as_tensor(np.asarray(var, np.float64).reshape(-1), device=self.device)
        self.state[2 * self.d] = float(count)
        _capi.check(self._L, self._L.myo_running_moments_export(_p(self.state), self.d, _p(self.mean_f), _p(self.var_f), _stream_ptr(self.device)))

    @property
    def mean(self):
        return self.state[: self.d]

    @property
    def var(self):
        return self.state[self.d: 2 * self.d]

    @property
    def count(self):
        return self.state[2 * self.d]

    def sync(self, base: "torch.Tensor | None" = None):
        """Merge the moments of all ranks (each rank saw its own worlds). ``base``: the state THIS rank started the
        interval from; every rank contributes what it added since (its state minus its own base) and the contributions
        are merged in rank order onto rank 0's base, so all ranks end with the same state even if their bases differed.
        Without ``base`` the ranks' states are merged as independent samples. Stays on the device (no host round trip)."""
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return
        mine = self.state if base is None else torch.cat([self.state, base.to(self.state)])
        got = torch.stack(_all_gather(mine))
        n = 2 * self.d + 1
        merged = merge_moment_states(got[:, :n], self.d, bases=None if base is None else got[:, n:])
        self.state.copy_(merged)
        _capi.check(self._L, self._L.myo_running_moments_export(_p(self.state), self.d, _p(self.mean_f), _p(self.var_f), _stream_ptr(self.device)))


def _all_gather(t):
    import torch.distributed as dist

    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return out


def merge_moment_states(states, d, base=None, bases=None):
    """Chan merge, in rank order, of per-rank RunningMeanStd states [mean(d), var(d), count] (fp64; numpy arrays or
    torch tensors on any device, result of the same kind). ``bases`` (one per rank) or ``base`` (shared): the state each
    rank started the interval from - a rank then contributes only what it added since (its state minus ITS base), merged
    onto rank 0's base; a rank whose base differs from rank 0's still contributes exactly its own additions, so every
    rank computes the same result. Branch-free, so the device version never synchronises with the host."""
    as_numpy = not torch.is_tensor(states) and not torch.is_tensor(states[0])
    S = torch.stack([torch.as_tensor(np.asarray(s) if as_numpy else s, dtype=torch.float64) for s in states]) if not torch.is_tensor(states) else states
    K = S.shape[0]
    if bases is not None:
        B = torch.stack([torch.as_tensor(np.asarray(b) if as_numpy else b, dtype=torch.float64) for b in bases]) if not torch.is_tensor(bases) else bases
    elif base is not None:
        B = torch.as_tensor(np.asarray(base) if as_numpy else base, dtype=torch.float64).to(S.device).expand(K, -1)
    else:
        B = None

    def split(s):
        return s[:d], s[d: 2 * d], s[2 * d]

    def merge(a, b):
        (ma, va, na), (mb, vb, nb) = a, b
        tot = na + nb
        safe = torch.clamp(tot, min=1e-300)
        delta = mb - ma
        return ma + delta * nb / safe, (va * na + vb * nb + delta * delta * na * nb / safe) / safe, tot

    def subtract(s, b):      # inverse of merge: the batch that turns b into s (count 0 when nothing was added)
        (ms, vs, ns), (mb, vb, nb) = s, b
        nx = torch.clamp(ns - nb, min=0.0)
        safe = torch.clamp(nx, min=1e-300)
        mx = torch.where(nx > 0, (ms * ns - mb * nb) / safe, ms)
        delta = mx - mb
        vx = torch.where(nx > 0, (vs * ns - vb * nb - delta * delta * nb * nx / torch.clamp(ns, min=1e-300)) / safe, vs)
        return mx, torch.clamp(vx, min=0.0), nx

    if B is None:
        acc = split(S[0])
        for k in range(1, K):
            acc = merge(acc, split(S[k]))
    else:
        acc = split(B[0])
        for k in range(K):
            acc = merge(acc, subtract(split(S[k]), split(B[k])))
    out = torch.cat([acc[0], acc[1], acc[2].reshape(1)])
    return out.numpy() if as_numpy else out


class DeviceVecNormalize:
    """VecNormalize over the device path of a ``MyoVecEnv``: observations stay raw in HBM and are normalised inside
    the policy kernel's input load (``policy.set_obs_norm`` is pointed at this object's fp32 moments, which every
    ``obs_rms`` update refreshes); rewards are scaled by the std of the discounted return as SB3 does."""

    def __init__(self, venv, policy=None, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8):
        self.venv, self.device = venv, venv.sim.device
        self.num_envs = venv.num_envs
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.obs_rms = DeviceRunningMeanStd(venv.sim.nobs, self.device)
        self.ret_rms = DeviceRunningMeanStd(1, self.device)
        self.returns = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)
        self._out_r = torch.empty(self.num_envs, dtype=torch.float32, device=self.device)
        self._L = _capi.lib()
        self.launch_count = 0
        self.policy = None
        if policy is not None:
            self.attach(policy)

    def attach(self, policy):
        self.policy = policy
        self._push_obs_norm()

    def _push_obs_norm(self):
        if self.policy is not None and self.norm_obs:
            self.policy.set_obs_norm(self.obs_rms.mean_f, self.obs_rms.var_f, self.epsilon, self.clip_obs)

    def reset_device(self):
        obs = self.venv.reset_device()
        self.returns.zero_()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
            self._push_obs_norm()
        return obs

    def step_device(self, actions):
        obs, rew, done, trunc = self.venv.step_device(actions)
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
            self._push_obs_norm()
        s = self.ret_rms._scratch_for(self.num_envs)
        _capi.check(self._L, self._L.myo_vecnorm_reward(_p(self.ret_rms.state), _p(self.returns), _p(rew), _p(done), _p(self._out_r), self.num_envs,
                                                        self.gamma, self.epsilon, self.clip_reward, int(self.training), int(self.norm_reward),
                                                        _p(s), _stream_ptr(self.device)))
        self.launch_count += 4 if self.training else 1
        return obs, self._out_r, done, trunc

    @property
    def terminal_obs(self):
        return self.venv.terminal_obs

    # -- VecNormalize.save / VecNormalize.load(path, venv) (/root/reference/src/main_eval.py:65-67) ----------------------------
    def stats(self):
        o, r = self.obs_rms.state.cpu().numpy(), self.ret_rms.state.cpu().numpy()
        d = self.obs_rms.d
        return dict(obs_mean=o[:d].copy(), obs_var=o[d: 2 * d].copy(), obs_count=float(o[2 * d]), ret_mean=float(r[0]), ret_var=float(r[1]),
                    ret_count=float(r[2]), clip_obs=self.clip_obs, clip_reward=self.clip_reward, gamma=self.gamma, epsilon=self.epsilon,
                    training=self.training, norm_obs=self.norm_obs, norm_reward=self.norm_reward)

    def save(self, path: str):
        from . import checkpoint

        checkpoint.save_vecnormalize(path, self.stats(), self.num_envs, self.venv.sim.nu)

    @classmethod
    def load(cls, path: str, venv, policy=None):
        from . import checkpoint

        st = checkpoint.load_vecnormalize(path)
        check_obs_width(st["obs_mean"], venv.sim.nobs, path)
        vn = cls(venv, None, training=st["training"], norm_obs=st["norm_obs"], norm_reward=st["norm_reward"], clip_obs=st["clip_obs"],
                 clip_reward=st["clip_reward"], gamma=st["gamma"], epsilon=st["epsilon"])
        vn.obs_rms.load(st["obs_mean"], st["obs_var"], st["obs_count"])
        vn.ret_rms.load([st["ret_mean"]], [st["ret_var"]], st["ret_count"])
        if policy is not None:
            vn.attach(policy)
        return vn


class RecurrentRolloutBuffer:
    """sb3-contrib ``RecurrentRolloutBuffer`` storage, step-major on the device: observations (as the policy saw them,
    i.e. normalised when the env is a ``DeviceVecNormalize``), actions, rewards, episode_starts, values, log_probs and
    the LSTM states the rollout started from (``h0`` / ``c0``). sb3-contrib stores the states of every step because its
    minibatches may start anywhere; the update here (``ppo.PPOUpdate``) takes whole sequences, whose only start states
    that matter are those of step 0 - every later sequence start is an episode start, where the state is zeroed."""

    def __init__(self, n_steps, n_envs, obs_dim, act_dim, lstm_hidden, device, gamma=0.99, gae_lambda=0.95):
        dev = torch.device(device)
        f = dict(dtype=torch.float32, device=dev)
        self.n_steps, self.n_envs, self.gamma, self.gae_lambda, self.device = n_steps, n_envs, gamma, gae_lambda, dev
        self.observations = torch.zeros(n_steps, n_envs, obs_dim, **f)
        self.actions = torch.zeros(n_steps, n_envs, act_dim, **f)
        self.rewards = torch.zeros(n_steps, n_envs, **f)
        self.values = torch.zeros(n_steps, n_envs, **f)
        self.log_probs = torch.zeros(n_steps, n_envs, **f)
        self.advantages = torch.zeros(n_steps, n_envs, **f)
        self.returns = torch.zeros(n_steps, n_envs, **f)
        self.episode_starts = torch.zeros(n_steps, n_envs, dtype=torch.uint8, device=dev)
        self.h0 = torch.zeros(2, n_envs, lstm_hidden, **f)      # [0] actor, [1] critic
        self.c0 = torch.zeros(2, n_envs, lstm_hidden, **f)
        self.pos, self.full = 0, False
        self._L = _capi.lib()
        self.launch_count = 0
        # reward terms (the env's ``info`` dict entries) summed over the rollout, for TensorboardCallback-style logging
        self.info_sum = torch.zeros(_capi.MYO_INFO_TERMS, dtype=torch.float64, device=dev)
        self.info_count = 0

    def reset(self):
        self.pos, self.full = 0, False
        self.info_sum.zero_(); self.info_count = 0

    def add_info(self, info: torch.Tensor) -> None:
        """``info`` [n, MYO_INFO_TERMS]: the reward terms of this env step (``BatchSim.info``)."""
        self.info_sum += info.sum(0, dtype=torch.float64)
        self.info_count += info.shape[0]

    def info_means(self):
        """Mean of every info term over the steps and worlds of the rollout (host numpy array)."""
        return (self.info_sum / max(self.info_count, 1)).cpu().numpy()

    def put_obs(self, obs, obs_norm=None):
        """Store the observation of the current step. ``obs_norm``: a ``DeviceVecNormalize`` whose CURRENT moments (the
        ones the policy's fused normalisation uses for this step: call before the env step updates them) normalise
        ``obs`` on the way in (one streaming kernel); None stores ``obs`` as given."""
        t = self.pos
        if obs_norm is not None and obs_norm.norm_obs:
            _capi.check(self._L, self._L.myo_normalize_obs(_p(obs), _p(obs_norm.obs_rms.mean_f), _p(obs_norm.obs_rms.var_f), obs_norm.epsilon,
                                                           obs_norm.clip_obs, _p(self.observations[t]), self.n_envs, obs.shape[1],
                                                           _stream_ptr(self.device)))
            self.launch_count += 1
        else:
            self.observations[t].copy_(obs)

    def add(self, obs, action, reward, episode_start, value, log_prob, h=None, c=None):
        """``obs`` None: already stored by ``put_obs``. ``h`` / ``c``: LSTM states this step started from (kept for step 0)."""
        t = self.pos
        if obs is not None:
            self.observations[t].copy_(obs)
        self.actions[t].copy_(action); self.rewards[t].copy_(reward)
        self.episode_starts[t].copy_(episode_start); self.values[t].copy_(value); self.log_probs[t].copy_(log_prob)
        if t == 0 and h is not None:
            self.h0.copy_(h); self.c0.copy_(c)
        self.pos += 1
        self.full = self.pos == self.n_steps

    def compute_returns_and_advantage(self, last_values, dones):
        assert self.full, "rollout buffer is not full"
        _capi.check(self._L, self._L.myo_gae(_p(self.rewards), _p(self.values), _p(self.episode_starts), _p(last_values.contiguous()),
                                             _p(dones.contiguous()), self.n_steps, self.n_envs, self.gamma, self.gae_lambda,
                                             _p(self.advantages), _p(self.returns), _stream_ptr(self.device)))
        self.launch_count += 1


def collect_rollouts(env, policy, buffer: RecurrentRolloutBuffer, state, obs, episode_starts, clip_actions=True, sde_sample_freq=-1):
    """``RecurrentPPO.collect_rollouts``: n_steps of policy forward -> env step -> buffer.add, with the TimeLimit
    bootstrap (reward += gamma * V(terminal_observation) for truncated worlds, values from the critic state the step
    ended in) and the final GAE pass. ``env``: MyoVecEnv or DeviceVecNormalize (device path); ``state`` = (h, c) as
    ``policy.initial_state`` returns them (updated in place). Returns (obs, episode_starts) for the next call."""
    h, c = state
    buffer.reset()
    norm = env if isinstance(env, DeviceVecNormalize) else None
    use_sde = getattr(policy, "use_sde", False)
    for t in range(buffer.n_steps):
        if t == 0:
            buffer.h0.copy_(h); buffer.c0.copy_(c)
        if use_sde and (t == 0 or (sde_sample_freq > 0 and t % sde_sample_freq == 0)):
            policy.reset_noise(obs.shape[0])          # RecurrentPPO.collect_rollouts: new exploration matrices
        actions, values, logp, _ = policy.forward(obs, (h, c), episode_starts)
        buffer.put_obs(obs, norm)
        env_actions = actions.clamp(-1.0, 1.0) if clip_actions else actions
        new_obs, rewards, dones, trunc = env.step_device(env_actions)
        rewards = rewards.clone()
        idx = torch.nonzero(trunc, as_tuple=False).flatten()
        if idx.numel():       # bootstrap with the value of the terminal observation (critic state after this step)
            tv = policy.predict_values(env.terminal_obs.index_select(0, idx), (h.index_select(1, idx), c.index_select(1, idx)))
            rewards.index_add_(0, idx, buffer.gamma * tv)
        buffer.add(None, actions, rewards, episode_starts, values, logp)
        sim = getattr(getattr(env, "venv", env), "sim", None)
        if sim is not None:
            buffer.add_info(sim.info)
        obs, episode_starts = new_obs.clone(), dones.clone()
    last_values = policy.predict_values(obs, (h.clone(), c.clone()), episode_starts)
    buffer.compute_returns_and_advantage(last_values, episode_starts)
    return obs, episode_starts


class PipelinedStepper:
    """Device-resident stepping of the worlds as ``k`` sub-batches on ``k`` CUDA streams. The rollout's two kernels have opposite
    shapes - the world kernel is one long persistent launch that owns every SM, the policy forward a short tensor-core launch - and
    with one stream they alternate, the policy waiting for the world kernel's last wave. With two sub-batches the policy forward
    of one half (and the head of its next world launch) runs on the SMs the other half's world kernel frees as it drains, so the
    policy's time and the drain tail disappear from the step. Worlds are independent, so the results of a sub-batch do not depend
    on the split (``envs[i]`` is an ordinary ``MyoVecEnv``); the policy handle is shared (read-only weights, per-call state).

    ``step()`` enqueues one env step of every sub-batch and returns without synchronising; ``obs[i]``, ``rewards[i]``,
    ``dones[i]`` hold the latest results of sub-batch ``i`` (valid on ``streams[i]``; ``join()`` makes the current stream wait)."""

    def __init__(self, envs, policy, deterministic: bool = False, clip_actions: bool = True):
        self.envs, self.policy = list(envs), policy
        dev = self.envs[0].device
        self.device = dev
        self.streams = [torch.cuda.Stream(dev) for _ in self.envs]
        self.states = [policy.initial_state(e.num_envs) for e in self.envs]
        self.starts = [torch.ones(e.num_envs, dtype=torch.uint8, device=dev) for e in self.envs]
        self.out = [(torch.empty(e.num_envs, e.sim.nu, device=dev), torch.empty(e.num_envs, device=dev), torch.empty(e.num_envs, device=dev))
                    for e in self.envs]
        self.obs = [None] * len(self.envs)
        self.rewards = [None] * len(self.envs)
        self.dones = [None] * len(self.envs)
        self.deterministic, self.clip_actions = deterministic, clip_actions
        self.num_envs = sum(e.num_envs for e in self.envs)

    def reset(self):
        cur = torch.cuda.current_stream(self.device)
        for i, e in enumerate(self.envs):
            self.streams[i].wait_stream(cur)
            with torch.cuda.stream(self.streams[i]):
                self.obs[i] = e.reset_device()
                self.starts[i].fill_(1)
        return self.obs

    def step(self):
        for i, e in enumerate(self.envs):
            with torch.cuda.stream(self.streams[i]):
                a, _, _, _ = self.policy.forward(self.obs[i], self.states[i], self.starts[i], deterministic=self.deterministic, out=self.out[i])
                if self.clip_actions:
                    a = a.clamp_(-1.0, 1.0)
                self.obs[i], self.rewards[i], d, _ = e.step_device(a)
                self.dones[i] = d
                self.starts[i] = d
        return self.obs, self.rewards, self.dones

    def spin_up(self, steps: int):
        """Untimed steps to the steady state of the workload with the episode phases of the worlds staggered uniformly over the
        horizon (world w of a sub-batch is reset once more at step ``w mod horizon``); see bench.py."""
        horizon = int(self.envs[0].cfg.max_episode_steps)
        for t in range(steps):
            if horizon > 0 and t < horizon:
                for i, e in enumerate(self.envs):
                    with torch.cuda.stream(self.streams[i]):
                        mask = (torch.arange(e.num_envs, device=self.device) % horizon) == t
                        e.sim.reset(mask)
                        self.starts[i] = torch.maximum(self.starts[i], mask.to(torch.uint8))
            self.step()

    def join(self):
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            cur.wait_stream(s)

    def synchronize(self):
        for s in self.streams:
            s.synchronize()
