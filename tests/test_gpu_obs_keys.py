"""GPU: MyoSuite's ``obs_keys`` and ``reward_mode`` env kwargs through the CUDA library. Two ``MyoVecEnv``s with the same seed, one with
the default layout and one with a permuted subset of keys plus ``t``, step the same actions: physics, rewards and infos agree bit for
bit, and the custom observations are the gathered columns of the default ones. Also the sparse reward through the Monitor returns, a
short RecurrentPPO run on a reduced observation, and the Baoding kernel's occupancy with custom keys. The host build runs the same
contract in tests/test_obs_keys_host.py."""
import numpy as np
import pytest
import torch

from myochallenge_b200.envs import make_vec_env
from myochallenge_b200.vec_env import DEFAULT_OBS_KEYS
from test_obs_keys_host import CASES, _expand, default_columns, expected_obs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

GPU_CASES = {
    "baoding": CASES["baoding"],
    "die": CASES["die"],
    "hand_pose": ("CustomMyoHandPoseRandom-v0", ["pose_err", "t", "qpos", "act", "pose_err"]),
    "reach": CASES["reach"],
    "elbow": CASES["elbow"],
}


@pytest.mark.parametrize("tag", sorted(GPU_CASES))
def test_custom_keys_gather_the_default_columns(product_lib, tag):
    env_id, keys = GPU_CASES[tag]
    n, steps = 256, 50
    kw = dict(device=DEV, seed=7, clip_actions=True, max_episode_steps=20)      # two auto-resets per world in the run, at least
    d, c = make_vec_env(env_id, n, **kw), make_vec_env(env_id, n, obs_keys=keys, **kw)
    full = keys if "act" in keys else keys + ["act"]
    assert c.obs_keys == tuple(full) and c.observation_space.shape == (c.sim.nobs,)
    sim = d.sim
    cols = default_columns(d.cfg.kind, sim.nq, sim.nv, sim.na, max(d.cfg.reach_nsite, 1))
    tcol = np.array([i for i, k in enumerate(_expand(full, d.cfg.kind, cols)) if k == "t"])
    assert c.sim.nobs == len(_expand(full, d.cfg.kind, cols))
    od, oc = d.reset_device().cpu().numpy(), c.reset_device().cpu().numpy()
    np.testing.assert_array_equal(oc, expected_obs(full, od, np.zeros(n), cols))
    dt = np.float32(d.cfg.frame_skip * sim.model.opt("timestep"))
    gen = torch.Generator(device=DEV).manual_seed(0)
    ended = 0
    for k in range(steps):
        a = torch.rand(n, sim.nu, device=DEV, generator=gen) * 2 - 1
        t_prev = c.sim.get_state()[3].cpu().numpy()
        rd, rc = d.step_device(a), c.step_device(a)
        for x, y in zip(rd[1:], rc[1:]):             # reward, done, truncated
            assert torch.equal(x, y), f"{tag} step {k}"
        assert torch.equal(d.sim.info, c.sim.info), f"{tag} step {k}: info"
        for x, y in zip(d.sim.get_state(), c.sim.get_state()):
            assert torch.equal(x, y), f"{tag} step {k}: state"
        time = c.sim.get_state()[3].cpu().numpy()
        od, oc = rd[0].cpu().numpy(), rc[0].cpu().numpy()
        np.testing.assert_array_equal(oc, expected_obs(full, od, time, cols), err_msg=f"{tag} step {k}")
        done = rd[2].cpu().numpy().astype(bool)
        if done.any():
            ended += int(done.sum())
            assert np.all(time[done] == 0)
            got = c.terminal_obs.cpu().numpy()[done]
            exp = expected_obs(full, d.terminal_obs.cpu().numpy()[done], np.full(done.sum(), np.nan), cols)
            np.testing.assert_array_equal(np.delete(got, tcol, 1), np.delete(exp, tcol, 1), err_msg=f"{tag} step {k}: terminal obs")
            t_end = (t_prev + dt)[done][:, None]
            assert np.allclose(got[:, tcol], t_end, rtol=1e-6) and np.all(got[:, tcol] > 0), f"{tag} step {k}: terminal t"
    assert ended >= 2 * n
    np.testing.assert_array_equal(c.sim.get_obs().cpu().numpy(), expected_obs(full, d.sim.get_obs().cpu().numpy(), c.sim.get_state()[3].cpu().numpy(), cols))
    assert d.sim.status() & ~1 == 0 and c.sim.status() & ~1 == 0


@pytest.mark.parametrize("tag", sorted(GPU_CASES))
def test_explicit_default_keys_are_bit_identical(product_lib, tag):
    env_id, _ = GPU_CASES[tag]
    n = 128
    kw = dict(device=DEV, seed=3, clip_actions=True, max_episode_steps=15)
    d = make_vec_env(env_id, n, **kw)
    e = make_vec_env(env_id, n, obs_keys=list(DEFAULT_OBS_KEYS[d.cfg.kind]), **kw)
    assert e.cfg.n_obs_keys > 0 and e.obs_keys == d.obs_keys
    assert torch.equal(d.reset_device(), e.reset_device())
    gen = torch.Generator(device=DEV).manual_seed(1)
    for _ in range(30):
        a = torch.rand(n, d.sim.nu, device=DEV, generator=gen) * 2 - 1
        for x, y in zip(d.step_device(a), e.step_device(a)):
            assert torch.equal(x, y)
        assert torch.equal(d.terminal_obs, e.terminal_obs) and torch.equal(d.sim.info, e.sim.info)


@pytest.mark.parametrize("tag", ["baoding", "die", "reach", "elbow"])
def test_sparse_reward_and_monitor_returns(product_lib, tag):
    env_id, keys = GPU_CASES[tag]
    n = 64
    env = make_vec_env(env_id, n, device=DEV, seed=5, clip_actions=True, max_episode_steps=10, reward_mode="sparse", obs_keys=keys)
    env.reset()
    rng = np.random.default_rng(0)
    ret = np.zeros(n, np.float32)
    finished = 0
    for _ in range(25):
        obs, rew, done, infos = env.step(rng.uniform(-1, 1, (n, env.sim.nu)).astype(np.float32))
        info = env.sim.info.cpu().numpy()
        np.testing.assert_array_equal(rew, info[:, 4])
        assert obs.shape == (n, env.sim.nobs)
        ret += rew
        for w in np.nonzero(done)[0]:
            assert infos[w]["episode"]["r"] == pytest.approx(float(ret[w]), rel=1e-6, abs=1e-6)
            assert infos[w]["rwd_dense"] == pytest.approx(float(info[w, 7]))
            ret[w] = 0
            finished += 1
    assert finished >= 2 * n


def test_recurrent_ppo_learns_on_reduced_keys(product_lib):
    from myochallenge_b200.ppo import RecurrentPPO
    from myochallenge_b200.rollout import DeviceVecNormalize

    n, T = 64, 8
    env = make_vec_env("myoFingerReachRandom-v0", n, device=DEV, seed=2, clip_actions=True, obs_keys=["reach_err", "t"])
    assert env.observation_space.shape == (3 + 1 + 5,)
    vn = DeviceVecNormalize(env, gamma=0.99)
    assert vn.obs_rms.d == 9
    agent = RecurrentPPO("MlpLstmPolicy", vn, n_steps=T, batch_size=T * 32, n_epochs=1, learning_rate=1e-4,
                         policy_kwargs=dict(lstm_hidden_size=64, net_arch=[dict(pi=[32], vf=[32])], log_std_init=-2.0), seed=1)
    agent.learn(total_timesteps=2 * n * T)
    assert len(agent.logs) == 2
    for log in agent.logs:
        assert all(np.isfinite(v) for v in log.values() if isinstance(v, (int, float))), log


def test_baoding_p2_custom_keys_keep_16_worlds_per_cta(product_lib):
    env = make_vec_env("CustomMyoChallengeBaodingP2-v1", 4096, device=DEV, seed=0, clip_actions=True, obs_keys=GPU_CASES["baoding"][1])
    info = env.sim.launch_info()
    assert info["lanes_per_world"] == 32 and info["worlds_per_cta"] == 16 and info["regs_per_thread"] <= 128, info
