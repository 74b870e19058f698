"""GPU: the finger reach task through the CUDA library. The reach fixtures (tests/reach_fixture_checks.py, the same checks the
host build runs in tests/test_reach_host.py), the MyoVecEnv contract, a multi-step rollout against the shim's ReachEnvV0 over
the fp64 oracle, and a short RecurrentPPO run."""
import numpy as np
import pytest
import torch
from scipy import stats as sps

import reach_fixture_checks as fx
from myochallenge_b200 import _capi
from myochallenge_b200.envs import make_vec_env
from myochallenge_b200.vec_env import REACH_KEYS

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("tag", fx.STEP_TAGS)
def test_reach_step_reproduces_the_shim_env(product_lib, tag):
    fx.check_step_cases(product_lib, DEV, tag)


@pytest.mark.parametrize("tag", fx.RESET_TAGS)
def test_reach_reset_reproduces_the_shim_distribution(product_lib, tag):
    fx.check_reset_distribution(product_lib, DEV, tag, n=4096)


@pytest.mark.parametrize("env_id", ["myoFingerReachFixed-v0", "myoFingerReachRandom-v0"])
def test_reach_vec_env_contract(product_lib, env_id):
    n = 32
    env = make_vec_env(env_id, n, device=DEV, seed=4, max_episode_steps=3)
    assert env.observation_space.shape == (19,) and env.info_keys == REACH_KEYS
    obs = env.reset()
    assert obs.shape == (n, 19)
    sid = env.cfg.reach_target_site[0]
    t0 = env.sim.get_param(_capi.PARAM_SITE_POS, sid).cpu().numpy().copy()
    rng = np.random.default_rng(0)
    for _ in range(3):
        obs, rew, done, infos = env.step(rng.uniform(-1, 1, (n, 5)).astype(np.float32))
    assert done.all()
    t1 = env.sim.get_param(_capi.PARAM_SITE_POS, sid).cpu().numpy()
    if "Fixed" in env_id:
        np.testing.assert_array_equal(t1, t0)
    else:
        assert np.all(np.abs(t1 - t0).max(1) > 0)           # auto-reset drew new targets
    for i in range(n):
        d = infos[i]
        assert set(d["rwd_dict"]) == set(REACH_KEYS) and d["TimeLimit.truncated"]
        tob = d["terminal_observation"]          # the finished episode's last observation: its own target
        np.testing.assert_allclose(tob[11:14], t0[i] - tob[8:11], atol=1e-5)
        np.testing.assert_allclose(obs[i, 11:14], t1[i] - obs[i, 8:11], atol=1e-5)
    # the host-array API and the device API step the same worlds alike
    e1, e2 = make_vec_env(env_id, n, device=DEV, seed=7, max_episode_steps=4), make_vec_env(env_id, n, device=DEV, seed=7, max_episode_steps=4)
    np.testing.assert_array_equal(e1.reset(), e2.reset_device().cpu().numpy())
    for _ in range(6):
        a = rng.uniform(-1, 1, (n, 5)).astype(np.float32)
        o1, r1, d1, _ = e1.step(a)
        o2, r2, d2, _ = e2.step_device(torch.as_tensor(a, device=DEV))
        np.testing.assert_array_equal(o1, o2.cpu().numpy())
        np.testing.assert_array_equal(r1, r2.cpu().numpy())
        np.testing.assert_array_equal(d1, d2.cpu().numpy().astype(bool))


def test_reach_rollout_matches_the_shim_env(product_lib):
    """64 myoFingerReachRandom worlds, 200 env steps (1000 mj_steps) under seeded random actions, against the shim's ReachEnvV0
    (fp64 oracle) replaying every world from its reset with that world's targets and actions. fp32 and fp64 trajectories of the
    finger drift apart slowly and, in a few worlds, far enough to cross far_th at different steps, so the bars are: episode
    lengths agree for >= 90 % of the worlds; returns of >= 90 % of the agreeing worlds within 1 % (+0.05 absolute); the two
    return samples pass a KS test (p > 0.05); done flags agree in >= 99.9 % of the steps where both distances are 2 cm clear
    of far_th."""
    g_len, g_ret, o_len, o_ret, flags, _ = fx.check_rollout(product_lib, DEV, n=64, steps=200)
    same = g_len == o_len
    assert same.mean() >= 0.9, f"episode lengths agree for {same.mean():.2f} of the worlds"
    ok = np.abs(g_ret - o_ret)[same] <= 0.01 * np.abs(o_ret[same]) + 0.05
    assert ok.mean() >= 0.9, f"returns agree for {ok.mean():.2f} of the worlds of equal length"
    assert sps.ks_2samp(g_ret, o_ret).pvalue > 0.05
    clear = flags[:, 0] > 0.02
    assert flags[clear, 1].mean() >= 0.999


def test_recurrent_ppo_learns_on_reach(product_lib):
    from myochallenge_b200.ppo import RecurrentPPO
    from myochallenge_b200.rollout import DeviceVecNormalize

    n, T = 64, 8
    env = make_vec_env("myoFingerReachRandom-v0", n, device=DEV, seed=2, clip_actions=True)
    vn = DeviceVecNormalize(env, gamma=0.99)
    agent = RecurrentPPO("MlpLstmPolicy", vn, n_steps=T, batch_size=T * 32, n_epochs=1, learning_rate=1e-4,
                         policy_kwargs=dict(lstm_hidden_size=64, net_arch=[dict(pi=[32], vf=[32])], log_std_init=-2.0), seed=1)
    agent.learn(total_timesteps=2 * n * T)
    assert len(agent.logs) == 2
    for log in agent.logs:
        assert all(np.isfinite(v) for v in log.values() if isinstance(v, (int, float))), log
    assert env.sim.status() & ~1 == 0        # bit 0: the finger model's advisory flag (DESIGN.md 5)
