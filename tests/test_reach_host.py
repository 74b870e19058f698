"""CPU: the finger reach task (MyoSuite ReachEnvV0 behind MyoFingerReachFixed / MyoFingerReachRandom). Registry and factory
mapping, config errors, the far_th time gate, and - through the host build of the kernel sources (tests/emul) - the reach
fixtures of tests/golden/make_reach_fixtures.py (checks in tests/reach_fixture_checks.py; the GPU run is tests/test_gpu_reach.py)."""
import numpy as np
import pytest
import torch

import reach_fixture_checks as fx
from myochallenge_b200 import _capi
from myochallenge_b200.assets import asset_path
from myochallenge_b200.envs import FACTORY_NAMES, REGISTRY, UNSUPPORTED, EnvironmentFactory, make_task_cfg, reach_far_steps
from myochallenge_b200.sim import BatchSim, Model
from myochallenge_b200.vec_env import REACH_KEYS

FINGER = "finger/myo_finger_v0.mjb"


@pytest.mark.parametrize("name,env_id,lo,hi", [
    ("MyoFingerReachFixed", "myoFingerReachFixed-v0", (0.2, 0.05, 0.2), (0.2, 0.05, 0.2)),
    ("MyoFingerReachRandom", "myoFingerReachRandom-v0", (0.1, -0.1, 0.1), (0.27, 0.1, 0.3))])
def test_reach_registrations(product_lib, name, env_id, lo, hi):
    assert FACTORY_NAMES[name] == env_id and name not in UNSUPPORTED
    assert REGISTRY[env_id]["kind"] == _capi.TASK_REACH and REGISTRY[env_id]["model"] == FINGER
    m = Model(asset_path(FINGER), lib=product_lib)
    cfg = make_task_cfg(m, env_id)
    assert cfg.kind == _capi.TASK_REACH and cfg.max_episode_steps == 200 and cfg.frame_skip == 5 and cfg.normalize_act == 1
    assert cfg.reach_nsite == 1
    assert m.id2name("site", cfg.reach_tip_site[0]) == "IFtip" and m.id2name("site", cfg.reach_target_site[0]) == "IFtip_target"
    np.testing.assert_allclose([list(cfg.reach_range[0][0]), list(cfg.reach_range[0][1])], [lo, hi], rtol=1e-6)
    np.testing.assert_allclose(list(cfg.rwd_weight)[:7], [1, 4, 0, 50, 0, 0, 0])         # reach bonus act_reg penalty sparse solved done
    assert cfg.far_th == pytest.approx(0.35) and cfg.reach_near_th == pytest.approx(0.0125) and cfg.reach_far_steps == 2


def test_reach_default_cfg_matches_the_registration(product_lib):
    m = Model(asset_path(FINGER), lib=product_lib)
    d, r = m.default_task_cfg(_capi.TASK_REACH), make_task_cfg(m, "myoFingerReachFixed-v0")
    for f in ("frame_skip", "max_episode_steps", "reach_nsite", "far_th", "reach_near_th", "reach_far_steps"):
        assert getattr(d, f) == getattr(r, f), f
    assert list(d.rwd_weight) == list(r.rwd_weight) and d.reach_target_site[0] == r.reach_target_site[0]


def test_reach_kwargs(product_lib):
    h = Model(asset_path("hand/myo_hand_pose.mjb"), lib=product_lib)
    rng = {s: ((0, 0, 0), (0.1, 0.2, 0.3)) for s in ("IFtip", "MFtip", "RFtip", "LFtip")}
    cfg = make_task_cfg(h, "myoFingerReachRandom-v0", target_reach_range=rng, far_th=0.5, frame_skip=10, max_episode_steps=50, normalize_act=False,
                        weighted_reward_keys={"reach": 2.0, "solved": 3.0})
    assert cfg.reach_nsite == 4 and [h.id2name("site", cfg.reach_target_site[k]) for k in range(4)] == ["IFtip_target", "MFtip_target", "RFtip_target", "LFtip_target"]
    assert cfg.far_th == pytest.approx(2.0) and cfg.reach_near_th == pytest.approx(0.05)     # both scale with the number of sites
    assert cfg.frame_skip == 10 and cfg.reach_far_steps == 2 and cfg.max_episode_steps == 50 and cfg.normalize_act == 0
    np.testing.assert_allclose(list(cfg.rwd_weight)[:7], [2, 0, 0, 0, 0, 3, 0])
    np.testing.assert_allclose(list(cfg.reach_range[3][1]), [0.1, 0.2, 0.3], rtol=1e-6)


def test_reach_errors(product_lib, emul_lib):
    m = Model(asset_path(FINGER), lib=product_lib)
    with pytest.raises(ValueError):
        make_task_cfg(m, "myoFingerReachRandom-v0", target_reach_range={"MFtip": ((0, 0, 0), (0, 0, 0))})      # not in the finger model
    with pytest.raises(ValueError):
        make_task_cfg(m, "myoFingerReachRandom-v0", target_reach_range={})
    h = Model(asset_path("hand/myo_hand_pose.mjb"), lib=product_lib)
    with pytest.raises(ValueError):
        make_task_cfg(h, "myoFingerReachRandom-v0", target_reach_range={s: ((0, 0, 0), (0, 0, 0)) for s in ("THtip", "IFtip", "MFtip", "RFtip", "LFtip")})
    with pytest.raises(TypeError):
        make_task_cfg(m, "myoFingerReachRandom-v0", pose_thd=0.1)
    with pytest.raises(ValueError):
        make_task_cfg(m, "myoFingerReachRandom-v0", weighted_reward_keys={"pose": 1.0})
    # the library refuses what make_task_cfg would not produce: more sites than override slots, bad site ids
    me = Model(asset_path(FINGER), lib=emul_lib)
    cfg = make_task_cfg(me, "myoFingerReachRandom-v0")
    cfg.reach_nsite = _capi.MYO_MAX_OVERRIDE + 1
    with pytest.raises(_capi.MyoError, match="MAX_OVERRIDE"):
        BatchSim(me, 4, cfg, device="cpu")
    cfg = make_task_cfg(me, "myoFingerReachRandom-v0")
    cfg.reach_target_site[0] = me.nsite
    with pytest.raises(_capi.MyoError):
        BatchSim(me, 4, cfg, device="cpu")


def test_far_th_gate_step_count():
    """MuJoCo sums time in fp64, one timestep per substep: after two env steps the sum is 0.020000000000000004 > 2 dt = 0.02
    (frame skip 5), and likewise for frame skip 10, so far_th applies from the second env step on; after one it does not."""
    assert reach_far_steps(0.002, 5) == 2 and reach_far_steps(0.002, 10) == 2
    t = 0.0
    for _ in range(10):
        t += 0.002
    assert t > 2 * 0.002 * 5 and not 0.01 > 2 * 0.002 * 5


def test_factory_creates_reach():
    """No longer NotImplementedError. Without a GPU it fails like every other config: no CPU path."""
    if torch.cuda.is_available():
        env = EnvironmentFactory.create("MyoFingerReachRandom", num_envs=4, device="cuda:0")
        assert env.observation_space.shape == (19,) and env.info_keys == REACH_KEYS
        return
    with pytest.raises(_capi.MyoError):
        EnvironmentFactory.create("MyoFingerReachRandom", num_envs=4, device="cuda:0")


@pytest.mark.parametrize("tag", fx.STEP_TAGS)
def test_reach_step_reproduces_the_shim_env(emul_lib, tag):
    fx.check_step_cases(emul_lib, "cpu", tag)


@pytest.mark.parametrize("tag", fx.RESET_TAGS)
def test_reach_reset_reproduces_the_shim_distribution(emul_lib, tag):
    fx.check_reset_distribution(emul_lib, "cpu", tag, n=768)
