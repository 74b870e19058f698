"""CPU: MyoSuite's ``obs_keys`` and ``reward_mode`` env kwargs. Key translation per task kind, the "act" append rule and the error
cases; then, through the host build of the kernel sources (tests/emul), the gathered observation against the columns of the default
one for every kind, the sparse reward, and the finger reach env against the shim's ReachEnvV0 over the fp64 oracle.
The GPU run of the same contract is tests/test_gpu_obs_keys.py."""
import numpy as np
import pytest
import torch

import reach_fixture_checks as fx
from env_fixture_checks import _rel
from myochallenge_b200 import _capi
from myochallenge_b200.assets import asset_path
from myochallenge_b200.envs import REGISTRY, make_task_cfg
from myochallenge_b200.sim import BatchSim, Model
from myochallenge_b200.vec_env import DEFAULT_OBS_KEYS, OBS_KEYS

# env id, a permuted subset of keys with t (and a duplicate where the kind has enough keys); "act" is appended unless listed
CASES = {
    "baoding": ("CustomMyoChallengeBaodingP2-v1", ["target2_err", "t", "act", "object1_pos", "hand_pos", "object2_velp", "target1_pos", "target1_pos"]),
    "die": ("CustomMyoChallengeDieReorientP2-v0", ["rot_err", "t", "hand_qvel", "obj_pos", "pos_err", "goal_rot"]),
    "elbow": ("CustomMyoElbowPoseRandom-v0", ["pose_err", "t", "qvel"]),
    "reach": ("myoFingerReachRandom-v0", ["reach_err", "target_pos", "t", "act", "qpos"]),
}


def default_columns(kind, nq, nv, na, nsite=1):
    """key -> column indices in the kind's default observation ("t" and reach's "target_pos" have none)."""
    if kind == _capi.TASK_BAODING:
        widths = [("hand_pos", nq - 14)] + [(k, 3) for k in DEFAULT_OBS_KEYS[kind][1:]]
    elif kind == _capi.TASK_REORIENT:
        widths = [("hand_qpos", nq - 7), ("hand_qvel", nv - 6)] + [(k, 3) for k in DEFAULT_OBS_KEYS[kind][2:]]
    elif kind == _capi.TASK_POSE:
        widths = [("qpos", nq), ("qvel", nv), ("pose_err", nq)]
    else:
        widths = [("qpos", nq), ("qvel", nv), ("tip_pos", 3 * nsite), ("reach_err", 3 * nsite)]
    cols, o = {}, 0
    for k, w in widths + [("act", na)]:
        cols[k] = np.arange(o, o + w)
        o += w
    return cols


def expected_obs(keys, default_obs, time, cols):
    """The custom observation assembled from the default one: t from the world's time, target_pos = tip_pos + reach_err."""
    parts = []
    for k in keys:
        if k == "t":
            parts.append(np.asarray(time, np.float32).reshape(-1, 1))
        elif k == "target_pos":
            parts.append(default_obs[:, cols["tip_pos"]] + default_obs[:, cols["reach_err"]])
        else:
            parts.append(default_obs[:, cols[k]])
    return np.concatenate(parts, axis=1)


def _model(env_id, lib):
    return Model(asset_path(REGISTRY[env_id]["model"]), lib=lib)


# ---- key translation -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", sorted(CASES))
def test_key_translation(product_lib, tag):
    env_id, keys = CASES[tag]
    m = _model(env_id, product_lib)
    cfg = make_task_cfg(m, env_id, obs_keys=keys)
    known = OBS_KEYS[cfg.kind]
    want = keys if "act" in keys else keys + ["act"]
    assert cfg.n_obs_keys == len(want) and [known[cfg.obs_keys[i]] for i in range(cfg.n_obs_keys)] == want
    assert cfg.reward_sparse == 0
    assert make_task_cfg(m, env_id).n_obs_keys == 0                    # no obs_keys: the default layout
    assert make_task_cfg(m, env_id, reward_mode="sparse").reward_sparse == 1
    assert make_task_cfg(m, env_id, reward_mode="dense").reward_sparse == 0


def test_key_ids_follow_the_header():
    """The Python key tables are numbered as the MYO_OBS_<KIND>_* enums of include/myo_b200.h."""
    import os
    import re

    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "myo_b200.h")).read()
    for kind, name in ((_capi.TASK_BAODING, "BAODING"), (_capi.TASK_REORIENT, "REORIENT"), (_capi.TASK_POSE, "POSE"), (_capi.TASK_REACH, "REACH")):
        ids = {k.lower(): int(v) for k, v in re.findall(rf"MYO_OBS_{name}_(\w+) = (\d+)", src)}
        assert ids.pop("count") == len(OBS_KEYS[kind])
        assert ids == {k: i for i, k in enumerate(OBS_KEYS[kind])}


def test_act_append_rule(product_lib):
    m = _model("myoFingerReachRandom-v0", product_lib)
    cfg = make_task_cfg(m, "myoFingerReachRandom-v0", obs_keys=["act", "qpos"])          # already listed: not appended again
    assert cfg.n_obs_keys == 2 and list(cfg.obs_keys)[:2] == [OBS_KEYS[_capi.TASK_REACH].index(k) for k in ("act", "qpos")]
    cfg = make_task_cfg(m, "myoFingerReachRandom-v0", obs_keys=["qpos", "qpos"])        # duplicates stay
    assert cfg.n_obs_keys == 3
    # a model without activations (na = 0) gets no "act"
    motor = Model(asset_path("finger/motor_finger_v0.mjb"), lib=product_lib)
    assert motor.na == 0
    cfg = make_task_cfg(motor, "myoFingerPoseRandom-v0", obs_keys=["qpos", "t"])
    assert cfg.n_obs_keys == 2


def test_errors(product_lib):
    m = _model("CustomMyoChallengeBaodingP2-v1", product_lib)
    with pytest.raises(ValueError, match="hand_pos"):                       # names the known keys
        make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", obs_keys=["qpos"])
    with pytest.raises(ValueError, match="empty"):
        make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", obs_keys=[])
    with pytest.raises(ValueError, match="at most 16"):
        make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", obs_keys=["t"] * 16)     # 16 + "act"
    assert make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", obs_keys=["t"] * 15).n_obs_keys == 16
    with pytest.raises(ValueError):
        make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", obs_keys="hand_pos")
    with pytest.raises(ValueError, match="reward_mode"):
        make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", reward_mode="shaped")


def test_library_refuses_bad_keys(emul_lib):
    m = _model("myoFingerReachRandom-v0", emul_lib)
    cfg = make_task_cfg(m, "myoFingerReachRandom-v0", obs_keys=["qpos"])
    cfg.obs_keys[0] = len(OBS_KEYS[_capi.TASK_REACH])                        # one past the kind's last key
    with pytest.raises(_capi.MyoError, match="key id") as e:
        BatchSim(m, 2, cfg, device="cpu")
    assert "error -1" in str(e.value)                                         # MYO_E_ARG
    cfg = make_task_cfg(m, "myoFingerReachRandom-v0")
    cfg.n_obs_keys = _capi.MYO_MAX_OBS_KEYS + 1
    with pytest.raises(_capi.MyoError, match="error -6"):                     # MYO_E_LIMIT
        BatchSim(m, 2, cfg, device="cpu")


@pytest.mark.parametrize("keys,width", [(None, 19), (["t"], 1 + 5), (["qpos", "qvel", "tip_pos", "reach_err", "act"], 19),
                                        (["target_pos", "target_pos", "t"], 3 + 3 + 1 + 5), (["act", "t", "act"], 5 + 1 + 5)])
def test_nobs(emul_lib, keys, width):
    """Finger reach: nq = nv = 4, na = 5, one site."""
    m = _model("myoFingerReachRandom-v0", emul_lib)
    kw = {} if keys is None else dict(obs_keys=keys)
    B = BatchSim(m, 2, make_task_cfg(m, "myoFingerReachRandom-v0", **kw), device="cpu")
    assert B.nobs == width and tuple(B.obs.shape) == (2, width)


# ---- the emulated kernel ---------------------------------------------------------------------------------------------------
def _pair(env_id, keys, lib, n, seed=3, **kw):
    m = _model(env_id, lib)
    d = BatchSim(m, n, make_task_cfg(m, env_id, **kw), device="cpu", seed=seed)
    c = BatchSim(m, n, make_task_cfg(m, env_id, obs_keys=keys, **kw), device="cpu", seed=seed)
    return m, d, c


@pytest.mark.parametrize("tag", sorted(CASES))
def test_emulated_gather_matches_default_columns(emul_lib, tag):
    env_id, keys = CASES[tag]
    n, steps = 3, 6
    m, d, c = _pair(env_id, keys, emul_lib, n, max_episode_steps=4)      # one auto-reset inside the run
    full = keys if "act" in keys else keys + ["act"]
    cols = default_columns(d.cfg.kind, d.nq, d.nv, d.na, max(d.cfg.reach_nsite, 1))
    od, oc = d.reset().numpy().copy(), c.reset().numpy().copy()
    np.testing.assert_array_equal(oc, expected_obs(full, od, np.zeros(n), cols))
    rng = np.random.default_rng(0)
    dt = np.float32(d.cfg.frame_skip * m.opt("timestep"))
    for k in range(steps):
        a = torch.as_tensor(rng.uniform(-1, 1, (n, d.nu)).astype(np.float32))
        t_prev = c.get_state()[3].numpy().copy()
        rd, rc = d.step(a), c.step(a)
        od, oc = rd[0].numpy().copy(), rc[0].numpy().copy()
        for x, y in zip(rd[1:], rc[1:]):
            np.testing.assert_array_equal(x.numpy(), y.numpy())
        np.testing.assert_array_equal(d.info.numpy(), c.info.numpy())
        time = c.get_state()[3].numpy()
        np.testing.assert_array_equal(d.get_state()[3].numpy(), time)
        np.testing.assert_array_equal(oc, expected_obs(full, od, time, cols), err_msg=f"{tag} step {k}")
        done = rd[2].numpy().astype(bool)
        if done.any():
            assert np.all(time[done] == 0)
            # the terminal observation carries the time of the step that ended the episode
            t_end = (t_prev + dt)[done][:, None]
            exp_t = expected_obs(full, d.terminal_obs.numpy()[done], np.full(done.sum(), np.nan), cols)
            got_t = c.terminal_obs.numpy()[done]
            tcol = np.array([i for i, kk in enumerate(_expand(full, d.cfg.kind, cols)) if kk == "t"])
            np.testing.assert_array_equal(np.delete(got_t, tcol, 1), np.delete(exp_t, tcol, 1))
            assert np.allclose(got_t[:, tcol], t_end, rtol=1e-6) and np.all(got_t[:, tcol] > 0)
    assert d.get_task_state()[0][:, 1].min() >= 2                          # every world went through an auto-reset
    # get_obs (MODE_GET_OBS) goes through the same gather
    np.testing.assert_array_equal(c.get_obs().numpy(), expected_obs(full, d.get_obs().numpy(), c.get_state()[3].numpy(), cols))


def _expand(keys, kind, cols):
    """Per output column, the key it belongs to."""
    out = []
    for k in keys:
        w = 1 if k == "t" else len(cols["tip_pos"] if k == "target_pos" else cols[k])
        out += [k] * w
    return out


@pytest.mark.parametrize("tag", sorted(CASES))
def test_emulated_sparse_reward(emul_lib, tag):
    env_id, _ = CASES[tag]
    m = _model(env_id, emul_lib)
    dense = BatchSim(m, 2, make_task_cfg(m, env_id), device="cpu", seed=1)
    sparse = BatchSim(m, 2, make_task_cfg(m, env_id, reward_mode="sparse"), device="cpu", seed=1)
    dense.reset(); sparse.reset()
    rng = np.random.default_rng(1)
    for _ in range(3):
        a = torch.as_tensor(rng.uniform(-1, 1, (2, dense.nu)).astype(np.float32))
        rd, rs = dense.step(a), sparse.step(a)
        np.testing.assert_array_equal(dense.info.numpy(), sparse.info.numpy())      # info columns do not change
        np.testing.assert_array_equal(rd[1].numpy(), dense.info.numpy()[:, 7])
        np.testing.assert_array_equal(rs[1].numpy(), sparse.info.numpy()[:, 4])
        np.testing.assert_array_equal(rd[0].numpy(), rs[0].numpy())


def test_reach_against_the_shim_env(emul_lib):
    """Custom obs_keys + reward_mode="sparse" on myoFingerReachRandom: the emulated kernel against ReachEnvV0 of tests/shim over the
    fp64 oracle, from the same reset (the kernel's drawn targets copied into the shim env) under the same actions."""
    keys = ["reach_err", "t", "target_pos", "qvel"]
    meta = dict(env_id="myoFingerReachRandom-v0", model="finger/myo_finger_v0.mjb", config=dict(obs_keys=keys, reward_mode="sparse"))
    n, steps = 3, 8
    model, cfg, B = fx._make(emul_lib, "cpu", meta, n, seed=2, auto_reset=0, max_episode_steps=steps + 1)
    obs0 = B.reset().numpy().copy()
    tgt = B.get_param(_capi.PARAM_SITE_POS, cfg.reach_target_site[0]).numpy().astype(np.float64)
    rng = np.random.default_rng(2)
    acts = rng.uniform(-1, 1, (steps, n, B.nu)).astype(np.float32)
    got_obs, got_rew = [], []
    for t in range(steps):
        o, r, _, _ = B.step(torch.as_tensor(acts[t]))
        got_obs.append(o.numpy().copy()); got_rew.append(r.numpy().copy())
    env = fx.shim_env(meta)
    assert env.obs_keys == keys + ["act"] and env.rwd_mode == "sparse"
    for w in range(n):
        env.reset()
        env.sim.model.site_pos[env.target_sids[0]] = tgt[w]
        env.sim.forward()
        o = env.get_obs()
        assert o.shape == obs0[w].shape and _rel(obs0[w], o, 1e-2) < 2e-4
        for t in range(steps):
            o, r, _, info = env.step(acts[t][w].astype(np.float64))
            assert _rel(got_obs[t][w], o, 1e-2) < 2e-4, f"world {w} step {t}: observation"
            assert r == info["rwd_sparse"]
            assert abs(got_rew[t][w] - r) <= 2e-4 * max(1.0, abs(r)), f"world {w} step {t}: sparse reward {got_rew[t][w]} vs {r}"


# ---- Python front end ------------------------------------------------------------------------------------------------------
class _Stub:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def test_vecnormalize_load_names_both_widths(tmp_path):
    from myochallenge_b200 import checkpoint
    from myochallenge_b200.rollout import DeviceVecNormalize
    from myochallenge_b200.vec_env import Box, VecNormalize

    path = str(tmp_path / "vn.pkl")
    checkpoint.save_vecnormalize(path, dict(obs_mean=np.zeros(86), obs_var=np.ones(86), obs_count=1.0, ret_mean=0.0, ret_var=1.0, ret_count=1.0),
                                 4, 39)
    venv = _Stub(num_envs=4, observation_space=Box(-10, 10, (50,)), action_space=Box(-1, 1, (39,)), sim=_Stub(nobs=50))
    with pytest.raises(ValueError, match="86.*50"):
        VecNormalize.load(path, venv)
    with pytest.raises(ValueError, match="86.*50"):
        DeviceVecNormalize.load(path, venv)
    venv.observation_space = Box(-10, 10, (86,))
    assert VecNormalize.load(path, venv).obs_rms.mean.shape == (86,)


def test_classifier_refuses_a_custom_layout():
    from myochallenge_b200.ensemble import MixtureOfEnsembles, TaskClassifier, evaluate_mixture

    default = DEFAULT_OBS_KEYS[_capi.TASK_BAODING] + ("act",)
    TaskClassifier.check_env(_Stub(cfg=_Stub(kind=_capi.TASK_BAODING), obs_keys=default))
    custom = _Stub(cfg=_Stub(kind=_capi.TASK_BAODING), obs_keys=("t",) + default)
    with pytest.raises(ValueError, match="obs\\[29:47\\]"):
        TaskClassifier.check_env(custom)
    with pytest.raises(ValueError, match="obs\\[29:47\\]"):
        evaluate_mixture(MixtureOfEnsembles.__new__(MixtureOfEnsembles), custom)
