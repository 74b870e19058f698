"""Kernel vs the reach fixtures (tests/golden/make_reach_fixtures.py: MyoSuite's ReachEnvV0 as restated in tests/shim, over the
fp64 oracle). Run through the single-lane host build of the kernel sources (CPU, tests/test_reach_host.py) and through the
CUDA library (tests/test_gpu_reach.py).

* step cases   : same pre-step state, target sites, env steps since the reset and action -> observation, the continuous reward
                 terms and the post-step state; done / solved / bonus bit-exact wherever the distance is clear of the threshold.
* reset samples: the target sites are compared in distribution (two-sample KS per coordinate; constant for a fixed range), the
                 state exactly (init_qpos, zero velocities and activations) and the observation through reach_err = target - tip.
"""
import json
import os

import numpy as np
import torch

from conftest import GOLDEN
from env_fixture_checks import _ks, _rel
from myochallenge_b200 import _capi, sim
from myochallenge_b200.assets import asset_path
from myochallenge_b200.envs import make_task_cfg

STEP_TAGS = ["finger_fixed", "finger_random", "finger_far", "hand_4tips"]
RESET_TAGS = ["finger_fixed", "finger_random", "hand_4tips"]
_FX = None


def fixtures():
    global _FX
    if _FX is None:
        f = np.load(os.path.join(GOLDEN, "reach_fixtures.npz"))
        _FX = (f, json.loads(str(f["meta"])))
    return _FX


def _get(group, tag):
    f, meta = fixtures()
    pre = f"{group}/{tag}/"
    return {k[len(pre):]: f[k] for k in f.files if k.startswith(pre)}, meta[group][tag]


def _make(lib, device, meta, n, seed=0, **extra):
    model = sim.Model(asset_path(meta["model"]), lib=lib)
    kw = dict(meta["config"])
    kw.update(extra)
    cfg = make_task_cfg(model, meta["env_id"], **kw)
    return model, cfg, sim.BatchSim(model, n, cfg, device=device, seed=seed)


def check_step_cases(lib, device, tag, obs_tol=2e-4):
    d, meta = _get("step", tag)
    n, ns = d["pre_target"].shape[:2]
    model, cfg, B = _make(lib, device, meta, n, auto_reset=0, max_episode_steps=100000)
    assert {0, 1} <= set(d["pre_elapsed"].tolist())          # the first two steps of an episode: far_th applies from the second on
    B.reset()
    B.set_state(d["pre_qpos"], d["pre_qvel"], d["pre_act"])
    for k in range(ns):
        B.set_param(_capi.PARAM_SITE_POS, cfg.reach_target_site[k], d["pre_target"][:, k])
    ti = np.zeros((n, _capi.TASK_STATE_I), np.int32)
    ti[:, 0], ti[:, 1] = d["pre_elapsed"], 1
    B.set_task_state(ti)
    obs, rew, done, trunc = [t.cpu().numpy().copy() for t in B.step(torch.as_tensor(d["action"], dtype=torch.float32).to(device))]
    info = B.info.cpu().numpy()
    q, v, a, _ = [t.cpu().numpy() for t in B.get_state()]
    assert not trunc.any()
    near, far = cfg.reach_near_th, cfg.far_th
    worst = 0.0
    for w in range(n):
        e = _rel(obs[w], d["obs"][w], 1e-2)
        worst = max(worst, e)
        assert e < obs_tol, f"{tag} case {w}: observation differs from the shim env's by {e:.2e}"
        np.testing.assert_allclose(info[w, [0, 2, 4]], d["terms"][w, [0, 2, 4]], rtol=2e-4, atol=2e-5, err_msg=f"{tag} case {w}: reward terms")
        dist = -d["terms"][w, 0]
        gated = d["pre_elapsed"][w] + 1 >= cfg.reach_far_steps
        if not gated:
            assert not done[w] and not d["done"][w] and info[w, 3] == 0, f"{tag} case {w}: far_th applied before the gate opened"
        if not gated or abs(dist - far) > 2e-5:
            assert bool(done[w]) == bool(d["done"][w]), f"{tag} case {w}: done flag"
            assert float(info[w, 6]) == float(d["terms"][w, 6]) and float(info[w, 3]) == float(d["terms"][w, 3]), f"{tag} case {w}: done / penalty"
        if min(abs(dist - near), abs(dist - 2 * near)) > 2e-5:
            assert float(info[w, 5]) == float(d["terms"][w, 5]), f"{tag} case {w}: solved flag"
            assert float(info[w, 1]) == float(d["terms"][w, 1]), f"{tag} case {w}: bonus"
            if not gated or abs(dist - far) > 2e-5:
                assert abs(rew[w] - d["reward"][w]) <= 2e-4 * max(1.0, abs(d["reward"][w])), f"{tag} case {w}: dense reward {rew[w]} vs {d['reward'][w]}"
        assert _rel(q[w], d["post_qpos"][w], 0.1) < obs_tol and _rel(a[w], d["post_act"][w], 0.1) < obs_tol
        assert _rel(v[w], d["post_qvel"][w], 1.0) < 2e-3
    assert B.status() & ~1 == 0
    return worst


def check_reset_distribution(lib, device, tag, n=1536, seed=11):
    d, meta = _get("reset", tag)
    model, cfg, B = _make(lib, device, meta, n, seed=seed)
    ns = cfg.reach_nsite
    obs = B.reset().cpu().numpy().copy()
    q, v, a, _ = [t.cpu().numpy() for t in B.get_state()]
    tgt = np.stack([B.get_param(_capi.PARAM_SITE_POS, cfg.reach_target_site[k]).cpu().numpy() for k in range(ns)], 1)
    for k in range(ns):
        for e in range(3):
            _ks(f"{tag}: target {k} site_pos[{e}]", tgt[:, k, e], d["target"][:, k, e])
            lo, hi = cfg.reach_range[k][0][e], cfg.reach_range[k][1][e]
            assert lo <= tgt[:, k, e].min() and tgt[:, k, e].max() <= hi
    # MujocoEnv.reset: init_qpos (the model's qpos0), zero velocities and activations, in every sample of both
    q0 = model.array("qpos0")
    np.testing.assert_allclose(q, np.tile(q0, (n, 1)), atol=1e-7)
    np.testing.assert_allclose(d["qpos"], np.tile(q0, (len(d["qpos"]), 1)), atol=1e-12)
    assert np.all(v == 0) and np.all(d["qvel"] == 0) and np.all(a == 0) and np.all(d["act"] == 0)
    # observation: tip_pos is the same in every reset; reach_err = target - tip, the targets hanging on the world body
    assert np.all(model.array("site_bodyid")[[cfg.reach_target_site[k] for k in range(ns)]] == 0)
    o0 = B.nq + B.nv
    for got, ref_tgt in ((obs, tgt), (d["obs"], d["target"])):
        tip, err = got[:, o0: o0 + 3 * ns], got[:, o0 + 3 * ns: o0 + 6 * ns]
        np.testing.assert_allclose(err, ref_tgt.reshape(len(got), -1) - tip, atol=2e-6)
    np.testing.assert_allclose(obs[:, o0: o0 + 3 * ns], np.tile(d["obs"][0, o0: o0 + 3 * ns], (n, 1)), atol=2e-6)
    np.testing.assert_array_equal(obs[:, o0 + 6 * ns:], 0)


def shim_env(meta):
    """ReachEnvV0 of tests/shim for a fixture-style meta (env_id, model, config); make_reach_fixtures puts the shim on sys.path."""
    import sys

    if GOLDEN not in sys.path:
        sys.path.insert(0, GOLDEN)
    import make_reach_fixtures

    return make_reach_fixtures.make_env(meta)


def check_rollout(lib, device, n=64, steps=200, seed=5):
    """``n`` myoFingerReachRandom worlds, ``steps`` env steps under seeded random actions (held for 5 steps); the shim env (fp64
    oracle) replays every world from the same reset with that world's targets and actions. Returns per-world (device length,
    device return, shim length, shim return), (margin of the distance to far_th, done flags agree) per compared step and the
    distance difference per compared step."""
    meta = dict(env_id="myoFingerReachRandom-v0", model="finger/myo_finger_v0.mjb", config={})
    model, cfg, B = _make(lib, device, meta, n, seed=seed, auto_reset=0, max_episode_steps=steps + 1)
    B.reset()
    tgt = B.get_param(_capi.PARAM_SITE_POS, cfg.reach_target_site[0]).cpu().numpy().astype(np.float64)
    rng = np.random.default_rng(seed)
    acts, rews, dones, dists = [], [], [], []
    a = None
    for t in range(steps):
        if t % 5 == 0:
            a = rng.uniform(-1, 1, (n, B.nu)).astype(np.float32)
        _, rew, done, _ = B.step(torch.as_tensor(a).to(device))
        acts.append(a.copy()); rews.append(rew.cpu().numpy().copy()); dones.append(done.cpu().numpy().astype(bool))
        dists.append(-B.info[:, 0].cpu().numpy().copy())
    rews, dones, dists = np.array(rews), np.array(dones), np.array(dists)
    first = np.where(dones.any(0), dones.argmax(0), steps - 1)
    g_len, g_ret = first + 1, np.array([rews[: first[w] + 1, w].sum() for w in range(n)])
    env = shim_env(meta)
    o_len, o_ret = np.full(n, steps), np.zeros(n)
    flags, dist_err = [], []
    for w in range(n):
        env.reset()
        env.sim.model.site_pos[env.target_sids[0]] = tgt[w]
        env.sim.forward()
        for t in range(steps):
            _, r, done, info = env.step(acts[t][w].astype(np.float64))
            o_ret[w] += r
            dist = -float(np.squeeze(info["rwd_dict"]["reach"]))
            if t < g_len[w]:
                margin = min(abs(dist - cfg.far_th), abs(dists[t, w] - cfg.far_th))
                flags.append((margin, bool(done) == bool(dones[t, w])))
                dist_err.append(abs(dist - dists[t, w]))
            if done:
                o_len[w] = t + 1
                break
    assert B.status() & ~1 == 0
    return g_len, g_ret, o_len, o_ret, np.array(flags), np.array(dist_err)
