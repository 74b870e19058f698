"""TEST INFRASTRUCTURE - generates tests/golden/reach_fixtures.npz from the ReachEnvV0 restatement in tests/shim (MyoSuite 1.2.3
envs/myo/reach_v0.py from memory, [3P-MEM]) over the fp64 oracle. No file of the reference builds on that env, so it needs no
reference sources: tests/shim goes on sys.path directly (shim.install() is not called).

* ``reset/<tag>/...``  raw samples of what ``reset()`` decides: target site_pos of every site, post-reset qpos / qvel / act and
  the observation - the distribution the device reset (csrc/myo_task.cuh task_reset) has to reproduce;
* ``step/<tag>/...``   deterministic cases: pre-step state, target sites, env steps since the reset, action -> observation,
  every reward term, done flag and post-step state. Each episode's first steps are all kept, so that the cases cover the
  steps before and after ReachEnvV0 starts applying far_th (data.time > 2 dt).

Tags: the two finger registrations; ``finger_far`` (far_th small enough that episodes end); ``hand_4tips`` (the hand pose model,
four tips, a user range around each tip). Everything is seeded.

    python tests/golden/make_reach_fixtures.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for _p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "shim"), ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

M_RESET = 256
TERMS = ("reach", "bonus", "act_reg", "penalty", "sparse", "solved", "done", "dense")
HAND_TIPS = ("IFtip", "MFtip", "RFtip", "LFtip")


def asset(rel):
    return os.path.join(ROOT, "myochallenge_b200", "assets", rel)


def make_env(meta):
    """The shim env for a fixture tag: the registration's kwargs (myochallenge_b200.envs.REGISTRY) updated by the tag's config."""
    from myochallenge_b200.envs import REGISTRY
    from myosuite.envs.myo.reach_v0 import ReachEnvV0

    reg = REGISTRY[meta["env_id"]]
    kw = dict(reg["kwargs"])
    kw.update(meta["config"])
    kw["target_reach_range"] = {s: (tuple(lo), tuple(hi)) for s, (lo, hi) in kw["target_reach_range"].items()}
    return ReachEnvV0(model_path=asset(meta["model"]), **kw)


def targets(env):
    m = env.sim.model
    return np.array([np.array(m.site_pos[sid]) for sid in env.target_sids])


def reset_samples(meta, n, seed):
    env = make_env(meta)
    env.seed(seed)
    out = []
    for _ in range(n):
        obs = env.reset()
        d = env.sim.data
        out.append(dict(target=targets(env), qpos=np.array(d.qpos), qvel=np.array(d.qvel), act=np.array(d.act), obs=np.array(obs, np.float32)))
    return {k: np.array([s[k] for s in out]) for k in out[0]}


def step_cases(meta, n_cases, seed, every=4, horizon=40, first=4):
    env = make_env(meta)
    env.seed(seed)
    rng = np.random.RandomState(seed + 1)
    nu = env.sim.model.nu
    cases = []
    while len(cases) < n_cases:
        env.reset()
        a = None
        for t in range(horizon):
            if t % 5 == 0:
                a = rng.uniform(-1, 1, nu)
            d = env.sim.data
            pre = dict(pre_qpos=np.array(d.qpos), pre_qvel=np.array(d.qvel), pre_act=np.array(d.act), pre_target=targets(env), pre_elapsed=t)
            obs, rew, done, info = env.step(a)
            if t < first or t % every == 0 or done:
                c = dict(pre)
                c.update(action=np.array(a), obs=np.array(obs, np.float32), reward=float(rew), done=bool(info["done"]),
                         terms=np.array([float(np.squeeze(info["rwd_dict"][k])) for k in TERMS]), post_qpos=np.array(d.qpos),
                         post_qvel=np.array(d.qvel), post_act=np.array(d.act))
                cases.append(c)
            if done:
                break
    return {k: np.array([c[k] for c in cases[:n_cases]]) for k in cases[0]}


def hand_range():
    """IF / MF / RF / LF tips of the hand pose model at qpos0, and a box around each (the targets a user range would give)."""
    from oracle import oracle

    path = asset("hand/myo_hand_pose.mjb")
    om, od = oracle.load(path)
    from oracle import mjb
    names = mjb.load(path).names_of("site")
    od.reset()
    od.call("o_kinematics")
    rng = {}
    for s in HAND_TIPS:
        p = np.array(od.site_xpos[names.index(s)])
        rng[s] = [list(np.round(p + [-0.04, -0.04, -0.04], 4)), list(np.round(p + [0.02, 0.02, 0.02], 4))]
    return rng


def main():
    out = {}
    meta = {"reset": {}, "step": {}}
    tags = [("finger_fixed", dict(env_id="myoFingerReachFixed-v0", model="finger/myo_finger_v0.mjb", config={}), True),
            ("finger_random", dict(env_id="myoFingerReachRandom-v0", model="finger/myo_finger_v0.mjb", config={}), True),
            ("finger_far", dict(env_id="myoFingerReachRandom-v0", model="finger/myo_finger_v0.mjb", config=dict(far_th=0.05)), False),
            ("hand_4tips", dict(env_id="myoFingerReachRandom-v0", model="hand/myo_hand_pose.mjb",
                                config=dict(target_reach_range=hand_range(), far_th=0.02)), True)]
    for i, (tag, m, with_reset) in enumerate(tags):
        groups = [("step", step_cases(m, 48, 700 + i))]
        if with_reset:
            groups.append(("reset", reset_samples(m, M_RESET, 300 + i)))
        for group, data in groups:
            meta[group][tag] = m
            for k, v in data.items():
                out[f"{group}/{tag}/{k}"] = np.asarray(v)
        print(tag, flush=True)
    out["meta"] = np.array(json.dumps(meta))
    path = os.path.join(HERE, "reach_fixtures.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
