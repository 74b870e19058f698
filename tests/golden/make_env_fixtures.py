"""TEST INFRASTRUCTURE - generates tests/golden/env_fixtures.npz by RUNNING THE REFERENCE'S OWN ENV CODE.

/root/reference/src/envs/{baoding,pose}.py are imported unmodified (through tests/shim: stand-ins for gym / MyoSuite / SB3,
physics = the fp64 oracle) and driven through ``EnvironmentFactory.create(name, **config)``, ``reset()`` and ``step()``:

* ``reset/<tag>/...``  raw samples of everything ``reset()`` decides (task, start angles, radii, period, ball mass / size /
  friction, counter, post-reset qpos / act / target sites / observation) for the 32 steps of the winning curriculum
  (myochallenge_b200/assets/curriculum/baoding_winner.json = the reference's config.json files), the two stock registrations
  and the pose envs - the distributions the device reset (csrc/myo_task.cuh task_reset) has to reproduce;
* ``step/<tag>/...``   deterministic cases: full pre-step state + task attributes + action -> the reference's observation,
  every term of its ``get_reward_dict``, done flag and post-step state, for the kernel to reproduce from the same state.

All three host RNGs the reference draws from (env.np_random, numpy's global, ``random``) are seeded; the recorded streams
are what make the fixtures reproducible. Only runs where /root/reference exists; the .npz travels with the repository.
``shrink`` keeps the stored file under 1 MB (see its docstring).

    python tests/golden/make_env_fixtures.py
"""
import json
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

M_RESET = 256
STEP_KEEP = 0.4         # share of each tag's non-terminal step cases that is stored (shrink)
BAODING_RESET_OBS = [23, 24, 29, 30, 35, 36, 38, 39]      # ball xy and target xy: the reset observation columns the checks read
BAODING_TERMS = ("pos_dist_1", "pos_dist_2", "act_reg", "alive", "sparse", "solved", "done", "dense")
POSE_TERMS = ("pose", "bonus", "penalty", "act_reg", "sparse", "solved", "done", "dense")
REORIENT_TERMS = ("pos_dist", "rot_dist", "act_reg", "alive", "sparse", "solved", "done", "dense", "pos_dist_diff", "rot_dist_diff")


def seed_all(env, s):
    np.random.seed(s)
    random.seed(s)
    env.seed(s)


def instrument(u):
    """Capture the time period handed to create_goal_trajectory (the HOLD task's goal table is all zeros)."""
    orig = u.create_goal_trajectory
    u._fx_period = np.nan

    def wrapped(time_step=0.1, time_period=6):
        u._fx_period = float(time_period)
        return orig(time_step=time_step, time_period=time_period)

    u.create_goal_trajectory = wrapped


def baoding_snapshot(u):
    m, d = u.sim.model, u.sim.data
    b = [getattr(u, "object%d_bid" % k, m.body_name2id("ball%d" % k)) for k in (1, 2)]
    g = [u.object1_gid, u.object2_gid]
    return dict(task=u.which_task.value, angle1=u.ball_1_starting_angle, angle2=u.ball_2_starting_angle, xr=u.x_radius, yr=u.y_radius,
                period=u._fx_period, counter=u.counter, mass=[m.body_mass[b[0]], m.body_mass[b[1]]],
                size=[m.geom_size[g[0]][0], m.geom_size[g[1]][0]], fric=[np.array(m.geom_friction[g[0]]), np.array(m.geom_friction[g[1]])],
                target_xy=[m.site_pos[u.target1_sid][0], m.site_pos[u.target1_sid][1], m.site_pos[u.target2_sid][0], m.site_pos[u.target2_sid][1]],
                qpos=np.array(d.qpos), qvel=np.array(d.qvel), act=np.array(d.act))


def reorient_snapshot(u):
    m, d = u.sim.model, u.sim.data
    g0, gn = u.object_gid0, u.object_gidn
    return dict(goal_pos=np.array(m.body_pos[u.goal_bid]), goal_quat=np.array(m.body_quat[u.goal_bid]), die_size=np.array(m.geom_size[g0:gn]),
                die_fric=np.array(m.geom_friction[g0:gn]), pos_dist=float(u.pos_dist), rot_dist=float(u.rot_dist),
                qpos=np.array(d.qpos), qvel=np.array(d.qvel), act=np.array(d.act))


def env_kind(u):
    return "baoding" if hasattr(u, "which_task") else ("reorient" if hasattr(u, "goal_bid") else "pose")


def stack(snaps):
    return {k: np.array([s[k] for s in snaps]) for k in snaps[0]}


def reset_samples(env_name, config, n, seed, instances=1):
    """n resets of one env object - or, with ``instances`` > 1, n / instances resets of each of that many env objects (what
    ``_setup`` decides once per object, e.g. the fixed task's start angles, only varies between objects)."""
    if instances > 1:
        np.random.seed(seed); random.seed(seed)
        parts = []
        for k in range(instances):
            part = reset_samples(env_name, config, n // instances, None)
            part["instance"] = np.full(n // instances, k)
            parts.append(part)
        return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    cfg = {k: (tuple(v) if isinstance(v, list) else v) for k, v in config.items()}
    env = EnvironmentFactory.create(env_name, **cfg)
    u = env.unwrapped
    if seed is not None:
        seed_all(env, seed)
    out = []
    if env_kind(u) == "baoding":
        instrument(u)
        for _ in range(n):
            obs = env.reset()
            s = baoding_snapshot(u)
            s["obs"] = np.array(obs)
            out.append(s)
    elif env_kind(u) == "reorient":
        for _ in range(n):
            obs = env.reset()
            s = reorient_snapshot(u)
            s["obs"] = np.array(obs)
            out.append(s)
    else:
        for _ in range(n):
            obs = env.reset()
            rec = dict(target=np.array(u.target_jnt_value, float), qpos=np.array(u.sim.data.qpos), qvel=np.array(u.sim.data.qvel),
                       act=np.array(u.sim.data.act), obs=np.array(obs))
            if u.weight_bodyname is not None:
                bid = u.sim.model.body_name2id(u.weight_bodyname)
                rec["weight_mass"] = float(u.sim.model.body_mass[bid])
                rec["weight_size0"] = float(u.sim.model.geom_size[u.sim.model.body_geomadr[bid]][0])
            out.append(rec)
    return stack(out)


def step_cases(env_name, config, n_cases, seed, every=3, horizon=40):
    cfg = {k: (tuple(v) if isinstance(v, list) else v) for k, v in config.items()}
    env = EnvironmentFactory.create(env_name, **cfg)
    u = env.unwrapped
    seed_all(env, seed)
    rng = np.random.RandomState(seed + 1)
    kind = env_kind(u)
    baoding = kind == "baoding"
    if baoding:
        instrument(u)
    terms = dict(baoding=BAODING_TERMS, pose=POSE_TERMS, reorient=REORIENT_TERMS)[kind]
    cases = []
    while len(cases) < n_cases:
        env.reset()
        a = None
        for t in range(horizon):
            if t % 5 == 0:
                a = rng.uniform(-1, 1, u.sim.model.nu)
            pre = baoding_snapshot(u) if baoding else (reorient_snapshot(u) if kind == "reorient" else
                                                       dict(target=np.array(u.target_jnt_value, float), qpos=np.array(u.sim.data.qpos),
                                                            qvel=np.array(u.sim.data.qvel), act=np.array(u.sim.data.act)))
            obs, rew, done, info = env.step(a)
            if t % every == 0 or done:
                c = {"pre_" + k: v for k, v in pre.items()}
                c.update(action=np.array(a), obs=np.array(obs), reward=float(rew), done=bool(info["done"]),
                         terms=np.array([float(np.squeeze(info["rwd_dict"][k])) for k in terms]), post_qpos=np.array(u.sim.data.qpos),
                         post_qvel=np.array(u.sim.data.qvel), post_act=np.array(u.sim.data.act))
                if baoding:
                    c["post_counter"] = u.counter
                cases.append(c)
            if done:
                break
    return stack(cases[:n_cases])


def shrink(out, meta, seed=0):
    """Cuts the recorded fixtures down to what tests/env_fixture_checks.py reads, so that the .npz stays under 1 MB:
    step observations in float32 (the checks compare them to 2e-4); reset observations (float64: their distributions are
    compared value by value) only in the columns the checks read (``obs_cols`` names them; pose resets keep none); of each
    tag's step cases every terminal one and a seeded ``STEP_KEEP`` share of the others."""
    rng = np.random.default_rng(seed)
    out = dict(out)
    for tag in meta["reset"]:
        pre = f"reset/{tag}/"
        obs = out.pop(pre + "obs")
        if pre + "task" in out:
            cols = np.array(BAODING_RESET_OBS)
        elif pre + "goal_quat" in out:          # die: object and goal pose, their errors (obs[o0 : o0 + 18])
            o0 = (out[pre + "qpos"].shape[1] - 7) + (out[pre + "qvel"].shape[1] - 6)
            cols = np.arange(o0, o0 + 18)
        else:
            continue
        out[pre + "obs"] = obs[:, cols]
        out[pre + "obs_cols"] = cols.astype(np.int32)
    for tag in meta["step"]:
        pre = f"step/{tag}/"
        done = np.asarray(out[pre + "done"], bool)
        rest = np.flatnonzero(~done)
        keep = np.sort(np.concatenate([np.flatnonzero(done), rng.choice(rest, int(np.ceil(STEP_KEEP * len(rest))), replace=False)]))
        for k in [k for k in out if k.startswith(pre)]:
            out[k] = out[k][keep]
        out[pre + "obs"] = out[pre + "obs"].astype(np.float32)
    return out


def main():
    global EnvironmentFactory
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import shim

    shim.install()                  # the reference's sources: imported here so that ``shrink`` imports without them
    import envs  # noqa: F401  (the reference's registrations)
    from envs.environment_factory import EnvironmentFactory
    from myosuite.envs.myo.myochallenge.baoding_v1 import Task  # noqa: F401
    cur = json.load(open(os.path.join(ROOT, "myochallenge_b200", "assets", "curriculum", "baoding_winner.json")))["steps"]
    out = {}
    meta = {"reset": {}, "step": {}}

    def put(group, tag, env_name, config, data):
        meta[group][tag] = dict(env_name=env_name, config=config)
        for k, v in data.items():
            v = np.asarray(v)
            out[f"{group}/{tag}/{k}"] = v.astype(np.float32) if v.dtype == np.float64 and k not in ("obs", "terms", "reward") else v

    for i, st in enumerate(cur):
        put("reset", "cur%02d" % (i + 1), st["env_name"], st["config"], reset_samples(st["env_name"], st["config"], M_RESET, 100 + i))
        print("reset", st["step"], flush=True)
    extra = [("p2_default", "CustomMyoBaodingBallsP2", {}), ("p1_default", "CustomMyoBaodingBallsP1", {}),
             ("p2_knobs", "CustomMyoBaodingBallsP2", dict(enable_rsi=True, rsi_probability=0.6, balls_overlap=False, overlap_probability=0.3,
                                                          limit_init_angle=0.8, beta_init_angle=[2.0, 5.0], beta_ball_size=[2.0, 2.0], beta_ball_mass=[5.0, 2.0],
                                                          noise_fingers=0.5)),
             ("p2_fixed_task", "CustomMyoBaodingBallsP2", dict(task_choice="fixed", overlap_probability=0.5)),
             ("p1_noise", "CustomMyoBaodingBallsP1", dict(task="random", enable_rsi=True, rsi_probability=0.7, noise_palm=0.6, noise_fingers=0.4, noise_balls=0.004)),
             ("finger_random", "CustomMyoFingerPoseRandom", {}), ("finger_fixed", "CustomMyoFingerPoseFixed", {}),
             ("elbow_random", "CustomMyoElbowPoseRandom", {}), ("hand_random", "CustomMyoHandPoseRandom", {}),
             ("hand_fixed", "CustomMyoHandPoseFixed", {}),
             ("finger_distance", "CustomMyoFingerPoseRandom", dict(target_distance=0.4, reset_type="init")),
             ("elbow_sds", "CustomMyoElbowPoseRandom", dict(reset_type="sds", sds_distance=0.3, target_distance=0.6, weight_bodyname=None, weight_range=None)),
             ("finger_sds0", "CustomMyoFingerPoseRandom", dict(reset_type="sds", sds_distance=0, weight_bodyname=None, weight_range=None)),
             ("elbow_weight", "CustomMyoElbowPoseRandom", dict(weight_bodyname="forearm", weight_range=(0.5, 2.0))),
             ("die_p1", "CustomMyoReorientP1", {}), ("die_p2", "CustomMyoReorientP2", {}),
             ("die_axes", "CustomMyoReorientP2", dict(goal_rot_x=[(-0.5, 0.5), (1.0, 1.2)], goal_rot_z=[(0.0, 0.0)], enable_rsi=True,
                                                      rsi_distance_pos=0.5, rsi_distance_rot=0.5))]
    for tag, name, cfg in extra:
        put("reset", tag, name, cfg, reset_samples(name, cfg, M_RESET, 500 + len(meta["reset"]), instances=32 if tag == "p2_fixed_task" else 1))
        print("reset", tag, flush=True)
    step_sets = [("p2_default", "CustomMyoBaodingBallsP2", {}, 72), ("p2_cur32", cur[31]["env_name"], cur[31]["config"], 48),
                 ("p2_rsi", "CustomMyoBaodingBallsP2", dict(enable_rsi=True, rsi_probability=1.0, balls_overlap=False), 48),
                 ("p1_cur02", cur[1]["env_name"], cur[1]["config"], 48),
                 ("p2_drop", "CustomMyoBaodingBallsP2", dict(drop_th=1.436, proximity_th=0.03), 48),
                 ("finger_random", "CustomMyoFingerPoseRandom", {}, 48), ("elbow_random", "CustomMyoElbowPoseRandom", {}, 32),
                 ("hand_random", "CustomMyoHandPoseRandom", {}, 32),
                 ("die_p2", "CustomMyoReorientP2", {}, 64),
                 ("die_drop", "CustomMyoReorientP2", dict(drop_th=0.03, pos_th=0.05, rot_th=3.0,
                                                          weighted_reward_keys=dict(pos_dist=1.0, rot_dist=0.2, pos_dist_diff=100.0, rot_dist_diff=10.0,
                                                                                    alive=1.0, act_reg=0.5, solved=2.0, done=-3.0, sparse=0.1)), 48)]
    for tag, name, cfg, n in step_sets:
        put("step", tag, name, cfg, step_cases(name, cfg, n, 900 + len(meta["step"])))
        print("step", tag, flush=True)
    out = shrink(out, meta)
    out["meta"] = np.array(json.dumps(meta))
    path = os.path.join(HERE, "env_fixtures.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
