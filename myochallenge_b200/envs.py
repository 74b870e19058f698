"""Environment registry and factory: the gym registrations of /root/reference/src/envs/__init__.py and the
name dispatch of /root/reference/src/envs/environment_factory.py:8-63, producing batched ``MyoVecEnv`` objects
instead of one ``gym.Env`` per process.

``EnvironmentFactory.create(env_name, num_envs=..., **kwargs)`` accepts the same names and the same kwargs
the reference passes through ``gym.make(id, **kwargs)`` into ``CustomBaodingP2Env._setup``
(/root/reference/src/envs/baoding.py:300-401), ``CustomBaodingEnv._setup`` (:96-176) and
``CustomPoseEnv._setup`` (/root/reference/src/envs/pose.py:7-51); they are translated into the C-ABI task
configuration (``myo_task_cfg``) that the world kernel evaluates per world on the device.
"""
from __future__ import annotations

import math
from typing import Any, Dict

import numpy as np

from . import _capi
from .assets import asset_path
from .sim import Model
from .vec_env import BAODING_KEYS, OBS_KEYS, POSE_KEYS, REACH_KEYS, REORIENT_KEYS, MyoVecEnv

_JNT_HAND = ['pro_sup', 'deviation', 'flexion', 'cmc_abduction', 'cmc_flexion', 'mp_flexion', 'ip_flexion', 'mcp2_flexion',
             'mcp2_abduction', 'pm2_flexion', 'md2_flexion', 'mcp3_flexion', 'mcp3_abduction', 'pm3_flexion', 'md3_flexion',
             'mcp4_flexion', 'mcp4_abduction', 'pm4_flexion', 'md4_flexion', 'mcp5_flexion', 'mcp5_abduction', 'pm5_flexion',
             'md5_flexion']
# per-joint (min, max) over the ten ASL poses of /root/reference/src/envs/__init__.py:174-183,204-207
_ASL = np.array([
    [0, 0, 0, 0.5624, 0.28272, -0.75573, -1.309, 1.30045, -0.006982, 1.45492, 0.998897, 1.26466, 0, 1.40604, 0.227795, 1.07614, -0.020944, 1.46103, 0.06284, 0.83263, -0.14399, 1.571, 1.38248],
    [0, 0, 0, 0.0248, 0.04536, -0.7854, -1.309, 0.366605, 0.010473, 0.269258, 0.111722, 1.48459, 0, 1.45318, 1.44532, 1.44532, -0.204204, 1.46103, 1.44532, 1.48459, -0.2618, 1.47674, 1.48459],
    [0, 0, 0, 0.0248, 0.04536, -0.7854, -1.13447, 0.514973, 0.010473, 0.128305, 0.111722, 0.510575, 0, 0.37704, 0.117825, 1.44532, -0.204204, 1.46103, 1.44532, 1.48459, -0.2618, 1.47674, 1.48459],
    [0, 0, 0, 0.3384, 0.25305, 0.01569, -0.0262045, 0.645885, 0.010473, 0.128305, 0.111722, 0.510575, 0, 0.37704, 0.117825, 1.571, -0.036652, 1.52387, 1.45318, 1.40604, -0.068068, 1.39033, 1.571],
    [0, 0, 0, 0.6392, -0.147495, -0.7854, -1.309, 0.637158, 0.010473, 0.128305, 0.111722, 0.510575, 0, 0.37704, 0.117825, 0.306345, -0.010472, 0.400605, 0.133535, 0.21994, -0.068068, 0.274925, 0.01571],
    [0, 0, 0, 0.3384, 0.25305, 0.01569, -0.0262045, 0.645885, 0.010473, 0.128305, 0.111722, 0.510575, 0, 0.37704, 0.117825, 0.306345, -0.010472, 0.400605, 0.133535, 0.21994, -0.068068, 0.274925, 0.01571],
    [0, 0, 0, 0.6392, -0.147495, -0.7854, -1.309, 0.637158, 0.010473, 0.128305, 0.111722, 0.510575, 0, 0.37704, 0.117825, 0.306345, -0.010472, 0.400605, 0.133535, 1.1861, -0.2618, 1.35891, 1.48459],
    [0, 0, 0, 0.524, 0.01569, -0.7854, -1.309, 0.645885, -0.006982, 0.128305, 0.111722, 0.510575, 0, 0.37704, 0.117825, 1.28036, -0.115192, 1.52387, 1.45318, 0.432025, -0.068068, 0.18852, 0.149245],
    [0, 0, 0, 0.428, 0.22338, -0.7854, -1.309, 0.645885, -0.006982, 0.128305, 0.194636, 1.39033, 0, 1.08399, 0.573415, 0.667675, -0.020944, 0, 0.06284, 0.432025, -0.068068, 0.18852, 0.149245],
    [0, 0, 0, 0.5624, 0.28272, -0.75573, -1.309, 1.30045, -0.006982, 1.45492, 0.998897, 0.39275, 0, 0.18852, 0.227795, 0.667675, -0.020944, 0, 0.06284, 0.432025, -0.068068, 0.18852, 0.149245],
])

# id -> (task kind, model, horizon, default kwargs)   [REF src/envs/__init__.py:12-229]
REGISTRY: Dict[str, Dict[str, Any]] = {
    "CustomMyoChallengeBaodingP1-v1": dict(kind=_capi.TASK_BAODING, model="hand/myo_hand_baoding.mjb", horizon=200, phase=1,
                                           kwargs=dict(normalize_act=True, goal_xrange=(0.025, 0.025), goal_yrange=(0.028, 0.028))),
    "CustomMyoChallengeBaodingP2-v1": dict(kind=_capi.TASK_BAODING, model="hand/myo_hand_baoding.mjb", horizon=200, phase=2,
                                           kwargs=dict(normalize_act=True, goal_time_period=(4, 6), goal_xrange=(0.020, 0.030),
                                                       goal_yrange=(0.022, 0.032), obj_size_range=(0.018, 0.024),
                                                       obj_mass_range=(0.030, 0.300), obj_friction_change=(0.2, 0.001, 0.00002),
                                                       task_choice="random")),
    # die reorientation   [REF src/envs/__init__.py:26-55]
    "CustomMyoChallengeDieReorientP1-v0": dict(kind=_capi.TASK_REORIENT, model="hand/myo_hand_die.mjb", horizon=150,
                                               kwargs=dict(normalize_act=True, frame_skip=5, goal_pos=(-.010, .010), goal_rot=(-1.57, 1.57))),
    "CustomMyoChallengeDieReorientP2-v0": dict(kind=_capi.TASK_REORIENT, model="hand/myo_hand_die.mjb", horizon=150,
                                               kwargs=dict(normalize_act=True, frame_skip=5, goal_pos=(-.020, .020), goal_rot=(-3.14, 3.14),
                                                           obj_size_change=0.007, obj_friction_change=(0.2, 0.001, 0.00002))),
    "CustomMyoElbowPoseFixed-v0": dict(kind=_capi.TASK_POSE, model="arm/myo_elbow_1dof6muscles.mjb", horizon=100,
                                       kwargs=dict(target_jnt_range={"r_elbow_flex": (2, 2)}, normalize_act=True, pose_thd=.175, reset_type="random")),
    "CustomMyoElbowPoseRandom-v0": dict(kind=_capi.TASK_POSE, model="arm/myo_elbow_1dof6muscles.mjb", horizon=100,
                                        kwargs=dict(target_jnt_range={"r_elbow_flex": (0, 2.27)}, normalize_act=True, pose_thd=.175, reset_type="random")),
    "CustomMyoFingerPoseFixed-v0": dict(kind=_capi.TASK_POSE, model="finger/myo_finger_v0.mjb", horizon=100,
                                        kwargs=dict(target_jnt_range={"IFadb": (0, 0), "IFmcp": (0, 0), "IFpip": (.75, .75), "IFdip": (.75, .75)},
                                                    normalize_act=True)),
    "CustomMyoFingerPoseRandom-v0": dict(kind=_capi.TASK_POSE, model="finger/myo_finger_v0.mjb", horizon=100,
                                         kwargs=dict(target_jnt_range={"IFadb": (-.2, .2), "IFmcp": (-.4, 1), "IFpip": (.1, 1), "IFdip": (.1, 1)},
                                                     normalize_act=True)),
    "CustomMyoHandPoseFixed-v0": dict(kind=_capi.TASK_POSE, model="hand/myo_hand_pose.mjb", horizon=100,
                                      kwargs=dict(target_jnt_value=np.array([0, 0, 0, -0.0904, 0.0824475, -0.681555, -0.514888, 0, -0.013964, -0.0458132, 0,
                                                                             0.67553, -0.020944, 0.76979, 0.65982, 0, 0, 0, 0, 0.479155, -0.099484, 0.95831, 0]),
                                                  normalize_act=True, pose_thd=.7, reset_type="init", target_type="fixed")),
    "CustomMyoHandPoseRandom-v0": dict(kind=_capi.TASK_POSE, model="hand/myo_hand_pose.mjb", horizon=100,
                                       kwargs=dict(target_jnt_range={n: (float(_ASL[:, i].min()), float(_ASL[:, i].max())) for i, n in enumerate(_JNT_HAND)},
                                                   normalize_act=True, pose_thd=.8, reset_type="random", target_type="generate")),
}
for _k in range(10):
    REGISTRY[f"CustomMyoHandPose{_k}Fixed-v0"] = dict(kind=_capi.TASK_POSE, model="hand/myo_hand_pose.mjb", horizon=100,
                                                      kwargs=dict(target_jnt_value=_ASL[_k].copy(), normalize_act=True, pose_thd=.7,
                                                                  reset_type="init", target_type="fixed"))
# stock MyoSuite ids the factory also exposes (same models and defaults as MyoSuite 1.2.3 registers them)
REGISTRY["myoFingerPoseRandom-v0"] = REGISTRY["CustomMyoFingerPoseRandom-v0"]
REGISTRY["myoFingerPoseFixed-v0"] = REGISTRY["CustomMyoFingerPoseFixed-v0"]
REGISTRY["myoChallengeBaodingP2-v1"] = REGISTRY["CustomMyoChallengeBaodingP2-v1"]
REGISTRY["myoChallengeBaodingP1-v1"] = REGISTRY["CustomMyoChallengeBaodingP1-v1"]
REGISTRY["myoHandPoseRandom-v0"] = REGISTRY["CustomMyoHandPoseRandom-v0"]
REGISTRY["myoElbowPose1D6MRandom-v0"] = REGISTRY["CustomMyoElbowPoseRandom-v0"]
# MyoSuite 1.2.3 envs/myo/__init__.py finger reach registrations (ReachEnvV0), as best recalled [3P-MEM]. The Random range has
# one check: at the model's qpos0 the oracle puts IFtip at (0.270, 0.000, 0.300), that range's upper corner. The frame skip and
# the horizon have no such check.
REGISTRY["myoFingerReachFixed-v0"] = dict(kind=_capi.TASK_REACH, model="finger/myo_finger_v0.mjb", horizon=200,
                                          kwargs=dict(target_reach_range={"IFtip": ((0.2, 0.05, 0.20), (0.2, 0.05, 0.20))},
                                                      normalize_act=True, frame_skip=5))
REGISTRY["myoFingerReachRandom-v0"] = dict(kind=_capi.TASK_REACH, model="finger/myo_finger_v0.mjb", horizon=200,
                                           kwargs=dict(target_reach_range={"IFtip": ((.1, -.1, .1), (.27, .1, .3))},
                                                       normalize_act=True, frame_skip=5))

# EnvironmentFactory names -> gym ids   [REF src/envs/environment_factory.py:22-61]
FACTORY_NAMES = {
    "MyoFingerPoseFixed": "myoFingerPoseFixed-v0", "MyoFingerPoseRandom": "myoFingerPoseRandom-v0",
    "MyoBaodingBallsP1": "myoChallengeBaodingP1-v1", "CustomMyoBaodingBallsP1": "CustomMyoChallengeBaodingP1-v1",
    "MyoBaodingBallsP2": "myoChallengeBaodingP2-v1", "CustomMyoBaodingBallsP2": "CustomMyoChallengeBaodingP2-v1",
    "CustomMyoElbowPoseFixed": "CustomMyoElbowPoseFixed-v0", "CustomMyoElbowPoseRandom": "CustomMyoElbowPoseRandom-v0",
    "CustomMyoFingerPoseFixed": "CustomMyoFingerPoseFixed-v0", "CustomMyoFingerPoseRandom": "CustomMyoFingerPoseRandom-v0",
    "CustomMyoHandPoseFixed": "CustomMyoHandPoseFixed-v0", "CustomMyoHandPoseRandom": "CustomMyoHandPoseRandom-v0",
    "CustomMyoReorientP1": "CustomMyoChallengeDieReorientP1-v0", "CustomMyoReorientP2": "CustomMyoChallengeDieReorientP2-v0",
    "MyoFingerReachFixed": "myoFingerReachFixed-v0", "MyoFingerReachRandom": "myoFingerReachRandom-v0",
}
# names the reference factory knows whose models / task kernels are outside this build (pen, key-turn, mixture)
UNSUPPORTED = {"MyoHandKeyTurnFixed", "MyoHandKeyTurnRandom", "MixtureModelBaodingEnv", "CustomMyoPenTwirlRandom"}


def reach_far_steps(timestep: float, frame_skip: int) -> int:
    """First env step count after which ReachEnvV0 applies far_th (``data.time > 2 dt``): MuJoCo adds ``timestep`` to ``time``
    in fp64 once per substep, so the sum is replayed here (the kernel keeps time in fp32 and compares step counts instead)."""
    dt, t, k = timestep * frame_skip, 0.0, 0
    while not t > 2 * dt:
        for _ in range(frame_skip):
            t += timestep
        k += 1
    return k


def _weights(cfg, keys, weighted_reward_keys):
    for i in range(_capi.MYO_INFO_TERMS):
        cfg.rwd_weight[i] = 0.0
    for k, w in weighted_reward_keys.items():
        if k not in keys:
            raise ValueError(f"unknown reward key {k!r} (known: {keys})")
        cfg.rwd_weight[keys.index(k)] = float(w)


def _obs_keys(cfg, model, obs_keys) -> None:
    """MujocoEnv._setup's ``obs_keys``: the observation concatenates these obs-dict entries in order (duplicates allowed), and
    BaseV0._setup appends "act" when the model has activations and the list lacks it."""
    known = OBS_KEYS[cfg.kind]
    if isinstance(obs_keys, str):
        raise ValueError(f"obs_keys: a list of keys, got the string {obs_keys!r} (known: {list(known)})")
    keys = list(obs_keys)
    if not keys:
        raise ValueError(f"obs_keys: empty list (known: {list(known)})")
    unknown = [k for k in keys if k not in known]
    if unknown:
        raise ValueError(f"obs_keys: unknown key(s) {unknown} (known: {list(known)})")
    if model.size("na") > 0 and "act" not in keys:
        keys.append("act")
    if len(keys) > _capi.MYO_MAX_OBS_KEYS:
        raise ValueError(f"obs_keys: at most {_capi.MYO_MAX_OBS_KEYS} keys (\"act\" included), got {len(keys)}")
    cfg.n_obs_keys = len(keys)
    for i, k in enumerate(keys):
        cfg.obs_keys[i] = known.index(k)


def make_task_cfg(model: Model, env_id: str, **overrides) -> _capi.TaskCfg:
    """Translate a registration + kwargs into the C-ABI task configuration."""
    if env_id not in REGISTRY:
        raise ValueError("Environment name not recognized:", env_id)
    reg = REGISTRY[env_id]
    kw = dict(reg["kwargs"])
    kw.update(overrides)
    cfg = model.default_task_cfg(reg["kind"])
    cfg.max_episode_steps = int(kw.pop("max_episode_steps", reg["horizon"]))
    cfg.frame_skip = int(kw.pop("frame_skip", 5 if reg["kind"] == _capi.TASK_REORIENT else 10))
    cfg.normalize_act = int(bool(kw.pop("normalize_act", True)))
    cfg.auto_reset = int(bool(kw.pop("auto_reset", True)))
    cfg.clip_actions = int(bool(kw.pop("clip_actions", False)))
    if reg["kind"] == _capi.TASK_BAODING:
        if "weighted_reward_keys" in kw:
            _weights(cfg, BAODING_KEYS, kw.pop("weighted_reward_keys"))
        cfg.drop_th = float(kw.pop("drop_th", 1.25))
        cfg.proximity_th = float(kw.pop("proximity_th", 0.015))
        for name, default in (("goal_time_period", (5, 5)), ("goal_xrange", (0.025, 0.025)), ("goal_yrange", (0.028, 0.028)),
                              ("obj_size_range", (0.018, 0.024)), ("obj_mass_range", (0.030, 0.300))):
            lo, hi = kw.pop(name, default)
            # the curriculum's first step holds the targets still with goal_time_period = 1e100: keep it finite in fp32
            getattr(cfg, name)[0], getattr(cfg, name)[1] = min(float(lo), 1e30), min(float(hi), 1e30)
        fc = kw.pop("obj_friction_change", (0.2, 0.001, 0.00002))
        for i in range(3):
            cfg.obj_friction_change[i] = float(fc[i])
        cfg.p1_reset = int(reg.get("phase", 2) == 1)
        if cfg.p1_reset:        # CustomBaodingEnv._setup: task=None | "cw" | "ccw" | "random" (sample_task, :285-296)
            task = kw.pop("task", None)
            if task not in (None, "cw", "ccw", "random"):
                raise ValueError("Unknown task for baoding: ", task)
            cfg.task_choice_random = int(task == "random")
            if task in ("cw", "ccw"):
                cfg.fixed_task = 1 if task == "cw" else 2
            cfg.noise_palm = float(kw.pop("noise_palm", 0.0))
            cfg.noise_balls = float(kw.pop("noise_balls", 0.0))
            for name, v in (("noise_palm", cfg.noise_palm), ("noise_fingers", float(kw.get("noise_fingers", 0.0)))):
                if not 0 <= v <= 1:
                    raise AssertionError(f"{name} must be between 0 and 1")
        else:
            task_choice = kw.pop("task_choice", "fixed")
            if task_choice not in ("fixed", "random"):
                raise ValueError(f"task_choice must be 'fixed' or 'random', got {task_choice!r}")
            cfg.task_choice_random = int(task_choice == "random")
        cfg.randomize_physics = int(reg.get("phase", 2) == 2)     # P1's reset keeps the nominal balls
        cfg.overlap_probability = float(kw.pop("overlap_probability", 0.0))
        cfg.balls_overlap = int(bool(kw.pop("balls_overlap", False)))    # read only inside the RSI branch (/root/reference/src/envs/baoding.py:634)
        lim = kw.pop("limit_init_angle", False)
        cfg.limit_init_angle = float(lim) if lim else 0.0
        cfg.noise_fingers = float(kw.pop("noise_fingers", 0.0))
        cfg.enable_rsi = int(bool(kw.pop("enable_rsi", False)))
        cfg.rsi_probability = float(kw.pop("rsi_probability", 1))
        for k in ("beta_init_angle", "beta_ball_size", "beta_ball_mass"):
            v = kw.pop(k, None)
            if v:
                if len(v) != 2 or min(v) <= 0:
                    raise ValueError(f"{k} must be the (a, b) > 0 of a beta distribution, got {v!r}")
                getattr(cfg, k)[0], getattr(cfg, k)[1] = float(v[0]), float(v[1])
    elif reg["kind"] == _capi.TASK_REORIENT:
        # CustomReorientEnv._setup (/root/reference/src/envs/reorient.py:58-125)
        if "weighted_reward_keys" in kw:
            _weights(cfg, REORIENT_KEYS, kw.pop("weighted_reward_keys"))
        for name, default in (("goal_pos", (0.0, 0.0)), ("goal_rot", (0.785, 0.785))):
            lo, hi = kw.pop(name, default)
            getattr(cfg, name)[0], getattr(cfg, name)[1] = float(lo), float(hi)
        cfg.obj_size_change = float(kw.pop("obj_size_change", 0.0))
        fc = kw.pop("obj_friction_change", (0, 0, 0))
        for i in range(3):
            cfg.obj_friction_change[i] = float(fc[i])
        cfg.pos_th, cfg.rot_th, cfg.drop_th = float(kw.pop("pos_th", 0.025)), float(kw.pop("rot_th", 0.262)), float(kw.pop("drop_th", 0.200))
        for ax, name in enumerate(("goal_rot_x", "goal_rot_y", "goal_rot_z")):
            ranges = kw.pop(name, None)
            if ranges is not None:
                if not 0 < len(ranges) <= _capi.MYO_MAX_ROT_RANGES:
                    raise ValueError(f"{name}: between 1 and {_capi.MYO_MAX_ROT_RANGES} (low, high) ranges")
                cfg.n_goal_rot[ax] = len(ranges)
                for k, (lo, hi) in enumerate(ranges):
                    cfg.goal_rot_axis[ax][k][0], cfg.goal_rot_axis[ax][k][1] = float(lo), float(hi)
        # enable_rsi / rsi_distance_*: the reference's RSI branch only rewrites body_pos / body_quat of the free-jointed die, which
        # MuJoCo's kinematics never reads (a free body's pose is its qpos), so these knobs change nothing there - nor here
        for k in ("enable_rsi", "rsi_distance_pos", "rsi_distance_rot"):
            kw.pop(k, None)
    elif reg["kind"] == _capi.TASK_REACH:
        # ReachEnvV0._setup(target_reach_range, far_th=.35, ...) [3P-MEM]: thresholds scale with the number of sites
        if "weighted_reward_keys" in kw:
            _weights(cfg, REACH_KEYS, kw.pop("weighted_reward_keys"))
        sites = dict(kw.pop("target_reach_range"))
        if not 0 < len(sites) <= _capi.MYO_MAX_OVERRIDE:
            raise ValueError(f"target_reach_range: between 1 and {_capi.MYO_MAX_OVERRIDE} sites (the targets use the per-world site overrides)")
        cfg.reach_nsite = len(sites)
        for k, (site, (lo, hi)) in enumerate(sites.items()):
            try:
                cfg.reach_tip_site[k], cfg.reach_target_site[k] = model.name2id("site", site), model.name2id("site", site + "_target")
            except KeyError:
                raise ValueError(f"target_reach_range: the model has no sites {site!r} and {site + '_target'!r}") from None
            lo, hi = np.asarray(lo, float).reshape(3), np.asarray(hi, float).reshape(3)
            for e in range(3):
                cfg.reach_range[k][0][e], cfg.reach_range[k][1][e] = lo[e], hi[e]
        cfg.far_th = float(kw.pop("far_th", 0.35)) * len(sites)
        cfg.reach_near_th = 0.0125 * len(sites)
        cfg.reach_far_steps = reach_far_steps(model.opt("timestep"), cfg.frame_skip)
    else:
        if "weighted_reward_keys" in kw:
            _weights(cfg, POSE_KEYS, kw.pop("weighted_reward_keys"))
        cfg.pose_thd = float(kw.pop("pose_thd", 0.35))
        cfg.target_distance = float(kw.pop("target_distance", 1.0))
        rt = kw.pop("reset_type", "init")
        if rt is None:
            rt = "none"
        if rt not in ("none", "init", "random", "sds"):
            raise ValueError(f"Reset Type not found: {rt!r}")
        cfg.reset_type = {"none": 0, "init": 1, "random": 2, "sds": 3}[rt]
        cfg.sds_distance = float(kw.pop("sds_distance", 0) or 0)
        tt = kw.pop("target_type", "generate")
        if tt not in ("generate", "fixed"):
            raise NotImplementedError(f"target_type {tt!r}")
        cfg.target_type = {"fixed": 0, "generate": 1}[tt]
        rng = kw.pop("target_jnt_range", None)
        val = kw.pop("target_jnt_value", None)
        if rng:
            if len(rng) > 64:
                raise ValueError("at most 64 target joints")
            cfg.n_target_jnt = len(rng)
            for i, (jn, (lo, hi)) in enumerate(rng.items()):
                cfg.target_jnt_ids[i] = model.name2id("joint", jn)
                cfg.target_jnt_range[i][0], cfg.target_jnt_range[i][1] = float(lo), float(hi)
        elif val is not None:
            cfg.n_target_jnt = 0
            for i, v in enumerate(np.asarray(val, float).reshape(-1)):
                cfg.target_jnt_value[i] = float(v)
        kw.pop("viz_site_targets", None)
        kw.pop("sds_distance", None)
        wb, wr = kw.pop("weight_bodyname", None), kw.pop("weight_range", None)
        if wb is not None:       # CustomPoseEnv.reset: body_mass[bid] ~ U(weight_range); geom_size[body_geomadr[bid]][0] follows (pose.py:55-66)
            if wr is None or len(wr) != 2:
                raise ValueError("weight_bodyname needs weight_range=(low, high)")
            bid = model.name2id("body", wb)
            gid = int(model.array("body_geomadr")[bid])
            cfg.weight_body, cfg.weight_geom = bid, gid
            cfg.weight_range[0], cfg.weight_range[1] = float(wr[0]), float(wr[1])
            cfg.n_ovr_body, cfg.ovr_body[0] = 1, bid
            if gid >= 0:
                cfg.n_ovr_geom, cfg.ovr_geom[0] = 1, gid
    kw.pop("model_path", None)
    obs_keys = kw.pop("obs_keys", None)
    if obs_keys is not None:
        _obs_keys(cfg, model, obs_keys)
    reward_mode = kw.pop("reward_mode", "dense")
    if reward_mode not in ("dense", "sparse"):
        raise ValueError(f"reward_mode must be 'dense' or 'sparse', got {reward_mode!r}")
    cfg.reward_sparse = int(reward_mode == "sparse")
    if kw:
        raise TypeError(f"unexpected env kwargs: {sorted(kw)}")
    return cfg


def make_vec_env(env_id: str, num_envs: int, device="cuda:0", seed: int = 0, **kwargs) -> MyoVecEnv:
    reg = REGISTRY.get(env_id)
    if reg is None:
        raise ValueError("Environment name not recognized:", env_id)
    model = Model(kwargs.pop("model_path", None) or asset_path(reg["model"]))
    cfg = make_task_cfg(model, env_id, **kwargs)
    return MyoVecEnv(model, cfg, num_envs, device=device, seed=seed)


class EnvironmentFactory:
    """Same static interface as the reference's factory; ``num_envs`` worlds instead of one env."""

    @staticmethod
    def create(env_name: str, num_envs: int = 1, device="cuda:0", seed: int = 0, **kwargs) -> MyoVecEnv:
        if env_name in UNSUPPORTED:
            raise NotImplementedError(f"{env_name}: the model / task kernel for this reference env is outside this build")
        if env_name not in FACTORY_NAMES:
            raise ValueError("Environment name not recognized:", env_name)
        return make_vec_env(FACTORY_NAMES[env_name], num_envs, device=device, seed=seed, **kwargs)
