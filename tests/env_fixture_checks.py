"""Kernel vs the fixtures recorded from the reference's OWN env code (tests/golden/make_env_fixtures.py: the unmodified
/root/reference/src/envs/{baoding,pose}.py driven over the oracle through tests/shim). Run twice: through the single-lane host
build of the kernel sources (CPU, tests/test_env_fixtures_emul.py) and through the CUDA library (tests/test_gpu_env_fixtures.py).

* step cases   : same pre-step state + env attributes + action -> observation, every reward term, the dense reward and the
                 post-step state must reproduce the reference's; done / solved flags bit-exact.
* reset samples: what ``reset()`` decides is random (three unseedable host RNGs in the reference, SURVEY.md 7), so the device
                 reset is compared in distribution (two-sample KS per continuous knob, frequencies of the discrete ones) and
                 through the deterministic relations the reference's code implies (angle pairs, RSI ball placement, post-RSI
                 activations, finger-noise groups).
"""
import json
import os

import numpy as np
import torch
from scipy import stats as sps

from conftest import GOLDEN
from myochallenge_b200 import _capi, sim
from myochallenge_b200.assets import asset_path
from myochallenge_b200.envs import FACTORY_NAMES, REGISTRY, make_task_cfg

_FX = None


def fixtures():
    global _FX
    if _FX is None:
        f = np.load(os.path.join(GOLDEN, "env_fixtures.npz"))
        _FX = (f, json.loads(str(f["meta"])))
    return _FX


def _get(group, tag):
    f, meta = fixtures()
    pre = f"{group}/{tag}/"
    d = {k[len(pre):]: f[k] for k in f.files if k.startswith(pre)}
    if "obs_cols" in d:          # reset observations are stored in the columns the checks read; any other column reads as NaN
        cols = d.pop("obs_cols")
        obs = np.full((len(d["obs"]), int(cols.max()) + 1), np.nan)
        obs[:, cols] = d["obs"]
        d["obs"] = obs
    return d, meta[group][tag]


def _make(lib, device, meta, n, seed=0, **extra):
    env_id = FACTORY_NAMES[meta["env_name"]]
    model = sim.Model(asset_path(REGISTRY[env_id]["model"]), lib=lib)
    kw = dict(meta["config"])
    kw.update(extra)
    cfg = make_task_cfg(model, env_id, **kw)
    return model, cfg, sim.BatchSim(model, n, cfg, device=device, seed=seed)


def _quat2mat(q):
    w, x, y, z = [q[:, i] for i in range(4)]
    R = np.stack([w*w + x*x - y*y - z*z, 2*(x*y - w*z), 2*(x*z + w*y), 2*(x*y + w*z), w*w - x*x + y*y - z*z, 2*(y*z - w*x),
                  2*(x*z - w*y), 2*(y*z + w*x), w*w - x*x - y*y + z*z], 1)
    return R / (w*w + x*x + y*y + z*z)[:, None]


def _rel(got, ref, floor):
    return float(np.abs(np.asarray(got, float) - np.asarray(ref, float)).max() / max(float(np.abs(ref).max()), floor))


# ---------------------------------------------------------------------------------------------------------------- step cases
def check_step_cases(lib, device, tag, obs_tol=2e-4):
    d, meta = _get("step", tag)
    n = len(d["done"])
    model, cfg, B = _make(lib, device, meta, n, auto_reset=0, max_episode_steps=100000)
    baoding = "pre_task" in d
    reorient = "pre_goal_quat" in d
    B.reset()
    B.set_state(d["pre_qpos"], d["pre_qvel"], d["pre_act"])
    if baoding:
        for k in range(2):
            B.set_param(_capi.PARAM_BODY_MASS, cfg.ball_body[k], d["pre_mass"][:, k: k + 1])
            B.set_param(_capi.PARAM_GEOM_SIZE, cfg.ball_geom[k], np.repeat(d["pre_size"][:, k: k + 1], 3, 1))
            B.set_param(_capi.PARAM_GEOM_FRICTION, cfg.ball_geom[k], d["pre_fric"][:, k])
            z = model.array("site_pos")[cfg.target_site[k], 2]
            B.set_param(_capi.PARAM_SITE_POS, cfg.target_site[k], np.concatenate([d["pre_target_xy"][:, 2 * k: 2 * k + 2], np.full((n, 1), z)], 1))
        ti = np.zeros((n, _capi.TASK_STATE_I), np.int32)
        ti[:, 0] = d["pre_counter"]; ti[:, 1] = 1; ti[:, 2] = d["pre_task"]
        tf = np.zeros((n, _capi.TASK_STATE_F), np.float32)
        tf[:, 0], tf[:, 1], tf[:, 2], tf[:, 3] = d["pre_angle1"], d["pre_angle2"], d["pre_xr"], d["pre_yr"]
        tf[:, 4] = np.where(np.isfinite(d["pre_period"]), np.minimum(d["pre_period"], 1e30), 5.0)
        B.set_task_state(ti, tf)
    elif reorient:
        B.set_param(_capi.PARAM_BODY_POS, cfg.goal_body, d["pre_goal_pos"])
        B.set_param(_capi.PARAM_BODY_MAT, cfg.goal_body, _quat2mat(d["pre_goal_quat"].astype(np.float64)))
        for k in range(cfg.object_ngeom):
            B.set_param(_capi.PARAM_GEOM_SIZE, cfg.object_geom0 + k, d["pre_die_size"][:, k])
            B.set_param(_capi.PARAM_GEOM_FRICTION, cfg.object_geom0 + k, d["pre_die_fric"][:, k])
        tf = np.zeros((n, _capi.TASK_STATE_F), np.float32)
        tf[:, 5], tf[:, 6] = d["pre_pos_dist"], d["pre_rot_dist"]
        B.set_task_state(tf=tf)
    else:
        B.set_task_state(pose_target=d["pre_target"])
    obs, rew, done, trunc = [t.cpu().numpy().copy() for t in B.step(torch.as_tensor(d["action"], dtype=torch.float32).to(device))]
    info = B.info.cpu().numpy()
    q, v, a, _ = [t.cpu().numpy() for t in B.get_state()]
    assert not trunc.any()
    worst = 0.0
    for w in range(n):
        e = _rel(obs[w], d["obs"][w], 1e-2)
        worst = max(worst, e)
        assert e < obs_tol, f"{tag} case {w}: observation differs from the reference's by {e:.2e}"
        cont = [0, 1, 2, 4] if baoding else ([0, 1, 2, 4, 8, 9] if reorient else [0, 3, 4])      # the continuous reward terms
        np.testing.assert_allclose(info[w, cont], d["terms"][w, cont], rtol=2e-4, atol=3e-5 if reorient else 2e-5, err_msg=f"{tag} case {w}: reward terms")
        assert bool(done[w]) == bool(d["done"][w]), f"{tag} case {w}: done flag"
        assert float(info[w, 6]) == float(d["terms"][w, 6])
        # flags that hinge on a threshold are compared where the reference's margin exceeds fp32 resolution of the distance
        if baoding:
            d1, d2 = -d["terms"][w, 0], -d["terms"][w, 1]
            z1, z2 = d["obs"][w, 25], d["obs"][w, 31]
            clear = min(abs(d1 - cfg.proximity_th), abs(d2 - cfg.proximity_th), abs(z1 - cfg.drop_th), abs(z2 - cfg.drop_th)) > 2e-5
        elif reorient:
            pd, rd = -d["terms"][w, 0], -d["terms"][w, 1]
            clear = min(abs(pd - cfg.pos_th), abs(pd - cfg.drop_th)) > 2e-5 and abs(rd - cfg.rot_th) > 2e-4
        else:
            dist = -d["terms"][w, 0]
            clear = min(abs(dist - cfg.pose_thd), abs(dist - 1.5 * cfg.pose_thd)) > 2e-5
        if clear:
            assert float(info[w, 5]) == float(d["terms"][w, 5]), f"{tag} case {w}: solved flag"
            assert float(info[w, 1 if not (baoding or reorient) else 3]) == float(d["terms"][w, 1 if not (baoding or reorient) else 3]), f"{tag} case {w}: alive / bonus term"
            assert abs(rew[w] - d["reward"][w]) <= 2e-4 * max(1.0, abs(d["reward"][w])), f"{tag} case {w}: dense reward {rew[w]} vs {d['reward'][w]}"
        assert _rel(q[w], d["post_qpos"][w], 0.1) < obs_tol and _rel(a[w], d["post_act"][w], 0.1) < obs_tol
        assert _rel(v[w], d["post_qvel"][w], 1.0) < 2e-3
    if baoding:
        ti2, _, _ = B.get_task_state()
        np.testing.assert_array_equal(ti2.cpu().numpy()[:, 0], d["post_counter"])       # self.counter after the step
    if reorient:      # step(): self.pos_dist / self.rot_dist <- this step's distances
        tf2 = B.get_task_state()[1].cpu().numpy()
        np.testing.assert_allclose(tf2[:, 5], -d["terms"][:, 0], rtol=2e-4, atol=3e-5)
        np.testing.assert_allclose(tf2[:, 6], -d["terms"][:, 1], rtol=2e-4, atol=3e-5)
    assert B.status() & ~1 == 0
    return worst


# ------------------------------------------------------------------------------------------------------------ reset samples
def _ks(name, got, ref, alpha=1e-5, ctol=2e-6):      # ~1000 comparisons against fixed reference samples: a real mismatch gives p << 1e-10
    got, ref = np.asarray(got, float).reshape(-1), np.asarray(ref, float).reshape(-1)
    if np.ptp(ref) < 1e-6:       # the reference never varies this knob (up to rounding noise): neither may the device
        assert np.abs(got - ref[0]).max() <= ctol * max(1.0, abs(ref[0])), f"{name}: constant {ref[0]} in the reference, device spread {np.ptp(got)}"
        return
    p = sps.ks_2samp(got, ref).pvalue
    assert p > alpha, f"{name}: distributions differ (KS p = {p:.2e}; device mean {got.mean():.5g} std {got.std():.3g}, reference mean {ref.mean():.5g} std {ref.std():.3g})"


def _freq(name, got, ref, values):
    for val in values:
        pg, pr = float(np.mean(got == val)), float(np.mean(ref == val))
        sd = np.sqrt(max(pr * (1 - pr), 1e-4) * (1.0 / len(got) + 1.0 / len(ref)))
        assert abs(pg - pr) < 4.5 * sd + 1e-9, f"{name}: P({val}) device {pg:.3f} vs reference {pr:.3f}"


def _wrap(x):
    return np.mod(np.asarray(x, float) + np.pi, 2 * np.pi) - np.pi


def check_reset_distribution(lib, device, tag, n=1536, seed=11):
    d, meta = _get("reset", tag)
    model, cfg, B = _make(lib, device, meta, n, seed=seed)
    obs = B.reset().cpu().numpy().copy()
    q, v, a, _ = [t.cpu().numpy() for t in B.get_state()]
    assert np.all(v == 0) and np.all(d["qvel"] == 0)
    if "goal_quat" in d:         # die reorientation: goal pose, die friction and size
        gp = B.get_param(_capi.PARAM_BODY_POS, cfg.goal_body).cpu().numpy()
        R = B.get_param(_capi.PARAM_BODY_MAT, cfg.goal_body).cpu().numpy().astype(np.float64)
        Rr = _quat2mat(d["goal_quat"].astype(np.float64))
        for e in range(3):
            _ks(f"{tag}: goal body_pos[{e}]", gp[:, e], d["goal_pos"][:, e])
        for e in range(9):       # the rotation matrix of body_quat, entry by entry (euler2quat of three uniform angles)
            _ks(f"{tag}: goal rotation[{e}]", R[:, e], Rr[:, e])
        np.testing.assert_allclose(np.einsum("nij,nkj->nik", R.reshape(-1, 3, 3), R.reshape(-1, 3, 3)), np.tile(np.eye(3), (n, 1, 1)), atol=1e-5)
        sizes = np.stack([B.get_param(_capi.PARAM_GEOM_SIZE, cfg.object_geom0 + k).cpu().numpy() for k in range(cfg.object_ngeom)], 1)
        fric = np.stack([B.get_param(_capi.PARAM_GEOM_FRICTION, cfg.object_geom0 + k).cpu().numpy() for k in range(cfg.object_ngeom)], 1)
        nominal = model.array("geom_size")[cfg.object_geom0: cfg.object_geom0 + cfg.object_ngeom]
        for arr, name in ((sizes, "device"), (d["die_size"], "reference")):      # ONE offset per reset, added to every half size of the three slabs
            delta = arr - nominal[None]
            assert np.abs(delta - delta[:, :1, :1]).max() < 1e-6, f"{tag}: {name} die sizes do not share one offset"
        _ks(f"{tag}: die size offset", sizes[:, 0, 0] - nominal[0, 0], d["die_size"][:, 0, 0] - nominal[0, 0])
        for k in range(cfg.object_ngeom):
            for e in range(3):
                _ks(f"{tag}: die geom {k} friction[{e}]", fric[:, k, e], d["die_fric"][:, k, e])
        for j in range(B.nq):
            _ks(f"{tag}: reset qpos[{j}]", q[:, j], d["qpos"][:, j])
        assert np.all(a == 0) and np.all(d["act"] == 0)
        tf = B.get_task_state()[1].cpu().numpy()
        o0 = (B.nq - 7) + (B.nv - 6)
        np.testing.assert_allclose(tf[:, 5], np.linalg.norm(obs[:, o0 + 6: o0 + 9], axis=1), rtol=1e-5, atol=1e-7)      # self.pos_dist from the reset obs
        np.testing.assert_allclose(tf[:, 6], np.linalg.norm(obs[:, o0 + 15: o0 + 18], axis=1), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(d["pos_dist"], np.linalg.norm(d["obs"][:, o0 + 6: o0 + 9], axis=1), rtol=1e-5, atol=1e-7)
        _ks(f"{tag}: pos_dist after reset", tf[:, 5], d["pos_dist"])
        if meta["config"].get("goal_rot_z") is None:       # (an angle pinned at 0 / +-pi makes rot_dist jump by 2 pi on rounding noise)
            _ks(f"{tag}: rot_dist after reset", tf[:, 6], d["rot_dist"])
        for e in range(9):
            _ks(f"{tag}: reset obs[{o0 + e}]", obs[:, o0 + e], d["obs"][:, o0 + e])
        # Euler angles (mat2euler): an angle at +-pi flips sign with the last bit of the matrix entry in the reference too, so
        # the angles are compared on the circle; rot_err = goal_rot - obj_rot inherits the same 2 pi ambiguity
        for e in range(9, 18):
            _ks(f"{tag}: cos reset obs[{o0 + e}]", np.cos(obs[:, o0 + e]), np.cos(d["obs"][:, o0 + e]), ctol=5e-5)
            _ks(f"{tag}: |sin| reset obs[{o0 + e}]", np.abs(np.sin(obs[:, o0 + e])), np.abs(np.sin(d["obs"][:, o0 + e])), ctol=5e-5)
        return
    if "task" not in d:          # pose envs: target + start pose
        _, _, tgt = B.get_task_state()
        tgt = tgt.cpu().numpy()
        for j in range(B.nq):
            _ks(f"{tag}: target_jnt_value[{j}]", tgt[:, j], d["target"][:, j])
            _ks(f"{tag}: reset qpos[{j}]", q[:, j], d["qpos"][:, j])
        np.testing.assert_allclose(obs[:, : B.nq], q, atol=1e-6)
        np.testing.assert_allclose(obs[:, B.nq + B.nv: 2 * B.nq + B.nv], tgt - q, atol=1e-5)          # pose_err
        if cfg.reset_type == 3:      # "sds": the start pose is tied to the target, sample by sample (pose.py:88-95)
            init = np.array([cfg_init for cfg_init in d["qpos"][0] * 0]) if False else None
            for got_q, got_t in ((q, tgt), (d["qpos"].astype(np.float64), d["target"].astype(np.float64))):
                # qpos = (1 - s) target + s init  =>  (qpos - (1 - s) target) / s is the same init_qpos in every sample
                if cfg.sds_distance > 0:
                    est = (got_q - (1 - cfg.sds_distance) * got_t) / cfg.sds_distance
                    assert np.abs(est - est[0]).max() < 1e-4
                else:
                    np.testing.assert_allclose(got_q, got_t, atol=1e-6)
        if "weight_mass" in d:       # CustomPoseEnv.reset: a new weight per reset and the geom size tied to it (pose.py:55-66)
            wm = B.get_param(_capi.PARAM_BODY_MASS, cfg.weight_body).cpu().numpy()[:, 0]
            ws = B.get_param(_capi.PARAM_GEOM_SIZE, cfg.weight_geom).cpu().numpy()[:, 0]
            _ks(f"{tag}: weight", wm, d["weight_mass"])
            np.testing.assert_allclose(ws, 0.01 + 2.5 * wm / 100, rtol=1e-6)
            np.testing.assert_allclose(d["weight_size0"], 0.01 + 2.5 * d["weight_mass"] / 100, rtol=1e-6)
        assert np.all(a == 0) and np.all(d["act"] == 0)
        return
    ti, tf, _ = B.get_task_state()
    ti, tf = ti.cpu().numpy(), tf.cpu().numpy()
    task, counter = ti[:, 2], ti[:, 0] + (ti[:, 3] & 1)
    _freq(f"{tag}: which_task", task, d["task"], (0, 1, 2))
    _freq(f"{tag}: counter after reset (1 = the RSI branch ran its in-reset step)", counter, d["counter"], (0, 1))
    # start angles: compared on the circle; the pair relation is deterministic in every branch of the reference's reset
    if "instance" in d:
        # decided once per env object (in _setup) and never redrawn by reset(): constant per object in the reference, constant
        # per world on the device (three more episodes), and the same two values with matching frequencies across objects
        for k in np.unique(d["instance"]):
            assert np.ptp(d["angle1"][d["instance"] == k]) == 0
        first = np.array([d["angle1"][d["instance"] == k][0] for k in np.unique(d["instance"])])
        for _ in range(3):
            B.reset()
            np.testing.assert_array_equal(B.get_task_state()[1].cpu().numpy()[:, 0], tf[:, 0])
        assert set(np.round(np.unique(tf[:, 0]), 5)) == set(np.round(np.unique(first), 5))
        _freq(f"{tag}: start angle per env object", np.round(tf[:, 0], 4), np.round(first, 4), np.round(np.unique(first), 4))
    else:
        _ks(f"{tag}: ball_1_starting_angle", _wrap(tf[:, 0]), _wrap(d["angle1"]))
    rel_g, rel_r = np.round(_wrap(tf[:, 1] - tf[:, 0]), 4), np.round(_wrap(d["angle2"] - d["angle1"]), 4)
    assert set(np.unique(np.abs(rel_g))) <= set(np.unique(np.abs(rel_r))), f"{tag}: angle2 - angle1 takes values {np.unique(rel_g)} (reference {np.unique(rel_r)})"
    for name, col in (("x_radius", 2), ("y_radius", 3), ("time_period", 4)):
        ref = d[{2: "xr", 3: "yr", 4: "period"}[col]]
        _ks(f"{tag}: {name}", tf[:, col], np.minimum(ref, 1e30))
    for k in range(2):
        _ks(f"{tag}: ball{k + 1} mass", B.get_param(_capi.PARAM_BODY_MASS, cfg.ball_body[k]).cpu().numpy()[:, 0], d["mass"][:, k])
        sz = B.get_param(_capi.PARAM_GEOM_SIZE, cfg.ball_geom[k]).cpu().numpy()
        _ks(f"{tag}: ball{k + 1} size", sz[:, 0], d["size"][:, k])
        fr = B.get_param(_capi.PARAM_GEOM_FRICTION, cfg.ball_geom[k]).cpu().numpy()
        for e in range(3):
            _ks(f"{tag}: ball{k + 1} friction[{e}]", fr[:, e], d["fric"][:, k, e])
    # hand pose after reset (noise knobs): per joint
    for j in range(B.nq - 14):
        _ks(f"{tag}: reset qpos[{j}]", q[:, j], d["qpos"][:, j])
    for grp in ((4, 5, 6), (7, 9, 10, 11, 13, 14, 15, 17, 18, 19, 21, 22)):        # one draw per group in the reference (:469-491)
        if np.ptp(d["qpos"][:, grp[0]]) > 0:
            assert np.allclose(q[:, grp], q[:, [grp[0]]]) and np.allclose(d["qpos"][:, grp], d["qpos"][:, [grp[0]]])
    # balls: z is never touched by a reset; xy either the model's or (RSI) the targets' world xy as the in-reset step left them
    bq = [cfg.ball_qposadr[0], cfg.ball_qposadr[1]]
    rsi_g, rsi_r = counter == 1, d["counter"] == 1
    for k in range(2):
        _ks(f"{tag}: ball{k + 1} z", q[:, bq[k] + 2], d["qpos"][:, bq[k] + 2])
        for e in range(2):
            _ks(f"{tag}: ball{k + 1} xy[{e}] (no RSI)", q[~rsi_g, bq[k] + e], d["qpos"][~rsi_r, bq[k] + e]) if (~rsi_r).sum() > 8 and (~rsi_g).sum() > 8 else None
    if rsi_r.sum() > 8 and rsi_g.sum() > 8:
        # observation: object xy - target xy right after an RSI reset. The reference places the balls on the targets' world xy
        # as observed AFTER its in-reset env.step and then restores the hand pose, so the targets (they ride on the palm) end up
        # a fraction of a millimetre away from the balls: the same offsets must come out of the device reset
        # (rotation tasks: a hold world's targets stay where that env's previous episode left them, :a7)
        rot_g, rot_r = rsi_g & (task > 0), rsi_r & (d["task"] > 0)
        for k, (o, t) in enumerate(((23, 35), (29, 38))):
            eg, er = obs[rot_g][:, o: o + 2] - obs[rot_g][:, t: t + 2], d["obs"][rot_r][:, o: o + 2] - d["obs"][rot_r][:, t: t + 2]
            if not cfg.p1_reset or (cfg.noise_balls == 0 and cfg.noise_palm == 0):
                assert np.abs(er).max() < 2e-3 and np.abs(eg).max() < 2e-3
                for e in range(2):
                    _ks(f"{tag}: RSI ball{k + 1} - target{k + 1} offset [{e}]", eg[:, e], er[:, e])
        # muscle activations after the in-reset zero-action step: the same vector in every RSI world
        ref_act = d["act"][rsi_r]
        assert np.abs(ref_act - ref_act[0]).max() < 1e-6
        np.testing.assert_allclose(a[rsi_g], np.tile(ref_act[0], (int(rsi_g.sum()), 1)), rtol=2e-5, atol=1e-7)
    assert np.all(a[~rsi_g] == 0) and np.all(d["act"][~rsi_r] == 0)
    # target sites (body frame): rotation-task worlds whose RSI step moved them sit on the goal ellipse of THIS reset's radii
    cx, cy = cfg.center_pos[0], cfg.center_pos[1]
    for k in range(2):
        sp = B.get_param(_capi.PARAM_SITE_POS, cfg.target_site[k]).cpu().numpy()
        moved_g, moved_r = rsi_g & (task > 0), rsi_r & (d["task"] > 0)
        if moved_g.sum() and moved_r.sum():
            eg = ((sp[moved_g, 0] - cx) / tf[moved_g, 2]) ** 2 + ((sp[moved_g, 1] - cy) / tf[moved_g, 3]) ** 2
            er = ((d["target_xy"][moved_r, 2 * k] - cx) / d["xr"][moved_r]) ** 2 + ((d["target_xy"][moved_r, 2 * k + 1] - cy) / d["yr"][moved_r]) ** 2
            np.testing.assert_allclose(er, 1.0, atol=1e-4)
            np.testing.assert_allclose(eg, 1.0, atol=1e-4)
    # the observation is assembled from the same state: hand_pos, velocities (zero), errors = target - object
    np.testing.assert_allclose(obs[:, : B.nq - 14], q[:, : B.nq - 14], atol=1e-6)
    np.testing.assert_allclose(obs[:, 41:44], obs[:, 35:38] - obs[:, 23:26], atol=1e-6)
    assert np.all(obs[:, 26:29] == 0) and np.all(obs[:, 32:35] == 0)
