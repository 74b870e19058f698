"""CPU: host logic of the env registry / factory (mirror of /root/reference/src/envs/__init__.py and
environment_factory.py), the VecNormalize arithmetic and the multi-rank moment merge (gloo, world_size 2)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import GOLDEN
from myochallenge_b200 import _capi
from myochallenge_b200.assets import asset_path
from myochallenge_b200.envs import FACTORY_NAMES, REGISTRY, EnvironmentFactory, make_task_cfg
from myochallenge_b200.sim import BatchSim, Model
from myochallenge_b200.vec_env import RunningMeanStd, VecNormalize, rank_seed

# trained_models/curriculum_steps_complete_baoding_winner/32_phase_2_smaller_rate_resume/config.json of the reference
STEP32 = {"weighted_reward_keys": {"pos_dist_1": 5, "pos_dist_2": 5, "act_reg": 0, "alive": 1, "solved": 5, "done": 0, "sparse": 0},
          "enable_rsi": False, "rsi_probability": 0, "balls_overlap": False, "overlap_probability": 0, "noise_fingers": 0,
          "limit_init_angle": 3.141592653589793, "goal_time_period": [4, 6], "goal_xrange": [0.02, 0.03], "goal_yrange": [0.022, 0.032],
          "obj_size_range": [0.018, 0.024], "obj_mass_range": [0.03, 0.3], "obj_friction_change": [0.2, 0.001, 2e-05], "task_choice": "random"}


def test_p2_registration_defaults(product_lib):
    m = Model(asset_path("hand/myo_hand_baoding.mjb"), lib=product_lib)
    cfg = make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1")
    assert cfg.kind == _capi.TASK_BAODING and cfg.max_episode_steps == 200 and cfg.frame_skip == 10 and cfg.normalize_act == 1
    assert tuple(cfg.goal_time_period) == (4.0, 6.0) and cfg.task_choice_random == 1 and cfg.randomize_physics == 1
    np.testing.assert_allclose(list(cfg.obj_mass_range), [0.03, 0.3], rtol=1e-6)
    np.testing.assert_allclose(list(cfg.obj_friction_change), [0.2, 0.001, 2e-5], rtol=1e-6)
    assert cfg.drop_th == pytest.approx(1.25) and cfg.proximity_th == pytest.approx(0.015)
    np.testing.assert_allclose(list(cfg.rwd_weight)[:7], [5, 5, 0, 0, 0, 0, 0])      # BaodingEnvV1 defaults


def test_curriculum_config_json_maps(product_lib):
    m = Model(asset_path("hand/myo_hand_baoding.mjb"), lib=product_lib)
    cfg = make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", **STEP32)
    # order: pos_dist_1 pos_dist_2 act_reg alive sparse solved done
    np.testing.assert_allclose(list(cfg.rwd_weight)[:7], [5, 5, 0, 1, 0, 5, 0])
    assert cfg.limit_init_angle == pytest.approx(np.pi) and cfg.overlap_probability == 0.0
    rsi = make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", enable_rsi=True, rsi_probability=0.9, beta_ball_mass=(2, 5))
    assert rsi.enable_rsi == 1 and rsi.rsi_probability == pytest.approx(0.9) and tuple(rsi.beta_ball_mass) == (2.0, 5.0)
    assert rsi.beta_init_angle[0] == 0.0 and rsi.balls_overlap == 0
    with pytest.raises(ValueError):
        make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", beta_ball_size=(0, 1))
    with pytest.raises(TypeError):
        make_task_cfg(m, "CustomMyoChallengeBaodingP2-v1", no_such_kwarg=1)


def test_p1_keeps_nominal_balls(product_lib):
    m = Model(asset_path("hand/myo_hand_baoding.mjb"), lib=product_lib)
    cfg = make_task_cfg(m, "CustomMyoChallengeBaodingP1-v1")
    assert cfg.randomize_physics == 0 and cfg.task_choice_random == 0 and cfg.fixed_task == 2     # WHICH_TASK = CCW
    assert tuple(cfg.goal_xrange) == pytest.approx((0.025, 0.025))


def test_pose_registrations(product_lib):
    m = Model(asset_path("finger/myo_finger_v0.mjb"), lib=product_lib)
    cfg = make_task_cfg(m, "CustomMyoFingerPoseRandom-v0")
    assert cfg.kind == _capi.TASK_POSE and cfg.max_episode_steps == 100 and cfg.n_target_jnt == 4
    names = [m.id2name("joint", cfg.target_jnt_ids[i]) for i in range(4)]
    assert names == ["IFadb", "IFmcp", "IFpip", "IFdip"]
    np.testing.assert_allclose([list(cfg.target_jnt_range[i]) for i in range(4)], [[-.2, .2], [-.4, 1], [.1, 1], [.1, 1]], rtol=1e-6)
    h = Model(asset_path("hand/myo_hand_pose.mjb"), lib=product_lib)
    cfg = make_task_cfg(h, "CustomMyoHandPoseRandom-v0")
    assert cfg.n_target_jnt == 23 and cfg.reset_type == 2 and cfg.pose_thd == pytest.approx(0.8)
    cfg = make_task_cfg(h, "CustomMyoHandPose3Fixed-v0")
    assert cfg.n_target_jnt == 0 and cfg.target_type == 0 and cfg.target_jnt_value[3] == pytest.approx(0.3384)
    e = Model(asset_path("arm/myo_elbow_1dof6muscles.mjb"), lib=product_lib)
    cfg = make_task_cfg(e, "myoElbowPose1D6MRandom-v0")
    assert cfg.n_target_jnt == 1 and cfg.pose_thd == pytest.approx(0.175)
    # the kwargs of the reference's pose mains (/root/reference/src/main_pose_elbow.py:30-43): reset_type "sds"
    cfg = make_task_cfg(e, "CustomMyoElbowPoseRandom-v0", reset_type="sds", sds_distance=0.3, weight_bodyname=None, weight_range=None, target_distance=0.5)
    assert cfg.reset_type == 3 and cfg.sds_distance == pytest.approx(0.3) and cfg.weight_body == -1
    cfg = make_task_cfg(e, "CustomMyoElbowPoseRandom-v0", weight_bodyname="forearm", weight_range=(0.5, 2.0))
    assert cfg.weight_body == e.name2id("body", "forearm") and cfg.n_ovr_body == 1 and cfg.n_ovr_geom == 1
    # die reorientation registrations (/root/reference/src/envs/__init__.py:26-55)
    d = Model(asset_path("hand/myo_hand_die.mjb"), lib=product_lib)
    cfg = make_task_cfg(d, "CustomMyoChallengeDieReorientP2-v0", goal_rot_x=[(-0.5, 0.5), (1.0, 1.2)])
    assert cfg.kind == _capi.TASK_REORIENT and cfg.frame_skip == 5 and cfg.max_episode_steps == 150 and cfg.object_ngeom == 3
    assert cfg.obj_size_change == pytest.approx(0.007) and cfg.n_goal_rot[0] == 2 and cfg.goal_rot_axis[0][1][1] == pytest.approx(1.2)
    assert tuple(cfg.rwd_weight)[:2] == (100.0, 1.0) and cfg.n_ovr_bodypose == 1


def test_factory_names_and_errors():
    assert set(FACTORY_NAMES.values()) <= set(REGISTRY)
    with pytest.raises(ValueError):
        EnvironmentFactory.create("NoSuchEnv")
    with pytest.raises(NotImplementedError):
        EnvironmentFactory.create("CustomMyoPenTwirlRandom")
    with pytest.raises(_capi.MyoError):           # no CPU path: creating worlds without a GPU fails loudly
        if torch.cuda.is_available():
            raise _capi.MyoError("gpu present")
        EnvironmentFactory.create("CustomMyoFingerPoseRandom", num_envs=4, device="cuda:0")


def test_running_mean_std_matches_numpy():
    rng = np.random.default_rng(0)
    x = rng.normal(3, 2, (1000, 5))
    r = RunningMeanStd((5,))
    for chunk in np.split(x, 10):
        r.update(chunk)
    # initial count 1e-4 with mean 0 / var 1 is part of SB3's definition
    np.testing.assert_allclose(r.mean, x.mean(0), atol=1e-5)
    np.testing.assert_allclose(r.var, x.var(0), rtol=1e-5)
    assert r.count == pytest.approx(1000 + 1e-4)


class _FakeVenv:
    num_envs = 3

    class _S:
        shape = (86,)
    observation_space = _S()
    action_space = None


def test_vecnormalize_constants_from_reference_pickle():
    g = np.load(os.path.join(GOLDEN, "vecnormalize_baoding_step32.npz"))
    v = VecNormalize.from_moments(_FakeVenv(), g["obs_mean"], g["obs_var"], g["obs_count"], g["ret_mean"], g["ret_var"], g["ret_count"],
                                  clip_obs=float(g["clip_obs"]), clip_reward=float(g["clip_reward"]), gamma=float(g["gamma"]), epsilon=float(g["epsilon"]))
    assert (v.clip_obs, v.clip_reward, v.gamma, v.epsilon) == (10.0, 10.0, 0.99, 1e-8)
    assert v.obs_rms.count == pytest.approx(2.567e8, rel=1e-3)
    obs = np.tile(g["obs_mean"], (3, 1)).astype(np.float32)
    obs[1] += 3 * np.sqrt(g["obs_var"])
    obs[2] += 1e6
    out = v.normalize_obs(obs)
    np.testing.assert_allclose(out[0], 0, atol=1e-3)
    np.testing.assert_allclose(out[1], 3, atol=0.05)      # float32 observations: sigma of the velocity slots is ~1e-4 of the values
    assert (out[2] == 10).all()
    r = v.normalize_reward(np.array([1.0, 1e9]))
    assert r[0] == pytest.approx(1 / np.sqrt(float(g["ret_var"]) + 1e-8), rel=1e-6) and r[1] == 10


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _moments_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(7)
    x = rng.normal(1, 3, (64, 6))                       # the global batch; each rank owns a shard of worlds
    shard = x[rank * 32:(rank + 1) * 32]
    r = RunningMeanStd((6,))
    for _ in range(3):
        r.update_distributed(shard)
    q.put((rank, r.mean, r.var, r.count, rank_seed(5, rank)))
    dist.destroy_process_group()


def test_two_rank_moment_merge_gloo():
    """World shards on 2 ranks: the all-reduced Chan merge gives every rank the single-process statistics."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_moments_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted([q.get(timeout=120) for _ in ps], key=lambda t: t[0])
    for p in ps:
        p.join(timeout=60)
    rng = np.random.default_rng(7)
    x = rng.normal(1, 3, (64, 6))
    ref = RunningMeanStd((6,))
    for _ in range(3):
        ref.update(x)
    for rank, mean, var, count, seed in res:
        np.testing.assert_allclose(mean, ref.mean, rtol=1e-12)
        np.testing.assert_allclose(var, ref.var, rtol=1e-10)
        assert count == pytest.approx(ref.count)
    assert res[0][4] != res[1][4]                    # ranks draw from disjoint world streams


def test_every_curriculum_step_maps_to_a_task_cfg(product_lib):
    """The reference's 32 training steps (config.json of each, packaged as data) all translate into the device task configuration:
    no knob of the winning curriculum is rejected or silently dropped."""
    from myochallenge_b200 import curriculum

    steps = curriculum.load()
    assert len(steps) == 32 and steps[0]["step"].startswith("01_") and steps[-1]["step"].startswith("32_")
    m = Model(asset_path("hand/myo_hand_baoding.mjb"), lib=product_lib)
    cfgs = {s["step"][:2]: curriculum.task_cfg(s, m) for s in steps}
    c01, c04, c06, c15, c18, c23, c32 = (cfgs[k] for k in ("01", "04", "06", "15", "18", "23", "32"))
    assert c01.p1_reset == 1 and c01.enable_rsi == 1 and c01.rsi_probability == 1.0 and 1e29 < c01.goal_time_period[0] < 3e38 and c01.goal_time_period[1] == c01.goal_time_period[0]      # static targets, finite in fp32
    assert c04.p1_reset == 1 and c04.task_choice_random == 1 and c04.rsi_probability == pytest.approx(0.9) and c04.drop_th == pytest.approx(1.3)
    assert c06.enable_rsi == 0 and tuple(c06.goal_time_period) == (10.0, 10.0)
    assert c15.p1_reset == 0 and c15.overlap_probability == pytest.approx(0.9)
    assert c18.limit_init_angle == pytest.approx(np.pi / 3, rel=1e-3)
    assert c23.noise_fingers == pytest.approx(0.2) and c23.randomize_physics == 1
    assert c32.limit_init_angle == pytest.approx(np.pi) and list(c32.rwd_weight)[:7] == [5, 5, 0, 1, 0, 5, 0]
    with pytest.raises(ValueError):
        make_task_cfg(m, "CustomMyoChallengeBaodingP1-v1", task="sideways")


def test_host_vecnormalize_save_load_round_trip(tmp_path):
    """``VecNormalize.load(path, venv)`` / ``.save(path)`` of the host-array class (the reference: src/main_eval.py:65-67,
    src/train/trainer.py:73-75): statistics and switches survive, including ``training = False`` as evaluation scripts set it."""
    class Venv(_FakeVenv):
        class _A:
            shape = (39,)
        action_space = _A()

    g = np.load(os.path.join(GOLDEN, "vecnormalize_baoding_step32.npz"))
    v = VecNormalize.from_moments(Venv(), g["obs_mean"], g["obs_var"], g["obs_count"], g["ret_mean"], g["ret_var"], g["ret_count"], training=False,
                                  norm_reward=False)
    p = str(tmp_path / "env.pkl")
    v.save(p)
    w = VecNormalize.load(p, Venv())
    np.testing.assert_array_equal(w.obs_rms.mean, v.obs_rms.mean); np.testing.assert_array_equal(w.obs_rms.var, v.obs_rms.var)
    assert w.obs_rms.count == v.obs_rms.count and w.ret_rms.var == v.ret_rms.var and (w.training, w.norm_obs, w.norm_reward) == (False, True, False)
    obs = np.tile(g["obs_mean"], (3, 1)).astype(np.float32) + 0.01
    np.testing.assert_array_equal(w.normalize_obs(obs), v.normalize_obs(obs))


def test_model_check_reports_every_blocking_feature(product_lib, tmp_path):
    """VERDICT r1 (row 37): one call tells whether an out-of-band .mjb runs, and if not, everything that blocks it."""
    from oracle import mjb

    for rel in ("hand/myo_hand_baoding.mjb", "hand/myo_hand_die.mjb", "hand/myo_hand_pose.mjb", "finger/myo_finger_v0.mjb", "arm/myo_elbow_1dof6muscles.mjb"):
        rep = Model(asset_path(rel), lib=product_lib).check()
        assert not any(line.startswith("- ") for line in rep.splitlines()), (rel, rep)
    m = mjb.load(asset_path("hand/myo_hand_baoding.mjb"))
    m.arrays["jnt_type"][3] = 1                      # a ball joint
    m.arrays["dof_frictionloss"][5] = 0.1
    m.arrays["geom_type"][m.name2id("geom", "ball2")] = 4       # an ellipsoid that collides with capsules and a sphere
    m.opt["cone"] = 1
    p = tmp_path / "odd.mjb"
    p.write_bytes(mjb.dump(m))
    rep = Model(str(p), lib=product_lib).check()
    for needle in ("ball joint", "frictionloss", "elliptic", "ellipsoid"):
        assert needle in rep, rep
    assert sum(line.startswith("- ") for line in rep.splitlines()) >= 3       # blocking features; "~ " lines are advisory


def test_contact_excludes_are_honoured(emul_lib, tmp_path):
    """<contact><exclude>: body pairs listed in exclude_signature never collide - same contact list in the oracle and the kernel."""
    from oracle import mjb, oracle
    from parity_common import many_contact_states

    src = asset_path("hand/myo_hand_baoding.mjb")
    m = mjb.load(src)
    b1, b2 = m.name2id("body", "palm"), m.name2id("body", "ball1")
    m.sizes["nexclude"] = 1
    m.arrays["exclude_signature"] = np.array([[(min(b1, b2) << 16) + max(b1, b2)]], np.int32)
    m.arrays["name_excludeadr"] = np.array([[0]], np.int32)
    p = tmp_path / "excl.mjb"
    p.write_bytes(mjb.dump(m))
    q = many_contact_states(src, 6, min_contacts=12)
    om, od = oracle.load(str(p))
    om0, od0 = oracle.load(src)
    model = Model(str(p), lib=emul_lib)
    assert "- " not in model.check()
    cfg = model.default_task_cfg(_capi.TASK_BAODING)
    cfg.randomize_physics = 0            # nominal ball sizes, as in the oracle
    B = BatchSim(model, 6, cfg, device="cpu")
    B.reset()
    B.set_state(q, np.zeros((6, B.nv), np.float32), np.zeros((6, B.na), np.float32))
    B.forward(None)
    geoms = B.stage("contact_geoms").numpy()
    ncon = B.stage("ncon").numpy()[:, 0]
    gb = np.asarray(om.geom_bodyid)
    fewer = 0
    for w in range(6):
        od.reset(); od.qpos[:] = q[w]; od.forward()
        od0.reset(); od0.qpos[:] = q[w]; od0.forward()
        ref = np.stack([od.contact_geom1[: od.ncon], od.contact_geom2[: od.ncon]], 1)
        assert ncon[w] == od.ncon and (geoms[w, : 2 * od.ncon] == ref.reshape(-1)).all()
        assert not any({gb[a], gb[b]} == {b1, b2} for a, b in ref)
        fewer += od0.ncon - od.ncon
    assert fewer > 0          # the excluded pair did collide in the unmodified model


def test_p1_reset_observation_matches_the_reference_checkpoint(emul_lib):
    """VERDICT r1 (missing 6): phase1_final.zip:_last_original_obs[0] is a just-reset Baoding P1 observation produced by MuJoCo on
    the real hand model. The authored stand-in is placed to reproduce it: hand pose, ball rest positions, zero velocities, target
    sites, errors, zero activations. ``ref`` is that vector to 6e-6 (its 5-decimal coordinates)."""
    ref = np.zeros(86)
    ref[0] = -1.57
    ref[23:26], ref[29:32] = (-0.227, -0.511, 1.452), (-0.256, -0.552, 1.442)
    ref[35:38], ref[38:41] = (-0.21591, -0.51066, 1.44507), (-0.25508, -0.54608, 1.45052)
    ref[41:44], ref[44:47] = ref[35:38] - ref[23:26], ref[38:41] - ref[29:32]
    m = Model(asset_path("hand/myo_hand_baoding.mjb"), lib=emul_lib)
    sim = BatchSim(m, 4, make_task_cfg(m, "CustomMyoChallengeBaodingP1-v1"), device="cpu", seed=0)
    obs = sim.reset().numpy()
    np.testing.assert_allclose(obs, np.tile(ref, (4, 1)), atol=1e-5)      # 10 micrometres: the stand-in was authored from 5-decimal coordinates
