"""CPU: checkpoint / normaliser interchange (SURVEY.md 8f rank 2). Files written by ``myochallenge_b200.checkpoint`` are read
back, and the written pickles are checked to name the SB3 / gym classes (by module and qualname, which is all a pickle stores of
a class) so SB3 can rebuild them."""
import os
import pickle
import pickletools

import numpy as np
import torch

from conftest import GOLDEN
from myochallenge_b200 import checkpoint as ck


def _golden_sd():
    g = np.load(os.path.join(GOLDEN, "policy_phase1.npz"))
    return {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w:")}, g


def _globals_named(b):
    out = set()
    strings = []
    for op, arg, _ in pickletools.genops(b):
        if op.name in ("SHORT_BINUNICODE", "BINUNICODE", "UNICODE"):
            strings.append(arg)
        if op.name == "GLOBAL":
            out.add(arg.replace(" ", "."))
        if op.name == "STACK_GLOBAL":
            out.add(strings[-2] + "." + strings[-1])
    return out


def test_zip_round_trip_and_sb3_layout(tmp_path):
    sd, _ = _golden_sd()
    p = str(tmp_path / "model.zip")
    opt = {"state": {0: {"step": torch.tensor(3.0), "exp_avg": torch.zeros(39), "exp_avg_sq": torch.ones(39)}}, "param_groups": [{"lr": 1e-4, "params": list(range(13))}]}
    ck.save_sb3_zip(p, sd, dict(n_steps=128, batch_size=4096, gamma=0.99, _last_obs=np.arange(6, dtype=np.float32).reshape(2, 3)), opt)
    import zipfile
    with zipfile.ZipFile(p) as z:
        assert {"data", "policy.pth", "policy.optimizer.pth", "pytorch_variables.pth", "_stable_baselines3_version", "system_info.txt"} <= set(z.namelist())
    c = ck.load_sb3_zip(p)
    assert list(c["state_dict"]) == ["log_std", "action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias"] + \
        [f"lstm_{n}.{k}_l0" for n in ("actor", "critic") for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
    for k, v in sd.items():
        assert torch.equal(c["state_dict"][k], v)
    assert c["data"]["n_steps"] == 128 and c["data"]["policy_kwargs"]["lstm_hidden_size"] == 128 and c["version"] == ck.SB3_VERSION
    np.testing.assert_array_equal(c["data"]["_last_obs"], np.arange(6, dtype=np.float32).reshape(2, 3))
    assert c["data"]["policy_class"].__name__ == "RecurrentActorCriticPolicy" and c["data"]["policy_class"].__module__ == "sb3_contrib.common.recurrent.policies"
    assert float(c["optimizer"]["state"][0]["step"]) == 3.0


def test_parameter_order_with_mlp_layers():
    names = ["log_std", "lstm_actor.weight_ih_l0", "lstm_critic.bias_hh_l0", "mlp_extractor.value_net.0.weight", "mlp_extractor.policy_net.2.bias",
             "mlp_extractor.policy_net.0.weight", "action_net.weight", "value_net.bias"]
    assert ck.sb3_parameter_order(names) == ["log_std", "mlp_extractor.policy_net.2.bias", "mlp_extractor.policy_net.0.weight", "mlp_extractor.value_net.0.weight",
                                             "action_net.weight", "value_net.bias", "lstm_actor.weight_ih_l0", "lstm_critic.bias_hh_l0"]


def test_vecnormalize_round_trip_names_sb3_classes(tmp_path):
    rng = np.random.default_rng(0)
    st = dict(obs_mean=rng.normal(size=86), obs_var=rng.random(86) + 0.1, obs_count=12345.5, ret_mean=2.5, ret_var=9.0, ret_count=777.0,
              clip_obs=10.0, clip_reward=10.0, gamma=0.99, epsilon=1e-8, training=False, norm_obs=True, norm_reward=False)
    p = str(tmp_path / "env.pkl")
    ck.save_vecnormalize(p, st, num_envs=16, act_dim=39)
    back = ck.load_vecnormalize(p)
    for k, v in st.items():
        assert np.array_equal(np.asarray(back[k]), np.asarray(v)), k
    named = _globals_named(open(p, "rb").read())
    assert {"stable_baselines3.common.vec_env.vec_normalize.VecNormalize", "stable_baselines3.common.running_mean_std.RunningMeanStd",
            "gym.spaces.box.Box"} <= named
    import sys
    assert "stable_baselines3" not in sys.modules and "gym" not in sys.modules          # the stand-in modules are gone again
    # the attribute set SB3 1.6.2's VecNormalize.__setstate__ / load expects (venv, class_attributes, returns are not pickled)
    with open(p, "rb") as f:
        v = ck._Unpickler(f).load()
    assert {"obs_rms", "ret_rms", "clip_obs", "clip_reward", "gamma", "epsilon", "training", "norm_obs", "norm_reward", "num_envs", "observation_space",
            "action_space", "old_obs", "old_reward", "norm_obs_keys"} <= set(v.__dict__) and "venv" not in v.__dict__
    assert v.observation_space.__dict__["_shape"] == (86,) and v.action_space.__dict__["high"].max() == 1.0


def test_unpickler_does_not_resolve_builtins_or_os(tmp_path):
    """ADVICE r1: the loader must not hand out eval / exec / os.system: a crafted pickle gets inert stand-ins."""
    import pickle

    class Evil:
        def __reduce__(self):
            import os
            return (os.system, ("echo pwned > %s" % (tmp_path / "pwned"),))

    class Evil2:
        def __reduce__(self):
            return (eval, ("__import__('os').getcwd()",))

    for obj in (Evil(), Evil2()):
        out = ck._loads(pickle.dumps(obj))
        assert isinstance(out, ck._Bag)
    assert not (tmp_path / "pwned").exists()


def test_save_and_load_paths_follow_sb3_open_path(tmp_path):
    assert ck.sb3_save_path("a/final_model.pkl") == "a/final_model.pkl"       # the reference's trainer.save name
    assert ck.sb3_save_path("a/rl_model_100_steps") == "a/rl_model_100_steps.zip"
    p = tmp_path / "final_model.pkl"
    p.write_bytes(b"x")
    assert ck.sb3_load_path(str(p)) == str(p)
    assert ck.sb3_load_path(str(tmp_path / "model")) == str(tmp_path / "model") + ".zip"
