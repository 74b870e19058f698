"""GPU: launch shape of the world kernel for the benchmark's Baoding P2 config. The fast scratch layout keeps one world small
enough that 16 one-warp worlds and the staged model tables share an SM's shared memory, at no more than 128 registers a
thread (16 warps x 32 lanes x 128 = the register file)."""
import pytest
import torch

from myochallenge_b200.envs import make_vec_env

pytestmark = pytest.mark.gpu


def test_baoding_p2_runs_16_worlds_per_cta(product_lib):
    env = make_vec_env("CustomMyoChallengeBaodingP2-v1", 4096, device="cuda:0", seed=0, clip_actions=True)
    info = env.sim.launch_info()
    assert info["lanes_per_world"] == 32
    assert info["worlds_per_cta"] == 16, info
    assert info["regs_per_thread"] <= 128, info
    obs = env.reset_device()
    gen = torch.Generator(device="cuda:0").manual_seed(0)
    for _ in range(5):
        obs, _, _, _ = env.step_device(torch.rand(4096, env.sim.nu, device="cuda:0", generator=gen) * 2 - 1)
    assert bool(torch.isfinite(obs).all())
    assert env.sim.status() == 0
    env.close()
