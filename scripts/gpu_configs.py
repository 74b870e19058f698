"""Throughput of the other BASELINE configs (elbow / finger / hand pose) with the policy in the loop (development aid; the
bench contract measures configs[4], Baoding)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from myochallenge_b200.envs import make_vec_env
from myochallenge_b200.policy import RecurrentPolicy

dev = "cuda:0"
for env_id, n in (("CustomMyoElbowPoseRandom-v0", 1), ("CustomMyoElbowPoseRandom-v0", 65536), ("CustomMyoFingerPoseRandom-v0", 4096),
                  ("CustomMyoFingerPoseRandom-v0", 65536), ("CustomMyoHandPoseRandom-v0", 16384), ("CustomMyoChallengeDieReorientP2-v0", 16384),
                  ("CustomMyoChallengeBaodingP1-v1", 32768), ("myoFingerReachRandom-v0", 4096), ("myoFingerReachRandom-v0", 65536)):
    env = make_vec_env(env_id, n, device=dev, seed=0, clip_actions=True)
    pol = RecurrentPolicy(env.sim.nobs, env.sim.nu, 256, (256, 256), (256, 256), max_batch=n, device=dev)
    pol.init_random(0, -2.0); pol.seed(1)
    obs = env.reset_device(); h, c = pol.initial_state(n); st = torch.ones(n, dtype=torch.uint8, device=dev)
    def step():
        global obs, st
        a, _, _, _ = pol.forward(obs, (h, c), st)
        obs, r, d, t = env.step_device(a); st = d
    for _ in range(110):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    K = 30
    e0.record()
    for _ in range(K):
        step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    print(f"{env_id:34s} n={n:6d}  {ms:8.3f} ms/step  {n / ms * 1e3:.3e} env-steps/s  status={env.sim.status()} done_frac={float(st.float().mean()):.4f} launch={env.sim.launch_info()}", flush=True)
    env.close(); del env, pol
