#!/usr/bin/env python
"""bench.py - Baoding env-steps/s with the recurrent policy in the loop (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W             # own arm (B200 kernels)
    python bench.py --impl reference --gpus N --steps K ...   # reference arm: CPU path on the host cores

A step = one pass of the hot path over every world of one GPU: policy forward on the current observations
(VecNormalize.normalize_obs fused, Gaussian sample) -> action clip -> env step (frame_skip x mj_step, obs, reward,
termination, TimeLimit, auto-reset).  Workload: configs[4] of BASELINE.json, myoChallengeBaodingP2-v1 with the
registration defaults of /root/reference/src/envs/__init__.py:58-74, 32768 worlds per GPU, random-init
MlpLstmPolicy (LSTM 256, pi = vf = [256, 256], ortho_init False, log_std_init -2) as the winning runs use
(/root/reference/trained_models/curriculum_steps_complete_baoding_winner/01_rsi_static/main.py:178-200).

One JSON line on stdout (rank 0).  `value` times the device-resident loop with CUDA events, max over ranks;
`e2e` times the same loop through the host-array VecEnv API (pinned host buffers, H2D + D2H every step);
`roofline` is the world kernel (dominant launch) against the measured HBM copy bandwidth; `cpu_baseline` times
the oracle (CPU restatement, the one thing bench.py may run from oracle/) on the host cores for a bounded sample.

`--dump-outputs DIR` writes what the last timed step of the `value` loop handed its caller (observations, rewards,
done flags, actions, values, log-probabilities; rank 0) as DIR/<name>.npy, so that two builds can be compared output
for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

sys.dont_write_bytecode = True          # the tree may be read-only; bench.py writes nothing into it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DUMP_LIMIT_BYTES = 64 << 20

METRIC = "Baoding env-steps/sec (1/2/4/8 B200, policy in loop) vs host MuJoCo SubprocVecEnv"
UNIT = "env-steps/s"
ENV_ID = "CustomMyoChallengeBaodingP2-v1"
# winning curriculum reward weights (step 32 config.json of the reference)
RWD = {"pos_dist_1": 5, "pos_dist_2": 5, "act_reg": 0, "alive": 1, "solved": 5, "done": 0, "sparse": 0}


def algorithmic_bytes_per_env_step(nq, nv, na, nu, nobs, nparam):
    """SURVEY.md 8(d): fp32 bytes one env step must move through HBM: action in, obs/reward/flags out, state +
    warm start read and written once, per-world randomised parameters read."""
    return 4 * (nu + nobs + 1) + 2 + 2 * 4 * (nq + nv + na + nv) + 4 * nparam


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason samples during the timed region (NVML)."""

    def __init__(self, index: int, period=0.1):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap", nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (fp64 C restatement of the MuJoCo 2.1.0 step subset) on the host cores, doing the SAME work per env step
# as the product arm: recurrent policy forward (torch, CPU) -> action clip -> env step (target update, muscle remap, frame_skip
# mj_steps, observation, reward, termination) -> reset of finished worlds. One Python thread per host core, 32 worlds per
# thread per call (ctypes and torch release the GIL), oracle built -O3 -march=native on this machine, Newton tolerance at
# MuJoCo's own default (1e-8).
def cpu_env_steps_per_s(seconds: float, threads: int, frame_skip: int = 10, states=None, per: int = 32, with_policy: bool = True):
    import ctypes

    import numpy as np
    import torch

    from myochallenge_b200.assets import asset_path
    from oracle import mjb, oracle

    path = asset_path("hand/myo_hand_baoding.mjb")
    L = oracle.lib(oracle.build_fast())
    L.o_set_solver_tol(1e-8)
    torch.set_num_threads(1)
    nw = threads * per
    src = mjb.load(path)
    models = [oracle.OracleModel(src) for _ in range(threads)]
    datas = [oracle.OracleData(m) for m in models]
    m0 = models[0]
    nobs = (m0.nq - 14) + 24 + m0.na
    q0r = np.array(m0.qpos0, np.float64).copy()
    q0r[:23] = 0.0
    q0r[0] = -1.57                             # reference init pose (/root/reference/src/envs/baoding.py:400-401)
    if states is None:
        qpos = np.tile(q0r, (nw, 1)); qvel = np.zeros((nw, m0.nv)); act = np.zeros((nw, m0.na))
    else:
        qpos, qvel, act = [np.ascontiguousarray(np.resize(np.asarray(a, np.float64), (nw, a.shape[1]))) for a in states]
    warm = np.zeros((nw, m0.nv))
    obs = np.zeros((nw, nobs)); reward = np.zeros(nw); done = np.zeros(nw, np.int32)
    rng0 = np.random.default_rng(0)

    def new_task(k):      # CustomBaodingP2Env.reset with the P2 registration's ranges
        a1 = rng0.uniform(0, 2 * np.pi, k)
        return np.stack([rng0.integers(0, 3, k).astype(float), a1, a1 - np.pi, rng0.uniform(0.020, 0.030, k), rng0.uniform(0.022, 0.032, k),
                         rng0.uniform(4, 6, k), np.zeros(k)], 1)

    task = np.ascontiguousarray(new_task(nw))
    ids = np.array([src.name2id("site", "ball1_site"), src.name2id("site", "ball2_site"), src.name2id("site", "target1_site"),
                    src.name2id("site", "target2_site"), m0.nv - 12, m0.nv - 6], np.int32)
    weights = np.array([5.0, 5.0, 0.0, 1.0, 0.0, 5.0, 0.0])      # the winning run's reward weights (RWD)
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)

    class Policy(torch.nn.Module):      # MlpLstmPolicy: LSTM-256 + [256, 256] for actor and critic, Gaussian head (log_std_init -2)
        def __init__(self):
            super().__init__()
            self.la, self.lc = torch.nn.LSTMCell(nobs, 256), torch.nn.LSTMCell(nobs, 256)
            self.pi = torch.nn.Sequential(torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, m0.nu))
            self.vf = torch.nn.Sequential(torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 1))

    torch.manual_seed(0)
    pol = Policy().double()
    counts = [0] * threads
    stop = time.perf_counter() + seconds

    def work(t):
        lo, hi = t * per, (t + 1) * per
        g = torch.Generator().manual_seed(t)
        ha, ca, hc, cc = [torch.zeros(per, 256, dtype=torch.float64) for _ in range(4)]
        action = np.zeros((nw, m0.nu))
        with torch.no_grad():
            while time.perf_counter() < stop:
                if with_policy:
                    o = torch.from_numpy(obs[lo:hi])
                    ha, ca = pol.la(o, (ha, ca)); hc, cc = pol.lc(o, (hc, cc))
                    mean, _value = pol.pi(ha), pol.vf(hc)
                    action[lo:hi] = (mean + np.exp(-2.0) * torch.randn(per, m0.nu, generator=g, dtype=torch.float64)).clamp_(-1, 1).numpy()
                else:
                    action[lo:hi] = np.random.default_rng(counts[t]).uniform(-1, 1, (per, m0.nu))
                L.o_batch_env_step(models[t]._p, datas[t]._p, lo, hi, frame_skip, qpos.ctypes.data_as(dp), qvel.ctypes.data_as(dp), act.ctypes.data_as(dp),
                                   warm.ctypes.data_as(dp), action.ctypes.data_as(dp), task.ctypes.data_as(dp), ids.ctypes.data_as(ip),
                                   weights.ctypes.data_as(dp), 1.25, 0.015, obs.ctypes.data_as(dp), reward.ctypes.data_as(dp), done.ctypes.data_as(ip))
                for w in range(lo, hi):      # SubprocVecEnv worker: reset on done (or a non-finite state) / TimeLimit
                    if done[w] or task[w, 6] >= 200 or not np.isfinite(qpos[w]).all():
                        qpos[w] = q0r; qvel[w] = 0; act[w] = 0; warm[w] = 0; task[w] = new_task(1)[0]
                        ha[w - lo] = 0; ca[w - lo] = 0; hc[w - lo] = 0; cc[w - lo] = 0
                counts[t] += per

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    dt = time.perf_counter() - t0
    total = sum(counts)
    what = "recurrent policy forward (torch CPU, fp64) + env step" if with_policy else "env step under uniform random actions"
    return total / dt, (f"{total} env steps ({what}: targets, remap, {frame_skip} mj_steps, obs, reward, reset; fp64 oracle -O3 -march=native, Newton tol 1e-8) "
                        f"of {nw} Baoding worlds in {dt:.1f} s on {threads} threads")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    # each "step" = a bounded sample: `--cpu-seconds` / steps of oracle stepping on all host cores
    per_step = max(0.5, args.cpu_seconds / max(1, args.steps))
    for _ in range(min(args.warmup, 1)):
        cpu_env_steps_per_s(0.5, threads)
    vals = []
    sample = ""
    for _ in range(args.steps):
        v, sample = cpu_env_steps_per_s(per_step, threads)
        vals.append(v)
    value = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{ENV_ID} (BASELINE configs[4]) on the host cores: policy forward + env step per world, 32 worlds per thread", "worlds_per_gpu": 0, "frame_skip": 10,
                   "note": "MuJoCo/MyoSuite/SB3 are not installable offline (no wheels, no network): the reference's CPU path is "
                           "represented by the fp64 C restatement of its mj_step subset (oracle/, built -O3 -march=native here, Newton "
                           "tolerance 1e-8 as MuJoCo's default), one thread per host core, with the same per-step work as the product arm "
                           "(recurrent policy forward, targets, remap, obs, reward, resets)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------------------
def dump_outputs(path, stepper):
    """What ``stepper.step()`` left for its caller after the last timed step - every sub-batch's results concatenated in world
    order - as float32 DIR/<name>.npy. Above DUMP_LIMIT_BYTES in all, the same seeded sample of worlds is kept in every file."""
    import numpy as np
    import torch

    outs = {"obs": stepper.obs, "reward": stepper.rewards, "done": stepper.dones, "actions": [o[0] for o in stepper.out],
            "values": [o[1] for o in stepper.out], "log_prob": [o[2] for o in stepper.out]}
    arrays = {k: torch.cat([t.float() for t in v]).cpu().numpy() for k, v in outs.items()}
    n = stepper.num_envs
    row_bytes = sum(a.nbytes for a in arrays.values()) // n
    rows = slice(None)
    if row_bytes * n > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(a[rows]))


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from myochallenge_b200 import _capi
    from myochallenge_b200.envs import make_vec_env
    from myochallenge_b200.policy import RecurrentPolicy
    from myochallenge_b200.vec_env import rank_seed

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path for the product arm)")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.worlds

    env = make_vec_env(ENV_ID, n, device=dev, seed=rank_seed(args.seed, rank), weighted_reward_keys=RWD, clip_actions=True)
    sim = env.sim
    pol = RecurrentPolicy(sim.nobs, sim.nu, lstm_hidden=256, pi=(256, 256), vf=(256, 256), max_batch=n, device=dev, use_sde=args.use_sde)
    pol.init_random(seed=0, log_std_init=-2.0)             # same weights on every rank
    pol.seed(0x5EED + rank)
    stats = os.path.join(ROOT, "myochallenge_b200", "assets", "vecnormalize", "baoding_step32.npz")
    if os.path.exists(stats):                               # the reference's own running moments (fixture), applied as
        g = np.load(stats)                                  # VecNormalize.normalize_obs in the policy's input load
        pol.set_obs_norm(torch.from_numpy(g["obs_mean"]).float(), torch.from_numpy(g["obs_var"]).float(), float(g["epsilon"]), float(g["clip_obs"]))
    h, c = pol.initial_state(n)
    out = (torch.empty(n, sim.nu, device=dev), torch.empty(n, device=dev), torch.empty(n, device=dev))
    starts = torch.ones(n, dtype=torch.uint8, device=dev)

    obs = env.reset_device()
    torch.cuda.synchronize()

    def step_device():
        nonlocal obs, starts
        actions, _, _, _ = pol.forward(obs, (h, c), starts, out=out)
        obs, rew, done, trunc = env.step_device(actions)
        starts = done

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # untimed spin-up to the steady state of the workload: right after a reset every world is in the cheap opening phase of
    # its episode (balls resting on the palm, few contacts); episodes end at random times (drop / TimeLimit), and only after
    # ~one horizon are the episode phases - and with them contact counts and Newton iterations per substep - mixed as they
    # are for the rest of a training run. Timing the first steps would overstate throughput by ~20 %.
    # With a policy that rarely drops the balls nearly every episode runs the full horizon, so worlds that start together stay
    # in phase for ever (all 32768 would truncate on the same step); the spin-up therefore staggers them - world w is reset
    # once, at spin-up step w mod horizon - so that any timed window averages over the phases of an episode.
    horizon = int(env.cfg.max_episode_steps)
    widx = torch.arange(n, device=dev)

    def stagger(sim_, t, starts_):
        if horizon > 0 and t < horizon:
            mask = (widx[: sim_.n] % horizon) == t
            sim_.reset(mask)
            return torch.maximum(starts_, mask.to(torch.uint8))
        return starts_

    for t in range(args.spinup):
        starts = stagger(sim, t, starts)
        step_device()
    for _ in range(args.warmup):
        step_device()
    barrier()
    l0 = sim.launch_count + pol.launch_count
    sampler = ClockSampler(local)
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 2)]
    ev[0].record()
    for i in range(args.steps):
        actions, _, _, _ = pol.forward(obs, (h, c), starts, out=out)
        ev[2 * i + 1].record()                              # brackets the world kernel on its own stream
        obs, rew, done, trunc = env.step_device(actions)
        ev[2 * i + 2].record()
        starts = done
    ev[-1].record()
    barrier()
    clocks = sampler.stop()
    launches = sim.launch_count + pol.launch_count - l0
    total_ms = ev[0].elapsed_time(ev[-1])
    world_ms = sum(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.steps)) / args.steps
    policy_ms = total_ms / args.steps - world_ms
    status = sim.status()

    # ---- value: the same step with the worlds split into two half-size sub-batches on two streams (rollout.PipelinedStepper):
    # the policy forward of one half runs on the SMs the other half's world kernel frees as it drains, so the policy's time and the
    # drain tail leave the step. The single-stream loop above stays for the per-kernel times the rooflines use.
    from myochallenge_b200.rollout import PipelinedStepper

    nh = n // 2
    halves = [make_vec_env(ENV_ID, nh, device=dev, seed=rank_seed(args.seed + 101 + k, rank), weighted_reward_keys=RWD, clip_actions=True)
              for k in range(2)]
    stepper = PipelinedStepper(halves, pol)
    stepper.reset()
    stepper.spin_up(args.spinup)                            # same steady state as the single-stream loop
    for _ in range(args.warmup):
        stepper.step()
    stepper.synchronize()
    barrier()
    lp0 = sum(hv.sim.launch_count for hv in halves) + pol.launch_count
    sampler = ClockSampler(local)
    sampler.start()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for s_ in stepper.streams:
        s_.wait_stream(torch.cuda.current_stream())
    for _ in range(args.steps):
        stepper.step()
    stepper.join()
    pe1.record()
    barrier()
    clocks = sampler.stop()
    pipe_ms = pe0.elapsed_time(pe1)
    pipe_launches = sum(hv.sim.launch_count for hv in halves) + pol.launch_count - lp0
    status |= halves[0].sim.status() | halves[1].sim.status()
    if args.dump_outputs and rank == 0:                     # before the e2e leg below steps the same sub-batches again
        dump_outputs(args.dump_outputs, stepper)

    # ---- e2e: the SB3-shaped host-array API, H2D + D2H inside the timed region -------------------------------
    # (1) one MyoVecEnv, synchronous loop: obs H2D -> policy -> actions D2H -> step_async (actions H2D) -> step_wait
    #     (obs / reward / done D2H). Every copy sits on the critical path.
    # (2) the same calls on two half-size MyoVecEnvs stepped alternately on two streams (a user-level double buffer,
    #     as one would run two SubprocVecEnvs): while one half's world kernel runs, the host drains and refills the
    #     other half. Reported as `e2e`; (1) is kept beside it as `sequential`.
    pin = dict(dtype=torch.float32, pin_memory=True)
    h_obs = torch.zeros(n, sim.nobs, **pin)
    h_act = torch.zeros(n, sim.nu, **pin)
    d_obs = torch.zeros(n, sim.nobs, device=dev)
    ob, _, dn, _ = env.step(np.zeros((n, sim.nu), np.float32))      # warm the host path
    h_obs.copy_(torch.from_numpy(ob))
    starts_h = torch.from_numpy(dn.astype(np.uint8)).to(dev)
    e2e_steps = max(2, min(args.steps, args.e2e_steps))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        d_obs.copy_(h_obs, non_blocking=True)                             # H2D: observations for the policy
        actions, _, _, _ = pol.forward(d_obs, (h, c), starts_h, out=out)
        h_act.copy_(actions, non_blocking=True)                           # D2H: sampled actions
        torch.cuda.current_stream().synchronize()
        env.step_async(np.clip(h_act.numpy(), -1.0, 1.0))                 # H2D: actions (inside step_async)
        ob, rw, dn, _ = env.step_wait(with_infos=False)                   # D2H: obs, reward, done
        h_obs.copy_(torch.from_numpy(ob))
        starts_h = torch.from_numpy(dn.astype(np.uint8)).to(dev, non_blocking=True)
    barrier()
    seq_s = time.perf_counter() - t0
    h2d = env.h2d_bytes_per_step + n * sim.nobs * 4 + n
    d2h = env.d2h_bytes_per_step + n * sim.nu * 4

    # K sub-batches, each with its own stream and pinned buffers (K = 2 reuses the halves of the device-resident loop). More parts
    # than two keep a world kernel queued on the GPU while the host handles one part's copies, at the price of shorter launches.
    K = max(2, args.e2e_parts)
    if K == 2:
        parts, strm, nk = halves, stepper.streams, nh
        pstate, pstarts, pout = stepper.states, [x.clone() for x in stepper.starts], stepper.out
        pobs = stepper.obs
    else:
        del halves
        nk = n // K
        parts = [make_vec_env(ENV_ID, nk, device=dev, seed=rank_seed(args.seed + 211 + k, rank), weighted_reward_keys=RWD, clip_actions=True)
                 for k in range(K)]
        pst = PipelinedStepper(parts, pol)
        pst.reset()
        pst.spin_up(args.spinup)
        pst.synchronize()
        strm, pstate, pstarts, pout, pobs = pst.streams, pst.states, [x.clone() for x in pst.starts], pst.out, pst.obs
    hb = [dict(h_obs=torch.zeros(nk, sim.nobs, **pin), h_act=torch.zeros(nk, sim.nu, **pin), d_obs=torch.zeros(nk, sim.nobs, device=dev),
               out=pout[k], state=pstate[k], starts=pstarts[k]) for k in range(K)]

    def issue(k):
        b = hb[k]
        with torch.cuda.stream(strm[k]):
            b["d_obs"].copy_(b["h_obs"], non_blocking=True)
            actions, _, _, _ = pol.forward(b["d_obs"], b["state"], b["starts"], out=b["out"])
            b["h_act"].copy_(actions, non_blocking=True)
            strm[k].synchronize()
            parts[k].step_async(np.clip(b["h_act"].numpy(), -1.0, 1.0))

    def collect(k):
        b = hb[k]
        with torch.cuda.stream(strm[k]):
            ob, rw, dn, _ = parts[k].step_wait(with_infos=False)
            b["h_obs"].copy_(torch.from_numpy(ob))
            b["starts"] = torch.from_numpy(dn.astype(np.uint8)).to(dev, non_blocking=True)

    for k in range(K):                                                     # the parts are at the steady state already
        with torch.cuda.stream(strm[k]):
            hb[k]["h_obs"].copy_(pobs[k])
            strm[k].synchronize()
    for _ in range(2):                                                     # warm the host path of every part
        for k in range(K):
            issue(k)
        for k in range(K):
            collect(k)
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        issue(k)
    for _ in range(e2e_steps - 1):
        for k in range(K):
            collect(k)
            issue(k)
    for k in range(K):
        collect(k)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_launches = sum(hv.sim.launch_count for hv in parts)

    # ---- whole PPO iteration (BASELINE configs[4]: "... with PPO training"): rollout of n_steps + RecurrentPPO.train ------
    ppo = None
    if not args.no_train:
        from myochallenge_b200.ppo import RecurrentPPO
        from myochallenge_b200.rollout import DeviceVecNormalize, collect_rollouts

        del parts, hb, stepper
        if K == 2:
            del halves
        else:
            del pst
        torch.cuda.empty_cache()
        vn = DeviceVecNormalize(env, gamma=0.99)
        bw = min(n, args.ppo_batch_worlds)
        # phase-2 hyper-parameters of the reference (/root/reference/docs/summary.md:103-117), winning architecture
        agent = RecurrentPPO("MlpLstmPolicy", vn, n_steps=args.ppo_steps, batch_size=args.ppo_steps * bw, n_epochs=args.ppo_epochs,
                             learning_rate=2.5e-5, clip_range=0.2, ent_coef=3e-5, max_grad_norm=0.8, gae_lambda=0.95, seed=0, use_sde=args.use_sde,
                             policy_kwargs=dict(lstm_hidden_size=256, net_arch=[dict(pi=[256, 256], vf=[256, 256])], log_std_init=-2.0,
                                                ortho_init=False, enable_critic_lstm=True))
        agent.policy.seed(0x5EED + rank)
        o = vn.reset_device().clone()
        st = torch.ones(n, dtype=torch.uint8, device=dev)
        state = agent.policy.initial_state(n)
        times = []
        for it in range(2):                                   # iteration 0 warms cuBLAS / allocator; iteration 1 is reported
            barrier()
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            lc0 = agent.update.launch_count
            e[0].record()
            o, st = collect_rollouts(vn, agent.policy, agent.buffer, state, o, st)
            e[1].record()
            log = agent.update.train(agent.buffer, args.ppo_epochs, agent._gen)
            e[2].record()
            barrier()
            times = [e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])]
        tt = torch.tensor(times, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        roll_ms, upd_ms = [float(x) for x in tt]
        ppo = {"value": world * n * args.ppo_steps / ((roll_ms + upd_ms) * 1e-3), "unit": UNIT, "rollout_ms": roll_ms, "update_ms": upd_ms,
               "n_steps": args.ppo_steps, "minibatch_worlds": bw, "n_epochs": args.ppo_epochs, "optimizer_steps": log["train/n_updates"],
               "update_samples_per_s": world * log["train/n_updates"] * bw * args.ppo_steps / (upd_ms * 1e-3),
               "update_launches": agent.update.launch_count - lc0, "approx_kl": log["train/approx_kl"], "clip_fraction": log["train/clip_fraction"],
               "note": "one full RecurrentPPO iteration: collect_rollouts (policy + env + VecNormalize + buffer + GAE) then n_epochs over the "
                       "rollout in minibatches of whole world sequences (bf16-operand cuBLAS GEMMs, own cell/loss/Adam kernels), "
                       "one flat-bucket gradient all-reduce per optimiser step when n_gpus > 1"}

    # max over ranks
    t = torch.tensor([total_ms, world_ms, e2e_s, seq_s, pipe_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, world_ms, e2e_s, seq_s, pipe_ms = [float(x) for x in t]
    single_ms_per_step = total_ms / args.steps
    ms_per_step = pipe_ms / args.steps
    value = world * 2 * nh * args.steps / (pipe_ms * 1e-3)
    single_value = world * n * args.steps / (total_ms * 1e-3)
    e2e_value = world * K * nk * e2e_steps / e2e_s
    seq_value = world * n * e2e_steps / seq_s

    # ---- roofline of the dominant kernel -----------------------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    b_env = algorithmic_bytes_per_env_step(sim.nq, sim.nv, sim.na, sim.nu, sim.nobs, sim.nparam)
    achieved = b_env * n / (world_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "world_kernel_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj.get("dram_bytes_per_launch_at_32768_worlds")
    roofline = {"kernel": "myo::world_kernel<32> (frame_skip x mj_step + obs/reward/reset, one launch per env step)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_env_step": b_env, "kernel_ms": world_ms, "kernel_share_of_step": world_ms / single_ms_per_step,
                "note": "state stays in shared memory across the 10 substeps: the kernel is FP32-issue/latency bound, not HBM bound (DESIGN.md)"}

    # ---- compute roofline: the bound that actually governs the world kernel (SURVEY.md 8d: FP32 issue / latency) ------------
    # FLOP and instruction counts per env step come from the committed ncu capture of this kernel (profiles/, per-launch
    # counters divided by the worlds of the launch); the peak is measured live on this GPU (myo_fp32_fma_peak).
    import ctypes as C
    compute = None
    cpath = os.path.join(ROOT, "profiles", "world_kernel_counters.json")
    if os.path.exists(cpath):
        cj = json.load(open(cpath))
        pk = C.c_double()
        _capi.check(_capi.lib(), _capi.lib().myo_fp32_fma_peak(local, C.byref(pk)))
        flop = float(cj["fp32_flop_per_env_step"])
        ach = flop * n / (world_ms * 1e-3) / 1e12
        compute = {"kernel": roofline["kernel"], "bound": "fp32-issue", "achieved": ach, "peak": pk.value, "unit": "TFLOP/s", "frac": ach / pk.value if pk.value else None,
                   "peak_source": "myo_fp32_fma_peak: FFMA microbenchmark run on this GPU just now (2 flop per FMA)",
                   "fp32_flop_per_env_step": flop, "thread_inst_per_env_step": cj.get("thread_inst_per_env_step"),
                   "warp_inst_per_env_step": cj.get("warp_inst_per_env_step"), "fp32_share_of_thread_inst": cj.get("fp32_share_of_thread_inst"),
                   "issue_slot_utilisation_pct": cj.get("issue_active_pct"), "active_lanes_per_warp_inst": cj.get("lanes_per_inst"),
                   "warps_per_sm": cj.get("warps_per_sm"), "counters_source": cj.get("source")}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 physics, bf16 x bf16 -> f32 policy GEMMs", "data": "synthetic",
        "config": {"workload": f"{ENV_ID} (BASELINE configs[4]), {n} worlds per GPU, frame_skip 10, horizon 200, full physics randomisation, "
                               "random-init MlpLstmPolicy LSTM-256 + [256,256] actor/critic in the loop",
                   "worlds_per_gpu": n, "parallelism": f"worlds sharded over {world} GPU(s), no data-path collective",
                   "l2": "per-step working set (state + LSTM h/c + obs, ~190 MB at 32768 worlds) exceeds the 126 MB L2; no explicit flush",
                   "use_sde": bool(args.use_sde), "spinup_steps": args.spinup, "steady_state": "untimed spin-up of one horizon before warm-up, worlds' episode phases staggered uniformly over the horizon",
                   "pipeline": "two half-size sub-batches stepped on two streams (rollout.PipelinedStepper): the policy forward of one half runs under "
                               "the drain of the other half's world kernel; `single_stream` = one full-size batch on one stream (its per-kernel times feed the rooflines)",
                   "single_stream": {"value": single_value, "ms_per_step": single_ms_per_step, "policy_ms": policy_ms, "world_kernel_ms": world_ms},
                   "policy_ms": policy_ms, "world_kernel_ms": world_ms, "status_flags": status},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "sequential": seq_value,
                "parts": K,
                "api": f"MyoVecEnv.step_async/step_wait with numpy arrays + RecurrentPolicy.forward on H2D-copied observations; {K} envs of {nk} worlds "
                       "stepped in turn on their own streams (`sequential`: one env, every copy on the critical path)"},
        "gpu_launches": int(pipe_launches), "clocks": clocks, "roofline": roofline, "compute_roofline": compute, "ppo_iteration": ppo,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        q, v, a, _ = [x.double().cpu().numpy() for x in sim.get_state()]
        threads = os.cpu_count() or 1
        val, sample = cpu_env_steps_per_s(args.cpu_seconds, threads, states=(q[:256], v[:256], a[:256]))
        line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--worlds", type=int, default=32768, help="worlds per GPU")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-parts", type=int, default=2, help="sub-batches of the end-to-end loop (each with its own stream and pinned buffers)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--spinup", type=int, default=200, help="untimed env steps before warm-up (one horizon: steady-state episode phases)")
    ap.add_argument("--use-sde", action="store_true", help="generalised state-dependent exploration (the reference's winning runs train with use_sde=True)")
    ap.add_argument("--no-train", action="store_true", help="skip the whole-PPO-iteration leg")
    ap.add_argument("--ppo-steps", type=int, default=128, help="n_steps of the PPO iteration leg")
    ap.add_argument("--ppo-batch-worlds", type=int, default=2048, help="world sequences per minibatch")
    ap.add_argument("--ppo-epochs", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path; the reference arm has none")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    return run_reference(args) if args.impl == "reference" else run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
