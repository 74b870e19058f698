// World kernel + the device half of the C ABI (myo_batch_*).
//
// One world per tile of G lanes (G = 8 / 16 / 32 by model size); the world's whole mjData subset
// lives in the tile's slice of shared memory for the duration of an env step: frame_skip mj_steps,
// then kinematics at the new state, observation, reward, termination, TimeLimit and auto-reset,
// all in one launch. HBM is touched once per env step: state + per-world parameters in (float4,
// world-major rows so a tile reads one contiguous row), state + obs/reward/flags out.
#include <cuda_runtime.h>
#ifndef MYO_EMUL
#include <cub/device/device_radix_sort.cuh>
#endif

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "myo_pack.hpp"
#include "myo_task.cuh"

const myo::Model& myo_model_host(const myo_model* m);

// kernel launch; tests/emul re-defines this to run the same kernels single-lane on the host
#ifndef MYO_LAUNCH
#define MYO_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif
#ifndef MYO_LANES_CASES
#define MYO_LANES_CASES(b, FN, ...)                 \
  switch ((b)->pm.lanes) {                          \
    case 8: rc = FN<8>(__VA_ARGS__); break;         \
    case 16: rc = FN<16>(__VA_ARGS__); break;       \
    default: rc = FN<32>(__VA_ARGS__); break;       \
  }
#endif

namespace myo {

constexpr int kThreads = 512;   // up to 16 one-warp worlds per CTA (register cap 128: 16 warps fill the register file)

// hand world w to the full-capacity kernel of this env step
MYO_DI void redo_push(const BatchPtrs& b, int w, int kind) {
#ifdef MYO_EMUL
  const int k = (*b.redo_count)++;
#else
  const int k = atomicAdd(b.redo_count, 1);
#endif
#ifdef MYO_EMUL
  b.redo_list[k] = w | (kind << 30);
#else
  *reinterpret_cast<volatile int*>(b.redo_list + k) = w | (kind << 30);      // consumers wait for the slot to turn non-negative
#endif
}

// One world, one env step / reset / test hook. SOLO: the CTA holds this world only (full-capacity layout), so phases may be
// called conditionally; otherwise every tile of the CTA must reach the same phase barriers and anything that needs extra
// physics (a reset with reference-state initialisation) or more room (more contacts / limit rows than the fast layout
// holds) is handed to the SOLO kernel through the redo list.
template <int G, int RMAX, bool SOLO, int V>
__device__ void run_world(int mslot, const myo_task_cfg& t, const BatchPtrs& b, const StepArgs& a, Ctx<G, V> c, int w, int kind) {
  MYO_M
  int status = 0;
  bool deferred_reset = false;
  int* ti = b.task_i + (size_t)w * TI_WORDS;
  float* tf = b.task_f + (size_t)w * TF_WORDS;
  float* ptarget = b.pose_target + (size_t)w * m.nq4;
  int* misc = SI(o_misc);
  const bool io = w < b.n_worlds;                    // padding worlds never touch caller buffers
  const int wi = io ? w : b.n_worlds - 1;
  const bool redo_reset = a.mode == MODE_REDO && kind == REDO_RESET;
  if (a.mode == MODE_RESET || redo_reset) {
    if (a.mode == MODE_RESET && a.mask && !a.mask[wi]) return;
    load_world<G>(mslot, c, b, w);
    task_reset<G, RMAX, SOLO>(mslot, t, c, b, w, ti, tf, ptarget);
    if (c.lane == 0) b.time[w] = 0.f;
    if (a.obs && io) {
      phase_tree_forward<G>(mslot, c, false);
      task_obs<G>(mslot, t, c, ptarget);
      write_obs<G>(mslot, c, a.obs + (size_t)w * m.nobs, b.time + w, false);
    }
    store_world<G>(mslot, c, b, w, true);
    return;
  }
  load_world<G>(mslot, c, b, w);
  if (a.mode == MODE_GET_OBS) {
    if (!io) return;
    phase_tree_forward<G>(mslot, c, false);
    task_obs<G>(mslot, t, c, ptarget);
    write_obs<G>(mslot, c, a.obs + (size_t)w * m.nobs, b.time + w, false);
    return;
  }
  if (a.mode == MODE_FORWARD || a.mode == MODE_MJ_STEP) {
    for (int i = c.lane; i < m.nu; i += G) SF(o_ctrl)[i] = a.in ? a.in[(size_t)wi * m.nu + i] : 0.f;
    c.tile.sync();
    if (a.mode == MODE_FORWARD) mj_forward_dev<G, RMAX, !SOLO>(mslot, c, &status, false);
    else {
      for (int s = 0; s < a.nsub; s++) mj_step_dev<G, RMAX, !SOLO>(mslot, c, &status, false);
      if (c.lane == 0) b.time[w] += (float)a.nsub * m.timestep;
    }
  } else {   // MODE_ENV_STEP (or its repetition with full capacities)
    if (t.kind == MYO_TASK_BAODING) baoding_targets<G>(mslot, t, c, ti, tf);
    task_action<G>(mslot, t, c, a.in + (size_t)wi * m.nu);
    c.tile.sync();
    for (int s = 0; s < a.nsub; s++) mj_step_dev<G, RMAX, !SOLO>(mslot, c, &status, true);
    if (!SOLO && b.redo_list) {
      // outgrew the fast layout in some substep: nothing of this attempt is kept, the full-capacity kernel steps the world again
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) status |= c.tile.shfl_xor(status, o);
      if (status & (ST_CON_OVERFLOW | ST_EFC_OVERFLOW)) {
        if (c.lane == 0 && io) redo_push(b, w, REDO_STEP);
        if (c.lane == 0 && b.work) b.work[w] = io ? 0 : 0x7fff;
        if (io) return;
        status &= ~(ST_CON_OVERFLOW | ST_EFC_OVERFLOW);
      }
    }
    // get_obs: kinematics at the post-step state (MyoSuite get_obs -> sim.forward)
    phase_tree_forward<G>(mslot, c, false);
    task_obs<G>(mslot, t, c, ptarget);
    float info[MYO_INFO_TERMS], reward;
    bool env_done;
    task_reward<G>(mslot, t, c, tf, ti[TI_ELAPSED] + 1, info, &reward, &env_done);
    if (t.reward_sparse) reward = info[4];      // reward_mode "sparse": the sparse term, slot 4 of every kind
    // a world whose state left the finite range ends its episode here (MuJoCo would warn and reset the data): the reset
    // below keeps NaNs out of the running moments downstream
    bool bad = false;
    for (int i = c.lane; i < m.nq; i += G) bad |= !isfinite(SF(o_qpos)[i]);
    for (int i = c.lane; i < m.nv; i += G) bad |= !isfinite(SF(o_qvel)[i]);
    bad = c.tile.ballot(bad) != 0u;
    if (bad) {
      status |= ST_NONFINITE; env_done = true; reward = 0.f;
#pragma unroll
      for (int k = 0; k < MYO_INFO_TERMS; k++) info[k] = 0.f;
      info[6] = 1.f;
      for (int i = c.lane; i < m.nobs_scr; i += G) SF(o_obs)[i] = 0.f;
      c.tile.sync();
    }
    const int elapsed = ti[TI_ELAPSED] + 1;
    const bool limit = t.max_episode_steps > 0 && elapsed >= t.max_episode_steps;
    const bool done = env_done || limit;
    c.tile.sync();
    if (c.lane == 0) {
      ti[TI_ELAPSED] = elapsed;
      b.time[w] += (float)a.nsub * m.timestep;
      if (io) {
        a.reward[w] = reward;
        a.done[w] = done ? 1 : 0;
        if (a.truncated) a.truncated[w] = (limit && !env_done) ? 1 : 0;
      }
    }
    if (a.info && io) for (int k = c.lane; k < MYO_INFO_TERMS; k += G) a.info[(size_t)w * MYO_INFO_TERMS + k] = info[k];
    if (done && t.auto_reset) {
      if (a.terminal_obs && io) write_obs<G>(mslot, c, a.terminal_obs + (size_t)w * m.nobs, b.time + w, bad);
      if (!SOLO && reset_needs_physics(t)) {
        // the reset runs an env step of its own (reference-state initialisation): done by a full-capacity pass, which also
        // writes the first observation of the new episode; the terminal state is stored as it is and the world is handed
        // over after that store (end of this function)
        deferred_reset = io;
      } else {
        task_reset<G, RMAX, SOLO>(mslot, t, c, b, w, ti, tf, ptarget);
        if (c.lane == 0) b.time[w] = 0.f;
        phase_tree_forward<G>(mslot, c, false);
        task_obs<G>(mslot, t, c, ptarget);
      }
    }
    if (io && !deferred_reset) write_obs<G>(mslot, c, a.obs + (size_t)w * m.nobs, b.time + w, bad);
  }
  // status flags
  for (int i = c.lane; i < m.nq; i += G) if (!isfinite(SF(o_qpos)[i])) status |= ST_NONFINITE;
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) status |= c.tile.shfl_xor(status, o);
  if (c.lane == 0) {
    misc[MI_STATUS] = status;
    if (status && io) atomicOr(b.status, status);
    if ((a.mode == MODE_ENV_STEP || a.mode == MODE_REDO) && b.work) b.work[w] = io ? 0x7ffe - min(misc[MI_NEFC], 0x7ffe) : 0x7fff;      // heavy worlds first (the partial last wave of CTAs gets the light ones), padding worlds last
  }
  store_world<G>(mslot, c, b, w, true);
  if (deferred_reset) {
    c.tile.sync();
    if (c.lane == 0) {
#ifndef MYO_EMUL
      __threadfence();
#endif
      redo_push(b, w, REDO_RESET);
    }
  }
  if (b.dump && (a.mode == MODE_FORWARD || a.mode == MODE_MJ_STEP)) {
    c.tile.sync();
    float* out = b.dump + (size_t)w * m.scratch_words;
    for (int i = c.lane; i < m.scratch_words; i += G) out[i] = c.sp()[i];
  }
}

// every kernel begins by staging the model's table block into shared memory (see myo_dev.hpp)
__device__ void stage_tables(const DevModel& m) {
  float4* dst = reinterpret_cast<float4*>(MYO_SMEM_WORDS);
  const float4* src = reinterpret_cast<const float4*>(m.g_tables);
#ifdef MYO_EMUL   // emulated threads run one after the other: each one stages the whole block
  for (int i = 0; i < m.tab_words / 4; i++) dst[i] = src[i];
#else
  for (int i = threadIdx.x; i < m.tab_words / 4; i += blockDim.x) dst[i] = src[i];
  __syncthreads();
#endif
}

// the full-capacity pass of the fast kernel goes through one noinline call, so that its (large, cold) code does not take part
// in the register allocation of the kernel body around the fast path
template <int G>
MYO_PHASE void heavy_world(int mslot_full, const myo_task_cfg& t, const BatchPtrs& b, const StepArgs& a, int soff, int entry) {
  cg::thread_block block = cg::this_thread_block();
  cg::thread_block_tile<G> tile = cg::tiled_partition<G>(block);
  Ctx<G, 1> ch(tile);
  ch.soff = soff;
  StepArgs ar = a;
  ar.mode = MODE_REDO;
  run_world<G, kSoloRowsPerLane, true>(mslot_full, t, b, ar, ch, entry & 0x3fffffff, entry >> 30);
}

#ifndef MYO_EMUL
MYO_DI int ld_volatile(const int* p) { return *reinterpret_cast<const volatile int*>(p); }
#endif

template <int G>
__global__ void __launch_bounds__(kThreads) world_kernel(int mslot, int mslot_full, const __grid_constant__ myo_task_cfg t,
                                                        const __grid_constant__ BatchPtrs b, const __grid_constant__ StepArgs a) {
  MYO_M
  stage_tables(m);
  cg::thread_block block = cg::this_thread_block();
  cg::thread_block_tile<G> tile = cg::tiled_partition<G>(block);
  Ctx<G, 0> c(tile);
  const int wpc = blockDim.x / G;
  const int tid = threadIdx.x / G;
  c.soff = m.tab_words + tid * m.scratch_words;
  constexpr int RMAX = kFastRows / G > 0 ? kFastRows / G : 1;
#ifndef MYO_EMUL
  if (b.sched && a.mode == MODE_ENV_STEP) {
    // Env step with dynamic scheduling: groups of wpc worlds (in the sorted order: heavy worlds first) are fetched from a
    // global counter; when none is left the CTA serves the redo list - worlds that outgrew the fast layout, resets that run
    // physics - with the full-capacity layout in its own shared memory. Overflows come from the heavy groups at the front,
    // so the list is complete long before the last (light) groups finish and the redone worlds fill the slack of the last wave.
    __shared__ int s_pick[3];
    const int ngroups = b.n_alloc / wpc;
    const DevModel& mf = c_models[mslot_full];
    bool exhausted = false;      // (thread 0) no group of worlds is left in the queue
    for (;;) {
      if (threadIdx.x == 0) {
        // what next: a full-capacity batch as soon as enough redo entries wait (so that work spreads over the whole launch and
        // not into a tail), else the next group of worlds, else - queue empty - whatever the redo list still holds
        int kind = 2, idx = 0, cnt = 0;
        for (;;) {
          if (b.redo_list) {
            const int avail = ld_volatile(b.redo_count), taken = ld_volatile(&b.sched[2]);
            if (taken < avail && (exhausted || avail - taken >= b.heavy_per_cta)) {
              const int want = min(taken + b.heavy_per_cta, avail);
              if (atomicCAS(&b.sched[2], taken, want) == taken) { kind = 1; idx = taken; cnt = want - taken; break; }
              continue;
            }
          }
          if (!exhausted) {
            const int g = atomicAdd(&b.sched[0], 1);
            if (g < ngroups) { kind = 0; idx = g; break; }
            exhausted = true;
            continue;
          }
          // Queue empty and no redo entry waiting: done. Nothing can be orphaned - an entry is pushed by a CTA while it works on
          // a group, and that CTA comes back here afterwards, where the entry is either already taken by someone or taken now -
          // so nobody has to wait for the other CTAs, and a kernel queued behind this one can start on the freed SMs.
          break;
        }
        s_pick[0] = kind; s_pick[1] = idx; s_pick[2] = cnt;
      }
      __syncthreads();
      const int kind = s_pick[0], idx = s_pick[1], cnt = s_pick[2];
      __syncthreads();
      if (kind == 2) break;
      if (kind == 0) {
        const int slot = idx * wpc + tid;
        run_world<G, RMAX, false>(mslot, t, b, a, c, b.order ? b.order[slot] : slot, 0);
      } else if (tid < cnt) {
        int e;
        while ((e = ld_volatile(b.redo_list + idx + tid)) < 0) __nanosleep(200);      // reserved but not written yet
        __threadfence();
        heavy_world<G>(mslot_full, t, b, a, m.tab_words + tid * mf.scratch_words, e);
      }
    }
    return;
  }
#endif
  // state arrays are padded to a multiple of wpc worlds, so every tile of a CTA runs the same number of
  // iterations (the phases contain CTA-wide barriers); padding worlds are stepped but have no I/O
  for (int slot = blockIdx.x * wpc + tid; slot < b.n_alloc; slot += gridDim.x * wpc) {
    const int w = b.order ? b.order[slot] : slot;
    run_world<G, RMAX, false>(mslot, t, b, a, c, w, 0);
    c.tile.sync();
  }
}

// Full-capacity kernel: ONE world per CTA (a single tile), scratch laid out with MuJoCo's own capacities (nconmax contacts,
// njmax rows). It serves the redo list of an env step (worlds that outgrew the fast layout; resets that run physics), explicit
// resets of tasks whose reset runs physics, and the parity hooks (forward / mj_step with stage dumps).
template <int G>
__global__ void __launch_bounds__(G < 32 ? 32 : G) solo_kernel(int mslot, const __grid_constant__ myo_task_cfg t,
                                                             const __grid_constant__ BatchPtrs b, const __grid_constant__ StepArgs a) {
  MYO_M
  const int count = a.mode == MODE_REDO ? *b.redo_count : b.n_worlds;
  if ((int)blockIdx.x >= count) return;
  stage_tables(m);
  cg::thread_block block = cg::this_thread_block();
  cg::thread_block_tile<G> tile = cg::tiled_partition<G>(block);
  Ctx<G, 1> c(tile);
  c.soff = m.tab_words;
  constexpr int RMAX = G == 1 ? kSoloRowsPerLane * 32 : kSoloRowsPerLane;
  for (int i = blockIdx.x; i < count; i += gridDim.x) {
    int w = i, kind = 0;
    if (a.mode == MODE_REDO) { const int e = b.redo_list[i]; w = e & 0x3fffffff; kind = e >> 30; }
    run_world<G, RMAX, true>(mslot, t, b, a, c, w, kind);
    c.tile.sync();
  }
}

// ---- stage extraction: factored scratch -> dense arrays, one thread per world ------------------
__global__ void extract_kernel(const __grid_constant__ DevModel m, const float* dump, int n, int stage, void* outv, int width) {
  stage_tables(m);
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n) return;
  const float* s = dump + (size_t)w * m.scratch_words;
  const int* si = reinterpret_cast<const int*>(s);
  float* of = reinterpret_cast<float*>(outv) + (size_t)w * width;
  int* oi = reinterpret_cast<int*>(outv) + (size_t)w * width;
  const int* misc = si + m.o_misc;
  const int nlim = misc[MI_NLIM], ncon = misc[MI_NCON], nefc = misc[MI_NEFC];
  auto copyf = [&](int off, int cnt) { for (int i = 0; i < cnt; i++) of[i] = s[off + i]; };
  switch (stage) {
    case MYO_STAGE_XPOS: copyf(m.o_xpos, 3 * m.nbody); break;
    case MYO_STAGE_XMAT: copyf(m.o_xmat, 9 * m.nbody); break;
    case MYO_STAGE_SITE_XPOS:
      for (int k = 0; k < m.nsite; k++) site_world(m, s, s + m.o_wparam, k, of + 3 * k);
      break;
    case MYO_STAGE_TEN_LENGTH: copyf(m.o_tenL, m.ntendon); break;
    case MYO_STAGE_TEN_J:
      for (int i = 0; i < m.ntendon * m.nv; i++) of[i] = 0.f;
      for (int t = 0; t < m.ntendon; t++)
        for (int e = 0; e < m.t_ndof[t]; e++) of[t * m.nv + m.t_dof[t * KT + e]] = s[m.o_tenJ + t * KT + e];
      break;
    case MYO_STAGE_QM:
      for (int i = 0; i < m.nv * m.nv; i++) of[i] = 0.f;
      for (int i = 0; i < m.nv; i++) {
        int adr = m.d_Madr[i], j = i;
        while (j >= 0) { of[i * m.nv + j] = of[j * m.nv + i] = s[m.o_M + adr++]; j = m.d_parent[j]; }
      }
      break;
    case MYO_STAGE_QFRC_BIAS: copyf(m.o_bias, m.nv); break;
    case MYO_STAGE_QFRC_PASSIVE: copyf(m.o_passive, m.nv); break;
    case MYO_STAGE_QFRC_ACTUATOR: copyf(m.o_qact, m.nv); break;
    case MYO_STAGE_ACT_FORCE: copyf(m.o_actF, m.nu); break;
    case MYO_STAGE_QACC_SMOOTH: copyf(m.o_qaccs, m.nv); break;
    case MYO_STAGE_QACC: copyf(m.o_qacc, m.nv); break;
    case MYO_STAGE_QFRC_CONSTRAINT: copyf(m.o_qcon, m.nv); break;
    case MYO_STAGE_ACT_DOT: copyf(m.o_actdot, m.na); break;
    case MYO_STAGE_NCON: oi[0] = ncon; break;
    case MYO_STAGE_NEFC: oi[0] = nefc; break;
    case MYO_STAGE_SOLVER_ITER: oi[0] = misc[MI_ITER]; break;
    case MYO_STAGE_STATUS: oi[0] = misc[MI_STATUS]; break;
    case MYO_STAGE_CONTACT_GEOMS:
      for (int k = 0; k < m.ncon_max; k++) {
        oi[2 * k] = k < ncon ? si[m.o_con + k * CON_WORDS + C_G1] : -1;
        oi[2 * k + 1] = k < ncon ? si[m.o_con + k * CON_WORDS + C_G2] : -1;
      }
      break;
    case MYO_STAGE_CONTACT_DIST:
      for (int k = 0; k < m.ncon_max; k++) of[k] = k < ncon ? s[m.o_con + k * CON_WORDS + C_DIST] : 0.f;
      break;
    case MYO_STAGE_EFC_TYPE_ID:
    case MYO_STAGE_EFC_J:
    case MYO_STAGE_EFC_AREF:
    case MYO_STAGE_EFC_D:
    case MYO_STAGE_EFC_FORCE: {
      const int per = stage == MYO_STAGE_EFC_J ? m.nv : (stage == MYO_STAGE_EFC_TYPE_ID ? 2 : 1);
      for (int i = 0; i < m.nefc_max * per; i++) { if (stage == MYO_STAGE_EFC_TYPE_ID) oi[i] = -1; else of[i] = 0.f; }
      for (int r = 0; r < nefc; r++) {
        const float* row = s + m.o_row + r * ROW_WORDS;
        if (stage == MYO_STAGE_EFC_AREF) of[r] = row[R_AREF];
        else if (stage == MYO_STAGE_EFC_D) of[r] = row[R_D];
        else if (stage == MYO_STAGE_EFC_FORCE) of[r] = row[R_JAR] < 0.f ? -row[R_D] * row[R_JAR] : 0.f;
      }
      if (stage == MYO_STAGE_EFC_TYPE_ID || stage == MYO_STAGE_EFC_J) {
        for (int r = 0; r < nlim; r++) {
          const float* lr = s + m.o_lim + r * LIM_WORDS; const int* li = reinterpret_cast<const int*>(lr);
          if (stage == MYO_STAGE_EFC_TYPE_ID) { oi[2 * r] = li[L_KIND]; oi[2 * r + 1] = li[L_ID]; }
          else for (int e = 0; e < li[L_NSUP]; e++) of[r * m.nv + lim_idx(li, e)] = lim_J(s, lr, li, e);
        }
        for (int k = 0; k < ncon; k++) {
          const float* cr = s + m.o_con + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
          const int row0 = ci[C_ROW0];
          if (row0 < 0) continue;
          const int nr = ci[C_DIM] == 1 ? 1 : 4;
          for (int q = 0; q < nr; q++) {
            const int r = row0 + q;
            if (stage == MYO_STAGE_EFC_TYPE_ID) { oi[2 * r] = nr == 1 ? EFC_CONTACT_FRICTIONLESS : EFC_CONTACT_PYRAMIDAL; oi[2 * r + 1] = k; }
            else {
              const float mu = cr[C_MU];
              for (int e = 0; e < ci[C_NSUP]; e++) {
                float jn, jt1, jt2;
                const int dof = contact_entry(m, s, cr, ci, e, &jn, &jt1, &jt2);
                float v = jn;
                if (nr == 4) v += ((q & 1) ? -mu : mu) * ((q < 2) ? jt1 : jt2);
                of[r * m.nv + dof] = v;
              }
            }
          }
        }
      }
    } break;
    default: break;
  }
}

__global__ void init_worlds_kernel(const __grid_constant__ DevModel m, BatchPtrs b, int fixed_task) {
  stage_tables(m);
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= b.n_alloc) return;
  for (int i = 0; i < m.nq4; i++) { b.qpos[(size_t)w * m.nq4 + i] = i < m.nq ? m.init_qpos[i] : 0.f; b.pose_target[(size_t)w * m.nq4 + i] = 0.f; }
  for (int i = 0; i < m.nv4; i++) { b.qvel[(size_t)w * m.nv4 + i] = 0.f; b.warm[(size_t)w * m.nv4 + i] = 0.f; }
  for (int i = 0; i < m.na4; i++) b.act[(size_t)w * m.na4 + i] = 0.f;
  for (int i = 0; i < m.nparam4; i++) b.wparam[(size_t)w * m.nparam4 + i] = m.param0[i];
  b.time[w] = 0.f;
  int* ti = b.task_i + (size_t)w * TI_WORDS;
  ti[TI_ELAPSED] = 0; ti[TI_EPISODE] = 0; ti[TI_TASK] = fixed_task; ti[TI_FLAGS] = 0;
  float* tf = b.task_f + (size_t)w * TF_WORDS;
  for (int k = 0; k < TF_WORDS; k++) tf[k] = 0.f;
  tf[TF_ANGLE1] = 0.25f * kPi; tf[TF_ANGLE2] = 0.25f * kPi - kPi; tf[TF_XR] = 0.025f; tf[TF_YR] = 0.028f; tf[TF_PERIOD] = 5.f;
}

// padded [n][w4] <-> packed [n][w] row copies for set_state / get_state / params
__global__ void repack_kernel(float* dst, int dst_stride, int dst_off, const float* src, int src_stride, int src_off, int width, int n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * width) return;
  const int w = (int)(i / width), k = (int)(i % width);
  dst[(size_t)w * dst_stride + dst_off + k] = src[(size_t)w * src_stride + src_off + k];
}

}  // namespace myo

// ------------------------------------------------------------------------------------------------
// The redo of worlds the fast layout cannot finish runs inside the fast kernel (dynamic scheduling) on the device; the host
// emulation has no such scheduler and runs it as a separate pass of the solo kernel.
#ifdef MYO_EMUL
constexpr bool kDynSched = false;
#else
constexpr bool kDynSched = true;
#endif

struct myo_batch {
  myo::PackedModel pm;
  myo_task_cfg cfg;
  myo::BatchPtrs p{};
  int device = 0, n = 0, slot = -1, slot_full = -1;
  int grid = 0, threads = myo::kThreads, smem = 0, regs = 0, wpc = 0, tab_bytes = 0;
  int solo_grid = 0, solo_smem = 0, solo_regs = 0;
  bool use_redo = false;       // worlds the fast layout cannot finish are redone with full capacities within the same env step
  int64_t launches = 0;
  std::vector<void*> allocs;
  // world grouping: after every env step the worlds are sorted by the constraint rows of their last substep, and the next
  // step walks them in that order, so the worlds that share a CTA (and its phase barriers) carry similar loads
  bool sort_worlds = false;
  int *order[2] = {nullptr, nullptr}, *iota = nullptr, *keys_out = nullptr;
  void* sort_tmp = nullptr;
  size_t sort_tmp_bytes = 0;
  int cur_order = -1;      // index of the order the next step uses (-1: identity)
};

namespace {

using namespace myo;

#define CK(call)                                                                                    \
  do {                                                                                              \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess) {                                                                        \
      set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                               \
      return MYO_E_CUDA;                                                                            \
    }                                                                                               \
  } while (0)

template <class T> int dev_alloc(myo_batch* b, T** p, size_t count) {
  void* q = nullptr;
  CK(cudaMalloc(&q, std::max<size_t>(count, 4) * sizeof(T)));
  CK(cudaMemset(q, 0, std::max<size_t>(count, 4) * sizeof(T)));
  b->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return MYO_OK;
}

// constant-memory model slots, per device
std::mutex g_slot_mu;
bool g_slot_busy[64][kModelSlots];
int acquire_slot(myo_batch* b) {      // two descriptors per batch: the fast layout and the full-capacity one
  std::lock_guard<std::mutex> lk(g_slot_mu);
  const int d = b->device & 63;
  int got[2] = {-1, -1}, k = 0;
  for (int s = 0; s < kModelSlots && k < 2; s++)
    if (!g_slot_busy[d][s]) got[k++] = s;
  if (k < 2) { set_error("too many live batches on one device (16 model slots in constant memory, two per batch)"); return MYO_E_LIMIT; }
  g_slot_busy[d][got[0]] = g_slot_busy[d][got[1]] = true;
  b->slot = got[0]; b->slot_full = got[1];
  return MYO_OK;
}
void release_slot(myo_batch* b) {
  std::lock_guard<std::mutex> lk(g_slot_mu);
  if (b->slot >= 0) g_slot_busy[b->device & 63][b->slot] = false;
  if (b->slot_full >= 0) g_slot_busy[b->device & 63][b->slot_full] = false;
  b->slot = b->slot_full = -1;
}
int upload_slot(myo_batch* b) {
#ifdef MYO_EMUL
  c_models[b->slot] = b->pm.dm;
  c_models[b->slot_full] = b->pm.dm_full;
#else
  CK(cudaMemcpyToSymbol(c_models, &b->pm.dm, sizeof(DevModel), (size_t)b->slot * sizeof(DevModel)));
  CK(cudaMemcpyToSymbol(c_models, &b->pm.dm_full, sizeof(DevModel), (size_t)b->slot_full * sizeof(DevModel)));
#endif
  return MYO_OK;
}

template <int G> int launch_world(myo_batch* b, const StepArgs& a, cudaStream_t st) {
  MYO_LAUNCH(world_kernel<G>, b->grid, b->threads, b->smem, st, b->slot, b->slot_full, b->cfg, b->p, a);
  b->launches++;
  CK(cudaGetLastError());
  return MYO_OK;
}
template <int G> int launch_solo(myo_batch* b, const StepArgs& a, cudaStream_t st) {
  const int want = a.mode == MODE_REDO ? b->solo_grid : std::min(b->n, b->solo_grid);
  MYO_LAUNCH(solo_kernel<G>, std::max(1, want), G, b->solo_smem, st, b->slot_full, b->cfg, b->p, a);
  b->launches++;
  CK(cudaGetLastError());
  return MYO_OK;
}
// fast kernel (many worlds per CTA, fast capacities)
int launch(myo_batch* b, const StepArgs& a, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CK(cudaSetDevice(b->device));
  int rc = MYO_OK;
  MYO_LANES_CASES(b, launch_world, b, a, st)
  return rc;
}
// full-capacity kernel (one world per CTA)
int launch_full(myo_batch* b, const StepArgs& a, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CK(cudaSetDevice(b->device));
  int rc = MYO_OK;
  MYO_LANES_CASES(b, launch_solo, b, a, st)
  return rc;
}
template <int G> int configure(myo_batch* b) {
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, world_kernel<G>));
  b->regs = fa.numRegs;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, b->device));
  const size_t world_bytes = (size_t)b->pm.dm.scratch_words * sizeof(float);
  const size_t tab_bytes = (size_t)b->pm.dm.tab_words * sizeof(float);
  if (tab_bytes + world_bytes > prop.sharedMemPerBlockOptin) { set_error("model tables + one world exceed shared memory per CTA"); return MYO_E_LIMIT; }
  const size_t max_smem = prop.sharedMemPerBlockOptin - tab_bytes;
  // worlds per CTA: fill the SM's shared memory with as few CTAs as keep threads <= kThreads
  int wpc = kThreads / G;
  while (wpc > 1 && wpc * world_bytes > max_smem) wpc--;
  if (wpc * world_bytes > max_smem) { set_error("one world's scratch exceeds shared memory per CTA"); return MYO_E_LIMIT; }
  // a batch smaller than one CTA steps no padding worlds beside its own; the CTA keeps room for one full-capacity world (redo)
  wpc = std::min(wpc, b->n);
  const size_t full_bytes = (size_t)b->pm.dm_full.scratch_words * sizeof(float);
  if (tab_bytes + full_bytes > prop.sharedMemPerBlockOptin) { set_error("model tables + one full-capacity world exceed shared memory per CTA"); return MYO_E_LIMIT; }
  b->wpc = wpc;
  b->tab_bytes = (int)tab_bytes;
  CK(cudaFuncSetAttribute(init_worlds_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tab_bytes));
  CK(cudaFuncSetAttribute(extract_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tab_bytes));
  b->threads = wpc * G;
  b->smem = (int)(tab_bytes + std::max(wpc * world_bytes, full_bytes));
  CK(cudaFuncSetAttribute(world_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, b->smem));
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, world_kernel<G>, b->threads, b->smem));
  if (per_sm < 1) per_sm = 1;
  const int need = (b->n + wpc - 1) / wpc;
  b->grid = std::max(1, std::min(need, prop.multiProcessorCount * per_sm));
  // full-capacity kernel: one world per CTA
  b->solo_smem = (int)(tab_bytes + full_bytes);
  CK(cudaFuncSetAttribute(solo_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, b->solo_smem));
  cudaFuncAttributes fs;
  CK(cudaFuncGetAttributes(&fs, solo_kernel<G>));
  b->solo_regs = fs.numRegs;
  int solo_per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&solo_per_sm, solo_kernel<G>, G, b->solo_smem));
  b->solo_grid = prop.multiProcessorCount * std::max(1, solo_per_sm);
  return MYO_OK;
}

}  // namespace

extern "C" {

int myo_task_cfg_default(const myo_model* mh, int kind, myo_task_cfg* cfg) {
  if (!mh || !cfg) { myo::set_error("null argument"); return MYO_E_ARG; }
  const myo::Model& m = myo_model_host(mh);
  memset(cfg, 0, sizeof *cfg);
  cfg->kind = kind; cfg->frame_skip = 10; cfg->max_episode_steps = kind == MYO_TASK_BAODING ? 200 : 100;
  cfg->normalize_act = 1; cfg->auto_reset = 1;
  cfg->solver_iterations = 0; cfg->solver_tolerance = 0.f;
  cfg->weight_body = -1; cfg->weight_geom = -1;
  if (kind == MYO_TASK_BAODING) {
    // BaodingEnvV1.DEFAULT_RWD_KEYS_AND_WEIGHTS (pos_dist 5/5, alive 0, act_reg 0), /root/reference/src/envs/baoding.py:16-22
    cfg->rwd_weight[0] = 5.f; cfg->rwd_weight[1] = 5.f;
    cfg->drop_th = 1.25f; cfg->proximity_th = 0.015f;
    cfg->goal_time_period[0] = cfg->goal_time_period[1] = 5.f;
    cfg->goal_xrange[0] = cfg->goal_xrange[1] = 0.025f; cfg->goal_yrange[0] = cfg->goal_yrange[1] = 0.028f;
    cfg->obj_size_range[0] = 0.018f; cfg->obj_size_range[1] = 0.024f;
    cfg->obj_mass_range[0] = 0.030f; cfg->obj_mass_range[1] = 0.300f;
    cfg->obj_friction_change[0] = 0.2f; cfg->obj_friction_change[1] = 0.001f; cfg->obj_friction_change[2] = 0.00002f;
    cfg->task_choice_random = 0; cfg->fixed_task = MYO_BAODING_CCW;
    cfg->center_pos[0] = -0.0125f; cfg->center_pos[1] = -0.07f;
    cfg->randomize_physics = 1;
    const char* bn[2] = {"ball1", "ball2"}; const char* sn[2] = {"ball1_site", "ball2_site"};
    const char* tn[2] = {"target1_site", "target2_site"};
    for (int k = 0; k < 2; k++) {
      cfg->ball_body[k] = m.name2id("body", bn[k]); cfg->ball_geom[k] = m.name2id("geom", bn[k]);
      cfg->ball_site[k] = m.name2id("site", sn[k]); cfg->target_site[k] = m.name2id("site", tn[k]);
      if (cfg->ball_body[k] < 0 || cfg->ball_geom[k] < 0 || cfg->ball_site[k] < 0 || cfg->target_site[k] < 0) {
        myo::set_error("model lacks the baoding names ball{1,2}, ball{1,2}_site, target{1,2}_site");
        return MYO_E_ARG;
      }
      const int j = m.i("body_jntadr")[cfg->ball_body[k]];
      cfg->ball_qposadr[k] = m.i("jnt_qposadr")[j]; cfg->ball_dofadr[k] = m.i("jnt_dofadr")[j];
    }
    cfg->n_ovr_body = 2; cfg->ovr_body[0] = cfg->ball_body[0]; cfg->ovr_body[1] = cfg->ball_body[1];
    cfg->n_ovr_geom = 2; cfg->ovr_geom[0] = cfg->ball_geom[0]; cfg->ovr_geom[1] = cfg->ball_geom[1];
    cfg->n_ovr_site = 2; cfg->ovr_site[0] = cfg->target_site[0]; cfg->ovr_site[1] = cfg->target_site[1];
  } else if (kind == MYO_TASK_REORIENT) {
    // ReorientEnvV0.DEFAULT_RWD_KEYS_AND_WEIGHTS (pos_dist 100, rot_dist 1) and CustomReorientEnv._setup's defaults
    // (/root/reference/src/envs/reorient.py:58-125); frame_skip 5, horizon 150 come from the registrations (src/envs/__init__.py:26-55)
    cfg->frame_skip = 5; cfg->max_episode_steps = 150;
    cfg->rwd_weight[0] = 100.f; cfg->rwd_weight[1] = 1.f;
    cfg->goal_pos[0] = cfg->goal_pos[1] = 0.f; cfg->goal_rot[0] = cfg->goal_rot[1] = 0.785f;
    cfg->pos_th = 0.025f; cfg->rot_th = 0.262f; cfg->drop_th = 0.2f;
    cfg->object_body = m.name2id("body", "Object"); cfg->goal_body = m.name2id("body", "target");
    cfg->object_site = m.name2id("site", "object_o"); cfg->goal_site = m.name2id("site", "target_o");
    if (cfg->object_body < 0 || cfg->goal_body < 0 || cfg->object_site < 0 || cfg->goal_site < 0) {
      myo::set_error("model lacks the reorient names: bodies Object / target, sites object_o / target_o");
      return MYO_E_ARG;
    }
    const int ob = cfg->object_body, gb = cfg->goal_body;
    cfg->object_geom0 = m.i("body_geomadr")[ob]; cfg->object_ngeom = m.i("body_geomnum")[ob];
    if (cfg->object_ngeom < 3 || cfg->object_ngeom > MYO_MAX_OVERRIDE) {
      myo::set_error("the Object body must carry 3 or 4 geoms (the reference's reset scales the last three as boxes)");
      return MYO_E_LIMIT;
    }
    const int j = m.i("body_jntadr")[ob];
    if (m.i("body_jntnum")[ob] != 1 || m.i("jnt_type")[j] != 0) { myo::set_error("the Object body must hang on a free joint"); return MYO_E_ARG; }
    cfg->object_qposadr = m.i("jnt_qposadr")[j]; cfg->object_dofadr = m.i("jnt_dofadr")[j];
    const double* sq = m.d("site_quat");
    for (int sid : {cfg->object_site, cfg->goal_site})
      if (sq[4 * sid] < 1.0 - 1e-9) { myo::set_error("object_o / target_o must share their bodies' frames (identity site_quat)"); return MYO_E_UNSUPPORTED; }
    if (m.i("body_parentid")[gb] != 0 || m.i("body_jntnum")[gb] != 0) { myo::set_error("the target body must be fixed to the world"); return MYO_E_UNSUPPORTED; }
    // goal_init_pos = site_xpos[target_o], goal_obj_offset = target_o - object_o, both at the model's qpos0 (the env reads them
    // right after MujocoEnv.__init__'s sim.forward(), reorient.py:88-92)
    const double* bp = m.d("body_pos") + 3 * gb; const double* bq = m.d("body_quat") + 4 * gb;
    const double* sp = m.d("site_pos"); const double* q0 = m.d("qpos0") + cfg->object_qposadr;
    auto rot = [](const double* q, const double* v, double* o) {
      const double w = q[0], x = q[1], y = q[2], z = q[3];
      const double R[9] = {w*w + x*x - y*y - z*z, 2*(x*y - w*z), 2*(x*z + w*y), 2*(x*y + w*z), w*w - x*x + y*y - z*z, 2*(y*z - w*x),
                           2*(x*z - w*y), 2*(y*z + w*x), w*w - x*x - y*y + z*z};
      for (int r = 0; r < 3; r++) o[r] = R[3*r] * v[0] + R[3*r + 1] * v[1] + R[3*r + 2] * v[2];
    };
    double tg[3], oo[3];
    rot(bq, sp + 3 * cfg->goal_site, tg);
    rot(q0 + 3, sp + 3 * cfg->object_site, oo);
    for (int e = 0; e < 3; e++) {
      tg[e] += bp[e]; oo[e] += q0[e];
      cfg->goal_init_pos[e] = (float)tg[e]; cfg->goal_obj_offset[e] = (float)(tg[e] - oo[e]);
    }
    cfg->n_ovr_geom = cfg->object_ngeom;
    for (int k = 0; k < cfg->object_ngeom; k++) {
      cfg->ovr_geom[k] = cfg->object_geom0 + k;
      const double* gp = m.d("geom_pos") + 3 * (cfg->object_geom0 + k);
      if (gp[0] != 0.0 || gp[1] != 0.0 || gp[2] != 0.0) { myo::set_error("die geoms away from the body origin (per-world geom_pos) are not supported"); return MYO_E_UNSUPPORTED; }
    }
    cfg->n_ovr_bodypose = 1; cfg->ovr_bodypose[0] = gb;
  } else if (kind == MYO_TASK_POSE) {
    // PoseEnvV0.DEFAULT_RWD_KEYS_AND_WEIGHTS: pose 1, bonus 4, penalty 50, act_reg 1 (order: pose bonus penalty act_reg)
    cfg->rwd_weight[0] = 1.f; cfg->rwd_weight[1] = 4.f; cfg->rwd_weight[2] = 50.f; cfg->rwd_weight[3] = 1.f;
    cfg->pose_thd = 0.35f; cfg->far_th = 4.f * 3.14159265358979f / 2.f; cfg->target_distance = 1.f;
    cfg->reset_type = 1; cfg->target_type = 1;
    cfg->weight_body = -1; cfg->weight_geom = -1;
  } else if (kind == MYO_TASK_REACH) {
    // ReachEnvV0._setup defaults (far_th .35, reach 1 / bonus 4 / penalty 50) and the myoFingerReach* registrations (frame_skip 5,
    // 200 steps), MyoSuite 1.2.3 [3P-MEM]. Sites: IFtip when the model has it, its target held at the model's site_pos.
    cfg->frame_skip = 5; cfg->max_episode_steps = 200;
    cfg->rwd_weight[0] = 1.f; cfg->rwd_weight[1] = 4.f; cfg->rwd_weight[3] = 50.f;
    const int tip = m.name2id("site", "IFtip"), tgt = m.name2id("site", "IFtip_target");
    if (tip >= 0 && tgt >= 0) {
      cfg->reach_nsite = 1; cfg->reach_tip_site[0] = tip; cfg->reach_target_site[0] = tgt;
      const double* sp = m.d("site_pos") + 3 * tgt;
      for (int e = 0; e < 3; e++) cfg->reach_range[0][0][e] = cfg->reach_range[0][1][e] = (float)sp[e];
    }
    cfg->far_th = 0.35f; cfg->reach_near_th = 0.0125f;
    // first env step after which time > 2 dt, with time summed in fp64 one substep at a time as MuJoCo does
    const double h = m.opt.at("timestep"), dt = h * cfg->frame_skip;
    double time = 0.0;
    int k = 0;
    while (!(time > 2.0 * dt)) { for (int s = 0; s < cfg->frame_skip; s++) time += h; k++; }
    cfg->reach_far_steps = k;
  }
  return MYO_OK;
}

int myo_model_check(const myo_model* mh, char* report, size_t report_len) {
  if (!mh) { myo::set_error("null model"); return MYO_E_ARG; }
  const std::string r = myo::check_model(myo_model_host(mh));
  if (report && report_len) { strncpy(report, r.c_str(), report_len - 1); report[report_len - 1] = 0; }
  if (r.rfind("- ", 0) == 0 || r.find("\n- ") != std::string::npos) { myo::set_error("model is outside the supported subset:\n" + r); return MYO_E_UNSUPPORTED; }
  return MYO_OK;      // "~ " lines, if any, are advisory
}

int myo_batch_create(const myo_model* mh, int n_worlds, int device, const myo_task_cfg* cfg, uint64_t seed, myo_batch** out) {
  if (!mh || !cfg || !out || n_worlds <= 0) { myo::set_error("bad argument to myo_batch_create"); return MYO_E_ARG; }
  if (cfg->kind == MYO_TASK_REACH) {
    if (cfg->reach_nsite > MYO_MAX_OVERRIDE) { myo::set_error("reach: more target sites than MYO_MAX_OVERRIDE"); return MYO_E_LIMIT; }
    const int nsite = myo_model_host(mh).sz("nsite");
    bool ok = cfg->reach_nsite >= 1;
    for (int k = 0; ok && k < cfg->reach_nsite; k++)
      ok = cfg->reach_tip_site[k] >= 0 && cfg->reach_tip_site[k] < nsite && cfg->reach_target_site[k] >= 0 && cfg->reach_target_site[k] < nsite;
    if (!ok) { myo::set_error("reach: needs 1..MYO_MAX_OVERRIDE tip / target sites with valid ids"); return MYO_E_ARG; }
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
    myo::set_error("no CUDA device available (this library has no CPU path)");
    return MYO_E_CUDA;
  }
  myo_batch* b = new myo_batch();
  b->cfg = *cfg; b->device = device; b->n = n_worlds;
  int status = MYO_OK;
  std::string err = myo::pack_model(myo_model_host(mh), *cfg, b->pm, status);
  if (!err.empty()) { delete b; myo::set_error(err); return status; }
  if (cfg->kind == MYO_TASK_POSE && cfg->n_target_jnt > 64) { delete b; myo::set_error("too many target joints"); return MYO_E_LIMIT; }
  auto fail = [&](int code) { myo_batch_destroy(b); return code; };
  if (cudaSetDevice(device) != cudaSuccess) { myo::set_error("cudaSetDevice failed"); return fail(MYO_E_CUDA); }
  const myo::DevModel& dm = b->pm.dm;
  int rc;
  if ((rc = dev_alloc(b, &b->pm.d_tables, b->pm.tables.size()))) return fail(rc);
  if (cudaMemcpy(b->pm.d_tables, b->pm.tables.data(), b->pm.tables.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
    myo::set_error("model upload failed");
    return fail(MYO_E_CUDA);
  }
  b->pm.dm.g_tables = b->pm.d_tables;
  b->pm.dm_full.g_tables = b->pm.d_tables;
  b->pm.dm_full.tab_words = b->pm.dm.tab_words;
  MYO_LANES_CASES(b, configure, b)
  if (rc) return fail(rc);
  if ((rc = acquire_slot(b)) || (rc = upload_slot(b))) return fail(rc);
  b->p.n_worlds = n_worlds; b->p.seed = seed;
  b->p.n_alloc = (n_worlds + b->wpc - 1) / b->wpc * b->wpc;
  const size_t n = (size_t)b->p.n_alloc;
  if ((rc = dev_alloc(b, &b->p.qpos, n * dm.nq4)) || (rc = dev_alloc(b, &b->p.qvel, n * dm.nv4)) ||
      (rc = dev_alloc(b, &b->p.act, n * dm.na4)) || (rc = dev_alloc(b, &b->p.warm, n * dm.nv4)) ||
      (rc = dev_alloc(b, &b->p.time, n)) || (rc = dev_alloc(b, &b->p.wparam, n * dm.nparam4)) ||
      (rc = dev_alloc(b, &b->p.task_f, n * myo::TF_WORDS)) || (rc = dev_alloc(b, &b->p.pose_target, n * dm.nq4)) ||
      (rc = dev_alloc(b, &b->p.task_i, n * myo::TI_WORDS)) || (rc = dev_alloc(b, &b->p.status, 4)))
    return fail(rc);
  b->p.dump = nullptr;
  b->p.order = nullptr; b->p.work = nullptr;
  b->p.redo_list = nullptr; b->p.redo_count = nullptr;
  {
    // the full-capacity pass after every env step is needed when the fast layout is smaller than MuJoCo's capacities or
    // when resets run physics
    const myo::DevModel& df = b->pm.dm_full;
    b->use_redo = df.ncon_max > dm.ncon_max || df.nlim_max > dm.nlim_max || df.nefc_max > dm.nefc_max || myo::reset_needs_physics(*cfg);
    if ((rc = dev_alloc(b, &b->p.redo_list, n)) || (rc = dev_alloc(b, &b->p.redo_count, 4)) || (rc = dev_alloc(b, &b->p.sched, 4))) return fail(rc);
    if (!b->use_redo) b->p.redo_list = nullptr;
    b->p.heavy_per_cta = std::max(1, std::min(b->wpc, (int)((b->smem - b->tab_bytes) / ((size_t)df.scratch_words * sizeof(float)))));
    if (!kDynSched) b->p.sched = nullptr;
  }
#ifndef MYO_EMUL
  {
    b->sort_worlds = b->p.n_alloc >= 4 * b->wpc * 148;      // worth it only when every SM sees several groups
    if (b->sort_worlds) {
      if ((rc = dev_alloc(b, &b->p.work, n)) || (rc = dev_alloc(b, &b->order[0], n)) || (rc = dev_alloc(b, &b->order[1], n)) ||
          (rc = dev_alloc(b, &b->iota, n)) || (rc = dev_alloc(b, &b->keys_out, n)))
        return fail(rc);
      std::vector<int> io(n);
      for (size_t i = 0; i < n; i++) io[i] = (int)i;
      if (cudaMemcpy(b->iota, io.data(), n * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) { myo::set_error("cudaMemcpy(iota) failed"); return fail(MYO_E_CUDA); }
      cub::DeviceRadixSort::SortPairs(nullptr, b->sort_tmp_bytes, b->p.work, b->keys_out, b->iota, b->order[0], (int)n, 0, 15);
      char* tmp = nullptr;
      if ((rc = dev_alloc(b, &tmp, b->sort_tmp_bytes))) return fail(rc);
      b->sort_tmp = tmp;
    }
  }
#endif
  MYO_LAUNCH(myo::init_worlds_kernel, (b->p.n_alloc + 127) / 128, 128, b->tab_bytes, (cudaStream_t)0, dm, b->p, cfg->fixed_task);
  b->launches++;
  if (cudaDeviceSynchronize() != cudaSuccess) { myo::set_error("world initialisation failed"); return fail(MYO_E_CUDA); }
  *out = b;
  return MYO_OK;
}

void myo_batch_destroy(myo_batch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  for (void* p : b->allocs) cudaFree(p);
  release_slot(b);
  delete b;
}

int myo_batch_dims(const myo_batch* b, int* n_worlds, int* nq, int* nv, int* na, int* nu, int* nobs, int* n_param) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  const myo::DevModel& d = b->pm.dm;
  if (n_worlds) *n_worlds = b->n;
  if (nq) *nq = d.nq;
  if (nv) *nv = d.nv;
  if (na) *na = d.na;
  if (nu) *nu = d.nu;
  if (nobs) *nobs = d.nobs;
  if (n_param) *n_param = d.nparam;
  return MYO_OK;
}

int myo_batch_launch_info(const myo_batch* b, int* lanes_per_world, int* worlds_per_cta, int* smem_bytes, int* regs_per_thread) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  if (lanes_per_world) *lanes_per_world = b->pm.lanes;
  if (worlds_per_cta) *worlds_per_cta = b->wpc;
  if (smem_bytes) *smem_bytes = b->smem;
  if (regs_per_thread) *regs_per_thread = b->regs;
  return MYO_OK;
}

int myo_batch_reset(myo_batch* b, const uint8_t* mask_dev, float* obs_dev, void* stream) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  myo::StepArgs a{};
  a.mode = myo::MODE_RESET; a.mask = mask_dev; a.obs = obs_dev;
  // a reset that runs physics (reference-state initialisation) is the full-capacity kernel's job
  return myo::reset_needs_physics(b->cfg) ? launch_full(b, a, stream) : launch(b, a, stream);
}

int myo_batch_step(myo_batch* b, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
                   uint8_t* truncated_dev, float* terminal_obs_dev, float* info_dev, void* stream) {
  if (!b || !actions_dev || !obs_dev || !reward_dev || !done_dev) { myo::set_error("null argument to myo_batch_step"); return MYO_E_ARG; }
  myo::StepArgs a{};
  a.mode = myo::MODE_ENV_STEP; a.nsub = b->cfg.frame_skip > 0 ? b->cfg.frame_skip : 1;
  a.in = actions_dev; a.obs = obs_dev; a.reward = reward_dev; a.done = done_dev; a.truncated = truncated_dev;
  a.terminal_obs = terminal_obs_dev; a.info = info_dev;
  b->p.order = (b->sort_worlds && b->cur_order >= 0) ? b->order[b->cur_order] : nullptr;
  cudaStream_t st_ = static_cast<cudaStream_t>(stream);
  if (b->use_redo) {
    CK(cudaMemsetAsync(b->p.redo_count, 0, sizeof(int), st_));
    if (kDynSched) CK(cudaMemsetAsync(b->p.redo_list, 0xFF, (size_t)b->p.n_alloc * sizeof(int), st_));
  }
  if (kDynSched) CK(cudaMemsetAsync(b->p.sched, 0, 4 * sizeof(int), st_));
  int rc = launch(b, a, stream);
  b->p.order = nullptr;
  if (!rc && b->use_redo && !kDynSched) {      // worlds the fast kernel could not finish: same step, full capacities, one world per CTA
    a.mode = myo::MODE_REDO;
    rc = launch_full(b, a, stream);
  }
  if (rc || !b->sort_worlds) return rc;
#ifndef MYO_EMUL
  // grouping for the next step: stable radix sort of (rows of the last substep, world); keys fit 15 bits
  const int nxt = b->cur_order == 0 ? 1 : 0;
  if (cub::DeviceRadixSort::SortPairs(b->sort_tmp, b->sort_tmp_bytes, b->p.work, b->keys_out, b->iota, b->order[nxt], b->p.n_alloc, 0, 15,
                                      static_cast<cudaStream_t>(stream)) != cudaSuccess) {
    myo::set_error("world grouping sort failed");
    return MYO_E_CUDA;
  }
  b->launches++;
  b->cur_order = nxt;
#endif
  return MYO_OK;
}

static int ensure_dump(myo_batch* b) {      // the parity hooks run in the full-capacity layout
  if (b->p.dump) return MYO_OK;
  return dev_alloc(b, &b->p.dump, (size_t)b->p.n_alloc * b->pm.dm_full.scratch_words);
}

int myo_batch_mj_step(myo_batch* b, const float* ctrl_dev, int nsub, void* stream) {
  if (!b || nsub < 0) { myo::set_error("bad argument to myo_batch_mj_step"); return MYO_E_ARG; }
  int rc = ensure_dump(b);
  if (rc) return rc;
  myo::StepArgs a{};
  a.mode = myo::MODE_MJ_STEP; a.nsub = nsub; a.in = ctrl_dev;
  return launch_full(b, a, stream);
}

int myo_batch_forward(myo_batch* b, const float* ctrl_dev, void* stream) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  int rc = ensure_dump(b);
  if (rc) return rc;
  myo::StepArgs a{};
  a.mode = myo::MODE_FORWARD; a.in = ctrl_dev;
  return launch_full(b, a, stream);
}

int myo_batch_get_obs(myo_batch* b, float* obs_dev, void* stream) {
  if (!b || !obs_dev) { myo::set_error("null argument"); return MYO_E_ARG; }
  myo::StepArgs a{};
  a.mode = myo::MODE_GET_OBS; a.obs = obs_dev;
  return launch(b, a, stream);
}

static int repack(myo_batch* b, float* dst, int ds, int doff, const float* src, int ss, int soff, int width, void* stream) {
  if (width <= 0) return MYO_OK;
  const long long total = (long long)b->n * width;
  MYO_LAUNCH(myo::repack_kernel, (unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), dst, ds, doff, src, ss, soff, width, b->n);
  b->launches++;
  CK(cudaGetLastError());
  return MYO_OK;
}

int myo_batch_set_state(myo_batch* b, const float* qpos_dev, const float* qvel_dev, const float* act_dev, const float* time_dev, void* stream) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  CK(cudaSetDevice(b->device));
  const myo::DevModel& d = b->pm.dm;
  int rc = MYO_OK;
  if (qpos_dev && (rc = repack(b, b->p.qpos, d.nq4, 0, qpos_dev, d.nq, 0, d.nq, stream))) return rc;
  if (qvel_dev && (rc = repack(b, b->p.qvel, d.nv4, 0, qvel_dev, d.nv, 0, d.nv, stream))) return rc;
  if (act_dev && d.na && (rc = repack(b, b->p.act, d.na4, 0, act_dev, d.na, 0, d.na, stream))) return rc;
  if (time_dev && (rc = repack(b, b->p.time, 1, 0, time_dev, 1, 0, 1, stream))) return rc;
  return MYO_OK;
}

int myo_batch_get_state(myo_batch* b, float* qpos_dev, float* qvel_dev, float* act_dev, float* time_dev, void* stream) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  CK(cudaSetDevice(b->device));
  const myo::DevModel& d = b->pm.dm;
  int rc = MYO_OK;
  if (qpos_dev && (rc = repack(b, qpos_dev, d.nq, 0, b->p.qpos, d.nq4, 0, d.nq, stream))) return rc;
  if (qvel_dev && (rc = repack(b, qvel_dev, d.nv, 0, b->p.qvel, d.nv4, 0, d.nv, stream))) return rc;
  if (act_dev && d.na && (rc = repack(b, act_dev, d.na, 0, b->p.act, d.na4, 0, d.na, stream))) return rc;
  if (time_dev && (rc = repack(b, time_dev, 1, 0, b->p.time, 1, 0, 1, stream))) return rc;
  return MYO_OK;
}

int myo_batch_get_task_state(myo_batch* b, int32_t* ti_dev, float* tf_dev, float* pose_target_dev, void* stream) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  static_assert(myo::TI_WORDS == MYO_TASK_STATE_I && myo::TF_WORDS == MYO_TASK_STATE_F, "task state layout");
  CK(cudaSetDevice(b->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (ti_dev) CK(cudaMemcpyAsync(ti_dev, b->p.task_i, (size_t)b->n * myo::TI_WORDS * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (tf_dev) CK(cudaMemcpyAsync(tf_dev, b->p.task_f, (size_t)b->n * myo::TF_WORDS * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (pose_target_dev) return repack(b, pose_target_dev, b->pm.dm.nq, 0, b->p.pose_target, b->pm.dm.nq4, 0, b->pm.dm.nq, stream);
  return MYO_OK;
}
int myo_batch_set_task_state(myo_batch* b, const int32_t* ti_dev, const float* tf_dev, const float* pose_target_dev, void* stream) {
  if (!b) { myo::set_error("null batch"); return MYO_E_ARG; }
  CK(cudaSetDevice(b->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (ti_dev) CK(cudaMemcpyAsync(b->p.task_i, ti_dev, (size_t)b->n * myo::TI_WORDS * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (tf_dev) CK(cudaMemcpyAsync(b->p.task_f, tf_dev, (size_t)b->n * myo::TF_WORDS * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (pose_target_dev) return repack(b, b->p.pose_target, b->pm.dm.nq4, 0, pose_target_dev, b->pm.dm.nq, 0, b->pm.dm.nq, stream);
  return MYO_OK;
}

static const myo::PackedModel::Slot* find_slot(const myo_batch* b, int kind, int id) {
  for (const auto& s : b->pm.slots) if (s.kind == kind && s.id == id) return &s;
  return nullptr;
}
int myo_batch_set_param(myo_batch* b, int kind, int id, const float* values_dev, void* stream) {
  if (!b || !values_dev) { myo::set_error("null argument"); return MYO_E_ARG; }
  const auto* s = find_slot(b, kind, id);
  if (!s) { myo::set_error("parameter was not declared as a per-world override in the task cfg"); return MYO_E_ARG; }
  CK(cudaSetDevice(b->device));
  return repack(b, b->p.wparam, b->pm.dm.nparam4, s->slot, values_dev, s->ncomp, 0, s->ncomp, stream);
}
int myo_batch_get_param(myo_batch* b, int kind, int id, float* values_dev, void* stream) {
  if (!b || !values_dev) { myo::set_error("null argument"); return MYO_E_ARG; }
  const auto* s = find_slot(b, kind, id);
  if (!s) { myo::set_error("parameter was not declared as a per-world override in the task cfg"); return MYO_E_ARG; }
  CK(cudaSetDevice(b->device));
  return repack(b, values_dev, s->ncomp, 0, b->p.wparam, b->pm.dm.nparam4, s->slot, s->ncomp, stream);
}

int myo_batch_stage_dump(myo_batch* b, int stage, void* out_dev, int* width, void* stream) {
  if (!b || stage < 0 || stage >= MYO_STAGE_COUNT) { myo::set_error("bad stage"); return MYO_E_ARG; }
  const myo::DevModel& d = b->pm.dm_full;
  int w = 0;
  switch (stage) {
    case MYO_STAGE_XPOS: w = 3 * d.nbody; break;
    case MYO_STAGE_XMAT: w = 9 * d.nbody; break;
    case MYO_STAGE_SITE_XPOS: w = 3 * d.nsite; break;
    case MYO_STAGE_TEN_LENGTH: w = d.ntendon; break;
    case MYO_STAGE_TEN_J: w = d.ntendon * d.nv; break;
    case MYO_STAGE_QM: w = d.nv * d.nv; break;
    case MYO_STAGE_ACT_FORCE: w = d.nu; break;
    case MYO_STAGE_ACT_DOT: w = d.na; break;
    case MYO_STAGE_NCON: case MYO_STAGE_NEFC: case MYO_STAGE_SOLVER_ITER: case MYO_STAGE_STATUS: w = 1; break;
    case MYO_STAGE_CONTACT_GEOMS: w = 2 * d.ncon_max; break;
    case MYO_STAGE_CONTACT_DIST: w = d.ncon_max; break;
    case MYO_STAGE_EFC_TYPE_ID: w = 2 * d.nefc_max; break;
    case MYO_STAGE_EFC_J: w = d.nefc_max * d.nv; break;
    case MYO_STAGE_EFC_AREF: case MYO_STAGE_EFC_D: case MYO_STAGE_EFC_FORCE: w = d.nefc_max; break;
    default: w = d.nv; break;
  }
  if (width) *width = w;
  if (!out_dev) return MYO_OK;
  if (!b->p.dump) { myo::set_error("no stage data: call myo_batch_forward or myo_batch_mj_step first"); return MYO_E_ARG; }
  CK(cudaSetDevice(b->device));
  MYO_LAUNCH(myo::extract_kernel, (b->n + 63) / 64, 64, b->tab_bytes, static_cast<cudaStream_t>(stream), d, b->p.dump, b->n, stage, out_dev, w);
  b->launches++;
  CK(cudaGetLastError());
  return MYO_OK;
}

int myo_batch_status(myo_batch* b, int* flags, void* stream) {
  if (!b || !flags) { myo::set_error("null argument"); return MYO_E_ARG; }
  CK(cudaSetDevice(b->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int h = 0;
  CK(cudaMemcpyAsync(&h, b->p.status, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaMemsetAsync(b->p.status, 0, sizeof(int), st));
  *flags = h;
  return MYO_OK;
}

int64_t myo_batch_launch_count(const myo_batch* b) { return b ? b->launches : 0; }

#ifdef MYO_PROFILE
// development builds only: cumulative per-phase cycles (lane 0 of every world), then cleared
int myo_debug_profile(unsigned long long* out16) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out16, myo::g_prof, sizeof(unsigned long long) * 16);
  unsigned long long z[16] = {0};
  cudaMemcpyToSymbol(myo::g_prof, z, sizeof z);
  return 0;
}
#endif

}  // extern "C"
