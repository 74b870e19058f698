// Recurrent policy forward for the rollout: sb3-contrib MlpLstmPolicy with separate actor / critic
// LSTMs (RecurrentActorCriticPolicy.forward as built by /root/reference/src/train/trainer.py:49-64;
// architecture of the winning runs:
// /root/reference/trained_models/curriculum_steps_complete_baoding_winner/01_rsi_static/main.py:178-200).
//
// One CTA owns a tile of 128 worlds of one network (grid.y: 0 = actor, 1 = critic) and runs the whole
// network on it with the activations resident in shared memory:
//   [x | h] (bf16, UMMA K-major core-matrix layout) --tcgen05.mma--> gates in TMEM (fp32, 4 gates x 64 units
//   per 256-column accumulator) --tcgen05.ld--> LSTM cell in registers -> h', c' (fp32, HBM) and h' (bf16, smem)
//   -> MLP layers (ReLU) -> head (Gaussian mean + sample + log-prob, or value).
// Weights are pre-packed once into the exact shared-memory image of every K-chunk, so the producer warp
// streams them from L2 with one cp.async.bulk (TMA engine, mbarrier complete_tx) per chunk into a 4-deep ring.
// Warp roles: warps 0-3 = loader / epilogue (one world per thread, TMEM lane = thread), warp 4 = weight
// producer, warp 5 = TMEM allocator + the single MMA-issuing thread.
#include <cublas_v2.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/myo_b200.h"

namespace myo {
void set_error(const std::string& msg);
}

namespace {

constexpr int TILE_M = 128;
constexpr int CHUNK_K = 32;                       // K elements per streamed weight chunk
constexpr int STAGES = 4;
constexpr int MAX_N = 256;
constexpr int STAGE_BYTES = MAX_N * CHUNK_K * 2;  // 16 KB
constexpr int MAX_OPS = 12;
constexpr int THREADS = 192;
constexpr int MAX_K1 = 128 + 256;                 // padded obs (hand pose: 108, die: 103) + hidden
constexpr int A1_BYTES = TILE_M * MAX_K1 * 2;     // 98304
constexpr int HB_BYTES = TILE_M * 256 * 2;        // 65536
constexpr int SMEM_BYTES = A1_BYTES + HB_BYTES + STAGES * STAGE_BYTES + 256;

enum { EPI_LSTM = 0, EPI_RELU = 1, EPI_HEAD_PI = 2, EPI_HEAD_VF = 3 };
enum { BUF_A1 = 0, BUF_HB = 1 };

struct GemmOp {
  int a_buf;        // A operand buffer
  int a_wait;       // 1: first reader of a new version of a_buf (wait for its writers)
  int K, N;         // K multiple of 16, N multiple of 16 and <= 256
  int epi, arg;     // epilogue kind; LSTM: hidden-unit tile index
  int out_buf;      // buffer the epilogue writes bf16 activations into
  int signal;       // 1: the epilogue completes a version of out_buf
  long long w_off;  // byte offset of the packed weights
  int b_off;        // float offset of the bias
};
struct NetProgram {
  int n_ops;
  GemmOp op[MAX_OPS];
};

struct FwdArgs {
  int n, obs_dim, obs_pad, H, act_dim;
  const float* obs;
  float* h;
  float* c;
  const uint8_t* start;
  const float* noise;
  float* actions;
  float* values;
  float* logp;
  const uint8_t* wpack[2];
  const float* bias[2];
  const float* log_std;
  const float* obs_mean;      // optional VecNormalize statistics (may be null)
  const float* obs_inv_std;
  float clip_obs;
  unsigned long long seed, step;   // seed != 0 and noise == null: sample with the in-kernel Philox stream
  float* latent;                   // optional [n][latent_dim]: the actor's last MLP activation (latent_pi, the input of action_net)
  int latent_dim;
};

// ---- PTX wrappers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor, K-major, no swizzle: 8x(16 B) core matrices; SBO = byte stride between
// 8-row groups, LBO = byte stride between the two K halves of one K=16 step (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (Blackwell)
  return d;
}
// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128
__device__ __forceinline__ uint32_t make_idesc(int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }
__device__ __forceinline__ float tanhf_(float x) { return 2.f / (1.f + __expf(-2.f * x)) - 1.f; }
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
// activation element (row, k) of a 128-row K-major buffer lives at (k/8)*2048 + row*16 + (k%8)*2
__device__ __forceinline__ uint32_t act_off(int row, int k) { return (uint32_t)((k >> 3) * (TILE_M * 16) + row * 16 + (k & 7) * 2); }

// Philox4x32-10 -> two standard normals per call (Box-Muller); stream keyed by (seed, world), counter (step, j)
__device__ __forceinline__ void philox_normal2(unsigned long long seed, uint32_t world, uint32_t step, uint32_t j, float* z0, float* z1) {
  uint32_t k0 = (uint32_t)seed ^ (world * 0x9E3779B9u), k1 = (uint32_t)(seed >> 32) ^ 0xBB67AE85u ^ world;
  uint32_t c0 = j, c1 = step, c2 = world, c3 = 0x2545F491u;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const float u0 = ((float)(c0 >> 8) + 0.5f) * (1.0f / 16777216.0f), u1 = (float)(c1 >> 8) * (1.0f / 16777216.0f);
  const float r = sqrtf(-2.f * __logf(u0));
  float sn, cs;
  __sincosf(6.283185307179586f * u1, &sn, &cs);
  *z0 = r * cs; *z1 = r * sn;
}

__global__ void __launch_bounds__(THREADS, 1)
policy_forward_kernel(const __grid_constant__ FwdArgs a, const __grid_constant__ NetProgram prog_pi, const __grid_constant__ NetProgram prog_vf) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int net = blockIdx.y;
  const NetProgram& prog = net == 0 ? prog_pi : prog_vf;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * TILE_M;

  uint8_t* sA1 = smem;
  uint8_t* sHB = smem + A1_BYTES;
  uint8_t* sRing = smem + A1_BYTES + HB_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + A1_BYTES + HB_BYTES + STAGES * STAGE_BYTES);
  // barriers: full[STAGES], empty[STAGES], acc_full[2], acc_empty[2], abuf_ready[2]; then the TMEM base word
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + STAGES), bar_accf = smem_u32(bars + 2 * STAGES),
                 bar_acce = smem_u32(bars + 2 * STAGES + 2), bar_abuf = smem_u32(bars + 2 * STAGES + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 6);

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    for (int s = 0; s < 2; s++) { mbar_init(bar_accf + 8 * s, 1); mbar_init(bar_acce + 8 * s, TILE_M); mbar_init(bar_abuf + 8 * s, TILE_M); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ================= loader: [x | h] tile -> bf16 core-matrix layout =================
    const int H = a.H;
    for (int rr = 0; rr < 32; rr++) {
      const int row = warp * 32 + rr, w = row0 + row;
      const bool live = w < a.n;
      const float keep = (live && !a.start[w]) ? 1.f : 0.f;
      // observation: obs_pad / 2 float2 slots, lanes take 2 consecutive k
      for (int k = 2 * lane; k < a.obs_pad; k += 64) {
        float x0 = 0.f, x1 = 0.f;
        if (live && k < a.obs_dim) {
          x0 = a.obs[(size_t)w * a.obs_dim + k];
          if (k + 1 < a.obs_dim) x1 = a.obs[(size_t)w * a.obs_dim + k + 1];
          if (a.obs_mean) {
            x0 = fminf(fmaxf((x0 - a.obs_mean[k]) * a.obs_inv_std[k], -a.clip_obs), a.clip_obs);
            if (k + 1 < a.obs_dim) x1 = fminf(fmaxf((x1 - a.obs_mean[k + 1]) * a.obs_inv_std[k + 1], -a.clip_obs), a.clip_obs);
          }
        }
        *reinterpret_cast<uint32_t*>(sA1 + act_off(row, k)) = pack_bf16(x0, x1);
      }
      const float* hrow = a.h + ((size_t)net * a.n + (live ? w : 0)) * H;
      for (int k = 4 * lane; k < H; k += 128) {
        float4 v = live ? *reinterpret_cast<const float4*>(hrow + k) : make_float4(0.f, 0.f, 0.f, 0.f);
        uint2 p;
        p.x = pack_bf16(v.x * keep, v.y * keep);
        p.y = pack_bf16(v.z * keep, v.w * keep);
        *reinterpret_cast<uint2*>(sA1 + act_off(row, a.obs_pad + k)) = p;
      }
    }
    fence_async_smem();
    mbar_arrive(bar_abuf + 8 * BUF_A1);

    // ================= epilogues =================
    const int row = threadIdx.x, w = row0 + row;
    const bool live = w < a.n;
    const float keep = (live && !a.start[w]) ? 1.f : 0.f;
    const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float* bias = a.bias[net];
    for (int i = 0; i < prog.n_ops; i++) {
      const GemmOp& op = prog.op[i];
      const int buf = i & 1;
      mbar_wait(bar_accf + 8 * buf, (i >> 1) & 1);
      tc_fence_after();
      const uint32_t acc = lane_base + buf * 256;
      uint8_t* sOut = op.out_buf == BUF_A1 ? sA1 : sHB;
      if (op.epi == EPI_LSTM) {
        const int u0 = op.arg * 64;
        float* crow = a.c + ((size_t)net * a.n + (live ? w : 0)) * H + u0;
        float* hrow = a.h + ((size_t)net * a.n + (live ? w : 0)) * H + u0;
        const float* b = bias + op.b_off;
        for (int jb = 0; jb < 4; jb++) {
          uint32_t gi[16], gf[16], gg[16], go[16];
          tmem_ld16(acc + 0 * 64 + jb * 16, gi);
          tmem_ld16(acc + 1 * 64 + jb * 16, gf);
          tmem_ld16(acc + 2 * 64 + jb * 16, gg);
          tmem_ld16(acc + 3 * 64 + jb * 16, go);
          float cold[16];
#pragma unroll
          for (int q = 0; q < 4; q++) {
            float4 v = live ? *reinterpret_cast<const float4*>(crow + jb * 16 + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
            cold[4 * q] = v.x * keep; cold[4 * q + 1] = v.y * keep; cold[4 * q + 2] = v.z * keep; cold[4 * q + 3] = v.w * keep;
          }
          tmem_ld_wait();
          float hn[16], cn[16];
#pragma unroll
          for (int u = 0; u < 16; u++) {
            const int col = jb * 16 + u;
            const float ig = sigmoidf_(__uint_as_float(gi[u]) + b[col]);
            const float fg = sigmoidf_(__uint_as_float(gf[u]) + b[64 + col]);
            const float gv = tanhf_(__uint_as_float(gg[u]) + b[128 + col]);
            const float og = sigmoidf_(__uint_as_float(go[u]) + b[192 + col]);
            cn[u] = fg * cold[u] + ig * gv;
            hn[u] = og * tanhf_(cn[u]);
          }
          if (live) {
#pragma unroll
            for (int q = 0; q < 4; q++) {
              *reinterpret_cast<float4*>(crow + jb * 16 + 4 * q) = make_float4(cn[4 * q], cn[4 * q + 1], cn[4 * q + 2], cn[4 * q + 3]);
              *reinterpret_cast<float4*>(hrow + jb * 16 + 4 * q) = make_float4(hn[4 * q], hn[4 * q + 1], hn[4 * q + 2], hn[4 * q + 3]);
            }
          }
#pragma unroll
          for (int q = 0; q < 2; q++) {
            uint4 p;
            p.x = pack_bf16(hn[8 * q], hn[8 * q + 1]); p.y = pack_bf16(hn[8 * q + 2], hn[8 * q + 3]);
            p.z = pack_bf16(hn[8 * q + 4], hn[8 * q + 5]); p.w = pack_bf16(hn[8 * q + 6], hn[8 * q + 7]);
            *reinterpret_cast<uint4*>(sOut + act_off(row, u0 + jb * 16 + 8 * q)) = p;
          }
        }
      } else if (op.epi == EPI_RELU) {
        const float* b = bias + op.b_off;
        for (int cb = 0; cb < op.N / 16; cb++) {
          uint32_t r[16];
          tmem_ld16(acc + cb * 16, r);
          tmem_ld_wait();
          float v[16];
#pragma unroll
          for (int u = 0; u < 16; u++) v[u] = fmaxf(__uint_as_float(r[u]) + b[cb * 16 + u], 0.f);
          if (a.latent && net == 0 && i == prog.n_ops - 2 && live) {      // latent_pi for state-dependent exploration (gSDE)
            float4* dst = reinterpret_cast<float4*>(a.latent + (size_t)w * a.latent_dim + cb * 16);
#pragma unroll
            for (int q = 0; q < 4; q++) dst[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          }
#pragma unroll
          for (int q = 0; q < 2; q++) {
            uint4 p;
            p.x = pack_bf16(v[8 * q], v[8 * q + 1]); p.y = pack_bf16(v[8 * q + 2], v[8 * q + 3]);
            p.z = pack_bf16(v[8 * q + 4], v[8 * q + 5]); p.w = pack_bf16(v[8 * q + 6], v[8 * q + 7]);
            *reinterpret_cast<uint4*>(sOut + act_off(row, cb * 16 + 8 * q)) = p;
          }
        }
      } else if (op.epi == EPI_HEAD_PI) {
        const float* b = bias + op.b_off;
        float lp = 0.f;
        for (int cb = 0; cb < op.N / 16; cb++) {
          uint32_t r[16];
          tmem_ld16(acc + cb * 16, r);
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 16; u += 2) {
            const int j = cb * 16 + u;
            if (j >= a.act_dim) continue;
            float z0 = 0.f, z1 = 0.f;
            if (live) {
              if (a.noise) { z0 = a.noise[(size_t)w * a.act_dim + j]; if (j + 1 < a.act_dim) z1 = a.noise[(size_t)w * a.act_dim + j + 1]; }
              else if (a.seed) philox_normal2(a.seed, (uint32_t)w, (uint32_t)a.step, (uint32_t)j, &z0, &z1);
            }
            const float ls0 = a.log_std[j];
            const float m0 = __uint_as_float(r[u]) + b[j];
            if (live) a.actions[(size_t)w * a.act_dim + j] = m0 + __expf(ls0) * z0;
            lp += -0.5f * z0 * z0 - ls0 - 0.9189385332046727f;
            if (j + 1 < a.act_dim) {
              const float ls1 = a.log_std[j + 1];
              const float m1 = __uint_as_float(r[u + 1]) + b[j + 1];
              if (live) a.actions[(size_t)w * a.act_dim + j + 1] = m1 + __expf(ls1) * z1;
              lp += -0.5f * z1 * z1 - ls1 - 0.9189385332046727f;
            }
          }
        }
        if (live && a.logp) a.logp[w] = lp;
      } else {   // EPI_HEAD_VF
        uint32_t r[16];
        tmem_ld16(acc, r);
        tmem_ld_wait();
        if (live && a.values) a.values[w] = __uint_as_float(r[0]) + bias[op.b_off];
      }
      tc_fence_before();
      mbar_arrive(bar_acce + 8 * buf);
      if (op.signal) {
        fence_async_smem();
        mbar_arrive(bar_abuf + 8 * op.out_buf);
      }
    }
  } else if (warp == 4) {
    // ================= weight producer =================
    if (lane == 0) {
      int chunk = 0;
      const uint8_t* wp = a.wpack[net];
      for (int i = 0; i < prog.n_ops; i++) {
        const GemmOp& op = prog.op[i];
        const uint8_t* src = wp + op.w_off;
        for (int k0 = 0; k0 < op.K; k0 += CHUNK_K, chunk++) {
          const int s = chunk % STAGES;
          const int ck = min(CHUNK_K, op.K - k0);
          const uint32_t bytes = (uint32_t)(op.N * ck * 2);
          if (chunk >= STAGES) mbar_wait(bar_empty + 8 * s, ((chunk / STAGES) - 1) & 1);
          mbar_expect_tx(bar_full + 8 * s, bytes);
          bulk_g2s(smem_u32(sRing + s * STAGE_BYTES), src, bytes, bar_full + 8 * s);
          src += bytes;
        }
      }
    }
  } else {
    // ================= MMA issuer =================
    if (lane == 0) {
      int chunk = 0;
      int abuf_phase[2] = {0, 0};
      for (int i = 0; i < prog.n_ops; i++) {
        const GemmOp& op = prog.op[i];
        const int buf = i & 1;
        if (op.a_wait) { mbar_wait(bar_abuf + 8 * op.a_buf, abuf_phase[op.a_buf] & 1); abuf_phase[op.a_buf]++; }
        if (i >= 2) mbar_wait(bar_acce + 8 * buf, ((i >> 1) - 1) & 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * 256;
        const uint32_t idesc = make_idesc(op.N);
        const uint32_t a_base = smem_u32(op.a_buf == BUF_A1 ? sA1 : sHB);
        const uint32_t b_lbo = (uint32_t)op.N * 16, a_lbo = TILE_M * 16;
        for (int k0 = 0; k0 < op.K; k0 += CHUNK_K, chunk++) {
          const int s = chunk % STAGES;
          const int ck = min(CHUNK_K, op.K - k0);
          mbar_wait(bar_full + 8 * s, (chunk / STAGES) & 1);
          tc_fence_after();
          const uint32_t b_base = smem_u32(sRing + s * STAGE_BYTES);
          for (int ks = 0; ks < ck; ks += 16) {
            const uint32_t a_addr = a_base + (uint32_t)((k0 + ks) >> 3) * a_lbo;
            const uint32_t b_addr = b_base + (uint32_t)(ks >> 3) * b_lbo;
            const uint64_t ad = make_desc(a_addr, a_lbo, 128);
            const uint64_t bd = make_desc(b_addr, b_lbo, 128);
            umma_bf16(d_tmem, ad, bd, idesc, (k0 + ks) > 0 ? 1u : 0u);
          }
          umma_commit(bar_empty + 8 * s);
        }
        umma_commit(bar_accf + 8 * buf);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// ---- weight packing: fp32 torch layout -> bf16 chunked core-matrix image ---------------------------
// element (n, k) of an N x K operand: chunk = k / CHUNK_K (all chunks before the last are CHUNK_K wide),
// inside the chunk (kk = k % CHUNK_K): (kk/8) * N*16 + (n/8)*128 + (n%8)*16 + (kk%8)*2 bytes
__device__ __forceinline__ size_t pack_off(int N, int n, int k) {
  const int chunk = k / CHUNK_K, kk = k % CHUNK_K;
  return (size_t)chunk * N * CHUNK_K * 2 + (size_t)(kk >> 3) * N * 16 + (size_t)(n >> 3) * 128 + (n & 7) * 16 + (kk & 7) * 2;
}
__global__ void pack_lstm_kernel(uint8_t* dst, float* bias_dst, const float* w_ih, const float* w_hh, const float* b_ih,
                                 const float* b_hh, int H, int obs_dim, int obs_pad, int tile) {
  const int K = obs_pad + H;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 256 * K) return;
  const int n = idx / K, k = idx % K;
  const int gate = n / 64, j = n % 64;
  const int srow = gate * H + tile * 64 + j;
  float v;
  if (k < obs_pad) v = k < obs_dim ? w_ih[(size_t)srow * obs_dim + k] : 0.f;
  else v = w_hh[(size_t)srow * H + (k - obs_pad)];
  *reinterpret_cast<__nv_bfloat16*>(dst + pack_off(256, n, k)) = __float2bfloat16_rn(v);
  if (k == 0) bias_dst[n] = b_ih[srow] + b_hh[srow];
}
__global__ void pack_dense_kernel(uint8_t* dst, float* bias_dst, const float* w, const float* b, int N, int K, int n_src, int k_src) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * K) return;
  const int n = idx / K, k = idx % K;
  const float v = (n < n_src && k < k_src) ? w[(size_t)n * k_src + k] : 0.f;
  *reinterpret_cast<__nv_bfloat16*>(dst + pack_off(N, n, k)) = __float2bfloat16_rn(v);
  if (k == 0) bias_dst[n] = n < n_src ? b[n] : 0.f;
}
__global__ void inv_std_kernel(float* mean_dst, float* inv_dst, const float* mean, const float* var, float eps, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { mean_dst[i] = mean[i]; inv_dst[i] = rsqrtf(var[i] + eps); }
}

int round_up(int x, int m) { return (x + m - 1) / m * m; }

}  // namespace

// ---- generalised state-dependent exploration (SB3 StateDependentNoiseDistribution, use_sde=True) ---------------------
// reset_noise: one exploration matrix per world, E[w][l][k] = exp(log_std[l][k]) * N(0, 1), kept in bf16; also the table
// s2[l][k] = exp(2 log_std[l][k]) the variance needs. Counter-based draws keyed by (seed, world), counter (epoch, pair index).
__global__ void sde_reset_noise_kernel(__nv_bfloat16* __restrict__ E, float* __restrict__ s2, const float* __restrict__ log_std, int n, int LA,
                                       unsigned long long seed, unsigned int epoch) {
  const int pairs = (LA + 1) / 2;
  const long long total = (long long)n * pairs;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int w = (int)(i / pairs), j = (int)(i - (long long)w * pairs);
    float z0, z1;
    philox_normal2(seed, (uint32_t)w, epoch, (uint32_t)j, &z0, &z1);
    const int e = 2 * j;
    E[(size_t)w * LA + e] = __float2bfloat16_rn(expf(log_std[e]) * z0);
    if (e + 1 < LA) E[(size_t)w * LA + e + 1] = __float2bfloat16_rn(expf(log_std[e + 1]) * z1);
  }
  if (blockIdx.x == 0) for (int e = threadIdx.x; e < LA; e += blockDim.x) s2[e] = expf(2.f * log_std[e]);
}

// one warp per world: noise_k = sum_l latent_l E[w][l][k], variance_k = sum_l latent_l^2 s2[l][k] + 1e-6 (StateDependentNoiseDistribution.
// get_noise / proba_distribution), action = mean + noise, log_prob = sum_k log N(noise_k; 0, variance_k). actions: mean in, action out.
__global__ void sde_sample_kernel(const float* __restrict__ latent, int ld, const __nv_bfloat16* __restrict__ E, const float* __restrict__ s2,
                                  float* __restrict__ actions, float* __restrict__ logp, int n, int L, int A) {
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= n) return;
  const __nv_bfloat16* Ew = E + (size_t)w * L * A;
  const float* lat = latent + (size_t)w * ld;
  float nz[2] = {0.f, 0.f}, var[2] = {0.f, 0.f};
  for (int l = 0; l < L; l++) {
    const float x = lat[l];
#pragma unroll
    for (int q = 0; q < 2; q++) {
      const int k = lane + 32 * q;
      if (k < A) { nz[q] += x * __bfloat162float(Ew[l * A + k]); var[q] += x * x * s2[l * A + k]; }
    }
  }
  float lp = 0.f;
#pragma unroll
  for (int q = 0; q < 2; q++) {
    const int k = lane + 32 * q;
    if (k < A) {
      const float v = var[q] + 1e-6f;
      actions[(size_t)w * A + k] += nz[q];
      lp += -0.5f * nz[q] * nz[q] / v - 0.5f * logf(v) - 0.9189385332046727f;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) lp += __shfl_xor_sync(0xffffffffu, lp, o);
  if (lane == 0 && logp) logp[w] = lp;
}

struct myo_policy {
  myo_policy_cfg cfg{};
  int device = 0, max_batch = 0, obs_pad = 0;
  std::map<std::string, float*> weights;   // fp32 staging copies by SB3 state-dict key
  std::map<std::string, int64_t> numel;
  NetProgram prog[2]{};
  uint8_t* wpack[2] = {nullptr, nullptr};
  float* bias[2] = {nullptr, nullptr};
  size_t wbytes[2] = {0, 0};
  int nbias[2] = {0, 0};
  float* log_std = nullptr;
  float *obs_mean = nullptr, *obs_inv_std = nullptr;
  float clip_obs = 10.f;
  bool has_norm = false, dirty = true;
  unsigned long long seed = 0, step = 0;
  int64_t launches = 0;
  float* latent_out = nullptr;   // caller-owned [max_batch][latent_dim], see myo_policy_set_latent_out
  // fp32 mode (myo_policy_set_precision): plain SGEMMs on the fp32 weights + elementwise kernels, for evaluating trained
  // checkpoints at the reference's own precision; scratch allocated on first use
  int precision = 0;
  cublasHandle_t blas = nullptr;
  float* f32_scratch = nullptr;
};

namespace {

#define PCK(call)                                                                   \
  do {                                                                              \
    cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess) {                                                        \
      myo::set_error(std::string(#call) + ": " + cudaGetErrorString(e_));           \
      return MYO_E_CUDA;                                                            \
    }                                                                               \
  } while (0)

// lay out the GEMM sequence of one network and the offsets of its packed weights / biases
void build_program(const myo_policy* p, int net, NetProgram& pr, size_t& wbytes, int& nbias) {
  const myo_policy_cfg& c = p->cfg;
  const int H = c.lstm_hidden, K1 = p->obs_pad + H;
  const int nl = net == 0 ? c.n_pi_layers : c.n_vf_layers;
  const int* widths = net == 0 ? c.pi_layers : c.vf_layers;
  size_t w = 0;
  int b = 0, n = 0;
  const int ntile = H / 64;
  for (int t = 0; t < ntile; t++) {
    GemmOp& op = pr.op[n++];
    op = GemmOp{BUF_A1, t == 0, K1, 256, EPI_LSTM, t, BUF_HB, t == ntile - 1, (long long)w, b};
    w += (size_t)256 * K1 * 2; b += 256;
  }
  int in_buf = BUF_HB, in_dim = H;
  for (int l = 0; l < nl; l++) {
    GemmOp& op = pr.op[n++];
    const int out_buf = in_buf == BUF_HB ? BUF_A1 : BUF_HB;
    op = GemmOp{in_buf, 1, in_dim, widths[l], EPI_RELU, 0, out_buf, 1, (long long)w, b};
    w += (size_t)widths[l] * in_dim * 2; b += widths[l];
    in_buf = out_buf; in_dim = widths[l];
  }
  {
    GemmOp& op = pr.op[n++];
    const int N = net == 0 ? round_up(c.act_dim, 16) : 16;
    op = GemmOp{in_buf, 1, in_dim, N, net == 0 ? EPI_HEAD_PI : EPI_HEAD_VF, 0, -1, 0, (long long)w, b};
    w += (size_t)N * in_dim * 2; b += N;
  }
  pr.n_ops = n;
  wbytes = w; nbias = b;
}

const float* find_w(const myo_policy* p, const std::string& name, int64_t need) {
  auto it = p->weights.find(name);
  if (it == p->weights.end()) { myo::set_error("policy weight not set: " + name); return nullptr; }
  if (p->numel.at(name) != need) { myo::set_error("policy weight has the wrong size: " + name); return nullptr; }
  return it->second;
}

int pack_weights(myo_policy* p, cudaStream_t st) {
  const myo_policy_cfg& c = p->cfg;
  const int H = c.lstm_hidden, K1 = p->obs_pad + H;
  for (int net = 0; net < 2; net++) {
    const std::string lstm = net == 0 ? "lstm_actor." : "lstm_critic.";
    const float* w_ih = find_w(p, lstm + "weight_ih_l0", (int64_t)4 * H * c.obs_dim);
    const float* w_hh = find_w(p, lstm + "weight_hh_l0", (int64_t)4 * H * H);
    const float* b_ih = find_w(p, lstm + "bias_ih_l0", 4 * H);
    const float* b_hh = find_w(p, lstm + "bias_hh_l0", 4 * H);
    if (!w_ih || !w_hh || !b_ih || !b_hh) return MYO_E_ARG;
    const NetProgram& pr = p->prog[net];
    int i = 0;
    for (; i < H / 64; i++) {
      const GemmOp& op = pr.op[i];
      pack_lstm_kernel<<<(256 * K1 + 255) / 256, 256, 0, st>>>(p->wpack[net] + op.w_off, p->bias[net] + op.b_off, w_ih, w_hh, b_ih, b_hh, H,
                                                               c.obs_dim, p->obs_pad, op.arg);
      p->launches++;
    }
    const int nl = net == 0 ? c.n_pi_layers : c.n_vf_layers;
    const int* widths = net == 0 ? c.pi_layers : c.vf_layers;
    int in_dim = H;
    for (int l = 0; l < nl; l++, i++) {
      const GemmOp& op = pr.op[i];
      const std::string base = std::string("mlp_extractor.") + (net == 0 ? "policy_net." : "value_net.") + std::to_string(2 * l);
      const float* w = find_w(p, base + ".weight", (int64_t)widths[l] * in_dim);
      const float* b = find_w(p, base + ".bias", widths[l]);
      if (!w || !b) return MYO_E_ARG;
      pack_dense_kernel<<<(op.N * op.K + 255) / 256, 256, 0, st>>>(p->wpack[net] + op.w_off, p->bias[net] + op.b_off, w, b, op.N, op.K, widths[l], in_dim);
      p->launches++;
      in_dim = widths[l];
    }
    {
      const GemmOp& op = pr.op[i];
      const int n_src = net == 0 ? c.act_dim : 1;
      const std::string base = net == 0 ? "action_net" : "value_net";
      const float* w = find_w(p, base + ".weight", (int64_t)n_src * in_dim);
      const float* b = find_w(p, base + ".bias", n_src);
      if (!w || !b) return MYO_E_ARG;
      pack_dense_kernel<<<(op.N * op.K + 255) / 256, 256, 0, st>>>(p->wpack[net] + op.w_off, p->bias[net] + op.b_off, w, b, op.N, op.K, n_src, in_dim);
      p->launches++;
    }
  }
  const float* ls = find_w(p, "log_std", c.act_dim);
  if (!ls) return MYO_E_ARG;
  PCK(cudaMemcpyAsync(p->log_std, ls, sizeof(float) * c.act_dim, cudaMemcpyDeviceToDevice, st));
  PCK(cudaGetLastError());
  p->dirty = false;
  return MYO_OK;
}

// ---- fp32 mode: the same function, plain fp32 arithmetic (library SGEMMs; this is the evaluation path, not the hot path) ----
__global__ void f32_prepare_kernel(float* xn, float* hm, const float* obs, const float* h, const uint8_t* start, const float* mean,
                                   const float* inv_std, float clip, int n, int O, int H) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (long long)n * O) {
    const int k = (int)(i % O);
    float v = obs[i];
    if (mean) v = fminf(fmaxf((v - mean[k]) * inv_std[k], -clip), clip);
    xn[i] = v;
  }
  if (i < (long long)n * H) hm[i] = start[i / H] ? 0.f : h[i];
}
__global__ void f32_cell_kernel(const float* gates, const float* b_ih, const float* b_hh, float* h, float* c, const uint8_t* start, int n, int H) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * H) return;
  const int w = (int)(i / H), u = (int)(i % H);
  const float* g = gates + (size_t)w * 4 * H;
  const float gi = g[u] + b_ih[u] + b_hh[u], gf = g[H + u] + b_ih[H + u] + b_hh[H + u];
  const float gg = g[2 * H + u] + b_ih[2 * H + u] + b_hh[2 * H + u], go = g[3 * H + u] + b_ih[3 * H + u] + b_hh[3 * H + u];
  const float cp = start[w] ? 0.f : c[i];
  const float cn = (1.f / (1.f + expf(-gf))) * cp + (1.f / (1.f + expf(-gi))) * tanhf(gg);
  c[i] = cn;
  h[i] = (1.f / (1.f + expf(-go))) * tanhf(cn);
}
__global__ void f32_bias_act_kernel(float* y, const float* b, int n, int N, int relu) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * N) return;
  const float v = y[i] + b[i % N];
  y[i] = relu ? fmaxf(v, 0.f) : v;
}
__global__ void f32_gauss_kernel(const float* mean, const float* log_std, const float* noise, unsigned long long seed, unsigned long long step,
                                 float* actions, float* logp, int n, int A) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n) return;
  float lp = 0.f;
  for (int j = 0; j < A; j += 2) {
    float z0 = 0.f, z1 = 0.f;
    if (noise) { z0 = noise[(size_t)w * A + j]; if (j + 1 < A) z1 = noise[(size_t)w * A + j + 1]; }
    else if (seed) philox_normal2(seed, (uint32_t)w, (uint32_t)step, (uint32_t)j, &z0, &z1);
    actions[(size_t)w * A + j] = mean[(size_t)w * A + j] + expf(log_std[j]) * z0;
    lp += -0.5f * z0 * z0 - log_std[j] - 0.9189385332046727f;
    if (j + 1 < A) {
      actions[(size_t)w * A + j + 1] = mean[(size_t)w * A + j + 1] + expf(log_std[j + 1]) * z1;
      lp += -0.5f * z1 * z1 - log_std[j + 1] - 0.9189385332046727f;
    }
  }
  if (logp) logp[w] = lp;
}

// Y[n][N] (row major) = X[n][K] W[N][K]' (+ Y if accumulate)
int f32_gemm(myo_policy* p, const float* X, const float* W, float* Y, int n, int N, int K, bool accumulate) {
  const float one = 1.f, beta = accumulate ? 1.f : 0.f;
  if (cublasSgemm(p->blas, CUBLAS_OP_T, CUBLAS_OP_N, N, n, K, &one, W, K, X, K, &beta, Y, N) != CUBLAS_STATUS_SUCCESS) {
    myo::set_error("cublasSgemm failed in the fp32 policy forward");
    return MYO_E_CUDA;
  }
  return MYO_OK;
}

int forward_fp32(myo_policy* p, int n, const float* obs, float* h, float* c, const uint8_t* start, const float* noise, float* actions,
                 float* values, float* logp, cudaStream_t st) {
  const myo_policy_cfg& cf = p->cfg;
  const int H = cf.lstm_hidden, O = cf.obs_dim, A = cf.act_dim, W = 256;
  if (!p->blas) {
    if (cublasCreate(&p->blas) != CUBLAS_STATUS_SUCCESS) { myo::set_error("cublasCreate failed"); return MYO_E_CUDA; }
    cublasSetMathMode(p->blas, CUBLAS_PEDANTIC_MATH);      // true fp32: no TF32, no reduced-precision accumulation
  }
  cublasSetStream(p->blas, st);
  const size_t per = (size_t)O + H + 4 * H + 2 * W + A;      // xn | hm | gates | two activation buffers | mean
  if (!p->f32_scratch) PCK(cudaMalloc(&p->f32_scratch, sizeof(float) * per * p->max_batch));
  float* xn = p->f32_scratch;
  float* hm = xn + (size_t)p->max_batch * O;
  float* gates = hm + (size_t)p->max_batch * H;
  float* act[2] = {gates + (size_t)p->max_batch * 4 * H, gates + (size_t)p->max_batch * (4 * H + W)};
  float* mean = act[1] + (size_t)p->max_batch * W;
  auto blocks = [](long long total) { return (unsigned)((total + 255) / 256); };
  int rc;
  for (int net = 0; net < 2; net++) {
    const std::string lstm = net == 0 ? "lstm_actor." : "lstm_critic.";
    const float* w_ih = find_w(p, lstm + "weight_ih_l0", (int64_t)4 * H * O);
    const float* w_hh = find_w(p, lstm + "weight_hh_l0", (int64_t)4 * H * H);
    const float* b_ih = find_w(p, lstm + "bias_ih_l0", 4 * H);
    const float* b_hh = find_w(p, lstm + "bias_hh_l0", 4 * H);
    if (!w_ih || !w_hh || !b_ih || !b_hh) return MYO_E_ARG;
    float* hn = h + (size_t)net * n * H;
    float* cn = c + (size_t)net * n * H;
    f32_prepare_kernel<<<blocks((long long)n * std::max(O, H)), 256, 0, st>>>(xn, hm, obs, hn, start, p->has_norm ? p->obs_mean : nullptr,
                                                                           p->obs_inv_std, p->clip_obs, n, O, H);
    if ((rc = f32_gemm(p, xn, w_ih, gates, n, 4 * H, O, false)) || (rc = f32_gemm(p, hm, w_hh, gates, n, 4 * H, H, true))) return rc;
    f32_cell_kernel<<<blocks((long long)n * H), 256, 0, st>>>(gates, b_ih, b_hh, hn, cn, start, n, H);
    p->launches += 4;
    const int nl = net == 0 ? cf.n_pi_layers : cf.n_vf_layers;
    const int* widths = net == 0 ? cf.pi_layers : cf.vf_layers;
    const float* x = hn;
    int in_dim = H;
    for (int l = 0; l < nl; l++) {
      const std::string base = std::string("mlp_extractor.") + (net == 0 ? "policy_net." : "value_net.") + std::to_string(2 * l);
      const float* w = find_w(p, base + ".weight", (int64_t)widths[l] * in_dim);
      const float* b = find_w(p, base + ".bias", widths[l]);
      if (!w || !b) return MYO_E_ARG;
      float* y = act[l & 1];
      if ((rc = f32_gemm(p, x, w, y, n, widths[l], in_dim, false))) return rc;
      f32_bias_act_kernel<<<blocks((long long)n * widths[l]), 256, 0, st>>>(y, b, n, widths[l], 1);
      p->launches += 2;
      x = y; in_dim = widths[l];
    }
    if (net == 0) {
      const float* w = find_w(p, "action_net.weight", (int64_t)A * in_dim);
      const float* b = find_w(p, "action_net.bias", A);
      const float* ls = find_w(p, "log_std", A);
      if (!w || !b || !ls) return MYO_E_ARG;
      if (p->latent_out && nl > 0) PCK(cudaMemcpyAsync(p->latent_out, x, sizeof(float) * (size_t)n * in_dim, cudaMemcpyDeviceToDevice, st));
      if ((rc = f32_gemm(p, x, w, mean, n, A, in_dim, false))) return rc;
      f32_bias_act_kernel<<<blocks((long long)n * A), 256, 0, st>>>(mean, b, n, A, 0);
      f32_gauss_kernel<<<blocks(n), 256, 0, st>>>(mean, ls, noise, p->seed, p->step, actions, logp, n, A);
      p->launches += 3;
    } else if (values) {
      const float* w = find_w(p, "value_net.weight", in_dim);
      const float* b = find_w(p, "value_net.bias", 1);
      if (!w || !b) return MYO_E_ARG;
      if ((rc = f32_gemm(p, x, w, values, n, 1, in_dim, false))) return rc;
      f32_bias_act_kernel<<<blocks(n), 256, 0, st>>>(values, b, n, 1, 0);
      p->launches += 2;
    }
  }
  p->step++;
  PCK(cudaGetLastError());
  return MYO_OK;
}

}  // namespace

extern "C" {

int myo_policy_create(const myo_policy_cfg* cfg, int max_batch, int device, myo_policy** out) {
  if (!cfg || !out || max_batch <= 0) { myo::set_error("bad argument to myo_policy_create"); return MYO_E_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
    myo::set_error("no CUDA device available (the policy kernels have no CPU path)");
    return MYO_E_CUDA;
  }
  const int H = cfg->lstm_hidden;
  if (H <= 0 || H % 64 || H > 256) { myo::set_error("lstm_hidden must be 64, 128, 192 or 256"); return MYO_E_LIMIT; }
  if (cfg->obs_dim <= 0 || cfg->obs_dim > 128) { myo::set_error("obs_dim must be in 1..128"); return MYO_E_LIMIT; }
  if (cfg->act_dim <= 0 || cfg->act_dim > 256) { myo::set_error("act_dim must be in 1..256"); return MYO_E_LIMIT; }
  if (cfg->n_pi_layers < 0 || cfg->n_pi_layers > 4 || cfg->n_vf_layers < 0 || cfg->n_vf_layers > 4) { myo::set_error("at most 4 MLP layers per head"); return MYO_E_LIMIT; }
  for (int l = 0; l < cfg->n_pi_layers; l++) if (cfg->pi_layers[l] <= 0 || cfg->pi_layers[l] % 16 || cfg->pi_layers[l] > 256) { myo::set_error("MLP widths must be multiples of 16 up to 256"); return MYO_E_LIMIT; }
  for (int l = 0; l < cfg->n_vf_layers; l++) if (cfg->vf_layers[l] <= 0 || cfg->vf_layers[l] % 16 || cfg->vf_layers[l] > 256) { myo::set_error("MLP widths must be multiples of 16 up to 256"); return MYO_E_LIMIT; }
  PCK(cudaSetDevice(device));
  myo_policy* p = new myo_policy();
  p->cfg = *cfg; p->device = device; p->max_batch = max_batch; p->obs_pad = round_up(cfg->obs_dim, 16);
  for (int net = 0; net < 2; net++) {
    build_program(p, net, p->prog[net], p->wbytes[net], p->nbias[net]);
    if (cudaMalloc(&p->wpack[net], p->wbytes[net]) != cudaSuccess || cudaMalloc(&p->bias[net], sizeof(float) * p->nbias[net]) != cudaSuccess) {
      myo::set_error("policy weight allocation failed");
      myo_policy_destroy(p);
      return MYO_E_CUDA;
    }
  }
  if (cudaMalloc(&p->log_std, sizeof(float) * cfg->act_dim) != cudaSuccess || cudaMalloc(&p->obs_mean, sizeof(float) * cfg->obs_dim) != cudaSuccess ||
      cudaMalloc(&p->obs_inv_std, sizeof(float) * cfg->obs_dim) != cudaSuccess) {
    myo::set_error("policy allocation failed");
    myo_policy_destroy(p);
    return MYO_E_CUDA;
  }
  if (cudaFuncSetAttribute(policy_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess) {
    myo::set_error("policy kernel needs 222 KB of shared memory per CTA");
    myo_policy_destroy(p);
    return MYO_E_CUDA;
  }
  *out = p;
  return MYO_OK;
}

void myo_policy_destroy(myo_policy* p) {
  if (!p) return;
  cudaSetDevice(p->device);
  for (auto& kv : p->weights) cudaFree(kv.second);
  for (int net = 0; net < 2; net++) { cudaFree(p->wpack[net]); cudaFree(p->bias[net]); }
  cudaFree(p->log_std); cudaFree(p->obs_mean); cudaFree(p->obs_inv_std);
  cudaFree(p->f32_scratch);
  if (p->blas) cublasDestroy(p->blas);
  delete p;
}

int myo_policy_set_weight(myo_policy* p, const char* name, const float* data_dev, int64_t numel, void* stream) {
  if (!p || !name || !data_dev || numel <= 0) { myo::set_error("bad argument to myo_policy_set_weight"); return MYO_E_ARG; }
  PCK(cudaSetDevice(p->device));
  const std::string key(name);
  auto it = p->weights.find(key);
  if (it != p->weights.end() && p->numel[key] != numel) { cudaFree(it->second); p->weights.erase(it); it = p->weights.end(); }
  if (it == p->weights.end()) {
    float* q = nullptr;
    PCK(cudaMalloc(&q, sizeof(float) * numel));
    p->weights[key] = q; p->numel[key] = numel;
  }
  PCK(cudaMemcpyAsync(p->weights[key], data_dev, sizeof(float) * numel, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  p->dirty = true;
  return MYO_OK;
}

int myo_policy_set_obs_norm(myo_policy* p, const float* mean_dev, const float* var_dev, float epsilon, float clip_obs, void* stream) {
  if (!p) { myo::set_error("null policy"); return MYO_E_ARG; }
  PCK(cudaSetDevice(p->device));
  if (!mean_dev || !var_dev) { p->has_norm = false; return MYO_OK; }
  inv_std_kernel<<<(p->cfg.obs_dim + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(p->obs_mean, p->obs_inv_std, mean_dev, var_dev, epsilon, p->cfg.obs_dim);
  p->launches++;
  PCK(cudaGetLastError());
  p->has_norm = true; p->clip_obs = clip_obs;
  return MYO_OK;
}

int myo_policy_set_latent_out(myo_policy* p, float* latent_dev) {
  if (!p) { myo::set_error("null policy"); return MYO_E_ARG; }
  p->latent_out = latent_dev;
  return MYO_OK;
}

int myo_policy_set_precision(myo_policy* p, int precision) {
  if (!p || (precision != 0 && precision != 1)) { myo::set_error("precision: 0 (bf16 operands on the tensor cores) or 1 (fp32)"); return MYO_E_ARG; }
  p->precision = precision;
  return MYO_OK;
}

int myo_policy_seed(myo_policy* p, uint64_t seed) {
  if (!p) { myo::set_error("null policy"); return MYO_E_ARG; }
  p->seed = seed; p->step = 0;
  return MYO_OK;
}

int myo_policy_forward(myo_policy* p, int n, const float* obs_dev, float* h_dev, float* c_dev, const uint8_t* episode_start_dev,
                       const float* noise_dev, float* actions_dev, float* values_dev, float* logp_dev, void* stream) {
  if (!p || n <= 0 || !obs_dev || !h_dev || !c_dev || !episode_start_dev || !actions_dev) { myo::set_error("bad argument to myo_policy_forward"); return MYO_E_ARG; }
  if (n > p->max_batch) { myo::set_error("batch exceeds max_batch given to myo_policy_create"); return MYO_E_ARG; }
  PCK(cudaSetDevice(p->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (p->precision == 1) return forward_fp32(p, n, obs_dev, h_dev, c_dev, episode_start_dev, noise_dev, actions_dev, values_dev, logp_dev, st);
  if (p->dirty) { int rc = pack_weights(p, st); if (rc) return rc; }
  FwdArgs a{};
  a.n = n; a.obs_dim = p->cfg.obs_dim; a.obs_pad = p->obs_pad; a.H = p->cfg.lstm_hidden; a.act_dim = p->cfg.act_dim;
  a.obs = obs_dev; a.h = h_dev; a.c = c_dev; a.start = episode_start_dev; a.noise = noise_dev;
  a.actions = actions_dev; a.values = values_dev; a.logp = logp_dev;
  a.wpack[0] = p->wpack[0]; a.wpack[1] = p->wpack[1]; a.bias[0] = p->bias[0]; a.bias[1] = p->bias[1];
  a.log_std = p->log_std;
  a.obs_mean = p->has_norm ? p->obs_mean : nullptr; a.obs_inv_std = p->has_norm ? p->obs_inv_std : nullptr; a.clip_obs = p->clip_obs;
  a.seed = p->seed; a.step = p->step++;
  a.latent = (p->cfg.n_pi_layers > 0) ? p->latent_out : nullptr;
  a.latent_dim = p->cfg.n_pi_layers > 0 ? p->cfg.pi_layers[p->cfg.n_pi_layers - 1] : p->cfg.lstm_hidden;
  dim3 grid((n + TILE_M - 1) / TILE_M, 2);
  policy_forward_kernel<<<grid, THREADS, SMEM_BYTES, st>>>(a, p->prog[0], p->prog[1]);
  p->launches++;
  PCK(cudaGetLastError());
  return MYO_OK;
}

int myo_sde_reset_noise(uint16_t* noise_mat_dev, float* std2_dev, const float* log_std_dev, int n, int latent_dim, int act_dim, uint64_t seed,
                        uint32_t epoch, void* stream) {
  if (!noise_mat_dev || !std2_dev || !log_std_dev || n <= 0 || latent_dim <= 0 || act_dim <= 0) { myo::set_error("bad argument to myo_sde_reset_noise"); return MYO_E_ARG; }
  const int LA = latent_dim * act_dim;
  const long long total = (long long)n * ((LA + 1) / 2);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  sde_reset_noise_kernel<<<(int)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<__nv_bfloat16*>(noise_mat_dev), std2_dev, log_std_dev, n, LA,
                                                                                    seed, epoch);
  PCK(cudaGetLastError());
  return MYO_OK;
}

int myo_sde_sample(const float* latent_dev, int latent_ld, const uint16_t* noise_mat_dev, const float* std2_dev, float* actions_dev, float* logp_dev,
                   int n, int latent_dim, int act_dim, void* stream) {
  if (!latent_dev || !noise_mat_dev || !std2_dev || !actions_dev || n <= 0 || latent_dim <= 0 || act_dim <= 0 || act_dim > 64 || latent_ld < latent_dim) {
    myo::set_error("bad argument to myo_sde_sample (act_dim <= 64)");
    return MYO_E_ARG;
  }
  sde_sample_kernel<<<(n * 32 + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(latent_dev, latent_ld, reinterpret_cast<const __nv_bfloat16*>(noise_mat_dev),
                                                                                        std2_dev, actions_dev, logp_dev, n, latent_dim, act_dim);
  PCK(cudaGetLastError());
  return MYO_OK;
}

int64_t myo_policy_launch_count(const myo_policy* p) { return p ? p->launches : 0; }

}  // extern "C"
