// PPO update of the recurrent policy on the device (SURVEY.md 8a row a18, 8f rank 1): what sb3-contrib's
// RecurrentPPO.train() does per minibatch - evaluate_actions over whole sequences (LSTM from the stored states,
// episode starts zero the state), advantage normalisation, clipped surrogate + value + entropy loss, backward
// (BPTT), clip_grad_norm_, Adam - reached from /root/reference/src/train/trainer.py:67-71 with the
// hyper-parameters of /root/reference/docs/summary.md:86-117.
//
// Design (not sb3's): a minibatch is a set of B worlds, each with its whole T-step sequence, stored step-major
// (row m = t * B + b). sb3-contrib splits sequences at episode starts and pads; here the sequences stay whole and
// the state is multiplied by (1 - episode_start) inside the recurrence, which is the same function and the same
// gradient (no gradient crosses a reset) without padding. GEMMs are plain library GEMMs (cuBLAS, bf16 operands with
// fp32 accumulation as in the rollout kernel, or fp32 for the parity tests); everything between them - gathers, LSTM
// cell forward / backward, bias + ReLU, the loss and its gradient, column sums, gradient-norm clipping and Adam - is
// hand-written here. The gradient leaves as one flat fp32 bucket so the cross-rank exchange is a single all-reduce.
//
// Reference semantics (third-party, restated in oracle/ppo_oracle.py):
//   sb3_contrib/ppo_recurrent/ppo_recurrent.py  RecurrentPPO.train
//   sb3_contrib/common/recurrent/policies.py    RecurrentActorCriticPolicy.evaluate_actions / _process_sequence
//   stable_baselines3/common/distributions.py   DiagGaussianDistribution.log_prob / entropy
//   torch.nn.utils.clip_grad_norm_, torch.optim.Adam
#include <cublas_v2.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/myo_b200.h"
#include "myo_lstm_seq.hpp"

namespace myo { void set_error(const std::string& msg); }

namespace {

#define QCK(call)                                                                 \
  do {                                                                            \
    cudaError_t e_ = (call);                                                      \
    if (e_ != cudaSuccess) {                                                      \
      myo::set_error(std::string(#call) + ": " + cudaGetErrorString(e_));        \
      return MYO_E_CUDA;                                                          \
    }                                                                             \
  } while (0)
#define BCK(call)                                                                 \
  do {                                                                            \
    cublasStatus_t s_ = (call);                                                   \
    if (s_ != CUBLAS_STATUS_SUCCESS) {                                            \
      myo::set_error(std::string(#call) + ": cuBLAS status " + std::to_string((int)s_)); \
      return MYO_E_CUDA;                                                          \
    }                                                                             \
  } while (0)
#define RCK(call) do { int rc_ = (call); if (rc_) return rc_; } while (0)

typedef __nv_bfloat16 bf16;
constexpr int kStatSlots = 8;          // policy_loss value_loss entropy_loss approx_kl clip_fraction loss adv_mean adv_std
constexpr int kLossBlocks = 592;       // 4 x 148 CTAs, grid-stride over rows; partial sums merged in CTA order
constexpr int kColsumRows = 296;       // row chunks of the two-stage column sum
constexpr int kNormBlocks = 296;
constexpr size_t kBlasWorkspace = 64u << 20;   // per cuBLAS handle (the library's own default for this architecture class is 32 MiB)

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

template <typename T> __device__ __forceinline__ T to_op(float x);
template <> __device__ __forceinline__ float to_op<float>(float x) { return x; }
template <> __device__ __forceinline__ bf16 to_op<bf16>(float x) { return __float2bfloat16_rn(x); }
__device__ __forceinline__ float from_op(float x) { return x; }
__device__ __forceinline__ float from_op(bf16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// ---- operand copies of the weights: fp32 [rows][cols] -> OpT [rows_pad][cols_pad], zero padded -----------------
template <typename T>
__global__ void convert_pad_kernel(const float* __restrict__ src, T* __restrict__ dst, int rows, int cols, int rows_pad, int cols_pad) {
  const int64_t total = (int64_t)rows_pad * cols_pad;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols_pad), c = (int)(i % cols_pad);
    dst[i] = to_op<T>((r < rows && c < cols) ? src[(int64_t)r * cols + c] : 0.f);
  }
}

// ---- minibatch gather: rows m = t * B + b from the step-major rollout buffers [T][n][.] -------------------------
template <typename T>
__global__ void gather_rows_kernel(int Tn, int B, int n, int O, int Op, int A, const int32_t* __restrict__ idx,
                                   const float* __restrict__ obs, const float* __restrict__ actions, const uint8_t* __restrict__ starts,
                                   const float* __restrict__ old_values, const float* __restrict__ old_logp, const float* __restrict__ adv,
                                   const float* __restrict__ ret, T* __restrict__ X, float* __restrict__ act, float* __restrict__ keep,
                                   float* __restrict__ ov, float* __restrict__ ol, float* __restrict__ ad, float* __restrict__ rt) {
  const int warps = (gridDim.x * blockDim.x) >> 5, lane = threadIdx.x & 31;
  const int M = Tn * B;
  for (int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; m < M; m += warps) {
    const int t = m / B, b = m - t * B;
    const int64_t src = (int64_t)t * n + idx[b];
    for (int j = lane; j < Op; j += 32) X[(int64_t)m * Op + j] = to_op<T>(j < O ? obs[src * O + j] : 0.f);
    for (int j = lane; j < A; j += 32) act[(int64_t)m * A + j] = actions[src * A + j];
    if (lane == 0) {
      keep[m] = starts[src] ? 0.f : 1.f;
      ov[m] = old_values[src]; ol[m] = old_logp[src]; ad[m] = adv[src]; rt[m] = ret[src];
    }
  }
}

// initial LSTM state of one net for the minibatch worlds, already multiplied by keep_0:
//   HP[0][b][:] = keep_0 h0[idx[b]][:]   (operand of the first recurrent GEMM),  C0[b][:] = keep_0 c0[idx[b]][:]
template <typename T>
__global__ void gather_state_kernel(int B, int H, const int32_t* __restrict__ idx, const float* __restrict__ h0, const float* __restrict__ c0,
                                    const float* __restrict__ keep, T* __restrict__ HP, float* __restrict__ C0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H) return;
  const int b = i / H, j = i - b * H;
  const int64_t src = (int64_t)idx[b] * H + j;
  HP[i] = to_op<T>(keep[b] * h0[src]);
  C0[i] = keep[b] * c0[src];
}

// four consecutive elements at once (H is a multiple of 8, rows are 16-byte aligned)
__device__ __forceinline__ void store4(float* p, float a, float b, float c, float d) { *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d); }
__device__ __forceinline__ void store4(bf16* p, float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 v;
  v.x = *reinterpret_cast<uint32_t*>(&lo); v.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = v;
}
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 add4(float4 a, float4 b, float4 c) { return make_float4(a.x + b.x + c.x, a.y + b.y + c.y, a.z + b.z + c.z, a.w + b.w + c.w); }

// ---- LSTM cell, step t of the sequence forward (torch gate order i f g o) -------------------------------------------
// G[t]: x W_ih^T + h_prev W_hh^T (no bias yet) -> activated gates in place; Cs[t] = c_t; Hs[t] = h_t;
// HP[t+1] = keep_{t+1} h_t (operand of the next recurrent GEMM). A thread owns four consecutive units of one world.
template <typename T>
__global__ void lstm_cell_fwd_kernel(int t, int Tn, int B, int H, float* __restrict__ G, const float* __restrict__ bih, const float* __restrict__ bhh,
                                     const float* __restrict__ keep, const float* __restrict__ C0, float* __restrict__ Cs,
                                     T* __restrict__ Hs, T* __restrict__ HP) {
  const int i4 = blockIdx.x * blockDim.x + threadIdx.x;
  const int H4 = H >> 2;
  if (i4 >= B * H4) return;
  const int b = i4 / H4, j = (i4 - b * H4) << 2;
  const int64_t m = (int64_t)t * B + b;
  float* g = G + m * 4 * H;
  const float4 pi = add4(ld4(g + j), ld4(bih + j), ld4(bhh + j));
  const float4 pf = add4(ld4(g + H + j), ld4(bih + H + j), ld4(bhh + H + j));
  const float4 pg = add4(ld4(g + 2 * H + j), ld4(bih + 2 * H + j), ld4(bhh + 2 * H + j));
  const float4 po = add4(ld4(g + 3 * H + j), ld4(bih + 3 * H + j), ld4(bhh + 3 * H + j));
  float4 cp = t == 0 ? ld4(C0 + (int64_t)b * H + j) : ld4(Cs + (m - B) * H + j);
  if (t > 0) { const float k = keep[m]; cp.x *= k; cp.y *= k; cp.z *= k; cp.w *= k; }
  const float kn = t + 1 < Tn ? keep[m + B] : 0.f;
  float gi[4] = {pi.x, pi.y, pi.z, pi.w}, gf[4] = {pf.x, pf.y, pf.z, pf.w}, gg[4] = {pg.x, pg.y, pg.z, pg.w}, go[4] = {po.x, po.y, po.z, po.w};
  const float cpv[4] = {cp.x, cp.y, cp.z, cp.w};
  float c[4], h[4];
#pragma unroll
  for (int q = 0; q < 4; q++) {
    gi[q] = sigmoidf_(gi[q]); gf[q] = sigmoidf_(gf[q]); gg[q] = tanhf(gg[q]); go[q] = sigmoidf_(go[q]);
    c[q] = gf[q] * cpv[q] + gi[q] * gg[q];
    h[q] = go[q] * tanhf(c[q]);
  }
  store4(g + j, gi[0], gi[1], gi[2], gi[3]); store4(g + H + j, gf[0], gf[1], gf[2], gf[3]);
  store4(g + 2 * H + j, gg[0], gg[1], gg[2], gg[3]); store4(g + 3 * H + j, go[0], go[1], go[2], go[3]);
  store4(Cs + m * H + j, c[0], c[1], c[2], c[3]);
  store4(Hs + m * H + j, h[0], h[1], h[2], h[3]);
  if (t + 1 < Tn) store4(HP + (m + B) * H + j, kn * h[0], kn * h[1], kn * h[2], kn * h[3]);
}

// step t of the backward recurrence. dHs: dL/dh_t from the layers above; dh_carry = dG_{t+1} W_hh (not yet masked);
// dc_carry = dL/dc_t through c_{t+1} (already masked). Writes dG_t (gate pre-activations) and the new dc_carry.
template <typename T>
__global__ void lstm_cell_bwd_kernel(int t, int Tn, int B, int H, const float* __restrict__ G, const float* __restrict__ keep,
                                     const float* __restrict__ C0, const float* __restrict__ Cs, const float* __restrict__ dHs,
                                     const float* __restrict__ dh_carry, float* __restrict__ dc_carry, T* __restrict__ dG) {
  const int i4 = blockIdx.x * blockDim.x + threadIdx.x;
  const int H4 = H >> 2;
  if (i4 >= B * H4) return;
  const int b = i4 / H4, j = (i4 - b * H4) << 2;
  const int64_t m = (int64_t)t * B + b, bo = (int64_t)b * H + j;
  const float* g = G + m * 4 * H;
  const float4 vi = ld4(g + j), vf = ld4(g + H + j), vg = ld4(g + 2 * H + j), vo = ld4(g + 3 * H + j);
  const float4 vdh = ld4(dHs + m * H + j), vc = ld4(Cs + m * H + j);
  float4 vcar = make_float4(0.f, 0.f, 0.f, 0.f), vdc = vcar;
  float kn = 0.f;
  if (t + 1 < Tn) { vcar = ld4(dh_carry + bo); vdc = ld4(dc_carry + bo); kn = keep[m + B]; }
  float4 vcp = t == 0 ? ld4(C0 + bo) : ld4(Cs + (m - B) * H + j);
  const float k = keep[m];
  if (t > 0) { vcp.x *= k; vcp.y *= k; vcp.z *= k; vcp.w *= k; }
  const float gi[4] = {vi.x, vi.y, vi.z, vi.w}, gf[4] = {vf.x, vf.y, vf.z, vf.w}, gg[4] = {vg.x, vg.y, vg.z, vg.w}, go[4] = {vo.x, vo.y, vo.z, vo.w};
  const float dhs[4] = {vdh.x, vdh.y, vdh.z, vdh.w}, cs[4] = {vc.x, vc.y, vc.z, vc.w}, car[4] = {vcar.x, vcar.y, vcar.z, vcar.w};
  const float dcs[4] = {vdc.x, vdc.y, vdc.z, vdc.w}, cp[4] = {vcp.x, vcp.y, vcp.z, vcp.w};
  float di[4], df[4], dg[4], dO[4], dcn[4];
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const float dh = dhs[q] + kn * car[q];
    const float tc = tanhf(cs[q]);
    const float dc = dcs[q] + dh * go[q] * (1.f - tc * tc);
    di[q] = dc * gg[q] * gi[q] * (1.f - gi[q]);
    df[q] = dc * cp[q] * gf[q] * (1.f - gf[q]);
    dg[q] = dc * gi[q] * (1.f - gg[q] * gg[q]);
    dO[q] = dh * tc * go[q] * (1.f - go[q]);
    dcn[q] = dc * gf[q] * k;
  }
  T* d = dG + m * 4 * H;
  store4(d + j, di[0], di[1], di[2], di[3]); store4(d + H + j, df[0], df[1], df[2], df[3]);
  store4(d + 2 * H + j, dg[0], dg[1], dg[2], dg[3]); store4(d + 3 * H + j, dO[0], dO[1], dO[2], dO[3]);
  store4(dc_carry + bo, dcn[0], dcn[1], dcn[2], dcn[3]);
}

// The same backward step on the activation records the persistent forward kernel writes (myo_lstm_seq.cu: per (row, 8 units)
// the activated gates i f g o as 8 x bf16 each, then c_t as 8 x fp32). A thread owns one record.
__device__ __forceinline__ void unpack8(const uint4 v, float* o) {
  const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int q = 0; q < 4; q++) { o[2 * q] = __low2float(p[q]); o[2 * q + 1] = __high2float(p[q]); }
}
__device__ __forceinline__ uint4 pack8(const float* x) {
  uint4 v;
  __nv_bfloat162 a = __floats2bfloat162_rn(x[0], x[1]), b = __floats2bfloat162_rn(x[2], x[3]), c = __floats2bfloat162_rn(x[4], x[5]), d = __floats2bfloat162_rn(x[6], x[7]);
  v.x = *reinterpret_cast<uint32_t*>(&a); v.y = *reinterpret_cast<uint32_t*>(&b); v.z = *reinterpret_cast<uint32_t*>(&c); v.w = *reinterpret_cast<uint32_t*>(&d);
  return v;
}
__global__ void lstm_cell_bwd_rec_kernel(int t, int Tn, int B, int H, const uint8_t* __restrict__ Rec, const float* __restrict__ keep,
                                         const float* __restrict__ C0, const float* __restrict__ dHs, const float* __restrict__ dh_carry,
                                         float* __restrict__ dc_carry, bf16* __restrict__ dG) {
  const int i8 = blockIdx.x * blockDim.x + threadIdx.x;
  const int H8 = H >> 3;
  if (i8 >= B * H8) return;
  const int b = i8 / H8, j = (i8 - b * H8) << 3;
  const int64_t m = (int64_t)t * B + b, bo = (int64_t)b * H + j;
  const uint8_t* rec = Rec + (m * H8 + (j >> 3)) * myo::kLstmRecBytes;
  const uint4* rg = reinterpret_cast<const uint4*>(rec);
  float gi[8], gf[8], gg[8], go[8], cs[8], cp[8], dhs[8], car[8], dcs[8];
  unpack8(rg[0], gi); unpack8(rg[1], gf); unpack8(rg[2], gg); unpack8(rg[3], go);
  auto ld8 = [](const float* p, float* o) { const float4 a = ld4(p), c = ld4(p + 4); o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = c.x; o[5] = c.y; o[6] = c.z; o[7] = c.w; };
  ld8(reinterpret_cast<const float*>(rec + 64), cs);
  ld8(dHs + m * H + j, dhs);
  const float k = keep[m];
  float kn = 0.f;
  if (t + 1 < Tn) { ld8(dh_carry + bo, car); ld8(dc_carry + bo, dcs); kn = keep[m + B]; }
  else {
#pragma unroll
    for (int q = 0; q < 8; q++) { car[q] = 0.f; dcs[q] = 0.f; }
  }
  if (t == 0) ld8(C0 + bo, cp);
  else {
    ld8(reinterpret_cast<const float*>(rec - (int64_t)B * H8 * myo::kLstmRecBytes + 64), cp);
#pragma unroll
    for (int q = 0; q < 8; q++) cp[q] *= k;
  }
  float di[8], df[8], dg[8], dO[8], dcn[8];
#pragma unroll
  for (int q = 0; q < 8; q++) {
    const float dh = dhs[q] + kn * car[q];
    const float tc = tanhf(cs[q]);
    const float dc = dcs[q] + dh * go[q] * (1.f - tc * tc);
    di[q] = dc * gg[q] * gi[q] * (1.f - gi[q]);
    df[q] = dc * cp[q] * gf[q] * (1.f - gf[q]);
    dg[q] = dc * gi[q] * (1.f - gg[q] * gg[q]);
    dO[q] = dh * tc * go[q] * (1.f - go[q]);
    dcn[q] = dc * gf[q] * k;
  }
  bf16* d = dG + m * 4 * H;
  *reinterpret_cast<uint4*>(d + j) = pack8(di); *reinterpret_cast<uint4*>(d + H + j) = pack8(df);
  *reinterpret_cast<uint4*>(d + 2 * H + j) = pack8(dg); *reinterpret_cast<uint4*>(d + 3 * H + j) = pack8(dO);
  store4(dc_carry + bo, dcn[0], dcn[1], dcn[2], dcn[3]); store4(dc_carry + bo + 4, dcn[4], dcn[5], dcn[6], dcn[7]);
}

// ---- MLP glue ----------------------------------------------------------------------------------------------------------
// four elements per thread (widths are multiples of 8, buffers 16-byte aligned)
template <typename T>
__global__ void bias_relu_kernel(const float* __restrict__ Z, const float* __restrict__ bias, T* __restrict__ A, int64_t total, int W) {
  const int64_t n4 = total >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 z = ld4(Z + 4 * i), bb = ld4(bias + (4 * i) % W);
    store4(A + 4 * i, fmaxf(z.x + bb.x, 0.f), fmaxf(z.y + bb.y, 0.f), fmaxf(z.z + bb.z, 0.f), fmaxf(z.w + bb.w, 0.f));
  }
}
__device__ __forceinline__ float4 ld4op(const float* p) { return ld4(p); }
__device__ __forceinline__ float4 ld4op(const bf16* p) {
  const uint2 v = *reinterpret_cast<const uint2*>(p);
  const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&v.x), hi = *reinterpret_cast<const __nv_bfloat162*>(&v.y);
  return make_float4(__low2float(lo), __high2float(lo), __low2float(hi), __high2float(hi));
}
template <typename T>
__global__ void relu_bwd_kernel(const float* __restrict__ dA, const T* __restrict__ A, T* __restrict__ dZ, int64_t total) {
  const int64_t n4 = total >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 d = ld4(dA + 4 * i), a = ld4op(A + 4 * i);
    store4(dZ + 4 * i, a.x > 0.f ? d.x : 0.f, a.y > 0.f ? d.y : 0.f, a.z > 0.f ? d.z : 0.f, a.w > 0.f ? d.w : 0.f);
  }
}

// column sums of Y[M][ld] (first N columns) -> part[chunk][N], then out[N] (and out2[N] if given): two stages, fixed order
template <typename T>
__global__ void colsum_partial_kernel(const T* __restrict__ Y, int64_t M, int N, int ld, float* __restrict__ part) {
  __shared__ float s[8][33];
  const int col = blockIdx.x * 32 + threadIdx.x;
  const int64_t rows_per = (M + gridDim.y - 1) / gridDim.y;
  const int64_t r0 = blockIdx.y * rows_per, r1 = min(M, r0 + rows_per);
  float acc = 0.f;
  if (col < N)
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) acc += from_op(Y[r * ld + col]);
  s[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && col < N) {
    for (int k = 1; k < 8; k++) acc += s[k][threadIdx.x];
    part[(int64_t)blockIdx.y * N + col] = acc;
  }
}
__global__ void colsum_final_kernel(const float* __restrict__ part, int chunks, int N, float* __restrict__ out, float* __restrict__ out2) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= N) return;
  float acc = 0.f;
  for (int k = 0; k < chunks; k++) acc += part[(int64_t)k * N + col];
  out[col] = acc;
  if (out2) out2[col] = acc;
}

// ---- loss ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// mean and unbiased std of the gathered advantages (torch: advantages.mean(), advantages.std()); one CTA, fp64 sums
__global__ void adv_stats_kernel(const float* __restrict__ adv, int64_t M, float* __restrict__ out) {
  __shared__ double s1[32], s2[32];
  double a = 0.0, q = 0.0;
  for (int64_t i = threadIdx.x; i < M; i += blockDim.x) { const double v = adv[i]; a += v; q += v * v; }
  a = warp_sum_d(a); q = warp_sum_d(q);
  if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a; s2[threadIdx.x >> 5] = q; }
  __syncthreads();
  if (threadIdx.x == 0) {
    a = 0.0; q = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) { a += s1[k]; q += s2[k]; }
    const double mean = a / (double)M;
    const double var = M > 1 ? fmax(q - a * mean, 0.0) / (double)(M - 1) : 0.0;
    out[0] = (float)mean; out[1] = (float)sqrt(var);
  }
}

// gSDE helpers: lat2 = latent^2 (operand of the variance GEMM), S2 = exp(2 log_std) zero-padded to [d][Ap]
template <typename T>
__global__ void square_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = from_op(x[i]);
    y[i] = to_op<T>(v * v);
  }
}
template <typename T>
__global__ void sde_std2_kernel(const float* __restrict__ log_std, T* __restrict__ S2, int d, int A, int Ap) {
  const int total = d * Ap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int l = i / Ap, k = i - l * Ap;
    S2[i] = to_op<T>(k < A ? expf(2.f * log_std[l * A + k]) : 0.f);
  }
}
// dL/dlog_std[l][k] = dL/dS2[l][k] * 2 exp(2 log_std[l][k])
__global__ void sde_logstd_grad_kernel(const float* __restrict__ dS2, const float* __restrict__ log_std, float* __restrict__ g, int d, int A, int Ap) {
  const int total = d * A;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int l = i / A, k = i - l * A;
    g[i] = dS2[l * Ap + k] * 2.f * expf(2.f * log_std[i]);
  }
}

struct LossArgs {
  int64_t M; int A, Ap;
  const float* var_raw;    // gSDE: [M][Ap] latent^2 . exp(2 log_std) (null: state-independent log_std[A])
  float ent_coef;
  const float* mean_raw;   // [M][Ap] action_net output without bias
  const float* ba;         // action_net.bias
  const float* log_std;
  const float* act; const float* old_logp; const float* adv; const float* adv_stats;
  float clip_range; int normalize_adv;
};

// policy part: one warp per row. dMEAN[m][k] = g_m z_k / sigma_k, partial sums of dlog_std and the statistics.
// part layout per CTA: [0] policy_loss [1] approx_kl [2] clip_fraction, [kStatSlots + k] dlog_std_k
template <typename T>
__global__ void policy_loss_kernel(LossArgs a, T* __restrict__ dMEAN, T* __restrict__ Q, float* __restrict__ part) {
  extern __shared__ float sh[];      // [warps][kStatSlots + A]
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int W = kStatSlots + a.A;
  float* mine = sh + wib * W;
  for (int k = lane; k < W; k += 32) mine[k] = 0.f;
  __syncwarp();
  const float invM = 1.f / (float)a.M;
  const float amean = a.normalize_adv ? a.adv_stats[0] : 0.f, ainv = a.normalize_adv ? 1.f / (a.adv_stats[1] + 1e-8f) : 1.f;
  float pl = 0.f, kl = 0.f, cf = 0.f;
  const bool sde = a.var_raw != nullptr;
  float ent = 0.f;
  for (int64_t m = (int64_t)blockIdx.x * nw + wib; m < a.M; m += (int64_t)gridDim.x * nw) {
    float lp = 0.f, en = 0.f;
    for (int k = lane; k < a.A; k += 32) {
      const float dlt = a.act[m * a.A + k] - (a.mean_raw[m * a.Ap + k] + a.ba[k]);
      if (sde) {
        const float v = a.var_raw[m * a.Ap + k] + 1e-6f;
        lp += -0.5f * dlt * dlt / v - 0.5f * logf(v) - 0.9189385332046727f;
        en += 1.4189385332046727f + 0.5f * logf(v);
      } else {
        const float ls = a.log_std[k];
        const float z = dlt * expf(-ls);
        lp += -0.5f * z * z - ls - 0.9189385332046727f;
      }
    }
    lp = warp_sum(lp);
    if (sde) ent += warp_sum(en);
    const float adv = (a.adv[m] - amean) * ainv;
    const float lr = lp - a.old_logp[m];
    const float ratio = expf(lr);
    const float u = adv * ratio, v = adv * fminf(fmaxf(ratio, 1.f - a.clip_range), 1.f + a.clip_range);
    const bool active = !(v < u);        // torch.min(u, v): the gradient reaches the ratio unless the clipped branch is the strict minimum
    const float g = active ? -adv * ratio * invM : 0.f;
    pl -= fminf(u, v); kl += (ratio - 1.f) - lr; cf += fabsf(ratio - 1.f) > a.clip_range ? 1.f : 0.f;
    for (int k = lane; k < a.Ap; k += 32) {
      float d = 0.f, q = 0.f;
      if (k < a.A) {
        const float dlt = a.act[m * a.A + k] - (a.mean_raw[m * a.Ap + k] + a.ba[k]);
        if (sde) {
          const float iv = 1.f / (a.var_raw[m * a.Ap + k] + 1e-6f);
          d = g * dlt * iv;
          q = 0.5f * (g * (dlt * dlt * iv - 1.f) - a.ent_coef * invM) * iv;     // dL/dsigma^2: log-prob and entropy terms
        } else {
          const float is = expf(-a.log_std[k]);
          const float z = dlt * is;
          d = g * z * is;
          mine[kStatSlots + k] += g * (z * z - 1.f);
        }
      }
      dMEAN[m * a.Ap + k] = to_op<T>(d);
      if (sde) Q[m * a.Ap + k] = to_op<T>(q);
    }
  }
  if (lane == 0) mine[3] = ent;
  if (lane == 0) { mine[0] = pl; mine[1] = kl; mine[2] = cf; }
  __syncthreads();
  for (int k = threadIdx.x; k < W; k += blockDim.x) {
    float acc = 0.f;
    for (int w = 0; w < nw; w++) acc += sh[w * W + k];
    part[(int64_t)blockIdx.x * W + k] = acc;
  }
}

// value part: v = raw + bias; optional clipping around the old value; dV = vf_coef * 2 (v_pred - ret) / M
template <typename T>
__global__ void value_loss_kernel(int64_t M, const float* __restrict__ vraw, const float* __restrict__ bv, const float* __restrict__ old_values,
                                  const float* __restrict__ ret, float clip_range_vf, float vf_coef, T* __restrict__ dV, float* __restrict__ part) {
  __shared__ float s[32];
  float vl = 0.f;
  const float invM = 1.f / (float)M;
  for (int64_t m = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; m < M; m += (int64_t)gridDim.x * blockDim.x) {
    float v = vraw[m] + bv[0];
    float pass = 1.f;
    if (clip_range_vf > 0.f) {
      const float dv = v - old_values[m];
      pass = fabsf(dv) <= clip_range_vf ? 1.f : 0.f;
      v = old_values[m] + fminf(fmaxf(dv, -clip_range_vf), clip_range_vf);
    }
    const float e = v - ret[m];
    vl += e * e;
    dV[m] = to_op<T>(vf_coef * 2.f * e * invM * pass);
  }
  vl = warp_sum(vl);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = vl;
  __syncthreads();
  if (threadIdx.x == 0) {
    vl = 0.f;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) vl += s[k];
    part[blockIdx.x] = vl;
  }
}

// merges the CTA partials in CTA order; writes the statistics and the log_std gradient
__global__ void loss_finalize_kernel(const float* __restrict__ ppart, int pblocks, const float* __restrict__ vpart, int vblocks, int A, int64_t M,
                                     const float* __restrict__ log_std, const float* __restrict__ adv_stats, float ent_coef, float vf_coef,
                                     float* __restrict__ stats, float* __restrict__ dlog_std, int sde) {
  const int W = kStatSlots + A;
  __shared__ float s[kStatSlots];
  const float invM = 1.f / (float)M;
  for (int k = threadIdx.x; k < W; k += blockDim.x) {
    float acc = 0.f;
    for (int b = 0; b < pblocks; b++) acc += ppart[(int64_t)b * W + k];
    if (k < kStatSlots) s[k] = acc;
    else if (!sde) dlog_std[k - kStatSlots] = acc - ent_coef;      // d(-ent_coef * mean entropy) / dlog_std_k = -ent_coef
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float vl = 0.f;
    for (int b = 0; b < vblocks; b++) vl += vpart[b];
    float ent = 0.f;
    if (sde) ent = s[3] * invM;       // per-sample entropies, summed by the loss kernel
    else for (int k = 0; k < A; k++) ent += 1.4189385332046727f + log_std[k];
    const float pl = s[0] * invM, value_loss = vl * invM, entropy_loss = -ent;
    stats[0] = pl; stats[1] = value_loss; stats[2] = entropy_loss; stats[3] = s[1] * invM; stats[4] = s[2] * invM;
    stats[5] = pl + ent_coef * entropy_loss + vf_coef * value_loss;
    stats[6] = adv_stats[0]; stats[7] = adv_stats[1];
  }
}

// ---- clip_grad_norm_ + Adam ------------------------------------------------------------------------------------------------
__global__ void sumsq_partial_kernel(const float* __restrict__ g, int64_t n, float scale, double* __restrict__ part) {
  __shared__ double s[32];
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = (double)(g[i] * scale);
    acc += v * v;
  }
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    acc = 0.0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) acc += s[k];
    part[blockIdx.x] = acc;
  }
}
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
                            const double* __restrict__ part, int nparts, float grad_scale, float max_grad_norm, float lr, float beta1,
                            float beta2, float eps, float bc1, float bc2_sqrt, float* __restrict__ gnorm_out) {
  double tot = 0.0;
  for (int k = 0; k < nparts; k++) tot += part[k];      // every thread walks the same short list: same value everywhere
  const float norm = (float)sqrt(tot);
  float coef = 1.f;
  if (max_grad_norm > 0.f) coef = fminf(max_grad_norm / (norm + 1e-6f), 1.f);
  if (gnorm_out && blockIdx.x == 0 && threadIdx.x == 0) gnorm_out[0] = norm;
  const float gs = grad_scale * coef, step = lr / bc1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * gs;
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] -= step * mi / (sqrtf(vi) / bc2_sqrt + eps);
  }
}

// ---- handle ------------------------------------------------------------------------------------------------------------------
struct NetLayout {
  int64_t wih, whh, bih, bhh;        // offsets into the flat parameter / gradient vector
  int nl, width[4];
  int64_t w[4], b[4];
  int64_t head_w, head_b;
  int head_n, head_np;               // outputs of the head (A or 1) and its padded operand width
  // offsets into the operand-copy buffer (elements)
  int64_t op_wih, op_whh, op_w[4], op_head;
};

}  // namespace

// activations / gradients of one network; the actor and the critic each own a set so their chains can run concurrently
struct NetBufs {
  void *dG = nullptr, *Hs = nullptr, *HP = nullptr, *Al[4] = {nullptr, nullptr, nullptr, nullptr}, *dZ = nullptr, *dhead = nullptr;
  float *G = nullptr, *Cs = nullptr, *C0 = nullptr, *T1 = nullptr, *head_out = nullptr, *dh_carry = nullptr, *dc_carry = nullptr, *cpart = nullptr;
  cublasHandle_t blas = nullptr;
  void* workspace = nullptr;
  uint8_t* seq_wpack = nullptr;      // persistent recurrent kernels (myo_lstm_seq.cu): packed W_hh images, combined bias
  float* seq_bias = nullptr;
  uint8_t* seq_rec = nullptr;        // activation records of the forward cluster kernel [M][H/8][kLstmRecBytes]
};

struct GradKey {      // everything a captured graph bakes in
  const void* ptr[12];
  int T, n, B;
  myo_ppo_hyper hp;
};

struct myo_ppo {
  myo_policy_cfg cfg{};
  int device = 0, precision = 1, maxT = 0, maxB = 0, use_sde = 0;
  int O = 0, Op = 0, A = 0, Ap = 0, H = 0, Dmax = 0;
  void *lat2 = nullptr, *S2 = nullptr, *Q = nullptr;      // gSDE: latent^2 [M][d], exp(2 log_std) [d][Ap], dL/dsigma^2 [M][Ap] (operand type)
  float *var_raw = nullptr, *dS2 = nullptr;               //       latent^2 . S2 [M][Ap], dL/dS2 [d][Ap]
  int64_t n_params = 0, n_op = 0;
  int64_t o_log_std = 0;
  NetLayout net[2];
  std::map<std::string, std::pair<int64_t, int64_t>> names;   // state-dict key -> (offset, numel)
  int64_t launches = 0;
  // device buffers
  void* wop = nullptr;
  void* X = nullptr;
  NetBufs nb[2];
  int32_t* idx = nullptr;
  float *act = nullptr, *keep = nullptr, *ov = nullptr, *ol = nullptr, *ad = nullptr, *rt = nullptr, *adv_stats = nullptr;
  float *ppart = nullptr, *vpart = nullptr;
  double* npart = nullptr;
  std::vector<void*> allocs;
  // the critic's chain runs on a second stream (fork / join by events) next to the actor's; the whole minibatch is
  // captured once into a CUDA graph (about 1 100 short launches) and replayed while the arguments stay the same
  cudaStream_t side = nullptr, main = nullptr;     // main: the graph's origin stream (the caller's may be the legacy default stream, which cannot be captured)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_in = nullptr, ev_out = nullptr;
  bool have_graph = false;
  long long* seq_prof = nullptr;     // MYO_PPO_SEQ_PROF=1: cycle counters of the forward cluster kernel (development)
  bool use_seq = false;              // bf16 mode with a supported hidden size: the recurrence runs in the persistent cluster kernels
  cudaGraphExec_t exec = nullptr;
  GradKey key{};
  int64_t graph_launches = 0;
};

namespace {

size_t op_size(const myo_ppo* p) { return p->precision ? sizeof(bf16) : sizeof(float); }

template <typename T>
int dev_alloc(myo_ppo* p, T** out, size_t bytes) {
  void* q = nullptr;
  if (cudaMalloc(&q, bytes ? bytes : 16) != cudaSuccess) {
    cudaGetLastError();
    myo::set_error("myo_ppo: device allocation of " + std::to_string(bytes) + " bytes failed");
    return MYO_E_CUDA;
  }
  p->allocs.push_back(q);
  *out = static_cast<T*>(q);
  return MYO_OK;
}

void build_layout(myo_ppo* p) {
  const myo_policy_cfg& c = p->cfg;
  const int H = c.lstm_hidden, O = c.obs_dim, A = c.act_dim;
  int64_t off = 0, op = 0;
  auto add = [&](const std::string& key, int64_t numel) {
    const int64_t o = off;
    p->names[key] = {o, numel};
    off += (numel + 7) / 8 * 8;
    return o;
  };
  {
    const int d_pi = c.n_pi_layers ? c.pi_layers[c.n_pi_layers - 1] : H;
    p->o_log_std = add("log_std", p->use_sde ? (int64_t)d_pi * A : A);
  }
  const char* lstm_name[2] = {"lstm_actor", "lstm_critic"};
  for (int k = 0; k < 2; k++) {
    NetLayout& n = p->net[k];
    n.wih = add(std::string(lstm_name[k]) + ".weight_ih_l0", (int64_t)4 * H * O);
    n.whh = add(std::string(lstm_name[k]) + ".weight_hh_l0", (int64_t)4 * H * H);
    n.bih = add(std::string(lstm_name[k]) + ".bias_ih_l0", 4 * H);
    n.bhh = add(std::string(lstm_name[k]) + ".bias_hh_l0", 4 * H);
  }
  const char* mlp_name[2] = {"mlp_extractor.policy_net.", "mlp_extractor.value_net."};
  for (int k = 0; k < 2; k++) {
    NetLayout& n = p->net[k];
    n.nl = k == 0 ? c.n_pi_layers : c.n_vf_layers;
    int d = H;
    for (int l = 0; l < n.nl; l++) {
      n.width[l] = k == 0 ? c.pi_layers[l] : c.vf_layers[l];
      n.w[l] = add(std::string(mlp_name[k]) + std::to_string(2 * l) + ".weight", (int64_t)n.width[l] * d);
      n.b[l] = add(std::string(mlp_name[k]) + std::to_string(2 * l) + ".bias", n.width[l]);
      d = n.width[l];
    }
  }
  for (int k = 0; k < 2; k++) {
    NetLayout& n = p->net[k];
    const int d = n.nl ? n.width[n.nl - 1] : H;
    n.head_n = k == 0 ? A : 1;
    n.head_np = k == 0 ? p->Ap : 1;
    n.head_w = add(k == 0 ? "action_net.weight" : "value_net.weight", (int64_t)n.head_n * d);
    n.head_b = add(k == 0 ? "action_net.bias" : "value_net.bias", n.head_n);
  }
  p->n_params = off;
  for (int k = 0; k < 2; k++) {
    NetLayout& n = p->net[k];
    n.op_wih = op; op += (int64_t)4 * H * p->Op;
    n.op_whh = op; op += (int64_t)4 * H * H;
    int d = H;
    for (int l = 0; l < n.nl; l++) { n.op_w[l] = op; op += (int64_t)n.width[l] * d; d = n.width[l]; }
    n.op_head = op; op += (int64_t)n.head_np * d;
  }
  p->n_op = op;
}

// row-major GEMMs on cuBLAS (column-major underneath). A, B: operand type; C: fp32.
// nt: C[M][N] (ldc) = A[M][K] (lda) . B[N][K]^T (ldb) + beta C
int gemm_nt(myo_ppo* p, cublasHandle_t blas, int64_t M, int N, int K, const void* A, int lda, const void* B, int ldb, float beta, float* C, int ldc) {
  const float alpha = 1.f;
  const cudaDataType dt = p->precision ? CUDA_R_16BF : CUDA_R_32F;
  BCK(cublasGemmEx(blas, CUBLAS_OP_T, CUBLAS_OP_N, N, (int)M, K, &alpha, B, dt, ldb, A, dt, lda, &beta, C, CUDA_R_32F, ldc,
                   CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT));
  p->launches++;
  return MYO_OK;
}
// nn: C[M][N] (ldc) = A[M][K] (lda) . B[K][N] (ldb)
int gemm_nn(myo_ppo* p, cublasHandle_t blas, int64_t M, int N, int K, const void* A, int lda, const void* B, int ldb, float* C, int ldc) {
  const float alpha = 1.f, beta = 0.f;
  const cudaDataType dt = p->precision ? CUDA_R_16BF : CUDA_R_32F;
  BCK(cublasGemmEx(blas, CUBLAS_OP_N, CUBLAS_OP_N, N, (int)M, K, &alpha, B, dt, ldb, A, dt, lda, &beta, C, CUDA_R_32F, ldc,
                   CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT));
  p->launches++;
  return MYO_OK;
}
// tn: dW[N][K] (ldc) = dY[M][N]^T (ldy) . X[M][K] (ldx)
int gemm_tn(myo_ppo* p, cublasHandle_t blas, int64_t M, int N, int K, const void* dY, int ldy, const void* X, int ldx, float* dW, int ldc) {
  const float alpha = 1.f, beta = 0.f;
  const cudaDataType dt = p->precision ? CUDA_R_16BF : CUDA_R_32F;
  BCK(cublasGemmEx(blas, CUBLAS_OP_N, CUBLAS_OP_T, K, N, (int)M, &alpha, X, dt, ldx, dY, dt, ldy, &beta, dW, CUDA_R_32F, ldc,
                   CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT));
  p->launches++;
  return MYO_OK;
}

inline int blocks_for(int64_t total, int threads, int cap = 148 * 16) {
  const int64_t b = (total + threads - 1) / threads;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

template <typename T>
int colsum(myo_ppo* p, float* cpart, const T* Y, int64_t M, int N, int ld, float* out, float* out2, cudaStream_t st) {
  int chunks = (int)((M + 63) / 64);
  if (chunks > kColsumRows) chunks = kColsumRows;
  dim3 grid((N + 31) / 32, chunks), block(32, 8);
  colsum_partial_kernel<T><<<grid, block, 0, st>>>(Y, M, N, ld, cpart);
  colsum_final_kernel<<<(N + 127) / 128, 128, 0, st>>>(cpart, chunks, N, out, out2);
  p->launches += 2;
  QCK(cudaGetLastError());
  return MYO_OK;
}

struct GradArgs {
  const float* params; int T, n, B; const int32_t* idx;
  const float *obs, *actions; const uint8_t* starts; const float *old_values, *old_logp, *adv, *ret, *h0, *c0;
  myo_ppo_hyper hp; float* grad; float* stats;
};

// forward, loss gradient at the head and backward of network k, all on stream st
template <typename T>
int net_chain(myo_ppo* p, const GradArgs& a, int k, cudaStream_t st) {
  const int H = p->H, O = p->O, Op = p->Op, A = p->A, Ap = p->Ap, B = a.B, Tn = a.T;
  const int64_t M = (int64_t)Tn * B;
  const NetLayout& n = p->net[k];
  NetBufs& nb = p->nb[k];
  cublasHandle_t blas = nb.blas;
  BCK(cublasSetStream(blas, st));
  T* wop = static_cast<T*>(p->wop);
  T* X = static_cast<T*>(p->X); T* dG = static_cast<T*>(nb.dG); T* Hs = static_cast<T*>(nb.Hs); T* HP = static_cast<T*>(nb.HP);
  T* dZ = static_cast<T*>(nb.dZ); T* dhead = static_cast<T*>(nb.dhead);
  const int cell_blocks = (B * (H / 4) + 255) / 256;
  // ---- forward over the sequences ----
  gather_state_kernel<T><<<(B * H + 255) / 256, 256, 0, st>>>(B, H, p->idx, a.h0 + (int64_t)k * a.n * H, a.c0 + (int64_t)k * a.n * H, p->keep, HP, nb.C0);
  p->launches++;
  RCK(gemm_nt(p, blas, M, 4 * H, Op, X, Op, wop + n.op_wih, Op, 0.f, nb.G, 4 * H));
  if (p->use_seq) {
    myo::LstmSeqFwd f{Tn, B, H, a.params + n.whh, a.params + n.bih, a.params + n.bhh, nb.seq_wpack, nb.seq_bias, nb.G, p->keep, nb.C0, nb.seq_rec, Hs, HP, k == 0 ? p->seq_prof : nullptr};
    p->launches++;
    RCK(myo::lstm_seq_forward(f, st));
    p->launches += 2;
  } else
  for (int t = 0; t < Tn; t++) {
    RCK(gemm_nt(p, blas, B, 4 * H, H, HP + (int64_t)t * B * H, H, wop + n.op_whh, H, 1.f, nb.G + (int64_t)t * B * 4 * H, 4 * H));
    lstm_cell_fwd_kernel<T><<<cell_blocks, 256, 0, st>>>(t, Tn, B, H, nb.G, a.params + n.bih, a.params + n.bhh, p->keep, nb.C0, nb.Cs, Hs, HP);
    p->launches++;
  }
  const T* in = Hs;
  int d = H;
  for (int l = 0; l < n.nl; l++) {
    T* Aout = static_cast<T*>(nb.Al[l]);
    RCK(gemm_nt(p, blas, M, n.width[l], d, in, d, wop + n.op_w[l], d, 0.f, nb.T1, n.width[l]));
    bias_relu_kernel<T><<<blocks_for(M * n.width[l] / 4, 256), 256, 0, st>>>(nb.T1, a.params + n.b[l], Aout, M * n.width[l], n.width[l]);
    p->launches++;
    in = Aout; d = n.width[l];
  }
  RCK(gemm_nt(p, blas, M, n.head_np, d, in, d, wop + n.op_head, d, 0.f, nb.head_out, n.head_np));
  // ---- loss and its gradient at the head ----
  const bool sde = k == 0 && p->use_sde;
  if (sde) {       // variance of the state-dependent noise: latent^2 . exp(2 log_std)  (latent detached: learn_features=False)
    square_kernel<T><<<blocks_for(M * d, 256), 256, 0, st>>>(in, static_cast<T*>(p->lat2), M * d);
    sde_std2_kernel<T><<<blocks_for((int64_t)d * Ap, 256), 256, 0, st>>>(a.params + p->o_log_std, static_cast<T*>(p->S2), d, A, Ap);
    p->launches += 2;
    RCK(gemm_nn(p, blas, M, Ap, d, p->lat2, d, p->S2, Ap, p->var_raw, Ap));
  }
  if (k == 0) {
    LossArgs la{M, A, Ap, sde ? p->var_raw : nullptr, a.hp.ent_coef, nb.head_out, a.params + n.head_b, a.params + p->o_log_std, p->act, p->ol, p->ad,
                p->adv_stats, a.hp.clip_range, a.hp.normalize_advantage};
    policy_loss_kernel<T><<<kLossBlocks, 256, sizeof(float) * 8 * (kStatSlots + A), st>>>(la, dhead, static_cast<T*>(p->Q), p->ppart);
    if (sde) {     // dL/dS2 = (latent^2)' . Q, then the chain rule through exp(2 log_std)
      RCK(gemm_tn(p, blas, M, d, Ap, p->lat2, d, p->Q, Ap, p->dS2, Ap));
      sde_logstd_grad_kernel<<<blocks_for((int64_t)d * A, 256), 256, 0, st>>>(p->dS2, a.params + p->o_log_std, a.grad + p->o_log_std, d, A, Ap);
      p->launches++;
    }
  } else {
    value_loss_kernel<T><<<kLossBlocks, 256, 0, st>>>(M, nb.head_out, a.params + n.head_b, p->ov, p->rt, a.hp.clip_range_vf, a.hp.vf_coef, dhead,
                                                       p->vpart);
  }
  p->launches++;
  QCK(cudaGetLastError());
  // ---- backward ----
  const int ldh = n.head_np;
  RCK(gemm_tn(p, blas, M, n.head_n, d, dhead, ldh, in, d, a.grad + n.head_w, d));
  RCK(colsum<T>(p, nb.cpart, dhead, M, n.head_n, ldh, a.grad + n.head_b, nullptr, st));
  // dA[M][d] = dhead[M][head_n] . W_head[head_n][d]
  RCK(gemm_nn(p, blas, M, d, n.head_np, dhead, ldh, wop + n.op_head, d, nb.T1, d));
  for (int l = n.nl - 1; l >= 0; l--) {
    const T* Aout = static_cast<const T*>(nb.Al[l]);
    const T* inl = l > 0 ? static_cast<const T*>(nb.Al[l - 1]) : Hs;
    const int din = l > 0 ? n.width[l - 1] : H;
    relu_bwd_kernel<T><<<blocks_for(M * n.width[l] / 4, 256), 256, 0, st>>>(nb.T1, Aout, dZ, M * n.width[l]);
    p->launches++;
    RCK(gemm_tn(p, blas, M, n.width[l], din, dZ, n.width[l], inl, din, a.grad + n.w[l], din));
    RCK(colsum<T>(p, nb.cpart, dZ, M, n.width[l], n.width[l], a.grad + n.b[l], nullptr, st));
    RCK(gemm_nn(p, blas, M, din, n.width[l], dZ, n.width[l], wop + n.op_w[l], din, nb.T1, din));
  }
  // T1 = dL/dHs [M][H]; backward through time
  for (int t = Tn - 1; t >= 0; t--) {
    if (p->use_seq)
      lstm_cell_bwd_rec_kernel<<<(B * (H / 8) + 255) / 256, 256, 0, st>>>(t, Tn, B, H, nb.seq_rec, p->keep, nb.C0, nb.T1, nb.dh_carry, nb.dc_carry,
                                                                          reinterpret_cast<bf16*>(nb.dG));
    else
      lstm_cell_bwd_kernel<T><<<cell_blocks, 256, 0, st>>>(t, Tn, B, H, nb.G, p->keep, nb.C0, nb.Cs, nb.T1, nb.dh_carry, nb.dc_carry, dG);
    p->launches++;
    if (t > 0) RCK(gemm_nn(p, blas, B, H, 4 * H, dG + (int64_t)t * B * 4 * H, 4 * H, wop + n.op_whh, H, nb.dh_carry, H));
  }
  RCK(gemm_tn(p, blas, M, 4 * H, O, dG, 4 * H, X, Op, a.grad + n.wih, O));
  RCK(gemm_tn(p, blas, M, 4 * H, H, dG, 4 * H, HP, H, a.grad + n.whh, H));
  RCK(colsum<T>(p, nb.cpart, dG, M, 4 * H, 4 * H, a.grad + n.bih, a.grad + n.bhh, st));
  QCK(cudaGetLastError());
  return MYO_OK;
}

// the whole minibatch: shared prologue on st, the actor's chain on st and the critic's on the side stream, join, finalize
template <typename T>
int minibatch_issue(myo_ppo* p, const GradArgs& a, cudaStream_t st) {
  const int H = p->H, O = p->O, Op = p->Op, A = p->A, B = a.B, Tn = a.T;
  const int64_t M = (int64_t)Tn * B;
  T* wop = static_cast<T*>(p->wop);
  T* X = static_cast<T*>(p->X);
  QCK(cudaMemsetAsync(a.grad, 0, sizeof(float) * p->n_params, st));
  // operand copies of the weights
  for (int k = 0; k < 2; k++) {
    const NetLayout& n = p->net[k];
    convert_pad_kernel<T><<<blocks_for((int64_t)4 * H * Op, 256), 256, 0, st>>>(a.params + n.wih, wop + n.op_wih, 4 * H, O, 4 * H, Op);
    convert_pad_kernel<T><<<blocks_for((int64_t)4 * H * H, 256), 256, 0, st>>>(a.params + n.whh, wop + n.op_whh, 4 * H, H, 4 * H, H);
    int d = H;
    for (int l = 0; l < n.nl; l++) {
      convert_pad_kernel<T><<<blocks_for((int64_t)n.width[l] * d, 256), 256, 0, st>>>(a.params + n.w[l], wop + n.op_w[l], n.width[l], d, n.width[l], d);
      d = n.width[l];
    }
    convert_pad_kernel<T><<<blocks_for((int64_t)n.head_np * d, 256), 256, 0, st>>>(a.params + n.head_w, wop + n.op_head, n.head_n, d, n.head_np, d);
    p->launches += 3 + n.nl;
  }
  gather_rows_kernel<T><<<blocks_for(M * 32, 256), 256, 0, st>>>(Tn, B, a.n, O, Op, A, p->idx, a.obs, a.actions, a.starts, a.old_values, a.old_logp,
                                                                   a.adv, a.ret, X, p->act, p->keep, p->ov, p->ol, p->ad, p->rt);
  adv_stats_kernel<<<1, 1024, 0, st>>>(p->ad, M, p->adv_stats);
  p->launches += 2;
  QCK(cudaGetLastError());
  QCK(cudaEventRecord(p->ev_fork, st));
  QCK(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
  int rc = net_chain<T>(p, a, 1, p->side);
  if (cudaEventRecord(p->ev_join, p->side) != cudaSuccess && !rc) { myo::set_error("cudaEventRecord(join) failed"); rc = MYO_E_CUDA; }
  const int rc0 = net_chain<T>(p, a, 0, st);
  if (cudaStreamWaitEvent(st, p->ev_join, 0) != cudaSuccess && !rc) { myo::set_error("cudaStreamWaitEvent(join) failed"); rc = MYO_E_CUDA; }
  if (rc0) return rc0;
  if (rc) return rc;
  loss_finalize_kernel<<<1, 128, 0, st>>>(p->ppart, kLossBlocks, p->vpart, kLossBlocks, A, M, a.params + p->o_log_std, p->adv_stats, a.hp.ent_coef,
                                          a.hp.vf_coef, a.stats, a.grad + p->o_log_std, p->use_sde);
  p->launches++;
  QCK(cudaGetLastError());
  return MYO_OK;
}

GradKey make_key(const GradArgs& a) {
  GradKey k;
  memset(&k, 0, sizeof(k));
  const void* ptrs[12] = {a.params, a.obs, a.actions, a.starts, a.old_values, a.old_logp, a.adv, a.ret, a.h0, a.c0, a.grad, a.stats};
  for (int i = 0; i < 12; i++) k.ptr[i] = ptrs[i];
  k.T = a.T; k.n = a.n; k.B = a.B; k.hp = a.hp;
  return k;
}

template <typename T>
int minibatch_grad(myo_ppo* p, const GradArgs& a, cudaStream_t st) {
  QCK(cudaMemcpyAsync(p->idx, a.idx, sizeof(int32_t) * a.B, cudaMemcpyDeviceToDevice, st));
  // the graph runs on the handle's own stream, ordered after / before the caller's stream by events
  QCK(cudaEventRecord(p->ev_in, st));
  QCK(cudaStreamWaitEvent(p->main, p->ev_in, 0));
  const GradKey key = make_key(a);
  if (!p->have_graph || memcmp(&key, &p->key, sizeof(key)) != 0) {
    if (p->exec) { cudaGraphExecDestroy(p->exec); p->exec = nullptr; }
    p->have_graph = false;
    const int64_t l0 = p->launches;
    QCK(cudaStreamBeginCapture(p->main, cudaStreamCaptureModeThreadLocal));
    const int rc = minibatch_issue<T>(p, a, p->main);
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(p->main, &graph);
    p->graph_launches = p->launches - l0;
    p->launches = l0;
    if (rc) { if (graph) cudaGraphDestroy(graph); cudaGetLastError(); return rc; }
    if (e != cudaSuccess || !graph) { myo::set_error(std::string("graph capture of the PPO minibatch failed: ") + cudaGetErrorString(e)); cudaGetLastError(); return MYO_E_CUDA; }
    const cudaError_t ei = cudaGraphInstantiate(&p->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) { myo::set_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ei)); cudaGetLastError(); return MYO_E_CUDA; }
    p->key = key; p->have_graph = true;
  }
  QCK(cudaGraphLaunch(p->exec, p->main));
  p->launches += p->graph_launches;
  QCK(cudaEventRecord(p->ev_out, p->main));
  QCK(cudaStreamWaitEvent(st, p->ev_out, 0));
  return MYO_OK;
}

}  // namespace

extern "C" {

int myo_ppo_create(const myo_policy_cfg* cfg, int max_steps, int max_worlds, int precision, int device, myo_ppo** out) {
  if (!cfg || !out || max_steps <= 0 || max_worlds <= 0 || precision < 0 || precision > 1) { myo::set_error("bad argument to myo_ppo_create"); return MYO_E_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
    cudaGetLastError();
    myo::set_error("no CUDA device available (the PPO update has no CPU path)");
    return MYO_E_CUDA;
  }
  if (cfg->lstm_hidden <= 0 || cfg->lstm_hidden % 8) { myo::set_error("lstm_hidden must be a multiple of 8"); return MYO_E_LIMIT; }
  if (cfg->obs_dim <= 0 || cfg->act_dim <= 0) { myo::set_error("obs_dim and act_dim must be positive"); return MYO_E_LIMIT; }
  if (cfg->n_pi_layers < 0 || cfg->n_pi_layers > 4 || cfg->n_vf_layers < 0 || cfg->n_vf_layers > 4) { myo::set_error("at most 4 MLP layers per head"); return MYO_E_LIMIT; }
  for (int l = 0; l < cfg->n_pi_layers; l++) if (cfg->pi_layers[l] <= 0 || cfg->pi_layers[l] % 8) { myo::set_error("MLP widths must be multiples of 8"); return MYO_E_LIMIT; }
  for (int l = 0; l < cfg->n_vf_layers; l++) if (cfg->vf_layers[l] <= 0 || cfg->vf_layers[l] % 8) { myo::set_error("MLP widths must be multiples of 8"); return MYO_E_LIMIT; }
  QCK(cudaSetDevice(device));
  myo_ppo* p = new myo_ppo();
  p->cfg = *cfg; p->device = device; p->precision = precision; p->maxT = max_steps; p->maxB = max_worlds; p->use_sde = cfg->use_sde != 0;
  p->O = cfg->obs_dim; p->Op = round_up(cfg->obs_dim, 8); p->A = cfg->act_dim; p->Ap = round_up(cfg->act_dim, 8); p->H = cfg->lstm_hidden;
  p->Dmax = p->H;
  for (int l = 0; l < cfg->n_pi_layers; l++) p->Dmax = cfg->pi_layers[l] > p->Dmax ? cfg->pi_layers[l] : p->Dmax;
  for (int l = 0; l < cfg->n_vf_layers; l++) p->Dmax = cfg->vf_layers[l] > p->Dmax ? cfg->vf_layers[l] : p->Dmax;
  build_layout(p);
  const size_t M = (size_t)max_steps * max_worlds, os = op_size(p), H = p->H, B = max_worlds;
  int rc = MYO_OK;
  auto A_ = [&](auto** q, size_t bytes) { if (!rc) rc = dev_alloc(p, q, bytes); };
  A_(&p->wop, os * p->n_op);
  A_(&p->X, os * M * p->Op);
  A_(&p->idx, sizeof(int32_t) * B);
  const size_t cpart_words = kColsumRows * (4 * H > (size_t)p->Dmax ? 4 * H : (size_t)p->Dmax);
  for (int k = 0; k < 2; k++) {
    NetBufs& nb = p->nb[k];
    const int nl = k == 0 ? cfg->n_pi_layers : cfg->n_vf_layers;
    A_(&nb.dG, os * M * 4 * H); A_(&nb.Hs, os * M * H); A_(&nb.HP, os * M * H);
    for (int l = 0; l < nl; l++) A_(&nb.Al[l], os * M * p->Dmax);
    A_(&nb.dZ, os * M * p->Dmax); A_(&nb.dhead, os * M * p->Ap);
    A_(&nb.G, sizeof(float) * M * 4 * H); A_(&nb.Cs, sizeof(float) * M * H); A_(&nb.C0, sizeof(float) * B * H);
    A_(&nb.T1, sizeof(float) * M * p->Dmax); A_(&nb.head_out, sizeof(float) * M * p->Ap);
    A_(&nb.dh_carry, sizeof(float) * B * H); A_(&nb.dc_carry, sizeof(float) * B * H);
    A_(&nb.cpart, sizeof(float) * cpart_words);
    A_(&nb.workspace, kBlasWorkspace);
    if (precision && myo::lstm_seq_supported((int)H) && getenv("MYO_PPO_SEQ") && atoi(getenv("MYO_PPO_SEQ"))) { A_(&nb.seq_wpack, 2 * myo::lstm_seq_wpack_bytes((int)H)); A_(&nb.seq_bias, sizeof(float) * 4 * H);
      A_(&nb.seq_rec, M * (H / 8) * myo::kLstmRecBytes); }
  }
  // The persistent cluster kernel is correct (tests compare it with the launch chain) but not faster yet (DESIGN.md 3.4b:
  // 9.1 vs 7.7 ms per minibatch on the bench shape), so the launch chain stays the default; MYO_PPO_SEQ=1 selects the kernel.
  p->use_seq = false;
  if (const char* e = getenv("MYO_PPO_SEQ")) p->use_seq = precision && myo::lstm_seq_supported((int)H) && atoi(e) != 0;
  if (const char* e = getenv("MYO_PPO_SEQ_PROF")) if (atoi(e)) { A_(&p->seq_prof, sizeof(long long) * 8); if (!rc) cudaMemset(p->seq_prof, 0, 64); }
  A_(&p->act, sizeof(float) * M * p->A); A_(&p->keep, sizeof(float) * M); A_(&p->ov, sizeof(float) * M); A_(&p->ol, sizeof(float) * M);
  A_(&p->ad, sizeof(float) * M); A_(&p->rt, sizeof(float) * M); A_(&p->adv_stats, sizeof(float) * 2);
  A_(&p->ppart, sizeof(float) * kLossBlocks * (kStatSlots + p->A)); A_(&p->vpart, sizeof(float) * kLossBlocks);
  A_(&p->npart, sizeof(double) * kNormBlocks);
  if (p->use_sde) {
    A_(&p->lat2, os * M * p->Dmax); A_(&p->S2, os * (size_t)p->Dmax * p->Ap); A_(&p->Q, os * M * p->Ap);
    A_(&p->var_raw, sizeof(float) * M * p->Ap); A_(&p->dS2, sizeof(float) * (size_t)p->Dmax * p->Ap);
  }
  if (rc) { myo_ppo_destroy(p); return rc; }
  for (int k = 0; k < 2; k++) {
    // an explicit workspace per handle: the two handles run concurrently, and cuBLAS must not allocate inside a graph capture
    if (cublasCreate(&p->nb[k].blas) != CUBLAS_STATUS_SUCCESS || cublasSetWorkspace(p->nb[k].blas, p->nb[k].workspace, kBlasWorkspace) != CUBLAS_STATUS_SUCCESS) {
      myo::set_error("cublasCreate / cublasSetWorkspace failed");
      myo_ppo_destroy(p);
      return MYO_E_CUDA;
    }
  }
  if (cudaStreamCreateWithFlags(&p->side, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&p->main, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&p->ev_in, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&p->ev_out, cudaEventDisableTiming) != cudaSuccess) {
    myo::set_error("stream / event creation failed");
    myo_ppo_destroy(p);
    return MYO_E_CUDA;
  }
  *out = p;
  return MYO_OK;
}

void myo_ppo_destroy(myo_ppo* p) {
  if (!p) return;
  cudaSetDevice(p->device);
  if (p->seq_prof) {
    long long h[8];
    cudaDeviceSynchronize();
    if (cudaMemcpy(h, p->seq_prof, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess)
      fprintf(stderr, "lstm_seq_fwd cycles (last launch, one thread): mma+wait %lld | epilogue math+global %lld | cluster wait #1 %lld | remote stores %lld | fences %lld | barrier #2 %lld\n",
              h[0], h[1], h[2], h[3], h[4], h[5]);
  }
  if (p->exec) cudaGraphExecDestroy(p->exec);
  for (int k = 0; k < 2; k++) if (p->nb[k].blas) cublasDestroy(p->nb[k].blas);
  if (p->side) cudaStreamDestroy(p->side);
  if (p->main) cudaStreamDestroy(p->main);
  if (p->ev_in) cudaEventDestroy(p->ev_in);
  if (p->ev_out) cudaEventDestroy(p->ev_out);
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->ev_join) cudaEventDestroy(p->ev_join);
  for (void* q : p->allocs) cudaFree(q);
  delete p;
}

int64_t myo_ppo_param_count(const myo_ppo* p) { return p ? p->n_params : 0; }

int myo_ppo_param_offset(const myo_ppo* p, const char* name, int64_t* offset, int64_t* numel) {
  if (!p || !name || !offset || !numel) { myo::set_error("bad argument to myo_ppo_param_offset"); return MYO_E_ARG; }
  auto it = p->names.find(name);
  if (it == p->names.end()) { myo::set_error(std::string("unknown parameter ") + name); return MYO_E_ARG; }
  *offset = it->second.first; *numel = it->second.second;
  return MYO_OK;
}

int myo_ppo_minibatch_grad(myo_ppo* p, const float* params_dev, int n_steps, int n_envs, const int32_t* world_idx_dev, int n_worlds,
                           const float* obs_dev, const float* actions_dev, const uint8_t* episode_starts_dev, const float* old_values_dev,
                           const float* old_logp_dev, const float* advantages_dev, const float* returns_dev, const float* h0_dev,
                           const float* c0_dev, const myo_ppo_hyper* hyper, float* grad_dev, float* stats_dev, void* stream) {
  if (!p || !params_dev || !world_idx_dev || !obs_dev || !actions_dev || !episode_starts_dev || !old_values_dev || !old_logp_dev ||
      !advantages_dev || !returns_dev || !h0_dev || !c0_dev || !hyper || !grad_dev || !stats_dev) {
    myo::set_error("null argument to myo_ppo_minibatch_grad");
    return MYO_E_ARG;
  }
  if (n_steps <= 0 || n_steps > p->maxT || n_worlds <= 0 || n_worlds > p->maxB || n_envs < n_worlds) {
    myo::set_error("minibatch exceeds the sizes given to myo_ppo_create");
    return MYO_E_ARG;
  }
  QCK(cudaSetDevice(p->device));
  GradArgs a{params_dev, n_steps, n_envs, n_worlds, world_idx_dev, obs_dev, actions_dev, episode_starts_dev, old_values_dev, old_logp_dev,
             advantages_dev, returns_dev, h0_dev, c0_dev, *hyper, grad_dev, stats_dev};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return p->precision ? minibatch_grad<bf16>(p, a, st) : minibatch_grad<float>(p, a, st);
}

int myo_ppo_adam_step(myo_ppo* p, float* params_dev, const float* grad_dev, float* exp_avg_dev, float* exp_avg_sq_dev, int step, float lr,
                      float beta1, float beta2, float eps, float max_grad_norm, float grad_scale, float* grad_norm_dev, void* stream) {
  if (!p || !params_dev || !grad_dev || !exp_avg_dev || !exp_avg_sq_dev || step <= 0) { myo::set_error("bad argument to myo_ppo_adam_step"); return MYO_E_ARG; }
  QCK(cudaSetDevice(p->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  sumsq_partial_kernel<<<kNormBlocks, 256, 0, st>>>(grad_dev, p->n_params, grad_scale, p->npart);
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<<<blocks_for(p->n_params, 256), 256, 0, st>>>(params_dev, grad_dev, exp_avg_dev, exp_avg_sq_dev, p->n_params, p->npart, kNormBlocks,
                                                            grad_scale, max_grad_norm, lr, beta1, beta2, eps, bc1, sqrtf(bc2), grad_norm_dev);
  p->launches += 2;
  QCK(cudaGetLastError());
  return MYO_OK;
}

int64_t myo_ppo_launch_count(const myo_ppo* p) { return p ? p->launches : 0; }

}  // extern "C"
