// K6b: packed bidirectional GRU recurrence (one layer), forward and backward through time.
//
// Replaces the nn.GRU context encoders: DGCNModule("GRU") (track_mm/dgcnv2.py: 2-layer BiGRU run unpacked over the
// seq-first padded batch) and SeqContext(rnn_type="gru") (track_mm/dgcn_models.py:46-47: 2-layer BiGRU over the packed
// sequence).  torch.nn.GRU semantics, gate order (r, z, n):
//     r = sigmoid(gx_r + W_hr h + b_hr),  z = sigmoid(gx_z + W_hz h + b_hz),  hn = W_hn h + b_hn
//     n = tanh(gx_n + r * hn),  h' = n + z (h - n)            (= (1 - z) n + z h, in ATen's order)
// gx = x W_ih^T + b_ih for ALL utterances and both directions is one hoisted GEMM (K2).  Unlike the LSTM (K6), b_hh
// cannot be folded into it -- b_hn sits inside r * (W_hn h + b_hn) -- so b_hh is an argument and is added in here.
//
// Same structure as K6: one CTA of 3*Hd threads per (direction, slice of dialogues), thread r keeps row r of W_hh in
// REGISTERS for the whole launch, h_{t-1} is broadcast from shared memory, 2 barriers per step; dialogue d occupies rows
// node_off[d] .. node_off[d+1] (packed-sequence semantics by construction, h0 = 0 per dialogue and direction).
// The weight gradients are NOT accumulated here: the backward stores the hidden-side pre-activation gradient
// dgh = [da_r, da_z, r * da_n] next to dgx = [da_r, da_z, da_n], and the caller forms dW_hh = dgh^T @ h_prev and
// db_hh = colsum(dgh) with the fixed-order reductions of K2.
#include "common.cuh"
#include <math.h>

namespace ercg {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// gates[t, dir*4Hd + (0|1|2|3)*Hd + j] = r, z, n, hn of unit j; hprev[t, dir*Hd + j] = h_{t-1}
template <int HD>
__global__ void __launch_bounds__(3 * HD, 1)
gru_fwd_kernel(const float* __restrict__ gx, long long ldgx, const float* __restrict__ whh, const float* __restrict__ bhh,
               const int* __restrict__ node_off, int B, float* __restrict__ out, long long ldo, float* __restrict__ gates,
               float* __restrict__ hprev) {
  __shared__ __align__(16) float sh[HD];
  __shared__ float srz[2 * HD];                   // r, z of the current step
  const int r = threadIdx.x;
  const int dir = blockIdx.x & 1;
  float w[HD];
  {
    const float* wr = whh + ((long long)dir * 3 * HD + r) * HD;
#pragma unroll
    for (int k = 0; k < HD; ++k) w[k] = wr[k];
  }
  const float bh = bhh[dir * 3 * HD + r];
  const int stride = gridDim.x >> 1;
  for (int d = blockIdx.x >> 1; d < B; d += stride) {
    const int o = node_off[d], L = node_off[d + 1] - o;
    if (r < HD) sh[r] = 0.f;
    __syncthreads();
    for (int s = 0; s < L; ++s) {
      const long long t = o + (dir == 0 ? s : L - 1 - s);
      const float g = gx[t * ldgx + dir * 3 * HD + r];
      float acc = bh;
#pragma unroll
      for (int k = 0; k < HD; k += 4) {
        const float4 h4 = *reinterpret_cast<const float4*>(&sh[k]);
        acc = fmaf(w[k], h4.x, acc); acc = fmaf(w[k + 1], h4.y, acc);
        acc = fmaf(w[k + 2], h4.z, acc); acc = fmaf(w[k + 3], h4.w, acc);
      }
      float* gt = gates + t * (8 * HD) + dir * 4 * HD;
      if (r < 2 * HD) {
        const float a = sigmoidf_(g + acc);
        srz[r] = a;
        gt[r] = a;
      }
      __syncthreads();
      if (r >= 2 * HD) {                          // the n-row threads hold gx_n and hn = W_hn h + b_hn: they finish the unit
        const int j = r - 2 * HD;
        const float rg = srz[j], zg = srz[HD + j], hp = sh[j];
        const float n = tanhf(fmaf(rg, acc, g));
        const float h = fmaf(zg, hp - n, n);
        gt[2 * HD + j] = n;
        gt[3 * HD + j] = acc;
        hprev[t * (2 * HD) + dir * HD + j] = hp;
        out[t * ldo + dir * HD + j] = h;
        sh[j] = h;
      }
      __syncthreads();
    }
  }
}

// thread (q, k) = (threadIdx.x / HD, threadIdx.x % HD) keeps W_hh[q*HD + j][k], j = 0..HD-1, in registers
template <int HD>
__global__ void __launch_bounds__(3 * HD, 1)
gru_bwd_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ gates,
               const float* __restrict__ hprev, const float* __restrict__ whh, const int* __restrict__ node_off, int B,
               float* __restrict__ dgx, long long lddgx, float* __restrict__ dgh, long long lddgh) {
  __shared__ __align__(16) float sdg[3 * HD];     // [da_r, da_z, dhn] of the current step
  __shared__ float sdan[HD];                      // da_n
  __shared__ float spart[3 * HD];                 // partial dh_{t-1} per gate block
  const int tid = threadIdx.x, q = tid / HD, k = tid % HD;
  const int dir = blockIdx.x & 1;
  float w[HD];
#pragma unroll
  for (int j = 0; j < HD; ++j) w[j] = whh[((long long)dir * 3 * HD + q * HD + j) * HD + k];
  const int stride = gridDim.x >> 1;
  for (int d = blockIdx.x >> 1; d < B; d += stride) {
    const int o = node_off[d], L = node_off[d + 1] - o;
    float dh_rec = 0.f;                           // meaningful for tid < HD
    __syncthreads();
    for (int s = L - 1; s >= 0; --s) {            // reverse of the forward traversal order
      const long long t = o + (dir == 0 ? s : L - 1 - s);
      if (tid < HD) {
        const float* g = gates + t * (8 * HD) + dir * 4 * HD;
        const float rg = g[tid], zg = g[HD + tid], n = g[2 * HD + tid], hn = g[3 * HD + tid];
        const float hp = hprev[t * (2 * HD) + dir * HD + tid];
        const float dh = dout[t * ldo + dir * HD + tid] + dh_rec;
        const float dan = dh * (1.f - zg) * (1.f - n * n);
        sdg[tid] = dan * hn * rg * (1.f - rg);
        sdg[HD + tid] = dh * (hp - n) * zg * (1.f - zg);
        sdg[2 * HD + tid] = dan * rg;
        sdan[tid] = dan;
        dh_rec = dh * zg;                         // direct path; the W_hh^T products are added below
      }
      __syncthreads();
      const float v = sdg[tid];
      dgh[t * lddgh + dir * 3 * HD + tid] = v;
      dgx[t * lddgx + dir * 3 * HD + tid] = tid < 2 * HD ? v : sdan[tid - 2 * HD];
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < HD; j += 4) {
        const float4 g4 = *reinterpret_cast<const float4*>(&sdg[q * HD + j]);
        acc = fmaf(w[j], g4.x, acc); acc = fmaf(w[j + 1], g4.y, acc);
        acc = fmaf(w[j + 2], g4.z, acc); acc = fmaf(w[j + 3], g4.w, acc);
      }
      spart[tid] = acc;
      __syncthreads();
      if (tid < HD) dh_rec += (spart[tid] + spart[HD + tid]) + spart[2 * HD + tid];
    }
  }
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_gru_fwd(const float* gx, int64_t ldgx, const float* whh, const float* bhh, const int32_t* node_off, int B,
                            int Hd, float* out, int64_t ldo, float* gates, float* hprev, void* stream) {
  if (B < 0) return ERCG_EINVAL;
  if (B == 0) return ERCG_OK;
  if (!gx || !whh || !bhh || !node_off || !out || !gates || !hprev) return ERCG_EINVAL;
  long long want = 2LL * B;
  int grid = (int)(want < 2 * kNumSMs ? want : 2 * kNumSMs);
#define ERCG_GRU_F(HD_)                                                                                                \
  case HD_:                                                                                                            \
    gru_fwd_kernel<HD_><<<grid, 3 * HD_, 0, (cudaStream_t)stream>>>(gx, ldgx, whh, bhh, node_off, B, out, ldo, gates,  \
                                                                    hprev);                                            \
    break;
  switch (Hd) {   // the reference instantiates 100 per direction (dgcnv2.py, dgcn_models.py); small sizes for tests
    ERCG_GRU_F(100) ERCG_GRU_F(64) ERCG_GRU_F(48) ERCG_GRU_F(32) ERCG_GRU_F(24) ERCG_GRU_F(16) ERCG_GRU_F(8)
    default: return ERCG_EINVAL;
  }
#undef ERCG_GRU_F
  return finish_launch();
}

extern "C" int ercg_gru_bwd(const float* dout, int64_t ldo, const float* gates, const float* hprev, const float* whh,
                            const int32_t* node_off, int B, int Hd, float* dgx, int64_t lddgx, float* dgh, int64_t lddgh,
                            void* stream) {
  if (B < 0) return ERCG_EINVAL;
  if (B == 0) return ERCG_OK;
  if (!dout || !gates || !hprev || !whh || !node_off || !dgx || !dgh) return ERCG_EINVAL;
  long long want = 2LL * B;
  int grid = (int)(want < 2 * kNumSMs ? want : 2 * kNumSMs);
#define ERCG_GRU_B(HD_)                                                                                                 \
  case HD_:                                                                                                             \
    gru_bwd_kernel<HD_><<<grid, 3 * HD_, 0, (cudaStream_t)stream>>>(dout, ldo, gates, hprev, whh, node_off, B, dgx,     \
                                                                    lddgx, dgh, lddgh);                                 \
    break;
  switch (Hd) {
    ERCG_GRU_B(100) ERCG_GRU_B(64) ERCG_GRU_B(48) ERCG_GRU_B(32) ERCG_GRU_B(24) ERCG_GRU_B(16) ERCG_GRU_B(8)
    default: return ERCG_EINVAL;
  }
#undef ERCG_GRU_B
  return finish_launch();
}
