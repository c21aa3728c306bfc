// K6: packed bidirectional LSTM recurrence (one layer), forward and backward through time.
//
// Replaces the cuDNN/ATen nn.LSTM behind SeqContext (track_mm/dgcn_models.py:10-33: pack_padded_sequence ->
// 2-layer BiLSTM(h = 100 per direction) -> pad_packed_sequence) and MMGCN's text LSTM (track_mm/mmgcn.py:69,114).
// The input transform x_t @ W_ih^T + b_ih + b_hh for ALL utterances and both directions is hoisted into one
// dense GEMM (K2) producing gx[N, 8*Hd] (gate order i,f,g,o per direction, PyTorch layout); this kernel only
// runs the sequential part
//     pre = gx[t] + W_hh h_{t-1};  i,f,o = sigmoid, g = tanh;  c_t = f c_{t-1} + i g;  h_t = o tanh(c_t)
// over the packed node layout (dialogue d occupies rows node_off[d] .. node_off[d+1]), which gives exactly the
// packed-sequence semantics of the reference (no padding step ever runs, h0 = c0 = 0 per dialogue/direction).
//
// One CTA of 4*Hd threads per (direction, slice of dialogues); thread r keeps row r of W_hh (Hd floats) in
// REGISTERS for the whole launch, h_{t-1} is broadcast from shared memory, so a step is Hd FFMAs + 2 barriers.
// The weight gradients are NOT accumulated here: the kernel stores dpre[N, 8*Hd] and h_{t-1}[N, 2*Hd] and the
// caller forms dW_hh = dpre^T @ h_prev, dW_ih = dpre^T @ x, db = colsum(dpre) with the split-K GEMM (K2).
#include "common.cuh"
#include "rnn_cluster.cuh"
#include <math.h>

namespace ercg {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

template <int HD>
__global__ void __launch_bounds__(4 * HD, 1)
lstm_fwd_kernel(const float* __restrict__ gx, long long ldgx, const float* __restrict__ whh,
                const int* __restrict__ node_off, int B, float* __restrict__ out, long long ldo,
                float* __restrict__ gates, float* __restrict__ cells, float* __restrict__ hprev) {
  __shared__ __align__(16) float sh[HD];
  __shared__ float sg[4 * HD];
  const int r = threadIdx.x;
  const int dir = blockIdx.x & 1;
  float w[HD];
  {
    const float* wr = whh + ((long long)dir * 4 * HD + r) * HD;
#pragma unroll
    for (int k = 0; k < HD; ++k) w[k] = wr[k];
  }
  const int stride = gridDim.x >> 1;
  for (int d = blockIdx.x >> 1; d < B; d += stride) {
    const int o = node_off[d], L = node_off[d + 1] - o;
    if (r < HD) sh[r] = 0.f;
    float c = 0.f;
    __syncthreads();
    for (int s = 0; s < L; ++s) {
      const long long t = o + (dir == 0 ? s : L - 1 - s);
      float acc = gx[t * ldgx + dir * 4 * HD + r];
#pragma unroll
      for (int k = 0; k < HD; k += 4) {
        const float4 h4 = *reinterpret_cast<const float4*>(&sh[k]);
        acc = fmaf(w[k], h4.x, acc); acc = fmaf(w[k + 1], h4.y, acc);
        acc = fmaf(w[k + 2], h4.z, acc); acc = fmaf(w[k + 3], h4.w, acc);
      }
      const float a = (r >= 2 * HD && r < 3 * HD) ? tanhf(acc) : sigmoidf_(acc);
      sg[r] = a;
      gates[t * (8 * HD) + dir * 4 * HD + r] = a;
      if (r < HD) hprev[t * (2 * HD) + dir * HD + r] = sh[r];
      __syncthreads();
      if (r < HD) {
        const float ig = sg[r], fg = sg[HD + r], gg = sg[2 * HD + r], og = sg[3 * HD + r];
        c = fmaf(fg, c, ig * gg);
        const float h = og * tanhf(c);
        cells[t * (2 * HD) + dir * HD + r] = c;
        out[t * ldo + dir * HD + r] = h;
        sh[r] = h;
      }
      __syncthreads();
    }
  }
}

// thread (q, k) = (threadIdx.x / HD, threadIdx.x % HD) keeps W_hh[q*HD + j][k], j = 0..HD-1, in registers
template <int HD>
__global__ void __launch_bounds__(4 * HD, 1)
lstm_bwd_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ gates,
                const float* __restrict__ cells, const float* __restrict__ whh, const int* __restrict__ node_off,
                int B, float* __restrict__ dgx, long long lddgx) {
  __shared__ __align__(16) float sdg[4 * HD];     // dpre of the current step
  __shared__ float spart[4 * HD];                 // partial dh_{t-1} per gate block
  const int tid = threadIdx.x, q = tid / HD, k = tid % HD;
  const int dir = blockIdx.x & 1;
  float w[HD];
#pragma unroll
  for (int j = 0; j < HD; ++j) w[j] = whh[((long long)dir * 4 * HD + q * HD + j) * HD + k];
  const int stride = gridDim.x >> 1;
  for (int d = blockIdx.x >> 1; d < B; d += stride) {
    const int o = node_off[d], L = node_off[d + 1] - o;
    float dh_rec = 0.f, dc_next = 0.f;            // meaningful for tid < HD
    __syncthreads();
    for (int s = L - 1; s >= 0; --s) {            // reverse of the forward traversal order
      const long long t = o + (dir == 0 ? s : L - 1 - s);
      if (tid < HD) {
        const float* g = gates + t * (8 * HD) + dir * 4 * HD;
        const float ig = g[tid], fg = g[HD + tid], gg = g[2 * HD + tid], og = g[3 * HD + tid];
        const float c = cells[t * (2 * HD) + dir * HD + tid];
        float cprev = 0.f;
        if (s > 0) {
          const long long tp = o + (dir == 0 ? s - 1 : L - s);
          cprev = cells[tp * (2 * HD) + dir * HD + tid];
        }
        const float dh = dout[t * ldo + dir * HD + tid] + dh_rec;
        const float tc = tanhf(c);
        const float dc = fmaf(dh * og, 1.f - tc * tc, dc_next);
        sdg[tid] = dc * gg * ig * (1.f - ig);
        sdg[HD + tid] = dc * cprev * fg * (1.f - fg);
        sdg[2 * HD + tid] = dc * ig * (1.f - gg * gg);
        sdg[3 * HD + tid] = dh * tc * og * (1.f - og);
        dc_next = dc * fg;
      }
      __syncthreads();
      dgx[t * lddgx + dir * 4 * HD + tid] = sdg[tid];
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < HD; j += 4) {
        const float4 g4 = *reinterpret_cast<const float4*>(&sdg[q * HD + j]);
        acc = fmaf(w[j], g4.x, acc); acc = fmaf(w[j + 1], g4.y, acc);
        acc = fmaf(w[j + 2], g4.z, acc); acc = fmaf(w[j + 3], g4.w, acc);
      }
      spart[tid] = acc;
      __syncthreads();
      if (tid < HD) dh_rec = (spart[tid] + spart[HD + tid]) + (spart[2 * HD + tid] + spart[3 * HD + tid]);
    }
  }
}

__global__ void dropout_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, float p, float scale,
                               unsigned long long seed) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = hash_uniform(seed, (unsigned long long)i) < p ? 0.f : x[i] * scale;
}

// dropout_kernel with the seed offset read from device memory (a step counter that a captured graph advances)
__global__ void dropout_dev_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, float p, float scale,
                                   unsigned long long seed, const unsigned long long* __restrict__ seed_dev) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = hash_uniform(seed + __ldg(seed_dev), (unsigned long long)i) < p ? 0.f : x[i] * scale;
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_lstm_fwd(const float* gx, int64_t ldgx, const float* whh, const int32_t* node_off, int B, int Hd,
                             float* out, int64_t ldo, float* gates, float* cells, float* hprev, void* stream) {
  if (B < 0) return ERCG_EINVAL;
  if (B == 0) return ERCG_OK;
  if (!gx || !whh || !node_off || !out || !gates || !cells || !hprev) return ERCG_EINVAL;
  if (Hd >= RNN_CLUSTER_MIN_HD && Hd <= RNN_CLUSTER_MAX_HD)     // K6c (rnn_cluster.cu)
    return lstm_cluster_fwd(gx, ldgx, whh, node_off, B, Hd, out, ldo, gates, cells, hprev, (cudaStream_t)stream);
  long long want = 2LL * B;
  int grid = (int)(want < 2 * kNumSMs ? want : 2 * kNumSMs);
#define ERCG_LSTM_F(HD_)                                                                                         \
  case HD_:                                                                                                      \
    lstm_fwd_kernel<HD_><<<grid, 4 * HD_, 0, (cudaStream_t)stream>>>(gx, ldgx, whh, node_off, B, out, ldo, gates, \
                                                                     cells, hprev);                              \
    break;
  switch (Hd) {   // the reference instantiates 100 per direction (dgcn.py:59-66, mmgcn.py:69); small sizes for tests
    ERCG_LSTM_F(100) ERCG_LSTM_F(64) ERCG_LSTM_F(48) ERCG_LSTM_F(32) ERCG_LSTM_F(24) ERCG_LSTM_F(16) ERCG_LSTM_F(8)
    default: return ERCG_EINVAL;
  }
#undef ERCG_LSTM_F
  return finish_launch();
}

extern "C" int ercg_lstm_bwd(const float* dout, int64_t ldo, const float* gates, const float* cells, const float* whh,
                             const int32_t* node_off, int B, int Hd, float* dgx, int64_t lddgx, void* stream) {
  if (B < 0) return ERCG_EINVAL;
  if (B == 0) return ERCG_OK;
  if (!dout || !gates || !cells || !whh || !node_off || !dgx) return ERCG_EINVAL;
  if (Hd >= RNN_CLUSTER_MIN_HD && Hd <= RNN_CLUSTER_MAX_HD)
    return lstm_cluster_bwd(dout, ldo, gates, cells, whh, node_off, B, Hd, dgx, lddgx, (cudaStream_t)stream);
  long long want = 2LL * B;
  int grid = (int)(want < 2 * kNumSMs ? want : 2 * kNumSMs);
#define ERCG_LSTM_B(HD_)                                                                                              \
  case HD_:                                                                                                           \
    lstm_bwd_kernel<HD_><<<grid, 4 * HD_, 0, (cudaStream_t)stream>>>(dout, ldo, gates, cells, whh, node_off, B, dgx,  \
                                                                     lddgx);                                          \
    break;
  switch (Hd) {
    ERCG_LSTM_B(100) ERCG_LSTM_B(64) ERCG_LSTM_B(48) ERCG_LSTM_B(32) ERCG_LSTM_B(24) ERCG_LSTM_B(16) ERCG_LSTM_B(8)
    default: return ERCG_EINVAL;
  }
#undef ERCG_LSTM_B
  return finish_launch();
}

extern "C" int ercg_dropout(const float* x, float* out, int64_t n, float p, uint64_t seed, void* stream) {
  if (n < 0 || !(p >= 0.f && p < 1.f)) return ERCG_EINVAL;
  if (n == 0) return ERCG_OK;
  if (!x || !out) return ERCG_EINVAL;
  dropout_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, n, p, 1.f / (1.f - p), seed);
  return finish_launch();
}

extern "C" int ercg_dropout_dev(const float* x, float* out, int64_t n, float p, uint64_t seed, const uint64_t* seed_dev,
                                void* stream) {
  if (!seed_dev || n < 0 || !(p >= 0.f && p < 1.f)) return ERCG_EINVAL;
  if (n == 0) return ERCG_OK;
  if (!x || !out) return ERCG_EINVAL;
  dropout_dev_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      x, out, n, p, 1.f / (1.f - p), seed, reinterpret_cast<const unsigned long long*>(seed_dev));
  return finish_launch();
}
