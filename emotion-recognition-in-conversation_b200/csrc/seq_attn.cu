// K13: dense masked MatchingAttention 'general' / 'general2' of the declare-lab sequence classifiers
// (track_mm/dgcnv2_models.py: MatchingAttention.forward with a mask, LSTMModel / GRUModel / DialogRNNModel's att2 loop),
// and the per-dialogue reversal of DialogRNNModel._reverse_seq.
//
// Query r = q*B + b of dialogue b attends over the L memory rows j*B + b (seq-first).  Per query, with s_j the score:
//   'general'  : s_j = <xq, M_j>,              alpha = softmax_j s_j
//   'general2' : s_j = m_j <xq, m_j M_j>,      p = softmax_j tanh(s_j) (over all L),  alpha_j = p_j m_j / sum_k p_k m_k
//   pool = sum_j alpha_j M_j
// Forward: one CTA per query, CTAs of one dialogue adjacent (block = b*Q + q) so that its L memory rows stay in L2 while
// its Q queries read them.  Warps take positions j (lanes split the D columns, scalar loads: any D, any row alignment),
// the softmax runs over the CTA with block reductions in a fixed order, then a thread per column sums alpha_j M_j in j order.
// Backward, with dalpha_j = <dpool, M_j>:
//   w_j = alpha_j (dalpha_j - sum_k alpha_k dalpha_k) [* (1 - tanh(s_j)^2) m_j^2 for 'general2']
//   dxq = sum_j w_j M_j  (by-query pass, which also stores w),   dM_j = sum_q (alpha_qj dpool_q + w_qj xq_q)  (by-memory-row
//   pass, q in order).  'general2': dp_j = m_j g_j / Z with g_j = dalpha_j - sum_k alpha_k dalpha_k; the softmax backward
//   p_j (dp_j - sum_k p_k dp_k) is alpha_j g_j because sum_k alpha_k g_k = 0 when sum_k alpha_k = 1.
// The dot products and the weighted sums over positions / queries accumulate in fp64 and round once, and the backward keeps
// dalpha, sum_k alpha_k dalpha_k, w and 1 - tanh^2 in fp64 (the difference dalpha_j - sum is a cancellation; fp32 there left
// dM and dx up to 2e-5 from the fp64 truth, four to eight times the reference's own fp32 error).
// No atomics; every sum has a fixed order, so results are bit-reproducible.
#include "common.cuh"
#include <math.h>

namespace ercg {

constexpr int MA_T = 128, MA_W = MA_T / 32;
constexpr int MA_MAXL = 4096, MA_MAXQ = 4096, MA_MAXD = 1024;   // shared memory: 8 L + 4 D bytes <= 48 KB

// fixed-order CTA reductions: lanes, then the warps in warp order
__device__ __forceinline__ float ma_block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = red[0];
#pragma unroll
  for (int w = 1; w < MA_W; ++w) t += red[w];
  return t;
}
__device__ __forceinline__ float ma_block_max(float v, float* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = red[0];
#pragma unroll
  for (int w = 1; w < MA_W; ++w) t = fmaxf(t, red[w]);
  return t;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double ma_block_sum_d(double v, double* red) {
  v = warp_sum_d(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = red[0];
#pragma unroll
  for (int w = 1; w < MA_W; ++w) t += red[w];
  return t;
}

// sc[j] = <v, M_j> for every j (v in shared memory), accumulated in fp64
template <typename T>
__device__ __forceinline__ void ma_dots(const float* __restrict__ M, long long ldm, int L, int B, int D, int b,
                                        const float* v, T* sc) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int j = warp; j < L; j += MA_W) {
    const float* row = M + ((long long)j * B + b) * ldm;
    double acc = 0.0;
    for (int d = lane; d < D; d += 32) acc = fma((double)v[d], (double)row[d], acc);
    acc = warp_sum_d(acc);
    if (lane == 0) sc[j] = (T)acc;
  }
}

__global__ void __launch_bounds__(MA_T)
match_att_fwd_kernel(const float* __restrict__ M, long long ldm, int L, int B, int D, int Q, const float* __restrict__ xq,
                     long long ldq, const float* __restrict__ mask, int general2, float* __restrict__ pool, long long ldp,
                     float* __restrict__ alpha, float* __restrict__ score) {
  extern __shared__ float ma_sm[];
  __shared__ float red[MA_W];
  float* xs = ma_sm;
  float* sc = ma_sm + D;
  const long long blk = blockIdx.x;
  const int b = (int)(blk / Q), q = (int)(blk % Q);
  const long long r = (long long)q * B + b;
  for (int d = threadIdx.x; d < D; d += MA_T) xs[d] = xq[r * ldq + d];
  __syncthreads();
  ma_dots(M, ldm, L, B, D, b, xs, sc);
  __syncthreads();
  const float* mrow = mask ? mask + (long long)b * L : nullptr;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < L; j += MA_T) {
    float s = sc[j];
    if (general2) {
      const float m = mrow ? mrow[j] : 1.f;
      s = m * (m * s);
    }
    score[r * L + j] = s;
    const float v = general2 ? tanhf(s) : s;
    sc[j] = v;
    mx = fmaxf(mx, v);
  }
  mx = ma_block_max(mx, red);
  float z = 0.f;
  for (int j = threadIdx.x; j < L; j += MA_T) {
    const float e = expf(sc[j] - mx);
    sc[j] = e;
    z += e;
  }
  z = ma_block_sum(z, red);
  float zm = 0.f;
  for (int j = threadIdx.x; j < L; j += MA_T) {
    float a = sc[j] / z;
    if (general2) a *= mrow ? mrow[j] : 1.f;
    sc[j] = a;
    zm += a;
  }
  if (general2) {
    zm = ma_block_sum(zm, red);
    for (int j = threadIdx.x; j < L; j += MA_T) sc[j] /= zm;     // an all-zero mask row: 0 / 0 = NaN, as the reference
  }
  __syncthreads();
  for (int j = threadIdx.x; j < L; j += MA_T) alpha[r * L + j] = sc[j];
  for (int d = threadIdx.x; d < D; d += MA_T) {
    double acc = 0.0;
    for (int j = 0; j < L; ++j) acc = fma((double)sc[j], (double)M[((long long)j * B + b) * ldm + d], acc);
    pool[r * ldp + d] = (float)acc;
  }
}

__global__ void __launch_bounds__(MA_T)
match_att_bwd_q_kernel(const float* __restrict__ M, long long ldm, int L, int B, int D, int Q, const float* __restrict__ mask,
                       int general2, const float* __restrict__ alpha, const float* __restrict__ score,
                       const float* __restrict__ dpool, long long lddp, float* __restrict__ w, float* __restrict__ dxq,
                       long long lddxq) {
  extern __shared__ double ma_smd[];
  __shared__ double red[MA_W];
  double* sc = ma_smd;                                           // [L]
  float* dps = reinterpret_cast<float*>(ma_smd + L);             // [D]
  const long long blk = blockIdx.x;
  const int b = (int)(blk / Q), q = (int)(blk % Q);
  const long long r = (long long)q * B + b;
  for (int d = threadIdx.x; d < D; d += MA_T) dps[d] = dpool[r * lddp + d];
  __syncthreads();
  ma_dots(M, ldm, L, B, D, b, dps, sc);                          // dalpha_j
  __syncthreads();
  const float* arow = alpha + r * L;
  double s = 0.0;
  for (int j = threadIdx.x; j < L; j += MA_T) s = fma((double)arow[j], sc[j], s);
  s = ma_block_sum_d(s, red);
  const float* mrow = mask ? mask + (long long)b * L : nullptr;
  for (int j = threadIdx.x; j < L; j += MA_T) {
    double g = (double)arow[j] * (sc[j] - s);
    if (general2) {
      const double u = tanh((double)score[r * L + j]), m = mrow ? mrow[j] : 1.0;
      g = g * (1.0 - u * u) * (m * m);
    }
    sc[j] = g;
    w[r * L + j] = (float)g;
  }
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += MA_T) {
    double acc = 0.0;
    for (int j = 0; j < L; ++j) acc = fma(sc[j], (double)M[((long long)j * B + b) * ldm + d], acc);
    dxq[r * lddxq + d] = (float)acc;
  }
}

constexpr int MA_QCHUNK = 256;
__global__ void __launch_bounds__(MA_T)
match_att_bwd_m_kernel(int L, int B, int D, int Q, const float* __restrict__ xq, long long ldq, const float* __restrict__ alpha,
                       const float* __restrict__ w, const float* __restrict__ dpool, long long lddp, float* __restrict__ dM,
                       long long lddm) {
  __shared__ float sa[MA_QCHUNK], sw[MA_QCHUNK];
  const long long blk = blockIdx.x;
  const int b = (int)(blk / L), j = (int)(blk % L);
  const int nd = (D + MA_T - 1) / MA_T;                          // <= 8 columns per thread
  double acc[MA_MAXD / MA_T];
#pragma unroll
  for (int k = 0; k < MA_MAXD / MA_T; ++k) acc[k] = 0.0;
  for (int q0 = 0; q0 < Q; q0 += MA_QCHUNK) {
    const int nq = min(MA_QCHUNK, Q - q0);
    __syncthreads();
    for (int t = threadIdx.x; t < nq; t += MA_T) {
      const long long idx = ((long long)(q0 + t) * B + b) * L + j;
      sa[t] = alpha[idx];
      sw[t] = w[idx];
    }
    __syncthreads();
    for (int t = 0; t < nq; ++t) {
      const long long r = (long long)(q0 + t) * B + b;
      const float a = sa[t], g = sw[t];
#pragma unroll
      for (int k = 0; k < MA_MAXD / MA_T; ++k) {
        const int d = threadIdx.x + k * MA_T;
        if (k < nd && d < D) acc[k] = fma((double)g, (double)xq[r * ldq + d], fma((double)a, (double)dpool[r * lddp + d], acc[k]));
      }
    }
  }
  const long long row = (long long)j * B + b;
#pragma unroll
  for (int k = 0; k < MA_MAXD / MA_T; ++k) {
    const int d = threadIdx.x + k * MA_T;
    if (k < nd && d < D) dM[row * lddm + d] = (float)acc[k];
  }
}

// out[t*B + b] = x[(c_b - 1 - t)*B + b] for t < c_b, 0 for c_b <= t < Lout;  c_b = counts[b] clamped to [0, Lin]
__global__ void __launch_bounds__(256)
reverse_seq_kernel(const float* __restrict__ x, long long ldx, int Lin, int B, int D, const int* __restrict__ counts,
                   float* __restrict__ out, long long ldo, long long total) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= total) return;
  const long long row = i / D;
  const int d = (int)(i - row * D);
  const int t = (int)(row / B), b = (int)(row - (long long)t * B);
  const int c = min(max(counts[b], 0), Lin);
  out[row * ldo + d] = t < c ? x[((long long)(c - 1 - t) * B + b) * ldx + d] : 0.f;
}

static int match_att_check(int L, int B, int D, int Q, long long ldm, long long ldq, int kind) {
  if (L < 1 || L > MA_MAXL || Q < 1 || Q > MA_MAXQ || D < 1 || D > MA_MAXD || B < 0 || (kind != ERCG_MATCH_GENERAL &&
      kind != ERCG_MATCH_GENERAL2) || ldm < D || ldq < D)
    return ERCG_EINVAL;
  if ((long long)B * Q > 0x7fffffffLL || (long long)B * L > 0x7fffffffLL) return ERCG_ERANGE;
  return ERCG_OK;
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_match_att_fwd(const float* M, int64_t ldm, int L, int B, int D, int Q, const float* xq, int64_t ldq,
                                  const float* mask, int kind, float* pool, int64_t ldp, float* alpha, float* score,
                                  void* stream) {
  const int rc = match_att_check(L, B, D, Q, ldm, ldq, kind);
  if (rc != ERCG_OK) return rc;
  if (B == 0) return ERCG_OK;
  if (!M || !xq || !pool || !alpha || !score || ldp < D) return ERCG_EINVAL;
  match_att_fwd_kernel<<<(unsigned)((long long)B * Q), MA_T, (size_t)(D + L) * sizeof(float), (cudaStream_t)stream>>>(
      M, ldm, L, B, D, Q, xq, ldq, kind == ERCG_MATCH_GENERAL2 ? mask : nullptr, kind == ERCG_MATCH_GENERAL2, pool, ldp, alpha,
      score);
  return finish_launch();
}

extern "C" int ercg_match_att_bwd(const float* M, int64_t ldm, int L, int B, int D, int Q, const float* xq, int64_t ldq,
                                  const float* mask, int kind, const float* alpha, const float* score, const float* dpool,
                                  int64_t lddp, float* w, float* dxq, int64_t lddxq, float* dM, int64_t lddm, void* stream) {
  const int rc = match_att_check(L, B, D, Q, ldm, ldq, kind);
  if (rc != ERCG_OK) return rc;
  if (B == 0) return ERCG_OK;
  if (!M || !xq || !alpha || !score || !dpool || !w || !dxq || !dM || lddp < D || lddxq < D || lddm < D) return ERCG_EINVAL;
  match_att_bwd_q_kernel<<<(unsigned)((long long)B * Q), MA_T, (size_t)L * sizeof(double) + (size_t)D * sizeof(float),
                           (cudaStream_t)stream>>>(
      M, ldm, L, B, D, Q, kind == ERCG_MATCH_GENERAL2 ? mask : nullptr, kind == ERCG_MATCH_GENERAL2, alpha, score, dpool, lddp,
      w, dxq, lddxq);
  int st = finish_launch();
  if (st != ERCG_OK) return st;
  match_att_bwd_m_kernel<<<(unsigned)((long long)B * L), MA_T, 0, (cudaStream_t)stream>>>(L, B, D, Q, xq, ldq, alpha, w, dpool,
                                                                                          lddp, dM, lddm);
  return finish_launch();
}

extern "C" int ercg_reverse_seq(const float* x, int64_t ldx, int Lin, int B, int D, const int32_t* counts, float* out,
                                int64_t ldo, int Lout, void* stream) {
  if (Lin < 0 || Lout < 0 || B < 0 || D < 0 || ldx < D || ldo < D) return ERCG_EINVAL;
  const long long total = (long long)Lout * B * D;
  if (total == 0) return ERCG_OK;
  if (!x || !counts || !out) return ERCG_EINVAL;
  reverse_seq_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, Lin, B, D, counts, out, ldo,
                                                                                         total);
  return finish_launch();
}
