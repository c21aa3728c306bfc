// K2 (exact-fp32 path): tiled SIMT GEMMs for the dense feature transforms.
//
//   gemm_nn : C[M,N]   = act(A[M,K] @ B[K,N] + bias)      forward transforms and input gradients
//   gemm_tn : C[K1,N1] = A[M,K1]^T @ B[M,N1]              weight gradients (contraction over utterances)
//   colsum  : out[N]   = sum_m A[m,N]                     bias gradients
// Replaces nn.Linear (track_mm/cogmen.py:103-105,116-122), the relation weights of RGCNConv
// (cogmen.py:65, models/rgcn.py:329-343) as one GEMM against [K,(R+1)*out], and the four Linears of
// TransformerConv (cogmen.py:66).  fp32 FFMA with fp32 accumulation: this is the parity path that
// meets the 1e-5 relative bound of BASELINE.json without any reduced-precision split.
//
// Tile: 128x128x16, 256 threads, 8x8 register micro-tile (two 4-wide halves 64 apart in each
// dimension so the shared-memory reads are conflict-free float4 / broadcasts), double-buffered
// shared memory with register prefetch of the next K-slab.
#include "common.cuh"
#include "gemm_skinny.cuh"
#include "col_stream.cuh"
#include <algorithm>

namespace ercg {

constexpr int BM = 128, BN = 128, BK = 16, GT = 256;

struct Epilogue {
  const float* bias; int act; const float* aux; long long ldaux; float aux_scale; float drop_p; unsigned long long seed;
  // GCNII epilogues (internal act codes, see ercg_gcnii_layer_fwd / ercg_gcnii_layer_bwd_input below)
  const float* aux2; long long ldaux2; float c_acc, c1, c2; int half;
  const unsigned long long* seed_dev = nullptr;   // optional device word added to `seed` (a step counter: fresh mask per graph replay)
};
constexpr int ACT_GCNII_FWD = 16;   // x = [relu if half](c_acc*acc + c1*aux[m,n] + c2*aux2[m,n]) (+ inverted dropout)
constexpr int ACT_GCNII_BWD = 17;   // x = c_acc*acc + (n < half ? c1*aux[m,n] : c2*aux[m,n-half])

__device__ __forceinline__ void mma_slab(const float (*As)[BM + 4], const float (*Bs)[BN + 4], float acc[8][8], int ty, int tx) {
#pragma unroll
  for (int k = 0; k < BK; ++k) {
    float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
    float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
    float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
    float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);
    float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
}

// ------------------------------------------------------------------------------------------ NN
// A-slab loader: thread t owns row (t & 127) and 8 consecutive k starting at (t >> 7) * 8.
template <bool VEC_A>
__device__ __forceinline__ void load_a_nn(const float* __restrict__ arow, bool row_ok, int k0, int K, float r[8]) {
  if (!row_ok) {
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = 0.f;
    return;
  }
  if (VEC_A && k0 + 8 <= K) {
    float4 v0 = ld4(arow + k0), v1 = ld4(arow + k0 + 4);
    r[0] = v0.x; r[1] = v0.y; r[2] = v0.z; r[3] = v0.w; r[4] = v1.x; r[5] = v1.y; r[6] = v1.z; r[7] = v1.w;
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = (k0 + i < K) ? __ldg(arow + k0 + i) : 0.f;
  }
}

// B-slab loader: thread t owns k rows (t >> 5) and (t >> 5) + 8, columns (t & 31) * 4 .. +3
template <bool VEC_B>
__device__ __forceinline__ void load_b_nn(const float* __restrict__ B, long long ldb, int k, int K, int n, int N, float r[4]) {
  if (k >= K) { r[0] = r[1] = r[2] = r[3] = 0.f; return; }
  const float* p = B + (long long)k * ldb + n;
  if (VEC_B && n + 4 <= N) {
    float4 v = ld4(p);
    r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) r[i] = (n + i < N) ? __ldg(p + i) : 0.f;
  }
}

#define ERCG_NN_KERNEL gemm_nn_kernel
#define ERCG_NN_GCNII_SEED ep.seed
#include "gemm_nn_kernel.cuh"

// ercg_gcnii_layer_fwd_dev: the GCNII layer with its dropout seed offset read from device memory
#define ERCG_NN_KERNEL gcnii_fwd_dev_kernel
#define ERCG_NN_GCNII_SEED (ep.seed + __ldg(ep.seed_dev))
#include "gemm_nn_kernel.cuh"

// ------------------------------------------------------------------------------------------ TN
// C[K1,N1] (+)= sum over rows m in this CTA's slab of A[m,k1] * B[m,n1]
// loaders: thread t owns slab rows (t >> 5) and (t >> 5) + 8, columns (t & 31) * 4 .. +3 of both A and B
template <bool VEC>
__device__ __forceinline__ void load_row4(const float* __restrict__ base, bool ok, int c, int Cn, float r[4]) {
  if (!ok) { r[0] = r[1] = r[2] = r[3] = 0.f; return; }
  if (VEC && c + 4 <= Cn) {
    float4 v = ld4(base + c);
    r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) r[i] = (c + i < Cn) ? __ldg(base + c + i) : 0.f;
  }
}

template <bool VEC_A, bool VEC_B>
__global__ void __launch_bounds__(GT, 2)
gemm_tn_kernel(const float* __restrict__ A, long long lda, const int* __restrict__ a_rows,
               const float* __restrict__ B, long long ldb, float* __restrict__ P /* [S,K1,N1] or C */, long long ldp,
               long long M, int K1, int N1, long long rows_per_split, long long split_stride) {
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Bs[2][BK][BN + 4];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int k0 = blockIdx.x * BM;     // K1 tile
  const int n0 = blockIdx.y * BN;     // N1 tile
  const long long mbeg = (long long)blockIdx.z * rows_per_split;
  long long mend = mbeg + rows_per_split;
  if (mend > M) mend = M;
  const int r0 = t >> 5, c4 = (t & 31) * 4;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  auto arow = [&](long long m) -> const float* { return A + (a_rows ? (long long)a_rows[m] : m) * lda + k0; };
  float ra0[4], ra1[4], rb0[4], rb1[4];
  auto fetch = [&](long long m) {
    const bool ok0 = m + r0 < mend, ok1 = m + r0 + 8 < mend;
    load_row4<VEC_A>(ok0 ? arow(m + r0) : A, ok0, c4, K1 - k0, ra0);
    load_row4<VEC_A>(ok1 ? arow(m + r0 + 8) : A, ok1, c4, K1 - k0, ra1);
    load_row4<VEC_B>(B + (m + r0) * ldb + n0, ok0, c4, N1 - n0, rb0);
    load_row4<VEC_B>(B + (m + r0 + 8) * ldb + n0, ok1, c4, N1 - n0, rb1);
  };
  auto stash = [&](int b) {
    *reinterpret_cast<float4*>(&As[b][r0][c4]) = make_float4(ra0[0], ra0[1], ra0[2], ra0[3]);
    *reinterpret_cast<float4*>(&As[b][r0 + 8][c4]) = make_float4(ra1[0], ra1[1], ra1[2], ra1[3]);
    *reinterpret_cast<float4*>(&Bs[b][r0][c4]) = make_float4(rb0[0], rb0[1], rb0[2], rb0[3]);
    *reinterpret_cast<float4*>(&Bs[b][r0 + 8][c4]) = make_float4(rb1[0], rb1[1], rb1[2], rb1[3]);
  };
  int buf = 0;
  if (mbeg < mend) {
    fetch(mbeg);
    stash(0);
    __syncthreads();
    for (long long m = mbeg; m < mend; m += BK) {
      const bool more = m + BK < mend;
      if (more) fetch(m + BK);
      mma_slab(As[buf], Bs[buf], acc, ty, tx);
      if (more) {
        stash(buf ^ 1);
        __syncthreads();
        buf ^= 1;
      }
    }
  }
  float* out = P + (long long)blockIdx.z * split_stride;
#pragma unroll
  for (int ih = 0; ih < 2; ++ih)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kk = k0 + ih * 64 + ty * 4 + i;
      if (kk >= K1) continue;
#pragma unroll
      for (int jh = 0; jh < 2; ++jh)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int nn = n0 + jh * 64 + tx * 4 + j;
          if (nn < N1) out[(long long)kk * ldp + nn] = acc[ih * 4 + i][jh * 4 + j];
        }
    }
}

// C[i] = sum_s P[s][i], fixed order
__global__ void reduce_splits_kernel(const float* __restrict__ P, long long split_stride, int S,
                                     float* __restrict__ C, long long ldc, int rows, int cols) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)rows * cols) return;
  float s = 0.f;
  for (int z = 0; z < S; ++z) s += P[(long long)z * split_stride + idx];
  const int r = (int)(idx / cols), c = (int)(idx % cols);
  C[(long long)r * ldc + c] = s;
}

// Same sum for MANY splits and few outputs (the skinny weight gradients: S ~ 600 slabs, K1*N1 ~ 600 outputs): 8 lanes per
// output take the splits round-robin, then a fixed 3-step shuffle tree => still bit-reproducible, 8x shorter serial chain.
__global__ void __launch_bounds__(256)
reduce_splits_wide_kernel(const float* __restrict__ P, long long split_stride, int S, float* __restrict__ C, long long ldc,
                          int rows, int cols) {
  const int sub = threadIdx.x & 7;
  const long long idx = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const bool ok = idx < (long long)rows * cols;
  float s = 0.f;
  if (ok)
    for (int z = sub; z < S; z += 8) s += P[(long long)z * split_stride + idx];
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  if (ok && sub == 0) {
    const int r = (int)(idx / cols), c = (int)(idx % cols);
    C[(long long)r * ldc + c] = s;
  }
}

// column sums: block b sums rows [b*CS_RPB, (b+1)*CS_RPB) -> partial[b][N]; the final kernel reduces the partials with
// the same (32 columns x 8 row-lanes) pattern in fp64.  Fixed order => bit-reproducible.
constexpr int CS_RPB = 256;
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const float* __restrict__ A, long long lda, long long M, int N, float* __restrict__ partial) {
  __shared__ float sm[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long rbeg = (long long)blockIdx.x * CS_RPB;
  long long rend = rbeg + CS_RPB;
  if (rend > M) rend = M;
  for (int c0 = 0; c0 < N; c0 += 32) {
    const int c = c0 + tx;
    float s = 0.f;
    if (c < N) {
      long long r = rbeg + ty;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      for (; r + 24 < rend; r += 32) {
        s0 += A[r * lda + c]; s1 += A[(r + 8) * lda + c]; s2 += A[(r + 16) * lda + c]; s3 += A[(r + 24) * lda + c];
      }
      for (; r < rend; r += 8) s0 += A[r * lda + c];
      s = (s0 + s1) + (s2 + s3);
    }
    sm[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && c < N) {
      float tot = 0.f;
#pragma unroll
      for (int y = 0; y < 8; ++y) tot += sm[y][tx];
      partial[(long long)blockIdx.x * N + c] = tot;
    }
    __syncthreads();
  }
}
// float4 version for 16-byte aligned rows: one warp load covers up to 512 bytes of a row, rows unrolled x4
__global__ void __launch_bounds__(256)
colsum_partial_v4_kernel(const float* __restrict__ A, long long lda, long long M, int N, float* __restrict__ partial) {
  __shared__ float4 sm[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long rbeg = (long long)blockIdx.x * CS_RPB;
  long long rend = rbeg + CS_RPB;
  if (rend > M) rend = M;
  for (int c0 = 0; c0 < N; c0 += 128) {
    const int c = c0 + 4 * tx;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < N) {
      long long r = rbeg + ty;
      for (; r + 24 < rend; r += 32) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ld4_stream(A + (r + 8 * u) * lda + c);
#pragma unroll
        for (int u = 0; u < 4; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
      }
      for (; r < rend; r += 8) {
        const float4 v = ld4_stream(A + r * lda + c);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
    }
    sm[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && c < N) {
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int y = 0; y < 8; ++y) { const float4 a = sm[y][tx]; t.x += a.x; t.y += a.y; t.z += a.z; t.w += a.w; }
      float* p0 = partial + (long long)blockIdx.x * N + c;
      p0[0] = t.x;
      if (c + 1 < N) p0[1] = t.y;
      if (c + 2 < N) p0[2] = t.z;
      if (c + 3 < N) p0[3] = t.w;
    }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(256)
colsum_final_kernel(const float* __restrict__ partial, int nblocks, int N, float* __restrict__ out) {
  __shared__ double sm[FIN_ROWS][FIN_COLS + 1];
  const int c = blockIdx.x * FIN_COLS + (threadIdx.x & (FIN_COLS - 1));
  const double tot = fin_reduce(partial, nblocks, N, c, c < N, sm);
  if (threadIdx.x < FIN_COLS && c < N) out[c] = (float)tot;
}

// skinny weight gradient (N1 <= 16, K1 <= 256, no row gather): slabs of rows, one block each
static bool tn_skinny(int64_t M, int K1, int N1, bool gather) { return !gather && N1 <= SK_MAXN && K1 <= 256 && M >= 1024; }
static void tn_skinny_plan(int64_t M, int K1, int& S, long long& rps, int& groups, int& KP) {
  KP = (K1 + 31) / 32 * 32;
  groups = 512 / KP;
  long long want = (long long)kNumSMs * 4;
  long long maxs = (M + 255) / 256;
  if (want > maxs) want = maxs;
  if (want < 1) want = 1;
  rps = (M + want - 1) / want;
  S = (int)((M + rps - 1) / rps);
}

static void tn_plan(int64_t M, int K1, int N1, int& S, long long& rows_per_split) {
  const long long tiles = (long long)((K1 + BM - 1) / BM) * ((N1 + BN - 1) / BN);
  long long want = (2LL * kNumSMs + tiles - 1) / tiles;      // ~2 CTAs per SM in flight
  long long maxs = (M + 511) / 512;                          // at least 512 rows per slab
  if (maxs < 1) maxs = 1;
  if (want > maxs) want = maxs;
  if (want < 1) want = 1;
  rows_per_split = (M + want - 1) / want;
  rows_per_split = (rows_per_split + BK - 1) / BK * BK;
  if (rows_per_split < BK) rows_per_split = BK;
  S = (int)((M + rows_per_split - 1) / rows_per_split);
  if (S < 1) S = 1;
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_gemm_nn(const float* A, int64_t lda, const int32_t* a_rows, const float* B, int64_t ldb,
                            const float* bias, float* C, int64_t ldc, int64_t M, int N, int K, int act,
                            const float* aux, int64_t ldaux, float aux_scale, float drop_p, uint64_t seed,
                            const uint64_t* seed_dev, void* stream) {
  if (M < 0 || N < 0 || K < 0) return ERCG_EINVAL;
  if (M == 0 || N == 0) return ERCG_OK;
  if (!A || !B || !C || lda < K || ldb < N || ldc < N) return ERCG_EINVAL;
  if (act < 0 || act > 3 || (act == ERCG_ACT_MASK_POS && !aux)) return ERCG_EINVAL;
  if (act == ERCG_ACT_RELU_DROPOUT && !(drop_p >= 0.f && drop_p < 1.f)) return ERCG_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (!a_rows && act == ERCG_ACT_NONE && M >= 1024 && K > 0) {          // skinny shapes: see gemm_skinny.cuh
    if (N <= SK_MAXN && K <= 2048) {
      const int NN = N <= 8 ? 8 : 16;
      const unsigned grid = (unsigned)std::min<long long>((long long)kNumSMs * 16, (long long)((M + 7) / 8));
      const size_t sm = (size_t)((K + 3) & ~3) * NN * sizeof(float);
      if (((lda & 3) == 0) && aligned16(A) && (K & 3) == 0 && K <= 128) {
        const unsigned g8 = (unsigned)std::min<long long>((long long)kNumSMs * 16, (long long)((M + 31) / 32));
        if (NN == 8) skinny_nn_small_n_q8_kernel<8><<<g8, 256, sm, st>>>(A, lda, B, ldb, bias, C, ldc, M, N, K);
        else skinny_nn_small_n_q8_kernel<16><<<g8, 256, sm, st>>>(A, lda, B, ldb, bias, C, ldc, M, N, K);
        return finish_launch();
      }
      if (NN == 8) skinny_nn_small_n_kernel<8><<<grid, 256, sm, st>>>(A, lda, B, ldb, bias, C, ldc, M, N, K);
      else skinny_nn_small_n_kernel<16><<<grid, 256, sm, st>>>(A, lda, B, ldb, bias, C, ldc, M, N, K);
      return finish_launch();
    }
    if (K <= SK_MAXN && N <= 1024) {
      const int NP = (N + 3) / 4 * 4;
      const long long total = M * (NP / 4);
      const unsigned grid = (unsigned)std::min<long long>((long long)kNumSMs * 16, (total + 255) / 256);
      skinny_nn_small_k_kernel<<<grid, 256, (size_t)(K + 1) * NP * sizeof(float), st>>>(A, lda, B, ldb, bias, C, ldc, M, N, K);
      return finish_launch();
    }
  }
  Epilogue ep{bias, act, aux, (long long)ldaux, aux_scale, drop_p, (unsigned long long)seed, nullptr, 0, 1.f, 0.f, 0.f, 0};
  ep.seed_dev = reinterpret_cast<const unsigned long long*>(seed_dev);
  const bool va = ((lda & 3) == 0) && aligned16(A);
  const bool vb = ((ldb & 3) == 0) && aligned16(B);
  long long gm = (M + BM - 1) / BM;
  if (gm > 2147483647LL) return ERCG_ERANGE;
  dim3 grid((unsigned)gm, (unsigned)((N + BN - 1) / BN));
  if (va && vb) gemm_nn_kernel<true, true><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, C, ldc, M, N, K, ep);
  else if (va) gemm_nn_kernel<true, false><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, C, ldc, M, N, K, ep);
  else if (vb) gemm_nn_kernel<false, true><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, C, ldc, M, N, K, ep);
  else gemm_nn_kernel<false, false><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, C, ldc, M, N, K, ep);
  return finish_launch();
}

extern "C" size_t ercg_gemm_tn_workspace_bytes(int64_t M, int K1, int N1) {
  if (M <= 0 || K1 <= 0 || N1 <= 0) return 0;
  int S; long long rps;
  tn_plan(M, K1, N1, S, rps);
  size_t need = S > 1 ? (size_t)S * K1 * N1 * sizeof(float) : 0;
  if (tn_skinny(M, K1, N1, false)) {
    int g, kp;
    tn_skinny_plan(M, K1, S, rps, g, kp);
    const size_t n2 = (size_t)S * K1 * N1 * sizeof(float);
    if (n2 > need) need = n2;
  }
  return need;
}

extern "C" int ercg_gemm_tn(const float* A, int64_t lda, const int32_t* a_rows, const float* B, int64_t ldb,
                            float* C, int64_t ldc, int64_t M, int K1, int N1,
                            void* workspace, size_t workspace_bytes, void* stream) {
  if (M < 0 || K1 < 0 || N1 < 0) return ERCG_EINVAL;
  if (K1 == 0 || N1 == 0) return ERCG_OK;
  if (!C || ldc < N1) return ERCG_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (M == 0) {   // empty contraction -> zeros
    cudaMemset2DAsync(C, ldc * sizeof(float), 0, (size_t)N1 * sizeof(float), K1, st);
    return ERCG_OK;
  }
  if (!A || !B || lda < K1 || ldb < N1) return ERCG_EINVAL;
  int S; long long rps;
  if (tn_skinny(M, K1, N1, a_rows != nullptr)) {
    int groups, KP;
    tn_skinny_plan(M, K1, S, rps, groups, KP);
    const size_t need2 = (size_t)S * K1 * N1 * sizeof(float);
    if (need2 <= workspace_bytes && workspace) {
      float* Pw = reinterpret_cast<float*>(workspace);
      const int NN = N1 <= 8 ? 8 : 16;
      if (((lda & 3) == 0) && aligned16(A) && (K1 & 3) == 0 && NN == 8) {
        const int KQ = K1 / 4;
        int g4 = 512 / KQ;
        const int cap = (int)(48 * 1024 / ((size_t)K1 * N1 * sizeof(float)));
        if (g4 > cap) g4 = cap;
        if (g4 >= 1) {
          const size_t sm4 = (size_t)g4 * K1 * N1 * sizeof(float);
          skinny_tn_small_n_v4_kernel<8><<<S, 512, sm4, st>>>(A, lda, B, ldb, Pw, M, K1, N1, rps, g4);
          int rc4 = finish_launch();
          if (rc4 != ERCG_OK) return rc4;
          const long long tot4 = (long long)K1 * N1;
          reduce_splits_wide_kernel<<<(unsigned)((tot4 * 8 + 255) / 256), 256, 0, st>>>(Pw, tot4, S, C, ldc, K1, N1);
          return finish_launch();
        }
      }
      const size_t sm = (size_t)groups * KP * NN * sizeof(float);
      if (NN == 8) skinny_tn_small_n_kernel<8><<<S, 512, sm, st>>>(A, lda, B, ldb, Pw, M, K1, N1, rps, groups, KP);
      else skinny_tn_small_n_kernel<16><<<S, 512, sm, st>>>(A, lda, B, ldb, Pw, M, K1, N1, rps, groups, KP);
      int rc2 = finish_launch();
      if (rc2 != ERCG_OK) return rc2;
      const long long tot = (long long)K1 * N1;
      reduce_splits_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(Pw, tot, S, C, ldc, K1, N1);
      return finish_launch();
    }
  }
  tn_plan(M, K1, N1, S, rps);
  const size_t need = S > 1 ? (size_t)S * K1 * N1 * sizeof(float) : 0;
  if (need > workspace_bytes || (need && !workspace)) return ERCG_EWORKSPACE;
  const bool va = ((lda & 3) == 0) && aligned16(A);
  const bool vb = ((ldb & 3) == 0) && aligned16(B);
  dim3 grid((K1 + BM - 1) / BM, (N1 + BN - 1) / BN, S);
  float* P = S > 1 ? reinterpret_cast<float*>(workspace) : C;
  const long long ldp = S > 1 ? N1 : ldc;
  const long long ss = S > 1 ? (long long)K1 * N1 : 0;
  if (va && vb) gemm_tn_kernel<true, true><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, P, ldp, M, K1, N1, rps, ss);
  else if (va) gemm_tn_kernel<true, false><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, P, ldp, M, K1, N1, rps, ss);
  else if (vb) gemm_tn_kernel<false, true><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, P, ldp, M, K1, N1, rps, ss);
  else gemm_tn_kernel<false, false><<<grid, GT, 0, st>>>(A, lda, a_rows, B, ldb, P, ldp, M, K1, N1, rps, ss);
  int rc = finish_launch();
  if (rc != ERCG_OK) return rc;
  if (S > 1) {
    const long long tot = (long long)K1 * N1;
    reduce_splits_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(P, ss, S, C, ldc, K1, N1);
    rc = finish_launch();
  }
  return rc;
}

extern "C" size_t ercg_colsum_workspace_bytes(int64_t M, int N) {
  if (M <= 0 || N <= 0) return 0;
  const size_t a = (size_t)((M + CS_RPB - 1) / CS_RPB) * N * sizeof(float), b = (size_t)CS_MAX_BLOCKS * N * sizeof(float);
  return a > b ? a : b;
}

extern "C" int ercg_colsum(const float* A, int64_t lda, int64_t M, int N, float* out,
                           void* workspace, size_t workspace_bytes, void* stream) {
  if (M < 0 || N < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!out) return ERCG_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (M == 0) { cudaMemsetAsync(out, 0, (size_t)N * sizeof(float), st); return ERCG_OK; }
  if (!A || lda < N) return ERCG_EINVAL;
  const size_t need = ercg_colsum_workspace_bytes(M, N);
  if (need > workspace_bytes || !workspace) return ERCG_EWORKSPACE;
  int nb = (int)((M + CS_RPB - 1) / CS_RPB);
  if (col_stream_ok(A, lda, N, M)) {      // contiguous rows: flat float4 stream (col_stream.cuh)
    const long long total4 = M * (long long)(N >> 2);
    nb = col_stream_blocks(N >> 2, total4);
    col_stream_kernel<2><<<nb, 256, 0, st>>>(A, nullptr, nullptr, nullptr, 0.f, nullptr, nullptr, 0.f, total4, N >> 2,
                                             reinterpret_cast<float*>(workspace));
  } else if (col_stream2_ok(A, lda, N, M)) {
    const long long total2 = M * (long long)(N >> 1);
    nb = col_stream_blocks(N >> 1, total2);
    col_stream2_kernel<<<nb, 256, 0, st>>>(A, total2, N >> 1, reinterpret_cast<float*>(workspace));
  } else if ((N & 3) == 0 && (lda & 3) == 0 && aligned16(A))
    colsum_partial_v4_kernel<<<nb, 256, 0, st>>>(A, lda, M, N, reinterpret_cast<float*>(workspace));
  else
    colsum_partial_kernel<<<nb, 256, 0, st>>>(A, lda, M, N, reinterpret_cast<float*>(workspace));
  int rc = finish_launch();
  if (rc != ERCG_OK) return rc;
  colsum_final_kernel<<<fin_blocks(N), 256, 0, st>>>(reinterpret_cast<const float*>(workspace), nb, N, out);
  return finish_launch();
}

// ---------------------------------------------------------------------------------------------
// GCNII layer (GraphConvolution.forward with variant=True, residual=False; track_mm/mmgcn_models.py:27-39)
//   out = dropout(relu(theta * [hi | h0] @ W + (1 - theta) * ((1 - alpha) * hi + alpha * h0)))
// [hi | h0] is never materialised: the A operand is read from two sources split at k = H.
// The ReLU and the NEXT layer's input dropout (GCNII_lyc.forward :388-392) are the epilogue.
// ---------------------------------------------------------------------------------------------
// argument checks of both GCNII forward entries; ERCG_OK with grid set = launch, ERCG_OK with grid.x == 0 = nothing to do
static int gcnii_fwd_check(const float* hi, int64_t ldhi, const float* h0, int64_t ldh0, const float* W, int64_t ldw,
                           const float* out, int64_t ldo, int64_t M, int H, float drop_p, dim3& grid) {
  grid = dim3(0, 0, 0);
  if (M < 0 || H <= 0 || (H & 7)) return ERCG_EINVAL;
  if (M == 0) return ERCG_OK;
  if (!hi || !h0 || !W || !out || ldhi < H || ldh0 < H || ldw < H || ldo < H) return ERCG_EINVAL;
  if (!(drop_p >= 0.f && drop_p < 1.f)) return ERCG_EINVAL;
  if (!aligned16(hi) || !aligned16(h0) || !aligned16(W) || (ldhi & 3) || (ldh0 & 3) || (ldw & 3)) return ERCG_EALIGN;
  long long gm = (M + BM - 1) / BM;
  if (gm > 2147483647LL) return ERCG_ERANGE;
  grid = dim3((unsigned)gm, (unsigned)((H + BN - 1) / BN));
  return ERCG_OK;
}

extern "C" int ercg_gcnii_layer_fwd(const float* hi, int64_t ldhi, const float* h0, int64_t ldh0, const float* W,
                                    int64_t ldw, float* out, int64_t ldo, int64_t M, int H, float theta, float alpha,
                                    int relu, float drop_p, uint64_t seed, void* stream) {
  dim3 grid;
  const int rc = gcnii_fwd_check(hi, ldhi, h0, ldh0, W, ldw, out, ldo, M, H, drop_p, grid);
  if (rc != ERCG_OK || grid.x == 0) return rc;
  Epilogue ep{nullptr, ACT_GCNII_FWD, hi, (long long)ldhi, 1.f, drop_p, (unsigned long long)seed,
              h0, (long long)ldh0, theta, (1.f - theta) * (1.f - alpha), (1.f - theta) * alpha, relu ? 1 : 0};
  gemm_nn_kernel<true, true><<<grid, GT, 0, (cudaStream_t)stream>>>(hi, ldhi, nullptr, W, ldw, out, ldo, M, H, 2 * H, ep,
                                                                   h0, ldh0, H);
  return finish_launch();
}

// ercg_gcnii_layer_fwd with the dropout mask drawn from seed + *seed_dev
extern "C" int ercg_gcnii_layer_fwd_dev(const float* hi, int64_t ldhi, const float* h0, int64_t ldh0, const float* W,
                                        int64_t ldw, float* out, int64_t ldo, int64_t M, int H, float theta, float alpha,
                                        int relu, float drop_p, uint64_t seed, const uint64_t* seed_dev, void* stream) {
  if (!seed_dev) return ERCG_EINVAL;
  dim3 grid;
  const int rc = gcnii_fwd_check(hi, ldhi, h0, ldh0, W, ldw, out, ldo, M, H, drop_p, grid);
  if (rc != ERCG_OK || grid.x == 0) return rc;
  Epilogue ep{nullptr, ACT_GCNII_FWD, hi, (long long)ldhi, 1.f, drop_p, (unsigned long long)seed,
              h0, (long long)ldh0, theta, (1.f - theta) * (1.f - alpha), (1.f - theta) * alpha, relu ? 1 : 0};
  ep.seed_dev = reinterpret_cast<const unsigned long long*>(seed_dev);
  gcnii_fwd_dev_kernel<true, true><<<grid, GT, 0, (cudaStream_t)stream>>>(hi, ldhi, nullptr, W, ldw, out, ldo, M, H, 2 * H,
                                                                         ep, h0, ldh0, H);
  return finish_launch();
}

// dS[M, 2H] = theta * dZ @ Wt + [ (1-theta)(1-alpha) dZ | (1-theta) alpha dZ ],  Wt = W^T [H, 2H]
// (left half = gradient w.r.t. hi, right half = this layer's contribution to the gradient w.r.t. h0)
extern "C" int ercg_gcnii_layer_bwd_input(const float* dZ, int64_t lddz, const float* Wt, int64_t ldwt, float* dS,
                                          int64_t ldds, int64_t M, int H, float theta, float alpha, void* stream) {
  if (M < 0 || H <= 0 || (H & 7)) return ERCG_EINVAL;
  if (M == 0) return ERCG_OK;
  if (!dZ || !Wt || !dS || lddz < H || ldwt < 2 * H || ldds < 2 * H) return ERCG_EINVAL;
  if (!aligned16(dZ) || !aligned16(Wt) || (lddz & 3) || (ldwt & 3)) return ERCG_EALIGN;
  Epilogue ep{nullptr, ACT_GCNII_BWD, dZ, (long long)lddz, 1.f, 0.f, 0ull,
              nullptr, 0, theta, (1.f - theta) * (1.f - alpha), (1.f - theta) * alpha, H};
  long long gm = (M + BM - 1) / BM;
  if (gm > 2147483647LL) return ERCG_ERANGE;
  dim3 grid((unsigned)gm, (unsigned)((2 * H + BN - 1) / BN));
  gemm_nn_kernel<true, true><<<grid, GT, 0, (cudaStream_t)stream>>>(dZ, lddz, nullptr, Wt, ldwt, dS, ldds, M, 2 * H, H, ep);
  return finish_launch();
}
