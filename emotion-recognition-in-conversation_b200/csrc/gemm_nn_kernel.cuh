// The SIMT NN GEMM kernel (gemm_simt.cu), written once and compiled under two names:
//   gemm_nn_kernel        ERCG_NN_GCNII_SEED = ep.seed                      (every host-seeded entry)
//   gcnii_fwd_dev_kernel  ERCG_NN_GCNII_SEED = ep.seed + *ep.seed_dev       (ercg_gcnii_layer_fwd_dev)
// The GCNII forward epilogue's dropout seed is the only difference.  Including the same text twice keeps the two from
// drifting apart and leaves gemm_nn_kernel's machine code as it was (a shared inline function does not: nvcc then
// allocates the existing kernel's registers differently).
// Include with ERCG_NN_KERNEL and ERCG_NN_GCNII_SEED defined; both are undefined at the end.
template <bool VEC_A, bool VEC_B>
__global__ void __launch_bounds__(GT, 2)
ERCG_NN_KERNEL(const float* __restrict__ A, long long lda, const int* __restrict__ a_rows,
               const float* __restrict__ B, long long ldb, float* __restrict__ C, long long ldc,
               long long M, int N, int K, Epilogue ep,
               const float* __restrict__ A2 = nullptr, long long lda2 = 0, int ksplit = 0x7fffffff) {
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Bs[2][BK][BN + 4];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const long long m0 = (long long)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;

  const int arow_l = t & 127, ak = (t >> 7) * 8;
  const long long am = m0 + arow_l;
  const bool a_ok = am < M;
  const float* arow = A;
  if (a_ok) arow = A + (a_rows ? (long long)a_rows[am] : am) * lda;
  // optional second source for the columns k >= ksplit of the A operand ([A | A2] without materialising the concat;
  // ksplit % 8 == 0 so every 8-wide thread chunk lies on one side)
  const float* arow2 = a_ok && A2 ? A2 + am * lda2 - ksplit : arow;
  const int bk = t >> 5, bn = (t & 31) * 4;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  float ra[8], rb0[4], rb1[4];
  load_a_nn<VEC_A>(ak >= ksplit ? arow2 : arow, a_ok, ak, K, ra);
  load_b_nn<VEC_B>(B, ldb, bk, K, n0 + bn, N, rb0);
  load_b_nn<VEC_B>(B, ldb, bk + 8, K, n0 + bn, N, rb1);
  const int nslab = (K + BK - 1) / BK;
  int buf = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) As[0][ak + i][arow_l] = ra[i];
  *reinterpret_cast<float4*>(&Bs[0][bk][bn]) = make_float4(rb0[0], rb0[1], rb0[2], rb0[3]);
  *reinterpret_cast<float4*>(&Bs[0][bk + 8][bn]) = make_float4(rb1[0], rb1[1], rb1[2], rb1[3]);
  __syncthreads();
  for (int s = 0; s < nslab; ++s) {
    const int kn = (s + 1) * BK;
    if (s + 1 < nslab) {
      load_a_nn<VEC_A>(kn + ak >= ksplit ? arow2 : arow, a_ok, kn + ak, K, ra);
      load_b_nn<VEC_B>(B, ldb, kn + bk, K, n0 + bn, N, rb0);
      load_b_nn<VEC_B>(B, ldb, kn + bk + 8, K, n0 + bn, N, rb1);
    }
    mma_slab(As[buf], Bs[buf], acc, ty, tx);
    if (s + 1 < nslab) {
      const int nb = buf ^ 1;
#pragma unroll
      for (int i = 0; i < 8; ++i) As[nb][ak + i][arow_l] = ra[i];
      *reinterpret_cast<float4*>(&Bs[nb][bk][bn]) = make_float4(rb0[0], rb0[1], rb0[2], rb0[3]);
      *reinterpret_cast<float4*>(&Bs[nb][bk + 8][bn]) = make_float4(rb1[0], rb1[1], rb1[2], rb1[3]);
      __syncthreads();
      buf = nb;
    }
  }

  // epilogue
  const bool vec_c = ((ldc & 3) == 0) && aligned16(C);
#pragma unroll
  for (int ih = 0; ih < 2; ++ih)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long m = m0 + ih * 64 + ty * 4 + i;
      if (m >= M) continue;
#pragma unroll
      for (int jh = 0; jh < 2; ++jh) {
        const int n = n0 + jh * 64 + tx * 4;
        if (n >= N) continue;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float x = acc[ih * 4 + i][jh * 4 + j];
          const int nn = n + j;
          if (nn < N) {
            if (ep.bias) x += __ldg(ep.bias + nn);
            if (ep.act == ERCG_ACT_RELU) {
              x = fmaxf(x, 0.f);
            } else if (ep.act == ERCG_ACT_RELU_DROPOUT) {
              x = fmaxf(x, 0.f);
              const bool drop = dropout_drop(dropout_group_hash(ep.seed + (ep.seed_dev ? __ldg(ep.seed_dev) : 0ull), m, nn, N), nn & 3, dropout_thr16(ep.drop_p));
              x = drop ? 0.f : x * (1.0f / (1.0f - ep.drop_p));
            } else if (ep.act == ERCG_ACT_MASK_POS) {
              x = __ldg(ep.aux + m * ep.ldaux + nn) > 0.f ? x * ep.aux_scale : 0.f;
            } else if (ep.act == ACT_GCNII_FWD) {
              x = ep.c_acc * x + (ep.c1 * __ldg(ep.aux + m * ep.ldaux + nn) + ep.c2 * __ldg(ep.aux2 + m * ep.ldaux2 + nn));
              if (ep.half) x = fmaxf(x, 0.f);
              if (ep.drop_p > 0.f) {
                const float u = hash_uniform(ERCG_NN_GCNII_SEED, (unsigned long long)m * (unsigned long long)N + nn);
                x = u < ep.drop_p ? 0.f : x * (1.0f / (1.0f - ep.drop_p));
              }
            } else if (ep.act == ACT_GCNII_BWD) {
              x = ep.c_acc * x + (nn < ep.half ? ep.c1 * __ldg(ep.aux + m * ep.ldaux + nn)
                                               : ep.c2 * __ldg(ep.aux + m * ep.ldaux + nn - ep.half));
            }
          }
          v[j] = x;
        }
        float* cp = C + m * ldc + n;
        if (vec_c && n + 4 <= N) {
          st4(cp, make_float4(v[0], v[1], v[2], v[3]));
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n + j < N) cp[j] = v[j];
        }
      }
    }
}

#undef ERCG_NN_KERNEL
#undef ERCG_NN_GCNII_SEED
