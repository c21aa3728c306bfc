// K4 / K5 warp-per-node kernels for the rows the float4 NC = 1..3 kernels of attn.cu do not take: any even H <= 1024 and
// rows that are only 8-byte aligned.  Included by attn.cu (inside namespace ercg, after AW and its own kernels).
//
// Same algorithm, edge order and per-chunk arithmetic as the attn.cu kernels, written over the chunk type V: a lane holds
// its part of an H-wide row as NC chunks, chunk c of lane l = elements [CW * (l + 32c), CW * (l + 32c) + CW), CW = 4 / 2.
//   * float4, NC = 4, 6, 8: every row 16-byte aligned with ld % 4 == 0 and 384 < H <= 1024;
//   * float2, NC = 4, 8, 12, 16: H % 4 == 2 or some row only 8-byte aligned (e.g. the key half of dgcnv2's [xt | e] at
//     odd hidden sizes), H <= 1024.
// The attn.cu kernels stay as they were tuned (their SASS is unchanged); these are separate instantiations because the
// compiler does not produce the same code for the float4 NC = 1..3 cases when they go through the generic template.
// All sums keep a fixed order (per lane over chunks, then the butterfly), so results are bit-reproducible and independent
// of the grid.  __launch_bounds__(256, 2): without the block count ptxas held some instantiations at 48-64 registers and
// spilled; with it none spills (-Xptxas -v) and the widest use 120-128 registers, two CTAs per SM.
#pragma once

template <typename V> struct Chunk;
template <> struct Chunk<float4> { static constexpr int SH = 2; };
template <> struct Chunk<float2> { static constexpr int SH = 1; };
template <typename V> __device__ __forceinline__ V ldv(const float* p);
template <> __device__ __forceinline__ float4 ldv<float4>(const float* p) { return ld4(p); }
template <> __device__ __forceinline__ float2 ldv<float2>(const float* p) { return *reinterpret_cast<const float2*>(p); }
template <typename V> __device__ __forceinline__ V zerov();
template <> __device__ __forceinline__ float4 zerov<float4>() { return make_float4(0.f, 0.f, 0.f, 0.f); }
template <> __device__ __forceinline__ float2 zerov<float2>() { return make_float2(0.f, 0.f); }
__device__ __forceinline__ void stv(float* p, float4 v) { st4(p, v); }
__device__ __forceinline__ void stv(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }
__device__ __forceinline__ float dotv(const float4& a, const float4& b) { return dot4(a, b); }
__device__ __forceinline__ float dotv(const float2& a, const float2& b) { return fmaf(a.x, b.x, a.y * b.y); }
__device__ __forceinline__ void fmav(float4& a, float s, const float4& b) { fma4(a, s, b); }
__device__ __forceinline__ void fmav(float2& a, float s, const float2& b) { a.x = fmaf(s, b.x, a.x); a.y = fmaf(s, b.y, a.y); }
__device__ __forceinline__ void scalev(float4& a, float s) { a.x *= s; a.y *= s; a.z *= s; a.w *= s; }
__device__ __forceinline__ void scalev(float2& a, float s) { a.x *= s; a.y *= s; }
__device__ __forceinline__ void addv(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
__device__ __forceinline__ void addv(float2& a, const float2& b) { a.x += b.x; a.y += b.y; }

template <typename V, int NC>
__device__ __forceinline__ void wload_row(const float* p, int nch, int lane, V r[NC]) {
  constexpr int CW = 1 << Chunk<V>::SH;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    r[c] = ch < nch ? ldv<V>(p + CW * ch) : zerov<V>();
  }
}
template <typename V, int NC>
__device__ __forceinline__ float wrow_dot(const V a[NC], const float* p, int nch, int lane) {
  constexpr int CW = 1 << Chunk<V>::SH;
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) s += dotv(a[c], ldv<V>(p + CW * ch));
  }
  return warp_sum(s);
}

// <a, row_q> for 4 rows at once: the 4 row loads are issued back to back, the 4 reductions interleave.
// Rows with live[q] == false are not read (warp-uniform) and yield 0.
template <typename V, int NC>
__device__ __forceinline__ void wrow_dot4(const V a[NC], const float* const p[4], const bool live[4], int nch, int lane,
                                         float out[4]) {
  constexpr int CW = 1 << Chunk<V>::SH;
  float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) {
      V v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = live[q] ? ldv<V>(p[q] + CW * ch) : zerov<V>();
#pragma unroll
      for (int q = 0; q < 4; ++q) s[q] += dotv(a[c], v[q]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int q = 0; q < 4; ++q) s[q] += __shfl_xor_sync(0xffffffffu, s[q], o);
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) out[q] = s[q];
}
// acc += sum_q w[q] * row_q (4 rows in flight)
template <typename V, int NC>
__device__ __forceinline__ void wrow_axpy4(V acc[NC], const float w[4], const float* const p[4], const bool live[4],
                                          int nch, int lane) {
  constexpr int CW = 1 << Chunk<V>::SH;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) {
      V v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = live[q] ? ldv<V>(p[q] + CW * ch) : zerov<V>();
#pragma unroll
      for (int q = 0; q < 4; ++q) fmav(acc[c], w[q], v[q]);
    }
  }
}

template <typename V, int NC>
__global__ void __launch_bounds__(AW * 32, 2)
attn_fwd_wide_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                     const float* __restrict__ s, long long ld, const int* __restrict__ rowptr,
                     const int* __restrict__ col, float scale, float* __restrict__ out, long long ldo,
                     float* __restrict__ alpha, float* __restrict__ dact, long long N, int H) {
  constexpr int CW = 1 << Chunk<V>::SH;
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  V qi[NC], acc[NC];
  wload_row<V, NC>(q + node * ld, nch, lane, qi);
#pragma unroll
  for (int c = 0; c < NC; ++c) acc[c] = zerov<V>();
  const int beg = rowptr[node], end = rowptr[node + 1];
  float run_max = -INFINITY, run_sum = 0.f;
  for (int cb = beg; cb < end; cb += 32) {
    const int cn = min(32, end - cb);
    float my = -INFINITY;                       // score of edge cb + lane
    const int mc = lane < cn ? col[cb + lane] : 0;      // sources of this batch, one coalesced load
    for (int u = 0; u < cn; u += 4) {
      const float* p[4];
      bool live[4];
      float d[4];
#pragma unroll
      for (int qq = 0; qq < 4; ++qq) {
        live[qq] = u + qq < cn;
        p[qq] = k + (long long)__shfl_sync(0xffffffffu, mc, min(u + qq, cn - 1)) * ld;
      }
      wrow_dot4<V, NC>(qi, p, live, nch, lane, d);
#pragma unroll
      for (int qq = 0; qq < 4; ++qq)
        if (lane == u + qq) my = d[qq] * scale;
    }
    if (dact && lane < cn) {                    // MatchingAttention 'general2' (dgcnv2_models.py:128-133): softmax of tanh(score)
      my = tanhf(my);
      dact[cb + lane] = 1.f - my * my;          // d tanh / d score, applied to dsig by the by-destination backward
    }
    const float cmax = warp_max(my);
    const float new_max = fmaxf(run_max, cmax);
    const float resc = run_max == -INFINITY ? 0.f : expf(run_max - new_max);   // first chunk: nothing to rescale
    const float ex = lane < cn ? expf(my - new_max) : 0.f;
    run_sum = run_sum * resc + warp_sum(ex);
#pragma unroll
    for (int c = 0; c < NC; ++c) scalev(acc[c], resc);
    if (alpha && lane < cn) alpha[cb + lane] = ex;        // un-normalised, relative to new_max; fixed below
    if (alpha && cb > beg && resc != 1.f) {               // rescale earlier chunks (rare: deg > 32)
      for (int e2 = beg + lane; e2 < cb; e2 += 32) alpha[e2] *= resc;
    }
    for (int u = 0; u < cn; u += 4) {
      const float* p[4];
      bool live[4];
      float a[4];
#pragma unroll
      for (int qq = 0; qq < 4; ++qq) {
        const int l = min(u + qq, cn - 1);
        live[qq] = u + qq < cn;
        a[qq] = __shfl_sync(0xffffffffu, ex, l);
        p[qq] = v + (long long)__shfl_sync(0xffffffffu, mc, l) * ld;
      }
      wrow_axpy4<V, NC>(acc, a, p, live, nch, lane);
    }
    run_max = new_max;
  }
  const float inv = 1.f / (run_sum + 1e-16f);
  if (alpha) {
    __syncwarp();
    for (int e2 = beg + lane; e2 < end; e2 += 32) alpha[e2] *= inv;
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) {
      V r = acc[c];
      scalev(r, inv);
      if (s) addv(r, ldv<V>(s + node * ld + CW * ch));
      stv(out + node * ldo + CW * ch, r);
    }
  }
}

// by-destination backward: dalpha_e = <dout_i, v_j>, D = sum alpha dalpha, dsig_e = alpha_e (dalpha_e - D),
// dq_i = scale * sum dsig_e k_j, ds_i = dout_i
template <typename V, int NC>
__global__ void __launch_bounds__(AW * 32, 2)
attn_bwd_dst_wide_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ k,
                         const float* __restrict__ v, long long ld, const int* __restrict__ rowptr,
                         const int* __restrict__ col, const float* __restrict__ alpha, float scale,
                         float* __restrict__ dq, float* __restrict__ ds, long long ldd, float* __restrict__ dsig,
                         const float* __restrict__ dact, long long N, int H) {
  constexpr int CW = 1 << Chunk<V>::SH;
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  V go[NC], acc[NC];
  wload_row<V, NC>(dout + node * ldo, nch, lane, go);
  const int beg = rowptr[node], end = rowptr[node + 1];
  if (end - beg <= 32) {
    // common case: every per-edge scalar of the row lives in one lane; no round trip through the dsig buffer
    const int cn = end - beg;
    const int mc = lane < cn ? col[beg + lane] : 0;
    const float al = lane < cn ? alpha[beg + lane] : 0.f;
    float my = 0.f;
    for (int u = 0; u < cn; u += 4) {
      const float* p[4];
      bool live[4];
      float d[4];
#pragma unroll
      for (int qq = 0; qq < 4; ++qq) {
        live[qq] = u + qq < cn;
        p[qq] = v + (long long)__shfl_sync(0xffffffffu, mc, min(u + qq, cn - 1)) * ld;
      }
      wrow_dot4<V, NC>(go, p, live, nch, lane, d);
#pragma unroll
      for (int qq = 0; qq < 4; ++qq)
        if (lane == u + qq) my = d[qq];
    }
    const float D = warp_sum(al * my);
    float g = al * (my - D);
    if (dact && lane < cn) g *= dact[beg + lane];
    if (lane < cn) dsig[beg + lane] = g;
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c] = zerov<V>();
    for (int u = 0; u < cn; u += 4) {
      const float* p[4];
      bool live[4];
      float gw[4];
#pragma unroll
      for (int qq = 0; qq < 4; ++qq) {
        const int l = min(u + qq, cn - 1);
        live[qq] = u + qq < cn;
        gw[qq] = __shfl_sync(0xffffffffu, g, l) * scale;
        p[qq] = k + (long long)__shfl_sync(0xffffffffu, mc, l) * ld;
      }
      wrow_axpy4<V, NC>(acc, gw, p, live, nch, lane);
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) {
        stv(dq + node * ldd + CW * ch, acc[c]);
        if (ds) stv(ds + node * ldd + CW * ch, go[c]);
      }
    }
    return;
  }
  // pass 1: dalpha per edge -> dsig buffer (temporarily), D
  float D = 0.f;
  for (int cb = beg; cb < end; cb += 32) {
    const int cn = min(32, end - cb);
    float my = 0.f;
    for (int u = 0; u < cn; ++u) {
      const float d = wrow_dot<V, NC>(go, v + (long long)col[cb + u] * ld, nch, lane);
      if (lane == u) my = d;
    }
    const float a = lane < cn ? alpha[cb + lane] : 0.f;
    D += warp_sum(a * my);
    if (lane < cn) dsig[cb + lane] = my;
  }
  __syncwarp();
#pragma unroll
  for (int c = 0; c < NC; ++c) acc[c] = zerov<V>();
  for (int cb = beg; cb < end; cb += 32) {
    const int cn = min(32, end - cb);
    float g = 0.f;
    if (lane < cn) {
      g = alpha[cb + lane] * (dsig[cb + lane] - D);
      if (dact) g *= dact[cb + lane];
      dsig[cb + lane] = g;
    }
    for (int u = 0; u < cn; ++u) {
      const float gu = __shfl_sync(0xffffffffu, g, u) * scale;
      const float* pk = k + (long long)col[cb + u] * ld;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const int ch = lane + 32 * c;
        if (ch < nch) fmav(acc[c], gu, ldv<V>(pk + CW * ch));
      }
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) {
      stv(dq + node * ldd + CW * ch, acc[c]);
      if (ds) stv(ds + node * ldd + CW * ch, go[c]);
    }
  }
}

// by-source backward: dk_j = scale * sum_i dsig[j->i] q_i,  dv_j = sum_i alpha[j->i] dout_i
template <typename V, int NC>
__global__ void __launch_bounds__(AW * 32, 2)
attn_bwd_src_wide_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ q, long long ld,
                         const int* __restrict__ t_rowptr, const int* __restrict__ t_col, const int* __restrict__ t_eid,
                         const float* __restrict__ alpha, const float* __restrict__ dsig, float scale,
                         float* __restrict__ dk, float* __restrict__ dv, long long ldd, long long N, int H) {
  constexpr int CW = 1 << Chunk<V>::SH;
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  V ak[NC], av[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) { ak[c] = zerov<V>(); av[c] = ak[c]; }
  const int beg = t_rowptr[node], end = t_rowptr[node + 1];
  for (int e = beg; e < end; ++e) {
    const int i = t_col[e], id = t_eid[e];
    const float a = alpha[id], g = dsig[id] * scale;
    const float* pq = q + (long long)i * ld;
    const float* pd = dout + (long long)i * ldo;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) {
        fmav(ak[c], g, ldv<V>(pq + CW * ch));
        fmav(av[c], a, ldv<V>(pd + CW * ch));
      }
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) {
      stv(dk + node * ldd + CW * ch, ak[c]);
      stv(dv + node * ldd + CW * ch, av[c]);
    }
  }
}

// ---- K5 EdgeAtt
// by-source softmax of <x_j, u_k> over k in out(j); result stored at the by-destination edge id.
template <typename V, int NC>
__global__ void __launch_bounds__(AW * 32, 2)
edgeatt_fwd_wide_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ u, long long ldu,
                        const int* __restrict__ t_rowptr, const int* __restrict__ t_col, const int* __restrict__ t_eid,
                        float* __restrict__ nu, long long N, int H) {
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  V xj[NC];
  wload_row<V, NC>(x + node * ldx, nch, lane, xj);
  const int beg = t_rowptr[node], end = t_rowptr[node + 1];
  // pass 1: raw scores -> nu[t_eid], running max
  float mx = -INFINITY;
  for (int cb = beg; cb < end; cb += 32) {
    const int cn = min(32, end - cb);
    float my = -INFINITY;
    for (int uu = 0; uu < cn; ++uu) {
      const float d = wrow_dot<V, NC>(xj, u + (long long)t_col[cb + uu] * ldu, nch, lane);
      if (lane == uu) my = d;
    }
    if (lane < cn) nu[t_eid[cb + lane]] = my;
    mx = fmaxf(mx, warp_max(my));
  }
  __syncwarp();
  float sum = 0.f;
  for (int e = beg + lane; e < end; e += 32) {
    const int id = t_eid[e];
    const float ex = expf(nu[id] - mx);
    nu[id] = ex;
    sum += ex;
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  for (int e = beg + lane; e < end; e += 32) nu[t_eid[e]] *= inv;
}

// by-source backward: dsig[e] = nu_e (dnu_e - sum nu dnu),  dx_j = sum_k dsig u_k   (dx is WRITTEN, not accumulated)
template <typename V, int NC>
__global__ void __launch_bounds__(AW * 32, 2)
edgeatt_bwd_src_wide_kernel(const float* __restrict__ dnu, const float* __restrict__ nu, const float* __restrict__ u,
                            long long ldu, const int* __restrict__ t_rowptr, const int* __restrict__ t_col,
                            const int* __restrict__ t_eid, float* __restrict__ dsig, float* __restrict__ dx, long long lddx,
                            long long N, int H) {
  constexpr int CW = 1 << Chunk<V>::SH;
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  const int beg = t_rowptr[node], end = t_rowptr[node + 1];
  float D = 0.f;
  for (int e = beg + lane; e < end; e += 32) {
    const int id = t_eid[e];
    D += nu[id] * dnu[id];
  }
  D = warp_sum(D);
  V acc[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) acc[c] = zerov<V>();
  for (int e = beg; e < end; ++e) {
    const int id = t_eid[e];
    const float g = nu[id] * (dnu[id] - D);
    if (lane == 0) dsig[id] = g;
    const float* pu = u + (long long)t_col[e] * ldu;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) fmav(acc[c], g, ldv<V>(pu + CW * ch));
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) stv(dx + node * lddx + CW * ch, acc[c]);
  }
}

// by-destination backward: du_k = sum_{j in in(k)} dsig[j->k] x_j
template <typename V, int NC>
__global__ void __launch_bounds__(AW * 32, 2)
edgeatt_bwd_dst_wide_kernel(const float* __restrict__ dsig, const float* __restrict__ x, long long ldx,
                            const int* __restrict__ rowptr, const int* __restrict__ col, float* __restrict__ du,
                            long long lddu, long long N, int H) {
  constexpr int CW = 1 << Chunk<V>::SH;
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  V acc[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) acc[c] = zerov<V>();
  const int beg = rowptr[node], end = rowptr[node + 1];
  for (int e = beg; e < end; ++e) {
    const float g = dsig[e];
    const float* px = x + (long long)col[e] * ldx;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) fmav(acc[c], g, ldv<V>(px + CW * ch));
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) stv(du + node * lddu + CW * ch, acc[c]);
  }
}
