// K4 / K5: fused edge attention over the packed CSR.
//
// K4 = PyG TransformerConv(heads=1) message/aggregate (track_mm/cogmen.py:66,72):
//   sigma[j->i] = <q_i, k_j> * scale,  alpha = softmax over the in-edges of i (max-subtracted,
//   denominator + 1e-16),  out_i = sum_j alpha[j->i] v_j + s_i.
// K5 = EdgeAtt of DialogueGCN (track_mm/dgcn_models.py:121-152): the same score/softmax machinery
//   normalised over the OUT-edges of each source (by-source traversal), no value aggregation.
//
// Warp-per-node kernels (any graph, any even H <= 1024, 8-byte aligned rows): one warp per node, lane l holds its part of
// an H-wide row as NC chunks of type V, chunk c = elements [CW * (l + 32c), CW * (l + 32c) + CW).  V = float4 (CW = 4) when
// H % 4 == 0 and every row is 16-byte aligned with ld % 4 == 0, float2 (CW = 2) otherwise (e.g. the key half of dgcnv2's
// [xt | e] at odd hidden sizes); ERCG_LAUNCH_NC picks V and NC from H and the operands.  Scores of up to 32 edges are
// kept one-per-lane in a register (deg <= 11 / 21 for the reference's windows); longer rows fall back to an online
// (running max / rescale) chunked loop.  Score, softmax and aggregation are one kernel: k_j and v_j rows are read once per
// edge from L1/L2, q_i/s_i/out_i once per node from HBM.  All sums keep a fixed order (per lane over chunks, then the
// butterfly), so results are bit-reproducible and independent of the grid.
// Algorithmic HBM bytes per node (SURVEY.md 8d): 5*4H (q,k,v,s,out) + 4 (rowptr) + 8*deg (col, alpha).
// The ercg_attn_window_* entry points run CTA tile kernels instead: attn_blk.cuh's for windows of up to 16 candidates, the
// round-1 tile kernels below for wider ones.
#include "common.cuh"
#include "attn_blk.cuh"
#include <math.h>
#include <stdlib.h>
#include <type_traits>

namespace ercg {

constexpr int AW = 8;
// Minimum resident CTAs per SM the warp-per-node kernels are compiled for: the float4 NC <= 3 instantiations were tuned
// without a block count (0), the wider ones spill without one (ptxas held some at 48-64 registers; with 2, none spills).
template <typename V, int NC>
constexpr int node_min_blocks = std::is_same<V, float4>::value && NC <= 3 ? 0 : 2;

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
__device__ __forceinline__ void load_row(const float* p, int nch, int lane, V r[NC]) {
  constexpr int CW = 1 << Chunk<V>::SH;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    r[c] = ch < nch ? ldv<V>(p + CW * ch) : zerov<V>();
  }
}
template <typename V, int NC>
__device__ __forceinline__ float row_dot(const V a[NC], const float* p, int nch, int lane) {
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
__device__ __forceinline__ void row_dot4(const V a[NC], const float* const p[4], const bool live[4], int nch, int lane,
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
__device__ __forceinline__ void row_axpy4(V acc[NC], const float w[4], const float* const p[4], const bool live[4],
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
__global__ void __launch_bounds__(AW * 32, node_min_blocks<V, NC>)
attn_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                const float* __restrict__ s, long long ld, const int* __restrict__ rowptr,
                const int* __restrict__ col, float scale, float* __restrict__ out, long long ldo,
                float* __restrict__ alpha, float* __restrict__ dact, long long N, int H) {
  constexpr int CW = 1 << Chunk<V>::SH;
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  V qi[NC], acc[NC];
  load_row<V, NC>(q + node * ld, nch, lane, qi);
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
      row_dot4<V, NC>(qi, p, live, nch, lane, d);
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
      row_axpy4<V, NC>(acc, a, p, live, nch, lane);
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
__global__ void __launch_bounds__(AW * 32, node_min_blocks<V, NC>)
attn_bwd_dst_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ k,
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
  load_row<V, NC>(dout + node * ldo, nch, lane, go);
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
      row_dot4<V, NC>(go, p, live, nch, lane, d);
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
      row_axpy4<V, NC>(acc, gw, p, live, nch, lane);
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
      const float d = row_dot<V, NC>(go, v + (long long)col[cb + u] * ld, nch, lane);
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
__global__ void __launch_bounds__(AW * 32, node_min_blocks<V, NC>)
attn_bwd_src_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ q, long long ld,
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

// ---------------------------------------------------------------------------------- K4 on WINDOW graphs: CTA tiles
// ncu on the warp-per-node kernels above (profiles/r01b_ncu_full_262k.csv): attn_fwd executes ~790 warp instructions
// per node at 63 % issue utilisation and 55 % occupancy -- issue- and latency-bound, DRAM at 20-30 %.  For the graphs
// K1 builds, the neighbours of node i are the contiguous rows [i - wlo, i + whi] of its dialogue, so a CTA that owns 32
// consecutive nodes needs only the 32 + wlo + whi rows around them.  These kernels stage those rows of k / v (and q or
// dout) in shared memory with coalesced cp.async copies (blk_stage_rows; all global latency is paid once, in parallel), then
//   * scores / dalpha: ONE LANE PER EDGE walks the 25 float4 chunks of "its" neighbour row in shared memory -- no
//     shuffle reduction at all; two nodes share a warp (16 lanes each) when wlo + whi + 1 <= 16,
//   * aggregation: one lane per float4 chunk, per-edge scalars broadcast by shuffle.
// ~210 instead of ~790 instructions per node.  Same arithmetic per edge; the summation order over edges is unchanged
// (ascending CSR order), so results stay bit-reproducible.  A source outside the promised window traps.
#ifndef ATTN_WT_
#define ATTN_WT_ 32
#endif
constexpr int WT = ATTN_WT_;  // nodes per CTA tile

// per-CTA column sums of two H-wide outputs: lane = float4 chunk, warps reduced in warp order through the staging buffer
// (8 KB of it, reused once every warp is done with the staged rows -- no extra shared memory, so occupancy is unchanged)
__device__ __forceinline__ void tile_colsum(float4* red /* [8][2][32] */, float4 a, float4 b, float* __restrict__ partial, int H) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nch = H >> 2;
  __syncthreads();
  red[(warp * 2 + 0) * 32 + lane] = a;
  red[(warp * 2 + 1) * 32 + lane] = b;
  __syncthreads();
  if (warp < 2 && lane < nch) {
    float4 t = red[warp * 32 + lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) {
      const float4 v = red[(w * 2 + warp) * 32 + lane];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    st4(partial + (long long)blockIdx.x * 2 * H + warp * H + 4 * lane, t);
  }
}

template <bool PAIR>
__global__ void __launch_bounds__(256)
attn_fwd_tile_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                     const float* __restrict__ s, long long ld, const int* __restrict__ rowptr,
                     const int* __restrict__ col, float scale, float* __restrict__ out, long long ldo,
                     float* __restrict__ alpha, long long N, int H, int wlo, int whi) {
  extern __shared__ float4 attn_sm[];
  const int nch = H >> 2, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long t0 = (long long)blockIdx.x * WT;
  const int tn = (int)min((long long)WT, N - t0);
  const long long r0 = max(0LL, t0 - wlo), r1 = min(N, t0 + tn + whi);
  const int R = (int)(r1 - r0), Rmax = WT + wlo + whi;
  float4* sq = attn_sm;
  float4* sk = sq + WT * nch;
  float4* sv = sk + Rmax * nch;
  blk_stage_rows<256>(sq, q, ld, t0, tn, nch);
  blk_stage_rows<256>(sk, k, ld, r0, R, nch);
  blk_stage_rows<256>(sv, v, ld, r0, R, nch);
  constexpr int NPW = WT / 8;                 // nodes per warp
  constexpr int G = PAIR ? 2 : 1;             // nodes handled together in the score phase
  constexpr int IT = NPW / G;
  const int half = PAIR ? lane >> 4 : 0, e = PAIR ? lane & 15 : lane;
  // Everything this warp needs from global memory besides the staged rows is requested NOW, while the cp.async traffic is
  // in flight: CSR metadata of its nodes and their skip rows.  (ncu, first tiled version: a third of the stall samples
  // were these small dependent loads issued one node at a time after the barrier.)
  int begs[IT], degs[IT], rows[IT];
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int nl = warp * NPW + it * G + half;
    const bool nok = nl < tn;
    begs[it] = nok ? rowptr[t0 + nl] : 0;
    degs[it] = nok ? rowptr[t0 + nl + 1] - begs[it] : 0;
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    rows[it] = 0;
    if (e < degs[it]) {
      const long long src = col[begs[it] + e];
      if (src < r0 || src >= r1) __trap();    // the caller promised a window graph
      rows[it] = (int)(src - r0);
    }
  }
  float4 skip[NPW];
#pragma unroll
  for (int h = 0; h < NPW; ++h) {
    const int nl = warp * NPW + h;
    skip[h] = (s && nl < tn && lane < nch) ? ld4(s + (t0 + nl) * ld + 4 * lane) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  cp_wait_all();
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int p = it * G;
    const int nl = warp * NPW + p + half;     // node of this lane's half
    const int beg = begs[it], deg = degs[it], row = rows[it];
    const bool live = e < deg;
    float d = 0.f;
    const float4* qi = sq + nl * nch;
    const float4* kr = sk + row * nch;
    if (live) {
#pragma unroll 5
      for (int c = 0; c < nch; ++c) d += dot4(qi[c], kr[c]);
    }
    d *= scale;
    const float x = live ? d : -INFINITY;
    const float mx = PAIR ? h16_max(x) : warp_max(x);
    const float ex = live ? expf(d - mx) : 0.f;
    const float inv = 1.f / ((PAIR ? h16_sum(ex) : warp_sum(ex)) + 1e-16f);
    const float al = ex * inv;
    if (live && alpha) alpha[beg + e] = al;
    // aggregation: lanes = float4 chunks, one node after the other
#pragma unroll
    for (int h = 0; h < G; ++h) {
      const int base = PAIR ? h * 16 : 0;
      const int hdeg = __shfl_sync(0xffffffffu, deg, base);
      const int hnl = warp * NPW + p + h;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);                 // out = (sum_j alpha v_j) + skip, in that order
      for (int u = 0; u < hdeg; ++u) {
        const float a = __shfl_sync(0xffffffffu, al, base + u);
        const int rw = __shfl_sync(0xffffffffu, row, base + u);
        if (lane < nch) fma4(acc, a, sv[rw * nch + lane]);
      }
      if (hnl < tn && lane < nch) {
        const float4 sk4 = skip[p + h];
        acc.x += sk4.x; acc.y += sk4.y; acc.z += sk4.z; acc.w += sk4.w;
        st4(out + (t0 + hnl) * ldo + 4 * lane, acc);
      }
    }
  }
}

template <bool PAIR>
__global__ void __launch_bounds__(256)
attn_bwd_dst_tile_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ k,
                         const float* __restrict__ v, long long ld, const int* __restrict__ rowptr,
                         const int* __restrict__ col, const float* __restrict__ alpha, float scale,
                         float* __restrict__ dq, float* __restrict__ ds, long long ldd, float* __restrict__ dsig,
                         float* __restrict__ colsum_partial /* [gridDim.x][2H]: column sums of dq | ds, or NULL */,
                         long long N, int H, int wlo, int whi) {
  extern __shared__ float4 attn_sm[];
  float4 cs_q = make_float4(0.f, 0.f, 0.f, 0.f), cs_s = cs_q;
  const int nch = H >> 2, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long t0 = (long long)blockIdx.x * WT;
  const int tn = (int)min((long long)WT, N - t0);
  const long long r0 = max(0LL, t0 - wlo), r1 = min(N, t0 + tn + whi);
  const int R = (int)(r1 - r0), Rmax = WT + wlo + whi;
  float4* sd = attn_sm;
  float4* sk = sd + WT * nch;
  float4* sv = sk + Rmax * nch;
  blk_stage_rows<256>(sd, dout, ldo, t0, tn, nch);
  blk_stage_rows<256>(sk, k, ld, r0, R, nch);
  blk_stage_rows<256>(sv, v, ld, r0, R, nch);
  constexpr int NPW = WT / 8;
  constexpr int G = PAIR ? 2 : 1;
  constexpr int IT = NPW / G;
  const int half = PAIR ? lane >> 4 : 0, e = PAIR ? lane & 15 : lane;
  int begs[IT], degs[IT], rows[IT];            // CSR metadata and alpha of this warp's nodes, requested before the wait
  float als[IT];
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int nl = warp * NPW + it * G + half;
    const bool nok = nl < tn;
    begs[it] = nok ? rowptr[t0 + nl] : 0;
    degs[it] = nok ? rowptr[t0 + nl + 1] - begs[it] : 0;
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    rows[it] = 0;
    als[it] = 0.f;
    if (e < degs[it]) {
      const long long src = col[begs[it] + e];
      if (src < r0 || src >= r1) __trap();
      rows[it] = (int)(src - r0);
      als[it] = alpha[begs[it] + e];
    }
  }
  cp_wait_all();
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int p = it * G;
    const int nl = warp * NPW + p + half;
    const int beg = begs[it], deg = degs[it], row = rows[it];
    const bool live = e < deg;
    const float al = als[it];
    float da = 0.f;
    const float4* gi = sd + nl * nch;
    const float4* vr = sv + row * nch;
    if (live) {
#pragma unroll 5
      for (int c = 0; c < nch; ++c) da += dot4(gi[c], vr[c]);
    }
    const float ad = al * da;
    const float D = PAIR ? h16_sum(ad) : warp_sum(ad);
    const float g = al * (da - D);
    if (live) dsig[beg + e] = g;
    const float gs = g * scale;
#pragma unroll
    for (int h = 0; h < G; ++h) {
      const int base = PAIR ? h * 16 : 0;
      const int hdeg = __shfl_sync(0xffffffffu, deg, base);
      const int hnl = warp * NPW + p + h;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int u = 0; u < hdeg; ++u) {
        const float a = __shfl_sync(0xffffffffu, gs, base + u);
        const int rw = __shfl_sync(0xffffffffu, row, base + u);
        if (lane < nch) fma4(acc, a, sk[rw * nch + lane]);
      }
      if (hnl < tn && lane < nch) {
        st4(dq + (t0 + hnl) * ldd + 4 * lane, acc);
        const float4 dsv = sd[hnl * nch + lane];
        if (ds) st4(ds + (t0 + hnl) * ldd + 4 * lane, dsv);
        cs_q.x += acc.x; cs_q.y += acc.y; cs_q.z += acc.z; cs_q.w += acc.w;
        cs_s.x += dsv.x; cs_s.y += dsv.y; cs_s.z += dsv.z; cs_s.w += dsv.w;
      }
    }
  }
  // bias gradient of the q/k/v/skip Linears = column sums of these outputs: reduced per CTA here (fixed order: nodes of a
  // warp ascending, then warps ascending) so that no kernel has to re-read the [N, 4H] gradient
  if (colsum_partial) tile_colsum(attn_sm, cs_q, cs_s, colsum_partial, H);
}

// by-source half on window graphs: the destinations of node j are rows [j - wlo, j + whi]
__global__ void __launch_bounds__(256, 5)      // <= 48 registers: 5 CTAs per SM (the 33.6 KB of staged rows allow 6)
attn_bwd_src_tile_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ q, long long ld,
                         const int* __restrict__ t_rowptr, const int* __restrict__ t_col, const int* __restrict__ t_eid,
                         const float* __restrict__ alpha, const float* __restrict__ dsig, float scale,
                         float* __restrict__ dk, float* __restrict__ dv, long long ldd,
                         float* __restrict__ colsum_partial /* [gridDim.x][2H]: column sums of dk | dv, or NULL */,
                         long long N, int H, int wlo, int whi) {
  extern __shared__ float4 attn_sm[];
  float4 cs_k = make_float4(0.f, 0.f, 0.f, 0.f), cs_v = cs_k;
  const int nch = H >> 2, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long t0 = (long long)blockIdx.x * WT;
  const int tn = (int)min((long long)WT, N - t0);
  const long long r0 = max(0LL, t0 - wlo), r1 = min(N, t0 + tn + whi);
  const int R = (int)(r1 - r0), Rmax = WT + wlo + whi;
  float4* sq = attn_sm;
  float4* sd = sq + Rmax * nch;
  blk_stage_rows<256>(sq, q, ld, r0, R, nch);
  blk_stage_rows<256>(sd, dout, ldo, r0, R, nch);
  constexpr int NPW = WT / 8;
  int degs[NPW], rows[NPW];                    // per-edge metadata of this warp's nodes, requested before the wait
  float as_[NPW], gs_[NPW];
#pragma unroll
  for (int p = 0; p < NPW; ++p) {
    const int nl = warp * NPW + p;
    const bool nok = nl < tn;
    const int beg = nok ? t_rowptr[t0 + nl] : 0;
    degs[p] = nok ? t_rowptr[t0 + nl + 1] - beg : 0;
    rows[p] = 0;
    as_[p] = 0.f;
    gs_[p] = 0.f;
    if (lane < degs[p]) {
      const long long dst = t_col[beg + lane];
      if (dst < r0 || dst >= r1) __trap();
      rows[p] = (int)(dst - r0);
      const int id = t_eid[beg + lane];
      as_[p] = alpha[id];
      gs_[p] = dsig[id] * scale;
    }
  }
  cp_wait_all();
#pragma unroll
  for (int p = 0; p < NPW; ++p) {
    const int nl = warp * NPW + p;
    if (nl >= tn) break;                       // warp-uniform
    const long long node = t0 + nl;
    const int deg = degs[p], row = rows[p];
    const float a = as_[p], g = gs_[p];
    float4 ak = make_float4(0.f, 0.f, 0.f, 0.f), av = ak;
    for (int u = 0; u < deg; ++u) {
      const float au = __shfl_sync(0xffffffffu, a, u), gu = __shfl_sync(0xffffffffu, g, u);
      const int rw = __shfl_sync(0xffffffffu, row, u);
      if (lane < nch) {
        fma4(ak, gu, sq[rw * nch + lane]);
        fma4(av, au, sd[rw * nch + lane]);
      }
    }
    if (lane < nch) {
      st4(dk + node * ldd + 4 * lane, ak);
      st4(dv + node * ldd + 4 * lane, av);
      cs_k.x += ak.x; cs_k.y += ak.y; cs_k.z += ak.z; cs_k.w += ak.w;
      cs_v.x += av.x; cs_v.y += av.y; cs_v.z += av.z; cs_v.w += av.w;
    }
  }
  if (colsum_partial) tile_colsum(attn_sm, cs_k, cs_v, colsum_partial, H);
}

// ---------------------------------------------------------------------------------- K5 EdgeAtt
// by-source softmax of <x_j, u_k> over k in out(j); result stored at the by-destination edge id.
template <typename V, int NC>
__global__ void __launch_bounds__(AW * 32, node_min_blocks<V, NC>)
edgeatt_fwd_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ u, long long ldu,
                   const int* __restrict__ t_rowptr, const int* __restrict__ t_col, const int* __restrict__ t_eid,
                   float* __restrict__ nu, long long N, int H) {
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * AW + (threadIdx.x >> 5);
  if (node >= N) return;
  const int nch = H >> Chunk<V>::SH;
  V xj[NC];
  load_row<V, NC>(x + node * ldx, nch, lane, xj);
  const int beg = t_rowptr[node], end = t_rowptr[node + 1];
  // pass 1: raw scores -> nu[t_eid], running max
  float mx = -INFINITY;
  for (int cb = beg; cb < end; cb += 32) {
    const int cn = min(32, end - cb);
    float my = -INFINITY;
    for (int uu = 0; uu < cn; ++uu) {
      const float d = row_dot<V, NC>(xj, u + (long long)t_col[cb + uu] * ldu, nch, lane);
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
__global__ void __launch_bounds__(AW * 32, node_min_blocks<V, NC>)
edgeatt_bwd_src_kernel(const float* __restrict__ dnu, const float* __restrict__ nu, const float* __restrict__ u,
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
__global__ void __launch_bounds__(AW * 32, node_min_blocks<V, NC>)
edgeatt_bwd_dst_kernel(const float* __restrict__ dsig, const float* __restrict__ x, long long ldx,
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

// window (tile) kernels: 16-byte aligned rows, H % 4 == 0, H <= 384
static int chk(const void* p, long long ld, int H) {
  if ((H & 3) || H <= 0 || H > 384) return ERCG_EINVAL;
  if (!p) return ERCG_EINVAL;
  if ((ld & 3) || !aligned16(p)) return ERCG_EALIGN;
  return ERCG_OK;
}

// warp-per-node kernels: any even H <= 1024, 8-byte aligned rows; *v4 stays true while every row so far also allows
// float4 chunks (16-byte aligned, ld % 4 == 0)
static int chk_row(const void* p, long long ld, int H, bool* v4) {
  if ((H & 1) || H <= 0 || H > 1024) return ERCG_EINVAL;
  if (!p) return ERCG_EINVAL;
  if ((ld & 1) || (reinterpret_cast<uintptr_t>(p) & 7u)) return ERCG_EALIGN;
  *v4 = *v4 && (ld & 3) == 0 && aligned16(p);
  return ERCG_OK;
}

}  // namespace ercg

using namespace ercg;

#define ERCG_CHK(p, ld) do { int rc_ = chk(p, ld, H); if (rc_) return rc_; } while (0)
#define ERCG_CHK_ROW(p, ld) do { int rc_ = chk_row(p, ld, H, &v4_); if (rc_) return rc_; } while (0)
// One warp per node, 8 per CTA.  Chunk type and count from H and the operands only: float4 chunks where every row allows
// them (NC = 1, 2, 3, 4, 6, 8 up to H = 128, 256, 384, 512, 768, 1024), float2 chunks when H % 4 == 2 or a row is only
// 8-byte aligned (NC = 4, 8, 12, 16 up to H = 256, 512, 768, 1024).
#define ERCG_LAUNCH_NC(kernel, ...)                                                                     \
  do {                                                                                                  \
    const unsigned blocks_ = (unsigned)((N + AW - 1) / AW);                                             \
    cudaStream_t st_ = (cudaStream_t)stream;                                                            \
    if (v4_ && H <= 128) kernel<float4, 1><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);                  \
    else if (v4_ && H <= 256) kernel<float4, 2><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);             \
    else if (v4_ && H <= 384) kernel<float4, 3><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);             \
    else if (v4_ && H <= 512) kernel<float4, 4><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);             \
    else if (v4_ && H <= 768) kernel<float4, 6><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);             \
    else if (v4_) kernel<float4, 8><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);                         \
    else if (H <= 256) kernel<float2, 4><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);                    \
    else if (H <= 512) kernel<float2, 8><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);                    \
    else if (H <= 768) kernel<float2, 12><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);                   \
    else kernel<float2, 16><<<blocks_, AW * 32, 0, st_>>>(__VA_ARGS__);                                 \
    return finish_launch();                                                                             \
  } while (0)

extern "C" int ercg_attn_fwd(const float* q, const float* k, const float* v, const float* s, int64_t ld,
                             const int32_t* rowptr, const int32_t* col, float scale,
                             float* out, int64_t ldo, float* alpha, float* dact, int64_t N, int H, void* stream) {
  if (N < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!rowptr || !col) return ERCG_EINVAL;
  bool v4_ = (H & 3) == 0;
  ERCG_CHK_ROW(q, ld); ERCG_CHK_ROW(k, ld); ERCG_CHK_ROW(v, ld); ERCG_CHK_ROW(out, ldo);
  if (s) ERCG_CHK_ROW(s, ld);
  ERCG_LAUNCH_NC(attn_fwd_kernel, q, k, v, s, ld, rowptr, col, scale, out, ldo, alpha, dact, N, H);
}

extern "C" int ercg_attn_bwd_dst(const float* dout, int64_t ldo, const float* k, const float* v, int64_t ld,
                                 const int32_t* rowptr, const int32_t* col, const float* alpha, float scale,
                                 float* dq, float* ds, int64_t ldd, float* dsig, const float* dact, int64_t N, int H,
                                 void* stream) {
  if (N < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!rowptr || !col || !alpha || !dsig) return ERCG_EINVAL;
  bool v4_ = (H & 3) == 0;
  ERCG_CHK_ROW(dout, ldo); ERCG_CHK_ROW(k, ld); ERCG_CHK_ROW(v, ld); ERCG_CHK_ROW(dq, ldd);
  if (ds) ERCG_CHK_ROW(ds, ldd);
  ERCG_LAUNCH_NC(attn_bwd_dst_kernel, dout, ldo, k, v, ld, rowptr, col, alpha, scale, dq, ds, ldd, dsig, dact, N, H);
}

extern "C" int ercg_attn_bwd_src(const float* dout, int64_t ldo, const float* q, int64_t ld,
                                 const int32_t* t_rowptr, const int32_t* t_col, const int32_t* t_eid,
                                 const float* alpha, const float* dsig, float scale,
                                 float* dk, float* dv, int64_t ldd, int64_t N, int H, void* stream) {
  if (N < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!t_rowptr || !t_col || !t_eid || !alpha || !dsig) return ERCG_EINVAL;
  bool v4_ = (H & 3) == 0;
  ERCG_CHK_ROW(dout, ldo); ERCG_CHK_ROW(q, ld); ERCG_CHK_ROW(dk, ldd); ERCG_CHK_ROW(dv, ldd);
  ERCG_LAUNCH_NC(attn_bwd_src_kernel, dout, ldo, q, ld, t_rowptr, t_col, t_eid, alpha, dsig, scale, dk, dv, ldd, N, H);
}

// ---- window-graph variants (contract: the in-neighbours of node i lie in [i - wlo, i + whi]; violated -> trap)
static size_t attn_tile_smem(int H, int wlo, int whi, int full_tiles /* tile-only matrices */, int halo_tiles) {
  const size_t rows = (size_t)(H >> 2) * 16 * ((size_t)full_tiles * WT + (size_t)halo_tiles * (WT + wlo + whi));
  return rows < 8192 ? 8192 : rows;        // tile_colsum reuses the first 8 KB as its reduction buffer (narrow H: rows alone are smaller)
}
static bool attn_tile_ok(int H, int wlo, int whi) { return H <= 128 && (H & 3) == 0 && wlo >= 0 && whi >= 0 && wlo + whi + 1 <= 32; }

static_assert(BT == WT, "the blocked kernels share the tile count (per-CTA column-sum partials) with the tile kernels");
// ERCG_ATTN_BLK=0 forces the round-1 tile kernels (A/B tests; read per call)
static bool attn_use_blk(int H, int wlo, int whi) {
  const char* e = getenv("ERCG_ATTN_BLK");
  return (!e || atoi(e) != 0) && attn_blk_ok(H, wlo, whi);
}
constexpr int ATTN_SMEM_LIMIT = 100 * 1024;   // dynamic shared memory limit of the window-attention kernels

extern "C" int ercg_attn_window_supported(int H, int wlo, int whi) { return attn_tile_ok(H, wlo, whi) ? 1 : 0; }
extern "C" int64_t ercg_attn_window_tiles(int64_t N) { return N <= 0 ? 0 : (N + WT - 1) / WT; }

extern "C" int ercg_attn_window_fwd(const float* q, const float* k, const float* v, const float* s, int64_t ld,
                                    const int32_t* rowptr, const int32_t* col, float scale, float* out, int64_t ldo,
                                    float* alpha, int64_t N, int H, int wlo, int whi, void* stream) {
  if (N < 0 || !attn_tile_ok(H, wlo, whi)) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!rowptr || !col) return ERCG_EINVAL;
  ERCG_CHK(q, ld); ERCG_CHK(k, ld); ERCG_CHK(v, ld); ERCG_CHK(out, ldo);
  if (s) ERCG_CHK(s, ld);
  const size_t sm = attn_tile_smem(H, wlo, whi, 1, 2);
  const unsigned blocks = (unsigned)((N + WT - 1) / WT);
  cudaStream_t st = (cudaStream_t)stream;
  if (attn_use_blk(H, wlo, whi)) {
    if (!smem_limit<attn_fwd_blk_kernel<BTH_FWD>>(ATTN_SMEM_LIMIT)) return ERCG_ECUDA;
    attn_fwd_blk_kernel<BTH_FWD><<<blocks, BTH_FWD, attn_blk_smem(H, wlo, whi, 0), st>>>(q, k, v, s, ld, rowptr, col, scale, out, ldo, alpha, N, H, wlo, whi);
    return finish_launch();
  }
  if (!smem_limit<attn_fwd_tile_kernel<true>>(ATTN_SMEM_LIMIT) || !smem_limit<attn_fwd_tile_kernel<false>>(ATTN_SMEM_LIMIT))
    return ERCG_ECUDA;
  if (wlo + whi + 1 <= 16) attn_fwd_tile_kernel<true><<<blocks, 256, sm, st>>>(q, k, v, s, ld, rowptr, col, scale, out, ldo, alpha, N, H, wlo, whi);
  else attn_fwd_tile_kernel<false><<<blocks, 256, sm, st>>>(q, k, v, s, ld, rowptr, col, scale, out, ldo, alpha, N, H, wlo, whi);
  return finish_launch();
}

extern "C" int ercg_attn_window_bwd_dst(const float* dout, int64_t ldo, const float* k, const float* v, int64_t ld,
                                        const int32_t* rowptr, const int32_t* col, const float* alpha, float scale,
                                        float* dq, float* ds, int64_t ldd, float* dsig, float* colsum_partial,
                                        int64_t N, int H, int wlo, int whi, void* stream) {
  if (N < 0 || !attn_tile_ok(H, wlo, whi)) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!rowptr || !col || !alpha || !dsig) return ERCG_EINVAL;
  ERCG_CHK(dout, ldo); ERCG_CHK(k, ld); ERCG_CHK(v, ld); ERCG_CHK(dq, ldd);
  if (ds) ERCG_CHK(ds, ldd);
  const size_t sm = attn_tile_smem(H, wlo, whi, 1, 2);
  const unsigned blocks = (unsigned)((N + WT - 1) / WT);
  cudaStream_t st = (cudaStream_t)stream;
  if (attn_use_blk(H, wlo, whi)) {
    if (!smem_limit<attn_bwd_dst_blk_kernel<BTH_DST>>(ATTN_SMEM_LIMIT)) return ERCG_ECUDA;
    attn_bwd_dst_blk_kernel<BTH_DST><<<blocks, BTH_DST, attn_blk_smem(H, wlo, whi, 1), st>>>(dout, ldo, k, v, ld, rowptr, col, alpha, scale, dq, ds, ldd, dsig, colsum_partial, N, H, wlo, whi);
    return finish_launch();
  }
  if (!smem_limit<attn_bwd_dst_tile_kernel<true>>(ATTN_SMEM_LIMIT) || !smem_limit<attn_bwd_dst_tile_kernel<false>>(ATTN_SMEM_LIMIT))
    return ERCG_ECUDA;
  if (wlo + whi + 1 <= 16) attn_bwd_dst_tile_kernel<true><<<blocks, 256, sm, st>>>(dout, ldo, k, v, ld, rowptr, col, alpha, scale, dq, ds, ldd, dsig, colsum_partial, N, H, wlo, whi);
  else attn_bwd_dst_tile_kernel<false><<<blocks, 256, sm, st>>>(dout, ldo, k, v, ld, rowptr, col, alpha, scale, dq, ds, ldd, dsig, colsum_partial, N, H, wlo, whi);
  return finish_launch();
}

extern "C" int ercg_attn_window_bwd_src(const float* dout, int64_t ldo, const float* q, int64_t ld,
                                        const int32_t* t_rowptr, const int32_t* t_col, const int32_t* t_eid,
                                        const float* alpha, const float* dsig, float scale, float* dk, float* dv,
                                        int64_t ldd, float* colsum_partial, int64_t N, int H, int wlo, int whi,
                                        void* stream) {
  if (N < 0 || !attn_tile_ok(H, wlo, whi)) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!t_rowptr || !t_col || !t_eid || !alpha || !dsig) return ERCG_EINVAL;
  ERCG_CHK(dout, ldo); ERCG_CHK(q, ld); ERCG_CHK(dk, ldd); ERCG_CHK(dv, ldd);
  const size_t sm = attn_tile_smem(H, wlo, whi, 0, 2);
  const unsigned blocks = (unsigned)((N + WT - 1) / WT);
  if (attn_use_blk(H, wlo, whi)) {
    if (!smem_limit<attn_bwd_src_blk_kernel<BTH_SRC>>(ATTN_SMEM_LIMIT)) return ERCG_ECUDA;
    attn_bwd_src_blk_kernel<BTH_SRC><<<blocks, BTH_SRC, attn_blk_smem(H, wlo, whi, 2), (cudaStream_t)stream>>>(dout, ldo, q, ld, t_rowptr, t_col, t_eid, alpha, dsig, scale, dk, dv, ldd, colsum_partial, N, H, wlo, whi);
    return finish_launch();
  }
  if (!smem_limit<attn_bwd_src_tile_kernel>(ATTN_SMEM_LIMIT)) return ERCG_ECUDA;
  attn_bwd_src_tile_kernel<<<blocks, 256, sm, (cudaStream_t)stream>>>(dout, ldo, q, ld, t_rowptr, t_col, t_eid, alpha, dsig, scale, dk, dv, ldd, colsum_partial, N, H, wlo, whi);
  return finish_launch();
}

extern "C" int ercg_edgeatt_fwd(const float* x, int64_t ldx, const float* u, int64_t ldu,
                                const int32_t* t_rowptr, const int32_t* t_col, const int32_t* t_eid,
                                float* nu, int64_t N, int H, void* stream) {
  if (N < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!t_rowptr || !t_col || !t_eid || !nu) return ERCG_EINVAL;
  bool v4_ = (H & 3) == 0;
  ERCG_CHK_ROW(x, ldx); ERCG_CHK_ROW(u, ldu);
  ERCG_LAUNCH_NC(edgeatt_fwd_kernel, x, ldx, u, ldu, t_rowptr, t_col, t_eid, nu, N, H);
}

extern "C" int ercg_edgeatt_bwd_src(const float* dnu, const float* nu, const float* u, int64_t ldu,
                                    const int32_t* t_rowptr, const int32_t* t_col, const int32_t* t_eid,
                                    float* dsig, float* dx, int64_t lddx, int64_t N, int H, void* stream) {
  if (N < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!dnu || !nu || !t_rowptr || !t_col || !t_eid || !dsig) return ERCG_EINVAL;
  bool v4_ = (H & 3) == 0;
  ERCG_CHK_ROW(u, ldu); ERCG_CHK_ROW(dx, lddx);
  ERCG_LAUNCH_NC(edgeatt_bwd_src_kernel, dnu, nu, u, ldu, t_rowptr, t_col, t_eid, dsig, dx, lddx, N, H);
}

extern "C" int ercg_edgeatt_bwd_dst(const float* dsig, const float* x, int64_t ldx,
                                    const int32_t* rowptr, const int32_t* col,
                                    float* du, int64_t lddu, int64_t N, int H, void* stream) {
  if (N < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!dsig || !rowptr || !col) return ERCG_EINVAL;
  bool v4_ = (H & 3) == 0;
  ERCG_CHK_ROW(x, ldx); ERCG_CHK_ROW(du, lddu);
  ERCG_LAUNCH_NC(edgeatt_bwd_dst_kernel, dsig, x, ldx, rowptr, col, du, lddu, N, H);
}
