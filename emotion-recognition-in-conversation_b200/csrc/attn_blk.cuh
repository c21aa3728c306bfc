// K4 on WINDOW graphs, register-blocked ("blk") kernels: the round-2 replacement of the one-lane-per-edge tile
// kernels.
//
// ncu on the round-1 tile kernels (profiles/r01d_ncu_full_graph_1M.csv): shared-memory wavefronts 50-62 % of peak, DRAM
// 35-38 %: every edge re-read a 400-byte k (or v, dout, q) row from shared memory -- ~110 wavefronts per node against the
// ~17 clocks per node the HBM traffic needs.  Two changes:
// (1) Register blocking over the window structure.  FOUR consecutive destinations i0 .. i0+3 share the 4 + wlo + whi candidate
//     sources [i0 - wlo, i0 + 3 + whi] (14 for COGMEN's 5/5 window), so
//     * score phase: one lane per (block of 4 destinations, candidate source): a k row chunk is read ONCE and used for four
//       dot products (the four q rows are broadcast reads); k is staged chunk-major ([chunk][row], odd row pitch), so lanes
//       with consecutive sources read consecutive float4 -- no bank conflicts.  With 256 threads the 25 chunks of a dot
//       product are split between two thread groups (chunks [0,13) and [13,25)) so that every thread works in this phase;
//     * aggregation phase: one thread per (block of 4 destinations, float4 chunk): 14 v-row chunks for four outputs instead
//       of 11 per output; the weights of a block travel through shared memory as one float4 per candidate.
//     Shared-memory wavefronts per node: ~110 -> ~70.
// (2) What was measured on the way (B200, 2^20 nodes, H = 100, window 5/5; tile kernels: fwd 0.753 / bwd_dst 0.818 / bwd_src
//     0.743 ms):
//     * one tile per 128-thread CTA (no chunk split), 4 CTAs/SM:            0.565 / 0.634 / 0.589 ms
//     * one tile per 256-thread CTA (chunk split, one aggregation round):   0.591 / 0.554 / 0.694 ms
//     * persistent 256-thread CTAs, double-buffered cp.async staging and metadata prefetched one tile ahead, 2 CTAs/SM:
//                                                                           0.718 / 0.781 / 0.855 ms  -- SLOWER: a tile's
//       phases (dots -> barrier -> softmax -> barrier -> weighted sums) are serial inside a CTA, and two resident CTAs per
//       SM (97-104 KB of buffers each) cannot fill each other's barrier gaps the way four independent ones do.  Dropped.
//     ncu of the first variant (profiles/r02d_ncu_attn_blk_v1.csv): no pipe saturated -- shared memory 50 %, issue 56 %,
//     DRAM 50 %, 23 % of the warp slots active: latency-bound.  Each kernel therefore uses the thread count that measured
//     fastest for it (template parameter TH): forward 128, by-destination backward 256, by-source backward 128, and its own
//     unroll factors (A/B runs with one .so per variant: forward / by-source weighted-sum loop not unrolled, by-destination x7;
//     256-thread dot loop not unrolled; 128-thread kernels compiled for 5 CTAs/SM; streaming vs plain stores: no difference).
//     Result: 0.559 / 0.528 / 0.590 ms = 0.59 / 0.63 / 0.47 of the HBM copy peak by each kernel's algorithmic bytes.
//     * packed fp32 FMAs (fma.rn.f32x2 = SASS FFMA2; common.cuh) in the dot-product and weighted-sum loops: 45 -> 29
//       instructions per weighted-sum iteration, yet forward 0.558 -> 0.539 ms, by-source 0.588 -> 0.584 ms (noise),
//       by-destination 0.531 -> 0.596 ms (slower): issue slots are not what these kernels wait for.  Forward only.
// Per-edge arithmetic (chunk order inside each half of the dot products, ascending-source order of the weighted sums) follows
// the tile kernels; the two half dot products and the softmax denominator are combined in a different order, so results
// agree with the tile / generic kernels to rounding (tests: 2e-6), not bit for bit; every order is fixed => run-to-run
// bit-reproducible.  Contract as for the tile kernels: row k's neighbours are the contiguous ascending window
// [k - wlo, k + whi] clipped to its dialogue (K1's graphs); requires 4 + wlo + whi <= 16 and H <= 128.
#pragma once
#include "common.cuh"

namespace ercg {

constexpr int BT = 32;        // destinations (sources, in the by-source kernel) per tile
constexpr int BD = 4;         // rows per register block
constexpr int BCAND = 16;     // candidate slots per block (>= BD + wlo + whi)
constexpr int BNB = BT / BD;  // blocks per tile
#ifndef BLK_STREAM
#define BLK_STREAM 1            // outputs are written once and read by a later kernel: keep them out of L1
#endif
#ifndef BLK_UNROLL2
#define BLK_UNROLL2 1
#endif
#ifndef BLK_MINB
#define BLK_MINB 5              // minimum resident CTAs per SM the 128-thread kernels are compiled for
#endif
constexpr int kBlkUnroll2 = BLK_UNROLL2;
__device__ __forceinline__ void blk_st(float* p, float4 v) {
#if BLK_STREAM
  st4_stream(p, v);
#else
  st4(p, v);
#endif
}

// Rows go global -> shared with 16-byte cp.async (LDGSTS): a lane issues all of its row chunks back to back, no registers
// are tied up and nobody waits until cp_wait_all(), so the whole tile's HBM latency is paid once and the CSR metadata loads
// issued right after overlap with it.  (The first tile kernels staged through registers -- ptxas kept only four loads in
// flight per lane -- and ran at 35-40 % of the HBM peak.)
__device__ __forceinline__ void cp16(float4* dst, const float* src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
  __syncthreads();
}
__device__ __forceinline__ float h16_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 8));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 4));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
}
__device__ __forceinline__ float h16_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 8);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v + __shfl_xor_sync(0xffffffffu, v, 1);
}
// rows [r0, r0 + rows) of a row-major [*, 4 * nch] matrix -> shared, row-major (lane = chunk)
template <int TH>
__device__ __forceinline__ void blk_stage_rows(float4* dst, const float* __restrict__ src, long long ld, long long r0, int rows, int nch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane < nch)
    for (int r = warp; r < rows; r += TH / 32) cp16(dst + r * nch + lane, src + (r0 + r) * ld + 4 * lane);
}
// same rows, chunk-major: element (r, c) at dst[c * RP + r]; RP odd => the 8 lanes of a quarter-warp (consecutive c) hit 8
// different 16-byte bank groups
template <int TH>
__device__ __forceinline__ void blk_stage_rows_t(float4* dst, const float* __restrict__ src, long long ld, long long r0, int rows, int nch, int RP) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane < nch)
    for (int r = warp; r < rows; r += TH / 32) cp16(dst + lane * RP + r, src + (r0 + r) * ld + 4 * lane);
}

struct BlkGeom {
  long long t0, r0;
  int tn, R;
};
__device__ __forceinline__ BlkGeom blk_geom(long long tile, long long N, int wlo, int whi) {
  BlkGeom g;
  g.t0 = tile * BT;
  g.tn = (int)min((long long)BT, N - g.t0);
  g.r0 = max(0LL, g.t0 - wlo);
  g.R = (int)(min(N, g.t0 + g.tn + whi) - g.r0);
  return g;
}

// CSR rows of the four nodes of this lane's block: first edge, degree, first neighbour (rows are contiguous ascending)
struct BlkRows {
  int beg[BD], deg[BD], first[BD];
};
__device__ __forceinline__ BlkRows blk_rows(const int* __restrict__ rowptr, const int* __restrict__ col, long long i0, int il0, int tn) {
  BlkRows m;
#pragma unroll
  for (int d = 0; d < BD; ++d) {
    const bool ok = il0 + d < tn;
    m.beg[d] = ok ? rowptr[i0 + d] : 0;
    m.deg[d] = ok ? rowptr[i0 + d + 1] - m.beg[d] : 0;
  }
#pragma unroll
  for (int d = 0; d < BD; ++d) m.first[d] = m.deg[d] > 0 ? col[m.beg[d]] : 0;
  return m;
}
// edge slot of candidate `cand` in row d of the block, or -1
__device__ __forceinline__ int blk_edge(const BlkRows& m, int d, long long cand, bool in_range) {
  const long long off = cand - (long long)m.first[d];
  return (in_range && m.deg[d] > 0 && off >= 0 && off < (long long)m.deg[d]) ? m.beg[d] + (int)off : -1;
}

// column sums over the blocks of a tile: every (block, chunk) item has written its two float4 into red[BNB][2][nch]; this
// adds them up in block order -> partial[tile][2H]
__device__ __forceinline__ void blk_colsum_finish(const float4* red, int nch, float* __restrict__ partial, long long tile, int H) {
  __syncthreads();
  const int tid = threadIdx.x;
  if (tid < 2 * nch) {
    const int which = tid / nch, cc = tid - which * nch;
    float4 t = red[which * nch + cc];
#pragma unroll
    for (int w = 1; w < BNB; ++w) {
      const float4 v = red[(w * 2 + which) * nch + cc];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    st4(partial + tile * 2 * H + which * H + 4 * cc, t);
  }
}

// Banded products of one tile, score phase: sc[d] = <a_{i0+d}, b_cand>.  arows: [BT][nch] row-major (tile rows); bt: [nch][RP]
// chunk-major.  GRP == 2 (256 threads): each thread group takes half of the chunks, group 1 hands its partial sums to group 0
// through `spart` (one barrier); GRP == 1: the whole dot product, in chunk order.
template <int GRP, bool PK = false>
__device__ __forceinline__ void blk_dots(const float4* __restrict__ arows, const float4* __restrict__ bt, int RP, int nch, int il0, int r,
                                         bool any, int grp, float4* __restrict__ spart, int slot, float sc[BD]) {
  const int cmid = (nch + 1) >> 1;
  const int c0 = (GRP == 2 && grp) ? cmid : 0, c1 = (GRP == 2 && !grp) ? cmid : nch;
  sc[0] = sc[1] = sc[2] = sc[3] = 0.f;
  if (PK) {                      // packed FMAs (FFMA2): even / odd partial sums per destination, added at the end
    float2 s2[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d) s2[d] = make_float2(0.f, 0.f);
    if (any) {
      const float4* br = bt + r;
      const float4* a0 = arows + il0 * nch;
#pragma unroll 5
      for (int c = c0; c < c1; ++c) {
        const float4 bc = br[c * RP];
#pragma unroll
        for (int d = 0; d < BD; ++d) dot4_acc2(s2[d], a0[d * nch + c], bc);
      }
    }
#pragma unroll
    for (int d = 0; d < BD; ++d) sc[d] = s2[d].x + s2[d].y;
  } else if (any) {
    const float4* br = bt + r;
    const float4* a0 = arows + il0 * nch;
    if (GRP == 2) {
#pragma unroll kBlkUnroll2
      for (int c = c0; c < c1; ++c) {
        const float4 bc = br[c * RP];
#pragma unroll
        for (int d = 0; d < BD; ++d) sc[d] += dot4(a0[d * nch + c], bc);
      }
    } else {
#pragma unroll 5
      for (int c = c0; c < c1; ++c) {
        const float4 bc = br[c * RP];
#pragma unroll
        for (int d = 0; d < BD; ++d) sc[d] += dot4(a0[d * nch + c], bc);
      }
    }
  }
  if (GRP == 2) {
    if (grp) spart[slot] = make_float4(sc[0], sc[1], sc[2], sc[3]);
    __syncthreads();
    if (!grp) {
      const float4 p = spart[slot];
      sc[0] += p.x; sc[1] += p.y; sc[2] += p.z; sc[3] += p.w;
    }
  }
}

// ------------------------------------------------------------------------------------------------ forward
template <int TH>
__global__ void __launch_bounds__(TH, TH == 128 ? BLK_MINB : 4)
attn_fwd_blk_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                    const float* __restrict__ s, long long ld, const int* __restrict__ rowptr, const int* __restrict__ col,
                    float scale, float* __restrict__ out, long long ldo, float* __restrict__ alpha, long long N, int H,
                    int wlo, int whi) {
  extern __shared__ float4 blk_sm[];
  constexpr int GRP = TH / 128;
  const int nch = H >> 2, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Rmax = BT + wlo + whi, RP = Rmax | 1, ncand = BD + wlo + whi;
  const BlkGeom g = blk_geom(blockIdx.x, N, wlo, whi);
  float4* sq = blk_sm;                       // [BT][nch]      q rows of the tile
  float4* skt = sq + BT * nch;               // [nch][RP]      k rows of tile + halo, chunk-major
  float4* sv = skt + nch * RP;               // [Rmax][nch]    v rows of tile + halo
  float4* sa = sv + Rmax * nch;              // [BNB][BCAND]   alpha of the 4 destinations of a block at each candidate
  float4* spart = sa + BNB * BCAND;          // [BNB][BCAND]   partial scores of thread group 1 (GRP == 2)
  blk_stage_rows<TH>(sq, q, ld, g.t0, g.tn, nch);
  blk_stage_rows_t<TH>(skt, k, ld, g.r0, g.R, nch, RP);
  blk_stage_rows<TH>(sv, v, ld, g.r0, g.R, nch);
  // ---- score phase: lane = (block b, candidate jj) [x thread group = half of the chunks]
  const int grp = warp >> 2, b = (warp & 3) * 2 + (lane >> 4), jj = lane & 15, il0 = b * BD, slot = b * BCAND + jj;
  const long long cand = g.t0 + il0 - wlo + jj;                    // global row of this lane's candidate source
  const BlkRows m = blk_rows(rowptr, col, g.t0 + il0, il0, g.tn);  // requested while the copies are in flight
  int e[BD];
  bool any = false;
#pragma unroll
  for (int d = 0; d < BD; ++d) {
    e[d] = blk_edge(m, d, cand, jj < ncand);
    any |= e[d] >= 0;
  }
  const int r = (int)min(max(cand - g.r0, 0LL), (long long)(g.R - 1));
  cp_wait_all();
  float sc[BD];
  blk_dots<GRP, true>(sq, skt, RP, nch, il0, r, any, grp, spart, slot, sc);
  if (!grp) {
    float al[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d) {
      const bool val = e[d] >= 0;
      const float x = sc[d] * scale;
      const float mx = h16_max(val ? x : -INFINITY);
      const float ex = val ? expf(x - mx) : 0.f;
      const float inv = 1.f / (h16_sum(ex) + 1e-16f);
      al[d] = ex * inv;
      if (val && alpha) alpha[e[d]] = al[d];
    }
    sa[slot] = make_float4(al[0], al[1], al[2], al[3]);
  }
  __syncthreads();
  // ---- aggregation phase: thread = (block bb, chunk c)
  for (int it = tid; it < BNB * nch; it += TH) {
    const int bb = it / nch, c = it - bb * nch, jl0 = bb * BD;
    float4 skip[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d)
      skip[d] = (s && jl0 + d < g.tn) ? ld4(s + (g.t0 + jl0 + d) * ld + 4 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 acc[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d) acc[d] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int rb = (int)(g.t0 + jl0 - wlo - g.r0);                 // row (may be < 0 in the first tile: clamped, weight 0)
#pragma unroll 1
    for (int j = 0; j < ncand; ++j) {
      const int rr = min(max(rb + j, 0), g.R - 1);
      const float4 a4 = sa[bb * BCAND + j];
      const float4 vv = sv[rr * nch + c];
      fma4_p(acc[0], a4.x, vv); fma4_p(acc[1], a4.y, vv); fma4_p(acc[2], a4.z, vv); fma4_p(acc[3], a4.w, vv);
    }
#pragma unroll
    for (int d = 0; d < BD; ++d)
      if (jl0 + d < g.tn) {
        acc[d].x += skip[d].x; acc[d].y += skip[d].y; acc[d].z += skip[d].z; acc[d].w += skip[d].w;
        blk_st(out + (g.t0 + jl0 + d) * ldo + 4 * c, acc[d]);
      }
  }
}

// ------------------------------------------------------------------------------------------------ backward, by destination
//   dalpha[j->i] = <dout_i, v_j>;  D_i = sum_j alpha dalpha;  dsig = alpha (dalpha - D_i);  dq_i = scale sum_j dsig k_j;  ds_i = dout_i
template <int TH>
__global__ void __launch_bounds__(TH, TH == 128 ? BLK_MINB : 4)
attn_bwd_dst_blk_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ k, const float* __restrict__ v,
                        long long ld, const int* __restrict__ rowptr, const int* __restrict__ col, const float* __restrict__ alpha,
                        float scale, float* __restrict__ dq, float* __restrict__ ds, long long ldd, float* __restrict__ dsig,
                        float* __restrict__ colsum_partial, long long N, int H, int wlo, int whi) {
  extern __shared__ float4 blk_sm[];
  constexpr int GRP = TH / 128;
  const int nch = H >> 2, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Rmax = BT + wlo + whi, RP = Rmax | 1, ncand = BD + wlo + whi;
  const BlkGeom g = blk_geom(blockIdx.x, N, wlo, whi);
  float4* sd = blk_sm;                       // [BT][nch]      dout rows of the tile
  float4* svt = sd + BT * nch;               // [nch][RP]      v rows, chunk-major (dot products)
  float4* sk = svt + nch * RP;               // [Rmax][nch]    k rows (weighted sums)
  float4* sa = sk + Rmax * nch;              // [BNB][BCAND]   dsig * scale of the 4 destinations of a block
  float4* spart = sa + BNB * BCAND;
  float4* red = spart + BNB * BCAND;         // [BNB][2][nch]
  blk_stage_rows<TH>(sd, dout, ldo, g.t0, g.tn, nch);
  blk_stage_rows_t<TH>(svt, v, ld, g.r0, g.R, nch, RP);
  blk_stage_rows<TH>(sk, k, ld, g.r0, g.R, nch);
  const int grp = warp >> 2, b = (warp & 3) * 2 + (lane >> 4), jj = lane & 15, il0 = b * BD, slot = b * BCAND + jj;
  const long long cand = g.t0 + il0 - wlo + jj;
  const BlkRows m = blk_rows(rowptr, col, g.t0 + il0, il0, g.tn);
  int e[BD];
  float al[BD];
  bool any = false;
#pragma unroll
  for (int d = 0; d < BD; ++d) {
    e[d] = blk_edge(m, d, cand, jj < ncand);
    any |= e[d] >= 0;
    al[d] = (e[d] >= 0 && !grp) ? alpha[e[d]] : 0.f;
  }
  const int r = (int)min(max(cand - g.r0, 0LL), (long long)(g.R - 1));
  cp_wait_all();
  float da[BD];
  blk_dots<GRP>(sd, svt, RP, nch, il0, r, any, grp, spart, slot, da);
  if (!grp) {
    float gs[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d) {
      const bool val = e[d] >= 0;
      const float x = val ? da[d] : 0.f;
      const float D = h16_sum(al[d] * x);
      const float gg = al[d] * (x - D);
      if (val) dsig[e[d]] = gg;
      gs[d] = val ? gg * scale : 0.f;
    }
    sa[slot] = make_float4(gs[0], gs[1], gs[2], gs[3]);
  }
  __syncthreads();
  for (int it = tid; it < BNB * nch; it += TH) {
    const int bb = it / nch, c = it - bb * nch, jl0 = bb * BD;
    float4 acc[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d) acc[d] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int rb = (int)(g.t0 + jl0 - wlo - g.r0);
#pragma unroll 7
    for (int j = 0; j < ncand; ++j) {
      const int rr = min(max(rb + j, 0), g.R - 1);
      const float4 a4 = sa[bb * BCAND + j];
      const float4 kk = sk[rr * nch + c];
      fma4(acc[0], a4.x, kk); fma4(acc[1], a4.y, kk); fma4(acc[2], a4.z, kk); fma4(acc[3], a4.w, kk);
    }
    float4 csq = make_float4(0.f, 0.f, 0.f, 0.f), css = csq;
#pragma unroll
    for (int d = 0; d < BD; ++d)
      if (jl0 + d < g.tn) {
        blk_st(dq + (g.t0 + jl0 + d) * ldd + 4 * c, acc[d]);
        const float4 dsv = sd[(jl0 + d) * nch + c];
        if (ds) blk_st(ds + (g.t0 + jl0 + d) * ldd + 4 * c, dsv);
        csq.x += acc[d].x; csq.y += acc[d].y; csq.z += acc[d].z; csq.w += acc[d].w;
        css.x += dsv.x; css.y += dsv.y; css.z += dsv.z; css.w += dsv.w;
      }
    red[(bb * 2 + 0) * nch + c] = csq;
    red[(bb * 2 + 1) * nch + c] = css;
  }
  // bias gradient of the q / skip Linears = column sums of dq | ds, reduced per tile here so nobody re-reads the [N,4H] gradient
  if (colsum_partial) blk_colsum_finish(red, nch, colsum_partial, blockIdx.x, H);
}

// ------------------------------------------------------------------------------------------------ backward, by source
//   dv_j = sum_i alpha[j->i] dout_i;  dk_j = scale sum_i dsig[j->i] q_i   over the out-edges of j (contiguous window of destinations)
template <int TH>
__global__ void __launch_bounds__(TH, TH == 128 ? BLK_MINB : 4)
attn_bwd_src_blk_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ q, long long ld,
                        const int* __restrict__ t_rowptr, const int* __restrict__ t_col, const int* __restrict__ t_eid,
                        const float* __restrict__ alpha, const float* __restrict__ dsig, float scale, float* __restrict__ dk,
                        float* __restrict__ dv, long long ldd, float* __restrict__ colsum_partial, long long N, int H, int wlo, int whi) {
  extern __shared__ float4 blk_sm[];
  const int nch = H >> 2, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Rmax = BT + wlo + whi, ncand = BD + wlo + whi;
  const BlkGeom g = blk_geom(blockIdx.x, N, wlo, whi);
  float4* sq = blk_sm;                       // [Rmax][nch] q rows of tile + halo
  float4* sd = sq + Rmax * nch;              // [Rmax][nch] dout rows of tile + halo
  float4* sa = sd + Rmax * nch;              // [BNB][BCAND] alpha of the 4 sources of a block at each candidate destination
  float4* sg = sa + BNB * BCAND;             // [BNB][BCAND] dsig * scale
  float4* red = sg + BNB * BCAND;            // [BNB][2][nch]
  blk_stage_rows<TH>(sq, q, ld, g.r0, g.R, nch);
  blk_stage_rows<TH>(sd, dout, ldo, g.r0, g.R, nch);
  if (warp < 4) {                            // lane = (block of 4 sources, candidate destination): per-edge weights via the transpose
    const int b = warp * 2 + (lane >> 4), jj = lane & 15, il0 = b * BD;
    const long long cand = g.t0 + il0 - wlo + jj;
    const BlkRows m = blk_rows(t_rowptr, t_col, g.t0 + il0, il0, g.tn);
    float a[BD], gg[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d) {
      const int te = blk_edge(m, d, cand, jj < ncand);
      a[d] = gg[d] = 0.f;
      if (te >= 0) {
        const int id = t_eid[te];
        a[d] = alpha[id];
        gg[d] = dsig[id] * scale;
      }
    }
    sa[b * BCAND + jj] = make_float4(a[0], a[1], a[2], a[3]);
    sg[b * BCAND + jj] = make_float4(gg[0], gg[1], gg[2], gg[3]);
  }
  cp_wait_all();
  for (int it = tid; it < BNB * nch; it += TH) {
    const int bb = it / nch, c = it - bb * nch, jl0 = bb * BD;
    float4 ak[BD], av[BD];
#pragma unroll
    for (int d = 0; d < BD; ++d) ak[d] = av[d] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int rb = (int)(g.t0 + jl0 - wlo - g.r0);
#pragma unroll 1
    for (int j = 0; j < ncand; ++j) {
      const int rr = min(max(rb + j, 0), g.R - 1);
      const float4 wa = sa[bb * BCAND + j], wg = sg[bb * BCAND + j];
      const float4 qq = sq[rr * nch + c], dd = sd[rr * nch + c];
      fma4(ak[0], wg.x, qq); fma4(ak[1], wg.y, qq); fma4(ak[2], wg.z, qq); fma4(ak[3], wg.w, qq);
      fma4(av[0], wa.x, dd); fma4(av[1], wa.y, dd); fma4(av[2], wa.z, dd); fma4(av[3], wa.w, dd);
    }
    float4 csk = make_float4(0.f, 0.f, 0.f, 0.f), csv = csk;
#pragma unroll
    for (int d = 0; d < BD; ++d)
      if (jl0 + d < g.tn) {
        blk_st(dk + (g.t0 + jl0 + d) * ldd + 4 * c, ak[d]);
        blk_st(dv + (g.t0 + jl0 + d) * ldd + 4 * c, av[d]);
        csk.x += ak[d].x; csk.y += ak[d].y; csk.z += ak[d].z; csk.w += ak[d].w;
        csv.x += av[d].x; csv.y += av[d].y; csv.z += av[d].z; csv.w += av[d].w;
      }
    red[(bb * 2 + 0) * nch + c] = csk;
    red[(bb * 2 + 1) * nch + c] = csv;
  }
  if (colsum_partial) blk_colsum_finish(red, nch, colsum_partial, blockIdx.x, H);
}

constexpr int BTH_FWD = 128, BTH_DST = 256, BTH_SRC = 128;       // measured fastest per kernel (see the header comment)

inline bool attn_blk_ok(int H, int wlo, int whi) {
  return H <= 128 && (H & 3) == 0 && wlo >= 0 && whi >= 0 && BD + wlo + whi <= BCAND;
}
inline size_t attn_blk_smem(int H, int wlo, int whi, int kind /* 0 fwd, 1 bwd_dst, 2 bwd_src */) {
  const int nch = H >> 2, Rmax = BT + wlo + whi, RP = Rmax | 1;
  size_t f4 = 0;
  if (kind == 0) f4 = (size_t)BT * nch + (size_t)nch * RP + (size_t)Rmax * nch + 2 * BNB * BCAND;
  else if (kind == 1) f4 = (size_t)BT * nch + (size_t)nch * RP + (size_t)Rmax * nch + 2 * BNB * BCAND + (size_t)BNB * 2 * nch;
  else f4 = (size_t)2 * Rmax * nch + 2 * BNB * BCAND + (size_t)BNB * 2 * nch;
  return f4 * 16;
}

}  // namespace ercg
