// K12: the DialogueRNN recurrence (DialogueRNN / DialogueRNNCell, track_mm/dgcnv2_models.py:235-348; declare-lab DialogueRNN,
// listener_state=False, context_attention 'simple' | 'general'), forward and backward through time.
//
// The reference runs a Python loop over utterance positions; per step it evaluates three GRUCells (the party cell for every
// party), a batched attention over the whole global-state history and re-concatenates that history.  Here one persistent
// cooperative kernel per direction runs every dialogue in lockstep, like K10 (dagerc.cu):
//  * the U-dependent input-gate terms of g_cell / p_cell and the 'general' query W_a U_t are one hoisted GEMM (K2) over all
//    L*B rows before the kernel ("pre", "xq");
//  * the sequential weights (W_ih^g[:, Dm:], W_hh^g, W_ih^p[:, Dm:], W_hh^p, W_ih^e, W_hh^e: 1.4 MB at 150/150/100, 4.7 MB at
//    256/256/256) stay resident in shared memory, sliced by hidden unit across the CTAs (each CTA owns a contiguous range
//    of the units of every cell, all three gate rows of each);
//  * a warp handles one dialogue at a time: the input vector [x ; h] of a cell is read once into registers and dotted with
//    the rows of every owned unit; the attention of dialogue b is done by one warp of CTA b % grid ("owner").
// Forward, step t: phase A = g cell (needs g_{t-1}, q_{t-1}[s]), attention c_t (needs g_0..g_{t-1}) and the e cell of step
// t-1 (needs q_{t-1}[s_{t-1}], trailing one phase behind because nothing reads e); grid.sync; phase B = the party cell (needs
// c_t); grid.sync.  Backward, step t in reverse: P2 = party-cell gates (W_ih^e^T dei_t), e-cell gates of t-1
// (W_hh^e^T deh_t) and g-cell gates (dG_t is complete); P3 = the transposed products of dpi, dph, dgi, dgh; P4 = attention
// backward (adds alpha dc + da xq to dG_j, j < t, per dialogue in j order).  The weight gradients are TN GEMMs (K2) of the
// saved rows, as for K6b.  All sums are in a fixed order and there are no atomics, so results are bit-reproducible.
#include <cooperative_groups.h>
#include "common.cuh"
namespace cg = cooperative_groups;

namespace ercg {

constexpr int RT = 512, RNW = RT / 32;
constexpr int RKC = 16;          // register chunks of 32 per lane: cell input vectors [x ; h] of up to 512 floats
constexpr int RQC = 8;           // chunks for Dg-wide vectors (Dg <= 256)
constexpr int RNN_MAXD = 256, RNN_MAXP = 16;

__device__ __forceinline__ float drnn_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }
// ercg_dropout's mask: kept iff hash_uniform(seed, idx) >= p, kept elements scaled by 1 / (1 - p)
__device__ __forceinline__ float drnn_keep(uint64_t seed, long long idx, float p, float scale) {
  return hash_uniform(seed, (uint64_t)idx) < p ? 0.f : scale;
}
// s = first argmax of the qmask row, m = its value
__device__ __forceinline__ void drnn_speaker(const float* __restrict__ qm, int P, int& s, float& m) {
  s = 0; m = __ldg(qm);
  for (int p = 1; p < P; ++p) { const float v = __ldg(qm + p); if (v > m) { m = v; s = p; } }
}
__device__ __forceinline__ void unit_range(int D, int& u0, int& n) {
  const long long G = gridDim.x, i = blockIdx.x;
  u0 = (int)(i * D / G);
  n = (int)((i + 1) * D / G) - u0;
}

// xr[c] = element lane + 32 c of [a (na) ; b (nb)], b == nullptr reads as zeros, 0 past the end
__device__ __forceinline__ void load_cat(float (&xr)[RKC], const float* a, int na, const float* b, int nb, int lane) {
#pragma unroll
  for (int c = 0; c < RKC; ++c) {
    const int k = lane + 32 * c;
    float v = 0.f;
    if (k < na) v = __ldcg(a + k);
    else if (k < na + nb && b != nullptr) v = __ldcg(b + k - na);
    xr[c] = v;
  }
}
// the four sums of one GRU unit over [x (nx) ; h]: r and z rows over both parts, the n row split into its x and h parts
struct Gate4 { float r, z, nx, nh; };
__device__ __forceinline__ Gate4 gate_dots(const float (&xr)[RKC], const float* w, int K, int nx, int lane) {
  float ar = 0.f, az = 0.f, anx = 0.f, anh = 0.f;
#pragma unroll
  for (int c = 0; c < RKC; ++c) {
    const int k = lane + 32 * c;
    if (k < K) {
      const float x = xr[c];
      ar = fmaf(w[k], x, ar);
      az = fmaf(w[K + k], x, az);
      if (k < nx) anx = fmaf(w[2 * K + k], x, anx); else anh = fmaf(w[2 * K + k], x, anh);
    }
  }
  return Gate4{warp_sum(ar), warp_sum(az), warp_sum(anx), warp_sum(anh)};
}
// dot of a shared-memory column with a global vector (K <= 768), lane-strided, fixed order; all loads are issued before
// the first FMA so a call waits for one memory latency, not K/32
constexpr int RCC = 24;
__device__ __forceinline__ float col_dot(const float* w, const float* x, int K, int lane) {
  float xv[RCC];
#pragma unroll
  for (int c = 0; c < RCC; ++c) { const int k = lane + 32 * c; xv[c] = k < K ? __ldcg(x + k) : 0.f; }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < RCC; ++c) { const int k = lane + 32 * c; if (k < K) s = fmaf(w[k], xv[c], s); }
  return warp_sum(s);
}
// lane's part of q . g_j for the four history rows j0 .. j0+3 (rows >= t read as zero), loads issued together
constexpr int RJ = 4;
__device__ __forceinline__ void hist_dots(float (&part)[RJ], const float (&q)[RQC], const float* g, long long B, int b, int Dg,
                                          int j0, int t, int lane) {
#pragma unroll
  for (int u = 0; u < RJ; ++u) {
    part[u] = 0.f;
    if (j0 + u < t) {
      const float* gj = g + ((long long)(j0 + u) * B + b) * Dg;
#pragma unroll
      for (int c = 0; c < RQC; ++c) { const int k = lane + 32 * c; if (k < Dg) part[u] = fmaf(q[c], __ldcg(gj + k), part[u]); }
    }
  }
}

struct DrnnParams {
  int L, B, Dg, Dp, De, P;
  float p, scale;
  uint64_t sg, sq, se;
  const float* qmask; const float* pre; long long ldpre; const float* xq; long long ldxq;
  const float *Wgq, *Whh_g, *bhh_g, *Wpc, *Whh_p, *bhh_p, *Wih_e, *Whh_e, *bih_e, *bhh_e;
  float *e, *g, *c, *qprev, *qcur, *gg, *gp, *ge, *alpha, *qstate;
  const float* de; float* dpre; long long lddpre; float* dxq; long long lddxq;
  float *dgh, *dph, *dei, *deh, *dG, *dQ, *dEh, *dc;
};

__device__ __forceinline__ float* alpha_block(const DrnnParams& p, int t, int b) {
  return p.alpha + (long long)p.B * t * (t - 1) / 2 + (long long)b * t;
}

__global__ void __launch_bounds__(RT, 1) drnn_fwd_kernel(DrnnParams p) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ float4 drnn_smem4[];
  float* sm = reinterpret_cast<float*>(drnn_smem4);
  const int Dg = p.Dg, Dp = p.Dp, De = p.De, B = p.B;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int g0, ng, p0, np, e0, ne;
  unit_range(Dg, g0, ng); unit_range(Dp, p0, np); unit_range(De, e0, ne);
  const int Kg = Dp + Dg, Kp = Dg + Dp, Ke = Dp + De;
  float* Wg = sm;                          // [ng][3][Kg]  rows (r,z,n) of [W_ih^g[:, Dm:] | W_hh^g]
  float* Wp = Wg + ng * 3 * Kg;            // [np][3][Kp]  rows of [W_ih^p[:, Dm:] | W_hh^p]
  float* We = Wp + np * 3 * Kp;            // [ne][3][Ke]  rows of [W_ih^e | W_hh^e]
  float* bs = We + ne * 3 * Ke;            // [ng][3] b_hh^g, [np][3] b_hh^p, [ne][6] b_ih^e, b_hh^e
  for (int i = tid; i < ng * 3 * Kg; i += RT) {
    const int uu = i / (3 * Kg), q = (i / Kg) % 3, k = i % Kg;
    const long long row = (long long)q * Dg + g0 + uu;
    Wg[i] = k < Dp ? p.Wgq[row * Dp + k] : p.Whh_g[row * Dg + k - Dp];
  }
  for (int i = tid; i < np * 3 * Kp; i += RT) {
    const int uu = i / (3 * Kp), q = (i / Kp) % 3, k = i % Kp;
    const long long row = (long long)q * Dp + p0 + uu;
    Wp[i] = k < Dg ? p.Wpc[row * Dg + k] : p.Whh_p[row * Dp + k - Dg];
  }
  for (int i = tid; i < ne * 3 * Ke; i += RT) {
    const int uu = i / (3 * Ke), q = (i / Ke) % 3, k = i % Ke;
    const long long row = (long long)q * De + e0 + uu;
    We[i] = k < Dp ? p.Wih_e[row * Dp + k] : p.Whh_e[row * De + k - Dp];
  }
  for (int i = tid; i < ng * 3; i += RT) bs[i] = p.bhh_g[(i % 3) * Dg + g0 + i / 3];
  for (int i = tid; i < np * 3; i += RT) bs[ng * 3 + i] = p.bhh_p[(i % 3) * Dp + p0 + i / 3];
  for (int i = tid; i < ne * 6; i += RT) {
    const int q = i % 6;
    bs[(ng + np) * 3 + i] = (q < 3 ? p.bih_e : p.bhh_e)[(q % 3) * De + e0 + i / 6];
  }
  for (long long i = tid; i < (long long)B * p.P * np; i += RT) p.qstate[(i / np) * Dp + p0 + i % np] = 0.f;
  __syncthreads();
  grid.sync();

  const float* bg = bs;
  const float* bp = bs + ng * 3;
  const float* be = bs + (ng + np) * 3;
  float xr[RKC];
  for (int t = 0; t <= p.L; ++t) {
    // ---------------- phase A: g cell and attention of step t, e cell of step t-1
    for (int b = warp; b < B; b += RNW) {
      const bool owner = (b % (int)gridDim.x) == (int)blockIdx.x;
      if (t < p.L && (ng > 0 || owner)) {
        const long long r = (long long)t * B + b;
        int s; float m;
        drnn_speaker(p.qmask + r * p.P, p.P, s, m);
        const float* qs = p.qstate + ((long long)b * p.P + s) * Dp;
        const float* gprev = t > 0 ? p.g + (r - B) * Dg : nullptr;
        load_cat(xr, qs, Dp, gprev, Dg, lane);
        if (owner) {
#pragma unroll
          for (int c = 0; c < RKC; ++c) { const int k = lane + 32 * c; if (k < Dp) p.qprev[r * Dp + k] = xr[c]; }
        }
        const float* pr = p.pre + r * p.ldpre;
        for (int uu = 0; uu < ng; ++uu) {
          const Gate4 a = gate_dots(xr, Wg + uu * 3 * Kg, Kg, Dp, lane);
          if (lane == 0) {
            const int u = g0 + uu;
            const float* b3 = bg + uu * 3;
            const float rg = drnn_sigmoid(__ldg(pr + u) + a.r + b3[0]);
            const float zg = drnn_sigmoid(__ldg(pr + Dg + u) + a.z + b3[1]);
            const float hn = a.nh + b3[2];
            const float n = tanhf(__ldg(pr + 2 * Dg + u) + a.nx + rg * hn);
            const float hp = gprev ? __ldcg(gprev + u) : 0.f;
            const float h = (1.f - zg) * n + zg * hp;
            p.g[r * Dg + u] = h * drnn_keep(p.sg, r * Dg + u, p.p, p.scale);
            float* gt = p.gg + r * 4 * Dg;
            gt[u] = rg; gt[Dg + u] = zg; gt[2 * Dg + u] = n; gt[3 * Dg + u] = hn;
          }
        }
        if (owner) {                       // c_t = sum_{j<t} softmax_j(xq . g_j) g_j over the dropped-out history
          float* crow = p.c + r * Dg;
          float acc[RQC];
#pragma unroll
          for (int c = 0; c < RQC; ++c) acc[c] = 0.f;
          if (t > 0) {
            const float* xq = p.xq + r * p.ldxq;
            float q[RQC];
#pragma unroll
            for (int c = 0; c < RQC; ++c) { const int k = lane + 32 * c; q[c] = k < Dg ? __ldg(xq + k) : 0.f; }
            float* al = alpha_block(p, t, b);
            float mx = -INFINITY;
            for (int j0 = 0; j0 < t; j0 += RJ) {
              float part[RJ];
              hist_dots(part, q, p.g, B, b, Dg, j0, t, lane);
#pragma unroll
              for (int u = 0; u < RJ; ++u) {
                if (j0 + u < t) {
                  const float sc = warp_sum(part[u]);
                  if (((j0 + u) & 31) == lane) al[j0 + u] = sc;
                  mx = fmaxf(mx, sc);
                }
              }
            }
            float z = 0.f;
            for (int j = lane; j < t; j += 32) z += expf(al[j] - mx);     // al[j] was written by this lane
            z = warp_sum(z);
            for (int j = lane; j < t; j += 32) al[j] = expf(al[j] - mx) / z;
            __syncwarp();
#pragma unroll 4
            for (int j = 0; j < t; ++j) {
              const float a = __ldcg(al + j);
              const float* gj = p.g + ((long long)j * B + b) * Dg;
#pragma unroll
              for (int c = 0; c < RQC; ++c) { const int k = lane + 32 * c; if (k < Dg) acc[c] = fmaf(a, __ldcg(gj + k), acc[c]); }
            }
          }
#pragma unroll
          for (int c = 0; c < RQC; ++c) { const int k = lane + 32 * c; if (k < Dg) crow[k] = acc[c]; }
        }
      }
      if (t >= 1 && ne > 0) {
        const long long r = (long long)(t - 1) * B + b;
        const float* eprev = t >= 2 ? p.e + (r - B) * De : nullptr;
        load_cat(xr, p.qcur + r * Dp, Dp, eprev, De, lane);
        for (int uu = 0; uu < ne; ++uu) {
          const Gate4 a = gate_dots(xr, We + uu * 3 * Ke, Ke, Dp, lane);
          if (lane == 0) {
            const int u = e0 + uu;
            const float* b6 = be + uu * 6;
            const float rg = drnn_sigmoid((a.r + b6[0]) + b6[3]);
            const float zg = drnn_sigmoid((a.z + b6[1]) + b6[4]);
            const float hn = a.nh + b6[5];
            const float n = tanhf(a.nx + b6[2] + rg * hn);
            const float hp = eprev ? __ldcg(eprev + u) : 0.f;
            const float h = (1.f - zg) * n + zg * hp;
            p.e[r * De + u] = h * drnn_keep(p.se, r * De + u, p.p, p.scale);
            float* gt = p.ge + r * 4 * De;
            gt[u] = rg; gt[De + u] = zg; gt[2 * De + u] = n; gt[3 * De + u] = hn;
          }
        }
      }
    }
    if (t == p.L) break;
    grid.sync();
    // ---------------- phase B: party cell of the speaker, q_t[s] = q_{t-1}[s] (1 - m) + m q~
    if (np > 0) {
      for (int b = warp; b < B; b += RNW) {
        const long long r = (long long)t * B + b;
        int s; float m;
        drnn_speaker(p.qmask + r * p.P, p.P, s, m);
        const float* qp = p.qprev + r * Dp;
        load_cat(xr, p.c + r * Dg, Dg, qp, Dp, lane);
        const float* pr = p.pre + r * p.ldpre + 3 * Dg;
        for (int uu = 0; uu < np; ++uu) {
          const Gate4 a = gate_dots(xr, Wp + uu * 3 * Kp, Kp, Dg, lane);
          if (lane == 0) {
            const int u = p0 + uu;
            const float* b3 = bp + uu * 3;
            const float rg = drnn_sigmoid(__ldg(pr + u) + a.r + b3[0]);
            const float zg = drnn_sigmoid(__ldg(pr + Dp + u) + a.z + b3[1]);
            const float hn = a.nh + b3[2];
            const float n = tanhf(__ldg(pr + 2 * Dp + u) + a.nx + rg * hn);
            const float hp = __ldcg(qp + u);
            const float qt = ((1.f - zg) * n + zg * hp) * drnn_keep(p.sq, r * Dp + u, p.p, p.scale);
            const float qc = hp * (1.f - m) + qt * m;
            p.qcur[r * Dp + u] = qc;
            p.qstate[((long long)b * p.P + s) * Dp + u] = qc;
            float* gt = p.gp + r * 4 * Dp;
            gt[u] = rg; gt[Dp + u] = zg; gt[2 * Dp + u] = n; gt[3 * Dp + u] = hn;
          }
        }
      }
    }
    grid.sync();
  }
}

// GRU backward of one unit: dh = gradient w.r.t. the cell output h = (1-z) n + z hp; gates (r, z, n, hn).
// dx = (dr, dz, dn) w.r.t. the input-side pre-activations, dhh = (dr, dz, r dn) w.r.t. W_hh h + b_hh; returns z dh.
__device__ __forceinline__ float gru_unit_bwd(float dh, const float* gt, int D, int u, float hp, float* dx, long long ldx,
                                              float* dhh) {
  const float rg = __ldcg(gt + u), zg = __ldcg(gt + D + u), n = __ldcg(gt + 2 * D + u), hn = __ldcg(gt + 3 * D + u);
  const float dn = dh * (1.f - zg) * (1.f - n * n);
  const float dz = dh * (hp - n) * zg * (1.f - zg);
  const float dr = dn * hn * rg * (1.f - rg);
  dx[u] = dr; dx[ldx + u] = dz; dx[2 * ldx + u] = dn;
  dhh[u] = dr; dhh[D + u] = dz; dhh[2 * D + u] = dn * rg;
  return dh * zg;
}

__global__ void __launch_bounds__(RT, 1) drnn_bwd_kernel(DrnnParams p) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ float4 drnn_smem4[];
  float* sm = reinterpret_cast<float*>(drnn_smem4);
  const int Dg = p.Dg, Dp = p.Dp, De = p.De, B = p.B;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int g0, ng, p0, np, e0, ne;
  unit_range(Dg, g0, ng); unit_range(Dp, p0, np); unit_range(De, e0, ne);
  const int Tg = 3 * Dp + 3 * Dg, Tp = 3 * De + 3 * Dp + 3 * Dg, Te = 3 * De;
  float* Cg = sm;                          // [ng][Tg]  column u of W_ih^p[:, Dm:] (3Dp) | of W_hh^g (3Dg)
  float* Cp = Cg + ng * Tg;                // [np][Tp]  column u of W_ih^e (3De) | W_hh^p (3Dp) | W_ih^g[:, Dm:] (3Dg)
  float* Ce = Cp + np * Tp;                // [ne][Te]  column u of W_hh^e
  for (int i = tid; i < ng * Tg; i += RT) {
    const int uu = i / Tg, k = i % Tg, u = g0 + uu;
    Cg[i] = k < 3 * Dp ? p.Wpc[(long long)k * Dg + u] : p.Whh_g[(long long)(k - 3 * Dp) * Dg + u];
  }
  for (int i = tid; i < np * Tp; i += RT) {
    const int uu = i / Tp, k = i % Tp, u = p0 + uu;
    Cp[i] = k < 3 * De ? p.Wih_e[(long long)k * Dp + u]
          : k < 3 * De + 3 * Dp ? p.Whh_p[(long long)(k - 3 * De) * Dp + u] : p.Wgq[(long long)(k - 3 * De - 3 * Dp) * Dp + u];
  }
  for (int i = tid; i < ne * Te; i += RT) Ce[i] = p.Whh_e[(long long)(i % Te) * De + e0 + i / Te];
  __syncthreads();
  const long long LB = (long long)p.L * B;
  {
    const long long nth = (long long)gridDim.x * RT, i0 = (long long)blockIdx.x * RT + tid;
    for (long long i = i0; i < LB * Dg; i += nth) p.dG[i] = 0.f;
  }
  for (long long i = tid; i < (long long)B * p.P * np; i += RT) p.dQ[(i / np) * Dp + p0 + i % np] = 0.f;
  // e cell of the last step
  for (int i = tid; i < B * ne; i += RT) {
    const int b = i / ne, u = e0 + i % ne;
    const long long r = (long long)(p.L - 1) * B + b;
    const float dh = __ldg(p.de + r * De + u) * drnn_keep(p.se, r * De + u, p.p, p.scale);
    const float hp = p.L >= 2 ? p.e[(r - B) * De + u] : 0.f;
    p.dEh[(long long)b * De + u] = gru_unit_bwd(dh, p.ge + r * 4 * De, De, u, hp, p.dei + r * 3 * De, De, p.deh + r * 3 * De);
  }
  grid.sync();

  for (int t = p.L - 1; t >= 0; --t) {
    // ---------------- P2: party-cell gates of step t, e-cell gates of step t-1, g-cell gates of step t (own units)
    for (int b = warp; b < B; b += RNW) {
      const long long r = (long long)t * B + b;
      if (np > 0) {
        int s; float m;
        drnn_speaker(p.qmask + r * p.P, p.P, s, m);
        float* dq = p.dQ + ((long long)b * p.P + s) * Dp;
        for (int uu = 0; uu < np; ++uu) {
          const float v = col_dot(Cp + uu * Tp, p.dei + r * 3 * De, 3 * De, lane);
          if (lane == 0) {
            const int u = p0 + uu;
            const float dqc = __ldcg(dq + u) + v;                                       // d q_t[s]
            const float dqt = dqc * m * drnn_keep(p.sq, r * Dp + u, p.p, p.scale);
            const float hp = __ldcg(p.qprev + r * Dp + u);
            const float dz = gru_unit_bwd(dqt, p.gp + r * 4 * Dp, Dp, u, hp, p.dpre + r * p.lddpre + 3 * Dg, Dp, p.dph + r * 3 * Dp);
            dq[u] = dqc * (1.f - m) + dz;                                      // d q_{t-1}[s] so far
          }
        }
      }
      if (t >= 1) {
        const long long rr = r - B;
        for (int uu = 0; uu < ne; ++uu) {
          const float v = col_dot(Ce + uu * Te, p.deh + r * 3 * De, 3 * De, lane);
          if (lane == 0) {
            const int u = e0 + uu;
            float* dEh = p.dEh + (long long)b * De + u;
            const float dh = (__ldg(p.de + rr * De + u) + __ldcg(dEh) + v) * drnn_keep(p.se, rr * De + u, p.p, p.scale);
            const float hp = t >= 2 ? __ldcg(p.e + (rr - B) * De + u) : 0.f;
            *dEh = gru_unit_bwd(dh, p.ge + rr * 4 * De, De, u, hp, p.dei + rr * 3 * De, De, p.deh + rr * 3 * De);
          }
        }
      }
      for (int i = lane; i < ng; i += 32) {
        const int u = g0 + i;
        const float dh = __ldcg(p.dG + r * Dg + u) * drnn_keep(p.sg, r * Dg + u, p.p, p.scale);
        const float hp = t >= 1 ? __ldcg(p.g + (r - B) * Dg + u) : 0.f;
        const float dz = gru_unit_bwd(dh, p.gg + r * 4 * Dg, Dg, u, hp, p.dpre + r * p.lddpre, Dg, p.dgh + r * 3 * Dg);
        if (t >= 1) p.dG[(r - B) * Dg + u] = __ldcg(p.dG + (r - B) * Dg + u) + dz;
      }
    }
    grid.sync();
    // ---------------- P3: dc_t = W_ih^p[:, Dm:]^T dpi, dG_{t-1} += W_hh^g^T dgh, d q_{t-1}[s] += W_hh^p^T dph + W_ih^g[:, Dm:]^T dgi
    for (int b = warp; b < B; b += RNW) {
      const long long r = (long long)t * B + b;
      const float* drow = p.dpre + r * p.lddpre;
      for (int uu = 0; uu < ng; ++uu) {
        const int u = g0 + uu;
        const float vc = col_dot(Cg + uu * Tg, drow + 3 * Dg, 3 * Dp, lane);
        if (lane == 0) p.dc[(long long)b * Dg + u] = vc;
        if (t >= 1) {
          const float vh = col_dot(Cg + uu * Tg + 3 * Dp, p.dgh + r * 3 * Dg, 3 * Dg, lane);
          if (lane == 0) p.dG[(r - B) * Dg + u] = __ldcg(p.dG + (r - B) * Dg + u) + vh;
        }
      }
      if (np > 0) {
        int s; float m;
        drnn_speaker(p.qmask + r * p.P, p.P, s, m);
        float* dq = p.dQ + ((long long)b * p.P + s) * Dp;
        for (int uu = 0; uu < np; ++uu) {
          const float v1 = col_dot(Cp + uu * Tp + 3 * De, p.dph + r * 3 * Dp, 3 * Dp, lane);
          const float v2 = col_dot(Cp + uu * Tp + 3 * De + 3 * Dp, drow, 3 * Dg, lane);
          if (lane == 0) dq[p0 + uu] = __ldcg(dq + p0 + uu) + (v1 + v2);
        }
      }
    }
    grid.sync();
    // ---------------- P4: attention backward of step t (owner warp of each dialogue)
    for (int b = warp; b < B; b += RNW) {
      if ((b % (int)gridDim.x) != (int)blockIdx.x) continue;
      const long long r = (long long)t * B + b;
      float acc[RQC];
#pragma unroll
      for (int c = 0; c < RQC; ++c) acc[c] = 0.f;
      if (t > 0) {
        const float* xq = p.xq + r * p.ldxq;
        float q[RQC], dcr[RQC];
#pragma unroll
        for (int c = 0; c < RQC; ++c) {
          const int k = lane + 32 * c;
          q[c] = k < Dg ? __ldg(xq + k) : 0.f;
          dcr[c] = k < Dg ? __ldcg(p.dc + (long long)b * Dg + k) : 0.f;
        }
        const float* al = alpha_block(p, t, b);
        float tot = 0.f;
        for (int j0 = 0; j0 < t; j0 += RJ) {
          float part[RJ];
          hist_dots(part, dcr, p.g, B, b, Dg, j0, t, lane);
#pragma unroll
          for (int u = 0; u < RJ; ++u)
            if (j0 + u < t) tot = fmaf(__ldcg(al + j0 + u), warp_sum(part[u]), tot);
        }
        for (int j0 = 0; j0 < t; j0 += RJ) {
          float part[RJ];
          hist_dots(part, dcr, p.g, B, b, Dg, j0, t, lane);
#pragma unroll
          for (int u = 0; u < RJ; ++u) {
            const int j = j0 + u;
            if (j < t) {
              const float a = __ldcg(al + j);
              const float da = a * (warp_sum(part[u]) - tot);
              const long long jr = (long long)j * B + b;
              const float* gj = p.g + jr * Dg;
              float* dgj = p.dG + jr * Dg;
#pragma unroll
              for (int c = 0; c < RQC; ++c) {
                const int k = lane + 32 * c;
                if (k < Dg) {
                  dgj[k] = __ldcg(dgj + k) + (a * dcr[c] + da * q[c]);
                  acc[c] = fmaf(da, __ldcg(gj + k), acc[c]);
                }
              }
            }
          }
        }
      }
#pragma unroll
      for (int c = 0; c < RQC; ++c) { const int k = lane + 32 * c; if (k < Dg) p.dxq[r * p.lddxq + k] = acc[c]; }
    }
    grid.sync();
  }
}

static int drnn_grid(const ercg_dialogue_rnn* a) {
  int G = device_sm_count();
  const int dmax = a->Dg > a->Dp ? (a->Dg > a->De ? a->Dg : a->De) : (a->Dp > a->De ? a->Dp : a->De);
  return G < dmax ? G : dmax;
}
static int cdiv(int a, int b) { return (a + b - 1) / b; }
static size_t drnn_fwd_smem(const ercg_dialogue_rnn* a, int G) {
  const int ug = cdiv(a->Dg, G), up = cdiv(a->Dp, G), ue = cdiv(a->De, G);
  return sizeof(float) * ((size_t)ug * 3 * (a->Dp + a->Dg) + (size_t)up * 3 * (a->Dg + a->Dp) + (size_t)ue * 3 * (a->Dp + a->De) +
                          3 * ug + 3 * up + 6 * ue);
}
static size_t drnn_bwd_smem(const ercg_dialogue_rnn* a, int G) {
  const int ug = cdiv(a->Dg, G), up = cdiv(a->Dp, G), ue = cdiv(a->De, G);
  return sizeof(float) * ((size_t)ug * 3 * (a->Dp + a->Dg) + (size_t)up * 3 * (a->De + a->Dp + a->Dg) + (size_t)ue * 3 * a->De);
}

static int drnn_check(const ercg_dialogue_rnn* a, int backward) {
  if (!a || a->L < 0 || a->B < 0) return ERCG_EINVAL;
  if (a->Dg < 1 || a->Dg > RNN_MAXD || a->Dp < 1 || a->Dp > RNN_MAXD || a->De < 1 || a->De > RNN_MAXD) return ERCG_EINVAL;
  if (a->P < 1 || a->P > RNN_MAXP || !(a->drop_p >= 0.f && a->drop_p < 1.f)) return ERCG_EINVAL;
  if (a->L == 0 || a->B == 0) return ERCG_OK;
  if (a->ldpre < 3LL * (a->Dg + a->Dp) || a->ldxq < 0) return ERCG_EINVAL;
  const void* need[] = {a->qmask, a->pre, a->xq, a->Wgq, a->Whh_g, a->bhh_g, a->Wpc, a->Whh_p, a->bhh_p, a->Wih_e, a->Whh_e,
                        a->bih_e, a->bhh_e, a->e, a->g, a->c, a->qprev, a->qcur, a->gates_g, a->gates_p, a->gates_e, a->qstate};
  for (const void* q : need) if (!q) return ERCG_EINVAL;
  if (a->L > 1 && !a->alpha) return ERCG_EINVAL;
  if (backward) {
    const void* bneed[] = {a->de, a->dpre, a->dxq, a->dgh, a->dph, a->dei, a->deh, a->dG, a->dQ, a->dEh, a->dc};
    for (const void* q : bneed) if (!q) return ERCG_EINVAL;
    if (a->lddpre < 3LL * (a->Dg + a->Dp) || a->lddxq < a->Dg) return ERCG_EINVAL;
  }
  return 1;
}

static DrnnParams drnn_params(const ercg_dialogue_rnn* a) {
  DrnnParams p;
  p.L = a->L; p.B = a->B; p.Dg = a->Dg; p.Dp = a->Dp; p.De = a->De; p.P = a->P;
  p.p = a->drop_p; p.scale = 1.0f / (1.0f - a->drop_p);
  p.sg = a->seed_g; p.sq = a->seed_q; p.se = a->seed_e;
  p.qmask = a->qmask; p.pre = a->pre; p.ldpre = a->ldpre; p.xq = a->xq; p.ldxq = a->ldxq;
  p.Wgq = a->Wgq; p.Whh_g = a->Whh_g; p.bhh_g = a->bhh_g; p.Wpc = a->Wpc; p.Whh_p = a->Whh_p; p.bhh_p = a->bhh_p;
  p.Wih_e = a->Wih_e; p.Whh_e = a->Whh_e; p.bih_e = a->bih_e; p.bhh_e = a->bhh_e;
  p.e = a->e; p.g = a->g; p.c = a->c; p.qprev = a->qprev; p.qcur = a->qcur; p.gg = a->gates_g; p.gp = a->gates_p;
  p.ge = a->gates_e; p.alpha = a->alpha; p.qstate = a->qstate;
  p.de = a->de; p.dpre = a->dpre; p.lddpre = a->lddpre; p.dxq = a->dxq; p.lddxq = a->lddxq; p.dgh = a->dgh; p.dph = a->dph; p.dei = a->dei;
  p.deh = a->deh; p.dG = a->dG; p.dQ = a->dQ; p.dEh = a->dEh; p.dc = a->dc;
  return p;
}

// CTAs of K resident per SM are asked at the largest shared memory it may use, so the answer is a lower bound for every
// size; set up and queried once per device (not per call, which may be inside a CUDA-graph capture).  The grid has at most
// one CTA per SM, so one resident CTA per SM makes it co-schedulable.
template <auto K>
static int drnn_launch(const ercg_dialogue_rnn* a, size_t smem, int G, void* stream) {
  if (smem > (size_t)kMaxSmemPerBlock) return ERCG_ERANGE;
  if (resident_capacity<K>(RT, kMaxSmemPerBlock) < 1) return ERCG_ECUDA;
  return launch_cooperative(K, G, RT, smem, (cudaStream_t)stream, drnn_params(a));
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_dialogue_rnn_fwd(const ercg_dialogue_rnn* args, void* stream) {
  const int rc = drnn_check(args, 0);
  if (rc <= 0) return rc;
  const int G = drnn_grid(args);
  return drnn_launch<drnn_fwd_kernel>(args, drnn_fwd_smem(args, G), G, stream);
}

extern "C" int ercg_dialogue_rnn_bwd(const ercg_dialogue_rnn* args, void* stream) {
  const int rc = drnn_check(args, 1);
  if (rc <= 0) return rc;
  const int G = drnn_grid(args);
  return drnn_launch<drnn_bwd_kernel>(args, drnn_bwd_smem(args, G), G, stream);
}
