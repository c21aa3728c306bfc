// K9 / K10: DAG-ERC (track_mm/dagerc.py:73-198, track_mm/dagerc_models.py:312-365) on packed dialogues.
//
// The reference walks every dialogue utterance by utterance in Python; per step and layer it launches ~40 small
// kernels (GAT over the growing prefix, two GRUCells) and re-applies Wr0 / Wr1 to the WHOLE prefix.  Here:
//
//  K9  dag_build   predecessor structure of get_adj_v1 (dagerc.py:109-129) in closed form: the predecessors of
//                  utterance i are the contiguous range [lo_i, i-1], lo_i = the windowp-th latest j < i with the
//                  same speaker (0 if there are fewer); get_s_mask (:131-154) is spk_i == spk_j on the fly.
//                  Integer kernel; dense adj / s_mask in the reference layout are emitted only on request.
//  K10 dag_layer   one persistent cooperative kernel per GNN layer.  Facts used:
//                  * softmax_j(w.[Q;K_j] + b - mask) does not depend on w_q.Q + b (constant over j), so the
//                    attention needs only a_j = w_k.H1_j, one scalar per utterance, computed when H1_j appears;
//                  * sum_j alpha_j (s_j Wr0 + (1-s_j) Wr1) H1_j = Wr0 S0 + Wr1 S1 with S0/S1 the alpha-weighted
//                    sums over same-/other-speaker predecessors: two mat-vecs per step instead of 2 i;
//                  * the GRU terms that depend only on H[l] (W_ih^c h, W_hh^p h) are hoisted into ONE GEMM over
//                    all utterances (K2) before the kernel: pre[N, 6D].
//                  What remains sequential per step is M = [Wr0|Wr1] S (2D -> D) and [W_hh^c; W_ih^p] M
//                  (D -> 6D).  Those weights (2.9 MB for D = 300) stay resident in shared memory, sliced by
//                  hidden unit across the CTAs of the grid; a step is two grid-wide phases (grid.sync between).
//                  Backward runs the same structure in reverse time (three phases per step) and emits the
//                  per-utterance pre-activation gradients; every weight gradient is then one TN GEMM (K2).
// All per-step sums have a fixed order => bit-reproducible.  No atomics.
#include <cooperative_groups.h>
#include "common.cuh"
namespace cg = cooperative_groups;

namespace ercg {

constexpr int DT = 256, DNW = DT / 32;
constexpr int DMAXCH = 4;        // float4 chunks per lane => D <= 512
constexpr int DB_F = 16;         // dialogues staged per chunk, forward
constexpr int DB_B = 8;          // backward (6D floats each)

struct DagParams {
  int B, D, Tmax, UN;
  const int* node_off; const int* order; const int* spk; const int* lo; const long long* eoff;
  const float* wk; const float* Wr0; const float* Wr1; const float* Whh_c; const float* bhh_c;
  const float* Wih_p; const float* bih_p;
  const float* Hin; const float* pre;
  float* H1; float* a; float* S; float* M; float* alpha; float* gc; float* hnc; float* gp;
  // backward only
  float* dH1; float* dpre; float* dGseq; float* dM; float* dS; float* dHdir; float* ga;
};

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ int dlg_len(const DagParams& p, int d) { return p.node_off[d + 1] - p.node_off[d]; }

// dot of two smem vectors of `n4` float4 chunks, lane-strided
__device__ __forceinline__ float sm_dot(const float* a, const float* b, int n4, int lane) {
  float s = 0.f;
  for (int c = lane; c < n4; c += 32) s += dot4(*reinterpret_cast<const float4*>(a + 4 * c), *reinterpret_cast<const float4*>(b + 4 * c));
  return s;
}

__global__ void __launch_bounds__(DT, 1) dag_fwd_kernel(DagParams p) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ float4 dag_smem4[];
  float* sm = reinterpret_cast<float*>(dag_smem4);
  const int D = p.D, nch = D >> 2, UN = p.UN;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int u0 = blockIdx.x * UN;
  const int un = min(UN, D - u0);
  float* WA = sm;                        // [UN][2D]   rows u of Wr0 | Wr1
  float* WB = WA + UN * 2 * D;           // [UN][6][D] rows (r,z,n) of W_hh^c and W_ih^p
  float* bB = WB + UN * 6 * D;           // [UN][8]
  float* wk = bB + UN * 8;               // [D]
  float* X = wk + D;                     // [DB_F][2D]
  for (int idx = tid; idx < un * 2 * D; idx += DT) {
    const int uu = idx / (2 * D), k = idx % (2 * D);
    WA[idx] = k < D ? p.Wr0[(long long)(u0 + uu) * D + k] : p.Wr1[(long long)(u0 + uu) * D + k - D];
  }
  for (int idx = tid; idx < un * 6 * D; idx += DT) {
    const int uu = idx / (6 * D), g = (idx / D) % 6, k = idx % D;
    const float* W = g < 3 ? p.Whh_c : p.Wih_p;
    WB[idx] = W[((long long)(g % 3) * D + u0 + uu) * D + k];
  }
  for (int idx = tid; idx < un * 6; idx += DT) {
    const int uu = idx / 6, g = idx % 6;
    bB[uu * 8 + g] = (g < 3 ? p.bhh_c : p.bih_p)[(g % 3) * D + u0 + uu];
  }
  for (int k = tid; k < D; k += DT) wk[k] = p.wk[k];
  __syncthreads();

  int nact = p.B;
  for (int i = 0; i < p.Tmax; ++i) {
    while (nact > 0 && dlg_len(p, p.order[nact - 1]) <= i) --nact;
    // ---------------- phase A: attention over the predecessor range, S0/S1, M = Wr0 S0 + Wr1 S1 (own units)
    for (int c0 = 0; c0 < nact; c0 += DB_F) {
      const int cn = min(DB_F, nact - c0);
      for (int bi = warp; bi < cn; bi += DNW) {
        const int d = p.order[c0 + bi];
        const int off = p.node_off[d];
        const long long n = off + i;
        const bool owner = (d % (int)gridDim.x) == (int)blockIdx.x;
        float4 s0[DMAXCH], s1[DMAXCH];
#pragma unroll
        for (int c = 0; c < DMAXCH; ++c) s0[c] = s1[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i > 0) {
          float part = 0.f;
#pragma unroll
          for (int c = 0; c < DMAXCH; ++c) {
            const int ch = lane + 32 * c;
            if (ch < nch) part += dot4(*reinterpret_cast<const float4*>(wk + 4 * ch), ldcg4(p.H1 + (n - 1) * D + 4 * ch));
          }
          const float an = warp_sum(part);                    // a_{i-1} = w_k . H1_{i-1}
          if (owner && lane == 0) p.a[n - 1] = an;
          const int lo = p.lo[n];
          float mx = an;
          for (int j = lo + lane; j < i - 1; j += 32) mx = fmaxf(mx, __ldcg(p.a + off + j));
          mx = warp_max(mx);
          float z = 0.f;
          for (int j = lo + lane; j < i - 1; j += 32) z += expf(__ldcg(p.a + off + j) - mx);
          z = warp_sum(z) + expf(an - mx);
          const int si = p.spk[n];
          const long long eo = p.eoff[n];
          for (int j = lo; j < i; ++j) {
            const float aj = (j == i - 1) ? an : __ldcg(p.a + off + j);
            const float al = expf(aj - mx) / z;
            if (owner && lane == 0) p.alpha[eo + j - lo] = al;
            const bool same = p.spk[off + j] == si;
            const float* row = p.H1 + (long long)(off + j) * D;
#pragma unroll
            for (int c = 0; c < DMAXCH; ++c) {
              const int ch = lane + 32 * c;
              if (ch < nch) {
                const float4 v = ldcg4(row + 4 * ch);
                if (same) fma4(s0[c], al, v); else fma4(s1[c], al, v);
              }
            }
          }
        }
#pragma unroll
        for (int c = 0; c < DMAXCH; ++c) {
          const int ch = lane + 32 * c;
          if (ch < nch) {
            *reinterpret_cast<float4*>(X + bi * 2 * D + 4 * ch) = s0[c];
            *reinterpret_cast<float4*>(X + bi * 2 * D + D + 4 * ch) = s1[c];
            if (owner) { st4(p.S + n * 2 * D + 4 * ch, s0[c]); st4(p.S + n * 2 * D + D + 4 * ch, s1[c]); }
          }
        }
      }
      __syncthreads();
      for (int item = warp; item < cn * un; item += DNW) {
        const int bi = item / un, uu = item % un;
        const float v = warp_sum(sm_dot(WA + uu * 2 * D, X + bi * 2 * D, 2 * nch, lane));
        if (lane == 0) {
          const int d = p.order[c0 + bi];
          p.M[((long long)p.node_off[d] + i) * D + u0 + uu] = v;
        }
      }
      __syncthreads();
    }
    grid.sync();
    // ---------------- phase B: the two GRU cells for the own units, H1_i = C + P
    for (int c0 = 0; c0 < nact; c0 += DB_F) {
      const int cn = min(DB_F, nact - c0);
      for (int idx = tid; idx < cn * nch; idx += DT) {
        const int bi = idx / nch, ch = idx % nch;
        const int d = p.order[c0 + bi];
        *reinterpret_cast<float4*>(X + bi * 2 * D + 4 * ch) = ldcg4(p.M + ((long long)p.node_off[d] + i) * D + 4 * ch);
      }
      __syncthreads();
      for (int item = warp; item < cn * un; item += DNW) {
        const int bi = item / un, uu = item % un;
        const float* x = X + bi * 2 * D;
        const float* w = WB + uu * 6 * D;
        float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int c = lane; c < nch; c += 32) {
          const float4 xv = *reinterpret_cast<const float4*>(x + 4 * c);
#pragma unroll
          for (int g = 0; g < 6; ++g) acc[g] += dot4(*reinterpret_cast<const float4*>(w + g * D + 4 * c), xv);
        }
#pragma unroll
        for (int g = 0; g < 6; ++g) acc[g] = warp_sum(acc[g]);
        if (lane == 0) {
          const int d = p.order[c0 + bi];
          const long long n = (long long)p.node_off[d] + i;
          const int u = u0 + uu;
          const float* pr = p.pre + n * 6 * D;
          const float* b = bB + uu * 8;
          const float Mu = x[u], hu = p.Hin[n * D + u];
          // GRU c: input H[l]_i (hoisted), hidden M
          const float hn_c = acc[2] + b[2];
          const float r = sigmoidf_(pr[u] + (acc[0] + b[0]));
          const float zc = sigmoidf_(pr[D + u] + (acc[1] + b[1]));
          const float nc = tanhf(pr[2 * D + u] + r * hn_c);
          const float C = (1.f - zc) * nc + zc * Mu;
          // GRU p: input M, hidden H[l]_i (hoisted)
          const float rp = sigmoidf_((acc[3] + b[3]) + pr[3 * D + u]);
          const float zp = sigmoidf_((acc[4] + b[4]) + pr[4 * D + u]);
          const float np_ = tanhf((acc[5] + b[5]) + rp * pr[5 * D + u]);
          const float P = (1.f - zp) * np_ + zp * hu;
          p.H1[n * D + u] = C + P;
          p.gc[n * 3 * D + u] = r; p.gc[n * 3 * D + D + u] = zc; p.gc[n * 3 * D + 2 * D + u] = nc;
          p.hnc[n * D + u] = hn_c;
          p.gp[n * 3 * D + u] = rp; p.gp[n * 3 * D + D + u] = zp; p.gp[n * 3 * D + 2 * D + u] = np_;
        }
      }
      __syncthreads();
    }
    grid.sync();
  }
}

__global__ void __launch_bounds__(DT, 1) dag_bwd_kernel(DagParams p) {
  cg::grid_group grid = cg::this_grid();
  extern __shared__ float4 dag_smem4[];
  float* sm = reinterpret_cast<float*>(dag_smem4);
  const int D = p.D, nch = D >> 2, UN = p.UN;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int u0 = blockIdx.x * UN;
  const int un = min(UN, D - u0);
  float* WT2 = sm;                       // [UN][6D]  column u of [W_hh^c; W_ih^p]
  float* WT3 = WT2 + UN * 6 * D;         // [UN][2][D] column u of Wr0, Wr1
  float* wk = WT3 + UN * 2 * D;          // [D]
  float* X = wk + D;                     // [DB_B][6D]
  for (int idx = tid; idx < un * 6 * D; idx += DT) {
    const int uu = idx / (6 * D), row = idx % (6 * D);
    WT2[idx] = row < 3 * D ? p.Whh_c[(long long)row * D + u0 + uu] : p.Wih_p[(long long)(row - 3 * D) * D + u0 + uu];
  }
  for (int idx = tid; idx < un * 2 * D; idx += DT) {
    const int uu = idx / (2 * D), h = (idx / D) & 1, k = idx % D;
    WT3[idx] = (h ? p.Wr1 : p.Wr0)[(long long)k * D + u0 + uu];
  }
  for (int k = tid; k < D; k += DT) wk[k] = p.wk[k];
  __syncthreads();

  int nact = 0;
  for (int i = p.Tmax - 1; i >= 0; --i) {
    while (nact < p.B && dlg_len(p, p.order[nact]) > i) ++nact;
    // ---------------- phase 1: gate gradients of both GRU cells for the own units (elementwise)
    for (int item = tid; item < nact * un; item += DT) {
      const int bi = item / un, uu = item % un;
      const int d = p.order[bi];
      const long long n = (long long)p.node_off[d] + i;
      const int u = u0 + uu;
      const float dH = __ldcg(p.dH1 + n * D + u);
      const float* pr = p.pre + n * 6 * D;
      const float r = p.gc[n * 3 * D + u], zc = p.gc[n * 3 * D + D + u], nc = p.gc[n * 3 * D + 2 * D + u];
      const float hn_c = p.hnc[n * D + u], Mu = p.M[n * D + u];
      const float rp = p.gp[n * 3 * D + u], zp = p.gp[n * 3 * D + D + u], np_ = p.gp[n * 3 * D + 2 * D + u];
      const float hn_p = pr[5 * D + u], hu = p.Hin[n * D + u];
      // C = (1-z) n + z M
      const float dnpre = dH * (1.f - zc) * (1.f - nc * nc);
      const float dzpre = dH * (Mu - nc) * zc * (1.f - zc);
      const float drpre = dnpre * hn_c * r * (1.f - r);
      float* dp = p.dpre + n * 6 * D;
      float* dg = p.dGseq + n * 6 * D;
      dp[u] = drpre; dp[D + u] = dzpre; dp[2 * D + u] = dnpre;             // d(W_ih^c h + b_ih^c)
      dg[u] = drpre; dg[D + u] = dzpre; dg[2 * D + u] = dnpre * r;         // d(W_hh^c M + b_hh^c)
      // P = (1-z') n' + z' h
      const float dnpre_p = dH * (1.f - zp) * (1.f - np_ * np_);
      const float dzpre_p = dH * (hu - np_) * zp * (1.f - zp);
      const float drpre_p = dnpre_p * hn_p * rp * (1.f - rp);
      dg[3 * D + u] = drpre_p; dg[4 * D + u] = dzpre_p; dg[5 * D + u] = dnpre_p;        // d(W_ih^p M + b_ih^p)
      dp[3 * D + u] = drpre_p; dp[4 * D + u] = dzpre_p; dp[5 * D + u] = dnpre_p * rp;   // d(W_hh^p h + b_hh^p)
      p.dM[n * D + u] = dH * zc;           // direct term; phase 2 adds the mat-vec part
      p.dHdir[n * D + u] = dH * zp;
    }
    grid.sync();
    // ---------------- phase 2: dM[u] += sum_rows dGseq[row] * [W_hh^c; W_ih^p][row][u]
    for (int c0 = 0; c0 < nact; c0 += DB_B) {
      const int cn = min(DB_B, nact - c0);
      for (int idx = tid; idx < cn * 6 * nch; idx += DT) {
        const int bi = idx / (6 * nch), ch = idx % (6 * nch);
        const int d = p.order[c0 + bi];
        *reinterpret_cast<float4*>(X + bi * 6 * D + 4 * ch) = ldcg4(p.dGseq + ((long long)p.node_off[d] + i) * 6 * D + 4 * ch);
      }
      __syncthreads();
      for (int item = warp; item < cn * un; item += DNW) {
        const int bi = item / un, uu = item % un;
        const float v = warp_sum(sm_dot(WT2 + uu * 6 * D, X + bi * 6 * D, 6 * nch, lane));
        if (lane == 0) {
          const int d = p.order[c0 + bi];
          float* q = p.dM + ((long long)p.node_off[d] + i) * D + u0 + uu;
          *q = __ldcg(q) + v;
        }
      }
      __syncthreads();
    }
    grid.sync();
    // ---------------- phase 3: dS0[u] = sum_k Wr0[k][u] dM[k], dS1[u] likewise (own units)
    if (i > 0) {
      for (int c0 = 0; c0 < nact; c0 += DB_B) {
        const int cn = min(DB_B, nact - c0);
        for (int idx = tid; idx < cn * nch; idx += DT) {
          const int bi = idx / nch, ch = idx % nch;
          const int d = p.order[c0 + bi];
          *reinterpret_cast<float4*>(X + bi * 6 * D + 4 * ch) = ldcg4(p.dM + ((long long)p.node_off[d] + i) * D + 4 * ch);
        }
        __syncthreads();
        for (int item = warp; item < cn * un * 2; item += DNW) {
          const int bi = item / (un * 2), uu = (item >> 1) % un, h = item & 1;
          const float v = warp_sum(sm_dot(WT3 + (uu * 2 + h) * D, X + bi * 6 * D, nch, lane));
          if (lane == 0) {
            const int d = p.order[c0 + bi];
            p.dS[((long long)p.node_off[d] + i) * 2 * D + h * D + u0 + uu] = v;
          }
        }
        __syncthreads();
      }
    }
    grid.sync();
    // ---------------- phase 4: through the weighted sums and the softmax back to the predecessors (own columns)
    if (i > 0) {
      for (int bi = warp; bi < nact; bi += DNW) {
        const int d = p.order[bi];
        const int off = p.node_off[d];
        const long long n = off + i;
        const bool owner = (d % (int)gridDim.x) == (int)blockIdx.x;
        const int lo = p.lo[n], si = p.spk[n];
        const long long eo = p.eoff[n];
        float4 g0[DMAXCH], g1[DMAXCH];
#pragma unroll
        for (int c = 0; c < DMAXCH; ++c) {
          const int ch = lane + 32 * c;
          g0[c] = g1[c] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ch < nch) { g0[c] = ldcg4(p.dS + n * 2 * D + 4 * ch); g1[c] = ldcg4(p.dS + n * 2 * D + D + 4 * ch); }
        }
        auto dalpha = [&](int j) {
          const bool same = p.spk[off + j] == si;
          const float* row = p.H1 + (long long)(off + j) * D;
          float part = 0.f;
#pragma unroll
          for (int c = 0; c < DMAXCH; ++c) {
            const int ch = lane + 32 * c;
            if (ch < nch) part += dot4(same ? g0[c] : g1[c], ld4(row + 4 * ch));
          }
          return warp_sum(part);
        };
        float tot = 0.f;
        for (int j = lo; j < i; ++j) tot += p.alpha[eo + j - lo] * dalpha(j);
        for (int j = lo; j < i; ++j) {
          const float al = p.alpha[eo + j - lo];
          const float da = al * (dalpha(j) - tot);
          const bool same = p.spk[off + j] == si;
          if (lane < un) {
            const int u = u0 + lane;
            float* dst = p.dH1 + (long long)(off + j) * D + u;
            const float ds = __ldcg(p.dS + n * 2 * D + (same ? 0 : D) + u);
            *dst = __ldcg(dst) + (al * ds + da * wk[u]);
          }
          if (owner && lane == 0) p.ga[off + j] += da;
        }
      }
    }
    __syncthreads();   // phase 1 of step i-1 reads the dH1 columns this CTA has just updated
  }
}

// ---------------------------------------------------------------------------------------------- K9
__global__ void dag_lo_kernel(const int* __restrict__ node_off, const int* __restrict__ node_dlg,
                              const int* __restrict__ spk, long long N, int windowp, int* __restrict__ lo,
                              int* __restrict__ cnt) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int off = node_off[node_dlg[n]];
  const int i = (int)(n - off), s = spk[n];
  int j = i - 1, c = 0, first = 0;
  for (; j >= 0; --j) {
    if (spk[off + j] == s && ++c == windowp) { first = j; break; }
  }
  lo[n] = first;
  cnt[n] = i - first;          // i = 0 -> 0 predecessors
}

// exclusive scan of cnt over all nodes: per-block totals -> serial scan of the totals -> per-node offsets
constexpr int SCAN_T = 256, SCAN_PER = 8, SCAN_TILE = SCAN_T * SCAN_PER;
__global__ void __launch_bounds__(SCAN_T) scan_tile_sums_kernel(const int* __restrict__ cnt, long long N, long long* __restrict__ tile) {
  __shared__ long long sh[SCAN_T];
  const long long base = (long long)blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_PER;
  long long s = 0;
  for (int k = 0; k < SCAN_PER; ++k) if (base + k < N) s += cnt[base + k];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = SCAN_T / 2; o > 0; o >>= 1) { if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) tile[blockIdx.x] = sh[0];
}
__global__ void scan_tiles_serial_kernel(long long* tile, int ntiles, long long* total) {
  long long run = 0;
  for (int t = 0; t < ntiles; ++t) { const long long v = tile[t]; tile[t] = run; run += v; }
  *total = run;
}
__global__ void __launch_bounds__(SCAN_T) scan_apply_kernel(const int* __restrict__ cnt, long long N, const long long* __restrict__ tile,
                                                            long long* __restrict__ eoff) {
  __shared__ long long sh[SCAN_T];
  const long long base = (long long)blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_PER;
  long long s = 0;
  for (int k = 0; k < SCAN_PER; ++k) if (base + k < N) s += cnt[base + k];
  sh[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long run = tile[blockIdx.x];
    for (int t = 0; t < SCAN_T; ++t) { const long long v = sh[t]; sh[t] = run; run += v; }
  }
  __syncthreads();
  long long run = sh[threadIdx.x];
  for (int k = 0; k < SCAN_PER; ++k) if (base + k < N) { eoff[base + k] = run; run += cnt[base + k]; }
}

// dense reference layout: adj [B,Lmax,Lmax] fp32 (get_adj_v1), s_mask [B,Lmax,Lmax] int64 (get_s_mask), from padded ids
__global__ void dag_dense_kernel(const int* __restrict__ spk_pad, int B, int Lmax, int windowp, float* __restrict__ adj,
                                 long long* __restrict__ smask) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)B * Lmax) return;
  const int b = (int)(idx / Lmax), i = (int)(idx % Lmax);
  const int* s = spk_pad + (long long)b * Lmax;
  int first = 0, c = 0;
  for (int j = i - 1; j >= 0; --j)
    if (s[j] == s[i] && ++c == windowp) { first = j; break; }
  float* arow = adj + idx * Lmax;
  long long* srow = smask + idx * Lmax;
  for (int j = 0; j < Lmax; ++j) {
    arow[j] = (j >= first && j < i) ? 1.f : 0.f;
    srow[j] = s[j] == s[i] ? 1 : 0;
  }
}

static int dag_units(int D, int* grid_out) {
  const int num_sms = device_sm_count();
  const int UN = (D + num_sms - 1) / num_sms;
  *grid_out = (D + UN - 1) / UN;
  return UN;
}
static size_t dag_fwd_smem(int D, int UN) { return sizeof(float) * ((size_t)UN * (8 * D + 8) + D + (size_t)DB_F * 2 * D); }
static size_t dag_bwd_smem(int D, int UN) { return sizeof(float) * ((size_t)UN * 8 * D + D + (size_t)DB_B * 6 * D); }

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_dag_build(const int32_t* node_off, const int32_t* node_dlg, const int32_t* spk, int64_t N, int windowp,
                              int32_t* lo, int32_t* cnt, int64_t* eoff, int64_t* total, void* workspace,
                              size_t workspace_bytes, void* stream) {
  if (N < 0 || windowp < 1) return ERCG_EINVAL;
  if (!total) return ERCG_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) { cudaMemsetAsync(total, 0, sizeof(int64_t), st); return ERCG_OK; }
  if (!node_off || !node_dlg || !spk || !lo || !cnt || !eoff) return ERCG_EINVAL;
  const int ntiles = (int)((N + SCAN_TILE - 1) / SCAN_TILE);
  if (!workspace || workspace_bytes < (size_t)ntiles * sizeof(long long)) return ERCG_EWORKSPACE;
  long long* tile = reinterpret_cast<long long*>(workspace);
  dag_lo_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(node_off, node_dlg, spk, N, windowp, lo, cnt);
  int rc = finish_launch();
  if (rc != ERCG_OK) return rc;
  scan_tile_sums_kernel<<<ntiles, SCAN_T, 0, st>>>(cnt, N, tile);
  if ((rc = finish_launch()) != ERCG_OK) return rc;
  scan_tiles_serial_kernel<<<1, 1, 0, st>>>(tile, ntiles, reinterpret_cast<long long*>(total));
  if ((rc = finish_launch()) != ERCG_OK) return rc;
  scan_apply_kernel<<<ntiles, SCAN_T, 0, st>>>(cnt, N, tile, reinterpret_cast<long long*>(eoff));
  return finish_launch();
}

extern "C" size_t ercg_dag_build_workspace_bytes(int64_t N) {
  return N <= 0 ? 0 : (size_t)((N + SCAN_TILE - 1) / SCAN_TILE) * sizeof(long long);
}

extern "C" int ercg_dag_dense_masks(const int32_t* spk_padded, int B, int Lmax, int windowp, float* adj, int64_t* s_mask,
                                    void* stream) {
  if (B < 0 || Lmax < 0 || windowp < 1) return ERCG_EINVAL;
  if (B == 0 || Lmax == 0) return ERCG_OK;
  if (!spk_padded || !adj || !s_mask) return ERCG_EINVAL;
  const long long rows = (long long)B * Lmax;
  dag_dense_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, (cudaStream_t)stream>>>(spk_padded, B, Lmax, windowp, adj,
                                                                                   reinterpret_cast<long long*>(s_mask));
  return finish_launch();
}

static int dag_check(const ercg_dag_layer* a, int backward) {
  if (!a || a->B < 0 || a->D <= 0 || (a->D & 3) || a->D > 128 * DMAXCH || a->Tmax < 0) return ERCG_EINVAL;
  if (a->B == 0 || a->Tmax == 0) return ERCG_OK;
  const void* need[] = {a->node_off, a->order, a->spk, a->lo, a->eoff, a->wk, a->Wr0, a->Wr1, a->Whh_c, a->bhh_c, a->Wih_p,
                        a->bih_p, a->Hin, a->pre, a->H1, a->a, a->S, a->M, a->alpha, a->gc, a->hnc, a->gp};
  for (const void* q : need) if (!q) return ERCG_EINVAL;
  if (backward && (!a->dH1 || !a->dpre || !a->dGseq || !a->dM || !a->dS || !a->dHdir || !a->ga)) return ERCG_EINVAL;
  return 1;
}

static DagParams dag_params(const ercg_dag_layer* a, int UN) {
  DagParams p;
  p.B = a->B; p.D = a->D; p.Tmax = a->Tmax; p.UN = UN;
  p.node_off = a->node_off; p.order = a->order; p.spk = a->spk; p.lo = a->lo;
  p.eoff = reinterpret_cast<const long long*>(a->eoff);
  p.wk = a->wk; p.Wr0 = a->Wr0; p.Wr1 = a->Wr1; p.Whh_c = a->Whh_c; p.bhh_c = a->bhh_c; p.Wih_p = a->Wih_p; p.bih_p = a->bih_p;
  p.Hin = a->Hin; p.pre = a->pre; p.H1 = a->H1; p.a = a->a; p.S = a->S; p.M = a->M; p.alpha = a->alpha; p.gc = a->gc;
  p.hnc = a->hnc; p.gp = a->gp;
  p.dH1 = a->dH1; p.dpre = a->dpre; p.dGseq = a->dGseq; p.dM = a->dM; p.dS = a->dS; p.dHdir = a->dHdir; p.ga = a->ga;
  return p;
}

// One cooperative launch of K.  The grid has at most one CTA per SM, so one CTA of K resident per SM, asked once per device
// at the largest shared memory K may use, makes every size co-schedulable; no set-up call is made per launch, so a layer
// can be captured in a CUDA graph.
template <auto K>
static int dag_launch(const ercg_dag_layer* a, int UN, int grid, size_t smem, void* stream) {
  if (smem > (size_t)kMaxSmemPerBlock) return ERCG_ERANGE;
  if (resident_capacity<K>(DT, kMaxSmemPerBlock) < 1) return ERCG_ECUDA;
  return launch_cooperative(K, grid, DT, smem, (cudaStream_t)stream, dag_params(a, UN));
}

extern "C" int ercg_dag_layer_fwd(const ercg_dag_layer* args, void* stream) {
  int rc = dag_check(args, 0);
  if (rc <= 0) return rc;
  int grid = 0;
  const int UN = dag_units(args->D, &grid);
  return dag_launch<dag_fwd_kernel>(args, UN, grid, dag_fwd_smem(args->D, UN), stream);
}

extern "C" int ercg_dag_layer_bwd(const ercg_dag_layer* args, void* stream) {
  int rc = dag_check(args, 1);
  if (rc <= 0) return rc;
  int grid = 0;
  const int UN = dag_units(args->D, &grid);
  return dag_launch<dag_bwd_kernel>(args, UN, grid, dag_bwd_smem(args->D, UN), stream);
}
