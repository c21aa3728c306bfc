// K6c: packed bidirectional LSTM / GRU recurrence for hidden sizes 101..384 per direction, forward and backward through
// time, on thread-block clusters with distributed shared memory.
//
// K6 / K6b keep one row of W_hh per thread in registers, which stops at Hd ~ 100 (an LSTM at Hd = 128 would need 512
// threads x 128 weight registers: the whole register file).  Here W_hh is spread over the C CTAs of a cluster (C = 8, or
// 16 when a CTA's slice does not fit in shared memory at 8):
//   - CTA q owns hidden units [q*U, (q+1)*U), U = ceil(Hd / C), with ALL their gate rows, so the cell update is CTA-local;
//     units past Hd are padding with zero weights (a padded LSTM unit keeps c = h = 0, a padded GRU unit h = 0).
//   - its W_hh rows stay in shared memory for the whole launch;
//   - forward: after each step every CTA writes its new h slice into every peer's copy of h (DSMEM) and the cluster meets
//     at one barrier.cluster; h is double-buffered, so one barrier per step is enough;
//   - backward: every CTA forms its partial W_hh^T da over its rows for all Hd columns and sends each owner CTA its
//     columns; the owner adds the C partials in CTA-rank order.
// A cluster advances NB dialogues ("lanes") of one direction in lockstep, so each shared-memory weight read serves NB
// dialogues.  Lane l of a direction runs dialogues l, l + lanes, l + 2 lanes, ... back to back: a lane whose dialogue ends
// sends h = 0 (forward) or ignores the received partials (backward) and starts its next dialogue on the following step,
// so lanes of unequal length do not wait for each other.  A dialogue's arithmetic depends only on its own rows: the
// summation orders are fixed by Hd (k-chunks of the mat-vec, then CTA rank), never by the grid or the lane, so results
// are bit-identical run to run and for any number of clusters.  FFMA only, fp32.
//
// Saved tensors and outputs are exactly K6's / K6b's (see lstm.cu, gru.cu), so the TN GEMM / column sums that form dW_hh
// and db_hh are unchanged.
#include "rnn_cluster.cuh"
#include <math.h>

namespace ercg {

constexpr int RC_NB = 8;                 // lanes (dialogues) per cluster advanced in lockstep
constexpr int RC_THREADS = 512;
constexpr int RC_SMEM_LIMIT = 227 * 1024 - 1024;   // dynamic shared memory per CTA we allow (227 KB less the static part)

__device__ __forceinline__ float rc_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ uint32_t rc_smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t rc_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t rc_clusterid() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t rc_nclusters() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void rc_st_peer(uint32_t local_addr, uint32_t rank, float v) {   // local smem address -> CTA `rank`
  uint32_t a;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(local_addr), "r"(rank));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory");
}
__device__ __forceinline__ void rc_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Geometry of one launch; a pure function of (cell, Hd, direction of time), see rc_geom.
struct RcGeom {
  int Hd, C, U, Hp, RWp;   // units per CTA, padded Hd (= C*U), gate rows per CTA padded to a multiple of 4
  int KS, chunk;           // the mat-vec splits its reduction dimension into KS chunks of `chunk` (multiple of 4)
};

// out[b][col] = sum over i of M[i][col] * v[b][i] for the NB lanes, i in this thread's chunk; M row-major with `cols`
// columns, v [NB][ld_v].  Threads of a warp take consecutive columns (conflict-free M reads, broadcast v reads).
__device__ __forceinline__ void rc_matvec(const float* __restrict__ M, int cols, int nrows, const float* __restrict__ v,
                                          int ld_v, const RcGeom& g, float* __restrict__ part) {
  const int tid = threadIdx.x, col = tid % cols, ks = tid / cols;
  if (ks >= g.KS) return;
  const int i0 = ks * g.chunk, i1 = min(nrows, i0 + g.chunk);
  float acc[RC_NB];
#pragma unroll
  for (int b = 0; b < RC_NB; ++b) acc[b] = 0.f;
  for (int i = i0; i < i1; i += 4) {
    const float m0 = M[(i + 0) * cols + col], m1 = M[(i + 1) * cols + col];
    const float m2 = M[(i + 2) * cols + col], m3 = M[(i + 3) * cols + col];
#pragma unroll
    for (int b = 0; b < RC_NB; ++b) {
      const float4 x = ld4(v + b * ld_v + i);
      acc[b] = fmaf(m0, x.x, acc[b]); acc[b] = fmaf(m1, x.y, acc[b]);
      acc[b] = fmaf(m2, x.z, acc[b]); acc[b] = fmaf(m3, x.w, acc[b]);
    }
  }
#pragma unroll
  for (int b = 0; b < RC_NB; ++b) part[(ks * RC_NB + b) * cols + col] = acc[b];
}

// Number of steps the cluster runs: the longest lane (sum of the lengths of its dialogues).
__device__ __forceinline__ int rc_steps(const int* __restrict__ node_off, int B, int lane0, int lanes, int* s_tot) {
  if (threadIdx.x < RC_NB) {
    int tot = 0;
    for (int d = lane0 + threadIdx.x; d < B; d += lanes) tot += node_off[d + 1] - node_off[d];
    s_tot[threadIdx.x] = tot;
  }
  __syncthreads();
  int m = 0;
#pragma unroll
  for (int b = 0; b < RC_NB; ++b) m = max(m, s_tot[b]);
  return m;
}

// A lane's position: dialogue d (>= B: the lane is done), its first row o and length L.
struct RcLane {
  int d, o, L;
  __device__ __forceinline__ void seek(const int* __restrict__ node_off, int B, int lanes) {   // skip empty dialogues
    for (; d < B; d += lanes) {
      o = node_off[d];
      L = node_off[d + 1] - o;
      if (L > 0) return;
    }
  }
};

// CELL 0 = LSTM (gates i, f, g, o; b_hh folded into gx), 1 = GRU (r, z, n; b_hh added here).
// smem: Wt [Hp][RWp] (W_hh slice, transposed: row = k, column = gate row g*U + u) | h [2][NB][Hp] | part [KS][NB][RWp]
template <int CELL>
__global__ void __launch_bounds__(RC_THREADS, 1)
rnn_cluster_fwd_kernel(const float* __restrict__ gx, long long ldgx, const float* __restrict__ whh,
                       const float* __restrict__ bhh, const int* __restrict__ node_off, int B, float* __restrict__ out,
                       long long ldo, float* __restrict__ gates, float* __restrict__ cells, float* __restrict__ hprev,
                       RcGeom g) {
  constexpr int G = CELL == 0 ? 4 : 3;
  extern __shared__ __align__(16) float smem[];
  __shared__ int s_tot[RC_NB];
  const int Hd = g.Hd, U = g.U, Hp = g.Hp, RWp = g.RWp;
  float* Wt = smem;
  float* hb = Wt + Hp * RWp;
  float* part = hb + 2 * RC_NB * Hp;
  const int tid = threadIdx.x, q = (int)rc_ctarank(), cid = (int)rc_clusterid();
  const int dir = cid & 1, lanes = ((int)rc_nclusters() >> 1) * RC_NB, lane0 = (cid >> 1) * RC_NB;

  for (int idx = tid; idx < G * U * Hp; idx += RC_THREADS) {      // coalesced along k in global memory
    const int r = idx / Hp, k = idx % Hp, gate = r / U, j = q * U + r % U;
    Wt[k * RWp + r] = (j < Hd && k < Hd) ? whh[((long long)dir * G * Hd + gate * Hd + j) * Hd + k] : 0.f;
  }
  for (int idx = tid; idx < Hp * (RWp - G * U); idx += RC_THREADS)
    Wt[(idx / (RWp - G * U)) * RWp + G * U + idx % (RWp - G * U)] = 0.f;
  for (int idx = tid; idx < 2 * RC_NB * Hp; idx += RC_THREADS) hb[idx] = 0.f;
  const int steps = rc_steps(node_off, B, lane0, lanes, s_tot);

  // cell threads: (lane b, unit u)
  const bool cell = tid < RC_NB * U;
  const int b = tid / U, u = tid % U, j = q * U + u;
  const bool live = cell && j < Hd;
  RcLane ln{lane0 + b, 0, 0};
  if (live) ln.seek(node_off, B, lanes);
  int s = 0;
  float c = 0.f, bh[G], gxv[G];           // gxv: gx of the lane's next step, loaded one step ahead (hides its latency)
  auto load_gx = [&]() {
    const long long t = ln.o + (dir == 0 ? s : ln.L - 1 - s);
#pragma unroll
    for (int i = 0; i < G; ++i) gxv[i] = gx[t * ldgx + dir * G * Hd + i * Hd + j];
  };
  if (live && ln.d < B) load_gx();
#pragma unroll
  for (int i = 0; i < G; ++i) bh[i] = (CELL == 1 && live) ? bhh[dir * 3 * Hd + i * Hd + j] : 0.f;
  rc_cluster_sync();                       // every CTA of the cluster has started and zeroed h before any DSMEM write

  for (int it = 0; it < steps; ++it) {
    const int cur = it & 1;
    const float* h = hb + cur * RC_NB * Hp;
    rc_matvec(Wt, RWp, Hp, h, Hp, g, part);
    __syncthreads();
    if (live && ln.d < B) {
      const long long t = ln.o + (dir == 0 ? s : ln.L - 1 - s);
      float acc[G];
#pragma unroll
      for (int i = 0; i < G; ++i) {
        float a = 0.f;
        for (int ks = 0; ks < g.KS; ++ks) a += part[(ks * RC_NB + b) * RWp + i * U + u];
        acc[i] = a;
      }
      float* gt = gates + t * (8 * Hd) + dir * 4 * Hd + j;
      const float hp = h[b * Hp + j];
      float hn;
      if constexpr (CELL == 0) {
        const float ig = rc_sigmoid(gxv[0] + acc[0]), fg = rc_sigmoid(gxv[1] + acc[1]);
        const float gg = tanhf(gxv[2] + acc[2]), og = rc_sigmoid(gxv[3] + acc[3]);
        c = fmaf(fg, c, ig * gg);
        hn = og * tanhf(c);
        gt[0] = ig; gt[Hd] = fg; gt[2 * Hd] = gg; gt[3 * Hd] = og;
        cells[t * (2 * Hd) + dir * Hd + j] = c;
      } else {
        const float ar = bh[0] + acc[0], az = bh[1] + acc[1], an = bh[2] + acc[2];
        const float rg = rc_sigmoid(gxv[0] + ar), zg = rc_sigmoid(gxv[1] + az);
        const float n = tanhf(fmaf(rg, an, gxv[2]));
        hn = fmaf(zg, hp - n, n);
        gt[0] = rg; gt[Hd] = zg; gt[2 * Hd] = n; gt[3 * Hd] = an;
      }
      hprev[t * (2 * Hd) + dir * Hd + j] = hp;
      out[t * ldo + dir * Hd + j] = hn;
      const bool last = ++s == ln.L;
      const uint32_t dst = rc_smem_addr(hb + (cur ^ 1) * RC_NB * Hp + b * Hp + j);
      for (int p = 0; p < g.C; ++p) rc_st_peer(dst, p, last ? 0.f : hn);   // a finished dialogue hands its lane h = 0
      if (last) {
        s = 0;
        c = 0.f;
        ln.d += lanes;
        ln.seek(node_off, B, lanes);
      }
      if (ln.d < B) load_gx();
    }
    rc_cluster_sync();
  }
}

// smem: W [RWp][Hp] (W_hh slice, row = gate row g*U + u, column = k) | da [NB][RWp] | recv [2][C][NB][U] |
// part [KS][NB][Hp].  da holds the hidden-side pre-activation gradients (LSTM dgx, GRU dgh) of this CTA's rows.
template <int CELL>
__global__ void __launch_bounds__(RC_THREADS, 1)
rnn_cluster_bwd_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ gates,
                       const float* __restrict__ cells, const float* __restrict__ hprev, const float* __restrict__ whh,
                       const int* __restrict__ node_off, int B, float* __restrict__ dgx, long long lddgx,
                       float* __restrict__ dgh, long long lddgh, RcGeom g) {
  constexpr int G = CELL == 0 ? 4 : 3;
  extern __shared__ __align__(16) float smem[];
  __shared__ int s_tot[RC_NB];
  const int Hd = g.Hd, U = g.U, Hp = g.Hp, RWp = g.RWp, C = g.C;
  float* W = smem;
  float* da = W + RWp * Hp;
  float* recv = da + RC_NB * RWp;
  float* part = recv + 2 * C * RC_NB * U;
  const int tid = threadIdx.x, q = (int)rc_ctarank(), cid = (int)rc_clusterid();
  const int dir = cid & 1, lanes = ((int)rc_nclusters() >> 1) * RC_NB, lane0 = (cid >> 1) * RC_NB;

  for (int idx = tid; idx < RWp * Hp; idx += RC_THREADS) {
    const int r = idx / Hp, k = idx % Hp, gate = r / U, j = q * U + r % U;
    W[idx] = (r < G * U && j < Hd && k < Hd) ? whh[((long long)dir * G * Hd + gate * Hd + j) * Hd + k] : 0.f;
  }
  for (int idx = tid; idx < RC_NB * RWp + 2 * C * RC_NB * U; idx += RC_THREADS) da[idx] = 0.f;   // da and recv
  const int steps = rc_steps(node_off, B, lane0, lanes, s_tot);

  const bool cell = tid < RC_NB * U;
  const int b = tid / U, u = tid % U, j = q * U + u;
  const bool live = cell && j < Hd;
  RcLane ln{lane0 + b, 0, 0};
  if (live) ln.seek(node_off, B, lanes);
  int s = ln.L - 1;                        // steps of a dialogue run in reverse of the forward traversal
  float dh_keep = 0.f;                     // LSTM: dc of the later step times f; GRU: dh of the later step times z
  // the saved values of the lane's next step, loaded one step ahead: gates (4), dout, LSTM c and c_{t-1} / GRU h_{t-1}
  float sv[7];
  auto load_step = [&]() {
    const long long t = ln.o + (dir == 0 ? s : ln.L - 1 - s);
    const float* gt = gates + t * (8 * Hd) + dir * 4 * Hd + j;
#pragma unroll
    for (int i = 0; i < 4; ++i) sv[i] = gt[i * Hd];
    sv[4] = dout[t * ldo + dir * Hd + j];
    if (CELL == 0) {
      sv[5] = cells[t * (2 * Hd) + dir * Hd + j];
      sv[6] = 0.f;
      if (s > 0) {
        const long long tp = ln.o + (dir == 0 ? s - 1 : ln.L - s);
        sv[6] = cells[tp * (2 * Hd) + dir * Hd + j];
      }
    } else {
      sv[5] = hprev[t * (2 * Hd) + dir * Hd + j];
    }
  };
  if (live && ln.d < B) load_step();
  rc_cluster_sync();

  for (int it = 0; it < steps; ++it) {
    const int cur = it & 1;
    if (live && ln.d < B) {
      const long long t = ln.o + (dir == 0 ? s : ln.L - 1 - s);
      const bool first = s == ln.L - 1;
      float rec = 0.f;
      if (!first)
        for (int p = 0; p < C; ++p) rec += recv[((cur * C + p) * RC_NB + b) * U + u];
      float* dxt = dgx + t * lddgx + dir * G * Hd + j;
      float* sda = da + b * RWp + u;
      if (CELL == 0) {
        const float ig = sv[0], fg = sv[1], gg = sv[2], og = sv[3], cc = sv[5], cprev = sv[6];
        const float dh = sv[4] + rec;
        const float tc = tanhf(cc);
        const float dc = fmaf(dh * og, 1.f - tc * tc, first ? 0.f : dh_keep);
        const float a0 = dc * gg * ig * (1.f - ig), a1 = dc * cprev * fg * (1.f - fg);
        const float a2 = dc * ig * (1.f - gg * gg), a3 = dh * tc * og * (1.f - og);
        sda[0] = a0; sda[U] = a1; sda[2 * U] = a2; sda[3 * U] = a3;
        dxt[0] = a0; dxt[Hd] = a1; dxt[2 * Hd] = a2; dxt[3 * Hd] = a3;
        dh_keep = dc * fg;
      } else {
        const float rg = sv[0], zg = sv[1], n = sv[2], hn = sv[3], hp = sv[5];
        const float dh = sv[4] + (first ? 0.f : dh_keep + rec);
        const float dan = dh * (1.f - zg) * (1.f - n * n);
        const float a0 = dan * hn * rg * (1.f - rg), a1 = dh * (hp - n) * zg * (1.f - zg), a2 = dan * rg;
        sda[0] = a0; sda[U] = a1; sda[2 * U] = a2;
        dxt[0] = a0; dxt[Hd] = a1; dxt[2 * Hd] = dan;
        float* dht = dgh + t * lddgh + dir * 3 * Hd + j;
        dht[0] = a0; dht[Hd] = a1; dht[2 * Hd] = a2;
        dh_keep = dh * zg;
      }
      if (s-- == 0) {
        ln.d += lanes;
        ln.seek(node_off, B, lanes);
        s = ln.L - 1;
      }
      if (ln.d < B) load_step();
    }
    __syncthreads();
    rc_matvec(W, Hp, RWp, da, RWp, g, part);
    __syncthreads();
    for (int idx = tid; idx < RC_NB * Hd; idx += RC_THREADS) {       // this CTA's partial of W_hh^T da -> owner of column k
      const int bb = idx / Hd, k = idx % Hd;
      float v = 0.f;
      for (int ks = 0; ks < g.KS; ++ks) v += part[(ks * RC_NB + bb) * Hp + k];
      rc_st_peer(rc_smem_addr(recv + (((cur ^ 1) * C + q) * RC_NB + bb) * U + k % U), k / U, v);
    }
    rc_cluster_sync();
  }
}

// ---- host side
static int rc_round4(int x) { return (x + 3) & ~3; }

// Shared-memory bytes of one CTA; fills g.  bwd: the backward kernel's layout.
static size_t rc_geom(int G, int Hd, int C, bool bwd, RcGeom& g) {
  g.Hd = Hd;
  g.C = C;
  g.U = (Hd + C - 1) / C;
  g.Hp = C * g.U;
  g.RWp = rc_round4(G * g.U);
  const int cols = bwd ? g.Hp : g.RWp, nrows = bwd ? g.RWp : g.Hp;
  g.KS = RC_THREADS / cols > 0 ? RC_THREADS / cols : 1;
  g.chunk = rc_round4((nrows + g.KS - 1) / g.KS);
  const size_t fl = bwd ? (size_t)g.RWp * g.Hp + (size_t)RC_NB * g.RWp + 2ull * C * RC_NB * g.U + (size_t)g.KS * RC_NB * g.Hp
                        : (size_t)g.Hp * g.RWp + 2ull * RC_NB * g.Hp + (size_t)g.KS * RC_NB * g.RWp;
  return fl * sizeof(float);
}

// Cluster size for (cell, Hd): the portable 8 when both kernels' slices fit at 8, else 16.  Same for fwd and bwd.
static int rc_cluster_size(int G, int Hd) {
  RcGeom g;
  return rc_geom(G, Hd, 8, false, g) <= (size_t)RC_SMEM_LIMIT && rc_geom(G, Hd, 8, true, g) <= (size_t)RC_SMEM_LIMIT ? 8 : 16;
}

// Clusters of C CTAs of `kern` that can be resident at once, queried once per device (and per C) at the largest shared
// memory the kernel is allowed, so it is a lower bound for every Hd.  0: this cluster shape cannot be scheduled.
template <typename K>
static int rc_capacity(K kern, int C, std::atomic<int>* cache) {
  const int d = current_device();
  if (d >= 0 && d < kMaxDevices) {
    const int c = cache[d].load(std::memory_order_acquire);
    if (c != 0) return c > 0 ? c : 0;
  }
  int n = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, RC_SMEM_LIMIT) == cudaSuccess &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C * 2, 1, 1);
    cfg.blockDim = dim3(RC_THREADS, 1, 1);
    cfg.dynamicSmemBytes = RC_SMEM_LIMIT;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) n = 0;
  }
  if (n == 0) cudaGetLastError();
  if (d >= 0 && d < kMaxDevices) cache[d].store(n > 0 ? n : -1, std::memory_order_release);
  return n;
}

// One launch: the grid holds an even number of clusters (half per direction), at most what is resident at once and at
// most one lane per dialogue.
template <typename K, typename... Args>
static int rc_launch(K kern, std::atomic<int> (*cache)[kMaxDevices], int G, int Hd, int B, bool bwd, cudaStream_t st,
                     Args... args) {
  RcGeom g;
  const int C = rc_cluster_size(G, Hd);
  const size_t smem = rc_geom(G, Hd, C, bwd, g);
  if (smem > (size_t)RC_SMEM_LIMIT) return ERCG_EINVAL;
  const int cap = rc_capacity(kern, C, cache[C == 16]);
  if (cap < 1) return ERCG_ECUDA;
  const long long want = 2LL * ((B + RC_NB - 1) / RC_NB);
  int ncl = (int)(want < cap ? want : cap) & ~1;
  if (ncl < 2) ncl = 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ncl * C, 1, 1);
  cfg.blockDim = dim3(RC_THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, kern, args..., g) != cudaSuccess) {
    cudaGetLastError();
    return ERCG_ECUDA;
  }
  return finish_launch();
}

static std::atomic<int> g_cap_lstm_fwd[2][kMaxDevices], g_cap_lstm_bwd[2][kMaxDevices];
static std::atomic<int> g_cap_gru_fwd[2][kMaxDevices], g_cap_gru_bwd[2][kMaxDevices];

int lstm_cluster_fwd(const float* gx, long long ldgx, const float* whh, const int* node_off, int B, int Hd, float* out,
                     long long ldo, float* gates, float* cells, float* hprev, cudaStream_t st) {
  return rc_launch(rnn_cluster_fwd_kernel<0>, g_cap_lstm_fwd, 4, Hd, B, false, st, gx, ldgx, whh, (const float*)nullptr,
                   node_off, B, out, ldo, gates, cells, hprev);
}

int lstm_cluster_bwd(const float* dout, long long ldo, const float* gates, const float* cells, const float* whh,
                     const int* node_off, int B, int Hd, float* dgx, long long lddgx, cudaStream_t st) {
  return rc_launch(rnn_cluster_bwd_kernel<0>, g_cap_lstm_bwd, 4, Hd, B, true, st, dout, ldo, gates, cells,
                   (const float*)nullptr, whh, node_off, B, dgx, lddgx, (float*)nullptr, 0LL);
}

int gru_cluster_fwd(const float* gx, long long ldgx, const float* whh, const float* bhh, const int* node_off, int B, int Hd,
                    float* out, long long ldo, float* gates, float* hprev, cudaStream_t st) {
  return rc_launch(rnn_cluster_fwd_kernel<1>, g_cap_gru_fwd, 3, Hd, B, false, st, gx, ldgx, whh, bhh, node_off, B, out, ldo,
                   gates, (float*)nullptr, hprev);
}

int gru_cluster_bwd(const float* dout, long long ldo, const float* gates, const float* hprev, const float* whh,
                    const int* node_off, int B, int Hd, float* dgx, long long lddgx, float* dgh, long long lddgh,
                    cudaStream_t st) {
  return rc_launch(rnn_cluster_bwd_kernel<1>, g_cap_gru_bwd, 3, Hd, B, true, st, dout, ldo, gates, (const float*)nullptr,
                   hprev, whh, node_off, B, dgx, lddgx, dgh, lddgh);
}

}  // namespace ercg
