// K11: MaskedEdgeAttention 'attn1' of the declare-lab DialogueGCN (track_mm/dgcnv2_models.py:517-562) in closed form.
//
// Reference: scale = Linear(2D -> max_seq_len, no bias)(M)  [L, B, 110];  alpha = softmax over the SEQUENCE axis (all L padded
// positions of the dialogue, padding included) -> [B, 110, L];  mask = 1 on the edges (i -> j) of the window graph, 1e-10
// elsewhere;  scores = alpha * mask / sum_j(alpha * mask), kept on the edges only.  batch_graphify then reads
// edge_norm[i -> j] = scores[b, i, j] one element at a time (dgcnv2_models.py:670-672).
// Here: S = M @ W^T is one GEMM over the dialogue-major rows [B * Lmax, 110] (row b * Lmax + j', column i); per source node
// (b, i) one warp computes m = max_j' S, e_j' = exp(S - m), Z_all, Z_win (targets j in [max(0, i - wp), min(len - 1, i + wf)]) and
//     nu[i -> j] = e_j / (Z_win + 1e-10 * (Z_all - Z_win))
// written straight into the packed by-destination edge order.  The dense [B, 110, L] tensors are never materialised.
// Backward: G = sum_{j in win} dnu_j nu_j;  dS[j', i] = [j' in win] dnu_j' nu_j' - c_j' e_j' / Den * G,  c = 1 (win) | 1e-10.
#include "common.cuh"
#include <math.h>

namespace ercg {

constexpr int EW = 8;      // warps (source nodes) per CTA

struct EdgeWin { int b, i, len, lo, hi; long long row0; };
__device__ __forceinline__ EdgeWin edge_win(const int* __restrict__ node_off, const int* __restrict__ node_dlg, long long node,
                                            long long Lmax, int wp, int wf) {
  EdgeWin w;
  w.b = node_dlg[node];
  const int o = node_off[w.b];
  w.len = node_off[w.b + 1] - o;
  w.i = (int)(node - o);
  w.lo = wp < 0 ? 0 : max(0, w.i - wp);
  w.hi = wf < 0 ? w.len - 1 : min(w.len - 1, w.i + wf);
  w.row0 = (long long)w.b * Lmax;
  return w;
}

__global__ void __launch_bounds__(EW * 32)
masked_edge_att_fwd_kernel(const float* __restrict__ S, long long ldS, const int* __restrict__ node_off,
                           const int* __restrict__ node_dlg, const int* __restrict__ t_rowptr, const int* __restrict__ t_eid,
                           long long Lmax, int wp, int wf, float* __restrict__ nu, float* __restrict__ stat /* [N][2]: m, Den */,
                           long long N) {
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * EW + (threadIdx.x >> 5);
  if (node >= N) return;
  const EdgeWin w = edge_win(node_off, node_dlg, node, Lmax, wp, wf);
  const float* col = S + w.row0 * ldS + w.i;
  float m = -INFINITY;
  for (long long j = lane; j < Lmax; j += 32) m = fmaxf(m, col[j * ldS]);
  m = warp_max(m);
  float zall = 0.f, zwin = 0.f;
  for (long long j = lane; j < Lmax; j += 32) {
    const float e = expf(col[j * ldS] - m);
    zall += e;
    if (j >= w.lo && j <= w.hi) zwin += e;
  }
  zall = warp_sum(zall);
  zwin = warp_sum(zwin);
  const float den = zwin + 1e-10f * (zall - zwin);
  const int te0 = t_rowptr[node];
  for (int j = w.lo + lane; j <= w.hi; j += 32) nu[t_eid[te0 + (j - w.lo)]] = expf(col[(long long)j * ldS] - m) / den;
  if (lane == 0) { stat[2 * node] = m; stat[2 * node + 1] = den; }
}

__global__ void __launch_bounds__(EW * 32)
masked_edge_att_bwd_kernel(const float* __restrict__ S, long long ldS, const int* __restrict__ node_off,
                           const int* __restrict__ node_dlg, const int* __restrict__ t_rowptr, const int* __restrict__ t_eid,
                           long long Lmax, int wp, int wf, const float* __restrict__ nu, const float* __restrict__ dnu,
                           const float* __restrict__ stat, float* __restrict__ dS /* zero-initialised */, long long ldd, long long N) {
  const int lane = threadIdx.x & 31;
  const long long node = (long long)blockIdx.x * EW + (threadIdx.x >> 5);
  if (node >= N) return;
  const EdgeWin w = edge_win(node_off, node_dlg, node, Lmax, wp, wf);
  const float* col = S + w.row0 * ldS + w.i;
  float* dcol = dS + w.row0 * ldd + w.i;
  const float m = stat[2 * node], den = stat[2 * node + 1];
  const int te0 = t_rowptr[node];
  float G = 0.f;
  for (int j = w.lo + lane; j <= w.hi; j += 32) {
    const int e = t_eid[te0 + (j - w.lo)];
    G += dnu[e] * nu[e];
  }
  G = warp_sum(G);
  for (long long j = lane; j < Lmax; j += 32) {
    const bool in = j >= w.lo && j <= w.hi;
    const float e = expf(col[j * ldS] - m);
    float g = -(in ? 1.f : 1e-10f) * e / den * G;
    if (in) {
      const int eid = t_eid[te0 + (int)(j - w.lo)];
      g += dnu[eid] * nu[eid];
    }
    dcol[j * ldd] = g;
  }
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_masked_edge_att_fwd(const float* S, int64_t ldS, const int32_t* node_off, const int32_t* node_dlg,
                                        const int32_t* t_rowptr, const int32_t* t_eid, int64_t Lmax, int wp, int wf,
                                        float* nu, float* stat, int64_t N, void* stream) {
  if (N < 0 || Lmax < 1 || ldS < Lmax) return ERCG_EINVAL;     // S holds a column per source position: ldS >= Lmax
  if (N == 0) return ERCG_OK;
  if (!S || !node_off || !node_dlg || !t_rowptr || !t_eid || !nu || !stat) return ERCG_EINVAL;
  masked_edge_att_fwd_kernel<<<(unsigned)((N + EW - 1) / EW), EW * 32, 0, (cudaStream_t)stream>>>(
      S, ldS, node_off, node_dlg, t_rowptr, t_eid, Lmax, wp, wf, nu, stat, N);
  return finish_launch();
}

extern "C" int ercg_masked_edge_att_bwd(const float* S, int64_t ldS, const int32_t* node_off, const int32_t* node_dlg,
                                        const int32_t* t_rowptr, const int32_t* t_eid, int64_t Lmax, int wp, int wf,
                                        const float* nu, const float* dnu, const float* stat, float* dS, int64_t ldd,
                                        int64_t N, void* stream) {
  if (N < 0 || Lmax < 1 || ldS < Lmax || ldd < Lmax) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!S || !node_off || !node_dlg || !t_rowptr || !t_eid || !nu || !dnu || !stat || !dS) return ERCG_EINVAL;
  masked_edge_att_bwd_kernel<<<(unsigned)((N + EW - 1) / EW), EW * 32, 0, (cudaStream_t)stream>>>(
      S, ldS, node_off, node_dlg, t_rowptr, t_eid, Lmax, wp, wf, nu, dnu, stat, dS, ldd, N);
  return finish_launch();
}
