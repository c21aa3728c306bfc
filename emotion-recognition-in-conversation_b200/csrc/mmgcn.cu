// K7 / K8: the MMGCN cross-modal utterance graph as a BLOCK adjacency, and GCNII propagation over it.
//
// Reference: MMGCN.create_big_adj (track_mm/mmgcn_models.py:582-646) builds a dense [M*N, M*N] matrix
// (M modalities, N utterances) that is ~98 % zeros: the only non-zeros are, per dialogue d of length L,
//   * one dense L x L angular-similarity block per modality m on the diagonal   (:603-611,618-620)
//   * for m != n the DIAGONAL of block (m,n): similarity of the same utterance across modalities (:621-634)
// and GraphConvolution (:27-39) multiplies that dense matrix into the node features 64 times
// (GCNII_lyc.forward :373-394).  Here the adjacency is stored in exactly that block form
//   blocks: a[m*SB + blk_off[d] + i*L + j]              (SB = sum_d L_d^2)
//   cross : a[M*SB + (m*(M-1) + nslot(m,n))*N + node]   (nslot = n < m ? n : n-1)
// with node order = modality-major then dialogue-major (row (m,i) = m*N + i, mmgcn_models.py:616), and
// every product with it touches only the non-zeros.
//
//   rownorm      xhat = x / |x|                                               (:606-607)
//   adj_fwd      c' = 0.99999 <xhat_i, xhat_j>, A = 1 - acos(c')/pi, deg = row sum, dinv = deg^-1/2
//   adj_norm     Ahat = (dinv_i * A_ij) * dinv_j   -- the same two roundings as D.mm(adj).mm(D) (:638-644)
//   spmm         out[(m,i)] = sum_j Ahat_m[i,j] h[(m,j)] + sum_{n!=m} Ahat_x[(m,n),i] h[(n,i)]   (torch.spmm, :29)
//   sddmm_acc    G[(i,j)] += <dhi_i, h_j> on the pattern (gradient w.r.t. Ahat, summed over the 64 layers)
//   adj_bwd      G -> d deg -> dA -> dc -> dxhat -> dx (create_big_adj is differentiable w.r.t. the features)
//
// One warp per (modality, utterance) row; lane c owns float4 chunks c, c+32 of the D-wide row (D <= 256);
// block scalars are read warp-uniformly.  Every sum has a fixed order (j ascending, then the other
// modalities ascending) => bit-reproducible.  No atomics.
#include "common.cuh"

namespace ercg {

constexpr int MW = 8;                 // warps per block
constexpr float kCosScale = 0.99999f; // mmgcn_models.py:609,629
constexpr float kPi = 3.14159265358979323846f;

struct BlockGraph {
  const int* node_off;        // [B+1]
  const int* node_dlg;        // [N]
  const long long* blk_off;   // [B+1] prefix of L^2
  long long N, SB;
  int M;
};

__device__ __forceinline__ long long cross_index(const BlockGraph& g, int m, int n, long long node) {
  const int slot = n < m ? n : n - 1;
  return (long long)g.M * g.SB + ((long long)(m * (g.M - 1) + slot)) * g.N + node;
}

__device__ __forceinline__ void load_row(const float* __restrict__ p, int nch, int lane, float4 r[2]) {
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int ch = lane + 32 * c;
    r[c] = ch < nch ? ld4(p + 4 * ch) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
__device__ __forceinline__ float row_dot(const float4 a[2], const float4 b[2]) {
  return warp_sum(dot4(a[0], b[0]) + dot4(a[1], b[1]));
}

__global__ void __launch_bounds__(MW * 32)
rownorm_kernel(const float* __restrict__ x, long long ldx, float* __restrict__ xhat, long long ldh,
               float* __restrict__ rinv, long long rows, int D) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int nch = D >> 2;
  float4 v[2];
  load_row(x + row * ldx, nch, lane, v);
  const float len = sqrtf(row_dot(v, v));
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) st4(xhat + row * ldh + 4 * ch, make_float4(v[c].x / len, v[c].y / len, v[c].z / len, v[c].w / len));
  }
  if (lane == 0) rinv[row] = 1.0f / len;
}

__device__ __forceinline__ float sim_of(float c) { return 1.0f - acosf(c) / kPi; }

// cs (scaled cosines) and a (raw similarities, normalised in place by adj_norm) share the flat layout
__global__ void __launch_bounds__(MW * 32)
adj_fwd_kernel(BlockGraph g, const float* __restrict__ xhat, long long ldh, int D, float* __restrict__ cs,
               float* __restrict__ a, float* __restrict__ dinv) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (row >= g.N * g.M) return;
  const int m = (int)(row / g.N);
  const long long node = row - (long long)m * g.N;
  const int d = g.node_dlg[node];
  const int s = g.node_off[d], L = g.node_off[d + 1] - s;
  const int li = (int)(node - s);
  const int nch = D >> 2;
  float4 xi[2], xj[2];
  load_row(xhat + row * ldh, nch, lane, xi);
  const long long base = (long long)m * g.SB + g.blk_off[d] + (long long)li * L;
  float deg = 0.f;
  for (int j = 0; j < L; ++j) {
    load_row(xhat + ((long long)m * g.N + s + j) * ldh, nch, lane, xj);
    const float c = row_dot(xi, xj) * kCosScale;
    const float sim = sim_of(c);
    deg += sim;
    if (lane == 0) { cs[base + j] = c; a[base + j] = sim; }
  }
  for (int n = 0; n < g.M; ++n) {
    if (n == m) continue;
    load_row(xhat + ((long long)n * g.N + node) * ldh, nch, lane, xj);
    const float c = row_dot(xi, xj) * kCosScale;
    const float sim = sim_of(c);
    deg += sim;
    if (lane == 0) { const long long ci = cross_index(g, m, n, node); cs[ci] = c; a[ci] = sim; }
  }
  if (lane == 0) dinv[row] = 1.0f / sqrtf(deg);
}

__global__ void __launch_bounds__(MW * 32)
adj_norm_kernel(BlockGraph g, float* __restrict__ a, const float* __restrict__ dinv) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (row >= g.N * g.M) return;
  const int m = (int)(row / g.N);
  const long long node = row - (long long)m * g.N;
  const int d = g.node_dlg[node];
  const int s = g.node_off[d], L = g.node_off[d + 1] - s;
  const long long base = (long long)m * g.SB + g.blk_off[d] + (long long)(node - s) * L;
  const float di = dinv[row];
  for (int j = lane; j < L; j += 32) a[base + j] = (di * a[base + j]) * dinv[(long long)m * g.N + s + j];
  if (lane < g.M && lane != m) {
    const long long ci = cross_index(g, m, lane, node);
    a[ci] = (di * a[ci]) * dinv[(long long)lane * g.N + node];
  }
}

// out[(m,i),:] = sum_j W_m[i,j] h[(m,j),:] + sum_{n != m} X[(m,n),i] h[(n,i),:]   (TRANS: W_m[j,i], X[(n,m),i])
// optional side job: acc_dst[row,:] += acc_src[row,:]  (the h0 gradient summed over the layers)
template <bool TRANS>
__global__ void __launch_bounds__(MW * 32)
spmm_kernel(BlockGraph g, const float* __restrict__ a, const float* __restrict__ h, long long ldh_,
            float* __restrict__ out, long long ldo, int H, const float* __restrict__ acc_src, long long lds,
            float* __restrict__ acc_dst, long long ldd) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (row >= g.N * g.M) return;
  const int m = (int)(row / g.N);
  const long long node = row - (long long)m * g.N;
  const int d = g.node_dlg[node];
  const int s = g.node_off[d], L = g.node_off[d + 1] - s;
  const int li = (int)(node - s);
  const int nch = H >> 2;
  const float* blk = a + (long long)m * g.SB + g.blk_off[d];
  const float* hb = h + ((long long)m * g.N + s) * ldh_;
  float4 acc[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
  int j = 0;
  for (; j + 4 <= L; j += 4) {
    float w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) w[u] = TRANS ? blk[(long long)(j + u) * L + li] : blk[(long long)li * L + j + u];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ld4(hb + (long long)(j + u) * ldh_ + 4 * ch);
#pragma unroll
        for (int u = 0; u < 4; ++u) fma4(acc[c], w[u], v[u]);
      }
    }
  }
  for (; j < L; ++j) {
    const float w = TRANS ? blk[(long long)j * L + li] : blk[(long long)li * L + j];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) fma4(acc[c], w, ld4(hb + (long long)j * ldh_ + 4 * ch));
    }
  }
  for (int n = 0; n < g.M; ++n) {
    if (n == m) continue;
    const float w = TRANS ? a[cross_index(g, n, m, node)] : a[cross_index(g, m, n, node)];
    const float* p = h + ((long long)n * g.N + node) * ldh_;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) fma4(acc[c], w, ld4(p + 4 * ch));
    }
  }
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) {
      st4(out + row * ldo + 4 * ch, acc[c]);
      if (acc_dst) {
        const float4 u = ld4(acc_src + row * lds + 4 * ch);
        float4 t = ld4(acc_dst + row * ldd + 4 * ch);
        t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
        st4(acc_dst + row * ldd + 4 * ch, t);
      }
    }
  }
}

// G[(m,i),(m,j)] (+)= <dhi[(m,i)], h[(m,j)]>,  Gx[(m,n),i] (+)= <dhi[(m,i)], h[(n,i)]>
__global__ void __launch_bounds__(MW * 32)
sddmm_kernel(BlockGraph g, const float* __restrict__ dhi, long long ldd, const float* __restrict__ h, long long ldh_,
             int H, float* __restrict__ G, int accumulate) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (row >= g.N * g.M) return;
  const int m = (int)(row / g.N);
  const long long node = row - (long long)m * g.N;
  const int d = g.node_dlg[node];
  const int s = g.node_off[d], L = g.node_off[d + 1] - s;
  const int nch = H >> 2;
  float4 di[2], hj[2];
  load_row(dhi + row * ldd, nch, lane, di);
  const long long base = (long long)m * g.SB + g.blk_off[d] + (long long)(node - s) * L;
  for (int j0 = 0; j0 < L; j0 += 32) {
    float mine = 0.f;
    const int jn = min(32, L - j0);
    for (int u = 0; u < jn; ++u) {
      load_row(h + ((long long)m * g.N + s + j0 + u) * ldh_, nch, lane, hj);
      const float v = row_dot(di, hj);
      if (lane == u) mine = v;
    }
    if (lane < jn) {
      const long long idx = base + j0 + lane;
      G[idx] = accumulate ? G[idx] + mine : mine;
    }
  }
  for (int n = 0; n < g.M; ++n) {
    if (n == m) continue;
    load_row(h + ((long long)n * g.N + node) * ldh_, nch, lane, hj);
    const float v = row_dot(di, hj);
    if (lane == 0) {
      const long long ci = cross_index(g, m, n, node);
      G[ci] = accumulate ? G[ci] + v : v;
    }
  }
}

// d deg[(m,i)] from G (gradient w.r.t. Ahat), the scaled cosines cs and dinv:
//   ddinv_k = sum_j G_kj A_kj dinv_j + sum_i G_ik A_ik dinv_i ;  ddeg_k = -1/2 ddinv_k dinv_k^3
__global__ void __launch_bounds__(MW * 32)
adj_bwd_deg_kernel(BlockGraph g, const float* __restrict__ G, const float* __restrict__ cs,
                   const float* __restrict__ dinv, float* __restrict__ ddeg) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (row >= g.N * g.M) return;
  const int m = (int)(row / g.N);
  const long long node = row - (long long)m * g.N;
  const int d = g.node_dlg[node];
  const int s = g.node_off[d], L = g.node_off[d + 1] - s;
  const int li = (int)(node - s);
  const long long blk = (long long)m * g.SB + g.blk_off[d];
  float t = 0.f;
  for (int j = lane; j < L; j += 32) {
    const long long ij = blk + (long long)li * L + j, ji = blk + (long long)j * L + li;
    const float dj = dinv[(long long)m * g.N + s + j];
    t += (G[ij] * sim_of(cs[ij]) + G[ji] * sim_of(cs[ji])) * dj;
  }
  if (lane < g.M && lane != m) {
    const long long mn = cross_index(g, m, lane, node), nm = cross_index(g, lane, m, node);
    t += (G[mn] * sim_of(cs[mn]) + G[nm] * sim_of(cs[nm])) * dinv[(long long)lane * g.N + node];
  }
  t = warp_sum(t);
  if (lane == 0) {
    const float di = dinv[row];
    ddeg[row] = -0.5f * t * di * di * di;
  }
}

__device__ __forceinline__ float dsim_dcos(float c) {   // d/dcos of 1 - acos(0.99999 cos)/pi, c = 0.99999 cos
  return kCosScale / (kPi * sqrtf(1.0f - c * c));
}

// dx[(m,i)] = (dxhat - xhat <xhat, dxhat>) / |x|,  dxhat_i = sum_j (e_ij + e_ji) xhat_j + cross terms,
// e_ij = (G_ij dinv_i dinv_j + ddeg_i) * dsim_dcos(c_ij)
__global__ void __launch_bounds__(MW * 32)
adj_bwd_x_kernel(BlockGraph g, const float* __restrict__ G, const float* __restrict__ cs,
                 const float* __restrict__ dinv, const float* __restrict__ ddeg, const float* __restrict__ xhat,
                 long long ldh, const float* __restrict__ rinv, int D, float* __restrict__ dx, long long ldx) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (row >= g.N * g.M) return;
  const int m = (int)(row / g.N);
  const long long node = row - (long long)m * g.N;
  const int d = g.node_dlg[node];
  const int s = g.node_off[d], L = g.node_off[d + 1] - s;
  const int li = (int)(node - s);
  const int nch = D >> 2;
  const long long blk = (long long)m * g.SB + g.blk_off[d];
  const float di = dinv[row], ddi = ddeg[row];
  float4 acc[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
  float4 xj[2];
  for (int j = 0; j < L; ++j) {
    const long long ij = blk + (long long)li * L + j, ji = blk + (long long)j * L + li;
    const long long rj = (long long)m * g.N + s + j;
    const float dj = dinv[rj];
    const float w = (G[ij] * di * dj + ddi) * dsim_dcos(cs[ij]) + (G[ji] * dj * di + ddeg[rj]) * dsim_dcos(cs[ji]);
    load_row(xhat + rj * ldh, nch, lane, xj);
    fma4(acc[0], w, xj[0]);
    fma4(acc[1], w, xj[1]);
  }
  for (int n = 0; n < g.M; ++n) {
    if (n == m) continue;
    const long long mn = cross_index(g, m, n, node), nm = cross_index(g, n, m, node);
    const long long rn = (long long)n * g.N + node;
    const float dn = dinv[rn];
    const float w = (G[mn] * di * dn + ddi) * dsim_dcos(cs[mn]) + (G[nm] * dn * di + ddeg[rn]) * dsim_dcos(cs[nm]);
    load_row(xhat + rn * ldh, nch, lane, xj);
    fma4(acc[0], w, xj[0]);
    fma4(acc[1], w, xj[1]);
  }
  float4 xi[2];
  load_row(xhat + row * ldh, nch, lane, xi);
  const float proj = row_dot(acc, xi);
  const float r = rinv[row];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch)
      st4(dx + row * ldx + 4 * ch, make_float4((acc[c].x - xi[c].x * proj) * r, (acc[c].y - xi[c].y * proj) * r,
                                               (acc[c].z - xi[c].z * proj) * r, (acc[c].w - xi[c].w * proj) * r));
  }
}

// ---- small helpers on the MMGCN path
// rows[i] = row of packed node i in a padded tensor: seq-first [Lmax,B,*] -> k*B + d, batch-first [B,Lmax,*] -> d*Lmax + k
__global__ void node_rows_kernel(const int* __restrict__ node_off, const int* __restrict__ node_dlg, long long N, int B,
                                 int Lmax, int seq_first, int* __restrict__ rows) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const int d = node_dlg[i];
  const int k = (int)(i - node_off[d]);
  rows[i] = seq_first ? k * B + d : d * Lmax + k;
}

// blk_off[d] = sum_{d' < d} L_{d'}^2 : one block, sequential over chunks (B is small next to N)
__global__ void blk_off_kernel(const int* __restrict__ node_off, int B, long long* __restrict__ blk_off) {
  __shared__ long long part[256];
  const int t = threadIdx.x;
  const int per = (B + 255) / 256;
  const int lo = min(B, t * per), hi = min(B, lo + per);
  long long s = 0;
  for (int d = lo; d < hi; ++d) { const long long L = node_off[d + 1] - node_off[d]; s += L * L; }
  part[t] = s;
  __syncthreads();
  if (t == 0) {
    long long run = 0;
    for (int i = 0; i < 256; ++i) { const long long v = part[i]; part[i] = run; run += v; }
    blk_off[B] = run;
  }
  __syncthreads();
  long long run = part[t];
  for (int d = lo; d < hi; ++d) { const long long L = node_off[d + 1] - node_off[d]; blk_off[d] = run; run += L * L; }
}

// l[i,:] += emb[argmax(qmask[rows[i],:]), :]   (MMGCN.forward, mmgcn_models.py:540-545); ids[i] = the argmax
__global__ void __launch_bounds__(MW * 32)
speaker_embed_add_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ qmask, int n_spk,
                         const int* __restrict__ rows, const float* __restrict__ emb, long long lde,
                         float* __restrict__ out, long long ldo, int* __restrict__ ids, float* __restrict__ onehot,
                         long long N, int D) {
  const int lane = threadIdx.x & 31;
  const long long i = (long long)blockIdx.x * MW + (threadIdx.x >> 5);
  if (i >= N) return;
  const float* q = qmask + (long long)rows[i] * n_spk;
  int best = 0;
  float bv = q[0];
  for (int k = 1; k < n_spk; ++k) { const float v = q[k]; if (v > bv) { bv = v; best = k; } }   // first maximum, like argmax
  if (lane == 0) ids[i] = best;
  for (int k = lane; k < n_spk; k += 32) onehot[i * n_spk + k] = k == best ? 1.f : 0.f;
  const int nch = D >> 2;
  for (int ch = lane; ch < nch; ch += 32) {
    const float4 a = ld4(x + i * ldx + 4 * ch), b = ld4(emb + (long long)best * lde + 4 * ch);
    st4(out + i * ldo + 4 * ch, make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w));
  }
}

__global__ void relu_dropout_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, float p, float scale,
                                    unsigned long long seed) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v = fmaxf(x[i], 0.f);
  if (p > 0.f) v = hash_uniform(seed, (unsigned long long)i) < p ? 0.f : v * scale;
  out[i] = v;
}

// relu_dropout_kernel with the seed offset read from device memory (a step counter that a captured graph advances)
__global__ void relu_dropout_dev_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, float p, float scale,
                                        unsigned long long seed, const unsigned long long* __restrict__ seed_dev) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v = fmaxf(x[i], 0.f);
  if (p > 0.f) v = hash_uniform(seed + __ldg(seed_dev), (unsigned long long)i) < p ? 0.f : v * scale;
  out[i] = v;
}

static int check_graph(const int32_t* node_off, const int32_t* node_dlg, const int64_t* blk_off, int64_t N, int64_t SB,
                       int M) {
  if (!node_off || !node_dlg || !blk_off || N < 0 || SB < 0 || M < 1 || M > 3) return ERCG_EINVAL;
  if ((long long)N * M > 2147483647LL * MW) return ERCG_ERANGE;
  return ERCG_OK;
}
static inline unsigned row_grid(long long rows) { return (unsigned)((rows + MW - 1) / MW); }
static inline bool row_ok(const float* p, int64_t ld, int D) { return p && aligned16(p) && (ld & 3) == 0 && ld >= D; }

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_node_rows(const int32_t* node_off, const int32_t* node_dlg, int64_t N, int B, int Lmax,
                              int seq_first, int32_t* rows, void* stream) {
  if (N < 0 || B < 0 || Lmax < 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!node_off || !node_dlg || !rows) return ERCG_EINVAL;
  if ((long long)B * Lmax > 2147483647LL) return ERCG_ERANGE;
  node_rows_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(node_off, node_dlg, N, B, Lmax, seq_first,
                                                                                rows);
  return finish_launch();
}

extern "C" int ercg_mmgcn_block_offsets(const int32_t* node_off, int B, int64_t* blk_off, void* stream) {
  if (B < 0 || !node_off || !blk_off) return ERCG_EINVAL;
  blk_off_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(node_off, B, reinterpret_cast<long long*>(blk_off));
  return finish_launch();
}

extern "C" int ercg_mmgcn_adj_fwd(const float* x, int64_t ldx, const int32_t* node_off, const int32_t* node_dlg,
                                  const int64_t* blk_off, int64_t N, int64_t SB, int M, int D, float* xhat, int64_t ldh,
                                  float* rinv, float* cs, float* ahat, float* dinv, void* stream) {
  int rc = check_graph(node_off, node_dlg, blk_off, N, SB, M);
  if (rc != ERCG_OK) return rc;
  if (N == 0) return ERCG_OK;
  if (D <= 0 || D > 256 || (D & 3) || !rinv || !cs || !ahat || !dinv) return ERCG_EINVAL;
  if (!row_ok(x, ldx, D) || !row_ok(xhat, ldh, D)) return ERCG_EALIGN;
  BlockGraph g{node_off, node_dlg, reinterpret_cast<const long long*>(blk_off), N, SB, M};
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)N * M;
  rownorm_kernel<<<row_grid(rows), MW * 32, 0, st>>>(x, ldx, xhat, ldh, rinv, rows, D);
  if ((rc = finish_launch()) != ERCG_OK) return rc;
  adj_fwd_kernel<<<row_grid(rows), MW * 32, 0, st>>>(g, xhat, ldh, D, cs, ahat, dinv);
  if ((rc = finish_launch()) != ERCG_OK) return rc;
  adj_norm_kernel<<<row_grid(rows), MW * 32, 0, st>>>(g, ahat, dinv);
  return finish_launch();
}

extern "C" int ercg_mmgcn_adj_bwd(const float* G, const float* cs, const float* dinv, const float* xhat, int64_t ldh,
                                  const float* rinv, const int32_t* node_off, const int32_t* node_dlg,
                                  const int64_t* blk_off, int64_t N, int64_t SB, int M, int D, float* ddeg, float* dx,
                                  int64_t ldx, void* stream) {
  int rc = check_graph(node_off, node_dlg, blk_off, N, SB, M);
  if (rc != ERCG_OK) return rc;
  if (N == 0) return ERCG_OK;
  if (D <= 0 || D > 256 || (D & 3) || !G || !cs || !dinv || !rinv || !ddeg) return ERCG_EINVAL;
  if (!row_ok(xhat, ldh, D) || !row_ok(dx, ldx, D)) return ERCG_EALIGN;
  BlockGraph g{node_off, node_dlg, reinterpret_cast<const long long*>(blk_off), N, SB, M};
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)N * M;
  adj_bwd_deg_kernel<<<row_grid(rows), MW * 32, 0, st>>>(g, G, cs, dinv, ddeg);
  if ((rc = finish_launch()) != ERCG_OK) return rc;
  adj_bwd_x_kernel<<<row_grid(rows), MW * 32, 0, st>>>(g, G, cs, dinv, ddeg, xhat, ldh, rinv, D, dx, ldx);
  return finish_launch();
}

extern "C" int ercg_mmgcn_spmm(const float* ahat, int transpose, const float* h, int64_t ldh, float* out, int64_t ldo,
                               const int32_t* node_off, const int32_t* node_dlg, const int64_t* blk_off, int64_t N,
                               int64_t SB, int M, int H, const float* acc_src, int64_t lds, float* acc_dst, int64_t ldd,
                               void* stream) {
  int rc = check_graph(node_off, node_dlg, blk_off, N, SB, M);
  if (rc != ERCG_OK) return rc;
  if (N == 0) return ERCG_OK;
  if (H <= 0 || H > 256 || (H & 3) || !ahat) return ERCG_EINVAL;
  if (!row_ok(h, ldh, H) || !row_ok(out, ldo, H)) return ERCG_EALIGN;
  if ((acc_dst != nullptr) != (acc_src != nullptr)) return ERCG_EINVAL;
  if (acc_dst && (!row_ok(acc_src, lds, H) || !row_ok(acc_dst, ldd, H))) return ERCG_EALIGN;
  BlockGraph g{node_off, node_dlg, reinterpret_cast<const long long*>(blk_off), N, SB, M};
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)N * M;
  if (transpose)
    spmm_kernel<true><<<row_grid(rows), MW * 32, 0, st>>>(g, ahat, h, ldh, out, ldo, H, acc_src, lds, acc_dst, ldd);
  else
    spmm_kernel<false><<<row_grid(rows), MW * 32, 0, st>>>(g, ahat, h, ldh, out, ldo, H, acc_src, lds, acc_dst, ldd);
  return finish_launch();
}

extern "C" int ercg_mmgcn_sddmm(const float* dhi, int64_t ldd, const float* h, int64_t ldh, const int32_t* node_off,
                                const int32_t* node_dlg, const int64_t* blk_off, int64_t N, int64_t SB, int M, int H,
                                float* G, int accumulate, void* stream) {
  int rc = check_graph(node_off, node_dlg, blk_off, N, SB, M);
  if (rc != ERCG_OK) return rc;
  if (N == 0) return ERCG_OK;
  if (H <= 0 || H > 256 || (H & 3) || !G) return ERCG_EINVAL;
  if (!row_ok(dhi, ldd, H) || !row_ok(h, ldh, H)) return ERCG_EALIGN;
  BlockGraph g{node_off, node_dlg, reinterpret_cast<const long long*>(blk_off), N, SB, M};
  const long long rows = (long long)N * M;
  sddmm_kernel<<<row_grid(rows), MW * 32, 0, (cudaStream_t)stream>>>(g, dhi, ldd, h, ldh, H, G, accumulate);
  return finish_launch();
}

extern "C" int ercg_speaker_embed_add(const float* x, int64_t ldx, const float* qmask, int n_speakers, const int32_t* rows,
                                      const float* emb, int64_t lde, float* out, int64_t ldo, int32_t* ids, float* onehot,
                                      int64_t N, int D, void* stream) {
  if (N < 0 || n_speakers < 1 || D <= 0 || (D & 3)) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!qmask || !rows || !ids || !onehot) return ERCG_EINVAL;
  if (!row_ok(x, ldx, D) || !row_ok(emb, lde, D) || !row_ok(out, ldo, D)) return ERCG_EALIGN;
  speaker_embed_add_kernel<<<row_grid(N), MW * 32, 0, (cudaStream_t)stream>>>(x, ldx, qmask, n_speakers, rows, emb, lde, out,
                                                                             ldo, ids, onehot, N, D);
  return finish_launch();
}

extern "C" int ercg_relu_dropout(const float* x, float* out, int64_t n, float p, uint64_t seed, void* stream) {
  if (n < 0 || !(p >= 0.f && p < 1.f)) return ERCG_EINVAL;
  if (n == 0) return ERCG_OK;
  if (!x || !out) return ERCG_EINVAL;
  relu_dropout_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, n, p, 1.f / (1.f - p), seed);
  return finish_launch();
}

extern "C" int ercg_relu_dropout_dev(const float* x, float* out, int64_t n, float p, uint64_t seed, const uint64_t* seed_dev,
                                     void* stream) {
  if (!seed_dev || n < 0 || !(p >= 0.f && p < 1.f)) return ERCG_EINVAL;
  if (n == 0) return ERCG_OK;
  if (!x || !out) return ERCG_EINVAL;
  relu_dropout_dev_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      x, out, n, p, 1.f / (1.f - p), seed, reinterpret_cast<const unsigned long long*>(seed_dev));
  return finish_launch();
}
