// K1: batch_graphify as one cooperative integer kernel (sm_100a).
//
// Replaces the python loops of the reference:
//   edge_perms      track_mm/cogmen_utils.py:147-172 (= dgcn_models.py:95-118)
//   batch_graphify  track_mm/cogmen_utils.py:109-144, track_mm/dgcn_models.py:51-92
// Everything is closed form: the in-edges of k are the window [max(0,k-wf), min(L-1,k+wp)], the
// out-edges of j are [max(0,j-wp), min(L-1,j+wf)], and the prefix of window sizes has a formula
// (deg_prefix), so no per-node scan is needed -- only a scan over the B dialogue lengths.
//
// One launch, three phases separated by grid.sync():
//   1. per-tile (256 dialogues) sums of node and edge counts
//   2. exclusive scan -> node_off[B+1], edge_off[B+1], edge_index_lengths[B]
//   3. one warp per dialogue fills node arrays, then walks its by-destination edge range and its
//      by-source edge range lane-per-edge (coalesced 4/1/8-byte stores).
// HBM traffic (algorithmic): 8B(lengths) + N speakers + 8(N+1) rowptrs + E*(4+1+4+1+4) (+4E inv_cnt,
// +24E when the reference-layout int64 edge_index/edge_type are requested).
#include <atomic>
#include "common.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace ercg {

__host__ __device__ inline void eff_window(long long L, int wp, int wf, long long& P, long long& F) {
  long long m = L > 0 ? L - 1 : 0;
  P = (wp < 0 || wp > m) ? m : wp;
  F = (wf < 0 || wf > m) ? m : wf;
}

__host__ __device__ inline long long dialog_edges(long long L, int wp, int wf) {
  if (L <= 0) return 0;
  long long P, F;
  eff_window(L, wp, wf, P, F);
  return L * (P + F + 1) - P * (P + 1) / 2 - F * (F + 1) / 2;
}

// sum_{k' < k} [ min(L-1, k'+A) - max(0, k'-Bk) + 1 ],  0 <= k <= L,  0 <= A,Bk <= L-1
__host__ __device__ inline long long deg_prefix(long long L, long long A, long long Bk, long long k) {
  long long t1 = L - A;                       // nodes k' < t1 are not clipped on the high side
  long long a = k < t1 ? k : t1;
  long long sum1 = a * A + a * (a - 1) / 2 + (k - a) * (L - 1);
  long long b = k - 1 - Bk;
  if (b < 0) b = 0;
  return sum1 + k - b * (b + 1) / 2;
}

struct GraphifyParams {
  const void* lengths; int len64; int B;
  const void* speakers; int spk64; long long spk_ld;
  int wp, wf, n_speakers;
  long long N, E;
  ercg_graph_out o;
  long long* tile_agg;   // [2 * numTiles]
};

__device__ __forceinline__ long long load_len(const GraphifyParams& p, int b) {
  long long L = p.len64 ? reinterpret_cast<const long long*>(p.lengths)[b]
                        : (long long)reinterpret_cast<const int*>(p.lengths)[b];
  return L < 0 ? 0 : L;
}

// block-wide inclusive scan of a pair of int64 (blockDim.x <= 1024, multiple of 32)
__device__ inline void block_scan_pair(long long& a, long long& b, long long* sm /* [2*32+2] */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    long long ta = __shfl_up_sync(0xffffffffu, a, o), tb = __shfl_up_sync(0xffffffffu, b, o);
    if (lane >= o) { a += ta; b += tb; }
  }
  __syncthreads();
  if (lane == 31) { sm[2 * wid] = a; sm[2 * wid + 1] = b; }
  __syncthreads();
  if (wid == 0) {
    long long wa = lane < nw ? sm[2 * lane] : 0, wb = lane < nw ? sm[2 * lane + 1] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      long long ta = __shfl_up_sync(0xffffffffu, wa, o), tb = __shfl_up_sync(0xffffffffu, wb, o);
      if (lane >= o) { wa += ta; wb += tb; }
    }
    if (lane < nw) { sm[2 * lane] = wa; sm[2 * lane + 1] = wb; }
  }
  __syncthreads();
  if (wid > 0) { a += sm[2 * (wid - 1)]; b += sm[2 * (wid - 1) + 1]; }
}

// sum_{k' < k} [ min(L-1, k'+A) - max(0, k'-Bk) + 1 ] in the index type I (int when L <= 46340: every product below is
// < 2^31 there; unsigned halves keep a*(a-1) exact)
template <typename I>
__device__ __forceinline__ I deg_prefix_t(I L, I A, I Bk, I k) {
  const I t1 = L - A;
  const I a = k < t1 ? k : t1;
  const I sum1 = a * A + (I)(((unsigned long long)(unsigned)a * (unsigned)(a - 1)) >> 1) + (k - a) * (L - 1);
  I b = k - 1 - Bk;
  if (b < 0) b = 0;
  return sum1 + k - (I)(((unsigned long long)(unsigned)b * (unsigned)(b + 1)) >> 1);
}
template <>
__device__ __forceinline__ long long deg_prefix_t<long long>(long long L, long long A, long long Bk, long long k) {
  return deg_prefix(L, A, Bk, k);
}

// One warp fills one dialogue: (a) node arrays lane-per-node, (b) by-destination edges, (c) by-source edges, lane-per-edge.
// Edge chunks are ROW-ALIGNED (a chunk holds whole rows whenever the row degree is <= 32), so the PyG mean weight
// 1/|{e' : dst = dst(e), type = type(e)}| is one __match_any_sync over (row, speaker, direction) instead of a loop over the
// window per edge (that loop was ~1/3 of this kernel's instructions); rows longer than a warp keep the loop.
template <typename I>
__device__ __forceinline__ void fill_dialogue(const GraphifyParams& p, int d, I L, I o, I eo) {
  const int lane = threadIdx.x & 31;
  const int n_spk = p.n_speakers;
  const I m = L - 1;
  const I P = (p.wp < 0 || (long long)p.wp > (long long)m) ? m : (I)p.wp;
  const I F = (p.wf < 0 || (long long)p.wf > (long long)m) ? m : (I)p.wf;
  for (I k = lane; k < L; k += 32) {
    long long s;
    int bad = 0;
    // a dialogue longer than the padded width would read the next dialogue's speakers (or past the array) and emit pad_row
    // values outside [0, B*Lmax): never dereference, clamp, and raise ERCG_GRAPH_ELENGTH in rel_info[513] (the reference
    // raises IndexError here, cogmen_utils.py:131-132)
    const long long kk = (p.spk_ld > 0 && (long long)k >= p.spk_ld) ? p.spk_ld - 1 : (long long)k;
    if (kk != (long long)k) bad |= 1;
    if (p.spk_ld > 0) {
      const long long idx = (long long)d * p.spk_ld + kk;
      s = p.spk64 ? reinterpret_cast<const long long*>(p.speakers)[idx]
                  : (long long)reinterpret_cast<const int*>(p.speakers)[idx];
    } else {
      s = p.spk64 ? reinterpret_cast<const long long*>(p.speakers)[(long long)o + k]
                  : (long long)reinterpret_cast<const int*>(p.speakers)[(long long)o + k];
    }
    if (s < 0 || s >= (long long)n_spk) { bad |= 2; s = 0; }       // would wrap in the uint8 relation id (reference: KeyError)
    if (bad && p.o.rel_info) atomicOr(p.o.rel_info + 513, bad);
    p.o.spk[o + k] = (int)s;
    p.o.node_dlg[o + k] = d;
    if (p.o.pad_row) p.o.pad_row[o + k] = (int)(p.spk_ld > 0 ? (long long)d * p.spk_ld + kk : (long long)(o + k));
    p.o.rowptr[o + k] = (int)(eo + deg_prefix_t<I>(L, P, F, k));
    p.o.t_rowptr[o + k] = (int)(eo + deg_prefix_t<I>(L, F, P, k));
  }
  __syncwarp();
  const int* spk = p.o.spk + o;
  for (int pass = 0; pass < 2; ++pass) {
    const I A = pass == 0 ? P : F;      // high-side reach of the row node
    const I Bk = pass == 0 ? F : P;     // low-side reach
    for (I k0 = 0; k0 < L; k0 += 32) {
      I kmine = k0 + lane;
      if (kmine > L) kmine = L;
      const I myS = deg_prefix_t<I>(L, A, Bk, kmine);          // first edge of row k0 + lane (clamped to the end)
      const I kend = k0 + 32 < L ? k0 + 32 : L;
      const I end = deg_prefix_t<I>(L, A, Bk, kend);
      I xb = __shfl_sync(0xffffffffu, myS, 0);
      while (xb < end) {
        // chunk = [xb, xe): as many WHOLE rows as fit in 32 lanes when a row starts at xb and fits; otherwise (row longer
        // than a warp, or xb in the middle of such a row) up to 32 edges of that one row
        const I nextS = __shfl_down_sync(0xffffffffu, myS, 1);
        const I rowEnd = lane == 31 ? end : nextS;              // lane l's row ends where row l + 1 starts
        const bool rowok = k0 + lane < kend;
        unsigned fits = 0u;
        if (__ballot_sync(0xffffffffu, rowok && myS == xb))
          fits = __ballot_sync(0xffffffffu, rowok && myS >= xb && rowEnd <= xb + 32);
        I xe;
        bool whole;
        if (fits) {
          xe = __shfl_sync(0xffffffffu, rowEnd, 31 - __clz(fits));
          whole = true;
        } else {
          const unsigned cont = __ballot_sync(0xffffffffu, rowok && myS <= xb && xb < rowEnd);
          const I re = __shfl_sync(0xffffffffu, rowEnd, cont ? __ffs(cont) - 1 : 31);
          xe = xb + 32 < re ? xb + 32 : re;
          whole = false;
        }
        const I x = xb + lane;
        const bool valid = x < xe;
        const I xs = valid ? x : xb;
        int lo = 0, hi = 31;
#pragma unroll
        for (int it = 0; it < 5; ++it) {
          const int mid = (lo + hi + 1) >> 1;
          const I v = __shfl_sync(0xffffffffu, myS, mid);
          if (v <= xs) lo = mid; else hi = mid - 1;
        }
        const I Srow = __shfl_sync(0xffffffffu, myS, lo);
        const I row = k0 + lo;                                  // k (pass 0) or j (pass 1)
        const I rlo = row - Bk > 0 ? row - Bk : 0;
        const I other = rlo + (xs - Srow);                      // j (pass 0) or k (pass 1)
        const I j = pass == 0 ? other : row;
        const I k = pass == 0 ? row : other;
        const int sj = spk[j], sk = spk[k];
        const int ty = (sj * n_spk + sk) * 2 + (j >= k ? 1 : 0);
        const long long e = (long long)eo + (long long)x;
        if (pass == 0) {
          unsigned same = 0u;
          if (p.o.inv_cnt && whole) {
            const unsigned key = valid ? (((unsigned)lo << 16) | ((unsigned)sj << 1) | (j >= k ? 1u : 0u)) : (0x80000000u | lane);
            same = __match_any_sync(0xffffffffu, key);
          }
          if (valid) {
            p.o.col[e] = (int)(o + j);
            p.o.etype[e] = (uint8_t)ty;
            if (p.o.edge_index) { p.o.edge_index[e] = (long long)(o + j); p.o.edge_index[p.E + e] = (long long)(o + k); }
            if (p.o.edge_type) p.o.edge_type[e] = ty;
            if (p.o.inv_cnt) {
              int c;
              if (whole) {
                c = __popc(same);
              } else {
                const I rhi = k + P < L - 1 ? k + P : L - 1;
                const bool dirj = j >= k;
                c = 0;
                for (I jj = rlo; jj <= rhi; ++jj) c += (spk[jj] == sj && ((jj >= k) == dirj)) ? 1 : 0;
              }
              p.o.inv_cnt[e] = 1.0f / (float)c;
            }
          }
        } else if (valid) {
          p.o.t_col[e] = (int)(o + k);
          p.o.t_etype[e] = (uint8_t)ty;
          const I klo = k - F > 0 ? k - F : 0;
          p.o.t_eid[e] = (int)(eo + deg_prefix_t<I>(L, P, F, k) + (j - klo));
        }
        xb = xe;
      }
    }
  }
}

__global__ void __launch_bounds__(256) graphify_kernel(GraphifyParams p) {
  cg::grid_group grid = cg::this_grid();
  __shared__ long long sm[66];
  const int T = blockDim.x;
  const int numTiles = (p.B + T - 1) / T;
  if (p.o.rel_info && blockIdx.x == 0)       // [0] count, [1..256] id -> slot, [257..512] slot -> id: see rel_census_kernel
    for (int i = threadIdx.x; i < 516; i += T) p.o.rel_info[i] = (i == 0 || i >= 513) ? 0 : -1;   // [513] = input-error flags

  // ---- phase 1: tile aggregates
  for (int tile = blockIdx.x; tile < numTiles; tile += gridDim.x) {
    int b = tile * T + threadIdx.x;
    long long n = 0, e = 0;
    if (b < p.B) { n = load_len(p, b); e = dialog_edges(n, p.wp, p.wf); }
    block_scan_pair(n, e, sm);
    if (threadIdx.x == T - 1) { p.tile_agg[2 * tile] = n; p.tile_agg[2 * tile + 1] = e; }
    __syncthreads();
  }
  grid.sync();

  // ---- phase 2: offsets
  for (int tile = blockIdx.x; tile < numTiles; tile += gridDim.x) {
    long long pn = 0, pe = 0;
    for (int t = threadIdx.x; t < tile; t += T) { pn += p.tile_agg[2 * t]; pe += p.tile_agg[2 * t + 1]; }
    block_scan_pair(pn, pe, sm);      // last thread holds the totals of all previous tiles
    __syncthreads();
    if (threadIdx.x == T - 1) { sm[64] = pn; sm[65] = pe; }
    __syncthreads();
    const long long basen = sm[64], basee = sm[65];
    int b = tile * T + threadIdx.x;
    long long n = 0, e = 0;
    if (b < p.B) { n = load_len(p, b); e = dialog_edges(n, p.wp, p.wf); }
    long long n0 = n, e0 = e;
    block_scan_pair(n, e, sm);
    if (b < p.B) {
      p.o.node_off[b] = (int)(basen + n - n0);
      p.o.edge_off[b] = (int)(basee + e - e0);
      if (p.o.edge_index_lengths) p.o.edge_index_lengths[b] = e0;
      if (b == p.B - 1) {
        long long Nt = basen + n, Et = basee + e;
        p.o.node_off[p.B] = (int)Nt;
        p.o.edge_off[p.B] = (int)Et;
        if (Nt <= p.N) { p.o.rowptr[Nt] = (int)Et; p.o.t_rowptr[Nt] = (int)Et; }
        if (p.o.totals) { p.o.totals[0] = Nt; p.o.totals[1] = Et; }
      }
    }
    __syncthreads();
  }
  if (p.B == 0 && blockIdx.x == 0 && threadIdx.x == 0) {
    p.o.node_off[0] = 0; p.o.edge_off[0] = 0; p.o.rowptr[0] = 0; p.o.t_rowptr[0] = 0;
    if (p.o.totals) { p.o.totals[0] = 0; p.o.totals[1] = 0; }
  }
  grid.sync();

  // ---- phase 3: one warp per dialogue
  const int warps_per_block = T >> 5;
  const long long gwarp = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * warps_per_block;
  for (long long d = gwarp; d < p.B; d += nwarps) {
    const long long L = load_len(p, (int)d);
    if (L == 0) continue;
    const long long o = p.o.node_off[d], eo = p.o.edge_off[d];
    if (o + L > p.N || eo + dialog_edges(L, p.wp, p.wf) > p.E) {   // caller passed too-small N / E: never write out of bounds
      if (p.o.rel_info && (threadIdx.x & 31) == 0) atomicOr(p.o.rel_info + 513, 4);
      continue;
    }
    // every in-dialogue quantity fits 32 bits when L <= 46340 (L^2 < 2^31): the integer pipe is the bound of this kernel
    if (L <= 46340) fill_dialogue<int>(p, (int)d, (int)L, (int)o, (int)eo);
    else fill_dialogue<long long>(p, (int)d, L, o, eo);
  }
}

// ---- relation census: which relation ids occur on at least one edge, and their compact numbering.  Consumers (RGCNConv)
// transform and gather only the relation slots that exist (one-speaker data such as MOSEI uses 2 of the 8 ids).
// Pass 1 streams etype[E] (16 ids per load) and marks the ids it sees: rel_info[1 + id] = 0 (every writer stores the same
// value -> no atomics on global memory); pass 2 (one block) turns the marks into slots.  Kept out of graphify_kernel: the
// extra live state there cost 0.12 ms per launch (spills in the edge loop), these two launches cost ~5 us.
__global__ void __launch_bounds__(256) rel_census_kernel(const uint8_t* __restrict__ etype, long long E, int* __restrict__ rel_info) {
  __shared__ unsigned bits[8];
  if (threadIdx.x < 8) bits[threadIdx.x] = 0u;
  __syncthreads();
  unsigned lo = 0u;
  auto see = [&](unsigned t) {
    if (t < 32u) lo |= 1u << t;
    else atomicOr(&bits[t >> 5], 1u << (t & 31u));
  };
  const long long nvec = aligned16(etype) ? E >> 4 : 0;       // (an unaligned caller buffer takes the scalar tail loop)
  const uint4* v = reinterpret_cast<const uint4*>(etype);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    const uint4 x = __ldg(v + i);
    const unsigned w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) see((w[a] >> (8 * b)) & 0xffu);
  }
  if (blockIdx.x == 0)
    for (long long e = (nvec << 4) + threadIdx.x; e < E; e += blockDim.x) see(etype[e]);
  lo = __reduce_or_sync(0xffffffffu, lo);
  if ((threadIdx.x & 31) == 0 && lo) atomicOr(&bits[0], lo);
  __syncthreads();
  if ((bits[threadIdx.x >> 5] >> (threadIdx.x & 31)) & 1u) rel_info[1 + threadIdx.x] = 0;
}

// A caller that already knows which relation ids can occur (from the speaker ids on the host) supplies its own id -> slot
// table and does not wait for the census; this check raises ERCG_GRAPH_ECENSUS if an edge carries an id the table lacks.
__global__ void __launch_bounds__(256) rel_check_kernel(const int* __restrict__ allowed, int n_allowed, int* __restrict__ rel_info) {
  const int t = threadIdx.x;
  if (rel_info[1 + t] >= 0 && (t >= n_allowed || allowed[t] < 0)) atomicOr(rel_info + 513, 8);
}

__global__ void __launch_bounds__(256) rel_slots_kernel(int* __restrict__ rel_info) {
  __shared__ int wcnt[8];
  const int t = threadIdx.x, lane = t & 31;
  const bool here = rel_info[1 + t] >= 0;
  const unsigned m = __ballot_sync(0xffffffffu, here);
  if (lane == 0) wcnt[t >> 5] = __popc(m);
  __syncthreads();
  int slot = __popc(m & ((1u << lane) - 1u));
  for (int w = 0; w < (t >> 5); ++w) slot += wcnt[w];
  if (here) { rel_info[1 + t] = slot; rel_info[257 + slot] = t; }
  if (t == 0) { int c = 0; for (int w = 0; w < 8; ++w) c += wcnt[w]; rel_info[0] = c; }
}

__global__ void graphify_count_kernel(const void* lengths, int len64, int B, int wp, int wf, long long* totals) {
  __shared__ long long sm[66];
  long long n = 0, e = 0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    long long L = len64 ? reinterpret_cast<const long long*>(lengths)[b] : (long long)reinterpret_cast<const int*>(lengths)[b];
    if (L < 0) L = 0;
    n += L; e += dialog_edges(L, wp, wf);
  }
  block_scan_pair(n, e, sm);
  if (threadIdx.x == blockDim.x - 1) { totals[0] = n; totals[1] = e; }
}

__global__ void pack_rows_kernel(const float* __restrict__ padded, long long ld, long long Lmax, int B, int seq_first,
                                 const int* __restrict__ node_off, const int* __restrict__ node_dlg,
                                 float* __restrict__ packed, long long ldp, long long N, int D, int unpack) {
  // one warp per node row
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= N) return;
  const int d = node_dlg[row];
  const long long pos = row - node_off[d];
  const long long prow = seq_first ? pos * B + d : (long long)d * Lmax + pos;
  const float* src = padded + prow * ld;
  float* dst = packed + row * ldp;
  if (unpack) {
    float* pd = const_cast<float*>(padded) + prow * ld;
    for (int c = lane; c < D; c += 32) pd[c] = dst[c];
  } else {
    for (int c = lane; c < D; c += 32) dst[c] = src[c];
  }
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_graphify_sizes_host(const int64_t* lengths_host, int B, int wp, int wf, int64_t* N_out, int64_t* E_out) {
  if (B < 0 || (B > 0 && !lengths_host) || !N_out || !E_out) return ERCG_EINVAL;
  long long n = 0, e = 0;
  for (int b = 0; b < B; ++b) {
    long long L = lengths_host[b] < 0 ? 0 : lengths_host[b];
    n += L; e += dialog_edges(L, wp, wf);
  }
  *N_out = n; *E_out = e;
  return ERCG_OK;
}

extern "C" int ercg_graphify_count(const void* lengths_dev, int lengths_is_i64, int B, int wp, int wf,
                                   int64_t* totals_dev, void* stream) {
  if (B < 0 || !totals_dev || (B > 0 && !lengths_dev)) return ERCG_EINVAL;
  graphify_count_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(lengths_dev, lengths_is_i64, B, wp, wf,
                                                              reinterpret_cast<long long*>(totals_dev));
  return finish_launch();
}

extern "C" size_t ercg_graphify_workspace_bytes(int B) {
  size_t tiles = (size_t)(B > 0 ? (B + 255) / 256 : 1);
  return tiles * 2 * sizeof(long long);
}

extern "C" int ercg_graphify_csr(const void* lengths_dev, int lengths_is_i64, int B,
                                 const void* speakers_dev, int speakers_is_i64, int64_t spk_ld,
                                 int wp, int wf, int n_speakers, int64_t N, int64_t E,
                                 const ercg_graph_out* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!out || B < 0 || N < 0 || E < 0 || n_speakers < 1 || spk_ld < 0) return ERCG_EINVAL;
  if (!out->node_off || !out->edge_off || !out->rowptr || !out->col || !out->etype || !out->t_rowptr ||
      !out->t_col || !out->t_etype || !out->t_eid || !out->spk || !out->node_dlg) return ERCG_EINVAL;
  if (B > 0 && (!lengths_dev || !speakers_dev)) return ERCG_EINVAL;
  if (2LL * n_speakers * n_speakers > 256) return ERCG_ERANGE;       // etype is uint8
  if (N >= 2147483647LL || E >= 2147483647LL) return ERCG_ERANGE;    // packed int32 indices
  if (workspace_bytes < ercg_graphify_workspace_bytes(B) || !workspace) return ERCG_EWORKSPACE;
  GraphifyParams p;
  p.lengths = lengths_dev; p.len64 = lengths_is_i64; p.B = B;
  p.speakers = speakers_dev; p.spk64 = speakers_is_i64; p.spk_ld = spk_ld;
  p.wp = wp; p.wf = wf; p.n_speakers = n_speakers; p.N = N; p.E = E; p.o = *out;
  p.tile_agg = reinterpret_cast<long long*>(workspace);
  const int num_sms = device_sm_count();
  const int max_blocks_per_sm = resident_capacity<graphify_kernel>(256, 0);
  if (max_blocks_per_sm < 1) return ERCG_ECUDA;
  long long want = (B + 7) / 8;                       // one warp per dialogue
  long long cap = (long long)max_blocks_per_sm * num_sms;
  int grid = (int)(want < 1 ? 1 : (want > cap ? cap : want));
  if (int rc = launch_cooperative(graphify_kernel, grid, 256, 0, (cudaStream_t)stream, p)) return rc;
  if (out->rel_info) {
    if (E > 0) {
      const long long want_c = (E / 16 + 255) / 256;
      const unsigned gc = (unsigned)(want_c < 1 ? 1 : (want_c > 4LL * num_sms ? 4LL * num_sms : want_c));
      rel_census_kernel<<<gc, 256, 0, (cudaStream_t)stream>>>(out->etype, E, out->rel_info);
      int rc = finish_launch();
      if (rc) return rc;
    }
    rel_slots_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(out->rel_info);
    return finish_launch();
  }
  return ERCG_OK;
}

extern "C" int ercg_graphify_check_census(const int32_t* allowed_slots, int n_allowed, int32_t* rel_info, void* stream) {
  if (!allowed_slots || !rel_info || n_allowed < 0 || n_allowed > 256) return ERCG_EINVAL;
  rel_check_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(allowed_slots, n_allowed, rel_info);
  return finish_launch();
}

// ---- ERCCollate's small tensors, built on the device from the packed layout (track_mm/mmbase.py:354-371,417-428)
namespace ercg {
__global__ void __launch_bounds__(256)
collate_masks_kernel(const int* __restrict__ node_off, const long long* __restrict__ spk_packed, int B, long long Lmax, int seq_first,
                     int n_onehot, float* __restrict__ attention_mask, long long* __restrict__ speaker_ids, float* __restrict__ speaker_onehot) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)B * Lmax) return;
  const int b = (int)(idx / Lmax);
  const long long l = idx - (long long)b * Lmax;
  const int o = node_off[b], len = node_off[b + 1] - o;
  const bool in = l < len;
  if (attention_mask) attention_mask[idx] = in ? 1.f : 0.f;                       // always [B, Lmax] (mmbase.py:361-363)
  const long long s = in ? spk_packed[o + l] : 0;                                 // padding = speaker 0 (zeros().long(), :370)
  const long long pos = seq_first ? l * B + b : idx;                              // transposed when not batch_first (:422-423)
  if (speaker_ids) speaker_ids[pos] = s;
  if (speaker_onehot)
    for (int c = 0; c < n_onehot; ++c) speaker_onehot[pos * n_onehot + c] = c == s ? 1.f : 0.f;   // onehot(), :425-426
}
}  // namespace ercg

extern "C" int ercg_collate_masks(const int32_t* node_off, const int64_t* speaker_packed, int B, int64_t Lmax, int seq_first,
                                  int n_onehot, float* attention_mask, int64_t* speaker_ids, float* speaker_onehot, void* stream) {
  if (B < 0 || Lmax < 0 || n_onehot < 0) return ERCG_EINVAL;
  if (B == 0 || Lmax == 0) return ERCG_OK;
  if (!node_off || !speaker_packed || (speaker_onehot && n_onehot < 1)) return ERCG_EINVAL;
  const long long total = (long long)B * Lmax;
  collate_masks_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      node_off, reinterpret_cast<const long long*>(speaker_packed), B, Lmax, seq_first, n_onehot, attention_mask,
      reinterpret_cast<long long*>(speaker_ids), speaker_onehot);
  return finish_launch();
}

static int pack_launch(const float* padded, int64_t ld, int64_t Lmax, int B, int seq_first,
                       const int32_t* node_off, const int32_t* node_dlg, float* packed, int64_t ldp,
                       int64_t N, int D, int unpack, void* stream) {
  if (N < 0 || D < 0 || B < 0) return ERCG_EINVAL;
  if (N == 0 || D == 0) return ERCG_OK;
  if (!padded || !packed || !node_off || !node_dlg) return ERCG_EINVAL;
  const int wpb = 8;
  long long blocks = (N + wpb - 1) / wpb;
  pack_rows_kernel<<<(unsigned)blocks, wpb * 32, 0, (cudaStream_t)stream>>>(padded, ld, Lmax, B, seq_first, node_off,
                                                                            node_dlg, packed, ldp, N, D, unpack);
  return finish_launch();
}

extern "C" int ercg_pack_rows(const float* padded, int64_t ld, int64_t Lmax, int B, int seq_first,
                              const int32_t* node_off, const int32_t* node_dlg, float* packed, int64_t ldp,
                              int64_t N, int D, void* stream) {
  return pack_launch(padded, ld, Lmax, B, seq_first, node_off, node_dlg, packed, ldp, N, D, 0, stream);
}

extern "C" int ercg_unpack_rows(const float* packed, int64_t ldp, const int32_t* node_off, const int32_t* node_dlg,
                                float* padded, int64_t ld, int64_t Lmax, int B, int seq_first, int64_t N, int D,
                                void* stream) {
  return pack_launch(padded, ld, Lmax, B, seq_first, node_off, node_dlg, const_cast<float*>(packed), ldp, N, D, 1, stream);
}
