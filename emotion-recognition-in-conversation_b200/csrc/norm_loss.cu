// BatchNorm1d(training statistics) + LeakyReLU (track_mm/cogmen.py:67-68,72) and the (class-weighted)
// mean cross entropy of the train steps (cogmen.py:185, dgcn.py:124), forward and backward.
// All reductions are two-level with a fixed order (per-block partials, then one thread per column
// summing the partials in fp64) => bit-reproducible and independent of scheduling.
#include "common.cuh"
#include "col_stream.cuh"
#include "p2p_dev.cuh"
#include <math.h>

namespace ercg {

constexpr int RPB = 256;    // rows per block in the column reductions

// partial[b][0:H] = sum f0, partial[b][H:2H] = sum f1 over the block's rows
template <int MODE>   // 0: (x, x^2)   1: (dy, dy*xhat) with dy = dout * lrelu'(gamma*xhat+beta)
__global__ void __launch_bounds__(256)
col_partials_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ dout, long long ldo,
                    const float* __restrict__ mean, const float* __restrict__ var, float eps,
                    const float* __restrict__ gamma, const float* __restrict__ beta, float slope,
                    long long N, int H, float* __restrict__ partial) {
  __shared__ float sm0[8][33], sm1[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long rbeg = (long long)blockIdx.x * RPB;
  long long rend = rbeg + RPB;
  if (rend > N) rend = N;
  for (int c0 = 0; c0 < H; c0 += 32) {
    const int c = c0 + tx;
    float s0 = 0.f, s1 = 0.f;
    if (c < H) {
      float mu = 0.f, istd = 0.f, g = 0.f, b = 0.f;
      if (MODE == 1) { mu = mean[c]; istd = (1.0f / sqrtf(var[c] + eps)); g = gamma[c]; b = beta[c]; }
      const float shift = MODE == 0 ? x[c] : 0.f;   // row 0 as a per-column shift: kills the E[x^2]-E[x]^2 cancellation
      for (long long r = rbeg + ty; r < rend; r += 8) {
        const float xv = x[r * ldx + c];
        if (MODE == 0) {
          const float xs = xv - shift;
          s0 += xs; s1 = fmaf(xs, xs, s1);
        } else {
          const float xh = (xv - mu) * istd;
          const float z = fmaf(g, xh, b);
          const float dy = dout[r * ldo + c] * (z > 0.f ? 1.f : slope);
          s0 += dy; s1 = fmaf(dy, xh, s1);
        }
      }
    }
    sm0[ty][tx] = s0; sm1[ty][tx] = s1;
    __syncthreads();
    if (ty == 0 && c < H) {
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int y = 0; y < 8; ++y) { t0 += sm0[y][tx]; t1 += sm1[y][tx]; }
      partial[(long long)blockIdx.x * 2 * H + c] = t0;
      partial[(long long)blockIdx.x * 2 * H + H + c] = t1;
    }
    __syncthreads();
  }
}

// float4 version of the above for 16-byte aligned rows: one pass over the columns (H <= 128 per pass), each warp load
// covers a whole 400-byte row instead of one 128-byte line, rows unrolled x4 -> 4x the bytes in flight per warp.
// Same row-to-warp assignment and the same fixed summation order inside a lane; only the partial sums differ in rounding.
template <int MODE>
__global__ void __launch_bounds__(256)
col_partials_v4_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ dout, long long ldo,
                       const float* __restrict__ mean, const float* __restrict__ var, float eps,
                       const float* __restrict__ gamma, const float* __restrict__ beta, float slope,
                       long long N, int H, float* __restrict__ partial) {
  __shared__ float4 sm0[8][33], sm1[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long rbeg = (long long)blockIdx.x * RPB;
  long long rend = rbeg + RPB;
  if (rend > N) rend = N;
  for (int c0 = 0; c0 < H; c0 += 128) {
    const int c = c0 + 4 * tx;
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
    if (c < H) {
      float4 mu = s0, istd = s0, g = s0, b = s0, shift = s0;
      if (MODE == 1) {
        mu = ld4(mean + c); g = ld4(gamma + c); b = ld4(beta + c);
        const float4 vv = ld4(var + c);
        istd = make_float4(1.0f / sqrtf(vv.x + eps), 1.0f / sqrtf(vv.y + eps), 1.0f / sqrtf(vv.z + eps), 1.0f / sqrtf(vv.w + eps));
      } else {
        shift = ld4(x + c);                       // row 0 as a per-column shift
      }
      auto acc = [&](const float4& xv, const float4& dv) {
        if (MODE == 0) {
          const float4 xs = make_float4(xv.x - shift.x, xv.y - shift.y, xv.z - shift.z, xv.w - shift.w);
          s0.x += xs.x; s0.y += xs.y; s0.z += xs.z; s0.w += xs.w;
          s1.x = fmaf(xs.x, xs.x, s1.x); s1.y = fmaf(xs.y, xs.y, s1.y); s1.z = fmaf(xs.z, xs.z, s1.z); s1.w = fmaf(xs.w, xs.w, s1.w);
        } else {
          const float4 xh = make_float4((xv.x - mu.x) * istd.x, (xv.y - mu.y) * istd.y, (xv.z - mu.z) * istd.z, (xv.w - mu.w) * istd.w);
          const float4 dy = make_float4(dv.x * (fmaf(g.x, xh.x, b.x) > 0.f ? 1.f : slope), dv.y * (fmaf(g.y, xh.y, b.y) > 0.f ? 1.f : slope),
                                        dv.z * (fmaf(g.z, xh.z, b.z) > 0.f ? 1.f : slope), dv.w * (fmaf(g.w, xh.w, b.w) > 0.f ? 1.f : slope));
          s0.x += dy.x; s0.y += dy.y; s0.z += dy.z; s0.w += dy.w;
          s1.x = fmaf(dy.x, xh.x, s1.x); s1.y = fmaf(dy.y, xh.y, s1.y); s1.z = fmaf(dy.z, xh.z, s1.z); s1.w = fmaf(dy.w, xh.w, s1.w);
        }
      };
      long long r = rbeg + ty;
      for (; r + 24 < rend; r += 32) {
        float4 xv[4], dv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          xv[u] = ld4_stream(x + (r + 8 * u) * ldx + c);
          dv[u] = MODE == 1 ? ld4_stream(dout + (r + 8 * u) * ldo + c) : xv[u];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) acc(xv[u], dv[u]);
      }
      for (; r < rend; r += 8) {
        const float4 xv = ld4_stream(x + r * ldx + c);
        acc(xv, MODE == 1 ? ld4_stream(dout + r * ldo + c) : xv);
      }
    }
    sm0[ty][tx] = s0; sm1[ty][tx] = s1;
    __syncthreads();
    if (ty == 0 && c < H) {
      float4 t0 = make_float4(0.f, 0.f, 0.f, 0.f), t1 = t0;
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        const float4 a = sm0[y][tx], bq = sm1[y][tx];
        t0.x += a.x; t0.y += a.y; t0.z += a.z; t0.w += a.w;
        t1.x += bq.x; t1.y += bq.y; t1.z += bq.z; t1.w += bq.w;
      }
      float* p0 = partial + (long long)blockIdx.x * 2 * H + c;
      p0[0] = t0.x; p0[H] = t1.x;
      if (c + 1 < H) { p0[1] = t0.y; p0[H + 1] = t1.y; }
      if (c + 2 < H) { p0[2] = t0.z; p0[H + 2] = t1.z; }
      if (c + 3 < H) { p0[3] = t0.w; p0[H + 3] = t1.w; }
    }
    __syncthreads();
  }
}

// second level of the BatchNorm reductions: fin_reduce (common.cuh) over partial[nb][2H]
__global__ void __launch_bounds__(256)
bn_stats_final_kernel(const float* __restrict__ partial, int nb, int H, long long N,
                      const float* __restrict__ x, float* __restrict__ mean, float* __restrict__ var) {
  __shared__ double sm[FIN_ROWS][FIN_COLS + 1];
  const int c = blockIdx.x * FIN_COLS + (threadIdx.x & (FIN_COLS - 1));
  const bool ok = c < H;
  const double s0 = fin_reduce(partial, nb, 2 * H, c, ok, sm);
  const double s1 = fin_reduce(partial, nb, 2 * H, H + c, ok, sm);
  if (!ok || threadIdx.x >= FIN_COLS) return;
  const double m = s0 / (double)N;          // mean of (x - shift)
  double v = s1 / (double)N - m * m;
  if (v < 0.0) v = 0.0;
  mean[c] = (float)(m + (double)x[c]); var[c] = (float)v;
}

// Data-parallel BatchNorm statistics in ONE kernel: the second level of the column reduction (as bn_stats_final_kernel), the
// exchange of the per-rank statistics over peer memory (p2p_dev.cuh), the global mean / biased variance and the running
// statistics of nn.BatchNorm1d -- instead of final-reduce, pack, all-reduce, unpack and running-update launches in a row on
// the critical path of the forward pass.  A CTA owns FIN_COLS columns from the partial sums to the result: it stages
// (mean n, (var + mean^2) n) of its columns in this rank's region, raises its flag in every peer's region, waits for the
// peers' CTA of the same index and adds the W staged values in rank order.  Arithmetic = ercg_bn_stats (fp32 results) then
// ercg_bn_sync_pack / all-reduce / ercg_bn_sync_unpack in fp64, step by step, so the result equals the unfused path bit for
// bit (and is the same on every rank).  count = rows over all ranks (host-known).
__global__ void __launch_bounds__(256)
bn_stats_final_p2p_kernel(const float* __restrict__ partial, int nb, int H, long long N, const float* __restrict__ x,
                          unsigned char* const* __restrict__ regions, int rank, int world, size_t slot_bytes, double count,
                          float* __restrict__ mean, float* __restrict__ var, float* __restrict__ rmean, float* __restrict__ rvar,
                          long long* __restrict__ nbt, float momentum, unsigned long long timeout_ns) {
  __shared__ double sm[FIN_ROWS][FIN_COLS + 1];
  const int c = blockIdx.x * FIN_COLS + (threadIdx.x & (FIN_COLS - 1));
  const bool ok = c < H, owner = ok && threadIdx.x < FIN_COLS;
  const double s0 = fin_reduce(partial, nb, 2 * H, c, ok, sm);
  const double s1 = fin_reduce(partial, nb, 2 * H, H + c, ok, sm);
  const P2pCall k = p2p_begin(regions, rank, slot_bytes, timeout_ns);
  if (owner) {
    const double m = s0 / (double)N;
    double v = s1 / (double)N - m * m;
    if (v < 0.0) v = 0.0;
    const double md = (double)(float)(m + (double)x[c]), vd = (double)(float)v, n = (double)N;   // the fp32 local statistics
    double* mine = reinterpret_cast<double*>(regions[rank] + k.slot_off);
    mine[c] = __dmul_rn(md, n);
    mine[H + c] = __dmul_rn(__dadd_rn(vd, __dmul_rn(md, md)), n);
  }
  p2p_signal_wait(regions, rank, world, blockIdx.x, k);
  if (owner) {
    double a[P2P_MAX_WORLD], b[P2P_MAX_WORLD];
#pragma unroll
    for (int p = 0; p < P2P_MAX_WORLD; ++p)
      if (p < world) {
        const double* d = reinterpret_cast<const double*>(regions[p] + k.slot_off);
        a[p] = ld_peer(d + c);
        b[p] = ld_peer(d + H + c);
      }
    double sa = a[0], sb = b[0];
#pragma unroll
    for (int p = 1; p < P2P_MAX_WORLD; ++p)
      if (p < world) { sa += a[p]; sb += b[p]; }
    const double gm = __ddiv_rn(sa, count);
    const double gv = __dsub_rn(__ddiv_rn(sb, count), __dmul_rn(gm, gm));
    const float m32 = (float)gm, v32 = (float)(gv > 0.0 ? gv : 0.0);
    mean[c] = m32;
    var[c] = v32;
    if (rmean) {                                              // = bn_running_update_kernel
      const long long seen = nbt ? nbt[0] + 1 : 1;            // nbt is bumped below, after every CTA has passed this point
      const float mom = momentum >= 0.f ? momentum : (float)(1.0 / (double)seen);
      const float cf = (float)count;
      const float unbias = mom * cf / fmaxf(cf - 1.0f, 1.0f);
      rmean[c] = fmaf(mom, m32, rmean[c] * (1.0f - mom));
      rvar[c] = fmaf(unbias, v32, rvar[c] * (1.0f - mom));
    }
  }
  if (p2p_close_call(k, gridDim.x) && rmean && nbt) nbt[0] += 1;
}

__global__ void __launch_bounds__(256)
sums_final_kernel(const float* __restrict__ partial, int nb, int H, float* __restrict__ sums) {
  __shared__ double sm[FIN_ROWS][FIN_COLS + 1];
  const int c = blockIdx.x * FIN_COLS + (threadIdx.x & (FIN_COLS - 1));
  const bool ok = c < 2 * H;
  const double s = fin_reduce(partial, nb, 2 * H, c, ok, sm);
  if (ok && threadIdx.x < FIN_COLS) sums[c] = (float)s;
}

// explicit _rn intrinsics: no FMA contraction, so the values equal the elementwise fp64 expression they replace
__global__ void __launch_bounds__(256)
bn_sync_pack_kernel(const float* __restrict__ mean, const float* __restrict__ var, double n, int H, double* __restrict__ buf) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < H) {
    const double m = (double)mean[c];
    buf[c] = __dmul_rn(m, n);
    buf[H + c] = __dmul_rn(__dadd_rn((double)var[c], __dmul_rn(m, m)), n);
  } else if (c == H) {
    buf[2 * H] = n;
    buf[2 * H + 1] = 0.0;                 // pad: the buffer is an even number of doubles = whole 16-byte units
  }
}
__global__ void __launch_bounds__(256)
bn_sync_unpack_kernel(const double* __restrict__ buf, int H, float* __restrict__ mean, float* __restrict__ var) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= H) return;
  const double count = buf[2 * H];
  const double gm = __ddiv_rn(buf[c], count);
  const double gv = __dsub_rn(__ddiv_rn(buf[H + c], count), __dmul_rn(gm, gm));
  mean[c] = (float)gm;
  var[c] = (float)(gv > 0.0 ? gv : 0.0);
}

__global__ void __launch_bounds__(256)
bn_running_update_kernel(const float* __restrict__ mean, const float* __restrict__ var, float* __restrict__ rmean,
                         float* __restrict__ rvar, long long* __restrict__ nbt, float momentum, float count, int H) {
  const long long seen = nbt ? nbt[0] + 1 : 1;
  const float m = momentum >= 0.f ? momentum : (float)(1.0 / (double)seen);
  const float unbias = m * count / fmaxf(count - 1.0f, 1.0f);
  for (int c = threadIdx.x; c < H; c += 256) {
    rmean[c] = fmaf(m, mean[c], rmean[c] * (1.0f - m));
    rvar[c] = fmaf(unbias, var[c], rvar[c] * (1.0f - m));
  }
  __syncthreads();                       // every thread has read nbt[0]
  if (threadIdx.x == 0 && nbt) nbt[0] = seen;
}

// BatchNorm backward sums (sum dy, sum dy * xhat) fused with their exchange: second level of the column reduction, then the
// per-rank sums meet over peer memory; `sums` keeps this rank's own values (= its dbeta / dgamma, which travel with the
// gradient all-reduce later), `gsums` the rank-ordered total the input gradient needs.  = sums_final_kernel + all-reduce.
__global__ void __launch_bounds__(256)
sums_final_p2p_kernel(const float* __restrict__ partial, int nb, int H, unsigned char* const* __restrict__ regions, int rank,
                      int world, size_t slot_bytes, float* __restrict__ sums, float* __restrict__ gsums,
                      unsigned long long timeout_ns) {
  __shared__ double sm[FIN_ROWS][FIN_COLS + 1];
  const int c = blockIdx.x * FIN_COLS + (threadIdx.x & (FIN_COLS - 1));
  const bool ok = c < 2 * H, owner = ok && threadIdx.x < FIN_COLS;
  const double s = fin_reduce(partial, nb, 2 * H, c, ok, sm);
  const P2pCall k = p2p_begin(regions, rank, slot_bytes, timeout_ns);
  if (owner) {
    const float v = (float)s;
    sums[c] = v;
    reinterpret_cast<float*>(regions[rank] + k.slot_off)[c] = v;
  }
  p2p_signal_wait(regions, rank, world, blockIdx.x, k);
  if (owner) {
    float a[P2P_MAX_WORLD];
#pragma unroll
    for (int p = 0; p < P2P_MAX_WORLD; ++p)
      if (p < world) a[p] = ld_peer(reinterpret_cast<const float*>(regions[p] + k.slot_off) + c);
    float t = a[0];
#pragma unroll
    for (int p = 1; p < P2P_MAX_WORLD; ++p)
      if (p < world) t += a[p];
    gsums[c] = t;
  }
  p2p_close_call(k, gridDim.x);
}

__global__ void __launch_bounds__(256)
bn_act_fwd_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ mean,
                  const float* __restrict__ var, float eps, const float* __restrict__ gamma,
                  const float* __restrict__ beta, float slope, float* __restrict__ out, long long ldo,
                  long long N, int H) {
  const int nch = H >> 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nch) return;
  const long long r = idx / nch;
  const int c = (int)(idx % nch) * 4;
  const float4 xv = ld4(x + r * ldx + c), mu = ld4(mean + c), vv = ld4(var + c), g = ld4(gamma + c), b = ld4(beta + c);
  float4 y;
  y.x = fmaf(g.x, (xv.x - mu.x) * (1.0f / sqrtf(vv.x + eps)), b.x);
  y.y = fmaf(g.y, (xv.y - mu.y) * (1.0f / sqrtf(vv.y + eps)), b.y);
  y.z = fmaf(g.z, (xv.z - mu.z) * (1.0f / sqrtf(vv.z + eps)), b.z);
  y.w = fmaf(g.w, (xv.w - mu.w) * (1.0f / sqrtf(vv.w + eps)), b.w);
  y.x = y.x > 0.f ? y.x : y.x * slope; y.y = y.y > 0.f ? y.y : y.y * slope;
  y.z = y.z > 0.f ? y.z : y.z * slope; y.w = y.w > 0.f ? y.w : y.w * slope;
  st4(out + r * ldo + c, y);
}

__global__ void __launch_bounds__(256)
bn_act_bwd_apply_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ x, long long ldx,
                        const float* __restrict__ mean, const float* __restrict__ var, float eps,
                        const float* __restrict__ gamma, const float* __restrict__ beta, float slope,
                        const float* __restrict__ sums, float inv_count, int use_batch_stats,
                        float* __restrict__ dx, long long lddx, long long N, int H) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * H) return;
  const long long r = idx / H;
  const int c = (int)(idx % H);
  const float istd = (1.0f / sqrtf(var[c] + eps)), g = gamma[c];
  const float xh = (x[r * ldx + c] - mean[c]) * istd;
  const float z = fmaf(g, xh, beta[c]);
  const float dy = dout[r * ldo + c] * (z > 0.f ? 1.f : slope);
  float v = dy;
  if (use_batch_stats) v = dy - sums[c] * inv_count - xh * (sums[H + c] * inv_count);
  dx[r * lddx + c] = g * istd * v;
}

__global__ void __launch_bounds__(256)
bn_act_bwd_apply_v4_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ x, long long ldx,
                           const float* __restrict__ mean, const float* __restrict__ var, float eps,
                           const float* __restrict__ gamma, const float* __restrict__ beta, float slope,
                           const float* __restrict__ sums, float inv_count, int use_batch_stats,
                           float* __restrict__ dx, long long lddx, long long N, int H) {
  const int nch = H >> 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * nch) return;
  const long long r = idx / nch;
  const int c = (int)(idx % nch) * 4;
  const float4 xv = ld4_stream(x + r * ldx + c), dv = ld4_stream(dout + r * ldo + c);
  const float4 mu = ld4(mean + c), vv = ld4(var + c), g = ld4(gamma + c), b = ld4(beta + c);
  float4 sa = make_float4(0.f, 0.f, 0.f, 0.f), sb = sa;
  if (use_batch_stats) { sa = ld4(sums + c); sb = ld4(sums + H + c); }
  auto one = [&](float xe, float de, float m, float v, float ge, float be, float s0, float s1) {
    const float istd = 1.0f / sqrtf(v + eps);
    const float xh = (xe - m) * istd;
    const float dy = de * (fmaf(ge, xh, be) > 0.f ? 1.f : slope);
    float t = dy;
    if (use_batch_stats) t = dy - s0 * inv_count - xh * (s1 * inv_count);
    return ge * istd * t;
  };
  st4_stream(dx + r * lddx + c, make_float4(one(xv.x, dv.x, mu.x, vv.x, g.x, b.x, sa.x, sb.x), one(xv.y, dv.y, mu.y, vv.y, g.y, b.y, sa.y, sb.y),
                                            one(xv.z, dv.z, mu.z, vv.z, g.z, b.z, sa.z, sb.z), one(xv.w, dv.w, mu.w, vv.w, g.w, b.w, sa.w, sb.w)));
}

// ------------------------------------------------------------------------------------------- CE
__global__ void __launch_bounds__(256)
ce_fwd_kernel(const float* __restrict__ logits, long long ld, const long long* __restrict__ labels,
              const float* __restrict__ cw, float* __restrict__ dlogits, long long ldd, long long N, int C,
              float* __restrict__ partial /* [blocks][2] */) {
  __shared__ float s0[256], s1[256];
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float num = 0.f, den = 0.f;
  if (i < N) {
    const float* z = logits + i * ld;
    float m = z[0];
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(z[c] - m);
    const float lse = m + logf(se);
    long long y = labels[i];
    const bool ok = y >= 0 && y < C;
    const float w = ok ? (cw ? cw[y] : 1.f) : 0.f;
    if (ok) { num = w * (lse - z[y]); den = w; }
    // a label outside [0, C) that is not F.cross_entropy's ignore_index (-100) is an input error (ATen raises a device
    // assert): poison the loss with NaN instead of silently giving the row weight 0
    else if (y != -100) num = __int_as_float(0x7fc00000);
    if (dlogits) {
      const float inv = 1.f / se;
      for (int c = 0; c < C; ++c) {
        const float p = expf(z[c] - m) * inv;
        dlogits[i * ldd + c] = w * (p - (c == y ? 1.f : 0.f));
      }
    }
  }
  s0[threadIdx.x] = num; s1[threadIdx.x] = den;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { s0[threadIdx.x] += s0[threadIdx.x + o]; s1[threadIdx.x] += s1[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { partial[2 * (long long)blockIdx.x] = s0[0]; partial[2 * (long long)blockIdx.x + 1] = s1[0]; }
}

__global__ void __launch_bounds__(256)
ce_final_kernel(const float* __restrict__ partial, long long nb, float* __restrict__ out) {
  // fixed order: thread-strided fp64 sums (256 threads: 16 loads per thread for 4096 partials, not 128 on one warp), a fixed
  // shuffle tree per warp, then the 8 warp sums in warp order
  __shared__ double sa[8], sb[8];
  double a = 0.0, b = 0.0;
  for (long long i = threadIdx.x; i < nb; i += 256) { a += (double)partial[2 * i]; b += (double)partial[2 * i + 1]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  if ((threadIdx.x & 31) == 0) { sa[threadIdx.x >> 5] = a; sb[threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0.0, tb = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) { ta += sa[w]; tb += sb[w]; }
    out[0] = (float)ta; out[1] = (float)tb;
  }
}

__global__ void scale_by_ratio_kernel(float* __restrict__ x, long long n, const float* __restrict__ num,
                                      const float* __restrict__ den) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] *= num[0] / den[0];
}

__global__ void mask_pos_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ ref, long long ldr,
                                float scale, float* __restrict__ out, long long ldo, long long M, int N) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * N) return;
  const long long r = idx / N;
  const int c = (int)(idx % N);
  out[r * ldo + c] = ref[r * ldr + c] > 0.f ? x[r * ldx + c] * scale : 0.f;
}

__global__ void __launch_bounds__(256)
mask_pos_v4_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ ref, long long ldr, float scale,
                   float* __restrict__ out, long long ldo, long long M, int N) {
  const int nch = N >> 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * nch) return;
  const long long r = idx / nch;
  const int c = (int)(idx % nch) * 4;
  const float4 xv = ld4_stream(x + r * ldx + c), rv = ld4_stream(ref + r * ldr + c);
  st4_stream(out + r * ldo + c, make_float4(rv.x > 0.f ? xv.x * scale : 0.f, rv.y > 0.f ? xv.y * scale : 0.f,
                                            rv.z > 0.f ? xv.z * scale : 0.f, rv.w > 0.f ? xv.w * scale : 0.f));
}

static inline bool v4_ok(const void* p, long long ld) { return aligned16(p) && (ld & 3) == 0; }

// ---------------------------------------------------------------------------------- classifier tail, backward
// cls = Linear(100,100) -> ReLU -> Dropout -> Linear(100,C) (track_mm/cogmen.py:116-122; dgcn_models.py:158-167).  Given the
// gradient of the logits, ONE pass over the hidden activations h [N,K] (post ReLU/dropout, K <= 128) produces everything
// the last Linear and the activation need:
//   dZ[m,:]  = (h[m,:] > 0 ? scale : 0) * (dl[m,:] @ W3)          gradient of the first Linear's pre-activation
//   dW3[c,k] = sum_m dl[m,c] * h[m,k],   db3[c] = sum_m dl[m,c],   db0[k] = sum_m dZ[m,k]
// instead of five launches (skinny TN, skinny NN, mask, two column sums) that read h or dZ again each time.
// One warp per row, lane = float4 chunk of the row: every sum is column-parallel, so the inner loop has no shuffle at
// all; rows are dealt to warps grid-stride and block partials are added in a fixed order => bit-reproducible.
constexpr int CT_MAXC = 8;
template <int C>
__global__ void __launch_bounds__(256)
cls_tail_bwd_kernel(const float* __restrict__ h, long long ldh, const float* __restrict__ dl /* [N,C] contiguous */,
                    const float* __restrict__ W3 /* [C,K] row-major (nn.Linear weight) */, float scale,
                    float* __restrict__ dZ, long long ldz, long long N, int K,
                    float* __restrict__ partial /* [gridDim.x][C*K + K + CT_MAXC] */) {
  __shared__ float4 red[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nch = K >> 2;
  const bool on = lane < nch;
  float4 w[C];
#pragma unroll
  for (int c = 0; c < C; ++c) w[c] = on ? ld4(W3 + (long long)c * K + 4 * lane) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 dw[C];
#pragma unroll
  for (int c = 0; c < C; ++c) dw[c] = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 cz = make_float4(0.f, 0.f, 0.f, 0.f);
  float cl = 0.f;                                            // lane c < C keeps sum_m dl[m,c]
  const long long stride = (long long)gridDim.x * 8;
  for (long long m0 = (long long)blockIdx.x * 8 + warp; m0 < N; m0 += 4 * stride) {
    float4 hv[4];
    float dv[4][C];
    bool ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long m = m0 + u * stride;
      ok[u] = m < N;
      hv[u] = (ok[u] && on) ? ld4_stream(h + m * ldh + 4 * lane) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int c = 0; c < C; ++c) dv[u][c] = ok[u] ? __ldg(dl + m * C + c) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (!ok[u]) continue;                                  // warp-uniform
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        fma4(g, dv[u][c], w[c]);
        fma4(dw[c], dv[u][c], hv[u]);
      }
      g.x = hv[u].x > 0.f ? g.x * scale : 0.f; g.y = hv[u].y > 0.f ? g.y * scale : 0.f;
      g.z = hv[u].z > 0.f ? g.z * scale : 0.f; g.w = hv[u].w > 0.f ? g.w * scale : 0.f;
      cz.x += g.x; cz.y += g.y; cz.z += g.z; cz.w += g.w;
      if (on) st4_stream(dZ + (m0 + u * stride) * ldz + 4 * lane, g);
      if (lane < C) {
        float mine = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) if (lane == c) mine = dv[u][c];
        cl += mine;
      }
    }
  }
  // block partial = warps added in warp order (through shared memory, one quantity at a time)
  float* out = partial + (long long)blockIdx.x * (C * K + K + CT_MAXC);
  auto reduce_store = [&](float4 v, float* dst) {
    __syncthreads();
    red[warp][lane] = v;
    __syncthreads();
    if (warp == 0 && on) {
      float4 t = red[0][lane];
#pragma unroll
      for (int q = 1; q < 8; ++q) { const float4 x = red[q][lane]; t.x += x.x; t.y += x.y; t.z += x.z; t.w += x.w; }
      st4(dst + 4 * lane, t);
    }
  };
#pragma unroll
  for (int c = 0; c < C; ++c) reduce_store(dw[c], out + c * K);
  reduce_store(cz, out + C * K);
  __syncthreads();
  red[warp][lane] = make_float4(cl, 0.f, 0.f, 0.f);
  __syncthreads();
  if (warp == 0 && lane < CT_MAXC) {
    float t = 0.f;
    if (lane < C)
      for (int q = 0; q < 8; ++q) t += red[q][lane].x;
    out[C * K + K + lane] = t;
  }
}

// fixed-order fp64 sum of the block partials [nb][width]; columns [0,CK) -> dW3, [CK,CK+K) -> db0, then C values -> db3
__global__ void __launch_bounds__(256)
cls_tail_final_kernel(const float* __restrict__ partial, int nb, int width, int CK, int K, int C, float* __restrict__ dW3,
                      float* __restrict__ db0, float* __restrict__ db3) {
  __shared__ double sm[FIN_ROWS][FIN_COLS + 1];
  const int c = blockIdx.x * FIN_COLS + (threadIdx.x & (FIN_COLS - 1));
  const bool ok = c < CK + K + C;
  const double s = fin_reduce(partial, nb, width, c, ok, sm);
  if (!ok || threadIdx.x >= FIN_COLS) return;
  if (c < CK) dW3[c] = (float)s;
  else if (c < CK + K) db0[c - CK] = (float)s;
  else db3[c - CK - K] = (float)s;
}

// ---------------------------------------------------------------------------------- log-softmax over the columns of a row
// F.log_softmax(x, dim=-1) of the sequence classifiers' heads: y = x - max - log(sum exp(x - max)); backward
// dx = dy - exp(y) * sum dy.  One warp per row, lanes over the columns (any C), fixed-order warp sums.
__global__ void __launch_bounds__(256)
log_softmax_fwd_kernel(const float* __restrict__ x, long long ldx, float* __restrict__ y, long long ldy, long long rows, int C) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + r * ldx;
  float m = -INFINITY;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, xr[c]);
  m = warp_max(m);
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += expf(xr[c] - m);
  const float ls = logf(warp_sum(s));
  for (int c = lane; c < C; c += 32) y[r * ldy + c] = xr[c] - m - ls;
}

__global__ void __launch_bounds__(256)
log_softmax_bwd_kernel(const float* __restrict__ y, long long ldy, const float* __restrict__ dy, long long lddy,
                       float* __restrict__ dx, long long lddx, long long rows, int C) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += dy[r * lddy + c];
  s = warp_sum(s);
  for (int c = lane; c < C; c += 32) dx[r * lddx + c] = dy[r * lddy + c] - expf(y[r * ldy + c]) * s;
}

}  // namespace ercg

using namespace ercg;

extern "C" int ercg_mask_pos(const float* x, int64_t ldx, const float* ref, int64_t ldr, float scale,
                             float* out, int64_t ldo, int64_t M, int N, void* stream) {
  if (M < 0 || N < 0) return ERCG_EINVAL;
  if (M == 0 || N == 0) return ERCG_OK;
  if (!x || !ref || !out) return ERCG_EINVAL;
  const long long tot = M * N;
  if ((N & 3) == 0 && v4_ok(x, ldx) && v4_ok(ref, ldr) && v4_ok(out, ldo)) {
    mask_pos_v4_kernel<<<(unsigned)((tot / 4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, ref, ldr, scale, out, ldo, M, N);
    return finish_launch();
  }
  mask_pos_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, ref, ldr, scale, out, ldo, M, N);
  return finish_launch();
}

extern "C" size_t ercg_bn_workspace_bytes(int64_t N, int H) {
  if (N <= 0 || H <= 0) return 0;
  const size_t a = (size_t)((N + RPB - 1) / RPB) * 2 * H * sizeof(float), b = (size_t)CS_MAX_BLOCKS * 2 * H * sizeof(float);
  return a > b ? a : b;
}

// first level of the BatchNorm statistics: per-block partial sums of (x - x[0,c]) and its square -> part[nb][2H]
static int bn_stats_partials(const float* x, int64_t ldx, int64_t N, int H, float* part, cudaStream_t st) {
  int nb = (int)((N + RPB - 1) / RPB);
  if (col_stream_ok(x, ldx, H, N)) {      // contiguous rows: flat float4 stream, every lane busy
    const long long total4 = N * (long long)(H >> 2);
    nb = col_stream_blocks(H >> 2, total4);
    col_stream_kernel<0><<<nb, 256, 0, st>>>(x, nullptr, nullptr, nullptr, 0.f, nullptr, nullptr, 0.f, total4, H >> 2, part);
  } else if (v4_ok(x, ldx))
    col_partials_v4_kernel<0><<<nb, 256, 0, st>>>(x, ldx, nullptr, 0, nullptr, nullptr, 0.f, nullptr, nullptr, 0.f, N, H, part);
  else
    col_partials_kernel<0><<<nb, 256, 0, st>>>(x, ldx, nullptr, 0, nullptr, nullptr, 0.f, nullptr, nullptr, 0.f, N, H, part);
  return nb;
}

extern "C" int ercg_bn_stats(const float* x, int64_t ldx, int64_t N, int H, float* mean, float* var,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (N <= 0 || H <= 0 || !x || !mean || !var || ldx < H) return ERCG_EINVAL;
  if (workspace_bytes < ercg_bn_workspace_bytes(N, H) || !workspace) return ERCG_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>(workspace);
  const int nb = bn_stats_partials(x, ldx, N, H, part, st);
  int rc = finish_launch();
  if (rc) return rc;
  bn_stats_final_kernel<<<fin_blocks(H), 256, 0, st>>>(part, nb, H, N, x, mean, var);
  return finish_launch();
}

extern "C" int ercg_p2p_bn_stats(void* const* regions_dev, int rank, int world, const float* x, int64_t ldx, int64_t N, int H,
                                 double count_global, float* mean, float* var, float* running_mean, float* running_var,
                                 int64_t* num_batches_tracked, float momentum, void* workspace, size_t workspace_bytes,
                                 size_t max_bytes, void* stream) {
  if (!regions_dev || world < 1 || world > P2P_MAX_WORLD || rank < 0 || rank >= world) return ERCG_EINVAL;
  if (N <= 0 || H <= 0 || !x || !mean || !var || ldx < H || !(count_global >= (double)N)) return ERCG_EINVAL;
  if ((running_mean == nullptr) != (running_var == nullptr)) return ERCG_EINVAL;
  if (running_mean && momentum < 0.f && !num_batches_tracked) return ERCG_EINVAL;
  if (fin_blocks(H) > (unsigned)P2P_MAX_CTAS) return ERCG_ERANGE;          // one flag word per CTA
  const size_t slot = (max_bytes + 255) / 256 * 256;
  if ((size_t)2 * H * sizeof(double) > slot) return ERCG_EWORKSPACE;
  if (workspace_bytes < ercg_bn_workspace_bytes(N, H) || !workspace) return ERCG_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>(workspace);
  const int nb = bn_stats_partials(x, ldx, N, H, part, st);
  int rc = finish_launch();
  if (rc) return rc;
  bn_stats_final_p2p_kernel<<<fin_blocks(H), 256, 0, st>>>(part, nb, H, N, x, reinterpret_cast<unsigned char* const*>(regions_dev),
                                                          rank, world, slot, count_global, mean, var, running_mean, running_var,
                                                          reinterpret_cast<long long*>(num_batches_tracked), momentum, p2p_timeout_ns());
  return finish_launch();
}

extern "C" int ercg_bn_running_update(const float* mean, const float* var, float* running_mean, float* running_var,
                                      int64_t* num_batches_tracked, float momentum, float count, int H, void* stream) {
  if (H <= 0 || H > 1024 || !mean || !var || !running_mean || !running_var) return ERCG_EINVAL;
  if (momentum < 0.f && !num_batches_tracked) return ERCG_EINVAL;
  bn_running_update_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(mean, var, running_mean, running_var,
                                                                reinterpret_cast<long long*>(num_batches_tracked), momentum, count, H);
  return finish_launch();
}

extern "C" int ercg_bn_sync_pack(const float* mean, const float* var, double n_local, int H, double* buf, void* stream) {
  if (H <= 0 || !mean || !var || !buf) return ERCG_EINVAL;
  bn_sync_pack_kernel<<<(H + 1 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(mean, var, n_local, H, buf);
  return finish_launch();
}
extern "C" int ercg_bn_sync_unpack(const double* buf, int H, float* mean, float* var, void* stream) {
  if (H <= 0 || !mean || !var || !buf) return ERCG_EINVAL;
  bn_sync_unpack_kernel<<<(H + 255) / 256, 256, 0, (cudaStream_t)stream>>>(buf, H, mean, var);
  return finish_launch();
}

extern "C" int ercg_bn_act_fwd(const float* x, int64_t ldx, const float* mean, const float* var, float eps,
                               const float* gamma, const float* beta, float slope,
                               float* out, int64_t ldo, int64_t N, int H, void* stream) {
  if (N < 0 || H <= 0 || (H & 3)) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!x || !mean || !var || !gamma || !beta || !out) return ERCG_EINVAL;
  if ((ldx & 3) || (ldo & 3) || !aligned16(x) || !aligned16(out) || !aligned16(mean) || !aligned16(var) ||
      !aligned16(gamma) || !aligned16(beta)) return ERCG_EALIGN;
  const long long tot = N * (H >> 2);
  bn_act_fwd_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, mean, var, eps, gamma, beta,
                                                                                     slope, out, ldo, N, H);
  return finish_launch();
}

// first level of the BatchNorm backward sums -> part[nb][2H]
static int bn_bwd_partials(const float* dout, int64_t ldo, const float* x, int64_t ldx, const float* mean, const float* var,
                           float eps, const float* gamma, const float* beta, float slope, int64_t N, int H, float* part,
                           cudaStream_t st) {
  int nb = (int)((N + RPB - 1) / RPB);
  if (col_stream_ok(x, ldx, H, N) && col_stream_ok(dout, ldo, H, N) && aligned16(mean) && aligned16(var) && aligned16(gamma) &&
      aligned16(beta)) {
    const long long total4 = N * (long long)(H >> 2);
    nb = col_stream_blocks(H >> 2, total4);
    col_stream_kernel<1><<<nb, 256, 0, st>>>(x, dout, mean, var, eps, gamma, beta, slope, total4, H >> 2, part);
  } else {
    // (the row-per-warp float4 variant measured slower for this two-input mode: 0.33 vs 0.29 ms at 2^20 x 100)
    col_partials_kernel<1><<<nb, 256, 0, st>>>(x, ldx, dout, ldo, mean, var, eps, gamma, beta, slope, N, H, part);
  }
  return nb;
}

extern "C" int ercg_bn_act_bwd_reduce(const float* dout, int64_t ldo, const float* x, int64_t ldx,
                                      const float* mean, const float* var, float eps,
                                      const float* gamma, const float* beta, float slope,
                                      float* sums, int64_t N, int H, void* workspace, size_t workspace_bytes, void* stream) {
  if (N <= 0 || H <= 0 || !dout || !x || !mean || !var || !gamma || !beta || !sums) return ERCG_EINVAL;
  if (workspace_bytes < ercg_bn_workspace_bytes(N, H) || !workspace) return ERCG_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>(workspace);
  const int nb = bn_bwd_partials(dout, ldo, x, ldx, mean, var, eps, gamma, beta, slope, N, H, part, st);
  int rc = finish_launch();
  if (rc) return rc;
  sums_final_kernel<<<fin_blocks(2 * H), 256, 0, st>>>(part, nb, H, sums);
  return finish_launch();
}

extern "C" int ercg_p2p_bn_act_bwd_reduce(void* const* regions_dev, int rank, int world, const float* dout, int64_t ldo,
                                          const float* x, int64_t ldx, const float* mean, const float* var, float eps,
                                          const float* gamma, const float* beta, float slope, float* sums, float* sums_global,
                                          int64_t N, int H, void* workspace, size_t workspace_bytes, size_t max_bytes,
                                          void* stream) {
  if (!regions_dev || world < 1 || world > P2P_MAX_WORLD || rank < 0 || rank >= world) return ERCG_EINVAL;
  if (N <= 0 || H <= 0 || !dout || !x || !mean || !var || !gamma || !beta || !sums || !sums_global) return ERCG_EINVAL;
  if (fin_blocks(2 * H) > (unsigned)P2P_MAX_CTAS) return ERCG_ERANGE;      // one flag word per CTA
  const size_t slot = (max_bytes + 255) / 256 * 256;
  if ((size_t)2 * H * sizeof(float) > slot) return ERCG_EWORKSPACE;
  if (workspace_bytes < ercg_bn_workspace_bytes(N, H) || !workspace) return ERCG_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>(workspace);
  const int nb = bn_bwd_partials(dout, ldo, x, ldx, mean, var, eps, gamma, beta, slope, N, H, part, st);
  int rc = finish_launch();
  if (rc) return rc;
  sums_final_p2p_kernel<<<fin_blocks(2 * H), 256, 0, st>>>(part, nb, H, reinterpret_cast<unsigned char* const*>(regions_dev), rank,
                                                          world, slot, sums, sums_global, p2p_timeout_ns());
  return finish_launch();
}

extern "C" int ercg_bn_act_bwd_apply(const float* dout, int64_t ldo, const float* x, int64_t ldx,
                                     const float* mean, const float* var, float eps,
                                     const float* gamma, const float* beta, float slope,
                                     const float* sums, double count, int use_batch_stats,
                                     float* dx, int64_t lddx, int64_t N, int H, void* stream) {
  if (N < 0 || H <= 0) return ERCG_EINVAL;
  if (N == 0) return ERCG_OK;
  if (!dout || !x || !mean || !var || !gamma || !beta || !dx || (use_batch_stats && (!sums || count <= 0))) return ERCG_EINVAL;
  const long long tot = N * H;
  if ((H & 3) == 0 && v4_ok(dout, ldo) && v4_ok(x, ldx) && v4_ok(dx, lddx) && aligned16(mean) && aligned16(var) &&
      aligned16(gamma) && aligned16(beta) && (!use_batch_stats || aligned16(sums))) {
    bn_act_bwd_apply_v4_kernel<<<(unsigned)((tot / 4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        dout, ldo, x, ldx, mean, var, eps, gamma, beta, slope, sums, use_batch_stats ? (float)(1.0 / count) : 0.f,
        use_batch_stats, dx, lddx, N, H);
    return finish_launch();
  }
  bn_act_bwd_apply_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      dout, ldo, x, ldx, mean, var, eps, gamma, beta, slope, sums, use_batch_stats ? (float)(1.0 / count) : 0.f,
      use_batch_stats, dx, lddx, N, H);
  return finish_launch();
}

extern "C" size_t ercg_ce_workspace_bytes(int64_t N) {
  if (N <= 0) return 2 * sizeof(float);
  return (size_t)((N + 255) / 256) * 2 * sizeof(float);
}

extern "C" int ercg_ce_fwd(const float* logits, int64_t ld, const int64_t* labels, const float* class_weight,
                           float* lossnum_den, float* dlogits, int64_t ldd, int64_t N, int C,
                           void* workspace, size_t workspace_bytes, void* stream) {
  if (N <= 0 || C <= 0 || !logits || !labels || !lossnum_den || ld < C || (dlogits && ldd < C)) return ERCG_EINVAL;
  if (workspace_bytes < ercg_ce_workspace_bytes(N) || !workspace) return ERCG_EWORKSPACE;
  const long long nb = (N + 255) / 256;
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>(workspace);
  ce_fwd_kernel<<<(unsigned)nb, 256, 0, st>>>(logits, ld, reinterpret_cast<const long long*>(labels), class_weight, dlogits,
                                             ldd, N, C, part);
  int rc = finish_launch();
  if (rc) return rc;
  ce_final_kernel<<<1, 256, 0, st>>>(part, nb, lossnum_den);
  return finish_launch();
}

extern "C" int ercg_scale_by_ratio(float* x, int64_t n, const float* num, const float* den, void* stream) {
  if (n < 0) return ERCG_EINVAL;
  if (n == 0) return ERCG_OK;
  if (!x || !num || !den) return ERCG_EINVAL;
  scale_by_ratio_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, n, num, den);
  return finish_launch();
}

extern "C" size_t ercg_cls_tail_bwd_workspace_bytes(int K, int C) {
  if (K <= 0 || C <= 0) return 0;
  return (size_t)kNumSMs * 4 * ((size_t)C * K + K + CT_MAXC) * sizeof(float);
}

// see cls_tail_bwd_kernel.  dW3 [C,K], db3 [C], db0 [K] are written; dZ [N,K] (row pitch ldz).  K % 4 == 0, K <= 128, C <= 8.
extern "C" int ercg_cls_tail_bwd(const float* h, int64_t ldh, const float* dlogits, const float* W3, float scale,
                                 float* dZ, int64_t ldz, float* dW3, float* db3, float* db0, int64_t N, int K, int C,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (N < 0 || K <= 0 || (K & 3) || K > 128 || C < 1 || C > CT_MAXC) return ERCG_EINVAL;
  if (!dW3 || !db3 || !db0) return ERCG_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) {
    cudaMemsetAsync(dW3, 0, (size_t)C * K * sizeof(float), st);
    cudaMemsetAsync(db3, 0, (size_t)C * sizeof(float), st);
    cudaMemsetAsync(db0, 0, (size_t)K * sizeof(float), st);
    return ERCG_OK;
  }
  if (!h || !dlogits || !W3 || !dZ || ldh < K || ldz < K) return ERCG_EINVAL;
  if (!v4_ok(h, ldh) || !v4_ok(dZ, ldz) || !aligned16(W3)) return ERCG_EALIGN;
  if (workspace_bytes < ercg_cls_tail_bwd_workspace_bytes(K, C) || !workspace) return ERCG_EWORKSPACE;
  long long want = (N + 31) / 32;
  const int grid = (int)(want < 1 ? 1 : (want > 4LL * kNumSMs ? 4LL * kNumSMs : want));
  float* part = reinterpret_cast<float*>(workspace);
  const int width = C * K + K + CT_MAXC;
  switch (C) {
#define ERCG_CT_CASE(c) case c: cls_tail_bwd_kernel<c><<<grid, 256, 0, st>>>(h, ldh, dlogits, W3, scale, dZ, ldz, N, K, part); break;
    ERCG_CT_CASE(1) ERCG_CT_CASE(2) ERCG_CT_CASE(3) ERCG_CT_CASE(4) ERCG_CT_CASE(5) ERCG_CT_CASE(6) ERCG_CT_CASE(7) ERCG_CT_CASE(8)
#undef ERCG_CT_CASE
  }
  int rc = finish_launch();
  if (rc) return rc;
  cls_tail_final_kernel<<<fin_blocks(width), 256, 0, st>>>(part, grid, width, C * K, K, C, dW3, db0, db3);
  return finish_launch();
}

extern "C" int ercg_log_softmax_fwd(const float* x, int64_t ldx, float* y, int64_t ldy, int64_t rows, int C, void* stream) {
  if (rows < 0 || C < 1 || ldx < C || ldy < C) return ERCG_EINVAL;
  if (rows == 0) return ERCG_OK;
  if (!x || !y) return ERCG_EINVAL;
  log_softmax_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, ldx, y, ldy, rows, C);
  return finish_launch();
}

extern "C" int ercg_log_softmax_bwd(const float* y, int64_t ldy, const float* dy, int64_t lddy, float* dx, int64_t lddx,
                                    int64_t rows, int C, void* stream) {
  if (rows < 0 || C < 1 || ldy < C || lddy < C || lddx < C) return ERCG_EINVAL;
  if (rows == 0) return ERCG_OK;
  if (!y || !dy || !dx) return ERCG_EINVAL;
  log_softmax_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(y, ldy, dy, lddy, dx, lddx, rows, C);
  return finish_launch();
}
