// Shared helpers for the libercgraph kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <stdint.h>
#include "../../include/ercgraph.h"

namespace ercg {

extern std::atomic<unsigned long long> g_launches;   // counted on the host side, one per kernel launch (any thread)

inline int finish_launch() {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return cudaPeekAtLastError() == cudaSuccess ? ERCG_OK : ERCG_ECUDA;
}

__host__ __device__ inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// streaming variants: data touched once, keep it out of L1
__device__ __forceinline__ float4 ld4_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st4_stream(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
}
__device__ __forceinline__ void fma4(float4& a, float s, const float4& b) {
  a.x = fmaf(s, b.x, a.x); a.y = fmaf(s, b.y, a.y); a.z = fmaf(s, b.z, a.z); a.w = fmaf(s, b.w, a.w);
}
// Packed variants.  sm_100a has a packed fp32 FMA (fma.rn.f32x2 -> SASS FFMA2, one operand may be a broadcast scalar): two
// IEEE FMAs per issue slot, bit-identical to two fmaf.  It does not raise the FMA pipe's peak, it halves the issue slots of
// a weighted-sum / dot-product loop.  Measured on the graph kernels (tools/bench_graph.py, 2^20 nodes; DESIGN.md 7): window
// attention forward 0.558 -> 0.539 ms, by-source backward and both gathers unchanged (they wait on loads, not on issue
// slots), the 256-thread by-destination backward SLOWER (0.531 -> 0.596 ms) -- so only the forward kernel uses these.
__device__ __forceinline__ void fma2_p(float& a0, float& a1, float s, float b0, float b1) {
  asm("{\n\t.reg .b64 ra, rb, rs;\n\tmov.b64 ra, {%0, %1};\n\tmov.b64 rb, {%2, %3};\n\tmov.b64 rs, {%4, %4};\n\t"
      "fma.rn.f32x2 ra, rs, rb, ra;\n\tmov.b64 {%0, %1}, ra;\n\t}"
      : "+f"(a0), "+f"(a1) : "f"(b0), "f"(b1), "f"(s));
}
__device__ __forceinline__ void fma4_p(float4& a, float s, const float4& b) {
  fma2_p(a.x, a.y, s, b.x, b.y);
  fma2_p(a.z, a.w, s, b.z, b.w);
}
// acc (two partial sums: even / odd elements) += a . b as two packed FMAs; the caller adds acc.x + acc.y at the end
__device__ __forceinline__ void dot4_acc2(float2& acc, const float4& a, const float4& b) {
  asm("{\n\t.reg .b64 rc, ra, rb;\n\tmov.b64 rc, {%0, %1};\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "fma.rn.f32x2 rc, ra, rb, rc;\n\tmov.b64 ra, {%6, %7};\n\tmov.b64 rb, {%8, %9};\n\t"
      "fma.rn.f32x2 rc, ra, rb, rc;\n\tmov.b64 {%0, %1}, rc;\n\t}"
      : "+f"(acc.x), "+f"(acc.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(a.z), "f"(a.w), "f"(b.z), "f"(b.w));
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}

// Second level of the two-level column reductions (bias gradients, BatchNorm statistics and backward sums, classifier-tail
// gradients): column c of out = sum over the nb block partials, fixed order, fp64.  A block is FIN_COLS columns x FIN_ROWS
// row-lanes; a thread adds every FIN_ROWS-th partial of its column with four independent accumulators (four loads in
// flight), then the FIN_ROWS lane sums are added in lane order.  The first version (32 columns x 8 row-lanes, one
// accumulator) walked 600 partials in 75 load-latency-bound iterations: 11-19 us per launch, nine such launches per COGMEN
// step -- nothing at 2^20 utterances per GPU, ~5 % of the step when the same batch is sharded over 8 GPUs.
constexpr int FIN_COLS = 8, FIN_ROWS = 32;           // FIN_COLS * FIN_ROWS == 256 threads
__device__ __forceinline__ double fin_reduce(const float* __restrict__ partial, int nb, long long ld, int c, bool ok,
                                             double (*sm)[FIN_COLS + 1]) {
  const int tx = threadIdx.x & (FIN_COLS - 1), ty = threadIdx.x / FIN_COLS;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  if (ok) {
    const float* p = partial + c;
    int b = ty;
    for (; b + 3 * FIN_ROWS < nb; b += 4 * FIN_ROWS) {
      const float v0 = p[(long long)b * ld], v1 = p[(long long)(b + FIN_ROWS) * ld], v2 = p[(long long)(b + 2 * FIN_ROWS) * ld],
                  v3 = p[(long long)(b + 3 * FIN_ROWS) * ld];
      s0 += (double)v0; s1 += (double)v1; s2 += (double)v2; s3 += (double)v3;
    }
    for (; b < nb; b += FIN_ROWS) s0 += (double)p[(long long)b * ld];
  }
  __syncthreads();                                   // sm may still be read by a previous call
  sm[ty][tx] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  double tot = 0.0;
#pragma unroll
  for (int y = 0; y < FIN_ROWS; ++y) tot += sm[y][tx];
  return tot;
}
static inline unsigned fin_blocks(int ncols) { return (unsigned)((ncols + FIN_COLS - 1) / FIN_COLS); }

// counter-based hash RNG for dropout: uniform in [0,1) from (seed, element index)
__device__ __forceinline__ float hash_uniform(uint64_t seed, uint64_t idx) {
  uint64_t z = seed + idx * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (float)(z >> 40) * (1.0f / 16777216.0f);
}

// Dropout of the GEMM epilogues (ERCG_ACT_RELU_DROPOUT): ONE 64-bit hash per group of four consecutive columns of a row,
// 16 bits per element (drop iff bits < p * 65536).  The per-element splitmix64 above costs ~25 integer instructions;
// in the tcgen05 GEMM epilogue that was 2.5x the whole tile (ncu: 181 us vs 73 us for the same product without it).
__device__ __forceinline__ uint64_t hash64(uint64_t seed, uint64_t idx) {
  uint64_t z = seed + idx * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__host__ __device__ inline unsigned dropout_thr16(float p) {
  const float t = p * 65536.0f + 0.5f;
  return t <= 0.f ? 0u : (t >= 65535.f ? 65535u : (unsigned)t);
}
// element (m, n) of an [M, N] matrix: group index m * ceil(N/4) + n/4, lane n%4
__device__ __forceinline__ uint64_t dropout_group_hash(uint64_t seed, long long m, int n, int N) {
  return hash64(seed, (uint64_t)m * (uint64_t)((N + 3) >> 2) + (uint64_t)(n >> 2));
}
__device__ __forceinline__ bool dropout_drop(uint64_t h, int lane4, unsigned thr16) {
  return (unsigned)((h >> (16 * lane4)) & 0xffffull) < thr16;
}

constexpr int kNumSMs = 148;   // B200
constexpr int kMaxDevices = 64; // per-device caches of launch attributes are indexed by the CUDA device id
constexpr int kMaxSmemPerBlock = 227 * 1024;   // B200: the most dynamic shared memory one block may opt in to

// ---- launch set-up shared by every kernel that needs more than a plain <<<>>> launch: a dynamic shared-memory limit above
// 48 KB, a cluster shape, or a cooperative (co-resident) grid.  Everything below is per device: kernel attributes belong to
// the device context, and the answers are computed once so that a launch inside a CUDA-graph capture makes no set-up call.
inline int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return d;
}

// A value computed once per CUDA device id (one process may drive several GPUs, each needs its own set-up).  A result < 1
// means "unavailable" and is cached as such (read back as 0).  Safe to race on: at worst compute() runs twice.  Device ids
// >= kMaxDevices are not cached.
struct PerDevice {
  std::atomic<int> v[kMaxDevices];
  template <class F>
  int get(F compute) {
    const int d = current_device();
    const bool slot = d >= 0 && d < kMaxDevices;
    if (slot) {
      const int c = v[d].load(std::memory_order_acquire);
      if (c != 0) return c > 0 ? c : 0;
    }
    const int n = compute();
    if (slot) v[d].store(n > 0 ? n : -1, std::memory_order_release);
    return n > 0 ? n : 0;
  }
};

inline int device_sm_count() {
  static PerDevice sms;
  return sms.get([] {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, current_device());
    return n > 0 ? n : kNumSMs;
  });
}

// Raises kernel K's dynamic shared-memory limit to `bytes` on the current device, once per device.  Every caller of one K
// passes the same bytes.  false (with no error left pending) when the runtime refuses; the caller returns ERCG_ECUDA.
template <auto K>
bool smem_limit(int bytes) {
  static PerDevice done;
  return done.get([&] {
    if (cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess) return 1;
    cudaGetLastError();
    return 0;
  }) > 0;
}

// cudaLaunchKernelEx configuration of `grid` blocks in 1-D clusters of C
struct ClusterConfig {
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  ClusterConfig(int C, int grid, int threads, size_t smem, cudaStream_t st) {
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  ClusterConfig(const ClusterConfig&) = delete;      // cfg.attrs points into this object
};

// How many of kernel K can be resident at once: blocks per SM for C = 1, clusters of C blocks on the device for C > 1.
// Asked once per device at `smem`, the largest dynamic shared memory K may launch with (which becomes K's limit), so the
// answer is a lower bound for every launch.  0: K cannot be scheduled this way.
template <auto K, int C = 1>
int resident_capacity(int threads, int smem) {
  static PerDevice cap;
  return cap.get([&] {
    if (smem > 0 && !smem_limit<K>(smem)) return 0;
    int n = 0;
    cudaError_t err;
    if constexpr (C == 1) {
      err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, K, threads, smem);
    } else {
      err = C > 8 ? cudaFuncSetAttribute(K, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) : cudaSuccess;
      ClusterConfig c(C, C, threads, smem, 0);
      if (err == cudaSuccess) err = cudaOccupancyMaxActiveClusters(&n, K, &c.cfg);
    }
    if (err != cudaSuccess) {
      cudaGetLastError();
      n = 0;
    }
    return n;
  });
}

// Result of a launch made with cudaLaunchKernelEx / cudaLaunchCooperativeKernel.  A failed launch leaves its error
// pending, and finish_launch() of the next unrelated launch would report it as its own, so it is cleared here.
inline int launch_status(cudaError_t err) {
  if (err == cudaSuccess) return finish_launch();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaGetLastError();
  return ERCG_ECUDA;
}

template <typename... KArgs, typename... Args>
int launch_cluster(void (*kernel)(KArgs...), int C, int grid, int threads, size_t smem, cudaStream_t st, Args&&... args) {
  ClusterConfig c(C, grid, threads, smem, st);
  return launch_status(cudaLaunchKernelEx(&c.cfg, kernel, static_cast<Args&&>(args)...));
}

// For kernels that call grid.sync(): the caller first checks that the grid fits resident_capacity.
template <typename P>
int launch_cooperative(void (*kernel)(P), int grid, int threads, size_t smem, cudaStream_t st, P p) {
  void* args[] = {&p};
  return launch_status(cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(threads), args, smem, st));
}

}  // namespace ercg
