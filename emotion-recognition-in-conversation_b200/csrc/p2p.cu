// Peer-memory all-reduce for the exchanges of the dialogue-sharded train step (SURVEY.md 8e; reference: DDP's bucketed NCCL
// all-reduce under accelerate, lumo/trainer/trainer.py:62-64,315-327).
//
// What crosses GPUs per COGMEN step is small and latency-bound: BatchNorm statistics (2H doubles), their backward sums
// (2H floats) and the flat gradient buffer in two buckets (0.53 + 0.58 MB).  With the batch sharded over 8 GPUs the whole
// step is 1.7 ms and four NCCL launches cost ~10 % of it.  On one NVSwitch node every GPU can load every peer's memory at
// NVLink speed, so the exchange is ONE-SHOT:
//   1. a CTA copies its chunk of the local vector into this rank's REGION (cudaMalloc'ed once, opened by every peer through
//      CUDA IPC) and writes the call number into its flag word in EVERY peer's region (system-scope release store);
//   2. it waits until all W flag words of its own region show that call number (acquire loads of local memory);
//   3. it adds the W staged chunks in rank order, loading the peers' copies straight over NVLink.
// Every rank adds the same values in the same order: results are bit-identical across ranks and run to run.  There is no
// reduce-scatter / all-gather round trip, no proxy thread, no host involvement; the kernel is an ordinary launch, so it is
// captured in the step's CUDA graph like any other node.  128 threads and <= 48 registers per CTA, so a CTA fits NEXT TO
// the persistent weight-gradient GEMM on an SM (352 threads x 168 registers) and the first gradient bucket can overlap it.
//
// Slot discipline.  A region holds two data slots and two flag sets, selected by the parity of the rank's call counter.  A
// rank overwrites slot p again two calls later; by then it has passed the wait of the call in between, for which every peer
// had to signal, and a peer signals call k+1 only after its call-k kernel has finished reading (stream order).  CTAs never
// wait for each other inside a grid, only for the same-index CTA of the peers, so no co-residency of the grid is assumed.
// Every wait is bounded (30 s): on timeout the kernel records ERCG_P2P_ETIMEOUT in the region header and carries on with
// whatever is there -- a dead peer makes the step wrong and says so (ercg_p2p_status), it does not hang the GPU.
// The same protocol is the tail of two reducing kernels in norm_loss.cu (BatchNorm statistics and their backward sums are
// exchanged by the kernels that reduce them); p2p_dev.cuh holds the device side.
#include "p2p_dev.cuh"

namespace ercg {

// B units per thread per round, at most WP peers each (B * WP == 8 loads in flight); returns the first unit not processed
template <typename T, int B, int WP>
__device__ __forceinline__ long long reduce_rounds(unsigned char* const* __restrict__ regions, int world, size_t slot_off,
                                                   float4* __restrict__ o, long long u, long long u1) {
  for (; u + (long long)(B - 1) * P2P_THREADS < u1; u += (long long)B * P2P_THREADS) {
    float4 v[B][WP];
#pragma unroll
    for (int b = 0; b < B; ++b)
#pragma unroll
      for (int p = 0; p < WP; ++p)
        if (p < world) v[b][p] = ld_peer16(regions[p] + slot_off + 16 * (u + (long long)b * P2P_THREADS));
#pragma unroll
    for (int b = 0; b < B; ++b) {
      float4 acc = v[b][0];
#pragma unroll
      for (int p = 1; p < WP; ++p)
        if (p < world) add16(acc, v[b][p], T());
      o[u + (long long)b * P2P_THREADS] = acc;
    }
  }
  return u;
}

// regions[r] = base of rank r's region as mapped in THIS process (own region included).  n elements of T; slot_bytes = size
// of one data slot.  The first `units` 16-byte units are split evenly over the CTAs (units = 0 when in / out are not 16-byte
// aligned); the remaining elements go one by one to the last CTA.
template <typename T>
__global__ void __launch_bounds__(P2P_THREADS, 10)
p2p_allreduce_kernel(unsigned char* const* __restrict__ regions, int rank, int world, const T* __restrict__ in, T* __restrict__ out,
                     long long n, long long units, size_t slot_bytes, unsigned long long timeout_ns) {
  const int c = blockIdx.x, G = gridDim.x, tid = threadIdx.x;
  unsigned char* self = regions[rank];
  const P2pCall k = p2p_begin(regions, rank, slot_bytes, timeout_ns);
  const size_t slot_off = k.slot_off;
  constexpr int EPV = 16 / sizeof(T);                         // elements per 16-byte unit
  const long long per = (units + G - 1) / G;
  const long long u0 = min(units, (long long)c * per), u1 = min(units, u0 + per);
  const long long e0 = c == G - 1 ? units * EPV : n, e1 = n;  // scalar tail (last CTA only)
  // 1. stage this CTA's chunk in the local region
  {
    float4* dst = reinterpret_cast<float4*>(self + slot_off);
    const float4* src = reinterpret_cast<const float4*>(in);
    long long u = u0 + tid;
    for (; u + 3 * P2P_THREADS < u1; u += 4 * P2P_THREADS) {  // four independent 16-byte copies in flight
      const float4 a = src[u], b = src[u + P2P_THREADS], cc = src[u + 2 * P2P_THREADS], d = src[u + 3 * P2P_THREADS];
      dst[u] = a; dst[u + P2P_THREADS] = b; dst[u + 2 * P2P_THREADS] = cc; dst[u + 3 * P2P_THREADS] = d;
    }
    for (; u < u1; u += P2P_THREADS) dst[u] = src[u];
    T* dste = reinterpret_cast<T*>(self + slot_off);
    for (long long e = e0 + tid; e < e1; e += P2P_THREADS) dste[e] = in[e];
  }
  // 2. tell every peer (and ourselves) that chunk c of this call is in place; 3. wait for everybody's chunk c
  p2p_signal_wait(regions, rank, world, c, k);
  // 4. add the W staged chunks in rank order; the peers' copies are read over NVLink, up to eight loads in flight per thread
  //    (a load costs ~2 us: issuing them one by one would make the kernel W times slower)
  {
    float4* o = reinterpret_cast<float4*>(out);
    long long u = u0 + tid;
    // few peers: 4 (W <= 2) or 2 (W <= 4) units per thread per round keep 8 loads in flight all the same
    if (world <= 2) u = reduce_rounds<T, 4, 2>(regions, world, slot_off, o, u, u1);
    else if (world <= 4) u = reduce_rounds<T, 2, 4>(regions, world, slot_off, o, u, u1);
    for (; u < u1; u += P2P_THREADS) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int p0 = 0; p0 < world; p0 += 8) {
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (p0 + j < world) v[j] = ld_peer16(regions[p0 + j] + slot_off + 16 * u);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (p0 + j < world) {
            if (p0 + j == 0) acc = v[0];
            else add16(acc, v[j], T());
          }
      }
      o[u] = acc;
    }
    for (long long e = e0 + tid; e < e1; e += P2P_THREADS) {
      T acc = ld_peer(reinterpret_cast<const T*>(regions[0] + slot_off) + e);
      for (int p = 1; p < world; ++p) acc += ld_peer(reinterpret_cast<const T*>(regions[p] + slot_off) + e);
      out[e] = acc;
    }
  }
  // 5. the last CTA to finish closes the call
  p2p_close_call(k, G);
}

}  // namespace ercg

using namespace ercg;

extern "C" size_t ercg_p2p_region_bytes(size_t max_bytes) {
  const size_t slot = (max_bytes + 255) / 256 * 256;
  return sizeof(P2pHeader) + 2 * slot;
}

extern "C" int ercg_p2p_alloc(size_t region_bytes, void** region, unsigned char* ipc_handle) {
  static_assert(sizeof(cudaIpcMemHandle_t) == ERCG_P2P_HANDLE_BYTES, "IPC handle size");
  if (!region || !ipc_handle || region_bytes < sizeof(P2pHeader)) return ERCG_EINVAL;
  void* p = nullptr;
  if (cudaMalloc(&p, region_bytes) != cudaSuccess) return ERCG_ECUDA;
  if (cudaMemset(p, 0, region_bytes) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) { cudaFree(p); return ERCG_ECUDA; }
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, p) != cudaSuccess) { cudaFree(p); cudaGetLastError(); return ERCG_ECUDA; }
  memcpy(ipc_handle, &h, sizeof(h));
  *region = p;
  return ERCG_OK;
}

extern "C" int ercg_p2p_open(const unsigned char* ipc_handle, void** region) {
  if (!region || !ipc_handle) return ERCG_EINVAL;
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle, sizeof(h));
  void* p = nullptr;
  if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return ERCG_ECUDA; }
  *region = p;
  return ERCG_OK;
}

extern "C" int ercg_p2p_close(void* peer_region) {
  if (!peer_region) return ERCG_EINVAL;
  return cudaIpcCloseMemHandle(peer_region) == cudaSuccess ? ERCG_OK : ERCG_ECUDA;
}

extern "C" int ercg_p2p_free(void* region) {
  if (!region) return ERCG_EINVAL;
  return cudaFree(region) == cudaSuccess ? ERCG_OK : ERCG_ECUDA;
}

extern "C" int ercg_p2p_status(const void* region, int* status_host) {
  if (!region || !status_host) return ERCG_EINVAL;
  const P2pHeader* h = reinterpret_cast<const P2pHeader*>(region);
  return cudaMemcpy(status_host, &h->status, sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess ? ERCG_OK : ERCG_ECUDA;
}

// The device address of the same word, for kernels that must not consume the result of a failed exchange
// (ercg_adam_step_guarded).  No synchronisation: the word lives in this rank's own region.
extern "C" int ercg_p2p_status_word(void* region, int** status_dev) {
  if (!region || !status_dev) return ERCG_EINVAL;
  *status_dev = &reinterpret_cast<P2pHeader*>(region)->status;
  return ERCG_OK;
}

extern "C" int ercg_p2p_allreduce(void* const* regions_dev, int rank, int world, const void* in, void* out, int64_t n,
                                  int dtype, size_t max_bytes, void* stream) {
  if (!regions_dev || world < 1 || world > P2P_MAX_WORLD || rank < 0 || rank >= world || n < 0 || (dtype != 0 && dtype != 1))
    return ERCG_EINVAL;
  if (n == 0) return ERCG_OK;                                 // (every rank passes the same n: nobody waits for this call)
  if (!in || !out) return ERCG_EINVAL;
  const size_t esz = dtype == 0 ? 4 : 8;
  const size_t slot = (max_bytes + 255) / 256 * 256;
  if ((size_t)n * esz > slot) return ERCG_EWORKSPACE;
  if ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & (esz - 1)) return ERCG_EALIGN;
  const long long epv = (long long)(16 / esz);
  const long long units = (aligned16(in) && aligned16(out)) ? n / epv : 0;   // 16-byte units; the rest goes element by element
  // One CTA per ROUND of the reduce loop (128 threads x B units x 16 bytes, B x W = 8 loads in flight per thread), at most 128
  // CTAs: the payloads are <= ~1 MB and the kernel is bound by the NVLink load latency times the number of rounds, not by
  // bandwidth.
  const size_t per_cta = (size_t)P2P_THREADS * 16 * (world <= 2 ? 4 : world <= 4 ? 2 : 1);
  long long want = (long long)(((size_t)n * esz + per_cta - 1) / per_cta);
  const int grid = (int)(want < 1 ? 1 : (want > P2P_MAX_CTAS ? P2P_MAX_CTAS : want));
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* const* regs = reinterpret_cast<unsigned char* const*>(regions_dev);
  if (dtype == 0)
    p2p_allreduce_kernel<float><<<grid, P2P_THREADS, 0, st>>>(regs, rank, world, (const float*)in, (float*)out, n, units, slot, p2p_timeout_ns());
  else
    p2p_allreduce_kernel<double><<<grid, P2P_THREADS, 0, st>>>(regs, rank, world, (const double*)in, (double*)out, n, units, slot, p2p_timeout_ns());
  return finish_launch();
}
