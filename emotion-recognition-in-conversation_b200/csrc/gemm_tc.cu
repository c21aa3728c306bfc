// K2 (tensor-core path): C[M,N] = act(A[M,K] @ B[K,N] + bias) and C[K1,N1] = A^T @ B on tcgen05 with fp32-grade accuracy.
//
// Replaces the same reference code as gemm_simt.cu (nn.Linear of cogmen.py:103-105,116-122, the relation
// weights of RGCNConv cogmen.py:65 / models/rgcn.py:329-343, the Linears of TransformerConv cogmen.py:66).
//
// The reference is fp32 and BASELINE.json asks for 1e-5 relative parity, which plain TF32 (10-bit mantissa) cannot give.
// Every operand is split x = hi + lo (hi = upper 19 bits = what a tf32 operand read sees, lo = x - hi exact) and the product
// is accumulated in fp32 as  A_hi*B_hi + A_lo*B_hi + A_hi*B_lo  (the dropped lo*lo term is 2^-22 relative):
// A_hi*B_hi runs as kind::tf32 MMAs (exact products); the two correction terms, 2^-11 of the result, as kind::f16 (bf16)
// MMAs at twice the rate -- 8 instead of 12 instructions per 32-k chunk, in both kernels.
//
// Both kernels are persistent, warp-specialised CTAs of 352 threads, 1 CTA / SM:
//   warps 0-3  splitter : raw TMA tile of the streamed operand -> tf32 hi + bf16 pairs of hi and lo, written straight
//                         into TENSOR MEMORY with tcgen05.st; the MMAs take that operand from TMEM (TS form)
//   warps 4-7  epilogue : tcgen05.ld accumulator rows -> round-to-nearest register accumulation across k groups ->
//                         bias / activation -> swizzled staging slabs -> TMA bulk stores (NN); partials to the workspace (TN)
//   warp  8    TMA producer of the streamed operand (HBM), warp 10 TMA producer of the other operand (L2-resident)
//   warp  9    MMA issuer: warp-uniform loop, one elected lane issues, tcgen05.commit releases stages
// Tensor memory (512 columns): 2 accumulator stages x 128 + 4 operand stages x 64.
//
// Accumulation accuracy: the tensor core adds into TMEM with round-toward-zero, which on random-sign data shrinks
// |D| by ~0.3 ulp per instruction (measured on B200: -8.8e-6 relative at K=1443 with one long chain -- see
// DESIGN.md).  As in Ootomo & Yokota's error-corrected tensor-core GEMM, the long sum therefore lives OUTSIDE the
// tensor core: the MMA warp accumulates only a group of k-chunks (128 k in the NN kernel, 256 rows in the TN kernel) into a
// TMEM stage, the epilogue warps add each such partial into fp32 REGISTER accumulators with round-to-nearest, and the two
// TMEM stages ping-pong so the drain of group g overlaps the MMAs of group g+1.  Every mbarrier wait is bounded: a protocol
// bug traps instead of hanging the GPU.  DESIGN.md section 5 has the measurements behind each of these choices.
#include "common.cuh"
#include <cuda.h>
#include <cuda_bf16.h>
#include <cstdlib>

namespace ercg {

constexpr int TC_BM = 128;        // rows per tile (UMMA M)
constexpr int TC_BN = 128;        // max output columns per tile (UMMA N, multiple of 16)
constexpr int TC_BK = 32;         // k per stage: 32 floats = one 128-byte swizzle span
constexpr int TC_GROUP = 4;         // k-chunks accumulated inside TMEM before a round-to-nearest flush to registers
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 4;      // 16 KB
constexpr uint32_t TC_B_BYTES = TC_BN * TC_BK * 4;      // 16 KB

struct TcEpilogue {
  const float* bias; int act; const float* aux; long long ldaux; float aux_scale; float drop_p; unsigned long long seed;
  int dbg;   // ERCG_TC_DBG: performance experiments only (1 no MMA, 8 no B loads)
  long long* trace;   // ERCG_TC_TRACE: CTA 0 records clock64() per role and k-chunk (pipeline timeline, diagnostics only)
  const unsigned long long* seed_dev = nullptr;   // optional device word added to `seed` (fresh dropout mask per graph replay)
};
constexpr int TR_N = 160;          // traced chunks
constexpr int TR_ROLES = 5;        // 0 A producer, 1 splitter, 2 MMA, 3 epilogue (per group), 4 B producer
// compiled in only with -DERCG_TRACE (make EXTRA=-DERCG_TRACE): the marks sit in the MMA issue loop, which paces the kernels
#ifdef ERCG_TRACE
#define TC_TRACE(role, idx, slot)                                                                   \
  do {                                                                                              \
    if (ep.trace && blockIdx.x == 0 && (idx) < TR_N) ep.trace[((role) * TR_N + (idx)) * 4 + (slot)] = clock64(); \
  } while (0)
#else
#define TC_TRACE(role, idx, slot) do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Every wait is bounded in WALL TIME, not in polls: a pipeline bug must fail instead of hanging the GPU, but a slow and
// legitimate wait (a pre-empted context, a debugger, a contended L2) must never be mistaken for one -- a __trap() poisons
// the whole CUDA context.  The clock is read once per 65536 polls; the limit is 20 s, four orders of magnitude above
// the longest wait of a healthy launch (~1 ms).  Build with -DERCG_NO_WAIT_LIMIT to remove the check altogether.
__device__ __forceinline__ bool mbar_timed_out(unsigned long long& t0) {
#ifdef ERCG_NO_WAIT_LIMIT
  return false;
#else
  unsigned long long now;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
  if (t0 == 0ull) { t0 = now; return false; }
  return now - t0 > 20000000000ull;
#endif
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  unsigned long long t0 = 0ull;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if ((spin & 0xffffu) == 0xffffu && mbar_timed_out(t0)) __trap();
  }
}
// same wait for warps that are NOT on the latency-critical path (TMA producers): back off between polls so that the spin
// loop does not eat the issue slots of the splitter / epilogue warps that share the SM sub-partition
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  unsigned long long t0 = 0ull;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (!done) __nanosleep(96);
    if ((spin & 0xffffu) == 0xffffu && mbar_timed_out(t0)) __trap();
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// hi/lo split for 3xTF32.  The tensor core reads only the upper 19 bits of a tf32 operand, so hi = x with the low 13
// mantissa bits cleared is what it would see anyway, lo = x - hi is exact, and lo is passed unrounded (the hardware
// truncates it to 11 significant bits: error <= 2^-20 |x| worst case, ~2^-22 on average).  2 instructions per element
// instead of ~10 for two cvt.rna.tf32 -- the splitter warps were issue-bound (profiles/r01_tn_v2_hot.txt).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xFFFFE000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ float rn_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// K-major, 128-byte swizzle: rows are 128 B apart, 8-row atoms are 1024 B apart (SBO), LBO unused (=1), version 1
__device__ __forceinline__ uint64_t make_desc_k_sw128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}

// ---------------------------------------------------------------------------------------------- kernel
// NN kernel, A operand through TENSOR MEMORY (tcgen05.mma "TS" form).
//
// Measured on the first version (A_hi/A_lo/B_hi/B_lo all in shared memory, profiles/r01_ncu_full_262k.csv): the kernel was
// bound by shared-memory bandwidth, not by HBM or the tensor pipe -- per 32-k chunk the splitter read 16 KB and wrote
// 32 KB, TMA wrote 44 KB and the twelve SS-form MMAs read 92 KB of operands (~184 KB per 16 KB of HBM data at
// 128 B/clk/SM).  Here the splitter threads (one per row of the 128-row tile = one per TMEM lane) read the raw TMA tile
// once and write A_hi / A_lo straight into TMEM columns with tcgen05.st; the MMAs take A from TMEM and only B from
// shared memory.  Shared-memory traffic per chunk drops to ~100 KB.
//
//   shared memory: raw A ring TC_R x 16 KB (as TMA wrote it, 128-byte swizzle) | B ring TC_Q x (B_hi 16 KB + B_lo 16 KB)
//                  | epilogue staging 4 warps x 2 slabs x 4 KB (written out by TMA bulk stores)
//   tensor memory (512 columns): accumulator stages 2 x 128 | A stages TC_TA x (hi 32 + lo 32 columns)
//
// Loop nest: M tile -> N tile -> k chunk.  When the whole K extent fits the TMEM A stages (K <= 32*TC_TA = 128) and there
// are several N tiles ("resident" mode: the K = 100 transforms of COGMEN with N = 900 / 400), A is loaded and split ONCE
// per M tile and stays in TMEM while the N tiles stream B only; otherwise A is re-streamed per N tile (n_tiles is 1 for
// every long-K transform of the reference models).
#ifndef TC_R_
#define TC_R_ 4
#endif
#ifndef TC_Q_
#define TC_Q_ 3
#endif
constexpr int TC_TA = 4;          // TMEM A stages
#ifndef PAIR_N_GRAN_
#define PAIR_N_GRAN_ 32
#endif
constexpr int PAIR_N_GRAN = PAIR_N_GRAN_;   // UMMA N granularity of the pair kernels (half of it per CTA)
constexpr uint32_t TC_TMEM_A0 = 2 * TC_BN;                       // first A column
constexpr int TC_SLABS = 4;                                     // 32-column slabs of a 128-column tile
constexpr uint32_t TC_SLAB_BYTES = 32 * 128;                     // epilogue staging slab: 32 rows x 32 columns, 128-byte swizzle
constexpr int TC_THREADS = 352;   // 4 splitter + 4 epilogue warps, A producer, MMA, B producer
#ifndef TC_R2_
#define TC_R2_ 6
#endif
#ifndef TC_Q2_
#define TC_Q2_ 6
#endif
// Ring geometry and barrier indices.  Single CTA: R raw A stages of 16 KB, Q B stages of (B_hi 16 KB + B16 16 KB), staging
// for all four 32-column slabs of a tile per epilogue warp (64 KB).  CTA pair (cta_group::2, one N tile, long K): each CTA
// holds HALF of the B tile (8 + 8 KB per stage) and stages one slab at a time (16 KB), so both rings are deeper in the same
// shared memory -- the pipeline trace of the single-CTA kernel on K = 1443 (profiles/r02o_nn_trace_single_cta.txt) has the
// B ring as the critical loop: stage freed by the MMAs -> TMA from L2 (~2800 clk under load) -> MMAs (~500 clk) around a
// 3-stage ring = ~1100 clk per chunk, with the tensor pipe busy 42 % of the time.
#ifndef TC_R2S_
#define TC_R2S_ 4
#endif
template <bool TWO, bool WIDE = false>
struct NnCfg {
  // pair + short tiles (WIDE: K <= 512, i.e. the K = 100 transforms with A resident across N tiles and the K = 300 / 400 input
  // gradients) keep the 4-slab staging -- with 4-16 chunks per tile the epilogue is a large share of a tile and staging slab
  // by slab, with its column sums in between, measured slower in the step -- and spend the freed B bytes on ring depth only;
  // pair + long K (K = 1443: 46 chunks per tile) stages one slab at a time and takes two more A stages
  static constexpr int R = TWO ? (WIDE ? TC_R2S_ : TC_R2_) : TC_R_;
  static constexpr int Q = TWO ? TC_Q2_ : TC_Q_;
  static constexpr uint32_t BT_BYTES = TWO ? TC_B_BYTES / 2 : TC_B_BYTES;       // one B tile (fp32 hi, or bf16 pairs) of this CTA
  static constexpr int SLABS = (TWO && !WIDE) ? 1 : 4;                          // staging slabs per epilogue warp
  static constexpr uint32_t STAGE_BYTES = 4 * SLABS * TC_SLAB_BYTES;
  static constexpr uint32_t SMEM_BYTES = R * TC_A_BYTES + Q * 2 * BT_BYTES + STAGE_BYTES + 1024 /*align*/ + 512 /*barriers*/;
  static constexpr int A_FULL = 0;                   // [R]  TMA bytes of the raw A tile landed
  static constexpr int R_FREE = A_FULL + R;          // [R]  splitter has read the raw tile (128 arrivals)
  static constexpr int TA_FULL = R_FREE + R;         // [TC_TA] A_hi / A_lo written to TMEM
  static constexpr int TA_FREE = TA_FULL + TC_TA;    // [TC_TA] MMAs that read this TMEM A stage retired
  static constexpr int B_FULL = TA_FREE + TC_TA;     // [Q]  TMA bytes of B_hi/B_lo landed (pair: both halves, on the leader)
  static constexpr int Q_FREE = B_FULL + Q;          // [Q]  MMAs that read this B stage retired
  static constexpr int ACC_FULL = Q_FREE + Q;        // [2]
  static constexpr int ACC_EMPTY = ACC_FULL + 2;     // [2]
  static constexpr int COUNT = ACC_EMPTY + 2;
  static_assert(SMEM_BYTES <= kMaxSmemPerBlock, "shared memory budget");
  static_assert(COUNT * 8 + 8 <= 512, "barrier area");
};
constexpr uint32_t TC_SMEM_BYTES = NnCfg<false>::SMEM_BYTES;

__device__ __forceinline__ float4 lds4(uint32_t saddr) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(saddr) : "memory");
  return r;
}
__device__ __forceinline__ void sts4(uint32_t saddr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t saddr) {
  uint16_t r;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(r) : "r"(saddr) : "memory");
  return (uint32_t)r;
}
__device__ __forceinline__ float lds1(uint32_t saddr) {
  float r;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(saddr) : "memory");
  return r;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum) : "memory");
}
// 16-bit operands (bf16): A from tensor memory (two k-elements per 32-bit column), B from shared memory, K = 16
__device__ __forceinline__ void tc_mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum) : "memory");
}
// {hi16 = bf16(b), lo16 = bf16(a)} -> element a sits at the EVEN k position (low half), round-to-nearest
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- CTA-pair (cta_group::2) helpers: the two CTAs of a cluster on one TPC run ONE MMA of M = 256; each CTA keeps its 128
// rows of A / D in its own tensor memory and HALF of the B tile in its own shared memory (the hardware feeds both tensor
// cores from both halves), so the shared-memory and L2 -> SM bytes of the B operand per SM halve.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_cta(uint32_t saddr, uint32_t rank) {   // shared::cta address -> shared::cluster address in CTA `rank`
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (release at CTA scope), as CUTLASS's ClusterBarrier::arrive(cta_id): what the peer's tensor core reads
  // was ordered by tcgen05.wait::st + tcgen05.fence::before_thread_sync (tensor memory) or fence.proxy.async (shared memory)
  // before this arrive; a .release.cluster here costs a cluster-wide memory barrier per arrival (measured: ~1500 clk)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {   // acquire at cluster scope (peer arrivals)
  uint32_t done = 0;
  unsigned long long t0 = 0ull;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if ((spin & 0xffffu) == 0xffffu && mbar_timed_out(t0)) __trap();
  }
}
// TMA load of this CTA's part of a pair's tile; the bytes complete on `cluster_bar` (the leader's barrier, mapa'd)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t cluster_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_commit2(uint32_t bar) {   // arrives on the barrier at this offset in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma2_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void tc_mma2_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum) : "memory");
}

// bias of four consecutive columns (zeros without a bias): fetched BEFORE the loop that applies it -- the staging stores of the
// epilogue are asm volatile with a memory clobber, so a load inside that loop is issued, waited for and used one at a time
__device__ __forceinline__ float4 tc_bias4(const TcEpilogue& ep, int nn0, int N) {
  float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ep.bias) {
    if (nn0 + 4 <= N) {
      b = __ldg(reinterpret_cast<const float4*>(ep.bias + nn0));   // bias is 16-byte aligned (checked on host)
    } else {
      if (nn0 + 0 < N) b.x = __ldg(ep.bias + nn0 + 0);
      if (nn0 + 1 < N) b.y = __ldg(ep.bias + nn0 + 1);
      if (nn0 + 2 < N) b.z = __ldg(ep.bias + nn0 + 2);
    }
  }
  return b;
}
template <int ACT>
__device__ __forceinline__ uint64_t tc_drop_hash(const TcEpilogue& ep, long long m, int nn0, int N) {
  return ACT == ERCG_ACT_RELU_DROPOUT ? dropout_group_hash(ep.seed, m, nn0, N) : 0ull;   // nn0 % 4 == 0: one hash per float4
}
template <int ACT>
__device__ __forceinline__ float4 tc_finish4(float4 x, const TcEpilogue& ep, long long m, int nn0, int N, float4 b, uint64_t h) {
  x.x += b.x; x.y += b.y; x.z += b.z; x.w += b.w;
  if (ACT == ERCG_ACT_RELU || ACT == ERCG_ACT_RELU_DROPOUT) {
    x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f);
  }
  if (ACT == ERCG_ACT_RELU_DROPOUT) {
    const float sc = 1.0f / (1.0f - ep.drop_p);
    const unsigned thr = dropout_thr16(ep.drop_p);
    x.x = dropout_drop(h, 0, thr) ? 0.f : x.x * sc;
    x.y = dropout_drop(h, 1, thr) ? 0.f : x.y * sc;
    x.z = dropout_drop(h, 2, thr) ? 0.f : x.z * sc;
    x.w = dropout_drop(h, 3, thr) ? 0.f : x.w * sc;
  }
  if (ACT == ERCG_ACT_MASK_POS) {
    const float* a = ep.aux + m * ep.ldaux + nn0;
    x.x = (nn0 + 0 < N && __ldg(a + 0) > 0.f) ? x.x * ep.aux_scale : 0.f;
    x.y = (nn0 + 1 < N && __ldg(a + 1) > 0.f) ? x.y * ep.aux_scale : 0.f;
    x.z = (nn0 + 2 < N && __ldg(a + 2) > 0.f) ? x.z * ep.aux_scale : 0.f;
    x.w = (nn0 + 3 < N && __ldg(a + 3) > 0.f) ? x.w * ep.aux_scale : 0.f;
  }
  return x;
}

// ABF16: the streamed operand A is STORED in bf16 (bf16 input-feature mode: half the HBM bytes of the projection).  Its raw
// tile is 128 rows x 32 bf16 = 64-byte rows (TMA 64-byte swizzle); the splitter copies the 16 words of its row -- already the
// "two k-elements per 32-bit column" packing the bf16 MMAs read -- straight into TMEM; there is no A_lo, and B comes as
// bf16_rn(B) | bf16_rn(B - bf16_rn(B)) (16 significant bits of every weight): 4 bf16 MMAs per 32-k chunk instead of 4 tf32 +
// 4 bf16, and no fp32 B tile.  The arithmetic is exact products of bf16 A with 16-bit B, accumulated in fp32.
// TWO: CTA pairs (cluster of 2, cta_group::2) for one N tile and a long K: CTA rank r owns M tile 2p + r (its A rows go to
// its own tensor memory, its accumulator rows stay there), loads rows [bn/2 r, bn/2 r + bn/2) of the B tile, and the
// leader's MMA warp issues M = 256 instructions for both.  The peer's TMA completes its bytes on the LEADER's B_FULL
// barrier; splitter and epilogue warps of both CTAs arrive (one lane per warp) on the leader's TA_FULL / ACC_EMPTY; what
// the MMAs release is a multicast commit to both CTAs.
template <int ACT, bool SMALLK, bool ABF16, bool TWO = false, bool ONESLAB = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_nn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBh,
                  const __grid_constant__ CUtensorMap tmBl, const __grid_constant__ CUtensorMap tmC,
                  float* __restrict__ C, long long ldc, long long M, int N,
                  int K, int bn /* UMMA N for this launch: multiple of 16, <= 128 */, const TcEpilogue ep_in,
                  float* __restrict__ colsum_partial /* [gridDim.x][4][128] column sums of C (N <= 128 only), or NULL */) {
  using Cfg = NnCfg<TWO, !ONESLAB>;
  TcEpilogue ep = ep_in;                                   // the device seed word is read ONCE, not per float4 of the epilogue
  if (ACT == ERCG_ACT_RELU_DROPOUT && ep.seed_dev) { ep.seed += *ep.seed_dev; ep.seed_dev = nullptr; }
  static_assert(!TWO || !ABF16, "pair mode: fp32 features");
  static_assert(!ONESLAB || (TWO && !SMALLK), "one-slab staging: pair mode, long K");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* bring = smem + Cfg::R * TC_A_BYTES;
  uint8_t* stage_all = bring + Cfg::Q * 2 * Cfg::BT_BYTES;          // 1024-byte aligned (every ring is a multiple of 1 KB)
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_all + Cfg::STAGE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + Cfg::COUNT);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t rank = TWO ? cluster_ctarank() : 0u;     // 0 = leader (issues the MMAs of the pair)
  const uint32_t pair_arrivals = TWO ? 8u : 128u;          // pair mode: one arrival per warp of both CTAs
  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::R; ++i) { mbar_init(BAR(Cfg::A_FULL + i), 1); mbar_init(BAR(Cfg::R_FREE + i), 128); }
    for (int i = 0; i < TC_TA; ++i) { mbar_init(BAR(Cfg::TA_FULL + i), pair_arrivals); mbar_init(BAR(Cfg::TA_FREE + i), 1); }
    for (int i = 0; i < Cfg::Q; ++i) { mbar_init(BAR(Cfg::B_FULL + i), 1); mbar_init(BAR(Cfg::Q_FREE + i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(BAR(Cfg::ACC_FULL + i), 1); mbar_init(BAR(Cfg::ACC_EMPTY + i), pair_arrivals); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 9) {   // all 512 TMEM columns: 2 accumulator stages x 128 + TC_TA A stages x 64
    if (TWO) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (TWO) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  auto LBAR = [&](int i) { return TWO ? mapa_cta(BAR(i), 0u) : BAR(i); };
  auto arrive_leader = [&](uint32_t lbar) {
    if (TWO) {
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(lbar);
    } else {
      mbar_arrive(lbar);
    }
  };

  // tile walk: single CTA t = blockIdx.x, += gridDim.x; pair p = blockIdx.x / 2, += gridDim.x / 2 and t = 2 p + rank (a tile
  // past the end is all zero-filled loads and clipped stores)
  const long long m_tiles_real = (M + TC_BM - 1) / TC_BM;
  const long long m_tiles = TWO ? (m_tiles_real + 1) / 2 : m_tiles_real;
  const long long t_first = TWO ? blockIdx.x / 2 : blockIdx.x, t_step = TWO ? gridDim.x / 2 : gridDim.x;
  auto TILE = [&](long long t) { return TWO ? 2 * t + (long long)rank : t; };
  const int n_tiles = (N + bn - 1) / bn;
  const int k_chunks = (K + TC_BK - 1) / TC_BK;
  const bool resident = n_tiles > 1 && k_chunks <= TC_TA;     // A stays in TMEM across the N tiles of an M tile
  const int a_reps = resident ? 1 : n_tiles;                  // A chunk loads per M tile = a_reps * k_chunks
  const uint32_t raw_base = smem_u32(smem), b_base = smem_u32(bring);
  auto B_HI = [&](int q) { return b_base + q * 2 * Cfg::BT_BYTES; };
  auto B_LO = [&](int q) { return b_base + q * 2 * Cfg::BT_BYTES + Cfg::BT_BYTES; };
  auto TA_HI = [&](int s) { return tmem_base + TC_TMEM_A0 + (uint32_t)s * 64u; };

  if (warp == 8) {
    // ------------------------------------------------------------------ A producer (HBM stream)
    if (lane == 0) {
      uint32_t n = 0;
      for (long long t = t_first; t < m_tiles; t += t_step) {
        const int m0 = (int)TILE(t) * TC_BM;
        for (int rep = 0; rep < a_reps; ++rep)
          for (int kc = 0; kc < k_chunks; ++kc, ++n) {
            const int r = n % Cfg::R;
            TC_TRACE(0, n, 0);
            mbar_wait_relaxed(BAR(Cfg::R_FREE + r), ((n / Cfg::R) & 1) ^ 1);
            TC_TRACE(0, n, 1);
            mbar_expect_tx(BAR(Cfg::A_FULL + r), ABF16 ? TC_A_BYTES / 2 : TC_A_BYTES);
            tma_load_2d(raw_base + r * TC_A_BYTES, &tmA, kc * TC_BK, m0, BAR(Cfg::A_FULL + r));
          }
      }
    }
  } else if (warp == 10) {
    // ------------------------------------------------------------------ B producer (L2-resident weights)
    if (lane == 0) {
      uint32_t n = 0;
      const uint32_t tx = 2u * (uint32_t)bn * TC_BK * 4u;
      for (long long t = t_first; t < m_tiles; t += t_step)
        for (int nt = 0; nt < n_tiles; ++nt)
          for (int kc = 0; kc < k_chunks; ++kc, ++n) {
            const int q = n % Cfg::Q;
            TC_TRACE(4, n, 0);
            mbar_wait_relaxed(BAR(Cfg::Q_FREE + q), ((n / Cfg::Q) & 1) ^ 1);
            TC_TRACE(4, n, 1);
            if (TWO) {
              // this CTA's half of the B rows; the bytes of BOTH halves complete on the leader's barrier
              const uint32_t lbar = mapa_cta(BAR(Cfg::B_FULL + q), 0u);
              if (rank == 0) mbar_expect_tx(BAR(Cfg::B_FULL + q), tx);
              // (the last N tile only has n_cur columns, half of THEM per CTA; the box still brings bn / 2 rows)
              const int n_cur = nt == n_tiles - 1 ? ((N - nt * bn + PAIR_N_GRAN - 1) / PAIR_N_GRAN * PAIR_N_GRAN) : bn;
              tma_load_2d_pair(B_HI(q), &tmBh, kc * TC_BK, nt * bn + (int)rank * (n_cur / 2), lbar);
              tma_load_2d_pair(B_LO(q), &tmBl, kc * 64, nt * bn + (int)rank * (n_cur / 2), lbar);
              continue;
            }
            if (ep.dbg & 8) { mbar_arrive(BAR(Cfg::B_FULL + q)); continue; }
            mbar_expect_tx(BAR(Cfg::B_FULL + q), ABF16 ? tx / 2 : tx);
            if (!ABF16) tma_load_2d(B_HI(q), &tmBh, kc * TC_BK, nt * bn, BAR(Cfg::B_FULL + q));
            tma_load_2d(B_LO(q), &tmBl, kc * 64, nt * bn, BAR(Cfg::B_FULL + q));      // bf16(B_hi) | bf16(B_lo) of this chunk
          }
    }
  } else if (warp == 9 && rank == 0) {
    // ------------------------------------------------------------------ MMA issuer
    // The whole warp runs this loop with warp-uniform control flow and one ELECTED lane issues the tcgen05 instructions
    // (profiles/r01_*: inside an `if (lane == 0)` region every descriptor had to be moved vector -> uniform register
    // per instruction and the issue loop itself, ~150 clk per UTCHMMA, was the bottleneck of the kernel).
    // UMMA N per N tile: bn, except the LAST tile of a row of tiles, which only computes the columns that exist (rounded up
    // to 16) -- N = 400 is 3 x 128 + 16 and N = 300 is 2 x 128 + 44: the tail tile costs 1/8 resp. 3/8 of a full one
    const int n_tail = TWO ? ((N - (n_tiles - 1) * bn + PAIR_N_GRAN - 1) / PAIR_N_GRAN * PAIR_N_GRAN) : ((N - (n_tiles - 1) * bn + 15) & ~15);
    constexpr uint32_t MMA_M = TWO ? 2 * TC_BM : TC_BM;
    const uint32_t idesc_base = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(MMA_M >> 4) << 24);
    const uint32_t idesc16_base = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(MMA_M >> 4) << 24);   // bf16 x bf16 -> f32
    const uint64_t desc_hi = ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61) | ((uint64_t)1 << 16);
    uint32_t a_base = 0, nb_ = 0;     // A chunk loads before this M tile; B chunk loads so far
    int a = 0;
    uint32_t aph = 0;
    for (long long t = t_first; t < m_tiles; t += t_step) {
      for (int nt = 0; nt < n_tiles; ++nt) {
        for (int kc = 0; kc < k_chunks; ++kc, ++nb_) {
          const int in_group = kc % TC_GROUP;
          const uint32_t d_tmem = tmem_base + (uint32_t)(a * TC_BN);
          if (lane == 0) TC_TRACE(2, nb_, 0);
          if (in_group == 0) mbar_wait(BAR(Cfg::ACC_EMPTY + a), aph ^ 1);   // epilogue has drained this accumulator stage
          if (lane == 0) TC_TRACE(2, nb_, 1);
          const uint32_t an = a_base + (resident ? 0 : nt * k_chunks) + kc;
          const int s = an % TC_TA, q = nb_ % Cfg::Q;
          mbar_wait(BAR(Cfg::TA_FULL + s), (an / TC_TA) & 1);        // A_hi / A_lo of this chunk are in TMEM
          if (lane == 0) TC_TRACE(2, nb_, 2);
          mbar_wait(BAR(Cfg::B_FULL + q), (nb_ / Cfg::Q) & 1);         // B tiles landed
          if (lane == 0) TC_TRACE(2, nb_, 3);
          tc_fence_after();
          // k-steps that still hold real columns (TMA zero-fills the K tail: K = 100 needs 13 tf32 steps of 8, not 16)
          const uint32_t n_mma = (uint32_t)((nt == n_tiles - 1 ? n_tail : bn) >> 3) << 17;   // pairs: half of it per CTA
          const uint32_t idesc = idesc_base | n_mma, idesc16 = idesc16_base | n_mma;
          const int ks_n = (ep.dbg & 1) ? 0 : min(TC_BK / 8, (K - kc * TC_BK + 7) >> 3);
          const int k16_n = (ep.dbg & 1) ? 0 : min(TC_BK / 16, (K - kc * TC_BK + 15) >> 4);
          const uint32_t ah0 = TA_HI(s);
          const uint64_t bh0 = desc_hi | (uint64_t)((B_HI(q) >> 4) & 0x3FFF), b16 = desc_hi | (uint64_t)((B_LO(q) >> 4) & 0x3FFF);
          if (elect_one()) {
            if (ABF16) {
              // A (bf16, exact) * (bf16(B) + bf16(B - bf16(B))): two bf16 MMAs per 16 k
#pragma unroll
              for (int j = 0; j < TC_BK / 16; ++j) {
                if (j < k16_n) {
                  tc_mma_bf16_ts(d_tmem, ah0 + 32 + j * 8, b16 + (uint64_t)(j * 2), idesc16, (in_group | j) ? 1u : 0u);
                  tc_mma_bf16_ts(d_tmem, ah0 + 32 + j * 8, b16 + (uint64_t)(4 + j * 2), idesc16, 1u);
                }
              }
            } else {
            // A_hi * B_hi in tf32 (exact products); the two 2^-11-sized correction terms A_lo * B_hi + A_hi * B_lo in bf16
            // at twice the rate: 4 + 4 instructions per 32-k chunk instead of 12 tf32 ones (see top of file)
#pragma unroll
            for (int ks = 0; ks < TC_BK / 8; ++ks)
              if (ks < ks_n) {
                if (TWO) tc_mma2_tf32_ts(d_tmem, ah0 + ks * 8, bh0 + (uint64_t)(ks * 2), idesc, (in_group | ks) ? 1u : 0u);
                else tc_mma_tf32_ts(d_tmem, ah0 + ks * 8, bh0 + (uint64_t)(ks * 2), idesc, (in_group | ks) ? 1u : 0u);
              }
#pragma unroll
            for (int j = 0; j < TC_BK / 16; ++j) {
              if (j < k16_n) {
                if (TWO) {
                  tc_mma2_bf16_ts(d_tmem, ah0 + 48 + j * 8, b16 + (uint64_t)(j * 2), idesc16, 1u);
                  tc_mma2_bf16_ts(d_tmem, ah0 + 32 + j * 8, b16 + (uint64_t)(4 + j * 2), idesc16, 1u);
                } else {
                  tc_mma_bf16_ts(d_tmem, ah0 + 48 + j * 8, b16 + (uint64_t)(j * 2), idesc16, 1u);        // bf16(A_lo) * bf16(B_hi)
                  tc_mma_bf16_ts(d_tmem, ah0 + 32 + j * 8, b16 + (uint64_t)(4 + j * 2), idesc16, 1u);    // bf16(A_hi) * bf16(B_lo)
                }
              }
            }
            }
            if (TWO) {
              tc_commit2(BAR(Cfg::Q_FREE + q));
              if (!resident || nt == n_tiles - 1) tc_commit2(BAR(Cfg::TA_FREE + s));
              if (in_group == TC_GROUP - 1 || kc == k_chunks - 1) tc_commit2(BAR(Cfg::ACC_FULL + a));
            } else {
            tc_commit(BAR(Cfg::Q_FREE + q));
            if (!resident || nt == n_tiles - 1) tc_commit(BAR(Cfg::TA_FREE + s));
            if (in_group == TC_GROUP - 1 || kc == k_chunks - 1) tc_commit(BAR(Cfg::ACC_FULL + a));   // partial sum -> epilogue
            }
          }
          __syncwarp();
          if (in_group == TC_GROUP - 1 || kc == k_chunks - 1) {
            if (++a == 2) { a = 0; aph ^= 1; }
          }
        }
      }
      a_base += (uint32_t)a_reps * k_chunks;
    }
  } else if (warp < 4) {
    // ------------------------------------------------------------------ splitter: thread = row of the tile = TMEM lane
    const int row = threadIdx.x;
    const uint32_t lane_addr = (uint32_t)(warp * 32) << 16;
    uint32_t n = 0;
    for (long long t = t_first; t < m_tiles; t += t_step) {
      for (int rep = 0; rep < a_reps; ++rep)
        for (int kc = 0; kc < k_chunks; ++kc, ++n) {
          const int r = n % Cfg::R, s = n % TC_TA;
          if (threadIdx.x == 0) TC_TRACE(1, n, 0);
          mbar_wait(BAR(Cfg::A_FULL + r), (n / Cfg::R) & 1);          // raw tile landed
          if (threadIdx.x == 0) TC_TRACE(1, n, 1);
          const uint32_t src = raw_base + r * TC_A_BYTES + (ABF16 ? row * 64 : row * 128);
          uint32_t hi[32], p16[32];                                // tf32 A_hi | bf16 pairs: [0,16) A_hi, [16,32) A_lo
          if (ABF16) {
            // 64-byte rows, TMA 64-byte swizzle: logical 16-byte chunk c sits at position c ^ ((row >> 1) & 3)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float4 x = lds4(src + ((c ^ ((row >> 1) & 3)) << 4));
              p16[4 * c + 0] = __float_as_uint(x.x); p16[4 * c + 1] = __float_as_uint(x.y);
              p16[4 * c + 2] = __float_as_uint(x.z); p16[4 * c + 3] = __float_as_uint(x.w);
            }
#pragma unroll
            for (int c = 16; c < 32; ++c) p16[c] = 0u;
          } else {
#pragma unroll
          for (int c = 0; c < 8; ++c) {                            // logical 16-byte chunk c sits at position c ^ (row & 7)
            const float4 x = lds4(src + ((c ^ (row & 7)) << 4));
            uint32_t l0, l1, l2, l3;
            split_tf32(x.x, hi[4 * c + 0], l0);
            split_tf32(x.y, hi[4 * c + 1], l1);
            split_tf32(x.z, hi[4 * c + 2], l2);
            split_tf32(x.w, hi[4 * c + 3], l3);
            p16[2 * c + 0] = pack_bf16x2(__uint_as_float(hi[4 * c + 0]), __uint_as_float(hi[4 * c + 1]));
            p16[2 * c + 1] = pack_bf16x2(__uint_as_float(hi[4 * c + 2]), __uint_as_float(hi[4 * c + 3]));
            p16[16 + 2 * c + 0] = pack_bf16x2(__uint_as_float(l0), __uint_as_float(l1));
            p16[16 + 2 * c + 1] = pack_bf16x2(__uint_as_float(l2), __uint_as_float(l3));
          }
          }
          mbar_wait(BAR(Cfg::TA_FREE + s), ((n / TC_TA) & 1) ^ 1);   // MMAs that read this TMEM stage retired
          if (threadIdx.x == 0) TC_TRACE(1, n, 2);
          tc_fence_after();
          if (!ABF16) tc_st32(TA_HI(s) + lane_addr, hi);
          tc_st32(TA_HI(s) + 32 + lane_addr, p16);
          tc_wait_st();
          // The raw stage is released only HERE: the TMEM stores above consume every loaded register, so the
          // shared-memory loads have returned.  (An arrive placed right after the loads was scheduled by ptxas before
          // their data came back -- SASS: LD.E.128 x8, SYNCS.ARRIVE, then the first use -- and a refill by TMA could
          // overtake a slow warp: rare wrong 32-row x 128-column blocks, caught by test_tc_gemm_race_stress.)
          mbar_arrive(BAR(Cfg::R_FREE + r));
          tc_fence_before();
          arrive_leader(LBAR(Cfg::TA_FULL + s));
          if (threadIdx.x == 0) TC_TRACE(1, n, 3);
        }
    }
  } else if (warp < 8) {
    // ------------------------------------------------------------------ epilogue (warps 4-7 -> TMEM lanes 32*(warp%4))
    // Every 32-column slab of the tile is staged in shared memory (thread = row, 16-byte chunks XOR-swizzled like a
    // 128-byte-swizzle TMA box, so the st.shared are bank-conflict free) and leaves as ONE bulk tensor store per slab; TMA
    // clips the M and N tails.  All (up to four) slabs of a tile are staged before the stores are issued, so there is one
    // wait for the previous tile's stores per tile, not one per pair of slabs.
    //   SMALLK (the whole K extent is one accumulation group: the K = 100 transforms): accumulator columns stream
    //   TMEM -> registers -> staging 32 at a time.  (ncu on the first version, which kept a float acc[128] per thread for
    //   every shape: the epilogue warps were busy ~97 % of the kernel -- local-memory spills of acc[], generic-address
    //   stores into the staging buffer -- and the MMA warp waited on ACC_EMPTY; K = 100, N = 100 ran at 27 % of HBM.)
    //   otherwise: partial sums of TC_GROUP k-chunks are added into fp32 registers with round-to-nearest (see top of file).
    int a = 0;
    uint32_t aph = 0;
    const int ew = warp & 3;
    const uint32_t stg_u32 = smem_u32(stage_all + ew * Cfg::SLABS * TC_SLAB_BYTES);     // this warp's 4 slabs of 32 x 32
    const uint32_t my_row = stg_u32 + lane * 128;
    const int n_groups = (k_chunks + TC_GROUP - 1) / TC_GROUP;
    const uint32_t tmem_lane = tmem_base + ((uint32_t)(ew * 32) << 16);
    float colacc[TC_SLABS];                                        // lane = column of a slab: sums over this warp's rows
#pragma unroll
    for (int sl = 0; sl < TC_SLABS; ++sl) colacc[sl] = 0.f;
    for (long long t = t_first; t < m_tiles; t += t_step) {
      const long long m0 = TILE(t) * TC_BM + ew * 32;
      const long long m = m0 + lane;                               // this thread's row (TMEM lane)
      const long long mrow = m < M ? m : M - 1;
      for (int nt = 0; nt < n_tiles; ++nt) {
        const int n0 = nt * bn;
        if (SMALLK) {
          mbar_wait(BAR(Cfg::ACC_FULL + a), aph);
          tc_fence_after();
          if (lane == 0) tma_store_wait_read();                    // the previous tile's bulk stores have read the slabs
          __syncwarp();
#pragma unroll
          for (int sl = 0; sl < TC_SLABS; ++sl) {
            const int c = 32 * sl;
            if (c < bn && n0 + c < N) {
              uint32_t rr[32];
              tc_ld32(tmem_lane + (uint32_t)(a * TC_BN + c), rr);
              float4 bb[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) bb[j] = tc_bias4(ep, n0 + c + 4 * j, N);     // in flight with the TMEM load
              uint64_t hh[8];                        // the eight hash chains of a slab interleave (one warp per scheduler: no
#pragma unroll                                       // other warp hides the latency of a serial 64-bit multiply chain)
              for (int j = 0; j < 8; ++j) hh[j] = tc_drop_hash<ACT>(ep, mrow, n0 + c + 4 * j, N);
              tc_wait_ld();
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                float4 v = make_float4(__uint_as_float(rr[j]), __uint_as_float(rr[j + 1]), __uint_as_float(rr[j + 2]),
                                       __uint_as_float(rr[j + 3]));
                if (ACT != ERCG_ACT_NONE || ep.bias) v = tc_finish4<ACT>(v, ep, mrow, n0 + c + j, N, bb[j >> 2], hh[j >> 2]);
                sts4(my_row + sl * TC_SLAB_BYTES + (((j >> 2) ^ (lane & 7)) << 4), v);
              }
            }
          }
          tc_fence_before();
          arrive_leader(LBAR(Cfg::ACC_EMPTY + a));
          if (++a == 2) { a = 0; aph ^= 1; }
        } else {
          float acc[TC_BN];
          for (int g = 0; g < n_groups; ++g) {
            if (threadIdx.x == 128) TC_TRACE(3, (int)((t - t_first) / t_step) * n_groups + g, 0);
            mbar_wait(BAR(Cfg::ACC_FULL + a), aph);
            if (threadIdx.x == 128) TC_TRACE(3, (int)((t - t_first) / t_step) * n_groups + g, 1);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < TC_BN; c += 32) {
              if (c < bn && n0 + c < N) {
                uint32_t rr[32];
                tc_ld32(tmem_lane + (uint32_t)(a * TC_BN + c), rr);
                tc_wait_ld();
                if (g == 0) {
#pragma unroll
                  for (int j = 0; j < 32; ++j) acc[c + j] = __uint_as_float(rr[j]);
                } else {
#pragma unroll
                  for (int j = 0; j < 32; ++j) acc[c + j] += __uint_as_float(rr[j]);   // round-to-nearest accumulation
                }
              }
            }
            tc_fence_before();
            arrive_leader(LBAR(Cfg::ACC_EMPTY + a));
            if (threadIdx.x == 128) TC_TRACE(3, (int)((t - t_first) / t_step) * n_groups + g, 2);
            if (++a == 2) { a = 0; aph ^= 1; }
          }
          if (ONESLAB) {
            // one staging slab per warp: stage, store, (column sums), and only then re-use it for the next slab -- four
            // short waits per 46-chunk tile, in exchange for 48 KB of shared memory that went into the rings
#pragma unroll
            for (int sl = 0; sl < 4; ++sl) {
              const int c = 32 * sl;
              if (c < bn && n0 + c < N) {
                if (lane == 0) tma_store_wait_read();
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  float4 v = make_float4(acc[c + j], acc[c + j + 1], acc[c + j + 2], acc[c + j + 3]);
                  if (ACT != ERCG_ACT_NONE || ep.bias) v = tc_finish4<ACT>(v, ep, mrow, n0 + c + j, N, tc_bias4(ep, n0 + c + j, N), tc_drop_hash<ACT>(ep, mrow, n0 + c + j, N));
                  sts4(my_row + (((j >> 2) ^ (lane & 7)) << 4), v);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) { tma_store_2d(&tmC, stg_u32, n0 + c, (int)m0); tma_store_commit(); }
                if (colsum_partial) {
                  float sum = 0.f;
#pragma unroll 8
                  for (int r = 0; r < 32; ++r)
                    sum += lds1(stg_u32 + r * 128 + ((((lane >> 2) ^ (r & 7)) << 4) | ((lane & 3) << 2)));
                  colacc[sl] += sum;
                }
              }
            }
            continue;
          }
          if (lane == 0) tma_store_wait_read();
          __syncwarp();
#pragma unroll
          for (int sl = 0; sl < TC_SLABS; ++sl) {
            const int c = 32 * sl;
            if (c < bn && n0 + c < N) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                float4 v = make_float4(acc[c + j], acc[c + j + 1], acc[c + j + 2], acc[c + j + 3]);
                if (ACT != ERCG_ACT_NONE || ep.bias) v = tc_finish4<ACT>(v, ep, mrow, n0 + c + j, N, tc_bias4(ep, n0 + c + j, N), tc_drop_hash<ACT>(ep, mrow, n0 + c + j, N));
                sts4(my_row + sl * TC_SLAB_BYTES + (((j >> 2) ^ (lane & 7)) << 4), v);
              }
            }
          }
        }
        fence_proxy_async();                                       // generic-proxy stores -> visible to the TMA engine
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (int sl = 0; sl < TC_SLABS; ++sl) {
            const int c = 32 * sl;
            if (c < bn && n0 + c < N) tma_store_2d(&tmC, stg_u32 + sl * TC_SLAB_BYTES, n0 + c, (int)m0);
          }
          tma_store_commit();
        }
        // bias gradient of the upstream layer = column sums of this product: taken from the staged slabs while TMA reads
        // them (lane = column, 32 conflict-free 4-byte reads per slab; rows past M are zero), so nobody re-reads C from HBM
        if (colsum_partial) {
#pragma unroll
          for (int sl = 0; sl < TC_SLABS; ++sl) {
            if (32 * sl < bn && n0 + 32 * sl < N) {
              float sum = 0.f;
#pragma unroll 8
              for (int r = 0; r < 32; ++r)
                sum += lds1(stg_u32 + sl * TC_SLAB_BYTES + r * 128 + ((((lane >> 2) ^ (r & 7)) << 4) | ((lane & 3) << 2)));
              colacc[sl] += sum;
            }
          }
        }
      }
    }
    if (colsum_partial) {
#pragma unroll
      for (int sl = 0; sl < TC_SLABS; ++sl)
        colsum_partial[((long long)blockIdx.x * 4 + ew) * 128 + sl * 32 + lane] = colacc[sl];
    }
    if (lane == 0) tma_store_wait_all();                           // global writes complete before the kernel exits
  }
  tc_fence_before();
  if (TWO) cluster_sync_all(); else __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    if (TWO) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------- TN (weight gradients)
// C[K1,N1] = A[M,K1]^T @ B[M,N1]: the contraction runs over the M utterance rows.  Same design as the NN kernel: the WIDE
// operand W (the one with more columns; 128-column tiles = the MMA M side) streams from HBM through a raw shared-memory
// ring, is split by one thread per column and goes to TENSOR MEMORY (lane = column, TMEM column = row of the 32-row
// chunk, i.e. K-major by construction -- the transposition costs nothing); the NARROW operand (<= 128 columns, the
// MMA N side) stays in shared memory as an MN-major tile ("128-byte swizzle with 32-byte atoms", UMMA layout type 1,
// TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B; the plain 128-byte swizzle silently produces zeros for MN-major tf32) for the
// tf32 hi*hi MMAs, is loaded a second time as plain boxes, and the epilogue warps turn that copy into a K-major bf16 tile
// (bf16(hi) | bf16(lo), the NN kernel's B16 layout) for the two bf16 correction MMAs.  When N1 > K1 the roles of A and B are swapped and the transposed result is written back by
// the reduction kernel.  Work unit = (128-column tile of W, row slab); each unit writes its [128 x n] partial to the
// workspace and a fixed-order reduction sums the slabs (bit-reproducible).  Same grouped-TMEM / register accumulation.
#ifndef TN_R_
#define TN_R_ 4
#endif
#ifndef TN_Q_
#define TN_Q_ 4
#endif
constexpr int TN_TA = 4;          // TMEM stages of W: tf32 hi 32 + bf16 pairs (hi 16, lo 16) columns
#ifndef TN_R2_
#define TN_R2_ 6
#endif
#ifndef TN_Q2_
#define TN_Q2_ 6
#endif
// Ring geometry.  Single CTA: R raw W stages of 16 KB ([32 rows][128 columns], no swizzle) and Q narrow stages of
// (swizzled fp32 tile 16 KB + bf16 tile 16 KB).  CTA pair: each CTA holds HALF of the narrow tile (64 columns: 8 + 8 KB per
// stage), so the narrow ring can be twice as deep in the same shared memory -- the pipeline trace of the single-CTA kernel
// (profiles/r02n_tn_trace.txt) has the narrow ring as the critical loop: stage freed by the MMAs -> TMA (~3100 clk under
// load) -> bf16 conversion (~600 clk) -> MMAs (~550 clk), i.e. ~4250 clk around a 4-stage ring.
template <bool TWO>
struct TnCfg {
  static constexpr int R = TWO ? TN_R2_ : TN_R_;
  static constexpr int Q = TWO ? TN_Q2_ : TN_Q_;
  static constexpr uint32_t NT_BYTES = TWO ? TC_B_BYTES / 2 : TC_B_BYTES;     // one narrow tile (fp32 or bf16) of this CTA
  static constexpr uint32_t SMEM_BYTES = R * TC_A_BYTES + Q * 2 * NT_BYTES + 1024 + 512;
  static constexpr int W_FULL = 0, W_FREE = W_FULL + R, TA_FULL = W_FREE + R, TA_FREE = TA_FULL + TN_TA,
                       B_FULL = TA_FREE + TN_TA, B_SPLIT = B_FULL + Q, B_FREE = B_SPLIT + Q, ACC_FULL = B_FREE + Q,
                       ACC_EMPTY = ACC_FULL + 2, BARS = ACC_EMPTY + 2;
  static_assert(SMEM_BYTES <= kMaxSmemPerBlock, "shared memory budget");
  static_assert(BARS * 8 + 8 <= 512, "barrier area");
};
constexpr int TN_THREADS = 352;   // 4 splitter + 4 epilogue warps, W producer, MMA, narrow-operand producer
#ifndef TN_GROUP_
#define TN_GROUP_ 8
#endif
#ifndef TN_DRAIN_AT_
#define TN_DRAIN_AT_ 2
#endif
// k-chunks accumulated inside TMEM before the round-to-nearest flush to registers.  8 (256 rows) instead of the NN kernel's
// 4: the epilogue warps of this kernel also split the narrow operand, and the pipeline trace (ERCG_TC_TRACE=2) showed the
// MMA warp waiting ~2000 clk at every group boundary for "drain the previous group, then split the next chunk".  Fewer,
// and mid-group, drains take that off the critical path; the truncation drift of a 256-row chain is ~1.6e-6 relative.
constexpr int TN_GROUP = TN_GROUP_;
constexpr int TN_DRAIN_AT = TN_DRAIN_AT_;     // the drain of group g-1 runs after this many chunks of group g were split

__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(4096 >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)1 << 61);
}

// WBF16: the wide operand W is stored in bf16 (the input features of the projection's weight gradient): raw tile 32 rows x 128
// bf16 columns (256-byte rows), W_hi = the value itself (exact in tf32), no W_lo => 4 tf32 + 2 bf16 MMAs per chunk instead of
// 4 + 4 and half the HBM bytes of the wide stream.
// TWO: CTA pairs (cluster of 2, cta_group::2).  Work unit = (PAIR of adjacent W tiles, slab): CTA rank r streams and splits
// W tile 2p + r into its own tensor memory, loads and converts the narrow columns [64 r, 64 r + 64) only, and the leader's MMA
// warp issues M = 256, N = 128 instructions for both.  Arrivals that the MMA warp waits for (TMEM operand written, narrow
// half converted, accumulator drained) go to the LEADER's barriers from both CTAs; everything the MMAs release (TMEM
// operand stages, narrow stages, accumulator stages) is a multicast commit to both CTAs.
template <bool WBF16, bool TWO>
__global__ void __launch_bounds__(TN_THREADS, 1)
gemm_tc_tn_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmN,
                  float* __restrict__ P /* [S][Wc][Nc] */, long long M, int Wc /* columns of the wide operand */,
                  int Nc /* columns of the narrow operand */, int bn /* narrow columns per unit: multiple of 32, <= 128 */,
                  int w_tiles, int n_tiles, int S, long long rows_per_slab, long long* trace) {
  using Cfg = TnCfg<TWO>;
  extern __shared__ uint8_t smem_raw[];
#ifdef ERCG_TRACE
#define TN_TRACE(role, idx, slot)                                                                                     \
  do {                                                                                                                \
    if (trace && blockIdx.x == 0 && (idx) < (unsigned)TR_N) trace[((role) * TR_N + (idx)) * 4 + (slot)] = clock64();   \
  } while (0)
#else
#define TN_TRACE(role, idx, slot) do { } while (0)
#endif
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* nring = smem + Cfg::R * TC_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(nring + Cfg::Q * 2 * Cfg::NT_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + Cfg::BARS);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = TWO ? cluster_ctarank() : 0u;     // 0 = leader (issues the MMAs of the pair)
  // barriers the MMA warp waits on collect both CTAs' warps: in pair mode ONE arrival per warp (lane 0, after __syncwarp)
  const uint32_t pair_arrivals = TWO ? 8u : 128u;
  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::R; ++i) { mbar_init(BAR(Cfg::W_FULL + i), 1); mbar_init(BAR(Cfg::W_FREE + i), 128); }
    for (int i = 0; i < TN_TA; ++i) { mbar_init(BAR(Cfg::TA_FULL + i), pair_arrivals); mbar_init(BAR(Cfg::TA_FREE + i), 1); }
    for (int i = 0; i < Cfg::Q; ++i) {
      mbar_init(BAR(Cfg::B_FULL + i), 1);
      mbar_init(BAR(Cfg::B_SPLIT + i), TWO ? 4u : 128u);     // pair mode: two conversion warps per CTA per chunk (teams)
      mbar_init(BAR(Cfg::B_FREE + i), 1);
    }
    for (int i = 0; i < 2; ++i) { mbar_init(BAR(Cfg::ACC_FULL + i), 1); mbar_init(BAR(Cfg::ACC_EMPTY + i), pair_arrivals); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 9) {
    if (TWO) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (TWO) cluster_sync_all(); else __syncthreads();      // the peer's barriers are initialised before anything arrives there
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int w_units = TWO ? (w_tiles + 1) / 2 : w_tiles;   // W tiles, or pairs of W tiles
  const long long units = (long long)w_units * n_tiles * S;
  const int nb = TWO ? bn / 64 : bn / 32;              // 32-wide boxes of the narrow operand THIS CTA loads and converts
  const int mma_n = TWO ? bn : (n_tiles == 1 ? (Nc + 15) / 16 * 16 : bn);   // UMMA N
  const long long u_first = TWO ? blockIdx.x / 2 : blockIdx.x, u_step = TWO ? gridDim.x / 2 : gridDim.x;
  // barriers of the leader as seen from this CTA (for the leader itself: its own)
  auto LBAR = [&](int i) { return TWO ? mapa_cta(BAR(i), 0u) : BAR(i); };
  auto arrive_leader = [&](uint32_t lbar) {
    if (TWO) {
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(lbar);
    } else {
      mbar_arrive(lbar);
    }
  };
  const uint32_t raw_base = smem_u32(smem), n_base = smem_u32(nring);
  // per narrow stage: [fp32 tile, MN-major swizzled: B of the tf32 MMAs AND the source of the bf16 conversion]
  //                   [bf16 tile, K-major 128-byte rows: bf16(hi) | bf16(lo) -- B of the bf16 MMAs, as in the NN kernel]
  auto N_HI = [&](int q) { return n_base + q * 2 * Cfg::NT_BYTES; };
  auto N_16 = [&](int q) { return n_base + q * 2 * Cfg::NT_BYTES + Cfg::NT_BYTES; };
  auto TA_HI = [&](int s) { return tmem_base + 2 * TC_BN + (uint32_t)s * 64u; };
  // unit -> (W tile, narrow tile, slab); slab fastest so that concurrently running CTAs stream different rows
  auto decode = [&](long long u, int& w0, int& n0, long long& mbeg, long long& mend, int& slab) {
    slab = (int)(u % S);
    const long long kn = u / S;
    w0 = TWO ? ((int)(kn / n_tiles) * 2 + (int)rank) * TC_BM : (int)(kn / n_tiles) * TC_BM;
    n0 = (int)(kn % n_tiles) * bn;
    mbeg = (long long)slab * rows_per_slab;
    mend = mbeg + rows_per_slab < M ? mbeg + rows_per_slab : M;
    if (mbeg > M) mbeg = M;
  };

  if (warp == 8) {
    if (lane == 0) {   // ---------------------------------------------------- wide-operand producer (HBM stream)
      uint32_t n = 0;
      for (long long u = u_first; u < units; u += u_step) {
        int w0, n0, slab; long long mbeg, mend;
        decode(u, w0, n0, mbeg, mend, slab);
        for (long long m = mbeg; m < mend; m += TC_BK, ++n) {
          const int r = n % Cfg::R;
          mbar_wait_relaxed(BAR(Cfg::W_FREE + r), ((n / Cfg::R) & 1) ^ 1);
          TN_TRACE(0, n, 1);
          mbar_expect_tx(BAR(Cfg::W_FULL + r), WBF16 ? TC_A_BYTES / 2 : TC_A_BYTES);
          tma_load_2d(raw_base + r * TC_A_BYTES, &tmW, w0, (int)m, BAR(Cfg::W_FULL + r));
        }
      }
    }
  } else if (warp == 10) {
    if (lane == 0) {   // ---------------------------------------------------- narrow-operand producer (mostly L2)
      uint32_t n = 0;
      const uint32_t tx = (uint32_t)nb * 4096u;
      for (long long u = u_first; u < units; u += u_step) {
        int w0, n0, slab; long long mbeg, mend;
        decode(u, w0, n0, mbeg, mend, slab);
        for (long long m = mbeg; m < mend; m += TC_BK, ++n) {
          const int q = n % Cfg::Q;
          mbar_wait_relaxed(BAR(Cfg::B_FREE + q), ((n / Cfg::Q) & 1) ^ 1);
          TN_TRACE(4, n, 1);
          mbar_expect_tx(BAR(Cfg::B_FULL + q), tx);
          for (int i = 0; i < nb; ++i)
            tma_load_2d(N_HI(q) + i * 4096, &tmN, n0 + (int)rank * (bn / 2) + 32 * i, (int)m, BAR(Cfg::B_FULL + q));
        }
      }
    }
  } else if (warp == 9 && rank == 0) {
    // ------------------------------------------------------------------------ MMA issuer (warp-uniform, elected lane)
    constexpr uint32_t MMA_M = TWO ? 2 * TC_BM : TC_BM;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) /* B is MN-major */ |
                           ((uint32_t)(mma_n >> 3) << 17) | ((uint32_t)(MMA_M >> 4) << 24);
    const uint32_t idesc16 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(mma_n >> 3) << 17) | ((uint32_t)(MMA_M >> 4) << 24);
    const uint64_t desc_k = ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61) | ((uint64_t)1 << 16);
    uint32_t n = 0;
    int a = 0;
    uint32_t aph = 0;
    for (long long u = u_first; u < units; u += u_step) {
      int w0, n0, slab; long long mbeg, mend;
      decode(u, w0, n0, mbeg, mend, slab);
      const long long chunks = (mend - mbeg + TC_BK - 1) / TC_BK;
      for (long long kc = 0; kc < chunks; ++kc, ++n) {
        const int in_group = (int)(kc % TN_GROUP);
        const uint32_t d_tmem = tmem_base + (uint32_t)(a * TC_BN);
        if (lane == 0) TN_TRACE(2, n, 0);
        if (in_group == 0) { if (TWO) mbar_wait_cluster(BAR(Cfg::ACC_EMPTY + a), aph ^ 1); else mbar_wait(BAR(Cfg::ACC_EMPTY + a), aph ^ 1); }
        if (lane == 0) TN_TRACE(2, n, 1);
        const int s = n % TN_TA, q = n % Cfg::Q;
        if (TWO) mbar_wait_cluster(BAR(Cfg::TA_FULL + s), (n / TN_TA) & 1); else mbar_wait(BAR(Cfg::TA_FULL + s), (n / TN_TA) & 1);
        if (lane == 0) TN_TRACE(2, n, 2);
        if (TWO) mbar_wait_cluster(BAR(Cfg::B_SPLIT + q), (n / Cfg::Q) & 1); else mbar_wait(BAR(Cfg::B_SPLIT + q), (n / Cfg::Q) & 1);
        if (lane == 0) TN_TRACE(2, n, 3);
        tc_fence_after();
        const uint32_t ah0 = TA_HI(s);
        const uint64_t bh0 = make_desc_mn_sw128(N_HI(q));
        const uint64_t b16 = desc_k | (uint64_t)((N_16(q) >> 4) & 0x3FFF);
        const bool last = in_group == TN_GROUP - 1 || kc == chunks - 1;
        if (elect_one()) {
          // W_hi * N_hi in tf32 (the fp32 tile is read with tf32 truncation = hi); the two correction terms in bf16
#pragma unroll
          for (int ks = 0; ks < TC_BK / 8; ++ks) {   // 8 rows = 1024 B
            if (TWO) tc_mma2_tf32_ts(d_tmem, ah0 + ks * 8, bh0 + (uint64_t)(ks * 64), idesc, (in_group | ks) ? 1u : 0u);
            else tc_mma_tf32_ts(d_tmem, ah0 + ks * 8, bh0 + (uint64_t)(ks * 64), idesc, (in_group | ks) ? 1u : 0u);
          }
#pragma unroll
          for (int j = 0; j < TC_BK / 16; ++j) {
            if (TWO) {
              if (!WBF16) tc_mma2_bf16_ts(d_tmem, ah0 + 48 + j * 8, b16 + (uint64_t)(j * 2), idesc16, 1u);
              tc_mma2_bf16_ts(d_tmem, ah0 + 32 + j * 8, b16 + (uint64_t)(4 + j * 2), idesc16, 1u);
            } else {
              if (!WBF16) tc_mma_bf16_ts(d_tmem, ah0 + 48 + j * 8, b16 + (uint64_t)(j * 2), idesc16, 1u);   // bf16(W_lo) * bf16(N_hi)
              tc_mma_bf16_ts(d_tmem, ah0 + 32 + j * 8, b16 + (uint64_t)(4 + j * 2), idesc16, 1u);    // bf16(W_hi) * bf16(N_lo)
            }
          }
          if (TWO) {
            tc_commit2(BAR(Cfg::TA_FREE + s));
            tc_commit2(BAR(Cfg::B_FREE + q));
            if (last) tc_commit2(BAR(Cfg::ACC_FULL + a));
          } else {
            tc_commit(BAR(Cfg::TA_FREE + s));
            tc_commit(BAR(Cfg::B_FREE + q));
            if (last) tc_commit(BAR(Cfg::ACC_FULL + a));
          }
        }
        __syncwarp();
        if (last) { if (++a == 2) { a = 0; aph ^= 1; } }
      }
    }
  } else if (warp < 4) {
    // ------------------------------------------------------------------------ splitter: thread = column of W = TMEM lane
    const int tid = threadIdx.x;
    const uint32_t lane_addr = (uint32_t)(warp * 32) << 16;
    uint32_t n = 0;
    for (long long u = u_first; u < units; u += u_step) {
      int w0, n0, slab; long long mbeg, mend;
      decode(u, w0, n0, mbeg, mend, slab);
      for (long long m = mbeg; m < mend; m += TC_BK, ++n) {
        const int r = n % Cfg::R, s = n % TN_TA;
        // raw [32 rows][128 columns] -> this thread's column, rows along the TMEM columns
        if (tid == 0) TN_TRACE(1, n, 0);
        mbar_wait(BAR(Cfg::W_FULL + r), (n / Cfg::R) & 1);
        if (tid == 0) TN_TRACE(1, n, 1);
        const uint32_t src = raw_base + r * TC_A_BYTES + (WBF16 ? tid * 2 : tid * 4);
        uint32_t hi[32], p16[32];                        // tf32 W_hi | bf16 pairs along the rows: [0,16) W_hi, [16,32) W_lo
        if (WBF16) {
#pragma unroll
          for (int j = 0; j < 32; j += 2) {               // raw [32 rows][128 bf16]: 256-byte rows
            const uint32_t b0 = lds_u16(src + j * 256), b1 = lds_u16(src + (j + 1) * 256);
            hi[j] = b0 << 16;                              // bf16 -> fp32 bit pattern: exact, and exact as a tf32 operand
            hi[j + 1] = b1 << 16;
            p16[j >> 1] = b0 | (b1 << 16);                 // element j at the even k position (low half)
            p16[16 + (j >> 1)] = 0u;
          }
        } else {
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          uint32_t l0, l1;
          split_tf32(lds1(src + j * 512), hi[j], l0);
          split_tf32(lds1(src + (j + 1) * 512), hi[j + 1], l1);
          p16[j >> 1] = pack_bf16x2(__uint_as_float(hi[j]), __uint_as_float(hi[j + 1]));
          p16[16 + (j >> 1)] = pack_bf16x2(__uint_as_float(l0), __uint_as_float(l1));
        }
        }
        mbar_wait(BAR(Cfg::TA_FREE + s), ((n / TN_TA) & 1) ^ 1);
        if (tid == 0) TN_TRACE(1, n, 2);
        tc_fence_after();
        tc_st32(TA_HI(s) + lane_addr, hi);
        tc_st32(TA_HI(s) + 32 + lane_addr, p16);
        tc_wait_st();
        mbar_arrive(BAR(Cfg::W_FREE + r));                 // after the TMEM stores: every loaded register has been consumed
        tc_fence_before();
        arrive_leader(LBAR(Cfg::TA_FULL + s));
        if (tid == 0) TN_TRACE(1, n, 3);
      }
    }
  } else if (warp < 8) {
    // ------------------------------------------------------------------------ epilogue warps: (1) hi/lo split of the narrow
    // operand, chunk by chunk (these warps are idle ~90 % of the time otherwise; on the splitter warps the split sat on
    // the critical path: profiles/r01_tn_v2_hot.txt), (2) accumulator drain, one group behind the split.
    int a = 0;
    uint32_t aph = 0;
    const int ew = warp & 3;
    const int te = threadIdx.x - 128;                  // 0..127
    uint32_t n = 0;                                    // chunk counter (narrow-operand ring)
    for (long long u = u_first; u < units; u += u_step) {
      int w0, n0, slab; long long mbeg, mend;
      decode(u, w0, n0, mbeg, mend, slab);
      const long long chunks = (mend - mbeg + TC_BK - 1) / TC_BK;
      const long long n_groups = (chunks + TN_GROUP - 1) / TN_GROUP;
      float acc[TC_BN];
#pragma unroll
      for (int j = 0; j < TC_BN; ++j) acc[j] = 0.f;
      auto drain = [&]() {
        mbar_wait(BAR(Cfg::ACC_FULL + a), aph);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < TC_BN; c += 32) {
          if (c < mma_n) {
            uint32_t rr[32];
            tc_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(a * TC_BN + c), rr);
            tc_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[c + j] += __uint_as_float(rr[j]);
          }
        }
        tc_fence_before();
        arrive_leader(LBAR(Cfg::ACC_EMPTY + a));
        if (++a == 2) { a = 0; aph ^= 1; }
      };
      for (long long g = 0; g < n_groups; ++g) {
        const long long kc_end = (g + 1) * TN_GROUP < chunks ? (g + 1) * TN_GROUP : chunks;
        bool pending = g > 0;                          // group g-1 still has to be drained (its MMAs retired long ago)
        for (long long kc = g * TN_GROUP; kc < kc_end; ++kc, ++n) {
          // pair mode: the conversion loop (barrier wait -> loads -> split -> stores -> proxy fence -> remote arrive, ~950 clk
          // per chunk for one warp however little it converts: profiles/r02o_tn_pair_trace.txt) was the slowest stage of the
          // pipeline, so the four warps form two TEAMS that take alternate chunks (thread = column, 64 columns per CTA).
          // Ownership goes by the parity of the GLOBAL chunk counter n and the ring depth is even, so a narrow stage
          // (q = n % Q) always belongs to the same team and only that team ever waits on its B_FULL barrier -- in every
          // phase.  (A first version had the other team wait on the skipped chunks' barriers "to keep the phase": a warp
          // whose arrival is not needed for a stage's reuse can be lapped by two phases, and a parity wait then blocks for
          // good.  It never happened in normal runs -- the conversion warps are ahead of the data -- but ncu's
          // instrumented replay pass slowed the warps enough to hang the kernel; profiles/README.md.)
          static_assert(!TWO || Cfg::Q % 2 == 0, "conversion teams own the narrow stages by parity");
          const int q = n % Cfg::Q;
          if (TWO && ((int)(n & 1u) != (ew >> 1))) continue;
          if (te == 0) TN_TRACE(3, n, 0);
          if (pending && kc - g * TN_GROUP >= TN_DRAIN_AT) { drain(); pending = false; if (te == 0) TN_TRACE(3, n, 3); }
          mbar_wait(BAR(Cfg::B_FULL + q), (n / Cfg::Q) & 1);
          if (te == 0) TN_TRACE(3, n, 1);
          // thread te = column te of the narrow tile: its 32 rows are read from the SAME swizzled MN-major tile the tf32 MMAs
          // use (layout type 1 = Swizzle<2,5,2>: the 32-byte atom index of a 128-byte row is XORed with the row index mod 4;
          // a warp reads one whole row per load, so the permutation inside the row keeps the 4-byte reads conflict-free --
          // a second, unswizzled TMA copy of the tile used to be the source: it doubled the L2 -> SM traffic of this operand,
          // and the kernel is bound by L2 slice throughput), are split hi / lo and go, as bf16 pairs along k, into row te
          // of the K-major bf16 tile (128-byte rows, 16-byte chunks XOR-swizzled with the row like a 128-byte-swizzle TMA
          // box: chunks 0-3 = bf16(hi), 4-7 = bf16(lo))
          if (TWO) {
            const int col = te & 63;                     // this team's 64 threads <-> the 64 columns of this CTA's half
            if (col < nb * 32) {
              const uint32_t src = N_HI(q) + (uint32_t)(col >> 5) * 4096u;
              const uint32_t cb = (uint32_t)(col & 31) * 4u;
              uint32_t p[32];
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                uint32_t h0, h1, l0, l1;
                split_tf32(lds1(src + j * 128 + (cb ^ (uint32_t)((j & 3) << 5))), h0, l0);
                split_tf32(lds1(src + (j + 1) * 128 + (cb ^ (uint32_t)(((j + 1) & 3) << 5))), h1, l1);
                p[j >> 1] = pack_bf16x2(__uint_as_float(h0), __uint_as_float(h1));
                p[16 + (j >> 1)] = pack_bf16x2(__uint_as_float(l0), __uint_as_float(l1));
              }
              const uint32_t dst = N_16(q) + (uint32_t)col * 128u;
#pragma unroll
              for (int c = 0; c < 8; ++c)
                sts4(dst + (uint32_t)((c ^ (col & 7)) << 4),
                     make_float4(__uint_as_float(p[4 * c]), __uint_as_float(p[4 * c + 1]), __uint_as_float(p[4 * c + 2]),
                                 __uint_as_float(p[4 * c + 3])));
            }
          } else
          if (te < nb * 32) {
            const uint32_t src = N_HI(q) + (uint32_t)(te >> 5) * 4096u;
            const uint32_t cb = (uint32_t)(te & 31) * 4u;
            uint32_t p[32];
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              uint32_t h0, h1, l0, l1;
              split_tf32(lds1(src + j * 128 + (cb ^ (uint32_t)((j & 3) << 5))), h0, l0);
              split_tf32(lds1(src + (j + 1) * 128 + (cb ^ (uint32_t)(((j + 1) & 3) << 5))), h1, l1);
              p[j >> 1] = pack_bf16x2(__uint_as_float(h0), __uint_as_float(h1));
              p[16 + (j >> 1)] = pack_bf16x2(__uint_as_float(l0), __uint_as_float(l1));
            }
            const uint32_t dst = N_16(q) + (uint32_t)te * 128u;
#pragma unroll
            for (int c = 0; c < 8; ++c)
              sts4(dst + (uint32_t)((c ^ (te & 7)) << 4),
                   make_float4(__uint_as_float(p[4 * c]), __uint_as_float(p[4 * c + 1]), __uint_as_float(p[4 * c + 2]),
                               __uint_as_float(p[4 * c + 3])));
          }
          fence_proxy_async();
          arrive_leader(LBAR(Cfg::B_SPLIT + q));
          if (te == 0) TN_TRACE(3, n, 2);
        }
        if (pending) drain();                          // (group shorter than TN_DRAIN_AT chunks)
      }
      drain();
      const int wc = w0 + ew * 32 + lane;
      if (wc < Wc) {
        float* prow = P + ((long long)slab * Wc + wc) * Nc + n0;
#pragma unroll
        for (int j = 0; j < TC_BN; ++j)
          if (j < bn && n0 + j < Nc) prow[j] = acc[j];
      }
    }
  }
  tc_fence_before();
  if (TWO) cluster_sync_all(); else __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    if (TWO) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// C = sum over slabs of P[s]; P[s] is [rows, cols] or, when the operand roles were swapped, [cols, rows] (transposed)
__global__ void tn_reduce_kernel(const float* __restrict__ P, long long stride, int S, float* __restrict__ C, long long ldc,
                                 int rows, int cols, int transposed) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)rows * cols) return;
  const int r = (int)(idx / cols), c = (int)(idx % cols);
  const long long src = transposed ? (long long)c * rows + r : idx;
  // four interleaved partial sums (slabs z, z+1, z+2, z+3 mod 4), fixed order: the S loads of a thread are independent, a
  // single running sum made them wait for each other (10 us per launch for a 100 x 100 result; four launches per step)
  const float* p = P + src;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int z = 0;
  for (; z + 3 < S; z += 4) {
    const float v0 = p[(long long)z * stride], v1 = p[(long long)(z + 1) * stride], v2 = p[(long long)(z + 2) * stride],
                v3 = p[(long long)(z + 3) * stride];
    s0 += v0; s1 += v1; s2 += v2; s3 += v3;
  }
  for (; z < S; ++z) s0 += p[(long long)z * stride];
  C[(long long)r * ldc + c] = (s0 + s1) + (s2 + s3);
}

// wide operand = the one with more columns; its 128-column tiles (or PAIRS of tiles, `two`) x row slabs are the work units
static bool tn_pairs_enabled() {
  static const bool on = [] { const char* e = getenv("ERCG_TN_PAIRS"); return !e || atoi(e) != 0; }();   // read once
  return on;
}
// CTA pairs that can be resident at once (1 CTA / SM, both SMs of a TPC).  A grid with more clusters than this runs in
// two waves.
static int tn_pair_capacity() {
  return resident_capacity<gemm_tc_tn_kernel<false, true>, 2>(TN_THREADS, TnCfg<true>::SMEM_BYTES);
}

static void tn_tc_plan(int64_t M, int K1, int N1, bool& swap, int& w_tiles, int& n_tiles, int& bn, int& S, long long& rps,
                       bool& two) {
  swap = N1 > K1;
  const int Wc = swap ? N1 : K1, Nc = swap ? K1 : N1;
  w_tiles = (Wc + TC_BM - 1) / TC_BM;
  const int cap = tn_pairs_enabled() && w_tiles % 2 == 0 ? tn_pair_capacity() : 0;
  two = cap > 0 && cap >= w_tiles / 2 * ((Nc + 127) / 128);         // CTA pairs need an even number of W tiles (no idle half pair)
  const int gran = two ? 64 : 32;                        // each CTA of a pair loads whole 32-column boxes of its half
  n_tiles = (Nc + 127) / 128;
  bn = ((Nc + n_tiles - 1) / n_tiles + gran - 1) / gran * gran;
  n_tiles = (Nc + bn - 1) / bn;
  const int w_units = two ? w_tiles / 2 : w_tiles;
  S = (two ? cap : kNumSMs) / (w_units * n_tiles);
  if (S < 1) S = 1;
  const long long quantum = (long long)TC_BK * TN_GROUP;
  long long maxS = (M + quantum - 1) / quantum;
  if (maxS < 1) maxS = 1;
  if (S > maxS) S = (int)maxS;
  rps = ((M + S - 1) / S + quantum - 1) / quantum * quantum;
  S = (int)((M + rps - 1) / rps);
}

// launch of either form; pairs = clusters of two CTAs on one TPC
template <bool WBF16>
static int tn_launch(bool two, const CUtensorMap& tmW, const CUtensorMap& tmN, float* P, long long M, int Wc, int Nc, int bn,
                     int wt, int nt, int S, long long rps, long long* tr, cudaStream_t st) {
  if (!smem_limit<gemm_tc_tn_kernel<WBF16, false>>(TnCfg<false>::SMEM_BYTES) ||
      !smem_limit<gemm_tc_tn_kernel<WBF16, true>>(TnCfg<true>::SMEM_BYTES))
    return ERCG_ECUDA;
  if (!two) {
    const long long units = (long long)wt * nt * S;
    const int grid = (int)(units < kNumSMs ? units : kNumSMs);
    gemm_tc_tn_kernel<WBF16, false><<<grid, TN_THREADS, TnCfg<false>::SMEM_BYTES, st>>>(tmW, tmN, P, M, Wc, Nc, bn, wt, nt, S, rps, tr);
    return finish_launch();
  }
  const long long units = (long long)(wt / 2) * nt * S;
  const int cap = tn_pair_capacity();
  const int pairs = (int)(units < cap ? units : cap);
  return launch_cluster(gemm_tc_tn_kernel<WBF16, true>, 2, 2 * pairs, TN_THREADS, TnCfg<true>::SMEM_BYTES, st, tmW, tmN, P, M,
                        Wc, Nc, bn, wt, nt, S, rps, tr);
}

// B[K,N] (row-major, ldb) -> Bt_hi [N, Kp] fp32 (K-major, tf32-rounded) and B16 [N, Kc, 64] bf16 (Kc = chunks of 32 k):
// per chunk the 32 values bf16(B_hi) followed by the 32 values bf16(B - B_hi), i.e. one 128-byte row per (n, chunk) so that
// a {64 x bn} TMA box lands as a 128-byte-swizzled K-major tile with the two bf16 operands side by side
__global__ void split_bt_kernel(const float* __restrict__ B, long long ldb, int K, int N, int Kp, int Kc, float* __restrict__ hi,
                                __nv_bfloat16* __restrict__ b16, int abf16 = 0) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int k = k0 + i, n = n0 + threadIdx.x;
    tile[i][threadIdx.x] = (k < K && n < N) ? B[(long long)k * ldb + n] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int n = n0 + i, k = k0 + threadIdx.x;
    if (n < N) {
      const float x = tile[threadIdx.x][i];                 // zero beyond K
      __nv_bfloat16* row = b16 + ((long long)n * Kc + blockIdx.x) * 64;
      if (abf16) {                                          // bf16-A kernel: B = b1 + b2, 16 significant bits, no fp32 copy
        const __nv_bfloat16 b1 = __float2bfloat16_rn(x);
        row[threadIdx.x] = b1;
        row[32 + threadIdx.x] = __float2bfloat16_rn(x - __bfloat162float(b1));
        continue;
      }
      const float h = rn_tf32(x);
      if (k < Kp) hi[(long long)n * Kp + k] = h;
      row[threadIdx.x] = __float2bfloat16_rn(h);
      row[32 + threadIdx.x] = __float2bfloat16_rn(x - h);
    }
  }
}

// out[c] = sum_b partial[b * ldp + c], fixed order, fp64 accumulation
__global__ void __launch_bounds__(256)
tc_colsum_final_kernel(const float* __restrict__ partial, int nblocks, int ldp, int N, float* __restrict__ out) {
  __shared__ double sm[FIN_ROWS][FIN_COLS + 1];
  const int c = blockIdx.x * FIN_COLS + (threadIdx.x & (FIN_COLS - 1));
  const double tot = fin_reduce(partial, nblocks, ldp, c, c < N, sm);
  if (threadIdx.x < FIN_COLS && c < N) out[c] = (float)tot;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  // cuTensorMapEncodeTiled is a DRIVER call: it needs a current context on the calling thread.  PyTorch runs backward passes on
  // its own autograd threads, where a tensor-core GEMM can be the first CUDA call (torch.empty served from the caching
  // allocator makes none) -> CUDA_ERROR_INVALID_CONTEXT (201).  One runtime call binds the primary context to the thread.
  static thread_local bool ctx_bound = false;
  if (!ctx_bound) {
    cudaFree(nullptr);
    ctx_bound = true;
  }
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D fp32 row-major [rows, cols] with row pitch `ld` floats; box {32 cols, box_rows}; 128-byte swizzle
static bool make_map(CUtensorMap* map, const float* base, long long rows, long long cols, long long ld, int box_rows,
                     CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// bf16 [rows, Kc*64] (row pitch Kc*128 bytes); box {64 elements = 128 bytes, box_rows}; 128-byte swizzle
static bool make_map_b16(CUtensorMap* map, const __nv_bfloat16* base, long long rows, long long kc, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {(cuuint64_t)kc * 64, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)kc * 128};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace ercg

using namespace ercg;

static long long* trace_buf = nullptr;      // ERCG_TC_TRACE=1: device buffer of the pipeline timeline (diagnostics only)

static bool nn_pairs_enabled() {
  static const bool on = [] { const char* e = getenv("ERCG_NN_PAIRS"); return !e || atoi(e) != 0; }();   // read once
  return on;
}
// CTA pairs of the NN kernel that can be resident at once (per device, queried once)
static int nn_pair_capacity() {
  const int n = resident_capacity<gemm_tc_nn_kernel<0, false, false, true, true>, 2>(TC_THREADS, NnCfg<true>::SMEM_BYTES);
  return n < kNumSMs / 2 ? n : kNumSMs / 2;
}

// dynamic shared memory of every NN kernel of activation ACT (the tables in ercg_gemm_nn_tc)
template <int ACT>
static bool nn_smem_limits() {
  return smem_limit<gemm_tc_nn_kernel<ACT, false, false>>(TC_SMEM_BYTES) &&
         smem_limit<gemm_tc_nn_kernel<ACT, true, false>>(TC_SMEM_BYTES) &&
         smem_limit<gemm_tc_nn_kernel<ACT, false, false, true, true>>(NnCfg<true, false>::SMEM_BYTES) &&
         smem_limit<gemm_tc_nn_kernel<ACT, true, false, true>>(NnCfg<true, true>::SMEM_BYTES) &&
         smem_limit<gemm_tc_nn_kernel<ACT, false, false, true>>(NnCfg<true, true>::SMEM_BYTES);
}

extern "C" size_t ercg_gemm_nn_tc_workspace_bytes(int N, int K) {
  if (N <= 0 || K <= 0) return 0;
  const size_t Kp = (size_t)(K + 3) / 4 * 4, Kc = (size_t)(K + TC_BK - 1) / TC_BK;
  return (size_t)N * Kp * sizeof(float) + (size_t)N * Kc * 128 /* bf16 pairs */ + 512 +
         (size_t)kNumSMs * 2 * 4 * 128 * sizeof(float) /* column-sum partials */;
}

// returns 1 when this shape/alignment can run on the tensor-core path
extern "C" int ercg_gemm_nn_tc_supported(const float* A, int64_t lda, const float* C, int64_t ldc, int64_t M, int N, int K) {
  if (M < 1 || N < 1 || K < 1) return 0;
  if ((lda & 3) || (ldc & 3) || !aligned16(A) || !aligned16(C)) return 0;
  if (M >= 2147483647LL || K >= (1 << 30)) return 0;
  return 1;
}

extern "C" int ercg_gemm_nn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                               int64_t ldc, int64_t M, int N, int K, int act, const float* aux, int64_t ldaux,
                               float aux_scale, float drop_p, uint64_t seed, const uint64_t* seed_dev, float* colsum_out,
                               void* workspace, size_t workspace_bytes, void* stream) {
  if (M < 0 || N < 0 || K < 0) return ERCG_EINVAL;
  if (colsum_out && (N > TC_BN || bias || act != ERCG_ACT_NONE)) return ERCG_EINVAL;
  if (M == 0 && colsum_out && N > 0) cudaMemsetAsync(colsum_out, 0, (size_t)N * sizeof(float), (cudaStream_t)stream);
  if (M == 0 || N == 0) return ERCG_OK;
  if (!A || !B || !C || lda < K || ldb < N || ldc < N || K == 0) return ERCG_EINVAL;
  if (act < 0 || act > 3 || (act == ERCG_ACT_MASK_POS && !aux)) return ERCG_EINVAL;
  if (act == ERCG_ACT_RELU_DROPOUT && !(drop_p >= 0.f && drop_p < 1.f)) return ERCG_EINVAL;
  if (!ercg_gemm_nn_tc_supported(A, lda, C, ldc, M, N, K) || (bias && !aligned16(bias))) return ERCG_EALIGN;
  if (workspace_bytes < ercg_gemm_nn_tc_workspace_bytes(N, K) || !workspace) return ERCG_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int Kp = (K + 3) / 4 * 4;
  const int Kc = (K + TC_BK - 1) / TC_BK;
  float* bhi = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  __nv_bfloat16* b16 = reinterpret_cast<__nv_bfloat16*>(
      (reinterpret_cast<uintptr_t>(bhi + (size_t)N * Kp) + 255) & ~uintptr_t(255));
  split_bt_kernel<<<dim3(Kc, (N + 31) / 32), dim3(32, 8), 0, st>>>(B, ldb, K, N, Kp, Kc, bhi, b16);
  int rc = finish_launch();
  if (rc) return rc;
  const int smallk = (K + TC_BK - 1) / TC_BK <= TC_GROUP ? 1 : 0;       // the whole K extent is one TMEM accumulation group
  const long long tiles = (M + TC_BM - 1) / TC_BM;          // a CTA owns whole M tiles (all their N tiles)
  // CTA pairs (cta_group::2): one N tile, or several with A resident in tensor memory; enough M tiles to fill the machine
  const bool pair_shape = N <= TC_BN || (K + TC_BK - 1) / TC_BK <= TC_TA;
  const int pair_cap = (pair_shape && tiles >= 2 * (kNumSMs / 2) && nn_pairs_enabled()) ? nn_pair_capacity() : 0;
  const bool two = pair_cap >= kNumSMs / 2 - 8;
  // UMMA N: multiple of 16 (pairs: of 32, half per CTA), <= 128, chosen to waste the fewest columns
  int bn = 128;
  if (N <= 128) bn = two ? (N + PAIR_N_GRAN - 1) / PAIR_N_GRAN * PAIR_N_GRAN : (N + 15) / 16 * 16;
  CUtensorMap tmA, tmBh, tmBl, tmC;
  const int b_box = two ? bn / 2 : bn;                      // B rows per TMA box: the whole tile, or this CTA's half
  if (!make_map(&tmA, A, M, K, lda, TC_BM) || !make_map(&tmBh, bhi, N, K, Kp, b_box) || !make_map_b16(&tmBl, b16, N, Kc, b_box) ||
      !make_map(&tmC, C, M, N, ldc, 32))                     // output: boxes of 32 rows x 32 columns (TMA bulk stores)
    return ERCG_ECUDA;
  typedef void (*NnKernel)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, float*, long long, long long, int, int, int,
                           TcEpilogue, float*);
  static const NnKernel kernels[4][2] = {
      {gemm_tc_nn_kernel<0, false, false>, gemm_tc_nn_kernel<0, true, false>}, {gemm_tc_nn_kernel<1, false, false>, gemm_tc_nn_kernel<1, true, false>},
      {gemm_tc_nn_kernel<2, false, false>, gemm_tc_nn_kernel<2, true, false>}, {gemm_tc_nn_kernel<3, false, false>, gemm_tc_nn_kernel<3, true, false>}};
  // [act][0 long K: one-slab staging | 1 small K | 2 medium K: wide staging]
  static const NnKernel pair_kernels[4][3] = {
      {gemm_tc_nn_kernel<0, false, false, true, true>, gemm_tc_nn_kernel<0, true, false, true>, gemm_tc_nn_kernel<0, false, false, true>},
      {gemm_tc_nn_kernel<1, false, false, true, true>, gemm_tc_nn_kernel<1, true, false, true>, gemm_tc_nn_kernel<1, false, false, true>},
      {gemm_tc_nn_kernel<2, false, false, true, true>, gemm_tc_nn_kernel<2, true, false, true>, gemm_tc_nn_kernel<2, false, false, true>},
      {gemm_tc_nn_kernel<3, false, false, true, true>, gemm_tc_nn_kernel<3, true, false, true>, gemm_tc_nn_kernel<3, false, false, true>}};
  const int pair_kind = smallk ? 1 : ((K + TC_BK - 1) / TC_BK > 16 ? 0 : 2);
  if (!nn_smem_limits<0>() || !nn_smem_limits<1>() || !nn_smem_limits<2>() || !nn_smem_limits<3>()) return ERCG_ECUDA;
  const int num_sms = device_sm_count();
  const int grid = two ? 2 * pair_cap : (int)(tiles < num_sms ? tiles : num_sms);
  static int dbg = -1;
  if (dbg < 0) { const char* e = getenv("ERCG_TC_DBG"); dbg = e ? atoi(e) : 0; }
  static int trace_on = -1;
  if (trace_on < 0) {
    const char* e = getenv("ERCG_TC_TRACE");
    trace_on = e ? atoi(e) : 0;
    if (trace_on && cudaMalloc(&trace_buf, sizeof(long long) * TR_ROLES * TR_N * 4) != cudaSuccess) trace_buf = nullptr;
  }
  long long* nn_trace = (trace_on & 1) ? trace_buf : nullptr;
  if (nn_trace) cudaMemsetAsync(nn_trace, 0, sizeof(long long) * TR_ROLES * TR_N * 4, st);
  TcEpilogue ep{bias, act, aux, (long long)ldaux, aux_scale, drop_p, (unsigned long long)seed, dbg, nn_trace};
  ep.seed_dev = reinterpret_cast<const unsigned long long*>(seed_dev);
  float* partial = colsum_out ? reinterpret_cast<float*>(b16 + (size_t)N * Kc * 64) : nullptr;   // [grid][4][128], after the B copies
  if (two) {
    const int pair_smem = pair_kind == 0 ? NnCfg<true, false>::SMEM_BYTES : NnCfg<true, true>::SMEM_BYTES;
    rc = launch_cluster(pair_kernels[act][pair_kind], 2, grid, TC_THREADS, pair_smem, st, tmA, tmBh, tmBl, tmC, C, ldc, M, N,
                        K, bn, ep, partial);
  } else {
    kernels[act][smallk]<<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(tmA, tmBh, tmBl, tmC, C, ldc, M, N, K, bn, ep, partial);
    rc = finish_launch();
  }
  if (rc || !colsum_out) return rc;
  tc_colsum_final_kernel<<<fin_blocks(N), 256, 0, st>>>(partial, grid * 4, 128, N, colsum_out);
  return finish_launch();
}

// diagnostics: copy out the pipeline timeline CTA 0 recorded during the last ercg_gemm_nn_tc launch (ERCG_TC_TRACE=1)
extern "C" int ercg_gemm_nn_tc_trace(long long* host_out /* [5][160][4] clock64 values, 0 = not recorded */) {
#ifndef ERCG_TRACE
  (void)host_out;
  return ERCG_EINVAL;                       // library built without -DERCG_TRACE
#endif
  if (!host_out || !trace_buf) return ERCG_EINVAL;
  return cudaMemcpy(host_out, trace_buf, sizeof(long long) * TR_ROLES * TR_N * 4, cudaMemcpyDeviceToHost) == cudaSuccess
             ? ERCG_OK : ERCG_ECUDA;
}

extern "C" size_t ercg_gemm_tn_tc_workspace_bytes(int64_t M, int K1, int N1) {
  if (M <= 0 || K1 <= 0 || N1 <= 0) return 0;
  bool swap, two; int wt, nt, bn, S; long long rps;
  tn_tc_plan(M, K1, N1, swap, wt, nt, bn, S, rps, two);
  return (size_t)S * K1 * N1 * sizeof(float) + 256;
}

extern "C" int ercg_gemm_tn_tc_supported(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int K1, int N1) {
  if (M < 1 || K1 < 1 || N1 < 1) return 0;
  if ((lda & 3) || (ldb & 3) || !aligned16(A) || !aligned16(B)) return 0;
  if (M >= 2147483647LL) return 0;
  return 1;
}

// 2-D fp32 row-major [rows, cols]; box {128 cols, 32 rows}, no swizzle (the raw W tile is only read by the splitter)
static bool make_map_plain(CUtensorMap* map, const float* base, long long rows, long long cols, long long ld) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)TC_BM, (cuuint32_t)TC_BK};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

extern "C" int ercg_gemm_tn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                               int K1, int N1, void* workspace, size_t workspace_bytes, void* stream) {
  if (M < 1 || K1 < 1 || N1 < 1 || !A || !B || !C || lda < K1 || ldb < N1 || ldc < N1) return ERCG_EINVAL;
  if (!ercg_gemm_tn_tc_supported(A, lda, B, ldb, M, K1, N1)) return ERCG_EALIGN;
  if (workspace_bytes < ercg_gemm_tn_tc_workspace_bytes(M, K1, N1) || !workspace) return ERCG_EWORKSPACE;
  bool swap, two; int wt, nt, bn, S; long long rps;
  tn_tc_plan(M, K1, N1, swap, wt, nt, bn, S, rps, two);
  float* P = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  const float* W = swap ? B : A;
  const float* Nw = swap ? A : B;
  const long long ldw = swap ? ldb : lda, ldn = swap ? lda : ldb;
  const int Wc = swap ? N1 : K1, Nc = swap ? K1 : N1;
  CUtensorMap tmW, tmN;
  if (!make_map_plain(&tmW, W, M, Wc, ldw) ||
      !make_map(&tmN, Nw, M, Nc, ldn, TC_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return ERCG_ECUDA;
  cudaStream_t st = (cudaStream_t)stream;
  static int tn_trace_on = -1;
  if (tn_trace_on < 0) {
    const char* e = getenv("ERCG_TC_TRACE");
    tn_trace_on = e ? atoi(e) : 0;
    if (tn_trace_on && !trace_buf && cudaMalloc(&trace_buf, sizeof(long long) * TR_ROLES * TR_N * 4) != cudaSuccess) trace_buf = nullptr;
  }
  long long* tr = (tn_trace_on & 2) ? trace_buf : nullptr;          // ERCG_TC_TRACE=2: trace the TN kernel instead of the NN one
  if (tr) cudaMemsetAsync(tr, 0, sizeof(long long) * TR_ROLES * TR_N * 4, st);
  int rc = tn_launch<false>(two, tmW, tmN, P, M, Wc, Nc, bn, wt, nt, S, rps, tr, st);
  if (rc) return rc;
  const long long tot = (long long)K1 * N1;
  tn_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(P, tot, S, C, ldc, K1, N1, swap ? 1 : 0);
  return finish_launch();
}


// ---------------------------------------------------------------------------------------------- bf16 input-feature mode
// The streamed operand of the input projection (x [N, hidden_all], 5.8 of the ~21 KB/utterance the step has to move) stored
// in bf16: ercg_gemm_nn_tc_bf16a = x @ W + b (forward), ercg_gemm_tn_tc_bf16a = x^T @ dF (weight gradient).  fp32
// accumulation, fp32 outputs, weights / gradients fp32 in HBM; the only approximation relative to the fp32 path is the
// rounding of x itself (done once, where the data set is stored) plus 16-bit weights inside the forward product.
namespace ercg {
static int g_last_map_result = 0;
static bool make_map_bf16_rows(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld_elems,
                               int box_cols, int box_rows, CUtensorMapSwizzle swz) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld_elems * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  g_last_map_result = (int)enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return g_last_map_result == 0;
}
}  // namespace ercg

extern "C" int ercg_gemm_bf16a_supported(const void* A, int64_t lda, int64_t M, int K) {
  if (M < 1 || K < 1 || !A) return 0;
  if ((lda & 7) || !aligned16(A) || lda < K) return 0;            // 16-byte aligned bf16 rows
  if (M >= 2147483647LL || K >= (1 << 30)) return 0;
  return 1;
}

extern "C" int ercg_gemm_nn_tc_bf16a(const void* A_bf16, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                                     int64_t ldc, int64_t M, int N, int K, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  if (M < 0 || N < 0 || K < 0) return ERCG_EINVAL;
  if (M == 0 || N == 0) return ERCG_OK;
  if (!A_bf16 || !B || !C || ldb < N || ldc < N || K == 0) return ERCG_EINVAL;
  if (!ercg_gemm_bf16a_supported(A_bf16, lda, M, K) || (ldc & 3) || !aligned16(C) || (bias && !aligned16(bias))) return ERCG_EALIGN;
  if (workspace_bytes < ercg_gemm_nn_tc_workspace_bytes(N, K) || !workspace) return ERCG_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int Kp = (K + 3) / 4 * 4;
  const int Kc = (K + TC_BK - 1) / TC_BK;
  float* bhi = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  __nv_bfloat16* b16 = reinterpret_cast<__nv_bfloat16*>(
      (reinterpret_cast<uintptr_t>(bhi + (size_t)N * Kp) + 255) & ~uintptr_t(255));
  split_bt_kernel<<<dim3(Kc, (N + 31) / 32), dim3(32, 8), 0, st>>>(B, ldb, K, N, Kp, Kc, bhi, b16, 1);
  int rc = finish_launch();
  if (rc) return rc;
  int bn = 128;
  if (N <= 128) bn = (N + 15) / 16 * 16;
  CUtensorMap tmA, tmBl, tmC;
  if (!make_map_bf16_rows(&tmA, A_bf16, M, K, lda, TC_BK, TC_BM, CU_TENSOR_MAP_SWIZZLE_64B) ||
      !make_map_b16(&tmBl, b16, N, Kc, bn) || !make_map(&tmC, C, M, N, ldc, 32))
    return ERCG_ECUDA;
  typedef void (*NnKernel)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, float*, long long, long long, int, int, int,
                           TcEpilogue, float*);
  static const NnKernel kernels[2] = {gemm_tc_nn_kernel<0, false, true>, gemm_tc_nn_kernel<0, true, true>};
  if (!smem_limit<gemm_tc_nn_kernel<0, false, true>>(TC_SMEM_BYTES) || !smem_limit<gemm_tc_nn_kernel<0, true, true>>(TC_SMEM_BYTES))
    return ERCG_ECUDA;
  const int num_sms = device_sm_count();
  const long long tiles = (M + TC_BM - 1) / TC_BM;
  const int grid = (int)(tiles < num_sms ? tiles : num_sms);
  TcEpilogue ep{bias, ERCG_ACT_NONE, nullptr, 0, 1.f, 0.f, 0ull, 0, nullptr};
  const int smallk = (K + TC_BK - 1) / TC_BK <= TC_GROUP ? 1 : 0;
  kernels[smallk]<<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(tmA, tmBl /* unused fp32 slot */, tmBl, tmC, C, ldc, M, N, K, bn, ep, nullptr);
  return finish_launch();
}

extern "C" int ercg_gemm_tn_tc_bf16a(const void* A_bf16, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                                     int64_t M, int K1, int N1, void* workspace, size_t workspace_bytes, void* stream) {
  if (M < 1 || K1 < 1 || N1 < 1 || !A_bf16 || !B || !C || ldb < N1 || ldc < N1) return ERCG_EINVAL;
  if (N1 > K1 || N1 > 128) return ERCG_EINVAL;                    // the bf16 operand must be the wide one (K1 >= N1), one narrow tile
  if (!ercg_gemm_bf16a_supported(A_bf16, lda, M, K1) || (ldb & 3) || !aligned16(B)) return ERCG_EALIGN;
  if (workspace_bytes < ercg_gemm_tn_tc_workspace_bytes(M, K1, N1) || !workspace) return ERCG_EWORKSPACE;
  bool swap, two; int wt, nt, bn, S; long long rps;
  tn_tc_plan(M, K1, N1, swap, wt, nt, bn, S, rps, two);
  if (swap) return ERCG_EINVAL;
  float* P = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  CUtensorMap tmW, tmN;
  if (!make_map_bf16_rows(&tmW, A_bf16, M, K1, lda, TC_BM, TC_BK, CU_TENSOR_MAP_SWIZZLE_NONE)) return ERCG_ECUDA;
  if (!make_map(&tmN, B, M, N1, ldb, TC_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) return ERCG_ECUDA;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = tn_launch<true>(two, tmW, tmN, P, M, K1, N1, bn, wt, nt, S, rps, nullptr, st);
  if (rc) return rc;
  const long long tot = (long long)K1 * N1;
  tn_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(P, tot, S, C, ldc, K1, N1, 0);
  return finish_launch();
}
