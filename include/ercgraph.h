/*
 * ercgraph.h -- C ABI of libercgraph.so: the B200 (sm_100a) conversation-graph hot path of
 * sailist/emotion-recognition-in-conversation (track_mm COGMEN / DialogueGCN / MMGCN / DAG-ERC).
 *
 * The reference has NO FFI / plugin registry: its boundary is "Python imports a function and calls
 * it with torch tensors" (SURVEY.md section 8b).  This header is therefore the boundary a binding
 * would use: every entry point takes raw DEVICE pointers + sizes + a CUDA stream (as void*), never
 * allocates, never synchronises, keeps no global state, launches on the stream it is given and
 * returns 0 or a negative ERCG_E* code (text via ercg_strerror).  Outputs and workspaces are
 * caller-allocated; the companion *_workspace_bytes functions say how much.
 *
 * Each entry point cites the reference code (path:line under the reference tree) it replaces.
 * Graph convention everywhere (track_mm/cogmen_utils.py:125-140, models/rgcn.py:133,158):
 *   edge (j -> k): j = source = edge_index[0], k = destination = edge_index[1]; messages are
 *   aggregated at k.  "CSR" = by destination (rowptr/col/etype), "transpose" = by source
 *   (t_rowptr/t_col/t_etype/t_eid, t_eid = position of that edge in the by-destination order).
 * All feature matrices are row-major fp32 with an explicit leading dimension in ELEMENTS.
 */
#ifndef ERCGRAPH_H_
#define ERCGRAPH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden: only this header is exported */
#endif

#define ERCG_OK 0
#define ERCG_EINVAL (-1)   /* bad argument (null pointer, negative size, unsupported combination) */
#define ERCG_EALIGN (-2)   /* pointer / leading dimension not aligned as the kernel requires */
#define ERCG_ERANGE (-3)   /* size exceeds what the packed int32/uint8 formats can hold */
#define ERCG_ECUDA (-4)    /* CUDA runtime reported an error at launch (cudaGetLastError) */
#define ERCG_EWORKSPACE (-5) /* workspace too small */
#define ERCG_P2P_ETIMEOUT (-6) /* a peer did not arrive at a peer-memory collective within 30 s (ercg_p2p_status) */

#define ERCG_GRAPH_ELENGTH 1   /* a dialogue is longer than the padded speaker width spk_ld */
#define ERCG_GRAPH_ESPEAKER 2  /* a speaker id outside [0, n_speakers) */
#define ERCG_GRAPH_ESIZE 4     /* the caller's N / E are smaller than the lengths imply: dialogues were skipped */
#define ERCG_GRAPH_ECENSUS 8   /* an edge carries a relation id missing from the caller's table (ercg_graphify_check_census) */

#define ERCG_ACT_NONE 0
#define ERCG_ACT_RELU 1
#define ERCG_ACT_RELU_DROPOUT 2   /* relu then inverted dropout (mask from a counter hash of seed,row,col) */
#define ERCG_ACT_MASK_POS 3       /* C = (A@B) * (aux[m,n] > 0 ? aux_scale : 0): relu/dropout backward */

const char* ercg_strerror(int code);
int ercg_version(void);
/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
unsigned long long ercg_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * K1  batch_graphify: window edges + speaker-pair/direction relation typing as ONE integer kernel
 * emitting a packed CSR (and its by-source transpose) over the whole batch of dialogues.
 * Replaces edge_perms (track_mm/cogmen_utils.py:147-172 = dgcn_models.py:95-118) and the per-edge
 * python loop of batch_graphify (cogmen_utils.py:109-144, dgcn_models.py:51-92).
 *   edges of dialogue d (length L): (j -> k) for max(0,j-wp) <= k <= min(L-1,j+wf); wp/wf = -1 unbounded
 *   type(j -> k) = ((spk_j * n_speakers + spk_k) * 2) + (j >= k)         (cogmen.py:124-129)
 * Canonical edge order = ascending dialogue, then destination k, then source j.
 * ------------------------------------------------------------------------------------------- */

/* Host-side closed form: N = sum L, E = sum |E_d|.  lengths_host is a HOST array. */
int ercg_graphify_sizes_host(const int64_t* lengths_host, int B, int wp, int wf, int64_t* N_out, int64_t* E_out);

/* Device-side totals when lengths live on the GPU: totals_dev[0]=N, totals_dev[1]=E. */
int ercg_graphify_count(const void* lengths_dev, int lengths_is_i64, int B, int wp, int wf,
                        int64_t* totals_dev, void* stream);

size_t ercg_graphify_workspace_bytes(int B);

typedef struct ercg_graph_out {
  /* required (device) */
  int32_t* node_off;   /* [B+1] first node of each dialogue */
  int32_t* edge_off;   /* [B+1] first edge of each dialogue */
  int32_t* rowptr;     /* [N+1] CSR by destination */
  int32_t* col;        /* [E]   source node of each edge */
  uint8_t* etype;      /* [E]   relation id */
  int32_t* t_rowptr;   /* [N+1] by source */
  int32_t* t_col;      /* [E]   destination node */
  uint8_t* t_etype;    /* [E] */
  int32_t* t_eid;      /* [E]   index of the same edge in by-destination order */
  int32_t* spk;        /* [N]   packed speaker ids */
  int32_t* node_dlg;   /* [N]   dialogue of each node */
  /* optional (may be NULL) */
  float* inv_cnt;      /* [E]   1/|{e' : dst(e')=dst(e), type(e')=type(e)}| -- PyG RGCNConv aggr='mean' weight */
  int64_t* edge_index; /* [2,E] reference layout (row0 = j, row1 = k), cogmen_utils.py:140 */
  int64_t* edge_type;  /* [E]   cogmen_utils.py:141 */
  int64_t* edge_index_lengths; /* [B] cogmen_utils.py:142 */
  int64_t* totals;     /* [2]   N, E as computed on the device (for validation) */
  int32_t* pad_row;    /* [N]   d*spk_ld + k: row of the node in a padded [B,spk_ld,*] tensor (node id if spk_ld=0) */
  int32_t* rel_info;   /* [516] relation census: [0] = P = number of relation ids that occur on at least one edge,
                          [1 + r] = compact slot of relation id r (-1 if no edge has it), [257 + s] = id of slot s (s < P).
                          One-speaker data (MOSEI, mosei_feature.py:211) uses 2 of the 2n^2 = 8 ids of cogmen.py:64.
                          [513] = input-error flags (0 = clean), OR of ERCG_GRAPH_E*: the kernel never reads or writes out
                          of bounds on bad input, it clamps and reports here (the reference raises IndexError / KeyError
                          at cogmen_utils.py:131-137); [514], [515] reserved (0). */
} ercg_graph_out;

/* speakers: padded [B, spk_ld] when spk_ld > 0 (reference layout), packed [N] when spk_ld == 0. */
int ercg_graphify_csr(const void* lengths_dev, int lengths_is_i64, int B,
                      const void* speakers_dev, int speakers_is_i64, int64_t spk_ld,
                      int wp, int wf, int n_speakers, int64_t N, int64_t E,
                      const ercg_graph_out* out, void* workspace, size_t workspace_bytes, void* stream);

/* For callers that know the possible relation ids up front (from the speaker ids on the host) and use their own
 * id -> slot table instead of waiting for the census of rel_info: ORs ERCG_GRAPH_ECENSUS into rel_info[513] when an edge
 * of the graph carries an id r with r >= n_allowed or allowed_slots[r] < 0.  Run it right after ercg_graphify_csr. */
int ercg_graphify_check_census(const int32_t* allowed_slots, int n_allowed, int32_t* rel_info, void* stream);

/* padded [B,Lmax,D] (row stride ld) -> packed [N,D]: the torch.cat of cogmen_utils.py:123,139 and
 * simple_batch_graphify (track_mm/mmgcn_utils.py:5-21, seq_first=1 for its [L,B,D] layout). */
int ercg_pack_rows(const float* padded, int64_t ld, int64_t Lmax, int B, int seq_first,
                   const int32_t* node_off, const int32_t* node_dlg, float* packed, int64_t ldp,
                   int64_t N, int D, void* stream);
/* backward of the above: scatter packed gradients into a zero-initialised padded tensor */
int ercg_unpack_rows(const float* packed, int64_t ldp, const int32_t* node_off, const int32_t* node_dlg,
                     float* padded, int64_t ld, int64_t Lmax, int B, int seq_first, int64_t N, int D, void* stream);

/* ERCCollate's small tensors (track_mm/mmbase.py:354-371,417-428) built on the device from the packed layout: the host
 * uploads packed rows only (no padding bytes cross PCIe) and the padded tensors the reference's batch dict carries are
 * produced here -- ercg_unpack_rows for the feature tensors, this call for
 *   attention_mask [B,Lmax] f32 (1 inside a dialogue), speaker ids [B,Lmax] int64 (padding = 0; [Lmax,B] when seq_first,
 *   i.e. not batch_first) and/or their one-hot [.., n_onehot] f32 (speaker_onehot).  Any output may be NULL. */
int ercg_collate_masks(const int32_t* node_off, const int64_t* speaker_packed, int B, int64_t Lmax, int seq_first,
                       int n_onehot, float* attention_mask, int64_t* speaker_ids, float* speaker_onehot, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  dense feature transforms.  C[M,N] = act(A[M,K] @ B[K,N] + bias[N]).
 * Replaces nn.Linear (cogmen.py:103-105,116-122), the per-relation weights of PyG RGCNConv
 * (cogmen.py:65) / vendored RGCNConv.message (models/rgcn.py:329-343) as one GEMM against the
 * concatenated [K,(R+1)*out] matrix, and the four Linears of TransformerConv (cogmen.py:66).
 * a_rows (optional): row m of the product reads A row a_rows[m] (fused padded->packed gather).
 * act = ERCG_ACT_*; aux/ldaux/aux_scale used by RELU_DROPOUT (aux_scale = keep prob handled via
 * drop_p) and MASK_POS.  fp32 in, fp32 accumulate, fp32 out.
 * ------------------------------------------------------------------------------------------- */
int ercg_gemm_nn(const float* A, int64_t lda, const int32_t* a_rows, const float* B, int64_t ldb,
                 const float* bias, float* C, int64_t ldc, int64_t M, int N, int K, int act,
                 const float* aux, int64_t ldaux, float aux_scale, float drop_p, uint64_t seed,
                 const uint64_t* seed_dev, void* stream);
/* seed_dev (optional, device): the dropout mask is drawn from seed + *seed_dev.  Point it at a device-resident step counter
 * (ercg_adam_step's) and a train step captured once in a CUDA graph draws a fresh mask on every replay. */

/* Tensor-core variant of ercg_gemm_nn (tcgen05 kind::tf32, TMA-staged 128-byte-swizzled tiles, TMEM
 * accumulators).  fp32-grade accuracy through the 3xTF32 split (hi/lo of both operands, fp32 accumulate);
 * same arguments and epilogues, plus a workspace for the K-major hi/lo copies of B.  Requirements
 * (ercg_gemm_nn_tc_supported): A and C 16-byte aligned with lda, ldc multiples of 4, no row gather. */
size_t ercg_gemm_nn_tc_workspace_bytes(int N, int K);
int ercg_gemm_nn_tc_supported(const float* A, int64_t lda, const float* C, int64_t ldc, int64_t M, int N, int K);
int ercg_gemm_nn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                    int64_t ldc, int64_t M, int N, int K, int act, const float* aux, int64_t ldaux,
                    float aux_scale, float drop_p, uint64_t seed, const uint64_t* seed_dev, float* colsum_out,
                    void* workspace, size_t workspace_bytes, void* stream);
/* colsum_out (optional, [N]; needs N <= 128, bias == NULL, act == ERCG_ACT_NONE): also returns the column sums of C,
 * reduced from the tiles while they sit in shared memory -- the bias gradient of the layer that produced A's operand
 * (the input gradient dX = dZ @ W^T of one Linear is the dZ whose column sums the previous Linear needs). */

/* Diagnostics (library built with -DERCG_TRACE and ERCG_TC_TRACE=1 / 2 in the environment): CTA 0 of ercg_gemm_nn_tc (1) or
 * ercg_gemm_tn_tc (2) records clock64() per pipeline role and k-chunk; this copies the [5 roles][160 chunks][4 marks] table
 * of the last launch to the host (synchronous).  Returns ERCG_EINVAL in a normal build. */
int ercg_gemm_nn_tc_trace(long long* host_out);

/* C[K1,N1] = A[M,K1]^T @ B[M,N1]  (weight gradients; contraction over the M utterance rows, split
 * across CTAs into fixed slabs and reduced in a fixed order => bit-reproducible). */
size_t ercg_gemm_tn_workspace_bytes(int64_t M, int K1, int N1);
int ercg_gemm_tn(const float* A, int64_t lda, const int32_t* a_rows, const float* B, int64_t ldb,
                 float* C, int64_t ldc, int64_t M, int K1, int N1,
                 void* workspace, size_t workspace_bytes, void* stream);

/* Tensor-core variant of ercg_gemm_tn (both operands MN-major for tcgen05, both hi/lo-split in shared memory). */
size_t ercg_gemm_tn_tc_workspace_bytes(int64_t M, int K1, int N1);
int ercg_gemm_tn_tc_supported(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int K1, int N1);
int ercg_gemm_tn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                    int K1, int N1, void* workspace, size_t workspace_bytes, void* stream);

/* bf16 INPUT-FEATURE MODE (BASELINE.json north_star: "stated separately for bf16").  The streamed operand A -- the
 * utterance features x [N, hidden_all] of the input projection nn.Linear(hidden_all, 100) (cogmen.py:103-105,146-147), 5.8 of
 * the ~21 KB/utterance a train step has to move -- is STORED in bf16 (uint16 bit patterns, row pitch lda ELEMENTS, a multiple
 * of 8 so rows are 16-byte aligned); weights, bias, outputs and gradients stay fp32, accumulation is fp32.
 *   ercg_gemm_nn_tc_bf16a   C[M,N]   = A @ B + bias        (forward; B enters with 16 significant bits)
 *   ercg_gemm_tn_tc_bf16a   C[K1,N1] = A^T @ Bg            (weight gradient; Bg fp32 through the hi/lo split; K1 >= N1, N1 <= 128)
 * Half the HBM (and host->device) bytes of the two largest kernels of the COGMEN step; results equal the fp32 path run on the
 * bf16-ROUNDED features to ~1e-5 (tests/test_gpu_bf16_mode.py), i.e. the mode's error is the rounding of the stored features.
 * Workspaces: ercg_gemm_nn_tc_workspace_bytes(N, K) / ercg_gemm_tn_tc_workspace_bytes(M, K1, N1). */
int ercg_gemm_bf16a_supported(const void* A_bf16, int64_t lda, int64_t M, int K);
int ercg_gemm_nn_tc_bf16a(const void* A_bf16, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                          int64_t ldc, int64_t M, int N, int K, void* workspace, size_t workspace_bytes, void* stream);
int ercg_gemm_tn_tc_bf16a(const void* A_bf16, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                          int64_t M, int K1, int N1, void* workspace, size_t workspace_bytes, void* stream);

/* out = ref > 0 ? x * scale : 0  -- backward of ReLU / ReLU+inverted-dropout given the forward OUTPUT
 * (cls of cogmen.py:116-122, Classifier of dgcn_models.py:163-170). */
int ercg_mask_pos(const float* x, int64_t ldx, const float* ref, int64_t ldr, float scale,
                  float* out, int64_t ldo, int64_t M, int N, void* stream);

/* out[n] = sum_m A[m,n]  (bias gradients), fixed-order two-level reduction */
size_t ercg_colsum_workspace_bytes(int64_t M, int N);
int ercg_colsum(const float* A, int64_t lda, int64_t M, int N, float* out,
                void* workspace, size_t workspace_bytes, void* stream);


/* ---------------------------------------------------------------------------------------------
 * K3  deterministic warp-segmented gather-reduce over the CSR (no atomics).
 *   out[k,:] = sum_{e in row k} w[e] * Y[col[e], etype[e]*H : +H]  (+ Y[k, root_off : +H]) (+ bias)
 * w == NULL -> 1, etype == NULL -> slot 0, root_off < 0 -> no root term, bias == NULL -> none.
 * Replaces MessagePassing.propagate + scatter_add of models/rgcn.py:188-221,15-46 (w = edge_norm),
 * PyG RGCNConv's per-relation mean (w = inv_cnt), and GraphConv's neighbour sum (dgcn_models.py:42,46).
 * Backward (by-source traversal):
 *   dY[j, r*H:+H] = sum_{e in out(j), type r} w[e] * dout[dst e]   for r in [0,R)   (all slots written)
 *   dY[j, root_off:+H] = dout[j]                                     (if root_off >= 0)
 *   dw[eid] = <dout[dst e], Y[src e, type e]>                        (if dw != NULL; needs Y)
 * rel_slot (optional, device int32 [R]): relation id -> column slot of Y / dY (K1's rel_info + 1), so that Y only holds
 * the P <= R relation ids that occur in the graph: Y is [N, P*H (+H root)], slot(e) = rel_slot[etype[e]]; ids with
 * rel_slot < 0 occur on no edge and are skipped by the backward.  NULL = identity (Y holds all R slots).
 * ------------------------------------------------------------------------------------------- */
int ercg_gather_fwd(const float* Y, int64_t ldy, const int32_t* rowptr, const int32_t* col,
                    const uint8_t* etype, const int32_t* rel_slot, const float* w, int root_off, const float* bias,
                    float* out, int64_t ldo, int64_t N, int H, void* stream);
int ercg_gather_bwd(const float* dout, int64_t ldo, const float* Y, int64_t ldy,
                    const int32_t* t_rowptr, const int32_t* t_col, const uint8_t* t_etype,
                    const int32_t* t_eid, const int32_t* rel_slot, const float* w, int R, int root_off,
                    float* dY, int64_t lddy, float* dw, int64_t N, int H, void* stream);
/* Backward on window graphs (every graph ercg_graphify_csr builds: the destinations of source j lie in [j - wlo, j + whi],
 * wlo = wp, whi = wf of batch_graphify; same limits as ercg_attn_window_supported): a CTA stages the dout rows around its 32
 * sources in shared memory.  n_slots = relation slots of dY (P with rel_slot, R without).  No dw (use ercg_gather_bwd when
 * the edge weights need a gradient).  Bit-identical to ercg_gather_bwd. */
int ercg_gather_window_bwd(const float* dout, int64_t ldo, const int32_t* t_rowptr, const int32_t* t_col,
                           const uint8_t* t_etype, const int32_t* t_eid, const int32_t* rel_slot, const float* w,
                           int n_slots, int root_off, float* dY, int64_t lddy, int64_t N, int H, int wlo, int whi,
                           void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4  fused edge attention of PyG TransformerConv(heads=1) (cogmen.py:66,72): score, segment
 * softmax over the in-edges of each destination (max-subtracted, denominator + 1e-16), weighted
 * aggregate of v, plus the skip row:  out[i] = sum_j alpha[j->i] v[j] + s[i].
 * alpha[E] (by-destination order) is saved for the backward.  q,k,v,s share one leading dimension.
 * H: any even value in [2, 1024] (odd, <= 0 or > 1024 -> ERCG_EINVAL).  Rows need 8-byte alignment: every pointer
 * 8-byte aligned and every leading dimension even (else ERCG_EALIGN).  16-byte aligned rows with H % 4 == 0 load
 * float4 chunks, others float2 chunks; both are bit-reproducible.  N == 0: no-op; N < 0: ERCG_EINVAL.
 * ------------------------------------------------------------------------------------------- */
int ercg_attn_fwd(const float* q, const float* k, const float* v, const float* s, int64_t ld,
                  const int32_t* rowptr, const int32_t* col, float scale,
                  float* out, int64_t ldo, float* alpha, float* dact, int64_t N, int H, void* stream);
/* dact (optional, [E]): the softmax runs over tanh(score) instead of the score -- nodal MatchingAttention 'general2' of the
 * declare-lab DialogueGCN (track_mm/dgcnv2_models.py:119-146, used over fully connected per-dialogue graphs, s = NULL,
 * scale = 1) -- and dact[e] = 1 - tanh^2 is saved for ercg_attn_bwd_dst, which folds it into dsig.  Same H range and
 * alignment as above, so the key half of dgcnv2's [xt | e] may start 8 bytes past a 16-byte boundary. */
/* by-destination half: dq[i], ds[i] = dout[i], dsig[e] = alpha_e (dalpha_e - sum alpha dalpha) [* dact_e] */
int ercg_attn_bwd_dst(const float* dout, int64_t ldo, const float* k, const float* v, int64_t ld,
                      const int32_t* rowptr, const int32_t* col, const float* alpha, float scale,
                      float* dq, float* ds, int64_t ldd, float* dsig, const float* dact, int64_t N, int H, void* stream);
/* by-source half: dk[j] = scale * sum_i dsig q[i], dv[j] = sum_i alpha dout[i] */
int ercg_attn_bwd_src(const float* dout, int64_t ldo, const float* q, int64_t ld,
                      const int32_t* t_rowptr, const int32_t* t_col, const int32_t* t_eid,
                      const float* alpha, const float* dsig, float scale,
                      float* dk, float* dv, int64_t ldd, int64_t N, int H, void* stream);

/* Window-graph variants of K4: same results, for graphs whose neighbourhoods are contiguous row ranges -- every graph
 * ercg_graphify_csr builds: the in-neighbours of node i lie in [i - wlo, i + whi] (wlo = wf, whi = wp of batch_graphify),
 * its out-neighbours in [i - wp, i + wf].  A CTA stages the rows around its 32 nodes in shared memory; a neighbour outside
 * the promised range traps.  Supported: H <= 128, H % 4 == 0, 0 <= wlo, whi, wlo + whi + 1 <= 32.
 * colsum_partial (optional, [ercg_attn_window_tiles(N)][2H]): per-CTA column sums of the two outputs (dq | ds, resp.
 * dk | dv), i.e. the bias gradients of the q/k/v/skip Linears (cogmen.py:66) once ercg_colsum has added the tiles up
 * (the partials are a [tiles, 2H] matrix, 1/16 of the gradient) -- the [N,4H] gradient is never re-read for them. */
int ercg_attn_window_supported(int H, int wlo, int whi);
int64_t ercg_attn_window_tiles(int64_t N);
int ercg_attn_window_fwd(const float* q, const float* k, const float* v, const float* s, int64_t ld,
                         const int32_t* rowptr, const int32_t* col, float scale, float* out, int64_t ldo, float* alpha,
                         int64_t N, int H, int wlo, int whi, void* stream);
int ercg_attn_window_bwd_dst(const float* dout, int64_t ldo, const float* k, const float* v, int64_t ld,
                             const int32_t* rowptr, const int32_t* col, const float* alpha, float scale, float* dq,
                             float* ds, int64_t ldd, float* dsig, float* colsum_partial, int64_t N, int H, int wlo,
                             int whi, void* stream);
int ercg_attn_window_bwd_src(const float* dout, int64_t ldo, const float* q, int64_t ld, const int32_t* t_rowptr,
                             const int32_t* t_col, const int32_t* t_eid, const float* alpha, const float* dsig,
                             float scale, float* dk, float* dv, int64_t ldd, float* colsum_partial, int64_t N, int H,
                             int wlo, int whi, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K5  EdgeAtt of DialogueGCN (dgcn_models.py:121-152): per-SOURCE window softmax
 *   nu[j->k] = softmax_{k in out(j)} <x_j, u_k>,  u = x @ W^T  (u computed by ercg_gemm_nn)
 * written in by-destination edge order (nu[t_eid]).  Backward: dsig per edge, dx_j += sum dsig u_k
 * (by source), du_k = sum_j dsig x_j (by destination).
 * H = g_dim: any even value in [2, 1024]; rows 8-byte aligned with even leading dimensions (same checks and return codes
 * as K4's ercg_attn_fwd).
 * ------------------------------------------------------------------------------------------- */
int ercg_edgeatt_fwd(const float* x, int64_t ldx, const float* u, int64_t ldu,
                     const int32_t* t_rowptr, const int32_t* t_col, const int32_t* t_eid,
                     float* nu, int64_t N, int H, void* stream);
int ercg_edgeatt_bwd_src(const float* dnu, const float* nu, const float* u, int64_t ldu,
                         const int32_t* t_rowptr, const int32_t* t_col, const int32_t* t_eid,
                         float* dsig, float* dx, int64_t lddx, int64_t N, int H, void* stream);
int ercg_edgeatt_bwd_dst(const float* dsig, const float* x, int64_t ldx,
                         const int32_t* rowptr, const int32_t* col,
                         float* du, int64_t lddu, int64_t N, int H, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K6  packed bidirectional LSTM recurrence, one layer (SeqContext, track_mm/dgcn_models.py:10-33;
 * MMGCN text LSTM, track_mm/mmgcn.py:69,114).  gx[N, 8*Hd] = x @ [W_ih; W_ih_reverse]^T + b_ih + b_hh is
 * produced by ercg_gemm_nn (gate order i,f,g,o per direction); whh = [2][4*Hd][Hd] (forward, reverse).
 * Dialogue d owns rows node_off[d]..node_off[d+1] (packed-sequence semantics, zero initial state).
 * fwd writes out[N,2*Hd] and saves gates[N,8*Hd] (post-activation), cells[N,2*Hd], hprev[N,2*Hd] (= h_{t-1}).
 * bwd writes dgx[N,8*Hd] (gradient w.r.t. the pre-activations); the caller forms
 *   dW_hh = dgx^T @ hprev, dW_ih = dgx^T @ x, db = colsum(dgx), dx = dgx @ [W_ih; W_ih_reverse] with K2.
 * Hd in {100 (the size the reference instantiates), 64, 48, 32, 24, 16, 8} runs K6 (lstm.cu: one CTA per direction and
 * dialogue slice, W_hh rows in registers); any Hd in 101..384 runs K6c (rnn_cluster.cu: W_hh spread over the shared memory
 * of a thread-block cluster of 8 CTAs, or a non-portable 16 when a slice does not fit at 8, with DSMEM exchange of h and of
 * the W_hh^T da partials).  Other sizes return ERCG_EINVAL; ERCG_ECUDA if the device cannot schedule the cluster shape.
 * ------------------------------------------------------------------------------------------- */
int ercg_lstm_fwd(const float* gx, int64_t ldgx, const float* whh, const int32_t* node_off, int B, int Hd,
                  float* out, int64_t ldo, float* gates, float* cells, float* hprev, void* stream);
int ercg_lstm_bwd(const float* dout, int64_t ldo, const float* gates, const float* cells, const float* whh,
                  const int32_t* node_off, int B, int Hd, float* dgx, int64_t lddgx, void* stream);
/* inverted dropout with a counter-hash mask (same (seed, index) -> same mask, so the backward re-applies it):
 * out[i] = hash(seed, i) < p ? 0 : x[i] / (1 - p).  nn.LSTM(dropout=.4) between layers, dgcn_models.py:17. */
int ercg_dropout(const float* x, float* out, int64_t n, float p, uint64_t seed, void* stream);
/* ercg_dropout with the mask drawn from seed + *seed_dev (seed_dev: device uint64, as ercg_gemm_nn's): the inter-layer
 * dropout of nn.LSTM (dgcn_models.py:17) inside a train step captured in a CUDA graph, which points seed_dev at its
 * device step counter so that every replay draws a fresh mask.  *seed_dev == 0 gives ercg_dropout(seed) bit for bit;
 * the backward calls it again with the same seed and word.  seed_dev NULL, n < 0 or p outside [0, 1): ERCG_EINVAL
 * before any launch. */
int ercg_dropout_dev(const float* x, float* out, int64_t n, float p, uint64_t seed, const uint64_t* seed_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K6b packed bidirectional GRU recurrence, one layer: the nn.GRU context encoders of DGCNModule("GRU")
 * (track_mm/dgcnv2.py, 2 layers run unpacked over the padded batch) and SeqContext(rnn_type="gru")
 * (track_mm/dgcn_models.py:46-47, 2 layers over the packed sequence).  torch.nn.GRU semantics, gate order r,z,n:
 *   r = sigmoid(gx_r + W_hr h + b_hr), z = sigmoid(gx_z + W_hz h + b_hz), n = tanh(gx_n + r (W_hn h + b_hn)),
 *   h' = (1 - z) n + z h.
 * gx[N, 6*Hd] = x @ [W_ih; W_ih_reverse]^T + b_ih (b_ih ONLY) is produced by ercg_gemm_nn; b_hh cannot be folded into it
 * (b_hn is multiplied by r) and is added inside the recurrence.  whh = [2][3*Hd][Hd], bhh = [2][3*Hd] (forward, reverse).
 * Dialogue d owns rows node_off[d]..node_off[d+1] (packed-sequence semantics, zero initial state).
 * fwd writes out[N,2*Hd] and saves gates[N,8*Hd] (per direction r, z, n, hn = W_hn h + b_hn) and hprev[N,2*Hd] (= h_{t-1}).
 * bwd writes dgx[N,6*Hd] = (da_r, da_z, da_n), the gradient w.r.t. gx, and dgh[N,6*Hd] = (da_r, da_z, r da_n), the
 * gradient w.r.t. W_hh h + b_hh; the caller forms dW_hh = dgh^T @ hprev, db_hh = colsum(dgh), dW_ih = dgx^T @ x,
 * db_ih = colsum(dgx), dx = dgx @ [W_ih; W_ih_reverse] with K2.
 * Hd in {100 (the size the reference instantiates), 64, 48, 32, 24, 16, 8} runs K6b (gru.cu); any Hd in 101..384 runs K6c
 * (rnn_cluster.cu, thread-block clusters of 8 or 16 CTAs, as for the LSTM).  Other values return ERCG_EINVAL; ERCG_ECUDA if
 * the device cannot schedule the cluster shape.
 * ------------------------------------------------------------------------------------------- */
int ercg_gru_fwd(const float* gx, int64_t ldgx, const float* whh, const float* bhh, const int32_t* node_off, int B, int Hd,
                 float* out, int64_t ldo, float* gates, float* hprev, void* stream);
int ercg_gru_bwd(const float* dout, int64_t ldo, const float* gates, const float* hprev, const float* whh,
                 const int32_t* node_off, int B, int Hd, float* dgx, int64_t lddgx, float* dgh, int64_t lddgh, void* stream);

/* ---------------------------------------------------------------------------------------------
 * BatchNorm1d (training statistics) + LeakyReLU of GNN.forward (cogmen.py:67-68,72).
 * stats: mean[H], var[H] (biased) over the N rows, fixed-order reduction.
 * ------------------------------------------------------------------------------------------- */
size_t ercg_bn_workspace_bytes(int64_t N, int H);
int ercg_bn_stats(const float* x, int64_t ldx, int64_t N, int H, float* mean, float* var,
                  void* workspace, size_t workspace_bytes, void* stream);
/* running statistics of nn.BatchNorm1d in train mode (cogmen.py:67; torch semantics): num_batches_tracked += 1;
 * m = momentum, or 1 / num_batches_tracked when momentum < 0 (momentum=None);
 * running_mean = (1 - m) running_mean + m mean;  running_var = (1 - m) running_var + m var count / max(count - 1, 1).
 * ONE launch instead of five elementwise ones; count = rows behind the statistics (all ranks).  H <= 1024. */
int ercg_bn_running_update(const float* mean, const float* var, float* running_mean, float* running_var,
                           int64_t* num_batches_tracked, float momentum, float count, int H, void* stream);
/* data-parallel BatchNorm statistics (global-batch mode): pack local (mean, biased var, n) into the fp64 all-reduce buffer
 * buf[2H+2] = (mean n | (var + mean^2) n | n | 0), and unpack the summed buffer into the global (mean, biased var) -- two
 * launches around the collective instead of a dozen elementwise ones.  Same arithmetic, in fp64, as the reference-style
 * torch expression it replaces (emotion-recognition-in-conversation_b200/dist.py). */
int ercg_bn_sync_pack(const float* mean, const float* var, double n_local, int H, double* buf, void* stream);
int ercg_bn_sync_unpack(const double* buf, int H, float* mean, float* var, void* stream);
int ercg_bn_act_fwd(const float* x, int64_t ldx, const float* mean, const float* var, float eps,
                    const float* gamma, const float* beta, float slope,
                    float* out, int64_t ldo, int64_t N, int H, void* stream);
/* backward with batch statistics (train) or with fixed statistics (eval, use_batch_stats = 0).
 * dgamma[H], dbeta[H], dx[N,H].  count = number of rows the statistics were taken over (N, or the
 * global count when the statistics were all-reduced across ranks; sums[2H] then holds the
 * all-reduced (sum dy, sum dy*xhat) produced by ercg_bn_act_bwd_reduce). */
int ercg_bn_act_bwd_reduce(const float* dout, int64_t ldo, const float* x, int64_t ldx,
                           const float* mean, const float* var, float eps,
                           const float* gamma, const float* beta, float slope,
                           float* sums /* [2H]: sum dy, sum dy*xhat */, int64_t N, int H,
                           void* workspace, size_t workspace_bytes, void* stream);
int ercg_bn_act_bwd_apply(const float* dout, int64_t ldo, const float* x, int64_t ldx,
                          const float* mean, const float* var, float eps,
                          const float* gamma, const float* beta, float slope,
                          const float* sums, double count, int use_batch_stats,
                          float* dx, int64_t lddx, int64_t N, int H, void* stream);

/* ---------------------------------------------------------------------------------------------
 * (class-weighted) cross entropy, mean reduction (F.cross_entropy at cogmen.py:185, dgcn.py:124).
 * fwd writes lossnum_den[0] = sum_i w[y_i] * nll_i, lossnum_den[1] = sum_i w[y_i] and the
 * un-normalised dlogits[i,c] = w[y_i] (softmax_ic - [c == y_i]).  The caller divides (possibly after an
 * all-reduce of lossnum_den across ranks); ercg_scale_by_ratio applies  x *= g[0] / den[0].
 * ------------------------------------------------------------------------------------------- */
size_t ercg_ce_workspace_bytes(int64_t N);
int ercg_ce_fwd(const float* logits, int64_t ld, const int64_t* labels, const float* class_weight,
                float* lossnum_den, float* dlogits, int64_t ldd, int64_t N, int C,
                void* workspace, size_t workspace_bytes, void* stream);
int ercg_scale_by_ratio(float* x, int64_t n, const float* num, const float* den, void* stream);

/* Backward of the classifier tail  Linear(K,K) -> ReLU -> Dropout -> Linear(K,C)  (cogmen.py:116-122) in one pass over the
 * hidden activations h [N,K] (post ReLU / dropout): dZ = (h > 0 ? scale : 0) * (dlogits @ W3)  (gradient of the first
 * Linear's pre-activation; scale = 1/(1-p) with dropout, 1 without), dW3 [C,K] = dlogits^T @ h, db3 [C] = column sums of
 * dlogits, db0 [K] = column sums of dZ.  dlogits is [N,C] contiguous, W3 the nn.Linear weight [C,K].  K % 4 == 0,
 * K <= 128, C <= 8.  Replaces five launches (ercg_gemm_tn, ercg_gemm_nn, ercg_mask_pos, 2 x ercg_colsum). */
size_t ercg_cls_tail_bwd_workspace_bytes(int K, int C);
int ercg_cls_tail_bwd(const float* h, int64_t ldh, const float* dlogits, const float* W3, float scale,
                      float* dZ, int64_t ldz, float* dW3, float* db3, float* db0, int64_t N, int K, int C,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K7  MMGCN cross-modal utterance graph as a block adjacency (MMGCN.create_big_adj,
 * track_mm/mmgcn_models.py:582-646).  M modalities, N utterances, node (m,i) = row m*N + i
 * (modality-major then dialogue-major, :616).  Non-zeros of the reference's dense [M*N, M*N] matrix:
 *   blocks: flat[m*SB + blk_off[d] + i*L + j]            L x L similarity block of dialogue d, modality m
 *   cross : flat[M*SB + (m*(M-1) + (n<m ? n : n-1))*N + node]   entry ((m,node),(n,node)), m != n
 * with SB = sum_d L_d^2 (ercg_mmgcn_block_offsets writes the prefix blk_off[B+1]); the flat array has
 * M*SB + M*(M-1)*N floats.
 *   adj_fwd: xhat = x/|x| (:606-607), cs = 0.99999 <xhat_i,xhat_j> (:608-609), A = 1 - acos(cs)/pi (:610),
 *            dinv = rowsum(A)^-1/2, ahat = (dinv_i A_ij) dinv_j  (D.mm(adj).mm(D), :638-644)
 *   adj_bwd: gradient G w.r.t. ahat (same flat layout) -> dx (create_big_adj is differentiable in the features)
 * D, H <= 256, multiples of 4; all feature rows 16-byte aligned.
 * ------------------------------------------------------------------------------------------- */
int ercg_mmgcn_block_offsets(const int32_t* node_off, int B, int64_t* blk_off, void* stream);
int ercg_mmgcn_adj_fwd(const float* x, int64_t ldx, const int32_t* node_off, const int32_t* node_dlg,
                       const int64_t* blk_off, int64_t N, int64_t SB, int M, int D, float* xhat, int64_t ldh,
                       float* rinv /*[M*N]*/, float* cs /*flat*/, float* ahat /*flat*/, float* dinv /*[M*N]*/, void* stream);
int ercg_mmgcn_adj_bwd(const float* G, const float* cs, const float* dinv, const float* xhat, int64_t ldh,
                       const float* rinv, const int32_t* node_off, const int32_t* node_dlg, const int64_t* blk_off,
                       int64_t N, int64_t SB, int M, int D, float* ddeg /*[M*N] scratch*/, float* dx, int64_t ldx,
                       void* stream);
/* out = Ahat @ h over the block pattern (torch.spmm(adj, input), mmgcn_models.py:29); transpose != 0 uses Ahat^T
 * (input gradient).  Optional side job for the backward: acc_dst[row,:] += acc_src[row,:]. */
int ercg_mmgcn_spmm(const float* ahat, int transpose, const float* h, int64_t ldh, float* out, int64_t ldo,
                    const int32_t* node_off, const int32_t* node_dlg, const int64_t* blk_off, int64_t N, int64_t SB,
                    int M, int H, const float* acc_src, int64_t lds, float* acc_dst, int64_t ldd, void* stream);
/* G[(i,j)] (+)= <dhi_i, h_j> on the block pattern: gradient w.r.t. ahat of out = Ahat @ h */
int ercg_mmgcn_sddmm(const float* dhi, int64_t ldd, const float* h, int64_t ldh, const int32_t* node_off,
                     const int32_t* node_dlg, const int64_t* blk_off, int64_t N, int64_t SB, int M, int H, float* G,
                     int accumulate, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K8  GCNII layer (GraphConvolution.forward, variant=True, residual=False; mmgcn_models.py:27-39) with the ReLU and
 * the next layer's input dropout of GCNII_lyc.forward (:388-392) as the epilogue:
 *   out = dropout(relu(theta * [hi | h0] @ W + (1-theta) * ((1-alpha) * hi + alpha * h0))),  W [2H, H]
 * (relu == 0: the bare GraphConvolution output, drop_p == 0: no dropout).  [hi | h0] is read from its two sources, never concatenated.  Backward w.r.t. the inputs:
 *   dS[M, 2H] = theta * dZ @ Wt + [(1-theta)(1-alpha) dZ | (1-theta) alpha dZ],  Wt = W^T [H, 2H], dZ = relu/dropout-masked dout
 * (weight gradient = theta * [hi | h0]^T dZ through ercg_gemm_tn).  H % 8 == 0.
 * ------------------------------------------------------------------------------------------- */
int ercg_gcnii_layer_fwd(const float* hi, int64_t ldhi, const float* h0, int64_t ldh0, const float* W, int64_t ldw,
                         float* out, int64_t ldo, int64_t M, int H, float theta, float alpha, int relu, float drop_p,
                         uint64_t seed, void* stream);
/* ercg_gcnii_layer_fwd with the dropout mask drawn from seed + *seed_dev (seed_dev: device uint64, as ercg_gemm_nn's): the
 * GCNII stack inside a train step captured in a CUDA graph, which points seed_dev at its device step counter so that every
 * replay draws a fresh mask.  *seed_dev == 0 gives ercg_gcnii_layer_fwd(seed) bit for bit.  seed_dev NULL and every
 * argument ercg_gcnii_layer_fwd rejects: the same error code before any launch. */
int ercg_gcnii_layer_fwd_dev(const float* hi, int64_t ldhi, const float* h0, int64_t ldh0, const float* W, int64_t ldw,
                             float* out, int64_t ldo, int64_t M, int H, float theta, float alpha, int relu, float drop_p,
                             uint64_t seed, const uint64_t* seed_dev, void* stream);
int ercg_gcnii_layer_bwd_input(const float* dZ, int64_t lddz, const float* Wt, int64_t ldwt, float* dS, int64_t ldds,
                               int64_t M, int H, float theta, float alpha, void* stream);

/* helpers of the MMGCN path */
/* rows[i] = row of packed node i in a padded tensor: seq-first [Lmax,B,*] -> k*B + d, batch-first -> d*Lmax + k
 * (simple_batch_graphify, track_mm/mmgcn_utils.py:5-21, fused into the consumer GEMM as its row gather) */
int ercg_node_rows(const int32_t* node_off, const int32_t* node_dlg, int64_t N, int B, int Lmax, int seq_first,
                   int32_t* rows, void* stream);
/* out[i,:] = x[i,:] + emb[argmax(qmask[rows[i], :]), :]; ids[i] = that argmax, onehot[N, n_speakers] for the
 * embedding gradient (onehot^T @ dout through ercg_gemm_tn).  MMGCN.forward, mmgcn_models.py:540-545. */
int ercg_speaker_embed_add(const float* x, int64_t ldx, const float* qmask, int n_speakers, const int32_t* rows,
                           const float* emb, int64_t lde, float* out, int64_t ldo, int32_t* ids, float* onehot, int64_t N,
                           int D, void* stream);
/* out = dropout(relu(x)) with the counter-hash mask (relu(dropout(x)) of mmgcn.py:117-118 is the same function) */
int ercg_relu_dropout(const float* x, float* out, int64_t n, float p, uint64_t seed, void* stream);
/* ercg_relu_dropout with the mask drawn from seed + *seed_dev (as ercg_dropout_dev): *seed_dev == 0 gives
 * ercg_relu_dropout(seed) bit for bit.  seed_dev NULL, n < 0 or p outside [0, 1): ERCG_EINVAL before any launch. */
int ercg_relu_dropout_dev(const float* x, float* out, int64_t n, float p, uint64_t seed, const uint64_t* seed_dev,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimizer tail of the train steps (SURVEY.md 8f-3) on ONE flat fp32 buffer of all live parameters and its gradient twin:
 *   torch.optim.Adam(lr, weight_decay) .step()           track_mm/cogmen.py:50,187-189, dgcn.py:41,127-129, mmgcn.py:34
 *   torch.optim.AdamW + clip_grad_norm_(params, 5)        track_mm/dagerc.py:39,229-231
 * ercg_sumsq: out[0] = sum x^2 (fixed-order fp64 partials; the squared global gradient norm).
 * ercg_adam_step: one launch updates p, m, v in place from g.  decoupled = 0: Adam (g += wd * p), 1: AdamW (p *= 1 - lr*wd).
 *   grad_scale multiplies every gradient (1/world_size after a summed all-reduce of per-rank MEAN losses; 1 otherwise).
 *   sumsq (optional, device): clip_grad_norm_ -- gradients are scaled by min(1, max_norm / (sqrt(*sumsq) * grad_scale + 1e-6)).
 *   step_dev: device int64 step counter; the update uses step + 1 for the bias corrections and a second tiny launch
 *   increments it, so a captured CUDA graph advances the optimizer state on every replay without host arithmetic.
 * ------------------------------------------------------------------------------------------- */
size_t ercg_sumsq_workspace_bytes(int64_t n);
int ercg_sumsq(const float* x, int64_t n, float* out, void* workspace, size_t workspace_bytes, void* stream);
int ercg_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                   float eps, float weight_decay, int decoupled, float grad_scale, const float* sumsq,
                   float max_norm, int64_t* step_dev, void* stream);
/* ercg_adam_step_guarded: ercg_adam_step (same arguments, same arithmetic bit for bit) that first reads the DEVICE int
 * *skip_if_nonzero: when it is not 0, both launches return before touching p, m, v or *step_dev.  The data-parallel trainer
 * passes the sticky status word of its peer-memory communicator (ercg_p2p_status_word), so the gradient of a timed-out
 * exchange is never applied -- DDP's all-reduce under accelerate (lumo/trainer/trainer.py:315-327) followed by
 * optimizer.step() (track_mm/cogmen.py:187-189, dgcn.py:127-129, mmgcn.py:141-157, dagerc.py:229-231) raises instead of
 * stepping on a failed collective.  skip_if_nonzero = NULL: ERCG_EINVAL. */
int ercg_adam_step_guarded(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                           float eps, float weight_decay, int decoupled, float grad_scale, const float* sumsq,
                           float max_norm, int64_t* step_dev, void* stream, const int* skip_if_nonzero);

/* ---------------------------------------------------------------------------------------------
 * Peer-memory all-reduce over NVLink / NVSwitch for the exchanges of the dialogue-sharded train step: BatchNorm statistics,
 * their backward sums, the flat gradient buffer.  Replaces the bucketed NCCL all-reduce the reference reaches through
 * accelerate / DDP (lumo/trainer/trainer.py:62-64,315-327, track_mm/cogmen.py:188) on ONE node.  One-shot: every rank stages
 * its vector in a region that all peers have opened through CUDA IPC, raises a flag in every peer's region, waits for the
 * peers' flags and adds the W staged vectors in rank order (bit-identical on all ranks, run to run).  See csrc/p2p.cu.
 *
 * Setup (the only entry points of this library that allocate or synchronise; call them once per communicator):
 *   ercg_p2p_region_bytes(max_bytes): size of a region for payloads up to max_bytes per call;
 *   ercg_p2p_alloc: cudaMalloc + zero a region on the current device, return it and its 64-byte IPC handle;
 *   ercg_p2p_open / ercg_p2p_close: map / unmap a PEER's region from its handle (exchange the handles over any host channel);
 *   ercg_p2p_free; ercg_p2p_status: copies the region's sticky status word to the host (0 or ERCG_P2P_ETIMEOUT).
 * ercg_p2p_allreduce: out[i] = sum over ranks of in[i] (in == out allowed), n elements of fp32 (dtype 0) or fp64 (dtype 1);
 *   regions_dev = DEVICE array of the W region base pointers as mapped in this process (own region at index rank).
 *   Every rank must issue the same sequence of calls (same n) on a communicator, all on one stream (or otherwise
 *   serialised); concurrent streams need one communicator each.  Plain kernel launch: capturable in a CUDA graph.
 *   Every wait for a peer is bounded (30 s; the environment variable ERCG_P2P_TIMEOUT_MS, read once per process, overrides
 *   it): a peer that never arrives makes the kernel return with the region's status word set to ERCG_P2P_ETIMEOUT.
 * ------------------------------------------------------------------------------------------- */
/* ercg_p2p_bn_stats: the data-parallel BatchNorm statistics of GNN.forward (cogmen.py:67,72 under DDP with the statistics
 *   taken over the GLOBAL batch) fused with their exchange: column reduction of this rank's rows, exchange over peer memory,
 *   global mean / biased variance (the same on every rank) and, when running_mean / running_var are given, the train-mode
 *   running statistics (as ercg_bn_running_update) -- two launches in all.  count_global = rows over all ranks.  Equals
 *   ercg_bn_stats + ercg_bn_sync_pack + all-reduce + ercg_bn_sync_unpack + ercg_bn_running_update bit for bit.
 *   workspace as for ercg_bn_stats; H <= 1024. */
#define ERCG_P2P_HANDLE_BYTES 64
size_t ercg_p2p_region_bytes(size_t max_bytes);
int ercg_p2p_alloc(size_t region_bytes, void** region, unsigned char* ipc_handle);
int ercg_p2p_open(const unsigned char* ipc_handle, void** region);
int ercg_p2p_close(void* peer_region);
int ercg_p2p_free(void* region);
int ercg_p2p_status(const void* region, int* status_host);
/* ercg_p2p_status_word: *status_dev = DEVICE address of the region's sticky status word (the value ercg_p2p_status copies),
 * for ercg_adam_step_guarded.  Host only, no synchronisation. */
int ercg_p2p_status_word(void* region, int** status_dev);
int ercg_p2p_allreduce(void* const* regions_dev, int rank, int world, const void* in, void* out, int64_t n, int dtype,
                       size_t max_bytes, void* stream);
/* ercg_p2p_bn_act_bwd_reduce: ercg_bn_act_bwd_reduce fused with the exchange of its result: sums[2H] = this rank's
 * (sum dy, sum dy*xhat) (its dbeta / dgamma), sums_global[2H] = the rank-ordered total over all ranks (what
 * ercg_bn_act_bwd_apply needs when the statistics were global).  H <= 512. */
int ercg_p2p_bn_act_bwd_reduce(void* const* regions_dev, int rank, int world, const float* dout, int64_t ldo,
                               const float* x, int64_t ldx, const float* mean, const float* var, float eps,
                               const float* gamma, const float* beta, float slope, float* sums, float* sums_global,
                               int64_t N, int H, void* workspace, size_t workspace_bytes, size_t max_bytes, void* stream);
int ercg_p2p_bn_stats(void* const* regions_dev, int rank, int world, const float* x, int64_t ldx, int64_t N, int H,
                      double count_global, float* mean, float* var, float* running_mean, float* running_var,
                      int64_t* num_batches_tracked, float momentum, void* workspace, size_t workspace_bytes,
                      size_t max_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K11  MaskedEdgeAttention 'attn1' of the declare-lab DialogueGCN (track_mm/dgcnv2_models.py:517-562) -- the edge weights of
 * dgcnv2's batch_graphify (:638-690) -- in closed form on the packed graph.  S [B*Lmax, >= max_seq_len] (row b*Lmax + j',
 * column i) = M @ scalar.weight^T from ercg_gemm_nn, M = the dialogue-major, full-length context rows.  Per source (b, i):
 *   nu[i -> j] = e_j / (Z_win + 1e-10 (Z_all - Z_win)),  e_j' = exp(S[j', i] - max_j' S[., i]) over ALL Lmax positions,
 *   Z_win over the targets j of i's window [max(0, i-wp), min(len-1, i+wf)] (wp / wf = -1: unbounded);
 * nu is written in by-destination edge order (through t_rowptr / t_eid of ercg_graphify_csr); stat [N,2] keeps (max, Den).
 * Backward: dS (zero-initialised by the caller, same layout as S) from dnu.
 * ERCG_EINVAL before any launch for Lmax < 1, ldS < Lmax or (backward) ldd < Lmax. */
int ercg_masked_edge_att_fwd(const float* S, int64_t ldS, const int32_t* node_off, const int32_t* node_dlg,
                             const int32_t* t_rowptr, const int32_t* t_eid, int64_t Lmax, int wp, int wf,
                             float* nu, float* stat, int64_t N, void* stream);
int ercg_masked_edge_att_bwd(const float* S, int64_t ldS, const int32_t* node_off, const int32_t* node_dlg,
                             const int32_t* t_rowptr, const int32_t* t_eid, int64_t Lmax, int wp, int wf,
                             const float* nu, const float* dnu, const float* stat, float* dS, int64_t ldd,
                             int64_t N, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K9  DAG-ERC predecessor structure (DAGERCModule.get_adj_v1 / get_s_mask, track_mm/dagerc.py:109-154) on packed
 * dialogues: the direct predecessors of utterance i are the contiguous local range [lo_i, i-1], lo_i = the
 * windowp-th latest j < i with spk_j == spk_i (0 if there are fewer); s_mask[i,j] = (spk_i == spk_j).
 *   lo[N], cnt[N] = i - lo_i, eoff[N] = exclusive scan of cnt (where node i's attention weights are stored),
 *   total[1] = sum cnt (device).  ercg_dag_dense_masks emits the reference's dense layout from PADDED speaker ids:
 *   adj [B,Lmax,Lmax] fp32, s_mask [B,Lmax,Lmax] int64 (computed over all Lmax positions, like the reference).
 * ------------------------------------------------------------------------------------------- */
size_t ercg_dag_build_workspace_bytes(int64_t N);
int ercg_dag_build(const int32_t* node_off, const int32_t* node_dlg, const int32_t* spk, int64_t N, int windowp,
                   int32_t* lo, int32_t* cnt, int64_t* eoff, int64_t* total, void* workspace, size_t workspace_bytes,
                   void* stream);
int ercg_dag_dense_masks(const int32_t* spk_padded, int B, int Lmax, int windowp, float* adj, int64_t* s_mask,
                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * K10  one DAG-ERC GNN layer over all dialogues (the i-loop of DAGERCModule.forward, dagerc.py:167-185, with
 * GAT_dialoggcn_v1.forward, dagerc_models.py:326-365, and the two nn.GRUCell of :89-90) as ONE persistent
 * cooperative kernel; backward = the same in reverse time.  D = hidden size (300 in the reference), D % 4 == 0.
 *   pre[N,6D] = Hin @ [W_ih^c ; W_hh^p]^T + [b_ih^c ; b_hh^p]   (hoisted, by ercg_gemm_nn)
 *   per step i: alpha = softmax_{j in [lo_i, i-1]} (wk . H1_j)      (the w_q.Q + b part of linear() is constant in j)
 *               S0/S1 = alpha-weighted sums of H1_j over same-/other-speaker j;  M = Wr0 S0 + Wr1 S1
 *               C = GRUCell_c(H_i, M), P = GRUCell_p(M, H_i), H1_i = C + P
 * order[B] = dialogues by decreasing length; Tmax = the longest.  Saved for the backward: a[N], S[N,2D], M[N,D],
 * alpha[total], gc[N,3D] (r,z,n of cell c), hnc[N,D] (W_hn^c M + b_hn^c), gp[N,3D].
 * Backward: dH1 [N,D] holds the incoming gradient and is used as the accumulator; outputs dpre[N,6D] (w.r.t. pre),
 * dGseq[N,6D] (w.r.t. [W_hh^c M + b ; W_ih^p M + b]), dM[N,D], dHdir[N,D] (direct z'*dP term of H_i), ga[N] (zero-
 * initialised; sum of the attention-logit gradients per utterance), dS[N,2D] scratch.  Weight gradients are TN GEMMs
 * of these against Hin / M / S / H1.
 * ------------------------------------------------------------------------------------------- */
typedef struct ercg_dag_layer {
  int32_t B, D, Tmax, reserved;
  const int32_t* node_off; const int32_t* order; const int32_t* spk; const int32_t* lo; const int64_t* eoff;
  const float* wk;      /* [D]     gather.linear.weight[0, D:2D] */
  const float* Wr0;     /* [D,D]   row-major (out, in) like nn.Linear.weight */
  const float* Wr1;
  const float* Whh_c;   /* [3D,D]  grus_c.weight_hh */
  const float* bhh_c;   /* [3D] */
  const float* Wih_p;   /* [3D,D]  grus_p.weight_ih */
  const float* bih_p;
  const float* Hin;     /* [N,D]   H[l] */
  const float* pre;     /* [N,6D] */
  float *H1, *a, *S, *M, *alpha, *gc, *hnc, *gp;
  float *dH1, *dpre, *dGseq, *dM, *dS, *dHdir, *ga;   /* backward only */
} ercg_dag_layer;
int ercg_dag_layer_fwd(const ercg_dag_layer* args, void* stream);
int ercg_dag_layer_bwd(const ercg_dag_layer* args, void* stream);

/* Stand-alone attention step = GAT_dialoggcn_v1.forward(Q, K, V, adj, s_mask) (track_mm/dagerc_models.py:326-365, mask_logic
 * :83-90) for B queries against N context rows each (the fused layer kernel above never materialises it):
 *   e[b,n] = w_linear[:D].Q[b] + w_linear[D:].K[b,n] + b_linear - (1 - adj[b,n]) * 1e30;  alpha[b,:] = softmax_n e[b,:]
 *   S01[b] = [ sum_n alpha*s*V[b,n] | sum_n alpha*(1-s)*V[b,n] ]   ([B, 2D]; attn_sum = S01 @ [Wr0 | Wr1]^T is a dense
 *   transform done by the caller with ercg_gemm_nn).  Q [B,D] (ldq), K / V [B,N,D] with batch / row strides in elements,
 *   adj / s_mask [B,N] fp32 (row stride ldm), alpha [B,N] and S01 [B,2D] contiguous.
 * Backward: dalpha (may be NULL) and dS01 in; de [B,N] = gradient of the pre-softmax logits (dw_k = sum de*K, dw_q = sum_b
 * (sum_n de) Q, db = sum de: the caller's transposed products), dQ [B,D], dK / dV [B,N,D] contiguous. */
int ercg_dag_gat_fwd(const float* Q, int64_t ldq, const float* K, int64_t ldk_b, int64_t ldk_n, const float* V,
                     int64_t ldv_b, int64_t ldv_n, const float* adj, const float* s_mask, int64_t ldm,
                     const float* w_linear, const float* b_linear, float* alpha, float* S01, int B, int N, int D,
                     void* stream);
int ercg_dag_gat_bwd(const float* V, int64_t ldv_b, int64_t ldv_n, const float* s_mask, int64_t ldm,
                     const float* w_linear, const float* alpha, const float* dalpha, const float* dS01, float* de,
                     float* dQ, float* dK, float* dV, int B, int N, int D, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K12  DialogueRNN recurrence (DialogueRNN / DialogueRNNCell of the declare-lab DialogueRNN, track_mm/dgcnv2_models.py:235-348,
 * listener_state=False, context_attention 'simple' or 'general') over B dialogues of L steps each (seq-first rows r = t*B + b;
 * every dialogue runs all L steps).  Per step, with s = argmax_p qmask[r] (first on ties) and m = qmask[r, s]:
 *   g_t = drop_g(GRUCell_g([U_t ; q_{t-1}[s]], g_{t-1}))
 *   c_t = sum_{j<t} alpha_j g_j, alpha = softmax_j(xq_r . g_j)  (c_0 = 0; xq_r = W_a U_t for 'general', the weight w of
 *         'simple' for every row)
 *   q_t[s] = q_{t-1}[s] (1 - m) + m drop_q(GRUCell_p([U_t ; c_t], q_{t-1}[s])),  q_t[p] = q_{t-1}[p] for p != s
 *   e_t = drop_e(GRUCell_e(q_t[s], e_{t-1}))
 * nn.GRUCell semantics (gate order r, z, n), zero initial states.  The reference runs the party cell for every party and
 * blends with qmask; running it for the speaker only is exact when each qmask row has at most one non-zero entry.
 * The U-dependent input-gate terms are hoisted: pre[L*B, >= 3Dg+3Dp] = U @ [W_ih^g[:, :Dm] ; W_ih^p[:, :Dm]]^T + [b_ih^g ;
 * b_ih^p] (ercg_gemm_nn), columns [0, 3Dg) for the g cell and [3Dg, 3Dg+3Dp) for the party cell.  Dropout (drop_p in
 * [0, 1)): element (r, u) of cell x in {g, q, e} is kept iff hash_uniform(seed_x, r*D_x + u) >= drop_p and then scaled by
 * 1 / (1 - drop_p) -- ercg_dropout's mask on a contiguous [L*B, D_x] tensor.
 * Dg, Dp, De in 1..256, P in 1..16; negative sizes, other widths or P, or drop_p outside [0, 1): ERCG_EINVAL before any
 * launch.  B == 0 or L == 0: no-op.  One persistent cooperative kernel per direction (weights sliced by hidden unit over
 * the CTAs' shared memory, all dialogues in lockstep, grid.sync between phases); ERCG_ECUDA if the device cannot
 * co-schedule the grid.  Fixed-order fp32 arithmetic, no atomics: results are bit-reproducible.
 * fwd writes e[L*B,De] and saves g[L*B,Dg] (after dropout), c[L*B,Dg], qprev / qcur[L*B,Dp] (q_{t-1}[s], q_t[s]),
 * gates_{g,p,e}[L*B, 4D] (r, z, n, W_hn h + b_hn) and alpha (step t >= 1 is the [B, t] block at offset B*t*(t-1)/2);
 * qstate[B*P*Dp] is workspace.
 * bwd reads de[L*B,De] and writes dpre (gradient w.r.t. the pre columns, row stride lddpre), dxq[L*B,Dg] (w.r.t. xq_r, row
 * stride lddxq;
 * 'simple': dw = column sums), dgh[L*B,3Dg], dph[L*B,3Dp], deh[L*B,3De] (w.r.t. W_hh h + b_hh of each cell: dW_hh = dgh^T @
 * h_{t-1}, db_hh = colsum) and dei[L*B,3De] (w.r.t. W_ih^e q_t[s] + b_ih^e).  dG[L*B,Dg], dQ[B*P*Dp], dEh[B*De] and
 * dc[B*Dg] are workspace.
 * ------------------------------------------------------------------------------------------- */
typedef struct ercg_dialogue_rnn {
  int32_t L, B, Dg, Dp, De, P;
  float drop_p;
  int32_t reserved;
  uint64_t seed_g, seed_q, seed_e;
  const float* qmask;                         /* [L*B, P] */
  const float* pre; int64_t ldpre;
  const float* xq; int64_t ldxq;              /* [L*B, Dg] rows, or one row with ldxq = 0 */
  const float *Wgq, *Whh_g, *bhh_g;           /* g_cell.weight_ih[:, Dm:] [3Dg,Dp], weight_hh [3Dg,Dg], bias_hh [3Dg] */
  const float *Wpc, *Whh_p, *bhh_p;           /* p_cell.weight_ih[:, Dm:] [3Dp,Dg], weight_hh [3Dp,Dp], bias_hh [3Dp] */
  const float *Wih_e, *Whh_e, *bih_e, *bhh_e; /* e_cell [3De,Dp], [3De,De], [3De], [3De] */
  float *e, *g, *c, *qprev, *qcur, *gates_g, *gates_p, *gates_e, *alpha, *qstate;
  const float* de;                            /* backward only from here on */
  float* dpre; int64_t lddpre;
  float* dxq; int64_t lddxq;
  float *dgh, *dph, *dei, *deh, *dG, *dQ, *dEh, *dc;
} ercg_dialogue_rnn;
int ercg_dialogue_rnn_fwd(const ercg_dialogue_rnn* args, void* stream);
int ercg_dialogue_rnn_bwd(const ercg_dialogue_rnn* args, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K13  dense masked MatchingAttention of the declare-lab sequence classifiers (MatchingAttention.forward(M, x, mask) and the
 * att2 loop of LSTMModel / GRUModel / DialogRNNModel, track_mm/dgcnv2_models.py).  B dialogues of L memory rows M (seq-first:
 * row j*B + b, row stride ldm); Q queries per dialogue, query q of dialogue b = row r = q*B + b of xq (= transform(x), ldq).
 *   kind ERCG_MATCH_GENERAL : alpha_j = softmax_j <xq_r, M_j>   (mask ignored)
 *   kind ERCG_MATCH_GENERAL2: s_j = m_j <xq_r, m_j M_j>, p = softmax_j tanh(s_j) over all L, alpha_j = p_j m_j / sum_k p_k m_k
 *        (m = mask[b*L + j], [B, L] contiguous; NULL = all ones; a row whose mask is all zero gives NaN, as the reference)
 *   pool_r = sum_j alpha_j M_j
 * fwd writes pool [Q*B, D] (row stride ldp), alpha [Q, B, L] and score [Q, B, L] (s_j, kept for the backward).
 * bwd reads dpool (row stride lddp) and writes dxq [Q*B, D] and dM [L*B, D] (both overwritten); w [Q, B, L] is workspace.
 * D in 1..1024 (any row alignment), L and Q in 1..4096, ld* >= D, B >= 0; other sizes or kinds: ERCG_EINVAL before any
 * launch; B*Q or B*L above 2^31 - 1: ERCG_ERANGE.  B == 0: no-op.  Fixed-order fp32, no atomics: bit-reproducible.
 * ------------------------------------------------------------------------------------------- */
#define ERCG_MATCH_GENERAL 0
#define ERCG_MATCH_GENERAL2 1
int ercg_match_att_fwd(const float* M, int64_t ldm, int L, int B, int D, int Q, const float* xq, int64_t ldq,
                       const float* mask, int kind, float* pool, int64_t ldp, float* alpha, float* score, void* stream);
int ercg_match_att_bwd(const float* M, int64_t ldm, int L, int B, int D, int Q, const float* xq, int64_t ldq,
                       const float* mask, int kind, const float* alpha, const float* score, const float* dpool,
                       int64_t lddp, float* w, float* dxq, int64_t lddxq, float* dM, int64_t lddm, void* stream);
/* DialogRNNModel._reverse_seq (pad_sequence of flip(x[:c_b]) per dialogue): x [Lin*B, D] seq-first (row stride ldx) ->
 * out [Lout*B, D] (row stride ldo), out[t*B + b] = x[(c_b - 1 - t)*B + b] for t < c_b and 0 for c_b <= t < Lout, with
 * c_b = counts[b] (device int32) clamped to [0, Lin].  Its backward is the same call with Lin and Lout swapped. */
int ercg_reverse_seq(const float* x, int64_t ldx, int Lin, int B, int D, const int32_t* counts, float* out, int64_t ldo,
                     int Lout, void* stream);
/* y = log_softmax(x) over the C columns of each row (F.log_softmax(., 2) of the classifiers' heads); bwd: dx = dy - exp(y) *
 * sum_c dy.  Any C >= 1; rows == 0: no-op. */
int ercg_log_softmax_fwd(const float* x, int64_t ldx, float* y, int64_t ldy, int64_t rows, int C, void* stream);
int ercg_log_softmax_bwd(const float* y, int64_t ldy, const float* dy, int64_t lddy, float* dx, int64_t lddx, int64_t rows,
                         int C, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* ERCGRAPH_H_ */
