/* aria_b200 — C ABI of the B200-native Aria hot path (libaria_b200.so).
 *
 * Every entry point is `extern "C"`, takes raw DEVICE pointers + sizes + a cudaStream_t, never allocates or
 * frees, launches asynchronously on the caller's stream and returns 0 or a negative error code.  There is
 * no CPU fallback: unsupported shapes are errors.  Pointers must be 16-byte aligned and rows contiguous.
 *
 * Each function names the reference interface (rhymes-ai/Aria @ 9b25fecb) it replaces.  The reference is
 * pure Python; its "FFI" for this path is the set of third-party kernels it imports (SURVEY.md §2b):
 *   grouped_gemm.ops.gmm (aria/model/moe_lm.py:432,484), flash-attn / SDPA behind the HF attention classes
 *   (moe_lm.py:594, vision_encoder.py:120), and the ATen ops of the router / dispatcher (moe_lm.py:261-269,
 *   329-332, 350-363).  INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 */
#ifndef ARIA_B200_H
#define ARIA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* aria_stream_t; /* == cudaStream_t */

#define ARIA_OK 0
#define ARIA_ERR_BAD_ARG (-1)
#define ARIA_ERR_UNSUPPORTED (-2)
#define ARIA_ERR_CUDA (-3)

/* Library/ABI version and build target ("sm_100a"). */
int aria_abi_version(void);
const char* aria_build_arch(void);

/* ------------------------------------------------------------------------------------------------
 * GEMM family (tcgen05 + TMA, bf16 in, fp32 accumulate in TMEM, bf16 out).
 * One descriptor drives: nn.Linear-layout dense GEMMs, the reference's grouped expert GEMM, and the fused
 * epilogues of the hot path.  Rounding points mirror the reference's op-by-op bf16 rounding.
 * ------------------------------------------------------------------------------------------------ */
enum { ARIA_B_NK = 0,  /* B[n_seg][N,K], K contiguous — torch.nn.Linear.weight                        */
       ARIA_B_GKN = 1, /* B[G,K,N],      N contiguous — GroupedGEMM.weight (moe_lm.py:465)            */
       ARIA_B_GNK = 2  /* B[G,N,K],      K contiguous — the same expert weight used transposed (dgrad) */ };
enum { ARIA_EPI_LINEAR = 0, /* out = act(acc + bias) (+ residual)                                      */
       ARIA_EPI_SWIGLU = 1, /* out = silu(acc_gate) * acc_up  (moe_lm.py:505-507 `glu`, LlamaMLP)      */
       ARIA_EPI_HEADS = 2   /* (+bias) (+RoPE) and scatter to [B, H, T, head_ld] head-major buffers    */ };
enum { ARIA_ACT_NONE = 0, ARIA_ACT_GELU_TANH = 1, /* F.gelu(approximate="tanh") — Idefics2 MLP       */
       ARIA_ACT_GELU_NEW = 2                       /* transformers NewGELU, op-by-op bf16 — projector  */ };

typedef struct aria_gemm_desc {
  /* A: activations [m, k] bf16, row stride lda (elements). For grouped GEMMs rows are grouped by expert. */
  const void* a;
  int64_t lda;
  int64_t m, n, k;   /* n = OUTPUT columns per segment (SWIGLU: B carries 2n columns: gate then up)       */
  /* B: weights. NK layout: up to 3 segments (e.g. q,k,v projections, or gate,up for SWIGLU), each [n,k]
   * (SWIGLU: b[0] = gate [n,k], b[1] = up [n,k]).  GKN layout: b[0] = [G, k, n] (SWIGLU: [G, k, 2n]).  */
  const void* b[3];
  int32_t n_seg;
  int32_t b_layout;
  /* grouping: num_groups = 1 and group_offsets = NULL for a dense GEMM; else group_offsets[G+1] (device,
   * int32) are the row offsets of each expert's contiguous row block inside A / out.                   */
  int32_t num_groups;
  const int32_t* group_offsets;
  int32_t group_mod;       /* grouped weights: group g uses weight block g % group_mod (> 0), g / -group_mod (< 0), g (0).
                            * Expert parallelism receives rows grouped by (source rank, local expert): num_groups = W*E_loc,
                            * mod = E_loc; or by (local expert, source rank): mod = -W, which keeps the W groups that share
                            * an expert's weights next to each other in the tile order (one HBM read, W-1 L2 hits) */
  /* epilogue */
  int32_t epilogue;
  int32_t act;
  const void* bias[3];     /* per segment [n] bf16 or NULL                                               */
  const void* residual;    /* [m, n] bf16 or NULL (LINEAR only), row stride ldr                          */
  int64_t ldr;
  void* out[3];            /* LINEAR/SWIGLU: out[0] = [m, n_seg*n] row stride ldo; HEADS: one per segment */
  int64_t ldo;
  /* HEADS epilogue: row r of A is (batch r / rows_per_batch, token r % rows_per_batch); column c of
   * segment s is (head c / head_dim, d c % head_dim); destination element
   *   out[s] + batch*stride_b + head*stride_h + (pos0 + token)*head_ld + d                              */
  int32_t head_dim, head_ld, rows_per_batch, pos0;
  int64_t stride_b, stride_h;
  int32_t rope_mask;       /* bit s set: apply rotate-half RoPE to segment s (needs head_dim == 128)     */
  const void* rope_cos;    /* [max_pos, head_dim] bf16 tables (aria_rope_table)                          */
  const void* rope_sin;
  const int32_t* position_ids; /* [m] or NULL (then position = pos0 + token)                              */
  /* debug overrides of the UMMA shared-memory descriptor fields (0 = default); bring-up only            */
  int32_t dbg_lbo, dbg_sbo, dbg_kadv;
  /* Expert parallelism over NVLink peer memory (fused compute + collective, SURVEY.md §8e):
   *   group_counts  non-NULL: group g = rows [group_offsets[g], group_offsets[g] + group_counts[g]) — fixed-capacity
   *                 regions a peer GPU fills without knowing the other senders' counts; a_rows = rows of the A buffer
   *                 (m then only feeds the tile-shape heuristics: pass the expected row count).
   *   out_group_base / out_group_row0 (LINEAR): row r of group g is stored at
   *                 (bf16*)out_group_base[g] + (out_group_row0[g] + r) * ldo — e.g. the SOURCE rank's combine buffer, so the
   *                 fc2 epilogue IS the return all-to-all (16-byte stores through NVSwitch). */
  const int32_t* group_counts;
  int64_t a_rows;
  const void* out_group_base;      /* uint64 device addresses [G] */
  const int32_t* out_group_row0;   /* [G] */
} aria_gemm_desc_t;

/* Generic entry.  Replaces: torch F.linear / cuBLAS on the path, and grouped_gemm.ops.gmm. */
int aria_gemm(const aria_gemm_desc_t* desc, aria_stream_t stream);

/* Drop-in for `grouped_gemm.ops.gmm(a, b, batch_sizes)` as called at moe_lm.py:484 (`experts_gemm`), except
 * that the per-expert row offsets stay on the device (no .cpu() sync, moe_lm.py:478):
 *   out[off[e]:off[e+1]] = a[off[e]:off[e+1]] @ b[e],  a [rows,k], b [G,k,n], out [rows,n], all bf16.      */
int aria_grouped_gemm(const void* a, const void* b, void* out, const int32_t* group_offsets, int64_t rows,
                      int64_t k, int64_t n, int32_t num_groups, aria_stream_t stream);

/* Weight gradient of a (grouped) linear layer — backward of gmm / F.linear:
 *   out[g, m, n] = sum_{r in group g} a[r, m] * b[r, n]   a [rows, md] (row stride lda), b [rows, nd] (ldb), out [G, md, nd] bf16.
 * group_offsets: device int32 row offsets, each a multiple of 16 (aria_build_permutation with row_align = 16).
 * num_sources = 1: offsets[G+1].  num_sources = S > 1 (expert parallelism): rows are grouped (source rank, g),
 * source-major, offsets[S*G+1], and out[g] sums the S partial products — no separate reduction pass. */
int aria_grouped_wgrad(const void* a, int64_t lda, const void* b, int64_t ldb, void* out, const int32_t* group_offsets,
                       int64_t rows, int64_t md, int64_t nd, int32_t num_groups, int32_t num_sources, aria_stream_t stream);

/* int64 counts (tokens_per_expert as the reference passes it, moe_lm.py:264-269) -> int32 offsets[G+1]. */
int aria_offsets_from_counts(const int64_t* counts, int32_t* offsets, int32_t num_groups, aria_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * MoE routing / dispatch (HBM-bound kernels)
 * ------------------------------------------------------------------------------------------------ */
/* TopKRouter.forward (moe_lm.py:275-293 = gating :190-201 + routing :261-269), eval path.
 *   x [T, d] bf16, w_router [E, d] bf16 -> logits [T, E] bf16 (required: the top-k runs on the rounded values),
 *   top_idx [T, k] int32 (descending logit, ties: lowest expert id), scores [T, k] bf16 (fp32 softmax over
 *   the k selected bf16 logits, rounded to bf16), counts [E] int32 (must be zeroed by this call: it is).
 * E <= 64, k <= 8. */
int aria_router_topk(const void* x, const void* w_router, void* logits_out, int32_t* top_idx, void* scores,
                     int32_t* counts, int64_t T, int32_t d, int32_t E, int32_t k, aria_stream_t stream);
/* Same routing from precomputed bf16 logits (exact integer/bit parity path; torch.topk + softmax + histc). */
int aria_route_from_logits(const void* logits, int32_t* top_idx, void* scores, int32_t* counts, int64_t T,
                           int32_t E, int32_t k, aria_stream_t stream);

/* Routing with the expert choice GIVEN (parity / replay hook): top_idx [T, k] int32 is an INPUT; scores = fp32 softmax over the
 * logits at those ids (same arithmetic as above), counts = their histogram.  Lets a test inject the oracle's top-k into the
 * CUDA path so that bf16 near-ties in the router cannot hide other differences. */
int aria_route_given_indices(const void* logits, const int32_t* top_idx, void* scores, int32_t* counts, int64_t T,
                             int32_t E, int32_t k, aria_stream_t stream);

/* TokenDispatcher.token_permutation (moe_lm.py:313-334): stable counting sort of the T*k expert ids.
 *   offsets [E+1] int32 (exclusive scan of counts), dest_row [T*k] int32 (row of flattened (token,slot) in
 *   the expert-sorted order == inverse of the reference's `sorted_indices`), src_token [T*k] int32 (token of
 *   each sorted row == sorted_indices // k).  Order inside an expert = ascending flattened index (stable). */
/* row_align = 1: dense layout (inference).  row_align = 16 (training): every expert's block starts on a multiple of 16
 * rows; src_token then needs T*k + E*(row_align-1) slots and pad rows carry -1 (permute_rows writes zeros for them). */
int aria_build_permutation(const int32_t* top_idx, const int32_t* counts, int32_t* offsets, int32_t* dest_row,
                           int32_t* src_token, int64_t T, int32_t E, int32_t k, int32_t row_align, aria_stream_t stream);
/*   permuted[r, :] = x[src_token[r], :]  (index_select, moe_lm.py:330) */
int aria_permute_rows(const void* x, const int32_t* src_token, void* permuted, int64_t rows, int32_t d,
                      aria_stream_t stream);
/* TokenDispatcher.token_unpermutation (moe_lm.py:336-365) fused with `output += shared` (moe_lm.py:576):
 *   out[t] = bf16( sum_j bf16(y[dest_row[t*k+j]] * scores[t,j]) ) (+ shared[t]) ; fp32 accumulate. */
int aria_unpermute_combine(const void* y, const int32_t* dest_row, const void* scores, const void* shared,
                           void* out, int64_t T, int32_t d, int32_t k, aria_stream_t stream);

/* MoELayer.forward as ONE call (moe_lm.py:548-577; SURVEY.md §8b "moe_block_fwd"): router -> stable sort by expert ->
 * grouped fc1 + glu -> grouped fc2 -> unpermute + score-weighted sum + shared experts.  Launches the kernels of the entries
 * above in order from C (no Python between them), the shared-expert branch on `side_stream` when one is given (forked from /
 * joined to `stream` with events: becomes a parallel branch under CUDA-graph capture), counts and offsets never leave the
 * device (the reference's tokens_per_expert.cpu(), moe_lm.py:478, is gone).
 *   x [T, d]; w_router [E, d]; fc1_w [E, d, 2I] / fc2_w [E, I, d] (GroupedGEMM.weight layout); gate_w / up_w [I_shared, d],
 *   down_w [d, I_shared] (nn.Linear layout; I_shared = 0: no shared experts); out [T, d]; all bf16.
 *   forced_top_idx [T, k] int32 or NULL: expert choice given (parity / replay hook, see aria_route_given_indices).
 *   workspace: aria_moe_block_fwd_workspace_bytes(...) bytes, 16-byte aligned; holds every intermediate. */
int64_t aria_moe_block_fwd_workspace_bytes(int64_t T, int32_t d, int32_t E, int32_t k, int32_t I, int32_t I_shared);
int aria_moe_block_fwd(const void* x, const void* w_router, const void* fc1_w, const void* fc2_w, const void* gate_w,
                       const void* up_w, const void* down_w, void* out, int64_t T, int32_t d, int32_t E, int32_t k, int32_t I,
                       int32_t I_shared, const int32_t* forced_top_idx, void* workspace, int64_t workspace_bytes,
                       aria_stream_t stream, aria_stream_t side_stream);

/* ---- backward of the MoE block (BASELINE cfg 5; autograd through moe_lm.py:548-577) ---- */
/* h = bf16(bf16(silu(g)) * u) with g = h1[:, :I], u = h1[:, I:]  (unfused `glu`, moe_lm.py:505-507; training keeps h1). */
int aria_swiglu_fwd(const void* h1, void* h, int64_t rows, int32_t I, aria_stream_t stream);
/* dh1 = [dh * u * silu'(g) | dh * silu(g)] */
int aria_swiglu_bwd(const void* h1, const void* dh, void* dh1, int64_t rows, int32_t I, aria_stream_t stream);
/* backward of aria_unpermute_combine w.r.t. y and scores:
 *   dy[dest_row[t*k+j]] = bf16(scores[t,j] * dout[t]),  dscores[t,j] = <dout[t], y[dest_row[t*k+j]]> (fp32).
 * dy rows that no (t,j) maps to (alignment pads) must be pre-zeroed by the caller. */
int aria_combine_bwd(const void* dout, const void* y, const int32_t* dest_row, const void* scores, void* dy, float* dscores,
                     int64_t T, int32_t d, int32_t k, aria_stream_t stream);
/* backward of softmax-over-top-k (moe_lm.py:261-262): dlogits[t, idx[t,j]] = s_j * (g_j - sum_i s_i g_i), zeros elsewhere. */
int aria_router_bwd(const float* dscores, const void* scores, const int32_t* top_idx, void* dlogits, int64_t T, int32_t E,
                    int32_t k, aria_stream_t stream);
/* Training-mode router losses (TopKRouter.apply_z_loss / apply_aux_loss, moe_lm.py:203-241; z_loss_func :128-140,
 * switch_load_balancing_loss_func :143-166).  logits [T,E] bf16, counts [E] int32 (tokens_per_expert), E <= 256.
 *   losses[0] = z_coeff * mean_t(logsumexp(logits_t)^2)
 *   losses[1] = aux_coeff * E/(T*k) * sum_e mean_t(softmax(logits)_te) * counts[e]          (fp32 softmax, :235)
 * The reference uses the values only through MoEAuxLossAutoScaler (:84-125): aria_router_aux_bwd ADDS
 * loss_scale * d(losses[0] + losses[1])/d(logits) to dlogits (bf16 [T,E], e.g. the output of aria_router_bwd);
 * loss_scale is MoEAuxLossAutoScaler.main_loss_backward_scale. */
size_t aria_router_aux_workspace_bytes(int32_t E);
int aria_router_aux_loss(const void* logits, const int32_t* counts, float* losses, int64_t T, int32_t E, int32_t k, float z_coeff,
                         float aux_coeff, void* workspace, size_t ws_bytes, aria_stream_t stream);
int aria_router_aux_bwd(const void* logits, const int32_t* counts, void* dlogits, int64_t T, int32_t E, int32_t k, float z_coeff,
                        float aux_coeff, float loss_scale, aria_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Norms, RoPE table, embedding, patches
 * ------------------------------------------------------------------------------------------------ */
/* LlamaRMSNorm (moe_lm.py:599-602,631): out = w * bf16(x * rsqrt(mean(x^2) + eps)).
 * If residual != NULL: first h = bf16(x + residual), written to sum_out, and the norm is taken of h. */
int aria_rmsnorm(const void* x, const void* residual, const void* weight, void* out, void* sum_out, int64_t rows,
                 int32_t d, float eps, aria_stream_t stream);
/* Backward of aria_rmsnorm without residual — replaces the autograd of LlamaRMSNorm (moe_lm.py:599-602):
 *   dx = r * (g - x * r^2 * mean(g * x)) (+ dres),  g = dy * w,  r = rsqrt(mean(x^2) + eps);   dw = sum_rows dy * bf16(x * r).
 * dres [rows, d] or NULL: the residual-stream gradient, added into dx in the same pass.  dw [d] bf16 is reduced
 * deterministically through fp32 per-block partials in the workspace (no atomics).
 * workspace: aria_rmsnorm_bwd_workspace_bytes(rows, d) = min(rows, 256) * d * 4 bytes. */
int64_t aria_rmsnorm_bwd_workspace_bytes(int64_t rows, int32_t d);
int aria_rmsnorm_bwd(const void* x, const void* weight, const void* dy, const void* dres, void* dx, void* dw, int64_t rows,
                     int32_t d, float eps, void* workspace, int64_t workspace_bytes, aria_stream_t stream);
/* Backward of rotate-half RoPE — replaces the autograd of apply_rotary_pos_emb (transformers modeling_llama), in place on
 * token-major x [rows, n_heads*128] bf16: dx1 = dy1*cos + dy2*sin, dx2 = dy2*cos - dy1*sin (x1 / x2 = the two 64-wide halves
 * of a head).  Positions as in the HEADS epilogue: position_ids[r] (int32) when given, else r % rows_per_batch; cos/sin
 * tables from aria_rope_table. */
int aria_rope_bwd(void* x, const void* cos, const void* sin, const int32_t* position_ids, int64_t rows, int32_t n_heads,
                  int32_t rows_per_batch, aria_stream_t stream);
/* nn.LayerNorm (Idefics2 encoder layers, projector): out = bf16((x-mean)*rstd*w + b). */
int aria_layernorm(const void* x, const void* weight, const void* bias, void* out, int64_t rows, int32_t d,
                   float eps, aria_stream_t stream);
/* LlamaRotaryEmbedding (moe_lm.py:632): cos/sin [n_pos, head_dim] bf16 from fp32 inv_freq[head_dim/2]. */
int aria_rope_table(const float* inv_freq, void* cos_out, void* sin_out, int32_t n_pos, int32_t head_dim,
                    aria_stream_t stream);
/* nn.Embedding gather: out[i] = table[ids[i]]. */
int aria_embedding(const int64_t* ids, const void* table, void* out, int64_t n, int32_t d, aria_stream_t stream);
/* masked_scatter merge (modeling_aria.py:272-283): rows where ids == image_token get consecutive rows of
 * `features`; `slot_index` [n] int32 scratch.  Returns the number of image slots through *count_out (device). */
int aria_merge_image_features(const int64_t* ids, int64_t image_token, const void* features, void* embeds,
                              int32_t* count_out, int64_t n, int32_t d, aria_stream_t stream);
/* Conv2d(3,C,14,14) as im2col: pixel_values [B,3,S,S] bf16 -> patches [B*N, k_pad] (k = 3*P*P zero padded). */
int aria_im2col_patches(const void* pixels, void* patches, int32_t B, int32_t S, int32_t P, int32_t k_pad,
                        aria_stream_t stream);
/* out[r,:] = bf16(x[r,:] + table[pos[r],:]) — position-embedding add of Idefics2VisionEmbeddings. */
int aria_add_pos_embedding(const void* x, const int64_t* pos_ids, const void* table, void* out, int64_t rows,
                           int32_t d, aria_stream_t stream);

/* Multi-GPU: allow kernels on the current device to load/store `peer_device`'s memory over NVLink (idempotent). */
int aria_enable_peer_access(int32_t peer_device);
/* CUDA IPC for peer-mapped arenas: export the 64-byte handle of the allocation containing `ptr` (+ byte offset of ptr in
 * it); open maps a peer's allocation into the current device's context (lazy peer access) and returns its base. */
int aria_ipc_export(const void* ptr, void* handle64, int64_t* offset_out);
int aria_ipc_open(const void* handle64, void** base_out);
int aria_ipc_close(void* base);

/* Expert-parallel exchange over NVLink peer memory (aria_b200/csrc/ep.cu): replaces the all-to-all the reference's
 * dispatcher lost (moe_lm.py:296-297).  `peer_*` arrays are device arrays of W addresses (one per rank, as mapped on THIS
 * GPU).  All calls are asynchronous and need no host sync. */
int aria_ep_publish_counts(const int32_t* counts, const uint64_t* peer_counts, int32_t rank, int32_t W, int32_t E,
                           aria_stream_t stream);                      /* my counts[E] -> counts_all[rank][:] on every rank */
int aria_peer_barrier(const uint64_t* peer_flags, int32_t rank, int32_t W, int32_t* epoch_dev /* device counter, advanced by the call */,
                      aria_stream_t stream);
int aria_ep_layout(const int32_t* counts_all, int32_t rank, int32_t W, int32_t E, int32_t* roff, int32_t* send_base,
                   int32_t* ret_base, aria_stream_t stream);          /* roff[W*E/W+1], send_base[E], ret_base[W*E/W] */
/* Fused permute + dispatch (and the way back): row i of group g -> rank g/group_div, row dst_row_base[g] + i - off[g];
 * source row = rows[src_token ? src_token[i] : i].  max_rows only sizes the grid. */
int aria_scatter_rows_grouped(const void* rows, const int32_t* src_token, const int32_t* group_offsets, int32_t G,
                              const int32_t* dst_row_base, int32_t group_div, const uint64_t* peer_bufs, int32_t d,
                              int64_t max_rows, aria_stream_t stream);
/* Fused exchange (fixed-capacity regions; see csrc/ep.cu): gathers the token rows in expert order (src_token / offsets from
 * aria_build_permutation) and stores each into region (e % E_loc, rank) = index (e % E_loc) * W + rank of owner e / E_loc — peer_recv[p] = rank p's receive
 * buffer [W*E_loc][cap][d] as mapped on this GPU — and publishes per-block (row count, first sorted row) into the owners'
 * meta arrays peer_counts[p] / peer_row0[p] ([W*E_loc] int32 each).  A peer barrier must follow before the owner reads. */
int aria_ep_dispatch(const void* x, const int32_t* src_token, const int32_t* offsets, const uint64_t* peer_recv,
                     const uint64_t* peer_counts, const uint64_t* peer_row0, int32_t rank, int32_t W, int32_t E,
                     int32_t cap, int32_t d, int64_t max_rows, aria_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Attention (tcgen05 QK^T / PV, fp32 online softmax)
 * ------------------------------------------------------------------------------------------------ */
/* softmax(q k^T * scale + mask) v for head_dim 128 (LM) — replaces flash_attn_func / SDPA behind
 * LLAMA_ATTENTION_CLASSES (moe_lm.py:594) and, with hd padded 72->128, the Idefics2 / projector attention.
 *   q [B, H, Tq, 128], k/v [B, H, Tk_max, 128] head-major bf16 (HF cache layout), first Tk rows valid.
 *   out [B, Tq, H*out_hd] token-major bf16 (only the first out_hd of 128 dims are written).
 *   causal != 0: query i (absolute position Tk - Tq + i) sees keys <= its position.
 *   key_mask [B, Tk] uint8 or NULL: 1 = key is masked OUT (image_attn_mask convention, vision_encoder.py:147). */
int aria_attention_fwd(const void* q, const void* k, const void* v, void* out, const uint8_t* key_mask,
                       int32_t B, int32_t H, int32_t Tq, int32_t Tk, int64_t q_stride_b, int64_t q_stride_h,
                       int64_t kv_stride_b, int64_t kv_stride_h, int32_t out_hd, float scale, int32_t causal,
                       void* workspace, int64_t workspace_bytes, aria_stream_t stream);
/* Scratch for the stream-K pieces of a persistent (non-causal) launch: when there are more (batch, head, 256-query) units than
 * SMs, the units left over after the whole rounds are cut along the keys and spread over all SMs; their partial (O, m, l) go
 * through this workspace and a merge kernel.  workspace may be NULL (or too small): the leftover units then run whole. */
int64_t aria_attention_fwd_workspace_bytes(int32_t B, int32_t H, int32_t Tq, int32_t Tk, int32_t out_hd, int32_t causal);
/* Single-token decode against a KV cache (HBM-bound, split-KV): q element (b,h,:) at q + b*q_stride_b + h*q_stride_h
 * (128 contiguous bf16), cache [B,H,Tk_max,128], out [B, H*128].  workspace: B*H*splits*(128+2) floats.
 * key_mask [B, Tk] uint8 or NULL: 1 = key is masked OUT (padded batch: the HF 2-D attention_mask inverted). */
int aria_attention_decode(const void* q, const void* k, const void* v, void* out, const uint8_t* key_mask, int32_t B, int32_t H, int32_t Tk,
                          int64_t q_stride_b, int64_t q_stride_h, int64_t kv_stride_b, int64_t kv_stride_h, float scale,
                          void* workspace, int64_t workspace_bytes, aria_stream_t stream);
int64_t aria_attention_decode_workspace_bytes(int32_t B, int32_t H, int32_t Tk);
/* Causal self-attention forward (Tq = Tk = T, head_dim 128) that also stores each query row's softmax normaliser — the
 * forward half of the autograd of eager_attention_forward / SDPA behind moe_lm.py:594.  Layouts as aria_attention_fwd:
 * q/k/v [B,H,T,128] head-major, out [B,T,H*128] token-major;  lse [B,H,T] fp32 = log2(sum_k 2^(s_k * scale * log2 e)) (the
 * log2 domain of the scaled scores), +INF for a query row that sees no key.  out is bit-identical to aria_attention_fwd's
 * for the launches that function runs on the same kernel (causal, T > 1024).  causal = 0 or head_dim != 128:
 * ARIA_ERR_UNSUPPORTED. */
int aria_attention_fwd_lse(const void* q, const void* k, const void* v, void* out, float* lse, const uint8_t* key_mask, int32_t B,
                           int32_t H, int32_t T, int64_t q_stride_b, int64_t q_stride_h, int64_t kv_stride_b, int64_t kv_stride_h,
                           float scale, int32_t head_dim, int32_t causal, aria_stream_t stream);
/* Causal attention backward — replaces the autograd of eager_attention_forward / SDPA behind moe_lm.py:594.
 *   q/k/v [B,H,T,128] head-major (the forward's buffers); out, dout, dq, dk, dv [B,T,H*128] token-major bf16 (the layout the
 *   q/k/v projection GEMMs read back); lse from aria_attention_fwd_lse; key_mask [B,T] uint8 or NULL, 1 = masked out.
 * Deterministic: repeated calls give bit-identical dq/dk/dv (no atomics).  causal = 0 or head_dim != 128:
 * ARIA_ERR_UNSUPPORTED.  workspace: aria_attention_bwd_workspace_bytes(B, H, T) = Delta [B,H,T] fp32, rounded up to 256 B. */
int64_t aria_attention_bwd_workspace_bytes(int32_t B, int32_t H, int32_t T);
int aria_attention_bwd(const void* q, const void* k, const void* v, const void* out, const void* dout, const float* lse, void* dq,
                       void* dk, void* dv, const uint8_t* key_mask, int32_t B, int32_t H, int32_t T, int64_t q_stride_b,
                       int64_t q_stride_h, int64_t kv_stride_b, int64_t kv_stride_h, float scale, int32_t head_dim, int32_t causal,
                       void* workspace, int64_t workspace_bytes, aria_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ARIA_B200_H */
