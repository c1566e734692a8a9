// Attention forward, third generation (round 2) — replaces attn_fwd2_kernel of attention.cu.
//
// Same contraction scheme (S = Q K^T and O += P V on tcgen05, S/P/O in TMEM, P consumed from TMEM) and the same 256-query
// CTA shape (two 128-row tiles ping-pong), rebuilt around what round 1 measured at the ViT shape (16 x 4900 x 4900, hd 72:
// 231 us/layer = 0.32 of the tensor roofline on real FLOPs):
//   * head dims 72 (ViT, projector) are staged 80 wide, not 128: a SW128 chunk of 64 columns + a SWIZZLE_32B chunk of 16
//     (Q, K: the 5th UMMA k-step; V: five 16-wide MN-major chunks) — 40 KB instead of 64 KB of K/V per key block through
//     L2 -> shared memory, three K/V stages instead of two;
//   * the exponentials are the bound at hd 72 (16 MUFU/clk/SM: 2048 clk per 256 x 128 block vs 1280 clk of MMA): a
//     compile-time share of them is evaluated on the FMA pipe (exp2_poly2, packed FFMA2), scaling and row sums are packed
//     f32x2 ops, the row max uses 3-input max;
//   * one MMA-issuing thread PER TILE (two warps) — each tile's QK / PV chain is independent, and a single thread
//     retiring both was the critical path in round 1 (profiles/r01_issue_loop_study.txt);
//   * warp-specialised register budgets (setmaxnreg): the softmax warpgroups hold a whole S row in registers without
//     spilling;
//   * non-causal launches are PERSISTENT with a hybrid stream-K split: CTA c runs units c, c + C, ... whole, and the
//     U mod C leftover units are cut along the keys into floor(C / leftover) chunks spread over the CTAs, their partial
//     (O, m, l) merged by attn_merge_kernel — 320 units on 148 SMs take 2.17 rounds instead of 3.
//   Causal launches (LM prefill) keep one unit per CTA, heaviest first (the hardware block scheduler is the LPT list
//   scheduler there).
// Where it stands (profiles/r02_attention_notes.txt): 185-192 us on that shape = 0.39-0.40 of the sustained tensor peak on real
// FLOPs.  ncu: MUFU pipe 56 %, tensor pipe 35 %: each tile is a serial chain S -> softmax -> P -> PV -> QK whose fixed latencies
// (five barrier hand-offs, TMEM load / store round trips), not a pipe, set the 3310-clk period per 256 x 128 block.  The share of
// exponentials on the FMA pipe (ARIA_ATTN_POLY) therefore stays 0: it measured slower (+40 % instructions for -25 % MUFU).
#include <stdlib.h>

#include "common.cuh"
#include "ptx.cuh"

namespace aria {

constexpr int A3_BM = 128, A3_BN = 128;
constexpr int A3_THREADS = 384;  // WG0 / WG1 (warps 0-7): softmax of tile 0 / 1; WG2: warp 8 TMA, warps 9 / 10 MMA issuers of tile 0 / 1, warp 11 TMEM owner
// ---- build-time switches (scripts/build_variant.sh; measurements in profiles/r02_attention_notes.txt)
#ifndef ARIA_ATTN_PF16
#define ARIA_ATTN_PF16 0    // 1 = P as packed fp16 from ex2.approx.f16x2 with a (fp16 A, bf16 B) PV descriptor. DEAD END, kept as a record:
                            // B200 raises cudaErrorIllegalInstruction on a kind::f16 MMA whose A and B formats differ
                            // (gpurun_out/r02 run 9), and ptxas lowers ex2.approx.f16x2 to TWO MUFU.EX2.F16 + PRMT, so it would
                            // not have halved the MUFU work either.  0: fp32 ex2 + bf16 pack
#endif
#ifndef ARIA_ATTN_POLY
#define ARIA_ATTN_POLY 0    // (PF16 = 0 only) of every 16 exponent pairs, how many go through exp2_poly2 instead of MUFU (0..16)
#endif
#ifndef ARIA_ATTN_SEQ
#define ARIA_ATTN_SEQ 0     // 1: the two softmax warpgroups take turns exponentiating (token passing; measured: no gain)
#endif
#ifndef ARIA_ATTN_ABLATE
#define ARIA_ATTN_ABLATE 0  // measurement-only variants (WRONG results): bit0 no exp math, bit1 no LDTM of S, bit2 no PV MMAs,
#endif                      // bit3 no QK MMAs, bit4 no STTM of P
#ifndef ARIA_ATTN_TRACE
#define ARIA_ATTN_TRACE 0   // measurement-only: per-role cycle accounting of CTA 0 written behind the workspace (scripts/trace_attn.py)
#endif
#if ARIA_ATTN_TRACE
#define TRACE_DECL long long tr_acc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long tr_t0 = clock64(); const long long tr_start = tr_t0
#define TRACE_MARK(slot) do { const long long tr_now = clock64(); tr_acc[slot] += tr_now - tr_t0; tr_t0 = tr_now; } while (0)
#define TRACE_DUMP(base) do { if (blockIdx.x == 0 && p.partial) { for (int z = 0; z < 12; ++z) p.partial[3200000 + (base) + z] = static_cast<float>(tr_acc[z]); \
                                p.partial[3200000 + (base) + 12] = static_cast<float>(clock64() - tr_start); } } while (0)
#else
#define TRACE_DECL
#define TRACE_MARK(slot)
#define TRACE_DUMP(base)
#endif

struct Attn3Params {
  int B, H, Tq, Tk;
  int out_hd;
  float scale_log2;
  const uint8_t* key_mask;  // [B, Tk] 1 = masked out
  __nv_bfloat16* out;       // [B, Tq, H*out_hd]
  float* partial;           // [slots][256][HD + 4] fp32 (O unnormalised | m | l | pad), stream-K pieces
  float* lse;               // [B, H, Tq] fp32 (LSE instantiations only): m + log2(l), +INF for a row without a visible key
  int n_q_pairs, n_kv_all;
  int units, n_cta, full_rounds, leftover, split;  // work distribution (see header)
};

// HD = contracted / produced head dim (80 for the 72-wide ViT heads, 128 for the LM); W = columns staged in shared memory:
// W = 80 is the lean layout described above, W = 128 stages the whole 128-wide row (two SW128 chunks; with HD = 80 only the
// first 80 columns are multiplied) — the LM layout, and the A/B fallback for hd 72 (env ARIA_ATTN_W=128).
template <int HD, int W>
struct A3Cfg {
  static_assert((W == 80 && HD == 80) || W == 128, "unsupported tile width");
  static constexpr int C1 = W - 64;                     // columns of the second chunk: 16 (SW32) or 64 (SW128)
  static constexpr int CH0 = A3_BM * 128;               // 16 KB: [128 rows][64 bf16], SW128
  static constexpr int CH1 = A3_BM * C1 * 2;            // 4 KB or 16 KB
  static constexpr int QK_TILE = CH0 + CH1;             // 20 KB / 32 KB
  static constexpr int V_TILE = A3_BN * W * 2;          // same size; W=80: five SW32 chunks, W=128: two SW128 chunks
  static constexpr int STAGES = W == 80 ? 3 : 2;
  static constexpr int SMEM = 2 * QK_TILE + STAGES * (QK_TILE + V_TILE) + 1024 + 512;
};

struct WorkItem {
  int bh, q_pair, kv0, kv1, slot;  // key blocks [kv0, kv1); slot >= 0: partial piece -> workspace slot
};

// item i of CTA c (same enumeration in every role)
ARIA_DEVICE bool get_item(const Attn3Params& p, int c, int i, WorkItem& w) {
  const int BH = p.B * p.H;
  int u;
  w.kv0 = 0;
  w.kv1 = p.n_kv_all;
  w.slot = -1;
  if (i < p.full_rounds) {
    u = i * p.n_cta + c;
  } else if (i == p.full_rounds && c < p.leftover * p.split) {
    const int lu = c / p.split, ch = c - lu * p.split;
    u = p.full_rounds * p.n_cta + lu;
    if (p.split > 1) {
      w.kv0 = static_cast<int>(static_cast<int64_t>(p.n_kv_all) * ch / p.split);
      w.kv1 = static_cast<int>(static_cast<int64_t>(p.n_kv_all) * (ch + 1) / p.split);
      w.slot = c;
    }
  } else {
    return false;
  }
  w.bh = u % BH;
  w.q_pair = p.n_q_pairs - 1 - u / BH;  // heaviest (latest rows) first for causal launches
  return true;
}

// LSE: the epilogue also stores each row's softmax normaliser in the log2 domain of scale*log2e*s the kernel tracks
// (the attention backward's input); whole units only (no stream-K pieces).
template <int HD, int W, bool CAUSAL, bool LSE = false>
__global__ void __launch_bounds__(A3_THREADS, 1)
attn_fwd3_kernel(const __grid_constant__ CUtensorMap tmQ0, const __grid_constant__ CUtensorMap tmQ1,
                 const __grid_constant__ CUtensorMap tmK0, const __grid_constant__ CUtensorMap tmK1,
                 const __grid_constant__ CUtensorMap tmV, const Attn3Params p) {
  using C = A3Cfg<HD, W>;
  constexpr int STAGES = C::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                          // [2 tiles][QK_TILE]
  uint8_t* sK = sQ + 2 * C::QK_TILE;           // [STAGES][QK_TILE]
  uint8_t* sV = sK + STAGES * C::QK_TILE;      // [STAGES][V_TILE]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + STAGES * C::V_TILE);
  uint64_t* q_full = bars;               // [2]
  uint64_t* q_empty = bars + 2;          // [2]
  uint64_t* k_full = bars + 4;           // [STAGES]
  uint64_t* v_full = bars + 4 + STAGES;  // [STAGES]
  uint64_t* kv_empty = bars + 4 + 2 * STAGES;  // [STAGES], 2 arrivals (one per issuer)
  uint64_t* s_full = bars + 4 + 3 * STAGES;    // [2]
  uint64_t* p_full = s_full + 2;               // [2 tiles][2 halves], 4 arrivals (one per softmax warp)
  uint64_t* o_full = p_full + 4;               // [2]
  uint64_t* o_empty = o_full + 2;              // [2], 4 arrivals
  uint64_t* seq = o_empty + 2;                 // [2], 4 arrivals: whose turn it is to exponentiate (ARIA_ATTN_SEQ)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(seq + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cw = warp - 8;  // control-warp index (0 TMA, 1 / 2 issuers, 3 TMEM owner); < 0: softmax warp
  if (cw == 0 && lane == 0) {
    prefetch_tmap(&tmQ0);
    prefetch_tmap(&tmK0);
    prefetch_tmap(&tmV);
    if (W == 80) {
      prefetch_tmap(&tmQ1);
      prefetch_tmap(&tmK1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
      mbar_init(&s_full[i], 1);
      // softmax -> issuer hand-offs: ONE arrival per warp (lane 0 after __syncwarp), not one per thread
      mbar_init(&p_full[2 * i], 4);
      mbar_init(&p_full[2 * i + 1], 4);
      mbar_init(&o_full[i], 1);
      mbar_init(&o_empty[i], 4);
      mbar_init(&seq[i], 4);
    }
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&kv_empty[i], 2);
    }
    fence_mbar_init();
  }
  if (cw == 3) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int cta = blockIdx.x;
#if ARIA_ATTN_TRACE
  uint64_t tr_g0 = 0;
  long long tr_c0 = 0;
  if (threadIdx.x == 0) {
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_g0));
    tr_c0 = clock64();
  }
#endif
  const int pos_off = p.Tk - p.Tq;

  // key blocks a tile of an item has to visit: [kv0, min(kv1, causal limit))
  auto tile_kv_end = [&](const WorkItem& w, int t) {
    int e = w.kv1;
    if (CAUSAL) {
      const int last_row = min(w.q_pair * 2 * A3_BM + (t + 1) * A3_BM, p.Tq) - 1;
      e = min(e, (pos_off + last_row) / A3_BN + 1);
    }
    if (w.q_pair * 2 * A3_BM + t * A3_BM >= p.Tq) e = w.kv0;  // tile has no valid row
    return max(e, w.kv0);
  };

  if (cw >= 0) {
    setmaxnreg_dec<88>();
    if (cw == 0) {
      // =========================== TMA producer ===========================
      if (elect_one()) {
        TRACE_DECL;
        uint32_t kv_it = 0;  // K/V blocks produced so far (ring position)
        WorkItem w;
        for (int i = 0; get_item(p, cta, i, w); ++i) {
          const int b = w.bh / p.H, h = w.bh % p.H;
          const int q0 = w.q_pair * 2 * A3_BM;
          for (int t = 0; t < 2; ++t) {
            mbar_wait(&q_empty[t], (i & 1) ^ 1);
            TRACE_MARK(0);
            mbar_arrive_expect_tx(&q_full[t], C::QK_TILE);
            tma_load_4d(sQ + t * C::QK_TILE, &tmQ0, &q_full[t], 0, q0 + t * A3_BM, h, b);
            tma_load_4d(sQ + t * C::QK_TILE + C::CH0, &tmQ1, &q_full[t], 64, q0 + t * A3_BM, h, b);
          }
          const int kv_end = max(tile_kv_end(w, 0), tile_kv_end(w, 1));
          for (int j = w.kv0; j < kv_end; ++j, ++kv_it) {
            const int s = kv_it % STAGES;
            TRACE_MARK(2);
            mbar_wait(&kv_empty[s], ((kv_it / STAGES) & 1) ^ 1);
            TRACE_MARK(1);
            uint8_t* dk = sK + s * C::QK_TILE;
            mbar_arrive_expect_tx(&k_full[s], C::QK_TILE);
            tma_load_4d(dk, &tmK0, &k_full[s], 0, j * A3_BN, h, b);
            tma_load_4d(dk + C::CH0, &tmK1, &k_full[s], 64, j * A3_BN, h, b);
            uint8_t* dv = sV + s * C::V_TILE;
            mbar_arrive_expect_tx(&v_full[s], C::V_TILE);
            if (W == 80) {
#pragma unroll
              for (int c = 0; c < 5; ++c) tma_load_4d(dv + c * (A3_BN * 32), &tmV, &v_full[s], c * 16, j * A3_BN, h, b);
            } else {
              tma_load_4d(dv, &tmV, &v_full[s], 0, j * A3_BN, h, b);
              tma_load_4d(dv + C::CH0, &tmV, &v_full[s], 64, j * A3_BN, h, b);
            }
          }
        }
        TRACE_MARK(2);
        TRACE_DUMP(0);
      }
    } else if (cw <= 2) {
      // =========================== MMA issuer of tile t ===========================
      const int t = cw - 1;
      if (elect_one()) {
        constexpr uint32_t idesc_qk = make_idesc_bf16(A3_BM, A3_BN, false, false);
        constexpr uint32_t idesc_pv = ARIA_ATTN_PF16 ? make_idesc_f16a_bf16b(A3_BM, HD, true) : make_idesc_bf16(A3_BM, HD, false, true);
        const uint32_t sQa = smem_u32(sQ) + t * C::QK_TILE, sKa = smem_u32(sK), sVa = smem_u32(sV);
        const uint64_t dQ0 = make_smem_desc_sw(sQa, 16, 1024, UMMA_SW128);
        const uint64_t dQ1 = W == 80 ? make_smem_desc_sw(sQa + C::CH0, 16, 256, UMMA_SW32) : make_smem_desc_sw(sQa + C::CH0, 16, 1024, UMMA_SW128);
        const uint64_t dK0 = make_smem_desc_sw(sKa, 16, 1024, UMMA_SW128);
        const uint64_t dK1 = W == 80 ? make_smem_desc_sw(sKa + C::CH0, 16, 256, UMMA_SW32) : make_smem_desc_sw(sKa + C::CH0, 16, 1024, UMMA_SW128);
        // V consumed MN-major: HD=80 five SW32 chunks (LBO = 4 KB chunk stride, SBO = 256, K step 512 B);
        //                      HD=128 two SW128 chunks (LBO = 16 KB, SBO = 1024, K step 2 KB)
        const uint64_t dV0 = W == 80 ? make_smem_desc_sw(sVa, A3_BN * 32, 256, UMMA_SW32) : make_smem_desc_sw(sVa, C::CH0, 1024, UMMA_SW128);
        constexpr uint32_t v_kadv = (W == 80 ? 512 : 2048) >> 4;
        const uint32_t tS = tmem_base + t * 128, tO = tmem_base + 256 + t * 128;
        const uint32_t s_full_a = smem_u32(&s_full[t]), p_full_a = smem_u32(&p_full[2 * t]);
        uint32_t kv_it = 0;   // ring position of the item's first block (all blocks of all items, as the producer counts)
        uint32_t blk = 0;     // blocks THIS tile has processed (phase of s_full / p_full)
        uint32_t done = 0;    // items in which this tile had work (phase of o_full / o_empty)
        WorkItem w;
        TRACE_DECL;
        auto issue_qk = [&](uint32_t ring) {
          const uint32_t st = ring % STAGES;
          TRACE_MARK(5);
          mbar_wait(&k_full[st], (ring / STAGES) & 1);
          TRACE_MARK(0);
          tc_fence_after();
          const uint64_t dk0 = dK0 + st * (C::QK_TILE >> 4), dk1 = dK1 + st * (C::QK_TILE >> 4);
          if (!(ARIA_ATTN_ABLATE & 8)) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16_ss(tS, dQ0 + k * 2, dk0 + k * 2, idesc_qk, k ? 1u : 0u);
            // second chunk: columns 64.. of the head (HD = 80: one more k-step, whichever way the chunk is staged)
#pragma unroll
            for (int k = 0; k < (HD - 64) / 16; ++k) umma_bf16_ss(tS, dQ1 + k * 2, dk1 + k * 2, idesc_qk, 1u);
          }
          umma_commit_addr(s_full_a);
        };
        for (int i = 0; get_item(p, cta, i, w); ++i) {
          const int n_all = max(tile_kv_end(w, 0), tile_kv_end(w, 1)) - w.kv0;  // blocks the producer streams for this item
          const int n_t = tile_kv_end(w, t) - w.kv0;                             // blocks this tile contracts
          if (n_t > 0) {
            TRACE_MARK(5);
            mbar_wait(&q_full[t], i & 1);
            TRACE_MARK(1);
            mbar_wait(&o_empty[t], (done & 1) ^ 1);  // previous item's epilogue has drained S/P/O of this tile
            TRACE_MARK(2);
            tc_fence_after();
            issue_qk(kv_it);
            ++done;
          }
          for (int j = 0; j < n_all; ++j) {
            const uint32_t ring = kv_it + j, st = ring % STAGES;
            if (j < n_t) {
              TRACE_MARK(5);
              mbar_wait(&v_full[st], (ring / STAGES) & 1);
              TRACE_MARK(3);
              const uint64_t dv = dV0 + st * (C::V_TILE >> 4);
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                TRACE_MARK(5);
                mbar_wait_addr(p_full_a + c * 8, blk & 1);
                TRACE_MARK(4);
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                  const int k = c * 4 + kk;
                  if (!(ARIA_ATTN_ABLATE & 4)) umma_bf16_ts(tO, tS + k * 8, dv + k * v_kadv, idesc_pv, (j | k) ? 1u : 0u);
                }
              }
              ++blk;
              if (j == n_t - 1) {
                umma_commit(&o_full[t]);
                umma_commit(&q_empty[t]);          // every QK of this item has been issued (and the PVs after them)
              }
              umma_commit(&kv_empty[st]);          // K(j) was read by QK(j), V(j) by PV(j): both issued by now
              if (j + 1 < n_t) issue_qk(ring + 1);
            } else {
              // this tile is done with the item (causal: the earlier rows need one block less): keep the ring's arrival count
              mbar_wait(&v_full[st], (ring / STAGES) & 1);
              mbar_arrive(&kv_empty[st]);
            }
          }
          if (n_t <= 0) {  // nothing to do for this tile: hand Q back so that the producer's phase bookkeeping stays uniform
            mbar_wait(&q_full[t], i & 1);
            mbar_arrive(&q_empty[t]);
          }
          kv_it += n_all;
        }
        TRACE_MARK(5);
        TRACE_DUMP(16 + 16 * t);
      }
    }
  } else {
    // =========================== softmax warpgroups ===========================
    setmaxnreg_inc<208>();
    const int t = warp >> 2;
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t tS = tmem_base + t * 128 + lane_addr;
    const uint32_t tO = tmem_base + 256 + t * 128 + lane_addr;
    const uint64_t scale2 = pack_f2(p.scale_log2, p.scale_log2);
    uint32_t blk = 0, done = 0, rounds = 0;
    WorkItem w;
    TRACE_DECL;
    for (int i = 0; get_item(p, cta, i, w); ++i) {
      const int b = w.bh / p.H, h = w.bh % p.H;
      const int q0 = w.q_pair * 2 * A3_BM + t * A3_BM;
      const int q = q0 + r;
      const bool row_ok = q < p.Tq;
      const int qpos = pos_off + q;
      const int kv_end = tile_kv_end(w, t);
      const int kv_end_all = ARIA_ATTN_SEQ ? max(tile_kv_end(w, 0), tile_kv_end(w, 1)) : kv_end;
      const uint8_t* km = p.key_mask ? p.key_mask + static_cast<int64_t>(b) * p.Tk : nullptr;
      float m_ref = -INFINITY, l = 0.f;

      // (ARIA_ATTN_SEQ: the exp phase is a token passed between the two softmax warpgroups — tile 0 block j, tile 1 block j,
      // tile 0 block j+1, ... — to force the tiles out of phase; a tile without work in a round still takes and passes it.)
      for (int j = w.kv0; j < kv_end_all; ++j, ++rounds) {
        const bool active = j < kv_end;
        uint32_t sr[4][32];
        float mx = -INFINITY;
        const int k0 = j * A3_BN;
        bool need_mask = false;
        if (active) {
          TRACE_MARK(7);
          mbar_wait(&s_full[t], blk & 1);
          TRACE_MARK(0);
          ++blk;
          tc_fence_after();
          need_mask = (k0 + A3_BN > p.Tk) || (CAUSAL && (k0 + A3_BN - 1 > pos_off + q0)) || km != nullptr;
          if (!(ARIA_ATTN_ABLATE & 2)) {
#pragma unroll
            for (int c = 0; c < 4; ++c) tmem_ld_32x32(tS + c * 32, sr[c]);
            tmem_ld_wait();
          } else {
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
              for (int e = 0; e < 32; ++e) sr[c][e] = __float_as_uint(static_cast<float>((e * 7 + c + lane) & 15) * 0.25f);
          }
          if (need_mask) {  // rare path (diagonal / tail / padded keys): -inf on dead keys
#pragma unroll
            for (int c = 0; c < 4; ++c) {
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                const int kc = k0 + c * 32 + e;
                const bool dead = kc >= p.Tk || (CAUSAL && kc > qpos) || (km && kc < p.Tk && km[kc]);
                if (dead) sr[c][e] = 0xff800000u;
              }
            }
          }
          float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            mx0 = fmax3(mx0, __uint_as_float(sr[0][e]), __uint_as_float(sr[0][e + 1]));
            mx1 = fmax3(mx1, __uint_as_float(sr[1][e]), __uint_as_float(sr[1][e + 1]));
            mx2 = fmax3(mx2, __uint_as_float(sr[2][e]), __uint_as_float(sr[2][e + 1]));
            mx3 = fmax3(mx3, __uint_as_float(sr[3][e]), __uint_as_float(sr[3][e + 1]));
          }
          mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        }
        TRACE_MARK(1);
        if (ARIA_ATTN_SEQ) mbar_wait(&seq[t], t == 0 ? ((rounds & 1) ^ 1) : (rounds & 1));   // my turn
        TRACE_MARK(2);
        if (active) {
          const float m_new = fmaxf(m_ref, mx * p.scale_log2);
          const bool want = (m_new - m_ref > 8.0f) || (m_ref == -INFINITY && m_new > -INFINITY);
          if (__any_sync(0xffffffffu, want)) {
            const float f = (m_ref == -INFINITY) ? 0.f : fast_ex2(m_ref - m_new);
            l *= f;
            m_ref = m_new;
            if (j > w.kv0) {
#pragma unroll 1
              for (int c = 0; c < HD; c += 16) {
                uint32_t v[16];
                tmem_ld_32x16(tO + c, v);
                tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * f);
                tmem_st_32x16(tO + c, v);
              }
            }
          }
          const float neg_m = (m_ref == -INFINITY) ? 0.f : -m_ref;
          const uint64_t negm2 = pack_f2(neg_m, neg_m);
          uint64_t lacc0 = 0ull, lacc1 = 0ull;  // packed (0.f, 0.f)
          float lh = 0.f;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t pk[16];
            if (ARIA_ATTN_PF16) {
#pragma unroll
              for (int e = 0; e < 16; ++e) {  // pair e = keys 2e, 2e+1 of this 32-key chunk: ONE MUFU op for both
                float x0, x1;
                unpack_f2(fma2(pack_u2(sr[c][2 * e], sr[c][2 * e + 1]), scale2, negm2), x0, x1);
                pk[e] = (ARIA_ATTN_ABLATE & 1) ? __float_as_uint(x0) : ex2_f16x2(x0, x1);
              }
              // row sum of the chunk: pairwise tree in fp16 (32 values, each <= 2^8), then fp32
              uint32_t t8[8], t4[4];
#pragma unroll
              for (int e = 0; e < 8; ++e) t8[e] = hadd2(pk[2 * e], pk[2 * e + 1]);
#pragma unroll
              for (int e = 0; e < 4; ++e) t4[e] = hadd2(t8[2 * e], t8[2 * e + 1]);
              lh += half2_sum_f32(hadd2(hadd2(t4[0], t4[1]), hadd2(t4[2], t4[3])));
            } else {
#pragma unroll
              for (int e = 0; e < 16; ++e) {  // pair e = keys 2e, 2e+1 of this 32-key chunk
                const uint64_t x = fma2(pack_u2(sr[c][2 * e], sr[c][2 * e + 1]), scale2, negm2);
                uint64_t pe;
                if (ARIA_ATTN_ABLATE & 1) {
                  pe = x;
                } else if (e < ARIA_ATTN_POLY) {
                  pe = need_mask ? exp2_poly2<true>(x) : exp2_poly2<false>(x);
                } else {
                  float x0, x1;
                  unpack_f2(x, x0, x1);
                  pe = pack_f2(fast_ex2(x0), fast_ex2(x1));
                }
                if (e & 1) lacc1 = add2(lacc1, pe); else lacc0 = add2(lacc0, pe);
                float p0, p1;
                unpack_f2(pe, p0, p1);
                pk[e] = pack_bf16(p0, p1);
              }
            }
            // P chunk (32 keys = 16 packed columns) overwrites S columns [16c, 16c+16): S is already in registers
            if (!(ARIA_ATTN_ABLATE & 16)) tmem_st_32x16(tS + c * 16, pk);
            if (c & 1) {  // 64 keys complete -> hand them to the PV MMA
              tmem_st_wait();
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(&p_full[2 * t + (c >> 1)]);
            }
          }
          TRACE_MARK(3);
          if (ARIA_ATTN_SEQ && lane == 0) mbar_arrive(&seq[1 - t]);   // pass the token (the p_full arrival synchronised the warp)
          float la, lb;
          unpack_f2(add2(lacc0, lacc1), la, lb);
          l += la + lb + lh;
        } else if (ARIA_ATTN_SEQ) {
          __syncwarp();
          if (lane == 0) mbar_arrive(&seq[1 - t]);
        }
      }
      if (kv_end <= w.kv0) continue;  // tile without work in this item (its issuer skipped it too)

      // ---- epilogue of the item: O (TMEM, fp32, relative to m_ref) -> out (normalised bf16) or -> partial slot
      TRACE_MARK(7);
      mbar_wait(&o_full[t], done & 1);
      TRACE_MARK(4);
      ++done;
      tc_fence_after();
      if (w.slot < 0) {
        const float inv_l = l > 0.f ? 1.0f / l : 0.f;
        if (LSE && row_ok) p.lse[static_cast<int64_t>(w.bh) * p.Tq + q] = l > 0.f ? m_ref + log2f(l) : INFINITY;
        __nv_bfloat16* orow = p.out + (static_cast<int64_t>(b) * p.Tq + q) * (static_cast<int64_t>(p.H) * p.out_hd) + h * p.out_hd;
#pragma unroll 1
        for (int c = 0; c < HD; c += 16) {
          uint32_t v[16];
          tmem_ld_32x16(tO + c, v);
          tmem_ld_wait();
          if (row_ok) {
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              if (c + g * 8 + 8 <= p.out_hd) {
                float x[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(v[g * 8 + e]) * inv_l;
                *reinterpret_cast<uint4*>(orow + c + g * 8) =
                    make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
              }
            }
          }
        }
      } else {
        float* prow = p.partial + (static_cast<int64_t>(w.slot) * 2 * A3_BM + t * A3_BM + r) * (HD + 4);  // = attn_merge_kernel's STRIDE
#pragma unroll 1
        for (int c = 0; c < HD; c += 16) {
          uint32_t v[16];
          tmem_ld_32x16(tO + c, v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 16; e += 2) *reinterpret_cast<uint2*>(prow + c + e) = make_uint2(v[e], v[e + 1]);
        }
        prow[HD] = m_ref;
        prow[HD + 1] = l;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[t]);
      TRACE_MARK(5);
    }
    if (r == 0) TRACE_DUMP(48 + 16 * t);
  }
  tc_fence_before();
  __syncthreads();
#if ARIA_ATTN_TRACE
  if (threadIdx.x == 0 && p.partial) {  // per-CTA: start / end on the global ns timer (low 32 bits), SM clocks, SM id
    uint64_t g1;
    uint32_t smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    float* d = p.partial + 3300000 + 4 * blockIdx.x;
    d[0] = __uint_as_float(static_cast<uint32_t>(tr_g0));
    d[1] = __uint_as_float(static_cast<uint32_t>(g1));
    d[2] = __uint_as_float(static_cast<uint32_t>(clock64() - tr_c0));
    d[3] = __uint_as_float(smid);
  }
#endif
  if (cw == 3) tmem_dealloc(tmem_base, 512);
}

// Merge of the stream-K pieces: unit `lu` (leftover unit) was cut into `split` key ranges, slot = lu * split + ch.
// One WARP per query row, one float4 of the head per lane (coalesced 16-byte loads of each piece's row);
// out = sum_i O_i 2^(m_i - M) / sum_i l_i 2^(m_i - M).  (Round 2: the first version used one thread per 8 columns in `leftover`
// blocks - 24 blocks for the ViT shape - and took 49 us per launch, a quarter of the attention kernel it follows.)
constexpr int A3_PSTRIDE_PAD = 4;  // floats after the HD columns of a partial row: m, l, 2 pad (keeps rows 16-byte aligned)
template <int HD>
__global__ void __launch_bounds__(256) attn_merge_kernel(const Attn3Params p) {
  constexpr int STRIDE = HD + A3_PSTRIDE_PAD;
  const int lane = threadIdx.x & 31;
  const int wg = blockIdx.x * 8 + (threadIdx.x >> 5);  // global warp = (leftover unit, row)
  const int lu = wg / (2 * A3_BM), row = wg - lu * (2 * A3_BM);
  const int BH = p.B * p.H;
  const int u = p.full_rounds * p.n_cta + lu;
  const int bh = u % BH, q_pair = p.n_q_pairs - 1 - u / BH;
  const int b = bh / p.H, h = bh % p.H;
  const int q = q_pair * 2 * A3_BM + row;
  if (q >= p.Tq) return;
  const float* base = p.partial + (static_cast<int64_t>(lu) * p.split * 2 * A3_BM + row) * STRIDE;
  const int64_t piece = static_cast<int64_t>(2 * A3_BM) * STRIDE;
  float M = -INFINITY;
  for (int ch = 0; ch < p.split; ++ch) M = fmaxf(M, __ldg(base + ch * piece + HD));
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float L = 0.f;
  const bool col_ok = lane * 4 < HD;
  for (int ch = 0; ch < p.split; ++ch) {
    const float* pr = base + ch * piece;
    const float m = __ldg(pr + HD);
    const float f = (m == -INFINITY) ? 0.f : exp2f(m - M);
    L += __ldg(pr + HD + 1) * f;
    if (col_ok) {
      const float4 o = __ldg(reinterpret_cast<const float4*>(pr) + lane);
      acc.x += o.x * f; acc.y += o.y * f; acc.z += o.z * f; acc.w += o.w * f;
    }
  }
  if (lane * 4 + 4 > p.out_hd) return;
  const float inv = L > 0.f ? 1.f / L : 0.f;
  __nv_bfloat16* orow = p.out + (static_cast<int64_t>(b) * p.Tq + q) * (static_cast<int64_t>(p.H) * p.out_hd) + h * p.out_hd;
  *reinterpret_cast<uint2*>(orow + lane * 4) = make_uint2(pack_bf16(acc.x * inv, acc.y * inv), pack_bf16(acc.z * inv, acc.w * inv));
}

static int make_tmap_heads3(CUtensorMap* tm, const void* ptr, int T, int H, int B, int64_t stride_b, int64_t stride_h,
                            uint32_t box_cols, CUtensorMapSwizzle swz) {
  uint64_t dims[4] = {128u, static_cast<uint64_t>(T), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
  uint64_t str[3] = {256u, static_cast<uint64_t>(stride_h) * 2, static_cast<uint64_t>(stride_b) * 2};
  uint32_t box[4] = {box_cols, 128, 1, 1};
  return make_tmap_bf16_swz(tm, ptr, 4, dims, str, box, swz);
}

template <int HD, int W, bool CAUSAL, bool LSE = false>
static int launch_attn3(const void* q, const void* k, const void* v, Attn3Params& p, int64_t q_stride_b, int64_t q_stride_h,
                        int64_t kv_stride_b, int64_t kv_stride_h, cudaStream_t stream) {
  using C = A3Cfg<HD, W>;
  CUtensorMap tmQ0, tmQ1, tmK0, tmK1, tmV;
  int rc = make_tmap_heads3(&tmQ0, q, p.Tq, p.H, p.B, q_stride_b, q_stride_h, 64, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = make_tmap_heads3(&tmK0, k, p.Tk, p.H, p.B, kv_stride_b, kv_stride_h, 64, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  if (W == 80) {
    rc = make_tmap_heads3(&tmQ1, q, p.Tq, p.H, p.B, q_stride_b, q_stride_h, 16, CU_TENSOR_MAP_SWIZZLE_32B);
    if (rc) return rc;
    rc = make_tmap_heads3(&tmK1, k, p.Tk, p.H, p.B, kv_stride_b, kv_stride_h, 16, CU_TENSOR_MAP_SWIZZLE_32B);
    if (rc) return rc;
    rc = make_tmap_heads3(&tmV, v, p.Tk, p.H, p.B, kv_stride_b, kv_stride_h, 16, CU_TENSOR_MAP_SWIZZLE_32B);
  } else {
    tmQ1 = tmQ0;
    tmK1 = tmK0;
    rc = make_tmap_heads3(&tmV, v, p.Tk, p.H, p.B, kv_stride_b, kv_stride_h, 64, CU_TENSOR_MAP_SWIZZLE_128B);
  }
  if (rc) return rc;
  auto kern = attn_fwd3_kernel<HD, W, CAUSAL, LSE>;
  static bool attr_set[kMaxDevices] = {};
  if (ensure_dynamic_smem(attr_set, kern, C::SMEM) != cudaSuccess) return ARIA_ERR_CUDA;
  kern<<<p.n_cta, A3_THREADS, C::SMEM, stream>>>(tmQ0, tmQ1, tmK0, tmK1, tmV, p);
  rc = check_launch("attn_fwd3_kernel");
  if (rc) return rc;
  if (p.leftover > 0 && p.split > 1) {
    attn_merge_kernel<HD><<<p.leftover * (2 * A3_BM / 8), 256, 0, stream>>>(p);
    rc = check_launch("attn_merge_kernel");
  }
  return rc;
}

}  // namespace aria

using namespace aria;

extern "C" int aria_attention_fwd_v2(const void* q, const void* k, const void* v, void* out, const uint8_t* key_mask, int32_t B, int32_t H,
                                     int32_t Tq, int32_t Tk, int64_t q_stride_b, int64_t q_stride_h, int64_t kv_stride_b,
                                     int64_t kv_stride_h, int32_t out_hd, float scale, int32_t causal, aria_stream_t stream_);  // attention.cu

extern "C" int64_t aria_attention_fwd_workspace_bytes(int32_t B, int32_t H, int32_t Tq, int32_t Tk, int32_t out_hd, int32_t causal) {
  (void)B; (void)H; (void)Tq; (void)Tk; (void)causal;
  // stream-K pieces of a persistent (non-causal) launch: at most one slot per CTA, 256 rows x (HD + 4) floats
  const int hd = out_hd <= 80 ? 80 : 128;
  return static_cast<int64_t>(sm_count()) * 2 * A3_BM * (hd + 4) * sizeof(float);
}

extern "C" int aria_attention_fwd(const void* q, const void* k, const void* v, void* out, const uint8_t* key_mask, int32_t B,
                                  int32_t H, int32_t Tq, int32_t Tk, int64_t q_stride_b, int64_t q_stride_h,
                                  int64_t kv_stride_b, int64_t kv_stride_h, int32_t out_hd, float scale, int32_t causal,
                                  void* workspace, int64_t workspace_bytes, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(q && k && v && out);
  ARIA_CHECK_ARG(B > 0 && H > 0 && Tq > 0 && Tk > 0 && Tk >= (causal ? Tq : 0));
  ARIA_CHECK_ARG(out_hd > 0 && out_hd <= 128 && out_hd % 8 == 0);
  ARIA_CHECK_ARG(q_stride_b % 8 == 0 && q_stride_h % 8 == 0 && kv_stride_b % 8 == 0 && kv_stride_h % 8 == 0);
  // short causal launches (the 768-token LM prefill: 60 units of <= 6 key blocks) are prologue-bound; the round-1 kernel, with
  // its lighter set-up, measures 23.3 us against 27.8 us there (profiles/r02_attn_v3_vs_v2.txt), and 1 % slower at T = 8192
  if (causal && Tk <= 1024 && static_cast<int64_t>(B) * H * ((Tq + 2 * A3_BM - 1) / (2 * A3_BM)) <= sm_count())
    return aria_attention_fwd_v2(q, k, v, out, key_mask, B, H, Tq, Tk, q_stride_b, q_stride_h, kv_stride_b, kv_stride_h, out_hd, scale,
                                 causal, stream_);
  Attn3Params p{};
  p.B = B;
  p.H = H;
  p.Tq = Tq;
  p.Tk = Tk;
  p.out_hd = out_hd;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.key_mask = key_mask;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.partial = static_cast<float*>(workspace);
  p.n_q_pairs = (Tq + 2 * A3_BM - 1) / (2 * A3_BM);
  p.n_kv_all = (Tk + A3_BN - 1) / A3_BN;
  const int64_t units = static_cast<int64_t>(B) * H * p.n_q_pairs;
  ARIA_CHECK_ARG(units < (1ll << 31));
  p.units = static_cast<int>(units);
  const int hd = out_hd <= 80 ? 80 : 128;
  const int sms = sm_count();
  static const int persist = [] { const char* e = getenv("ARIA_ATTN_PERSIST"); return e ? atoi(e) : 1; }();
  const bool can_split = workspace && workspace_bytes >= aria_attention_fwd_workspace_bytes(B, H, Tq, Tk, out_hd, causal);
  if (!causal && persist && units > sms) {
    // persistent: whole units round-robin, the leftover cut along the keys (needs the workspace; without it the leftover
    // units run whole on the first CTAs)
    p.n_cta = sms;
    p.full_rounds = static_cast<int>(units / sms);
    p.leftover = static_cast<int>(units - static_cast<int64_t>(p.full_rounds) * sms);
    p.split = 1;
    if (p.leftover > 0 && can_split) {
      p.split = sms / p.leftover;
      if (p.split > p.n_kv_all) p.split = p.n_kv_all;
      if (p.split < 1) p.split = 1;
    }
  } else if (!causal && persist && can_split && units * 2 <= sms && p.n_kv_all >= 4) {
    // fewer units than SMs (the projector's cross-attention: 16 heads x 256 queries against 4900 keys): every unit is cut
    // along the keys so that all SMs work, pieces merged as above
    p.full_rounds = 0;
    p.leftover = static_cast<int>(units);
    p.split = sms / p.leftover;
    if (p.split > p.n_kv_all / 2) p.split = p.n_kv_all / 2;
    p.n_cta = p.leftover * p.split;
  } else {
    p.n_cta = static_cast<int>(units);
    p.full_rounds = 1;
    p.leftover = 0;
    p.split = 1;
  }
  static const int tile_w = [] { const char* e = getenv("ARIA_ATTN_W"); return e ? atoi(e) : 80; }();
#define ARIA_A3(HD_, W_) \
  return causal ? launch_attn3<HD_, W_, true>(q, k, v, p, q_stride_b, q_stride_h, kv_stride_b, kv_stride_h, stream) \
                : launch_attn3<HD_, W_, false>(q, k, v, p, q_stride_b, q_stride_h, kv_stride_b, kv_stride_h, stream)
  if (hd == 80 && tile_w == 80) ARIA_A3(80, 80);
  if (hd == 80) ARIA_A3(80, 128);
  ARIA_A3(128, 128);
#undef ARIA_A3
}

// Causal self-attention forward that also returns lse (aria_attention_bwd's input): the v3 kernel with one unit per CTA,
// heaviest first, exactly as aria_attention_fwd runs causal launches that it does not route to the round-1 kernel.
extern "C" int aria_attention_fwd_lse(const void* q, const void* k, const void* v, void* out, float* lse, const uint8_t* key_mask,
                                      int32_t B, int32_t H, int32_t T, int64_t q_stride_b, int64_t q_stride_h, int64_t kv_stride_b,
                                      int64_t kv_stride_h, float scale, int32_t head_dim, int32_t causal, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (!causal || head_dim != 128) {
    fprintf(stderr, "aria_b200: attention forward with lse supports causal self-attention with head_dim 128 only\n");
    return ARIA_ERR_UNSUPPORTED;
  }
  ARIA_CHECK_ARG(q && k && v && out && lse);
  ARIA_CHECK_ARG(B > 0 && H > 0 && T > 0);
  ARIA_CHECK_ARG(q_stride_b % 8 == 0 && q_stride_h % 8 == 0 && kv_stride_b % 8 == 0 && kv_stride_h % 8 == 0);
  Attn3Params p{};
  p.B = B;
  p.H = H;
  p.Tq = T;
  p.Tk = T;
  p.out_hd = 128;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.key_mask = key_mask;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.lse = lse;
  p.n_q_pairs = (T + 2 * A3_BM - 1) / (2 * A3_BM);
  p.n_kv_all = (T + A3_BN - 1) / A3_BN;
  const int64_t units = static_cast<int64_t>(B) * H * p.n_q_pairs;
  ARIA_CHECK_ARG(units < (1ll << 31));
  p.units = static_cast<int>(units);
  p.n_cta = p.units;
  p.full_rounds = 1;
  p.leftover = 0;
  p.split = 1;
  return launch_attn3<128, 128, true, true>(q, k, v, p, q_stride_b, q_stride_h, kv_stride_b, kv_stride_h, stream);
}
