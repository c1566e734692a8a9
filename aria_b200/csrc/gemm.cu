// 1-CTA tcgen05 GEMM (M=128 x N=BN tiles): the HBM-bound regimes (few rows per expert, decode) and odd tile shapes.
// See gemm_common.cuh for the design notes; gemm2.cu holds the 2-CTA (cta_group::2, M=256) kernel used when the
// problem is large enough to be tensor-bound.
#include <stdlib.h>

#include "gemm_common.cuh"

namespace aria {

// pipeline depth: the classic 128-row A stage keeps the tuned depths; skinny-M stages fill ~200 KB (max 24)
constexpr int gemm_stages(int BN, int AM) {
  if (AM == 128) return (BN == 256) ? 4 : (BN >= 128 ? 6 : 8);
  const int s = (200 * 1024) / (AM * BK * 2 + BN * BK * 2);
  return s > 24 ? 24 : s;
}

// AM = rows of A staged per k-block (TMA box height).  128 in general; 32 for skinny-M (decode) GEMMs, where a 128-row A
// stage would be 75 % padding: the shared memory goes to more weight stages instead (bytes in flight are what bound a
// weight-streaming GEMM).  The MMA still reads 128 rows starting at the stage base; rows >= AM are whatever follows in
// shared memory and only reach accumulator lanes that the epilogue never stores.
template <int BN, bool B_MN, int EPI, int AM = 128>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB0,
            const __grid_constant__ CUtensorMap tmB1, const __grid_constant__ CUtensorMap tmB2, const GemmParams p) {
  constexpr int B_STAGE_BYTES = BN * BK * 2;
  constexpr int A_BYTES = AM * BK * 2;
  constexpr int STAGE_BYTES = A_BYTES + B_STAGE_BYTES;
  constexpr int STAGES = gemm_stages(BN, AM);
  constexpr int ACC_STRIDE = (BN <= 32) ? 32 : (BN <= 64) ? 64 : (BN <= 128) ? 128 : 256;  // TMEM columns per accumulator stage
  constexpr int TMEM_COLS = 2 * ACC_STRIDE;
  constexpr int OUT_BN = (EPI == ARIA_EPI_SWIGLU) ? BN / 2 : BN;  // output columns per tile
  static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "invalid UMMA N");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;  // [2]
  uint64_t* tempty_bar = tfull_bar + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB0);
    if (p.n_seg > 1 || EPI == ARIA_EPI_SWIGLU) prefetch_tmap(&tmB1);
    if (p.n_seg > 2) prefetch_tmap(&tmB2);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_out_total = p.N * (EPI == ARIA_EPI_SWIGLU ? 1 : p.n_seg);  // output columns overall
  const int n_tiles = (n_out_total + OUT_BN - 1) / OUT_BN;
  const int k_blocks = (p.K + BK - 1) / BK;

  // The two single-thread loops below are latency-bound instruction streams: every SASS instruction in them costs ~5-10
  // cycles of k-block time (measured with scripts/probes/mma_probe.cu: 0.32 us per k-block in the naive form, 0.12-0.15 us
  // when lean).  Hence: elect.sync guards (no vector->uniform register waterfalls), everything tile-invariant hoisted out of
  // the k loop, shared-memory addresses as running 32-bit values, descriptors as base + offset.
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (elect_one()) {
      TileSched sched;
      sched.init(p, n_tiles);
      uint32_t stage = 0, phase = 0;
      for (int t = blockIdx.x;; t += gridDim.x) {
        int grp, m_idx, n_idx, row0, rows;
        if (!sched.decode(t, grp, m_idx, n_idx, row0, rows)) break;
        const int a_row = row0 + m_idx * BM;
        const int bgrp = weight_block(p, grp);
        // B coordinates of this tile (k-invariant part)
        int b_c0 = 0, b_c1 = 0;          // K-major: row (n) coordinate of the two boxes; MN-major: base k row
        const CUtensorMap* tb0 = &tmB0;
        const CUtensorMap* tb1 = &tmB1;
        if constexpr (B_MN) {
          b_c0 = bgrp * p.K;
        } else if constexpr (EPI == ARIA_EPI_SWIGLU) {
          b_c0 = b_c1 = n_idx * OUT_BN;
        } else {
          const int col = n_idx * BN;
          const int seg = col / p.N;
          tb0 = seg == 0 ? &tmB0 : (seg == 1 ? &tmB1 : &tmB2);
          b_c0 = col - seg * p.N + bgrp * p.b_group_rows;
        }
        for (int kb = 0; kb < k_blocks; ++kb) {
          const uint32_t fb = full0 + stage * 8;
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint32_t sb = sa + A_BYTES;
          mbar_wait_addr(empty0 + stage * 8, phase ^ 1);
          mbar_arrive_expect_tx_addr(fb, STAGE_BYTES);
          tma_load_2d_addr(sa, &tmA, fb, kb * BK, a_row);
          if constexpr (B_MN) {
            // B = [G*K, Ncols] rows k, N contiguous; one box = 64 k-rows x 64 n (8 KB), BN/64 boxes per stage
            const int krow = b_c0 + kb * BK;
            constexpr int CH = BN / 64;
#pragma unroll
            for (int c = 0; c < CH; ++c) {
              int ncol;
              if constexpr (EPI == ARIA_EPI_SWIGLU) {
                constexpr int HALF = CH / 2;
                ncol = (c < HALF) ? (n_idx * OUT_BN + c * 64) : (p.N + n_idx * OUT_BN + (c - HALF) * 64);
              } else {
                ncol = n_idx * BN + c * 64;
              }
              tma_load_2d_addr(sb + c * (64 * BK * 2), &tmB0, fb, ncol, krow);
            }
          } else if constexpr (EPI == ARIA_EPI_SWIGLU) {
            tma_load_2d_addr(sb, tb0, fb, kb * BK, b_c0);
            tma_load_2d_addr(sb + (BN / 2) * BK * 2, tb1, fb, kb * BK, b_c1);
          } else {
            tma_load_2d_addr(sb, tb0, fb, kb * BK, b_c0);
          }
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, false, B_MN);
      const uint32_t b_lbo = p.dbg_lbo ? p.dbg_lbo : (B_MN ? 64 * BK * 2 : 16);
      const uint32_t b_sbo = p.dbg_sbo ? p.dbg_sbo : 1024;
      const uint32_t b_kadv = (p.dbg_kadv ? p.dbg_kadv : (B_MN ? 16 * 128 : 32)) >> 4;
      // descriptors of stage 0 / k-step 0; the start-address field is (addr >> 4) in the low 14 bits and shared-memory
      // addresses stay below 2^18, so adding (byte offset >> 4) never carries into the next field
      const uint64_t da0 = make_smem_desc(smem_base, 16, 1024);
      const uint64_t db0 = make_smem_desc(smem_base + A_BYTES, b_lbo, b_sbo);
      const uint32_t tfull0 = smem_u32(tfull_bar), tempty0 = smem_u32(tempty_bar);
      TileSched sched;
      sched.init(p, n_tiles);
      uint32_t stage = 0, phase = 0;
      int it = 0;
      for (int t = blockIdx.x;; t += gridDim.x, ++it) {
        int grp, m_idx, n_idx, row0, rows;
        if (!sched.decode(t, grp, m_idx, n_idx, row0, rows)) break;
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait_addr(tempty0 + as * 8, aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * ACC_STRIDE;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait_addr(full0 + stage * 8, phase);
          tc_fence_after();
          const uint64_t da = da0 + stage * (STAGE_BYTES >> 4);
          const uint64_t db = db0 + stage * (STAGE_BYTES >> 4);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) umma_bf16_ss(d_tmem, da + k * 2, db + k * b_kadv, idesc, (kb | k) ? 1u : 0u);
          umma_commit_addr(empty0 + stage * 8);  // frees the smem slot once these MMAs have read it
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_addr(tfull0 + as * 8);  // accumulator complete -> epilogue
      }
    }
  } else {
    // =========================== epilogue (warps 2..9) ===========================
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int r_in_tile = quad * 32 + lane;
    TileSched sched;
    sched.init(p, n_tiles);
    int it = 0;
    for (int t = blockIdx.x;; t += gridDim.x, ++it) {
      int grp, m_idx, n_idx, row0, rows;
      if (!sched.decode(t, grp, m_idx, n_idx, row0, rows)) break;
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + as * ACC_STRIDE + (static_cast<uint32_t>(quad * 32) << 16);
      const int r_in_grp = m_idx * BM + r_in_tile;
      const bool row_ok = r_in_grp < rows;
      const int64_t grow = static_cast<int64_t>(row0) + r_in_grp;

      epilogue_tile<BN, EPI>(p, taddr, n_out_total, n_idx, grow, row_ok, (warp - 2) >> 2, grp, r_in_grp);
      // release this accumulator stage back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
  (void)ACC_STRIDE;
}

template <int BN, bool B_MN, int EPI, int AM = 128>
static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap* tmB, const GemmParams& p, int max_tiles,
                       cudaStream_t stream) {
  constexpr int B_STAGE_BYTES = BN * BK * 2;
  constexpr int STAGES = gemm_stages(BN, AM);
  // + (128-AM) rows of slack: the M=128 MMA of the last stage reads 16 KB from a stage base whose A part is only AM rows
  constexpr int SMEM = STAGES * (AM * BK * 2 + B_STAGE_BYTES) + 1024 /*align*/ + 512 /*barriers*/ + (BM - AM) * BK * 2;
  auto kern = gemm_kernel<BN, B_MN, EPI, AM>;
  static bool attr_set[kMaxDevices] = {};
  if (ensure_dynamic_smem(attr_set, kern, SMEM) != cudaSuccess) return ARIA_ERR_CUDA;
  int grid = sm_count();
  if (max_tiles < grid) grid = max_tiles;
  if (grid < 1) grid = 1;
  kern<<<grid, GEMM_THREADS, SMEM, stream>>>(tmA, tmB[0], tmB[1], tmB[2], p);
  return check_launch("gemm_kernel");
}

}  // namespace aria

namespace aria {
int launch_gemm2_dispatch(int bn, bool b_mn, int epi, const CUtensorMap& tmA, const CUtensorMap* tmB, const GemmParams& p,
                          int max_tiles, cudaStream_t stream);  // gemm2.cu
}

using namespace aria;

namespace aria {
// aria_gemm with the epilogue given separately: `epi` may also be one of the internal modes of gemm_common.cuh (lm_loss.cu),
// whose arguments come in `xp`.  Those run dense, single-segment GEMMs on 128-row A stages.
int gemm_run(const aria_gemm_desc_t* d, int epi, const XentParams* xp, cudaStream_t stream) {
  ARIA_CHECK_ARG(d != nullptr);
  const bool xent = epi >= EPI_XENT_STATS;
  if (xent) ARIA_CHECK_ARG(xp != nullptr && d->n_seg == 1 && d->num_groups == 1 && d->residual == nullptr);
  ARIA_CHECK_ARG(d->a && d->b[0] && d->out[0]);
  ARIA_CHECK_ARG(d->m >= 0 && d->n > 0 && d->k > 0);
  ARIA_CHECK_ARG(d->n % 8 == 0 && d->k % 8 == 0 && d->lda % 8 == 0);
  ARIA_CHECK_ARG(d->n_seg >= 1 && d->n_seg <= 3);
  ARIA_CHECK_ARG(d->num_groups >= 1 && (d->group_mod >= 0 || d->num_groups % (-d->group_mod) == 0));
  ARIA_CHECK_ARG((reinterpret_cast<uintptr_t>(d->a) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->out[0]) & 15) == 0);
  if (d->m == 0) return ARIA_OK;
  const bool b_mn = d->b_layout == ARIA_B_GKN;
  const bool b_gnk = d->b_layout == ARIA_B_GNK;
  const bool swiglu = epi == ARIA_EPI_SWIGLU;
  if (b_mn) {
    ARIA_CHECK_ARG(d->n_seg == 1);
    // k-blocks must not straddle experts in the flattened [G*K, N] view (a single group has no neighbour: TMA zero-fills)
    ARIA_CHECK_ARG(d->k % BK == 0 || (d->num_groups == 1 && d->group_mod == 0));
    ARIA_CHECK_ARG(d->n % 64 == 0);
    ARIA_CHECK_ARG(epi != ARIA_EPI_HEADS);
  } else {
    ARIA_CHECK_ARG(d->num_groups == 1 || d->n_seg == 1);
    if (swiglu) ARIA_CHECK_ARG(d->n_seg == 2 && d->b[1]);
    if (b_gnk) ARIA_CHECK_ARG(d->n_seg == 1 && !swiglu && epi == ARIA_EPI_LINEAR && d->n % 128 == 0);
    else ARIA_CHECK_ARG(d->num_groups == 1);
  }
  if (d->num_groups > 1) ARIA_CHECK_ARG(d->group_offsets != nullptr);
  if (d->group_counts) ARIA_CHECK_ARG(d->group_offsets != nullptr);
  if (xent) ARIA_CHECK_ARG(epi == EPI_ACC_F32 ? b_mn : !b_mn && !b_gnk);
  if (d->out_group_base) ARIA_CHECK_ARG(d->out_group_row0 != nullptr && epi == ARIA_EPI_LINEAR && d->group_offsets != nullptr);
  ARIA_CHECK_ARG(d->a_rows == 0 || d->a_rows >= d->m);

  GemmParams p{};
  p.M = static_cast<int>(d->m);
  p.N = static_cast<int>(d->n);
  p.K = static_cast<int>(d->k);
  p.num_groups = d->num_groups;
  p.group_offsets = d->group_offsets;
  p.group_counts = d->group_counts;
  p.out_group_base = static_cast<const uint64_t*>(d->out_group_base);
  p.out_group_row0 = d->out_group_row0;
  p.group_mod = d->group_mod;
  p.pair = 0;
  p.b_group_rows = b_gnk ? static_cast<int>(d->n) : 0;
  p.n_seg = swiglu ? 1 : d->n_seg;
  p.act = d->act;
  for (int i = 0; i < 3; ++i) {
    p.bias[i] = static_cast<const __nv_bfloat16*>(d->bias[i]);
    p.out[i] = static_cast<__nv_bfloat16*>(d->out[i]);
  }
  p.residual = static_cast<const __nv_bfloat16*>(d->residual);
  p.ldr = d->ldr;
  p.ldo = d->ldo;
  p.head_dim = d->head_dim;
  p.head_ld = d->head_ld;
  p.rows_per_batch = d->rows_per_batch > 0 ? d->rows_per_batch : static_cast<int>(d->m);
  p.pos0 = d->pos0;
  p.stride_b = d->stride_b;
  p.stride_h = d->stride_h;
  p.rope_mask = d->rope_mask;
  p.rope_cos = static_cast<const __nv_bfloat16*>(d->rope_cos);
  p.rope_sin = static_cast<const __nv_bfloat16*>(d->rope_sin);
  p.position_ids = d->position_ids;
  p.dbg_lbo = d->dbg_lbo;
  p.dbg_sbo = d->dbg_sbo;
  p.dbg_kadv = d->dbg_kadv;
  if (xent) p.x = *xp;

  // ---- kernel / tile shape selection
  // 2-CTA pairs (M=256 tiles, gemm2.cu) whenever there are at least two 128-row tiles of work per group; the 1-CTA
  // kernel keeps the HBM-bound regimes (a few rows per expert, decode, lm_head on one row) and the 144-wide ViT tile.
  const int64_t n_out_total = d->n * (swiglu ? 1 : d->n_seg);
  bool two_cta = (d->num_groups == 1) ? (d->m > BM) : (d->m / d->num_groups >= 192);
  {  // bring-up / A-B switch: ARIA_GEMM_CTAS=1 forces the 1-CTA kernel, =2 the 2-CTA kernel where legal
    static int force = -1;
    if (force < 0) {
      const char* ev = getenv("ARIA_GEMM_CTAS");
      force = ev ? atoi(ev) : 0;
    }
    if (force == 1) two_cta = false;
    if (force == 2) two_cta = d->m > BM;
  }
  int BN;
  if (epi == ARIA_EPI_HEADS) {
    ARIA_CHECK_ARG(d->head_dim > 0 && d->head_dim % 8 == 0 && d->head_ld >= d->head_dim && d->n % d->head_dim == 0);
    if (d->rope_mask) ARIA_CHECK_ARG(d->head_dim == 128 && d->rope_cos && d->rope_sin);
    if (d->n % 128 == 0) {
      BN = 128;
    } else {
      ARIA_CHECK_ARG(!d->rope_mask && d->n % 144 == 0);
      BN = 144;
      two_cta = false;
    }
    for (int s = 0; s < d->n_seg; ++s) ARIA_CHECK_ARG(d->out[s] && d->b[s]);
  } else {
    BN = 128;
    if (swiglu) ARIA_CHECK_ARG(d->n % 64 == 0);
    if (d->n_seg > 1 && !swiglu) ARIA_CHECK_ARG(d->n % BN == 0);
  }
  if (two_cta && BN == 128) {
    // 2-CTA pays off with 256 x 256 tiles (twice the flops per byte pulled from L2, measured 1.28-1.38 PFLOP/s vs
    // 0.84 for 128 x 128); with too few such tiles (< ~1.3 waves of CTA pairs) the 1-CTA kernel fills the SMs better.
    const int64_t out_bn256 = swiglu ? 128 : 256;
    const bool divisible = swiglu ? (d->n % 128 == 0) : ((d->n_seg == 1 && !b_gnk) || d->n % 256 == 0);
    const int64_t m_tiles256 = (d->num_groups == 1) ? (d->m + 255) / 256 : (d->m / 256 + d->num_groups / 2);
    const int64_t tiles256 = m_tiles256 * ((n_out_total + out_bn256 - 1) / out_bn256);
    static const int mid = [] { const char* e = getenv("ARIA_GEMM_MID"); return e ? atoi(e) : 1; }();
    // short-K dense GEMMs whose 256 x 256 tiles fill the last round badly run better as 128 x 128 tiles: ViT o_proj
    // (4900 x 1152 x 1152: 100 pair tiles on 74 pairs = 0.68 of two rounds) 27.4 us on pairs, 23.3 us on single CTAs; with a long K
    // (ViT fc2, K = 4304, same tile count) the pair kernel stays ahead (57.9 vs 66.7 us).  profiles/r02_gemm_notes.txt
    const int64_t pairs = sm_count() / 2;
    const double fill2 = static_cast<double>(tiles256) / static_cast<double>((tiles256 + pairs - 1) / pairs * pairs);
    const bool poor_fill = d->num_groups == 1 && d->k <= 2048 && fill2 < 0.75;
    if (divisible && tiles256 * 10 >= 13 * pairs && !poor_fill) {
      BN = 256;
    } else if (mid && d->num_groups == 1 && d->m >= 256 && d->m <= 1024) {
      // mid-size dense GEMM (the T=768 LM projections): 256 x 128 pair tiles pull 24 KB per CTA per k-block from L2 instead of
      // 32 KB: qkv+RoPE 37.4 -> 33.7 us, shared gate|up 32.8 -> 29.2, o_proj 19.7 -> 19.2, down 19.0 -> 18.2 (ARIA_GEMM_MID=0 disables)
    } else {
      two_cta = false;
    }
  }

  // Expert-parallel regions ordered (expert, source rank) with an even number of source ranks: CTA pairs over neighbouring regions
  // (gemm2.cu pair mode).  OPT-IN (ARIA_GEMM_PAIR=1, read per call): isolated it is 11 % faster than the 1-CTA kernel (134 -> 120 us,
  // half the weight bytes per SM), inside the 2-GPU step it measured 5 % slower (profiles/r02_gemm_notes.txt), so the default stays.
  {
    const char* pe = getenv("ARIA_GEMM_PAIR");
    const bool pair_on = pe && pe[0] == '1';
    const bool ok = swiglu ? (d->n % 128 == 0) : (d->n % 256 == 0);
    if (pair_on && d->group_counts && d->group_mod < 0 && (-d->group_mod) % 2 == 0 && b_mn && ok && epi != ARIA_EPI_HEADS) {
      two_cta = true;
      BN = 256;
      p.pair = 1;
    }
  }

  // HBM-bound grouped regime on the 1-CTA kernel (few rows per expert): 128 x 256 tiles halve the A-tile share of the
  // L2 -> SM traffic per streamed weight byte (env ARIA_GEMM_WIDE=0 disables, for A/B measurements)
  if (!two_cta && b_mn && d->num_groups > 1 && BN == 128) {
    static int wide = -1;
    if (wide < 0) {
      const char* ev = getenv("ARIA_GEMM_WIDE");
      wide = ev ? atoi(ev) : 1;
    }
    const bool ok = swiglu ? (d->n % 128 == 0) : (d->n % 256 == 0);
    if (wide && ok) BN = 256;
  }

  // Skinny-M dense GEMMs (decode: m <= 32): 32-row A stages, narrow tiles so that ~80+ CTAs stream weights with many
  // stages each (bytes in flight bound a weight-streaming GEMM); very wide N (lm_head) keeps 128-column tiles.
  int AM = 128;
  static const bool skinny_on = [] { const char* e = getenv("ARIA_GEMM_SKINNY"); return !(e && e[0] == '0'); }();
  if (skinny_on && !xent && !two_cta && !b_mn && d->num_groups == 1 && d->m <= 32 && BN == 128) {
    AM = 32;
    if (epi == ARIA_EPI_LINEAR && d->n_seg == 1 && d->n % 32 == 0 && d->n < 16384) BN = 32;
    if (swiglu && d->n % 32 == 0) BN = 64;
  }

  CUtensorMap tmA, tmB[3];
  // a_rows: rows of the A buffer when groups live in fixed-capacity regions (m is then the EXPECTED row count that the
  // kernel-selection heuristics above use; the tensor map must cover the whole buffer)
  int rc = make_tmap_2d(&tmA, d->a, d->k, d->a_rows > 0 ? d->a_rows : d->m, d->lda * 2, BK, AM);
  if (rc) return rc;
  if (b_mn) {
    const uint64_t ncols = swiglu ? 2 * d->n : d->n;
    const uint64_t n_weights = d->group_mod > 0 ? d->group_mod : (d->group_mod < 0 ? d->num_groups / (-d->group_mod) : d->num_groups);
    rc = make_tmap_2d(&tmB[0], d->b[0], ncols, n_weights * d->k, ncols * 2, 64, BK);
    if (rc) return rc;
    tmB[1] = tmB[0];
    tmB[2] = tmB[0];
  } else {
    const int nb = swiglu ? 2 : d->n_seg;
    // rows of B staged per TMA box: the whole tile (1-CTA), half of it per CTA (2-CTA); SwiGLU splits gate | up
    uint32_t box_rows = swiglu ? BN / 2 : BN;
    if (two_cta && !swiglu) box_rows = BN / 2;
    for (int s = 0; s < 3; ++s) {
      const void* ptr = s < nb ? d->b[s] : d->b[0];
      const uint64_t b_rows = b_gnk ? static_cast<uint64_t>(d->group_mod > 0 ? d->group_mod : (d->group_mod < 0 ? d->num_groups / (-d->group_mod) : d->num_groups)) * d->n : d->n;
      rc = make_tmap_2d(&tmB[s], ptr, d->k, b_rows, d->k * 2, BK, box_rows);
      if (rc) return rc;
    }
  }

  const int out_bn = swiglu ? BN / 2 : BN;
  const int64_t n_tiles = (n_out_total + out_bn - 1) / out_bn;
  const int bm = two_cta ? 2 * BM : BM;
  const int64_t m_tiles_ub = p.pair ? (d->m + BM - 1) / BM + d->num_groups / 2
                                    : (d->m + bm - 1) / bm + (d->num_groups > 1 ? d->num_groups : 0);
  int64_t max_tiles = n_tiles * m_tiles_ub;
  if (max_tiles > (1 << 30)) max_tiles = 1 << 30;

  if (two_cta)
    return launch_gemm2_dispatch(BN, b_mn, epi, tmA, tmB, p, static_cast<int>(max_tiles), stream);

#define ARIA_LAUNCH(BN_, MN_, EPI_) return launch_gemm<BN_, MN_, EPI_>(tmA, tmB, p, static_cast<int>(max_tiles), stream)
  if (AM == 32) {
    if (epi == ARIA_EPI_HEADS) return launch_gemm<128, false, ARIA_EPI_HEADS, 32>(tmA, tmB, p, static_cast<int>(max_tiles), stream);
    if (swiglu) {
      if (BN == 64) return launch_gemm<64, false, ARIA_EPI_SWIGLU, 32>(tmA, tmB, p, static_cast<int>(max_tiles), stream);
      return launch_gemm<128, false, ARIA_EPI_SWIGLU, 32>(tmA, tmB, p, static_cast<int>(max_tiles), stream);
    }
    if (BN == 32) return launch_gemm<32, false, ARIA_EPI_LINEAR, 32>(tmA, tmB, p, static_cast<int>(max_tiles), stream);
    return launch_gemm<128, false, ARIA_EPI_LINEAR, 32>(tmA, tmB, p, static_cast<int>(max_tiles), stream);
  }
  if (epi == ARIA_EPI_HEADS) {
    if (BN == 128) ARIA_LAUNCH(128, false, ARIA_EPI_HEADS);
    ARIA_LAUNCH(144, false, ARIA_EPI_HEADS);
  }
  if (swiglu) {
    if (b_mn && BN == 256) ARIA_LAUNCH(256, true, ARIA_EPI_SWIGLU);
    if (b_mn) ARIA_LAUNCH(128, true, ARIA_EPI_SWIGLU);
    ARIA_LAUNCH(128, false, ARIA_EPI_SWIGLU);
  }
  if (xent) {  // BN = 128 here: the 256-wide tiles only run on CTA pairs
    if (epi == EPI_XENT_STATS) ARIA_LAUNCH(128, false, EPI_XENT_STATS);
    if (epi == EPI_XENT_GRAD) ARIA_LAUNCH(128, false, EPI_XENT_GRAD);
    ARIA_LAUNCH(128, true, EPI_ACC_F32);
  }
  if (b_mn && BN == 256) ARIA_LAUNCH(256, true, ARIA_EPI_LINEAR);
  if (b_mn) ARIA_LAUNCH(128, true, ARIA_EPI_LINEAR);
  ARIA_LAUNCH(128, false, ARIA_EPI_LINEAR);
#undef ARIA_LAUNCH
}
}  // namespace aria

extern "C" int aria_gemm(const aria_gemm_desc_t* d, aria_stream_t stream) {
  ARIA_CHECK_ARG(d != nullptr);
  ARIA_CHECK_ARG(d->epilogue == ARIA_EPI_LINEAR || d->epilogue == ARIA_EPI_SWIGLU || d->epilogue == ARIA_EPI_HEADS);
  return gemm_run(d, d->epilogue, nullptr, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int aria_grouped_gemm(const void* a, const void* b, void* out, const int32_t* group_offsets, int64_t rows,
                                 int64_t k, int64_t n, int32_t num_groups, aria_stream_t stream) {
  aria_gemm_desc_t d{};
  d.a = a;
  d.lda = k;
  d.m = rows;
  d.n = n;
  d.k = k;
  d.b[0] = b;
  d.n_seg = 1;
  d.b_layout = ARIA_B_GKN;
  d.num_groups = num_groups;
  d.group_offsets = group_offsets;
  d.epilogue = ARIA_EPI_LINEAR;
  d.out[0] = out;
  d.ldo = n;
  return aria_gemm(&d, stream);
}

extern "C" int aria_abi_version(void) { return 2; }
extern "C" const char* aria_build_arch(void) { return "sm_100a"; }
