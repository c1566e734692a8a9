// 2-CTA tcgen05 GEMM: a CTA pair (thread-block cluster of 2 on one TPC) computes a 256 x BN output tile with
// tcgen05.mma.cta_group::2 (UMMA M=256).  Each CTA stages its own 128 rows of A and HALF of the B tile in shared
// memory, so per-SM shared-memory traffic per MMA is halved compared with the 1-CTA kernel — the 1-CTA M=128 x N=128
// SS-mode MMA needs 128 B/clk of operand reads, all the shared memory has, which is why gemm.cu tops out near half
// the tensor peak — and each CTA holds its 128 accumulator rows in its own TMEM.
//
//   rank 0 (leader): TMA producer, MMA issuer (for both CTAs), epilogue of rows [0,128)
//   rank 1         : TMA producer (completion bytes credited to the leader's mbarrier), epilogue of rows [128,256)
//   smem full[]    : leader only, expect_tx = bytes of BOTH CTAs' loads
//   smem empty[]   : one per CTA, released by a multicast tcgen05.commit
//   tmem full[]    : one per CTA (multicast commit); tmem empty[]: leader only, 8 arrivals (4 epilogue warps x 2 CTAs)
//
// Pair mode (GemmParams::pair, expert parallelism): the rows live in fixed-capacity regions ordered (expert, source rank); the two
// CTAs of a pair take 128 rows each from two NEIGHBOURING regions of the same expert, so one weight tile (half staged per CTA) serves
// both source ranks' rows: half the weight bytes per SM of the 1-CTA kernel, which re-pulled the tile for every region
// (profiles/r02_gemm_notes.txt).
#include "gemm_common.cuh"

namespace aria {

constexpr int BM2 = 256;

template <int BN, bool B_MN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB0,
             const __grid_constant__ CUtensorMap tmB1, const __grid_constant__ CUtensorMap tmB2, const GemmParams p) {
  static_assert(BN == 128 || BN == 256, "2-CTA tiles are 256x128 or 256x256");
  constexpr int BH = BN / 2;                       // B rows (K-major) / columns (MN-major) staged per CTA
  constexpr int B_STAGE_BYTES = BH * BK * 2;
  constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  constexpr int STAGES = (BN == 256) ? 6 : 8;
  constexpr int ACC_STRIDE = BN;                   // TMEM columns per accumulator stage (128 lanes per CTA)
  constexpr int TMEM_COLS = 2 * ACC_STRIDE;
  constexpr int OUT_BN = (EPI == ARIA_EPI_SWIGLU) ? BN / 2 : BN;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;  // [2]
  uint64_t* tempty_bar = tfull_bar + 2;      // [2] (leader's copy is the live one)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1;
  const int n_clusters = gridDim.x >> 1;

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
      mbar_init(&tempty_bar[i], 2 * EPI_WARPS);
    }
    fence_mbar_init();
  }
  __syncthreads();
  cluster_sync_all();  // peer barriers are initialised before any remote arrive / multicast
  if (warp == 1) {
    tmem_alloc_2sm(tmem_slot, TMEM_COLS);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_out_total = p.N * (EPI == ARIA_EPI_SWIGLU ? 1 : p.n_seg);
  const int n_tiles = (n_out_total + OUT_BN - 1) / OUT_BN;
  const int k_blocks = (p.K + BK - 1) / BK;

  // Lean single-thread issue loops (see gemm.cu): tile-invariant math hoisted, 32-bit shared addresses, base descriptors.
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
  if (warp == 0) {
    // =========================== TMA producer (both CTAs) ===========================
    if (elect_one()) {
      TileSched sched;
      sched.init(p, n_tiles, BM2);
      uint32_t stage = 0, phase = 0;
      const uint32_t leader_full0 = full0 & 0xFEFFFFFFu;  // completion bytes are credited to the leader CTA's barrier
      for (int t = cluster_id;; t += n_clusters) {
        int grp, m_idx, n_idx, row0, rows;
        if (!sched.decode(t, grp, m_idx, n_idx, row0, rows)) break;
        // pair mode: this CTA's 128 rows come from ITS region of the super-group; both regions multiply the same expert's weights
        const int a_row = p.pair ? p.group_offsets[2 * grp + static_cast<int>(rank)] + m_idx * BM
                                 : row0 + m_idx * BM2 + static_cast<int>(rank) * BM;
        const int bgrp = weight_block(p, p.pair ? 2 * grp : grp);
        int b_c = 0;
        const CUtensorMap* tb = &tmB0;
        if constexpr (B_MN) {
          b_c = bgrp * p.K;
        } else if constexpr (EPI == ARIA_EPI_SWIGLU) {
          tb = rank == 0 ? &tmB0 : &tmB1;
          b_c = n_idx * OUT_BN;
        } else {
          const int col = n_idx * BN;
          const int seg = col / p.N;
          tb = seg == 0 ? &tmB0 : (seg == 1 ? &tmB1 : &tmB2);
          b_c = col - seg * p.N + static_cast<int>(rank) * BH + bgrp * p.b_group_rows;
        }
        for (int kb = 0; kb < k_blocks; ++kb) {
          const uint32_t fb = leader_full0 + stage * 8;
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint32_t sb = sa + A_STAGE_BYTES;
          mbar_wait_addr(empty0 + stage * 8, phase ^ 1);
          if (rank == 0) mbar_arrive_expect_tx_addr(full0 + stage * 8, 2 * STAGE_BYTES);
          tma_load_2d_2sm_addr(sa, &tmA, fb, kb * BK, a_row);
          if constexpr (B_MN) {
            // B = [G*K, Ncols], N contiguous.  This CTA stages N-columns [rank*BH, +BH) of the tile.
            const int krow = b_c + kb * BK;
            constexpr int CH = BH / 64;
#pragma unroll
            for (int c = 0; c < CH; ++c) {
              int ncol;
              if constexpr (EPI == ARIA_EPI_SWIGLU) {
                // rank 0 holds the gate columns, rank 1 the up columns (gate|up = first|second half of the 2I cols)
                ncol = static_cast<int>(rank) * p.N + n_idx * OUT_BN + c * 64;
              } else {
                ncol = n_idx * BN + static_cast<int>(rank) * BH + c * 64;
              }
              tma_load_2d_2sm_addr(sb + c * (64 * BK * 2), &tmB0, fb, ncol, krow);
            }
          } else {
            tma_load_2d_2sm_addr(sb, tb, fb, kb * BK, b_c);
          }
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (leader CTA only) ===========================
    if (rank == 0 && elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(BM2, BN, false, B_MN);
      constexpr uint32_t b_lbo = B_MN ? 64 * BK * 2 : 16;
      constexpr uint32_t b_kadv = (B_MN ? 16 * 128 : 32) >> 4;
      const uint64_t da0 = make_smem_desc(smem_base, 16, 1024);
      const uint64_t db0 = make_smem_desc(smem_base + A_STAGE_BYTES, b_lbo, 1024);
      const uint32_t tfull0 = smem_u32(tfull_bar), tempty0 = smem_u32(tempty_bar);
      TileSched sched;
      sched.init(p, n_tiles, BM2);
      uint32_t stage = 0, phase = 0;
      int it = 0;
      for (int t = cluster_id;; t += n_clusters, ++it) {
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
          for (int k = 0; k < BK / 16; ++k) umma_bf16_ss_2sm(d_tmem, da + k * 2, db + k * b_kadv, idesc, (kb | k) ? 1u : 0u);
          umma_commit_2sm_addr(empty0 + stage * 8);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_2sm_addr(tfull0 + as * 8);
      }
    }
  } else {
    // =========================== epilogue (warps 2..9 of both CTAs) ===========================
    const int quad = warp & 3;
    const int r_in_tile = static_cast<int>(rank) * BM + quad * 32 + lane;
    const uint32_t leader_tempty0 = mapa_shared(smem_u32(&tempty_bar[0]), 0);
    TileSched sched;
    sched.init(p, n_tiles, BM2);
    int it = 0;
    for (int t = cluster_id;; t += n_clusters, ++it) {
      int grp, m_idx, n_idx, row0, rows;
      if (!sched.decode(t, grp, m_idx, n_idx, row0, rows)) break;
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + as * ACC_STRIDE + (static_cast<uint32_t>(quad * 32) << 16);
      int r_in_grp = m_idx * BM2 + r_in_tile;
      int my_grp = grp;
      if (p.pair) {  // rows of this CTA = rows [m_idx * 128, +128) of region 2 grp + rank
        my_grp = 2 * grp + static_cast<int>(rank);
        r_in_grp = m_idx * BM + quad * 32 + lane;
        row0 = p.group_offsets[my_grp];
        rows = p.group_counts[my_grp];
      }
      const bool row_ok = r_in_grp < rows;
      const int64_t grow = static_cast<int64_t>(row0) + r_in_grp;
      epilogue_tile<BN, EPI>(p, taddr, n_out_total, n_idx, grow, row_ok, (warp - 2) >> 2, my_grp, r_in_grp);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(leader_tempty0 + as * 8);
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // both CTAs are done with each other's shared memory / barriers / TMEM pairing
  if (warp == 1) tmem_dealloc_2sm(tmem_base, TMEM_COLS);
}

template <int BN, bool B_MN, int EPI>
static int launch_gemm2(const CUtensorMap& tmA, const CUtensorMap* tmB, const GemmParams& p, int max_tiles, cudaStream_t stream) {
  constexpr int BH = BN / 2;
  constexpr int STAGES = (BN == 256) ? 6 : 8;
  constexpr int SMEM = STAGES * (A_STAGE_BYTES + BH * BK * 2) + 1024 + 256;
  auto kern = gemm2_kernel<BN, B_MN, EPI>;
  static bool attr_set[kMaxDevices] = {};
  if (ensure_dynamic_smem(attr_set, kern, SMEM) != cudaSuccess) return ARIA_ERR_CUDA;
  int clusters = sm_count() / 2;
  if (max_tiles < clusters) clusters = max_tiles;
  if (clusters < 1) clusters = 1;
  kern<<<clusters * 2, GEMM_THREADS, SMEM, stream>>>(tmA, tmB[0], tmB[1], tmB[2], p);
  return check_launch("gemm2_kernel");
}

// Entry used by aria_gemm (gemm.cu).  bn = 128 or 256.
int launch_gemm2_dispatch(int bn, bool b_mn, int epi, const CUtensorMap& tmA, const CUtensorMap* tmB, const GemmParams& p,
                          int max_tiles, cudaStream_t stream) {
#define G2(BN_, MN_, EPI_) return launch_gemm2<BN_, MN_, EPI_>(tmA, tmB, p, max_tiles, stream)
  if (epi == EPI_XENT_STATS) { if (bn == 256) G2(256, false, EPI_XENT_STATS); G2(128, false, EPI_XENT_STATS); }
  if (epi == EPI_XENT_GRAD) { if (bn == 256) G2(256, false, EPI_XENT_GRAD); G2(128, false, EPI_XENT_GRAD); }
  if (epi == EPI_ACC_F32) { if (bn == 256) G2(256, true, EPI_ACC_F32); G2(128, true, EPI_ACC_F32); }
  if (epi == ARIA_EPI_SWIGLU) {
    if (bn == 256) { if (b_mn) G2(256, true, ARIA_EPI_SWIGLU); G2(256, false, ARIA_EPI_SWIGLU); }
    if (b_mn) G2(128, true, ARIA_EPI_SWIGLU);
    G2(128, false, ARIA_EPI_SWIGLU);
  }
  if (epi == ARIA_EPI_HEADS) {
    if (bn == 256) G2(256, false, ARIA_EPI_HEADS);
    G2(128, false, ARIA_EPI_HEADS);
  }
  if (bn == 256) { if (b_mn) G2(256, true, ARIA_EPI_LINEAR); G2(256, false, ARIA_EPI_LINEAR); }
  if (b_mn) G2(128, true, ARIA_EPI_LINEAR);
  G2(128, false, ARIA_EPI_LINEAR);
#undef G2
}

}  // namespace aria
