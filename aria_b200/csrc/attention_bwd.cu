// Causal attention backward (head_dim 128) on tcgen05 — the autograd of the LM attention (attention_v3.cu's causal path).
//
// FlashAttention-2's split into three launches, each deterministic (every output element is written by exactly one CTA, no
// float atomics):
//   attn_bwd_pre_kernel   Delta = rowsum(dO o O) in fp32, one warp per (token, head) row;
//   attn_bwd_dkdv_kernel  one CTA per (b, h, 128-key block), looping over the query blocks at or after the diagonal:
//                           S^T = K Q^T, dP^T = V dO^T          (SS: both operands K-major in shared memory)
//                           P^T = exp2(S^T * scale*log2e - lse), dS^T = P^T o (dP^T - Delta)   (a thread owns a key row)
//                           dV += P^T dO, dK += dS^T Q           (TS: P^T / dS^T read back from TMEM as bf16, dO / Q MN-major)
//   attn_bwd_dq_kernel    one CTA per (b, h, 128-query block), looping over the key blocks up to the diagonal:
//                           S = Q K^T, dP = dO V^T, dS as above (a thread owns a query row), dQ += dS K (TS, K MN-major).
// The dQ kernel recomputes S and dP (two GEMMs more than the atomic FA2 variant, 7 instead of 5): in exchange dQ needs no fp32
// scratch of [B, H, T, 128] and no atomics, and the result is bit-reproducible run to run.  Both loops are a serial chain
// (MMA -> softmax-gradient warps -> MMA): the TMEM budget is spent on the four 128-column accumulators of the dK/dV kernel
// (S^T, dP^T, dV, dK = 512 columns), which leaves no room to double-buffer S; the operand tiles of the next block are
// prefetched by TMA while the current one is computed.
//
// lse comes from aria_attention_fwd_lse: m + log2(l) in the log2 domain of scale*log2e*s, +INF for a row without a visible key,
// so exp2(x - lse) is exactly 0 there.  Masked keys, the causal upper triangle of diagonal blocks and rows past T give P = 0.
// `scale` is folded into dK and dQ in their epilogues.
#include "common.cuh"
#include "ptx.cuh"

namespace aria {

constexpr int AB_BLK = 128;               // rows of every tile (keys or queries) = head dim
constexpr int AB_CH = AB_BLK * 128;       // 16 KB: one SW128 chunk [128 rows][64 bf16]
constexpr int AB_TILE = 2 * AB_CH;        // 32 KB: a 128 x 128 bf16 tile as two 64-column chunks
constexpr int AB_THREADS = 192;           // warps 0-3: softmax gradient (TMEM lanes 0-127); warp 4: TMA; warp 5: TMEM owner + MMA issuer
constexpr int AB_SMEM = 6 * AB_TILE + 2048 + 128 + 1024;  // 2 resident tiles + 2 stages x 2 tiles, lse / Delta staging, barriers, alignment

struct AttnBwdParams {
  int B, H, T, n_blk;
  float scale, scale_log2;
  const uint8_t* key_mask;  // [B, T], 1 = masked out
  const float* lse;         // [B, H, T]
  const float* delta;       // [B, H, T]
  __nv_bfloat16 *dq, *dk, *dv;  // [B, T, H*128]
};

ARIA_DEVICE void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// a 128 x 128 tile from a head-major [B, H, T, 128] tensor map (coordinates: column, token, head, batch)
ARIA_DEVICE void load_tile_hm(uint8_t* dst, const CUtensorMap* m, uint64_t* bar, int t0, int h, int b) {
  tma_load_4d(dst, m, bar, 0, t0, h, b);
  tma_load_4d(dst + AB_CH, m, bar, 64, t0, h, b);
}
// ... from a token-major [B, T, H*128] tensor map (coordinates: column, head, token, batch)
ARIA_DEVICE void load_tile_tm(uint8_t* dst, const CUtensorMap* m, uint64_t* bar, int t0, int h, int b) {
  tma_load_4d(dst, m, bar, 0, h, t0, b);
  tma_load_4d(dst + AB_CH, m, bar, 64, h, t0, b);
}
// k-th 16-wide step of a tile used K-major (K = head dim): two SW128 chunks, +32 B per step inside a chunk
ARIA_DEVICE uint64_t kmajor_desc(uint32_t tile, int k) {
  return make_smem_desc_sw(tile + (k >> 2) * AB_CH, 16, 1024, UMMA_SW128) + (k & 3) * 2;
}
// the same tile used MN-major (K = its 128 rows, N = head dim): LBO = chunk stride, +16 rows = +2 KB per step
ARIA_DEVICE uint64_t mnmajor_desc(uint32_t tile, int k) {
  return make_smem_desc_sw(tile, AB_CH, 1024, UMMA_SW128) + k * (2048 >> 4);
}

// 128 x 128 x 128 products: SS with both operands K-major, TS with A from TMEM (bf16, 2 per column) and B MN-major
ARIA_DEVICE void mma_ss_128(uint32_t tmem_d, uint32_t a_tile, uint32_t b_tile) {
  constexpr uint32_t idesc = make_idesc_bf16(AB_BLK, AB_BLK, false, false);
#pragma unroll
  for (int k = 0; k < 8; ++k) umma_bf16_ss(tmem_d, kmajor_desc(a_tile, k), kmajor_desc(b_tile, k), idesc, k ? 1u : 0u);
}
ARIA_DEVICE void mma_ts_128(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_tile, bool accumulate) {
  constexpr uint32_t idesc = make_idesc_bf16(AB_BLK, AB_BLK, false, true);
#pragma unroll
  for (int k = 0; k < 8; ++k) umma_bf16_ts(tmem_d, tmem_a + k * 8, mnmajor_desc(b_tile, k), idesc, (accumulate || k) ? 1u : 0u);
}

// 128 fp32 accumulator columns of this thread's TMEM lane -> one bf16 row of 128 (times `mul`); the load is warp-wide
ARIA_DEVICE void store_acc_row(uint32_t tacc, __nv_bfloat16* row, bool ok, float mul) {
#pragma unroll 1
  for (int c = 0; c < 128; c += 16) {
    uint32_t v[16];
    tmem_ld_32x16(tacc + c, v);
    tmem_ld_wait();
    if (ok) {
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(v[g * 8 + e]) * mul;
        *reinterpret_cast<uint4*>(row + c + g * 8) =
            make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
      }
    }
  }
}

__global__ void __launch_bounds__(256) attn_bwd_pre_kernel(const uint2* __restrict__ out, const uint2* __restrict__ dout,
                                                           float* __restrict__ delta, int B, int H, int T) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);  // (b, t, h), token-major order
  if (row >= static_cast<int64_t>(B) * T * H) return;
  const uint2 o = out[row * 32 + lane], g = dout[row * 32 + lane];
  float s = bf16_lo(o.x) * bf16_lo(g.x) + bf16_hi(o.x) * bf16_hi(g.x) + bf16_lo(o.y) * bf16_lo(g.y) + bf16_hi(o.y) * bf16_hi(g.y);
#pragma unroll
  for (int w = 16; w; w >>= 1) s += __shfl_xor_sync(0xffffffffu, s, w);
  if (lane == 0) {
    const int h = static_cast<int>(row % H);
    const int64_t bt = row / H;
    const int t = static_cast<int>(bt % T), b = static_cast<int>(bt / T);
    delta[(static_cast<int64_t>(b) * H + h) * T + t] = s;
  }
}

// shared memory: [resident tile 0][resident tile 1][stage 0: tile 0, tile 1][stage 1: tile 0, tile 1][lse | Delta x 2][barriers]
struct BwdSmem {
  uint8_t* base;
  ARIA_DEVICE uint8_t* resident(int i) const { return base + i * AB_TILE; }
  ARIA_DEVICE uint8_t* staged(int s, int i) const { return base + (2 + 2 * s + i) * AB_TILE; }
  ARIA_DEVICE float* rowvals() const { return reinterpret_cast<float*>(base + 6 * AB_TILE); }  // [2 buffers][lse 128 | Delta 128]
  ARIA_DEVICE uint64_t* bars() const { return reinterpret_cast<uint64_t*>(base + 6 * AB_TILE + 2048); }
};

// dK, dV of one (b, h, key block): resident K, V; streamed (Q, dO) per query block.
__global__ void __launch_bounds__(AB_THREADS, 1)
attn_bwd_dkdv_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO, const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const BwdSmem sm{reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023))};
  uint64_t* bars = sm.bars();
  uint64_t* kv_full = bars;        // K, V landed
  uint64_t* qd_full = bars + 1;    // [2] Q, dO of a stage landed
  uint64_t* qd_empty = bars + 3;   // [2] the MMAs reading a stage are done
  uint64_t* s_full = bars + 5;     // S^T, dP^T in TMEM
  uint64_t* p_full = bars + 6;     // P^T, dS^T written back (4 arrivals, one per warp)
  uint64_t* acc_full = bars + 7;   // dV, dK final
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int BH = p.B * p.H;
  const int kb = blockIdx.x / BH, bh = blockIdx.x % BH;  // key block 0 (the most query blocks) first
  const int b = bh / p.H, h = bh % p.H;
  const int k0 = kb * AB_BLK;
  const int n_it = p.n_blk - kb;  // query blocks kb .. n_blk-1
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQ);
    prefetch_tmap(&tmK);
    prefetch_tmap(&tmV);
    prefetch_tmap(&tmdO);
    mbar_init(kv_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&qd_full[i], 1);
      mbar_init(&qd_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 4);
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 5) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;  // columns: S^T [0,128) | dP^T [128,256) | dV [256,384) | dK [384,512)

  if (warp == 4) {
    if (elect_one()) {
      mbar_arrive_expect_tx(kv_full, 2 * AB_TILE);
      load_tile_hm(sm.resident(0), &tmK, kv_full, k0, h, b);
      load_tile_hm(sm.resident(1), &tmV, kv_full, k0, h, b);
      for (int it = 0; it < n_it; ++it) {
        const int s = it & 1, q0 = (kb + it) * AB_BLK;
        mbar_wait(&qd_empty[s], ((it >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&qd_full[s], 2 * AB_TILE);
        load_tile_hm(sm.staged(s, 0), &tmQ, &qd_full[s], q0, h, b);
        load_tile_tm(sm.staged(s, 1), &tmdO, &qd_full[s], q0, h, b);
      }
    }
  } else if (warp == 5) {
    if (elect_one()) {
      const uint32_t sK = smem_u32(sm.resident(0)), sV = smem_u32(sm.resident(1));
      const uint32_t tS = tmem, tdP = tmem + 128, tdV = tmem + 256, tdK = tmem + 384;
      mbar_wait(kv_full, 0);
      for (int it = 0; it < n_it; ++it) {
        const int s = it & 1;
        const uint32_t sQ = smem_u32(sm.staged(s, 0)), sdO = smem_u32(sm.staged(s, 1));
        mbar_wait(&qd_full[s], (it >> 1) & 1);
        tc_fence_after();
        // S^T(it) and dP^T(it) overwrite P^T / dS^T(it-1): the dV / dK MMAs reading those were issued first and
        // tcgen05.mma of one thread execute in order
        mma_ss_128(tS, sK, sQ);
        mma_ss_128(tdP, sV, sdO);
        umma_commit(s_full);
        mbar_wait(p_full, it & 1);
        tc_fence_after();
        mma_ts_128(tdV, tS, sdO, it > 0);
        mma_ts_128(tdK, tdP, sQ, it > 0);
        umma_commit(&qd_empty[s]);
      }
      umma_commit(acc_full);
    }
  } else {
    // ---- softmax gradient: thread = key row r of the block
    const int r = warp * 32 + lane;
    const int key = k0 + r;
    const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t tS = tmem + lane_addr, tdP = tmem + 128 + lane_addr;
    const bool key_dead = key >= p.T || (p.key_mask && p.key_mask[static_cast<int64_t>(b) * p.T + key]);
    const float* lse_bh = p.lse + static_cast<int64_t>(bh) * p.T;
    const float* delta_bh = p.delta + static_cast<int64_t>(bh) * p.T;
    for (int it = 0; it < n_it; ++it) {
      const int q0 = (kb + it) * AB_BLK;
      // lse / Delta of the block's 128 queries (columns here) through shared memory; two buffers, so one barrier per block
      // also keeps a fast warp from overwriting values a slow one still reads
      float* rv = sm.rowvals() + (it & 1) * 256;
      const int qr = q0 + r;
      rv[r] = qr < p.T ? lse_bh[qr] : INFINITY;
      rv[128 + r] = qr < p.T ? delta_bh[qr] : 0.f;
      named_bar_sync(1, 128);
      mbar_wait(s_full, it & 1);
      tc_fence_after();
      const bool diag = it == 0;  // query block == key block: causal triangle
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t sr[32], dpr[32];
        tmem_ld_32x32(tS + c * 32, sr);
        tmem_ld_32x32(tdP + c * 32, dpr);
        tmem_ld_wait();
        uint32_t pk[16], dk[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          float pp[2], ds[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int j = c * 32 + 2 * e + u;
            float pv = fast_ex2(fmaf(__uint_as_float(sr[2 * e + u]), p.scale_log2, -rv[j]));
            if (key_dead || (diag && q0 + j < key)) pv = 0.f;
            pp[u] = pv;
            ds[u] = pv * (__uint_as_float(dpr[2 * e + u]) - rv[128 + j]);
          }
          pk[e] = pack_bf16(pp[0], pp[1]);
          dk[e] = pack_bf16(ds[0], ds[1]);
        }
        // chunk c (32 queries = 16 packed columns) goes over columns [16c, 16c+16), already read
        tmem_st_32x16(tS + c * 16, pk);
        tmem_st_32x16(tdP + c * 16, dk);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
    }
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const bool ok = key < p.T;
    const int64_t off = (static_cast<int64_t>(b) * p.T + (ok ? key : 0)) * (static_cast<int64_t>(p.H) * 128) + h * 128;
    store_acc_row(tmem + 256 + lane_addr, p.dv + off, ok, 1.f);
    store_acc_row(tmem + 384 + lane_addr, p.dk + off, ok, p.scale);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem, 512);
}

// dQ of one (b, h, query block): resident Q, dO; streamed (K, V) per key block.
__global__ void __launch_bounds__(AB_THREADS, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmdO, const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const BwdSmem sm{reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023))};
  uint64_t* bars = sm.bars();
  uint64_t* qd_full = bars;        // Q, dO landed
  uint64_t* kv_full = bars + 1;    // [2]
  uint64_t* kv_empty = bars + 3;   // [2]
  uint64_t* s_full = bars + 5;     // S, dP in TMEM
  uint64_t* ds_full = bars + 6;    // dS written back (4 arrivals)
  uint64_t* acc_full = bars + 7;   // dQ final
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int BH = p.B * p.H;
  const int qb = p.n_blk - 1 - blockIdx.x / BH, bh = blockIdx.x % BH;  // last query block (the most key blocks) first
  const int b = bh / p.H, h = bh % p.H;
  const int q0 = qb * AB_BLK;
  const int n_it = qb + 1;  // key blocks 0 .. qb
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQ);
    prefetch_tmap(&tmK);
    prefetch_tmap(&tmV);
    prefetch_tmap(&tmdO);
    mbar_init(qd_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(ds_full, 4);
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 5) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;  // columns: S [0,128) | dP [128,256) | dQ [256,384)

  if (warp == 4) {
    if (elect_one()) {
      mbar_arrive_expect_tx(qd_full, 2 * AB_TILE);
      load_tile_hm(sm.resident(0), &tmQ, qd_full, q0, h, b);
      load_tile_tm(sm.resident(1), &tmdO, qd_full, q0, h, b);
      for (int it = 0; it < n_it; ++it) {
        const int s = it & 1;
        mbar_wait(&kv_empty[s], ((it >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&kv_full[s], 2 * AB_TILE);
        load_tile_hm(sm.staged(s, 0), &tmK, &kv_full[s], it * AB_BLK, h, b);
        load_tile_hm(sm.staged(s, 1), &tmV, &kv_full[s], it * AB_BLK, h, b);
      }
    }
  } else if (warp == 5) {
    if (elect_one()) {
      const uint32_t sQ = smem_u32(sm.resident(0)), sdO = smem_u32(sm.resident(1));
      const uint32_t tS = tmem, tdP = tmem + 128, tdQ = tmem + 256;
      mbar_wait(qd_full, 0);
      for (int it = 0; it < n_it; ++it) {
        const int s = it & 1;
        const uint32_t sK = smem_u32(sm.staged(s, 0)), sV = smem_u32(sm.staged(s, 1));
        mbar_wait(&kv_full[s], (it >> 1) & 1);
        tc_fence_after();
        mma_ss_128(tS, sQ, sK);
        mma_ss_128(tdP, sdO, sV);
        umma_commit(s_full);
        mbar_wait(ds_full, it & 1);
        tc_fence_after();
        mma_ts_128(tdQ, tdP, sK, it > 0);
        umma_commit(&kv_empty[s]);
      }
      umma_commit(acc_full);
    }
  } else {
    // ---- softmax gradient: thread = query row r of the block
    const int r = warp * 32 + lane;
    const int q = q0 + r;
    const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t tS = tmem + lane_addr, tdP = tmem + 128 + lane_addr;
    const bool row_ok = q < p.T;
    const float lse_r = row_ok ? p.lse[static_cast<int64_t>(bh) * p.T + q] : INFINITY;
    const float delta_r = row_ok ? p.delta[static_cast<int64_t>(bh) * p.T + q] : 0.f;
    const float neg_lse = -lse_r;
    const uint8_t* km = p.key_mask ? p.key_mask + static_cast<int64_t>(b) * p.T : nullptr;
    for (int it = 0; it < n_it; ++it) {
      const int kbase = it * AB_BLK;
      const bool need_mask = it == qb || kbase + AB_BLK > p.T || km != nullptr;
      mbar_wait(s_full, it & 1);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t dead = 0;  // bit e: key kbase + 32c + e is past T or masked out (one byte load per lane, then a ballot)
        if (need_mask) {
          const int kl = kbase + c * 32 + lane;
          dead = __ballot_sync(0xffffffffu, kl >= p.T || (km && km[kl]));
        }
        uint32_t sr[32], dpr[32];
        tmem_ld_32x32(tS + c * 32, sr);
        tmem_ld_32x32(tdP + c * 32, dpr);
        tmem_ld_wait();
        uint32_t dk[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          float ds[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int j = 2 * e + u;
            float pv = fast_ex2(fmaf(__uint_as_float(sr[j]), p.scale_log2, neg_lse));
            if (need_mask && (((dead >> j) & 1u) || kbase + c * 32 + j > q)) pv = 0.f;
            ds[u] = pv * (__uint_as_float(dpr[j]) - delta_r);
          }
          dk[e] = pack_bf16(ds[0], ds[1]);
        }
        tmem_st_32x16(tdP + c * 16, dk);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);
    }
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const int64_t off = (static_cast<int64_t>(b) * p.T + (row_ok ? q : 0)) * (static_cast<int64_t>(p.H) * 128) + h * 128;
    store_acc_row(tmem + 256 + lane_addr, p.dq + off, row_ok, p.scale);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem, 512);
}

static int make_tmap_head_major(CUtensorMap* tm, const void* ptr, int T, int H, int B, int64_t stride_b, int64_t stride_h) {
  uint64_t dims[4] = {128u, static_cast<uint64_t>(T), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
  uint64_t str[3] = {256u, static_cast<uint64_t>(stride_h) * 2, static_cast<uint64_t>(stride_b) * 2};
  uint32_t box[4] = {64, AB_BLK, 1, 1};
  return make_tmap_bf16(tm, ptr, 4, dims, str, box);
}
// token-major [B, T, H*128]: dims ordered (column, head, token, batch) so that the strides grow; a box of one head and 128
// tokens lands in shared memory exactly like a head-major box
static int make_tmap_token_major(CUtensorMap* tm, const void* ptr, int T, int H, int B) {
  uint64_t dims[4] = {128u, static_cast<uint64_t>(H), static_cast<uint64_t>(T), static_cast<uint64_t>(B)};
  uint64_t str[3] = {256u, static_cast<uint64_t>(H) * 256, static_cast<uint64_t>(T) * H * 256};
  uint32_t box[4] = {64, 1, AB_BLK, 1};
  return make_tmap_bf16(tm, ptr, 4, dims, str, box);
}

static int64_t delta_bytes(int32_t B, int32_t H, int32_t T) {
  return (static_cast<int64_t>(B) * H * T * static_cast<int64_t>(sizeof(float)) + 255) / 256 * 256;
}

}  // namespace aria

using namespace aria;

extern "C" int64_t aria_attention_bwd_workspace_bytes(int32_t B, int32_t H, int32_t T) {
  if (B <= 0 || H <= 0 || T <= 0) return ARIA_ERR_BAD_ARG;
  return delta_bytes(B, H, T);
}

extern "C" int aria_attention_bwd(const void* q, const void* k, const void* v, const void* out, const void* dout, const float* lse,
                                  void* dq, void* dk, void* dv, const uint8_t* key_mask, int32_t B, int32_t H, int32_t T,
                                  int64_t q_stride_b, int64_t q_stride_h, int64_t kv_stride_b, int64_t kv_stride_h, float scale,
                                  int32_t head_dim, int32_t causal, void* workspace, int64_t workspace_bytes,
                                  aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (!causal || head_dim != 128) {
    fprintf(stderr, "aria_b200: attention backward supports causal self-attention with head_dim 128 only\n");
    return ARIA_ERR_UNSUPPORTED;
  }
  ARIA_CHECK_ARG(q && k && v && out && dout && lse && dq && dk && dv && workspace);
  ARIA_CHECK_ARG(B > 0 && H > 0 && T > 0);
  ARIA_CHECK_ARG(q_stride_b % 8 == 0 && q_stride_h % 8 == 0 && kv_stride_b % 8 == 0 && kv_stride_h % 8 == 0);
  ARIA_CHECK_ARG(workspace_bytes >= delta_bytes(B, H, T));
  const int n_blk = (T + AB_BLK - 1) / AB_BLK;
  const int64_t ctas = static_cast<int64_t>(B) * H * n_blk;
  ARIA_CHECK_ARG(ctas < (1ll << 31));

  AttnBwdParams p{};
  p.B = B;
  p.H = H;
  p.T = T;
  p.n_blk = n_blk;
  p.scale = scale;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.key_mask = key_mask;
  p.lse = lse;
  p.delta = static_cast<float*>(workspace);
  p.dq = static_cast<__nv_bfloat16*>(dq);
  p.dk = static_cast<__nv_bfloat16*>(dk);
  p.dv = static_cast<__nv_bfloat16*>(dv);

  CUtensorMap tmQ, tmK, tmV, tmdO;
  int rc = make_tmap_head_major(&tmQ, q, T, H, B, q_stride_b, q_stride_h);
  if (!rc) rc = make_tmap_head_major(&tmK, k, T, H, B, kv_stride_b, kv_stride_h);
  if (!rc) rc = make_tmap_head_major(&tmV, v, T, H, B, kv_stride_b, kv_stride_h);
  if (!rc) rc = make_tmap_token_major(&tmdO, dout, T, H, B);
  if (rc) return rc;

  const int64_t rows = static_cast<int64_t>(B) * T * H;
  attn_bwd_pre_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, stream>>>(
      static_cast<const uint2*>(out), static_cast<const uint2*>(dout), static_cast<float*>(workspace), B, H, T);
  rc = check_launch("attn_bwd_pre_kernel");
  if (rc) return rc;
  static bool attr_dkdv[kMaxDevices] = {}, attr_dq[kMaxDevices] = {};
  if (ensure_dynamic_smem(attr_dkdv, attn_bwd_dkdv_kernel, AB_SMEM) != cudaSuccess) return ARIA_ERR_CUDA;
  if (ensure_dynamic_smem(attr_dq, attn_bwd_dq_kernel, AB_SMEM) != cudaSuccess) return ARIA_ERR_CUDA;
  attn_bwd_dkdv_kernel<<<static_cast<unsigned>(ctas), AB_THREADS, AB_SMEM, stream>>>(tmQ, tmK, tmV, tmdO, p);
  rc = check_launch("attn_bwd_dkdv_kernel");
  if (rc) return rc;
  attn_bwd_dq_kernel<<<static_cast<unsigned>(ctas), AB_THREADS, AB_SMEM, stream>>>(tmQ, tmK, tmV, tmdO, p);
  return check_launch("attn_bwd_dq_kernel");
}
