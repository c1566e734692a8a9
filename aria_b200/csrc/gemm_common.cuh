// Shared pieces of the tcgen05 GEMM kernels (gemm.cu: 1-CTA tiles, gemm2.cu: 2-CTA pairs): parameters, the
// device-side tile scheduler and the fused epilogues.
//
// Persistent, warp-specialised tcgen05 GEMM for sm_100a (bf16 x bf16 -> fp32 in TMEM -> bf16).
//
//   * warp 0  : TMA producer  (cp.async.bulk.tensor, SWIZZLE_128B tiles, mbarrier complete_tx)
//   * warp 1  : MMA issuer    (one elected thread, tcgen05.mma cta_group::1 M=128 x N=BN x K=16), owns TMEM
//   * warps 2-9: epilogue     (tcgen05.ld 32x32b, fused epilogue, 16-byte global stores; two warps per lane quadrant)
//   * TMEM accumulators are double buffered (2 x BN columns) so tile i+1's MMAs overlap tile i's epilogue.
//
// One kernel template serves (a) nn.Linear-layout dense GEMMs (B = [N,K], K-major), (b) the reference's
// grouped expert GEMM (aria/model/moe_lm.py:398-428,467-484: B = [E,K,N], consumed N-contiguous through an
// MN-major UMMA descriptor — the HF weight layout is used as is, no repack) with a device-side tile
// scheduler over the expert row offsets (no host sync, cf. moe_lm.py:478), and (c) the fused epilogues:
// bias/activation/residual, SwiGLU (moe_lm.py:505-507), and RoPE + head-major scatter for q/k/v.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace aria {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KB
constexpr int GEMM_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two warps per TMEM lane quadrant)
constexpr int EPI_WARPS = 8;

// Internal epilogues of the fused lm_head + cross-entropy (lm_loss.cu); never accepted by aria_gemm.
//   XENT_STATS: z = bf16(acc), columns >= V are -inf; per row, one (max, sum exp(z - max)) partial per 64 columns, and the
//               target's logit
//   XENT_GRAD : out = bf16((exp(z - lse[r]) - [v0 + c == target[r]]) * dloss / n_valid), 0 for ignored rows
//   ACC_F32   : acc32 = acc (+ acc32 unless first); the last call stores bf16(acc32) to out instead
constexpr int EPI_XENT_STATS = 3;
constexpr int EPI_XENT_GRAD = 4;
constexpr int EPI_ACC_F32 = 5;
constexpr int XENT_SLOT = 64;  // columns per (max, sum) partial

struct XentParams {
  const int32_t* target;   // [M], < 0: ignored row
  const float* lse;        // [M] natural log (GRAD)
  float2* part;            // [ceil(V / 64)][M] (STATS)
  float* tlogit;           // [M] (STATS)
  const float* dloss;      // [1] (GRAD)
  const int32_t* n_valid;  // [1] (GRAD)
  float* acc;              // [M, N] fp32 (ACC_F32)
  int64_t M;
  int V, v0;               // vocabulary size; global column of the tile's column 0 (GRAD)
  int first, last;         // ACC_F32
};

struct GemmParams {
  int M, N, K;  // N = output columns per segment
  int num_groups;
  const int32_t* group_offsets;
  const int32_t* group_counts;     // non-NULL: group g = rows [group_offsets[g], + group_counts[g]) (fixed-capacity regions)
  const uint64_t* out_group_base;  // non-NULL (LINEAR): rows of group g are stored at out_group_base[g] + (out_group_row0[g] + r)*ldo
  const int32_t* out_group_row0;   //   — e.g. straight into the source rank's combine buffer over NVLink (expert parallelism)
  int b_group_rows;  // K-major grouped weights [G, N, K]: B row of (group g, column c) is g*b_group_rows + c (0: dense)
  int group_mod;  // weight block of group g: g % group_mod (> 0: expert-parallel (source rank, expert) groups), g / -group_mod (< 0:
                  // (expert, source rank) groups - the groups of one expert are neighbours and share its weights in L2), g (0)
  int pair;       // 2-CTA kernel on fixed-capacity regions: groups (2s, 2s+1) form ONE 256-row tile, 128 rows of each (see gemm2.cu)
  int n_seg;
  int act;
  const __nv_bfloat16* bias[3];
  const __nv_bfloat16* residual;
  int64_t ldr;
  __nv_bfloat16* out[3];
  int64_t ldo;
  int head_dim, head_ld, rows_per_batch, pos0;
  int64_t stride_b, stride_h;
  int rope_mask;
  const __nv_bfloat16* rope_cos;
  const __nv_bfloat16* rope_sin;
  const int32_t* position_ids;
  int dbg_lbo, dbg_sbo, dbg_kadv;
  XentParams x;
};

ARIA_DEVICE int weight_block(const GemmParams& p, int grp) {
  return p.group_mod > 0 ? grp % p.group_mod : (p.group_mod < 0 ? grp / (-p.group_mod) : grp);
}

// Monotonic decoder of the persistent tile index -> (group, m-tile, n-tile).  Tiles are ordered group-major,
// then n-tile, with the m-tile innermost so that CTAs running concurrently share the same weight tile.
struct TileSched {
  const int32_t* offs;
  const int32_t* cnts;
  int G, n_tiles, M;
  int g, mt_prefix, g_row0, g_rows, g_mt, bm;
  bool pair;
  __device__ void init(const GemmParams& p, int n_tiles_, int bm_ = BM) {
    bm = bm_;
    pair = p.pair != 0;
    offs = p.group_offsets;
    cnts = p.group_counts;
    G = p.num_groups;
    n_tiles = n_tiles_;
    M = p.M;
    g = -1;
    mt_prefix = 0;
    g_mt = 0;
    g_row0 = 0;
    g_rows = 0;
  }
  __device__ bool load_group(int gi) {
    if (pair) {  // super-group gi = regions (2 gi, 2 gi + 1); each CTA of the pair walks ITS region in 128-row steps
      if (2 * gi + 1 >= G) return false;
      g_row0 = 0;
      g_rows = max(cnts[2 * gi], cnts[2 * gi + 1]);
      g_mt = (g_rows + BM - 1) / BM;
      return true;
    }
    if (gi >= G) return false;
    if (offs) {
      g_row0 = offs[gi];
      g_rows = cnts ? cnts[gi] : offs[gi + 1] - g_row0;
    } else {
      g_row0 = 0;
      g_rows = M;
    }
    g_mt = (g_rows + bm - 1) / bm;
    return true;
  }
  __device__ bool decode(int t, int& grp, int& m_idx, int& n_idx, int& row0, int& rows) {
    if (g < 0) {
      g = 0;
      if (!load_group(0)) return false;
    }
    while (t >= (mt_prefix + g_mt) * n_tiles) {
      mt_prefix += g_mt;
      ++g;
      if (!load_group(g)) return false;
    }
    int r = t - mt_prefix * n_tiles;
    n_idx = r / g_mt;
    m_idx = r - n_idx * g_mt;
    grp = g;
    row0 = g_row0;
    rows = g_rows;
    return true;
  }
};

ARIA_DEVICE float act_apply(float x, int act) {
  if (act == ARIA_ACT_GELU_TANH) {
    // torch gelu(approximate="tanh"): one fp32 evaluation, rounded once by the caller
    const float k0 = 0.7978845608028654f, k1 = 0.044715f;
    float inner = k0 * (x + k1 * x * x * x);
    return 0.5f * x * (1.f + fast_tanh(inner));
  }
  if (act == ARIA_ACT_GELU_NEW) {
    // transformers NewGELUActivation evaluated op by op on bf16 tensors (aria/model/projector.py:40-45):
    // 0.5 * x * (1.0 + tanh(sqrt(2/pi) * (x + 0.044715 * pow(x, 3))))
    float p3 = bf16r(x * x * x);
    float t = bf16r(0.044715f * p3);
    t = bf16r(x + t);
    t = bf16r(0.7978845608028654f * t);
    t = bf16r(fast_tanh(t));
    t = bf16r(1.0f + t);
    float h = bf16r(0.5f * x);
    return h * t;
  }
  return x;
}

// Fused epilogue of one accumulator tile: this thread owns one output row (TMEM lane) and walks the tile's columns
// in 32-column tcgen05.ld chunks.  `taddr` already carries the lane quadrant and accumulator-stage column offset.
//   LINEAR / HEADS : the tile covers output columns [n_idx*BN, +BN)
//   SWIGLU         : TMEM columns [0,BN/2) hold the gate, [BN/2,BN) the up projection; output columns
//                    [n_idx*BN/2, +BN/2)
// `half` (0/1) selects which half of the tile's column chunks this warp handles: the two warps that share a TMEM lane
// quadrant split the columns, so 8 epilogue warps drain one accumulator in half the time of 4.
template <int BN, int EPI>
ARIA_DEVICE void epilogue_tile(const GemmParams& p, const uint32_t taddr, const int n_out_total, const int n_idx,
                               const int64_t grow, const bool row_ok, const int half, const int grp = 0, const int r_in_grp = 0) {
  constexpr int OUT_BN = (EPI == ARIA_EPI_SWIGLU) ? BN / 2 : BN;
  if constexpr (EPI == ARIA_EPI_SWIGLU) {
    // out[:, n] = bf16( bf16(silu(bf16(gate))) * bf16(up) )  — rounding points of moe_lm.py:505-507
    __nv_bfloat16* orow = p.out[0] + grow * p.ldo + n_idx * OUT_BN;
    constexpr int NCH = OUT_BN / 32;
    const int cb = (half * NCH / 2) * 32, ce = half ? OUT_BN : (NCH / 2) * 32;
#pragma unroll 1
    for (int c = cb; c < ce; c += 32) {
      uint32_t g[32], u[32];
      tmem_ld_32x32(taddr + c, g);
      tmem_ld_32x32(taddr + OUT_BN + c, u);
      tmem_ld_wait();
      uint32_t o[16];
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        float g0 = __uint_as_float(g[j]), g1 = __uint_as_float(g[j + 1]);
        float u0 = __uint_as_float(u[j]), u1 = __uint_as_float(u[j + 1]);
        bf16r2(g0, g1);
        bf16r2(u0, u1);
        float s0 = fast_silu(g0), s1 = fast_silu(g1);
        bf16r2(s0, s1);
        o[j >> 1] = pack_bf16(s0 * u0, s1 * u1);
      }
      if (row_ok) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int col = n_idx * OUT_BN + c + q * 8;
          if (col + 8 <= p.N)
            *reinterpret_cast<uint4*>(orow + c + q * 8) = make_uint4(o[q * 4], o[q * 4 + 1], o[q * 4 + 2], o[q * 4 + 3]);
        }
      }
    }
  } else if constexpr (EPI == EPI_XENT_STATS) {
    // log-sum-exp partials of the bf16-rounded logits; this warp's half of the tile is 1 (BN = 128) or 2 (BN = 256) slots
    constexpr float L2E = 1.4426950408889634f;
    const int col0 = n_idx * BN + half * (BN / 2);
    const int t = row_ok ? p.x.target[grow] : -1;
    float m = -INFINITY, s = 0.f;
#pragma unroll 1
    for (int c = 0; c < BN / 2; c += 32) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + half * (BN / 2) + c, v);
      tmem_ld_wait();
      const int cb = col0 + c;
      float z[32], cm = -INFINITY, zt = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        z[j] = cb + j < p.x.V ? bf16r(__uint_as_float(v[j])) : -INFINITY;
        cm = fmaxf(cm, z[j]);
        if (cb + j == t) zt = z[j];
      }
      if (row_ok && t >= cb && t < cb + 32) p.x.tlogit[grow] = zt;
      if (cm > -INFINITY) {
        const float mn = fmaxf(m, cm);
        float a = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) a += exp2f((z[j] - mn) * L2E);
        s = s * exp2f((m - mn) * L2E) + a;
        m = mn;
      }
      if ((c & (XENT_SLOT - 1)) == XENT_SLOT - 32) {  // end of a 64-column slot
        const int slot0 = cb + 32 - XENT_SLOT;
        if (row_ok && slot0 < p.x.V) p.x.part[static_cast<int64_t>(slot0 / XENT_SLOT) * p.x.M + grow] = make_float2(m, s);
        m = -INFINITY;
        s = 0.f;
      }
    }
  } else if constexpr (EPI == EPI_XENT_GRAD) {
    // d loss / d z of one vocabulary chunk (tile columns are chunk columns; global column = v0 + chunk column)
    constexpr float L2E = 1.4426950408889634f;
    const int col0 = n_idx * BN;
    int t = -1;
    float lse = 0.f;
    if (row_ok) {
      t = p.x.target[grow];
      lse = p.x.lse[grow];
    }
    const int nv = *p.x.n_valid;
    const float scale = (t >= 0 && nv > 0) ? *p.x.dloss / static_cast<float>(nv) : 0.f;
    const int tc = t - p.x.v0;  // target as a chunk column
    __nv_bfloat16* orow = p.out[0] + grow * p.ldo;
#pragma unroll 1
    for (int c = half * (BN / 2); c < (half + 1) * (BN / 2); c += 32) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + c, v);
      tmem_ld_wait();
      if (!row_ok) continue;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int col = col0 + c + q * 8;
        if (col + 8 > p.N) continue;
        float g[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float z = bf16r(__uint_as_float(v[q * 8 + j]));
          g[j] = (exp2f((z - lse) * L2E) - (col + j == tc ? 1.f : 0.f)) * scale;
        }
        *reinterpret_cast<uint4*>(orow + col) =
            make_uint4(pack_bf16(g[0], g[1]), pack_bf16(g[2], g[3]), pack_bf16(g[4], g[5]), pack_bf16(g[6], g[7]));
      }
    }
  } else if constexpr (EPI == EPI_ACC_F32) {
    const int col0 = n_idx * BN;
    float* arow = p.x.acc + grow * p.N;
    __nv_bfloat16* orow = p.out[0] + grow * p.ldo;
#pragma unroll 1
    for (int c = half * (BN / 2); c < (half + 1) * (BN / 2); c += 32) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + c, v);
      tmem_ld_wait();
      if (!row_ok) continue;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int col = col0 + c + q * 8;
        if (col + 8 > p.N) continue;
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = __uint_as_float(v[q * 8 + j]);
        float4* a4 = reinterpret_cast<float4*>(arow + col);
        if (!p.x.first) {
          const float4 u = a4[0], w = a4[1];
          x[0] += u.x; x[1] += u.y; x[2] += u.z; x[3] += u.w;
          x[4] += w.x; x[5] += w.y; x[6] += w.z; x[7] += w.w;
        }
        if (p.x.last) {
          *reinterpret_cast<uint4*>(orow + col) =
              make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
        } else {
          a4[0] = make_float4(x[0], x[1], x[2], x[3]);
          a4[1] = make_float4(x[4], x[5], x[6], x[7]);
        }
      }
    }
  } else if constexpr (EPI == ARIA_EPI_LINEAR) {
    const int col0 = n_idx * BN;
    const int seg = col0 / p.N;  // bias is per segment; out is [m, n_seg*n]
    const __nv_bfloat16* bias = p.bias[seg];
    __nv_bfloat16* orow = p.out[0] + grow * p.ldo + col0;
    if (p.out_group_base)  // per-group destination (possibly a peer GPU's memory: the stores then travel over NVLink)
      orow = reinterpret_cast<__nv_bfloat16*>(p.out_group_base[grp]) + static_cast<int64_t>(p.out_group_row0[grp] + r_in_grp) * p.ldo + col0;
    const __nv_bfloat16* rrow = (p.residual && row_ok) ? p.residual + grow * p.ldr + col0 : nullptr;
    // Two-deep software pipeline over the 32-column chunks of this warp's half: the accumulator chunk (tcgen05.ld), the bias
    // vectors and the residual row pieces of chunk i + 1 are all in flight while chunk i is converted and stored.  Round 1
    // loaded bias / residual inside the per-8-column loop, each load followed by its use: ncu showed 16 - 32 serial global-load
    // latencies per thread and tile (long_scoreboard on the LDG consumers = 22 % of all samples of the ViT fc1 GEMM, tensor pipe
    // 39 % active), i.e. the epilogue, not the MMA loop, set the tile time (profiles/r02_gemm_notes.txt).
    constexpr int NCH = BN / 32, NCHH = NCH - NCH / 2;  // chunks of the tile / of the larger half (BN = 32: all in half 1)
    const int cb = half ? (NCH / 2) * 32 : 0;
    const int n_my = half ? NCH - NCH / 2 : NCH / 2;
    if (n_my == 0) return;
    uint32_t v[2][32];
    uint4 bv[2][4], rv[2][4];
    auto issue = [&](int c, int set) {
      tmem_ld_32x32(taddr + c, v[set]);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int col = col0 + c + q * 8;
        const bool ok = col + 8 <= n_out_total;
        bv[set][q] = (bias && ok) ? __ldg(reinterpret_cast<const uint4*>(bias + (col - seg * p.N))) : make_uint4(0, 0, 0, 0);
        rv[set][q] = (rrow && ok) ? *reinterpret_cast<const uint4*>(rrow + c + q * 8) : make_uint4(0, 0, 0, 0);
      }
    };
    issue(cb, 0);
#pragma unroll
    for (int i = 0; i < NCHH; ++i) {
      if (i >= n_my) break;
      const int c = cb + i * 32;
      const int set = i & 1;
      tmem_ld_wait();
      if (i + 1 < n_my) issue(c + 32, set ^ 1);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int col = col0 + c + q * 8;
        if (col + 8 > n_out_total) continue;
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = __uint_as_float(v[set][q * 8 + j]);
        if (bias) {
          const uint32_t bw[4] = {bv[set][q].x, bv[set][q].y, bv[set][q].z, bv[set][q].w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            x[2 * j] += bf16_lo(bw[j]);
            x[2 * j + 1] += bf16_hi(bw[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = bf16r(x[j]);
        if (p.act != ARIA_ACT_NONE) {
#pragma unroll
          for (int j = 0; j < 8; ++j) x[j] = bf16r(act_apply(x[j], p.act));
        }
        if (row_ok) {
          if (rrow) {
            const uint32_t rw[4] = {rv[set][q].x, rv[set][q].y, rv[set][q].z, rv[set][q].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              x[2 * j] += bf16_lo(rw[j]);
              x[2 * j + 1] += bf16_hi(rw[j]);
            }
          }
          *reinterpret_cast<uint4*>(orow + c + q * 8) =
              make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
        }
      }
    }
  } else {  // ARIA_EPI_HEADS
    const int col0 = n_idx * BN;
    const int seg = col0 / p.N;
    const int cseg0 = col0 - seg * p.N;
    const __nv_bfloat16* bias = p.bias[seg];
    const int b = static_cast<int>(grow / p.rows_per_batch);
    const int tok = static_cast<int>(grow - static_cast<int64_t>(b) * p.rows_per_batch);
    __nv_bfloat16* obase = p.out[seg] + b * p.stride_b + static_cast<int64_t>(p.pos0 + tok) * p.head_ld;
    const bool rope = (p.rope_mask >> seg) & 1;
    if (rope) {
      // head_dim == 128 and BN a multiple of it: the tile holds BN/128 whole heads. rotate-half RoPE with op-by-op
      // bf16 rounding:  out = bf16(bf16(x*cos) + bf16(rotate_half(x)*sin))
      const int pos = row_ok ? (p.position_ids ? p.position_ids[grow] : p.pos0 + tok) : 0;
      const __nv_bfloat16* cs = p.rope_cos + static_cast<int64_t>(pos) * p.head_dim;
      const __nv_bfloat16* sn = p.rope_sin + static_cast<int64_t>(pos) * p.head_dim;
      constexpr int NHC = BN / 64;
#pragma unroll 1
      for (int hc = half * NHC / 2; hc < (half ? NHC : NHC / 2); hc += 1) {
        // hc enumerates (head-in-tile, 32-column chunk of the low half): hh = hc / 2, c = (hc & 1) * 32
        const int hh = hc >> 1, c = (hc & 1) * 32;
        __nv_bfloat16* orow = obase + (cseg0 / p.head_dim + hh) * p.stride_h;
        const uint32_t th = taddr + hh * 128;
        uint32_t lo[32], hi[32];
        tmem_ld_32x32(th + c, lo);
        tmem_ld_32x32(th + 64 + c, hi);
        // all 16 table vectors of this chunk are requested before anything waits (they were loaded one group at a time
        // inside the loop below, each followed by its use)
        uint4 tc_lo[4], ts_lo[4], tc_hi[4], ts_hi[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          tc_lo[q] = __ldg(reinterpret_cast<const uint4*>(cs + c + q * 8));
          ts_lo[q] = __ldg(reinterpret_cast<const uint4*>(sn + c + q * 8));
          tc_hi[q] = __ldg(reinterpret_cast<const uint4*>(cs + 64 + c + q * 8));
          ts_hi[q] = __ldg(reinterpret_cast<const uint4*>(sn + 64 + c + q * 8));
        }
        tmem_ld_wait();
        if (row_ok) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 c_lo = tc_lo[q], s_lo = ts_lo[q], c_hi = tc_hi[q], s_hi = ts_hi[q];
            const uint32_t cl[4] = {c_lo.x, c_lo.y, c_lo.z, c_lo.w}, sl[4] = {s_lo.x, s_lo.y, s_lo.z, s_lo.w};
            const uint32_t ch[4] = {c_hi.x, c_hi.y, c_hi.z, c_hi.w}, sh[4] = {s_hi.x, s_hi.y, s_hi.z, s_hi.w};
            float ol[8], oh[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float xl = __uint_as_float(lo[q * 8 + j]);
              float xh = __uint_as_float(hi[q * 8 + j]);
              bf16r2(xl, xh);
              float cosl = (j & 1) ? bf16_hi(cl[j >> 1]) : bf16_lo(cl[j >> 1]);
              float sinl = (j & 1) ? bf16_hi(sl[j >> 1]) : bf16_lo(sl[j >> 1]);
              float cosh_ = (j & 1) ? bf16_hi(ch[j >> 1]) : bf16_lo(ch[j >> 1]);
              float sinh_ = (j & 1) ? bf16_hi(sh[j >> 1]) : bf16_lo(sh[j >> 1]);
              float a0 = xl * cosl, a1 = -xh * sinl, b0 = xh * cosh_, b1 = xl * sinh_;
              bf16r2(a0, a1);
              bf16r2(b0, b1);
              ol[j] = a0 + a1;
              oh[j] = b0 + b1;
            }
            *reinterpret_cast<uint4*>(orow + c + q * 8) =
                make_uint4(pack_bf16(ol[0], ol[1]), pack_bf16(ol[2], ol[3]), pack_bf16(ol[4], ol[5]), pack_bf16(ol[6], ol[7]));
            *reinterpret_cast<uint4*>(orow + 64 + c + q * 8) =
                make_uint4(pack_bf16(oh[0], oh[1]), pack_bf16(oh[2], oh[3]), pack_bf16(oh[4], oh[5]), pack_bf16(oh[6], oh[7]));
          }
        }
      }
    } else {
      constexpr int NCH = (BN + 31) / 32, NMAX = NCH - NCH / 2;
      const int cb = half ? (NCH / 2) * 32 : 0;
      const int n_my = half ? NCH - NCH / 2 : NCH / 2;
      // same two-deep pipeline as the LINEAR epilogue: accumulator chunk and bias vectors of chunk i + 1 in flight while chunk i
      // is converted and scattered to its heads
      uint32_t v[2][32];
      uint4 bvq[2][4];
      auto window = [&](int c) { return (c + 32 <= BN) ? c : BN - 32; };  // BN = 144: the tail re-reads an overlapping window
      auto issue = [&](int c, int set) {
        const int cbase = window(c);
        tmem_ld_32x32(taddr + cbase, v[set]);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int cs_ = cseg0 + cbase + q * 8;
          bvq[set][q] = (bias && cs_ + 8 <= p.N) ? __ldg(reinterpret_cast<const uint4*>(bias + cs_)) : make_uint4(0, 0, 0, 0);
        }
      };
      if (n_my > 0) issue(cb, 0);
#pragma unroll
      for (int i = 0; i < NMAX; ++i) {
        if (i >= n_my) break;
        const int c = cb + i * 32;
        const int set = i & 1;
        tmem_ld_wait();
        if (i + 1 < n_my) issue(c + 32, set ^ 1);
        const int cbase = window(c);
        const int qstart = (c + 32 <= BN) ? 0 : (c - cbase) / 8;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (q < qstart) continue;
          const int cs_ = cseg0 + cbase + q * 8;  // column inside the segment
          if (cs_ + 8 > p.N) continue;
          float x[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) x[j] = __uint_as_float(v[set][q * 8 + j]);
          if (bias) {
            const uint4 bv = bvq[set][q];
            const uint32_t bw[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              x[2 * j] += bf16_lo(bw[j]);
              x[2 * j + 1] += bf16_hi(bw[j]);
            }
          }
          if (row_ok) {
            const int head = cs_ / p.head_dim;
            const int d = cs_ - head * p.head_dim;
            *reinterpret_cast<uint4*>(obase + head * p.stride_h + d) =
                make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
          }
        }
      }
    }
  }
}

}  // namespace aria
