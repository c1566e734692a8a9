// Row-wise / gather kernels around the GEMMs (all HBM-bound, 128-bit accesses, one warp per row).
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace aria {

ARIA_DEVICE float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

static inline int rows_grid(int64_t rows, int wpb) {
  int64_t b = (rows + wpb - 1) / wpb;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

// LlamaRMSNorm: h = x (+res, bf16-rounded); out = w * bf16(h * (1/sqrt(mean(h^2)+eps))).
// One 128-thread block per row (prefill batches are only a few hundred rows: a warp per row leaves the SMs idle).
template <int MAXV>  // max uint4 per thread held in registers
__global__ void __launch_bounds__(128) rmsnorm_kernel(const uint4* __restrict__ x, const uint4* __restrict__ res,
                                                      const uint4* __restrict__ w, uint4* __restrict__ out,
                                                      uint4* __restrict__ sum_out, int64_t rows, int vpr, float eps, float inv_d) {
  __shared__ float red[4];
  const int tid = threadIdx.x;
  for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
    float h[MAXV][8];
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int v = tid + i * 128;
      if (v < vpr) {
        const uint4 q = x[r * vpr + v];
        const uint32_t a[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          h[i][2 * j] = bf16_lo(a[j]);
          h[i][2 * j + 1] = bf16_hi(a[j]);
        }
        if (res) {
          const uint4 q2 = res[r * vpr + v];
          const uint32_t b[4] = {q2.x, q2.y, q2.z, q2.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            h[i][2 * j] = bf16r(h[i][2 * j] + bf16_lo(b[j]));
            h[i][2 * j + 1] = bf16r(h[i][2 * j + 1] + bf16_hi(b[j]));
          }
          if (sum_out)
            sum_out[r * vpr + v] = make_uint4(pack_bf16(h[i][0], h[i][1]), pack_bf16(h[i][2], h[i][3]),
                                              pack_bf16(h[i][4], h[i][5]), pack_bf16(h[i][6], h[i][7]));
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) ss += h[i][j] * h[i][j];
      }
    }
    ss = warp_sum(ss);
    __syncthreads();  // red[] free (previous row consumed)
    if ((tid & 31) == 0) red[tid >> 5] = ss;
    __syncthreads();
    ss = red[0] + red[1] + red[2] + red[3];
    const float rstd = 1.0f / sqrtf(ss * inv_d + eps);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int v = tid + i * 128;
      if (v < vpr) {
        const uint4 q = __ldg(w + v);
        const uint32_t a[4] = {q.x, q.y, q.z, q.w};
        float o[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          o[2 * j] = bf16_lo(a[j]) * bf16r(h[i][2 * j] * rstd);
          o[2 * j + 1] = bf16_hi(a[j]) * bf16r(h[i][2 * j + 1] * rstd);
        }
        out[r * vpr + v] = make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
      }
    }
  }
}

// nn.LayerNorm, one WARP per row (rows of up to 32 * MAXV uint4 = 256 * MAXV elements): the row lives in the lanes' registers,
// mean and variance are two shuffle reductions, no shared memory and no block barrier.  Used for the ViT (d = 1152: 144 vectors,
// 4.5 per lane); the block-per-row kernel below spent its time in three __syncthreads per row with 16 of 128 threads active in
// the second vector round (12.7 us per launch for 22.6 MB = 28 % of the HBM roofline in profiles/r02_bench_b.json).
template <int MAXV>
__global__ void __launch_bounds__(256) layernorm_warp_kernel(const uint4* __restrict__ x, const uint4* __restrict__ w,
                                                             const uint4* __restrict__ b, uint4* __restrict__ out, int64_t rows,
                                                             int vpr, float eps, float inv_d) {
  const int lane = threadIdx.x & 31;
  const int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  float h[MAXV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < vpr) {
      const uint4 q = x[r * vpr + v];
      const uint32_t a[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        h[i][2 * j] = bf16_lo(a[j]);
        h[i][2 * j + 1] = bf16_hi(a[j]);
        s += h[i][2 * j] + h[i][2 * j + 1];
      }
    }
  }
  const float mean = warp_sum(s) * inv_d;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    if (lane + i * 32 < vpr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float dlt = h[i][j] - mean;
        ss += dlt * dlt;
      }
    }
  }
  const float rstd = 1.0f / sqrtf(warp_sum(ss) * inv_d + eps);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < vpr) {
      const uint4 qw = __ldg(w + v), qb = __ldg(b + v);
      const uint32_t aw[4] = {qw.x, qw.y, qw.z, qw.w}, ab[4] = {qb.x, qb.y, qb.z, qb.w};
      float o[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        o[2 * j] = (h[i][2 * j] - mean) * rstd * bf16_lo(aw[j]) + bf16_lo(ab[j]);
        o[2 * j + 1] = (h[i][2 * j + 1] - mean) * rstd * bf16_hi(aw[j]) + bf16_hi(ab[j]);
      }
      out[r * vpr + v] = make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
    }
  }
}

// nn.LayerNorm over the last dim: fp32 mean / variance (two-pass over registers), one rounding at the end.
// One 128-thread block per row (same reasoning as rmsnorm_kernel).
template <int MAXV>
__global__ void __launch_bounds__(128) layernorm_kernel(const uint4* __restrict__ x, const uint4* __restrict__ w,
                                                        const uint4* __restrict__ b, uint4* __restrict__ out, int64_t rows,
                                                        int vpr, float eps, float inv_d) {
  __shared__ float red[2][4];
  const int tid = threadIdx.x;
  for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
    float h[MAXV][8];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int v = tid + i * 128;
      if (v < vpr) {
        const uint4 q = x[r * vpr + v];
        const uint32_t a[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          h[i][2 * j] = bf16_lo(a[j]);
          h[i][2 * j + 1] = bf16_hi(a[j]);
          s += h[i][2 * j] + h[i][2 * j + 1];
        }
      }
    }
    s = warp_sum(s);
    __syncthreads();
    if ((tid & 31) == 0) red[0][tid >> 5] = s;
    __syncthreads();
    const float mean = (red[0][0] + red[0][1] + red[0][2] + red[0][3]) * inv_d;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int v = tid + i * 128;
      if (v < vpr) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float dlt = h[i][j] - mean;
          ss += dlt * dlt;
        }
      }
    }
    ss = warp_sum(ss);
    if ((tid & 31) == 0) red[1][tid >> 5] = ss;
    __syncthreads();
    const float rstd = 1.0f / sqrtf((red[1][0] + red[1][1] + red[1][2] + red[1][3]) * inv_d + eps);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int v = tid + i * 128;
      if (v < vpr) {
        const uint4 qw = __ldg(w + v), qb = __ldg(b + v);
        const uint32_t aw[4] = {qw.x, qw.y, qw.z, qw.w}, ab[4] = {qb.x, qb.y, qb.z, qb.w};
        float o[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          o[2 * j] = (h[i][2 * j] - mean) * rstd * bf16_lo(aw[j]) + bf16_lo(ab[j]);
          o[2 * j + 1] = (h[i][2 * j + 1] - mean) * rstd * bf16_hi(aw[j]) + bf16_hi(ab[j]);
        }
        out[r * vpr + v] = make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
      }
    }
  }
}

__global__ void rope_table_kernel(const float* __restrict__ inv_freq, __nv_bfloat16* __restrict__ cos_out,
                                  __nv_bfloat16* __restrict__ sin_out, int n_pos, int hd) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<int64_t>(n_pos) * hd) return;
  const int pos = static_cast<int>(i / hd), d = static_cast<int>(i % hd);
  const float ang = static_cast<float>(pos) * inv_freq[d % (hd / 2)];  // emb = cat(freqs, freqs)
  cos_out[i] = __float2bfloat16_rn(cosf(ang));
  sin_out[i] = __float2bfloat16_rn(sinf(ang));
}

__global__ void __launch_bounds__(256) embedding_kernel(const int64_t* __restrict__ ids, const uint4* __restrict__ table,
                                                        uint4* __restrict__ out, int64_t n, int vpr) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * wpb + (threadIdx.x >> 5); r < n;
       r += static_cast<int64_t>(gridDim.x) * wpb) {
    const uint4* src = table + ids[r] * vpr;
    for (int v = lane; v < vpr; v += 32) out[r * vpr + v] = __ldg(src + v);
  }
}

// Single block: exclusive scan of (ids == image_token) gives each image slot its feature row (masked_scatter
// consumes the source in order), then rows are copied.
__global__ void __launch_bounds__(1024) merge_kernel(const int64_t* __restrict__ ids, int64_t image_token,
                                                     const uint4* __restrict__ feats, uint4* __restrict__ embeds,
                                                     int32_t* __restrict__ count_out, int64_t n, int vpr) {
  __shared__ int warp_cnt[32];
  __shared__ int running_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) running_s = 0;
  __syncthreads();
  for (int64_t start = 0; start < n; start += blockDim.x) {
    const int64_t i = start + threadIdx.x;
    const bool hit = i < n && ids[i] == image_token;
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) warp_cnt[warp] = __popc(m);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 32; ++w) {
      const int c = warp_cnt[w];
      if (w < warp) before += c;
      total += c;
    }
    const int slot = running_s + before + __popc(m & ((1u << lane) - 1));
    // every thread of the warp helps copy the rows of its warp's hits
    for (int src_lane = 0; src_lane < 32; ++src_lane) {
      if ((m >> src_lane) & 1u) {
        const int s = __shfl_sync(0xffffffffu, slot, src_lane);
        const int64_t row = start + warp * 32 + src_lane;
        for (int v = lane; v < vpr; v += 32) embeds[row * vpr + v] = __ldg(feats + static_cast<int64_t>(s) * vpr + v);
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) running_s += total;
    __syncthreads();
  }
  if (threadIdx.x == 0 && count_out) *count_out = running_s;
}

// Multi-block variant for prompts of up to 16384 tokens: one warp per token; a warp whose token is an image slot counts the
// image tokens in front of it (lanes stride over ids[0..t)) to find its feature row, then copies the row.  The single-block kernel
// above copies the 256 x 5 KB rows of a cfg-2 prompt with ONE SM: 86 us per step in profiles/r02_launch_shares_final.txt.
__global__ void __launch_bounds__(256) merge_rows_kernel(const int64_t* __restrict__ ids, int64_t image_token,
                                                         const uint4* __restrict__ feats, uint4* __restrict__ embeds,
                                                         int32_t* __restrict__ count_out, int64_t n, int vpr) {
  const int lane = threadIdx.x & 31;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (t >= n) return;
  const bool hit = ids[t] == image_token;
  const bool last = t == n - 1;
  if (!hit && !(last && count_out)) return;
  int c = 0;
  for (int64_t i = lane; i < t; i += 32) c += ids[i] == image_token;
#pragma unroll
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (hit)
    for (int v = lane; v < vpr; v += 32) embeds[t * vpr + v] = __ldg(feats + static_cast<int64_t>(c) * vpr + v);
  if (last && count_out && lane == 0) *count_out = c + (hit ? 1 : 0);
}

// patches[(b*Np + py*Nside + px), c*P*P + i*P + j] = pixels[b, c, py*P + i, px*P + j]; k_pad zero padded.
__global__ void im2col_kernel(const __nv_bfloat16* __restrict__ pix, __nv_bfloat16* __restrict__ out, int B, int S, int P,
                              int k_pad) {
  const int nside = S / P;
  const int64_t total = static_cast<int64_t>(B) * nside * nside * k_pad;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int kk = static_cast<int>(i % k_pad);
    const int64_t patch = i / k_pad;
    __nv_bfloat16 v = __float2bfloat16_rn(0.f);
    if (kk < 3 * P * P) {
      const int c = kk / (P * P), rem = kk % (P * P), ii = rem / P, jj = rem % P;
      const int px = static_cast<int>(patch % nside), py = static_cast<int>((patch / nside) % nside);
      const int b = static_cast<int>(patch / (static_cast<int64_t>(nside) * nside));
      v = pix[((static_cast<int64_t>(b) * 3 + c) * S + (py * P + ii)) * S + (px * P + jj)];
    }
    out[i] = v;
  }
}

__global__ void __launch_bounds__(256) add_pos_kernel(const uint4* __restrict__ x, const int64_t* __restrict__ pos,
                                                      const uint4* __restrict__ table, uint4* __restrict__ out, int64_t rows,
                                                      int vpr) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * wpb + (threadIdx.x >> 5); r < rows;
       r += static_cast<int64_t>(gridDim.x) * wpb) {
    const uint4* t = table + pos[r] * vpr;
    for (int v = lane; v < vpr; v += 32) {
      const uint4 a = x[r * vpr + v], b = __ldg(t + v);
      const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        o[j] = pack_bf16(bf16_lo(aw[j]) + bf16_lo(bw[j]), bf16_hi(aw[j]) + bf16_hi(bw[j]));
      out[r * vpr + v] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}


// Backward of rmsnorm_kernel without residual (LlamaRMSNorm autograd): y = w o bf16(x r), r = rsqrt(mean(x^2) + eps).
//   dx = r (g - x r^2 mean(g o x)) (+ dres),  g = dy o w;   dw = sum_rows dy o bf16(x r)
// One 128-thread block per row (grid-stride over rows); dw is accumulated per block in registers and written as fp32 partials
// [gridDim.x][d] that rmsnorm_dw_reduce_kernel sums in a fixed order: deterministic, no atomics.
constexpr int RMS_BWD_BLOCKS = 256;  // fixed, so that the workspace size does not depend on the device
template <int MAXV>
__global__ void __launch_bounds__(128) rmsnorm_bwd_kernel(const uint4* __restrict__ x, const uint4* __restrict__ w,
                                                          const uint4* __restrict__ dy, const uint4* __restrict__ dres,
                                                          uint4* __restrict__ dx, float* __restrict__ partial, int64_t rows, int vpr,
                                                          float eps, float inv_d) {
  __shared__ float red[2][4];
  const int tid = threadIdx.x;
  float dw[MAXV][8];
#pragma unroll
  for (int i = 0; i < MAXV; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) dw[i][j] = 0.f;
  for (int64_t r = blockIdx.x; r < rows; r += gridDim.x) {
    float h[MAXV][8], g[MAXV][8];
    float ss = 0.f, sg = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int v = tid + i * 128;
      if (v < vpr) {
        const uint4 qx = x[r * vpr + v], qy = dy[r * vpr + v], qw = __ldg(w + v);
        const uint32_t a[4] = {qx.x, qx.y, qx.z, qx.w}, b[4] = {qy.x, qy.y, qy.z, qy.w}, c[4] = {qw.x, qw.y, qw.z, qw.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          h[i][2 * j] = bf16_lo(a[j]);
          h[i][2 * j + 1] = bf16_hi(a[j]);
          g[i][2 * j] = bf16_lo(b[j]);       // dy for now; g = dy o w below
          g[i][2 * j + 1] = bf16_hi(b[j]);
          const float w0 = bf16_lo(c[j]), w1 = bf16_hi(c[j]);
          ss += h[i][2 * j] * h[i][2 * j] + h[i][2 * j + 1] * h[i][2 * j + 1];
          sg += g[i][2 * j] * w0 * h[i][2 * j] + g[i][2 * j + 1] * w1 * h[i][2 * j + 1];
        }
      }
    }
    ss = warp_sum(ss);
    sg = warp_sum(sg);
    __syncthreads();  // red[] free (previous row consumed)
    if ((tid & 31) == 0) {
      red[0][tid >> 5] = ss;
      red[1][tid >> 5] = sg;
    }
    __syncthreads();
    ss = red[0][0] + red[0][1] + red[0][2] + red[0][3];
    sg = red[1][0] + red[1][1] + red[1][2] + red[1][3];
    const float rstd = 1.0f / sqrtf(ss * inv_d + eps);   // as the forward computes it
    const float c2 = rstd * rstd * sg * inv_d;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int v = tid + i * 128;
      if (v < vpr) {
        const uint4 qw = __ldg(w + v);
        const uint32_t c[4] = {qw.x, qw.y, qw.z, qw.w};
        float res[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (dres) {
          const uint4 qr = dres[r * vpr + v];
          const uint32_t e[4] = {qr.x, qr.y, qr.z, qr.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            res[2 * j] = bf16_lo(e[j]);
            res[2 * j + 1] = bf16_hi(e[j]);
          }
        }
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float wj = (j & 1) ? bf16_hi(c[j >> 1]) : bf16_lo(c[j >> 1]);
          dw[i][j] += g[i][j] * bf16r(h[i][j] * rstd);
          o[j] = rstd * (g[i][j] * wj - h[i][j] * c2) + res[j];
        }
        dx[r * vpr + v] = make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
      }
    }
  }
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int v = tid + i * 128;
    if (v < vpr) {
      float4* dst = reinterpret_cast<float4*>(partial + static_cast<int64_t>(blockIdx.x) * vpr * 8 + v * 8);
      dst[0] = make_float4(dw[i][0], dw[i][1], dw[i][2], dw[i][3]);
      dst[1] = make_float4(dw[i][4], dw[i][5], dw[i][6], dw[i][7]);
    }
  }
}

// dw[c] = bf16(sum_b partial[b][c]), blocks summed in index order
__global__ void __launch_bounds__(256) rmsnorm_dw_reduce_kernel(const float* __restrict__ partial, __nv_bfloat16* __restrict__ dw,
                                                                int n_part, int d) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= d) return;
  float s = 0.f;
  for (int b = 0; b < n_part; ++b) s += partial[static_cast<int64_t>(b) * d + c];
  dw[c] = __float2bfloat16_rn(s);
}

// Transpose of rotate-half RoPE, in place on token-major [rows, n_heads*128]: dx1 = dy1 c + dy2 s, dx2 = dy2 c - dy1 s.
// One warp per (row, head); lane l owns dims 2l, 2l+1 of each half.
__global__ void __launch_bounds__(256) rope_bwd_kernel(uint32_t* __restrict__ x, const uint32_t* __restrict__ cos_t,
                                                       const uint32_t* __restrict__ sin_t, const int32_t* __restrict__ position_ids,
                                                       int64_t rows, int n_heads, int rows_per_batch) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (wid >= rows * n_heads) return;
  const int64_t r = wid / n_heads;
  const int pos = position_ids ? position_ids[r] : static_cast<int>(r % rows_per_batch);
  uint32_t* row = x + wid * 64;                    // 128 bf16 = 64 words
  const uint32_t* cs = cos_t + static_cast<int64_t>(pos) * 64;
  const uint32_t* sn = sin_t + static_cast<int64_t>(pos) * 64;
  const uint32_t a = row[lane], b = row[32 + lane];
  const uint32_t c1 = __ldg(cs + lane), c2 = __ldg(cs + 32 + lane), s1 = __ldg(sn + lane), s2 = __ldg(sn + 32 + lane);
  const float y1[2] = {bf16_lo(a), bf16_hi(a)}, y2[2] = {bf16_lo(b), bf16_hi(b)};
  const float co1[2] = {bf16_lo(c1), bf16_hi(c1)}, co2[2] = {bf16_lo(c2), bf16_hi(c2)};
  const float si1[2] = {bf16_lo(s1), bf16_hi(s1)}, si2[2] = {bf16_lo(s2), bf16_hi(s2)};
  float o1[2], o2[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    // forward: out1 = x1 c1 - x2 s1, out2 = x2 c2 + x1 s2
    o1[u] = y1[u] * co1[u] + y2[u] * si2[u];
    o2[u] = y2[u] * co2[u] - y1[u] * si1[u];
  }
  row[lane] = pack_bf16(o1[0], o1[1]);
  row[32 + lane] = pack_bf16(o2[0], o2[1]);
}

}  // namespace aria

using namespace aria;

extern "C" int aria_rmsnorm(const void* x, const void* residual, const void* weight, void* out, void* sum_out, int64_t rows,
                            int32_t d, float eps, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(x && weight && out && d % 8 == 0 && d <= 128 * 8 * 4 && rows >= 0);
  if (rows == 0) return ARIA_OK;
  const int vpr = d / 8;
  int64_t grid64 = rows;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  if (grid64 > cap) grid64 = cap;
  const int grid = static_cast<int>(grid64);
#define RMS(MAXV)                                                                                                   \
  rmsnorm_kernel<MAXV><<<grid, 128, 0, stream>>>(static_cast<const uint4*>(x), static_cast<const uint4*>(residual), \
                                                 static_cast<const uint4*>(weight), static_cast<uint4*>(out),       \
                                                 static_cast<uint4*>(sum_out), rows, vpr, eps, 1.0f / d)
  if (vpr <= 128) RMS(1);
  else if (vpr <= 256) RMS(2);
  else if (vpr <= 384) RMS(3);
  else RMS(4);
#undef RMS
  return check_launch("rmsnorm_kernel");
}

extern "C" int aria_layernorm(const void* x, const void* weight, const void* bias, void* out, int64_t rows, int32_t d,
                              float eps, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(x && weight && bias && out && d % 8 == 0 && d <= 128 * 8 * 4 && rows >= 0);
  if (rows == 0) return ARIA_OK;
  const int vpr = d / 8;
  if (vpr <= 160 && rows >= 1024) {  // many short rows (the ViT): one warp per row
    layernorm_warp_kernel<5><<<static_cast<int>((rows + 7) / 8), 256, 0, stream>>>(
        static_cast<const uint4*>(x), static_cast<const uint4*>(weight), static_cast<const uint4*>(bias), static_cast<uint4*>(out), rows,
        vpr, eps, 1.0f / d);
    return check_launch("layernorm_warp_kernel");
  }
  int64_t grid64 = rows;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  if (grid64 > cap) grid64 = cap;
  const int grid = static_cast<int>(grid64);
#define LN(MAXV)                                                                                                    \
  layernorm_kernel<MAXV><<<grid, 128, 0, stream>>>(static_cast<const uint4*>(x), static_cast<const uint4*>(weight), \
                                                   static_cast<const uint4*>(bias), static_cast<uint4*>(out), rows, vpr, eps, 1.0f / d)
  if (vpr <= 128) LN(1);
  else if (vpr <= 256) LN(2);
  else if (vpr <= 384) LN(3);
  else LN(4);
#undef LN
  return check_launch("layernorm_kernel");
}

extern "C" int aria_rope_table(const float* inv_freq, void* cos_out, void* sin_out, int32_t n_pos, int32_t head_dim,
                               aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(inv_freq && cos_out && sin_out && n_pos > 0 && head_dim > 0 && head_dim % 2 == 0);
  const int64_t n = static_cast<int64_t>(n_pos) * head_dim;
  rope_table_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(inv_freq, static_cast<__nv_bfloat16*>(cos_out),
                                                                          static_cast<__nv_bfloat16*>(sin_out), n_pos, head_dim);
  return check_launch("rope_table_kernel");
}

extern "C" int aria_embedding(const int64_t* ids, const void* table, void* out, int64_t n, int32_t d, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(ids && table && out && d % 8 == 0 && n >= 0);
  if (n == 0) return ARIA_OK;
  embedding_kernel<<<rows_grid(n, 8), 256, 0, stream>>>(ids, static_cast<const uint4*>(table), static_cast<uint4*>(out), n, d / 8);
  return check_launch("embedding_kernel");
}

extern "C" int aria_merge_image_features(const int64_t* ids, int64_t image_token, const void* features, void* embeds,
                                         int32_t* count_out, int64_t n, int32_t d, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(ids && features && embeds && d % 8 == 0 && n >= 0);
  if (n == 0) return ARIA_OK;
  if (n <= 16384) {
    merge_rows_kernel<<<static_cast<int>((n + 7) / 8), 256, 0, stream>>>(ids, image_token, static_cast<const uint4*>(features),
                                                                         static_cast<uint4*>(embeds), count_out, n, d / 8);
    return check_launch("merge_rows_kernel");
  }
  merge_kernel<<<1, 1024, 0, stream>>>(ids, image_token, static_cast<const uint4*>(features), static_cast<uint4*>(embeds),
                                       count_out, n, d / 8);
  return check_launch("merge_kernel");
}

extern "C" int aria_im2col_patches(const void* pixels, void* patches, int32_t B, int32_t S, int32_t P, int32_t k_pad,
                                   aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(pixels && patches && B > 0 && S > 0 && P > 0 && S % P == 0 && k_pad >= 3 * P * P && k_pad % 8 == 0);
  im2col_kernel<<<sm_count() * 8, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(pixels),
                                                    static_cast<__nv_bfloat16*>(patches), B, S, P, k_pad);
  return check_launch("im2col_kernel");
}

extern "C" int aria_add_pos_embedding(const void* x, const int64_t* pos_ids, const void* table, void* out, int64_t rows,
                                      int32_t d, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(x && pos_ids && table && out && d % 8 == 0 && rows >= 0);
  if (rows == 0) return ARIA_OK;
  add_pos_kernel<<<rows_grid(rows, 8), 256, 0, stream>>>(static_cast<const uint4*>(x), pos_ids, static_cast<const uint4*>(table),
                                                         static_cast<uint4*>(out), rows, d / 8);
  return check_launch("add_pos_kernel");
}

// Lets kernels launched on the current device load/store memory of `peer_device` (NVLink P2P); idempotent.
extern "C" int aria_enable_peer_access(int32_t peer_device) {
  int cur = 0;
  if (cudaGetDevice(&cur) != cudaSuccess) return ARIA_ERR_CUDA;
  if (cur == peer_device) return ARIA_OK;
  int can = 0;
  if (cudaDeviceCanAccessPeer(&can, cur, peer_device) != cudaSuccess || !can) return ARIA_ERR_UNSUPPORTED;
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {
    cudaGetLastError();
    return ARIA_OK;
  }
  return e == cudaSuccess ? ARIA_OK : ARIA_ERR_CUDA;
}

// CUDA IPC plumbing for peer-mapped buffers (one arena per rank).  export: handle of the cudaMalloc allocation that
// contains `ptr` + byte offset of `ptr` inside it.  open: maps a peer's allocation into the CURRENT device's context with
// lazy peer access, so that kernels on this GPU can load/store it over NVLink.
extern "C" int aria_ipc_export(const void* ptr, void* handle64, int64_t* offset_out) {
  ARIA_CHECK_ARG(ptr && handle64 && offset_out);
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, const_cast<void*>(ptr)) != cudaSuccess) {
    fprintf(stderr, "aria_b200: cudaIpcGetMemHandle failed: %s\n", cudaGetErrorString(cudaGetLastError()));
    return ARIA_ERR_CUDA;
  }
  memcpy(handle64, &h, sizeof(h));
  typedef CUresult (*PFN_range)(CUdeviceptr*, size_t*, CUdeviceptr);
  static PFN_range fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return ARIA_ERR_CUDA;
    fn = reinterpret_cast<PFN_range>(p);
  }
  CUdeviceptr base = 0;
  size_t size = 0;
  if (fn(&base, &size, reinterpret_cast<CUdeviceptr>(ptr)) != CUDA_SUCCESS) return ARIA_ERR_CUDA;
  *offset_out = static_cast<int64_t>(reinterpret_cast<CUdeviceptr>(ptr) - base);
  return ARIA_OK;
}

extern "C" int aria_ipc_open(const void* handle64, void** base_out) {
  ARIA_CHECK_ARG(handle64 && base_out);
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof(h));
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) {
    fprintf(stderr, "aria_b200: cudaIpcOpenMemHandle failed: %s\n", cudaGetErrorString(e));
    cudaGetLastError();
    return ARIA_ERR_CUDA;
  }
  *base_out = p;
  return ARIA_OK;
}

extern "C" int aria_ipc_close(void* base) {
  return cudaIpcCloseMemHandle(base) == cudaSuccess ? ARIA_OK : ARIA_ERR_CUDA;
}

extern "C" int64_t aria_rmsnorm_bwd_workspace_bytes(int64_t rows, int32_t d) {
  if (rows <= 0 || d <= 0 || d % 8) return ARIA_ERR_BAD_ARG;
  const int64_t blocks = rows < RMS_BWD_BLOCKS ? rows : RMS_BWD_BLOCKS;
  return blocks * d * static_cast<int64_t>(sizeof(float));
}

extern "C" int aria_rmsnorm_bwd(const void* x, const void* weight, const void* dy, const void* dres, void* dx, void* dw, int64_t rows,
                                int32_t d, float eps, void* workspace, int64_t workspace_bytes, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(x && weight && dy && dx && dw && workspace && d > 0 && d % 8 == 0 && d <= 128 * 8 * 4 && rows > 0);
  ARIA_CHECK_ARG(workspace_bytes >= aria_rmsnorm_bwd_workspace_bytes(rows, d));
  const int vpr = d / 8;
  const int grid = static_cast<int>(rows < RMS_BWD_BLOCKS ? rows : RMS_BWD_BLOCKS);
  float* partial = static_cast<float*>(workspace);
#define RMSB(MAXV)                                                                                                          \
  rmsnorm_bwd_kernel<MAXV><<<grid, 128, 0, stream>>>(static_cast<const uint4*>(x), static_cast<const uint4*>(weight),       \
                                                     static_cast<const uint4*>(dy), static_cast<const uint4*>(dres),        \
                                                     static_cast<uint4*>(dx), partial, rows, vpr, eps, 1.0f / d)
  if (vpr <= 128) RMSB(1);
  else if (vpr <= 256) RMSB(2);
  else if (vpr <= 384) RMSB(3);
  else RMSB(4);
#undef RMSB
  int rc = check_launch("rmsnorm_bwd_kernel");
  if (rc) return rc;
  rmsnorm_dw_reduce_kernel<<<(d + 255) / 256, 256, 0, stream>>>(partial, static_cast<__nv_bfloat16*>(dw), grid, d);
  return check_launch("rmsnorm_dw_reduce_kernel");
}

extern "C" int aria_rope_bwd(void* x, const void* cos_t, const void* sin_t, const int32_t* position_ids, int64_t rows,
                             int32_t n_heads, int32_t rows_per_batch, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(x && cos_t && sin_t && rows >= 0 && n_heads > 0 && (position_ids || rows_per_batch > 0));
  if (rows == 0) return ARIA_OK;
  const int64_t warps = rows * n_heads;
  rope_bwd_kernel<<<static_cast<unsigned>((warps + 7) / 8), 256, 0, stream>>>(
      static_cast<uint32_t*>(x), static_cast<const uint32_t*>(cos_t), static_cast<const uint32_t*>(sin_t), position_ids, rows, n_heads,
      rows_per_batch);
  return check_launch("rope_bwd_kernel");
}
