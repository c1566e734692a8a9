// Training-side loss head and embedding gradient:
//
//   aria_lm_xent_fwd / aria_lm_xent_bwd: lm_head + shifted cross-entropy (modeling_aria.py:300-323: nn.CrossEntropyLoss over
//     lm_head(h).float()) without ever materialising the [M, V] logits.  The forward is one tcgen05 GEMM whose epilogue
//     (XENT_STATS, gemm_common.cuh) reduces each 64-column slice of a row to a (max, sum exp) partial, then a row kernel merges
//     the partials into lse and the loss.  The backward walks the vocabulary in chunks: a GEMM recomputes the chunk's logits
//     and its epilogue (XENT_GRAD) stores d loss / d logits as bf16; the wgrad kernel turns that into the chunk's rows of dW;
//     a dense GEMM (W read MN-major, ACC_F32 epilogue) adds chunk @ W[chunk] into an fp32 dh, rounded once at the end.
//   aria_embedding_bwd: the gradient of nn.Embedding as a stable counting sort of (id, position) and one block per distinct id
//     summing its rows in position order — bit-reproducible, no atomics on values.
//
// Everything is launched from C on the caller's stream: no allocation, no host sync, graph-capturable.
#include <string.h>

#include "gemm_common.cuh"

namespace aria {
int gemm_run(const aria_gemm_desc_t* d, int epi, const XentParams* xp, cudaStream_t stream);  // gemm.cu
}

namespace {
using namespace aria;

constexpr int64_t kAlign = 256;
inline int64_t al(int64_t n) { return (n + kAlign - 1) / kAlign * kAlign; }
constexpr float kL2E = 1.4426950408889634f;
constexpr int XENT_ROWS = 128;                                   // rows per block of the merge kernel
constexpr int64_t kBwdChunkBudget = int64_t(512) << 20;          // default bf16 chunk buffer of the backward

struct FwdWs {
  int64_t part, tlogit, blk_sum, blk_cnt, total;
};
FwdWs fwd_ws(int64_t M, int64_t V) {
  FwdWs w{};
  const int64_t slots = (V + XENT_SLOT - 1) / XENT_SLOT, nblk = (M + XENT_ROWS - 1) / XENT_ROWS;
  int64_t o = 0;
  w.part = o;    o += al(slots * M * 8);
  w.tlogit = o;  o += al(M * 4);
  w.blk_sum = o; o += al(nblk * 4);
  w.blk_cnt = o; o += al(nblk * 4);
  w.total = o;
  return w;
}

// fixed part of the backward workspace: [0, M] row offsets of the wgrad launch, then the fp32 dh accumulator
int64_t bwd_fixed(int64_t M, int64_t d) { return al(16) + al(M * d * 4); }

// One thread per row: merge the (max, sum) partials in slot order -> lse; loss contribution lse - z_target of a valid row
// (target >= V: NaN); per-block sums in a fixed order.
__global__ void __launch_bounds__(XENT_ROWS) xent_rows_kernel(const float2* __restrict__ part, const float* __restrict__ tlogit,
                                                              const int32_t* __restrict__ target, float* __restrict__ lse,
                                                              float* __restrict__ blk_sum, int32_t* __restrict__ blk_cnt, int64_t M,
                                                              int V, int slots) {
  __shared__ float ss[XENT_ROWS];
  __shared__ int sc[XENT_ROWS];
  const int64_t r = static_cast<int64_t>(blockIdx.x) * XENT_ROWS + threadIdx.x;
  float contrib = 0.f;
  int cnt = 0;
  if (r < M) {
    float m = -INFINITY, l = 0.f;
    for (int s = 0; s < slots; ++s) {
      const float2 ps = part[static_cast<int64_t>(s) * M + r];
      if (ps.x == -INFINITY) continue;
      if (ps.x > m) {
        l = l * exp2f((m - ps.x) * kL2E) + ps.y;
        m = ps.x;
      } else {
        l += ps.y * exp2f((ps.x - m) * kL2E);
      }
    }
    const float lr = m + logf(l);
    lse[r] = lr;
    const int t = target[r];
    if (t >= 0) {
      cnt = 1;
      contrib = t < V ? lr - tlogit[r] : NAN;
    }
  }
  ss[threadIdx.x] = contrib;
  sc[threadIdx.x] = cnt;
  __syncthreads();
  for (int w = XENT_ROWS / 2; w; w >>= 1) {
    if (threadIdx.x < w) {
      ss[threadIdx.x] += ss[threadIdx.x + w];
      sc[threadIdx.x] += sc[threadIdx.x + w];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    blk_sum[blockIdx.x] = ss[0];
    blk_cnt[blockIdx.x] = sc[0];
  }
}

// Single block: loss = sum / n_valid over the per-block partials (fixed order; 0 valid rows -> 0/0 = NaN, as torch).
__global__ void __launch_bounds__(256) xent_final_kernel(const float* __restrict__ blk_sum, const int32_t* __restrict__ blk_cnt,
                                                         int nblk, float* __restrict__ loss, int32_t* __restrict__ n_valid) {
  __shared__ float ss[256];
  __shared__ int sc[256];
  float s = 0.f;
  int c = 0;
  for (int i = threadIdx.x; i < nblk; i += 256) {
    s += blk_sum[i];
    c += blk_cnt[i];
  }
  ss[threadIdx.x] = s;
  sc[threadIdx.x] = c;
  __syncthreads();
  for (int w = 128; w; w >>= 1) {
    if (threadIdx.x < w) {
      ss[threadIdx.x] += ss[threadIdx.x + w];
      sc[threadIdx.x] += sc[threadIdx.x + w];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *loss = ss[0] / static_cast<float>(sc[0]);
    *n_valid = sc[0];
  }
}

__global__ void xent_offsets_kernel(int32_t* offs, int32_t M) {
  offs[0] = 0;
  offs[1] = M;
}

// ---------------------------------------------------------------------------------------------------- embedding backward
// key of a position: its id, or `vocab` (a bucket that is never summed) for skipped / out-of-range ids
__device__ __forceinline__ int emb_key(int64_t id, int64_t skip_id, int64_t vocab) {
  return (id < 0 || id >= vocab || id == skip_id) ? static_cast<int>(vocab) : static_cast<int>(id);
}

__global__ void __launch_bounds__(256) emb_count_kernel(const int64_t* __restrict__ ids, int32_t* __restrict__ counts, int64_t n,
                                                        int64_t skip_id, int64_t vocab) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * 256 + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * 256)
    atomicAdd(&counts[emb_key(ids[i], skip_id, vocab)], 1);  // integer counts: order-independent
}

// Single block: exclusive scan of counts[nb] -> offsets[nb + 1] and cursor[nb] (= offsets).
__global__ void __launch_bounds__(1024) emb_scan_kernel(const int32_t* __restrict__ counts, int32_t* __restrict__ offsets,
                                                        int32_t* __restrict__ cursor, int nb) {
  __shared__ int part[1024];
  const int per = (nb + 1023) / 1024;
  const int b = threadIdx.x * per, e = min(nb, b + per);
  int s = 0;
  for (int i = b; i < e; ++i) s += counts[i];
  part[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
    const int v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  int run = part[threadIdx.x] - s;
  for (int i = b; i < e; ++i) {
    offsets[i] = run;
    cursor[i] = run;
    run += counts[i];
  }
  if (threadIdx.x == 1023) offsets[nb] = part[1023];
}

// One warp, positions in order, 32 at a time: equal keys inside a step get consecutive slots in lane order, so every bucket
// lists its positions in ascending order (a stable scatter, independent of scheduling).
__global__ void __launch_bounds__(32) emb_scatter_kernel(const int64_t* __restrict__ ids, int32_t* cursor, int32_t* __restrict__ sorted,
                                                         int64_t n, int64_t skip_id, int64_t vocab) {
  const int lane = threadIdx.x;
  for (int64_t i0 = 0; i0 < n; i0 += 32) {
    const int64_t i = i0 + lane;
    const bool ok = i < n;
    const int key = ok ? emb_key(ids[i], skip_id, vocab) : -1;
    const unsigned same = __match_any_sync(0xffffffffu, key);
    const int rank = __popc(same & ((1u << lane) - 1));
    const int base = ok ? cursor[key] : 0;
    __syncwarp();
    if (ok) {
      sorted[base + rank] = static_cast<int32_t>(i);
      if (rank == 0) cursor[key] = base + __popc(same);
    }
    __syncwarp();
  }
}

// One block per bucket head: dtable[id] = bf16(sum over the bucket's positions, in order, of dout[p]) in fp32.
template <int MAXV>
__global__ void __launch_bounds__(128) emb_sum_kernel(const int64_t* __restrict__ ids, const int32_t* __restrict__ sorted,
                                                      const int32_t* __restrict__ offsets, const uint4* __restrict__ dout,
                                                      uint4* __restrict__ dtable, int64_t skip_id, int64_t vocab, int vpr) {
  const int j = blockIdx.x;
  const int n_kept = offsets[vocab];
  if (j >= n_kept) return;
  const int key = emb_key(ids[sorted[j]], skip_id, vocab);
  if (j > 0 && emb_key(ids[sorted[j - 1]], skip_id, vocab) == key) return;  // not the first position of its bucket
  const int end = offsets[key + 1];
  float acc[MAXV][8];
#pragma unroll
  for (int u = 0; u < MAXV; ++u)
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[u][e] = 0.f;
  for (int q = j; q < end; ++q) {
    const int64_t row = sorted[q];
#pragma unroll
    for (int u = 0; u < MAXV; ++u) {
      const int v = threadIdx.x + u * 128;
      if (v < vpr) {
        const uint4 x = __ldg(dout + row * vpr + v);
        const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          acc[u][2 * e] += bf16_lo(w[e]);
          acc[u][2 * e + 1] += bf16_hi(w[e]);
        }
      }
    }
  }
#pragma unroll
  for (int u = 0; u < MAXV; ++u) {
    const int v = threadIdx.x + u * 128;
    if (v < vpr)
      dtable[static_cast<int64_t>(key) * vpr + v] = make_uint4(pack_bf16(acc[u][0], acc[u][1]), pack_bf16(acc[u][2], acc[u][3]),
                                                               pack_bf16(acc[u][4], acc[u][5]), pack_bf16(acc[u][6], acc[u][7]));
  }
}

struct EmbWs {
  int64_t counts, offsets, cursor, sorted, total;
};
EmbWs emb_ws(int64_t n, int64_t vocab) {
  EmbWs w{};
  int64_t o = 0;
  w.counts = o;  o += al((vocab + 1) * 4);
  w.offsets = o; o += al((vocab + 2) * 4);
  w.cursor = o;  o += al((vocab + 1) * 4);
  w.sorted = o;  o += al(n * 4);
  w.total = o;
  return w;
}

}  // namespace

extern "C" int64_t aria_lm_xent_fwd_workspace_bytes(int64_t M, int64_t V) {
  if (M < 0 || V <= 0 || V % 8 || V >= (int64_t(1) << 31) || M >= (int64_t(1) << 31)) return ARIA_ERR_BAD_ARG;
  return fwd_ws(M, V).total;
}

extern "C" int aria_lm_xent_fwd(const void* h, const void* w, const int32_t* target, float* lse, float* loss, int32_t* n_valid,
                                int64_t M, int64_t V, int32_t d, void* workspace, int64_t workspace_bytes, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(h && w && target && lse && loss && n_valid && workspace);
  ARIA_CHECK_ARG(d > 0 && d % 8 == 0 && M >= 0 && M < (int64_t(1) << 31) && V > 0 && V % 8 == 0 && V < (int64_t(1) << 31));
  ARIA_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 15) == 0);
  const FwdWs ws = fwd_ws(M, V);
  ARIA_CHECK_ARG(workspace_bytes >= ws.total);
  if (M == 0) return ARIA_OK;
  uint8_t* base = static_cast<uint8_t*>(workspace);
  XentParams x{};
  x.target = target;
  x.part = reinterpret_cast<float2*>(base + ws.part);
  x.tlogit = reinterpret_cast<float*>(base + ws.tlogit);
  x.M = M;
  x.V = static_cast<int>(V);
  aria_gemm_desc_t g;
  memset(&g, 0, sizeof(g));
  g.a = h; g.lda = d; g.m = M; g.n = V; g.k = d;
  g.b[0] = w; g.n_seg = 1; g.b_layout = ARIA_B_NK; g.num_groups = 1;
  g.out[0] = workspace;  // not written by this epilogue
  int rc = gemm_run(&g, EPI_XENT_STATS, &x, stream);
  if (rc) return rc;
  const int nblk = static_cast<int>((M + XENT_ROWS - 1) / XENT_ROWS);
  float* blk_sum = reinterpret_cast<float*>(base + ws.blk_sum);
  int32_t* blk_cnt = reinterpret_cast<int32_t*>(base + ws.blk_cnt);
  xent_rows_kernel<<<nblk, XENT_ROWS, 0, stream>>>(x.part, x.tlogit, target, lse, blk_sum, blk_cnt, M, static_cast<int>(V),
                                                   static_cast<int>((V + XENT_SLOT - 1) / XENT_SLOT));
  if ((rc = check_launch("xent_rows_kernel"))) return rc;
  xent_final_kernel<<<1, 256, 0, stream>>>(blk_sum, blk_cnt, nblk, loss, n_valid);
  return check_launch("xent_final_kernel");
}

extern "C" int64_t aria_lm_xent_bwd_workspace_bytes(int64_t M, int64_t V, int32_t d) {
  if (M < 0 || V <= 0 || V % 8 || d <= 0 || d % 64) return ARIA_ERR_BAD_ARG;
  const int64_t v_pad = (V + 255) / 256 * 256;
  int64_t vc = M > 0 ? kBwdChunkBudget / (M * 2) / 256 * 256 : v_pad;
  if (vc < 256) vc = 256;
  if (vc > v_pad) vc = v_pad;
  return bwd_fixed(M, d) + al(M * vc * 2);
}

extern "C" int aria_lm_xent_bwd(const void* h, const void* w, const int32_t* target, const float* lse, const int32_t* n_valid,
                                const float* dloss, void* dh, void* dw, int64_t M, int64_t V, int32_t d, void* workspace,
                                int64_t workspace_bytes, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(h && w && target && lse && n_valid && dloss && dh && workspace);
  ARIA_CHECK_ARG(d > 0 && d % 64 == 0 && M >= 0 && M < (int64_t(1) << 31) && V > 0 && V % 8 == 0 && V < (int64_t(1) << 31));
  ARIA_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 15) == 0);
  const int64_t fixed = bwd_fixed(M, d);
  // chunk width: the largest multiple of 256 columns whose bf16 [M, Vc] buffer fits behind the fixed part, at least one tile
  const int64_t v_pad = (V + 255) / 256 * 256;
  int64_t vc = M > 0 && workspace_bytes > fixed ? (workspace_bytes - fixed) / (M * 2) / 256 * 256 : 0;
  if (vc > v_pad) vc = v_pad;
  ARIA_CHECK_ARG(M == 0 || vc >= 256);
  if (M == 0) return ARIA_OK;
  uint8_t* base = static_cast<uint8_t*>(workspace);
  int32_t* offs = reinterpret_cast<int32_t*>(base);
  float* acc = reinterpret_cast<float*>(base + al(16));
  void* chunk = base + fixed;
  xent_offsets_kernel<<<1, 1, 0, stream>>>(offs, static_cast<int32_t>(M));
  int rc = check_launch("xent_offsets_kernel");
  if (rc) return rc;
  const __nv_bfloat16* wb = static_cast<const __nv_bfloat16*>(w);
  for (int64_t v0 = 0; v0 < V; v0 += vc) {
    const int64_t vn = V - v0 < vc ? V - v0 : vc;
    const void* wc = wb + v0 * d;
    // 1. chunk = d loss / d z for columns [v0, v0 + vn)
    XentParams x{};
    x.target = target;
    x.lse = lse;
    x.dloss = dloss;
    x.n_valid = n_valid;
    x.M = M;
    x.V = static_cast<int>(V);
    x.v0 = static_cast<int>(v0);
    aria_gemm_desc_t g;
    memset(&g, 0, sizeof(g));
    g.a = h; g.lda = d; g.m = M; g.n = vn; g.k = d;
    g.b[0] = wc; g.n_seg = 1; g.b_layout = ARIA_B_NK; g.num_groups = 1;
    g.out[0] = chunk; g.ldo = vc;
    if ((rc = gemm_run(&g, EPI_XENT_GRAD, &x, stream))) return rc;
    // 2. dW[v0:v0+vn] = chunk^T h (disjoint rows of dW: nothing to accumulate)
    if (dw) {
      if ((rc = aria_grouped_wgrad(chunk, vc, h, d, static_cast<__nv_bfloat16*>(dw) + v0 * d, offs, M, vn, d, 1, 1, stream_))) return rc;
    }
    // 3. dh (+)= chunk @ W[v0:v0+vn]  (W as [K = vn, N = d], N contiguous), fp32 across chunks
    memset(&x, 0, sizeof(x));
    x.acc = acc;
    x.M = M;
    x.first = v0 == 0;
    x.last = v0 + vc >= V;
    memset(&g, 0, sizeof(g));
    g.a = chunk; g.lda = vc; g.m = M; g.n = d; g.k = vn;
    g.b[0] = wc; g.n_seg = 1; g.b_layout = ARIA_B_GKN; g.num_groups = 1;
    g.out[0] = dh; g.ldo = d;
    if ((rc = gemm_run(&g, EPI_ACC_F32, &x, stream))) return rc;
  }
  return ARIA_OK;
}

extern "C" int64_t aria_embedding_bwd_workspace_bytes(int64_t n, int64_t vocab) {
  if (n < 0 || vocab <= 0 || n >= (int64_t(1) << 31) || vocab >= (int64_t(1) << 31) - 2) return ARIA_ERR_BAD_ARG;
  return emb_ws(n, vocab).total;
}

extern "C" int aria_embedding_bwd(const int64_t* ids, const void* dout, void* dtable, int64_t n, int32_t d, int64_t vocab,
                                  int64_t skip_id, void* workspace, int64_t workspace_bytes, aria_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ARIA_CHECK_ARG(ids && dout && dtable && workspace);
  ARIA_CHECK_ARG(d > 0 && d % 8 == 0 && d <= 128 * 8 * 4 && n >= 0 && n < (int64_t(1) << 31) && vocab > 0 &&
                 vocab < (int64_t(1) << 31) - 2);
  const EmbWs ws = emb_ws(n, vocab);
  ARIA_CHECK_ARG(workspace_bytes >= ws.total);
  if (n == 0) return ARIA_OK;
  uint8_t* base = static_cast<uint8_t*>(workspace);
  int32_t* counts = reinterpret_cast<int32_t*>(base + ws.counts);
  int32_t* offsets = reinterpret_cast<int32_t*>(base + ws.offsets);
  int32_t* cursor = reinterpret_cast<int32_t*>(base + ws.cursor);
  int32_t* sorted = reinterpret_cast<int32_t*>(base + ws.sorted);
  if (cudaMemsetAsync(counts, 0, (vocab + 1) * 4, stream) != cudaSuccess) return ARIA_ERR_CUDA;
  int64_t cb = (n + 255) / 256;
  if (cb > sm_count() * 8) cb = sm_count() * 8;
  emb_count_kernel<<<static_cast<int>(cb), 256, 0, stream>>>(ids, counts, n, skip_id, vocab);
  int rc = check_launch("emb_count_kernel");
  if (rc) return rc;
  emb_scan_kernel<<<1, 1024, 0, stream>>>(counts, offsets, cursor, static_cast<int>(vocab + 1));
  if ((rc = check_launch("emb_scan_kernel"))) return rc;
  emb_scatter_kernel<<<1, 32, 0, stream>>>(ids, cursor, sorted, n, skip_id, vocab);
  if ((rc = check_launch("emb_scatter_kernel"))) return rc;
  const int vpr = d / 8;
#define EMB(MAXV)                                                                                                              \
  emb_sum_kernel<MAXV><<<static_cast<int>(n), 128, 0, stream>>>(ids, sorted, offsets, static_cast<const uint4*>(dout),       \
                                                                static_cast<uint4*>(dtable), skip_id, vocab, vpr)
  if (vpr <= 128) EMB(1);
  else if (vpr <= 256) EMB(2);
  else if (vpr <= 384) EMB(3);
  else EMB(4);
#undef EMB
  return check_launch("emb_sum_kernel");
}
