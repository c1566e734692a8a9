"""Torch-facing wrappers over the C ABI: tensors in, tensors out, raw pointers underneath.

PyTorch is used for device memory and streams only; every computation below is one of our CUDA kernels.
All wrappers launch on the current stream of the input's device and never synchronise.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib as L

bf16 = torch.bfloat16


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _chk(t: torch.Tensor, dtype=bf16, align: int = 16):
    if not t.is_cuda:
        raise RuntimeError("aria_b200 ops need CUDA tensors (there is no CPU path)")
    if t.dtype != dtype:
        raise RuntimeError(f"expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError("expected a contiguous tensor")
    if t.data_ptr() % align:
        raise RuntimeError(f"expected {align}-byte aligned storage")
    return t


# ------------------------------------------------------------------------------------------- GEMMs
def _run_gemm(d: L.GemmDesc, ref: torch.Tensor, what: str):
    with torch.cuda.device(ref.device):
        L.check(L.load().aria_gemm(C.byref(d), _stream(ref)), what)


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, act: int = L.ACT_NONE,
           residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """F.linear(x, weight, bias) -> act -> (+ residual); x [..., K], weight [N, K] (nn.Linear layout)."""
    _chk(x), _chk(weight)
    K = x.shape[-1]
    N = weight.shape[0]
    x2 = x.reshape(-1, K)
    M = x2.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=bf16, device=x.device)
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.n, d.k = x2.data_ptr(), K, M, N, K
    d.b[0] = weight.data_ptr()
    d.n_seg, d.b_layout, d.num_groups = 1, L.B_NK, 1
    d.epilogue, d.act = L.EPI_LINEAR, act
    if bias is not None:
        d.bias[0] = _chk(bias).data_ptr()
    if residual is not None:
        r2 = _chk(residual).reshape(-1, N)
        d.residual, d.ldr = r2.data_ptr(), N
    d.out[0], d.ldo = out.data_ptr(), N
    _run_gemm(d, x, "linear")
    return out.view(*x.shape[:-1], N)


def linear_multi(x: torch.Tensor, weights: Sequence[torch.Tensor]) -> torch.Tensor:
    """[x @ W0.T | x @ W1.T | ...] in one GEMM launch (up to 3 nn.Linear weights with equal out_features)."""
    _chk(x)
    K = x.shape[-1]
    N = weights[0].shape[0]
    x2 = x.reshape(-1, K)
    M = x2.shape[0]
    out = torch.empty((M, N * len(weights)), dtype=bf16, device=x.device)
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.n, d.k = x2.data_ptr(), K, M, N, K
    for s_, w in enumerate(weights):
        _chk(w)
        assert w.shape == weights[0].shape
        d.b[s_] = w.data_ptr()
    d.n_seg, d.b_layout, d.num_groups = len(weights), L.B_NK, 1
    d.epilogue = L.EPI_LINEAR
    d.out[0], d.ldo = out.data_ptr(), N * len(weights)
    _run_gemm(d, x, "linear_multi")
    return out


def linear_swiglu(x: torch.Tensor, gate_w: torch.Tensor, up_w: torch.Tensor) -> torch.Tensor:
    """silu(x @ gate_w.T) * (x @ up_w.T) in one GEMM (LlamaMLP front half, moe_lm.py:368-395)."""
    _chk(x), _chk(gate_w), _chk(up_w)
    K = x.shape[-1]
    N = gate_w.shape[0]
    x2 = x.reshape(-1, K)
    M = x2.shape[0]
    out = torch.empty((M, N), dtype=bf16, device=x.device)
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.n, d.k = x2.data_ptr(), K, M, N, K
    d.b[0], d.b[1] = gate_w.data_ptr(), up_w.data_ptr()
    d.n_seg, d.b_layout, d.num_groups = 2, L.B_NK, 1
    d.epilogue = L.EPI_SWIGLU
    d.out[0], d.ldo = out.data_ptr(), N
    _run_gemm(d, x, "linear_swiglu")
    return out.view(*x.shape[:-1], N)


def grouped_gemm(a: torch.Tensor, b: torch.Tensor, offsets: torch.Tensor, swiglu: bool = False,
                 dbg=(0, 0, 0), group_mod: int = 0, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[off[e]:off[e+1]] = a[off[e]:off[e+1]] @ b[e] (+ residual); b [E, K, N] (GroupedGEMM.weight, moe_lm.py:465).
    swiglu=True fuses `glu` (moe_lm.py:505-507): b has 2I columns, out has I."""
    _chk(a), _chk(b), _chk(offsets, torch.int32)
    rows, K = a.shape
    E, Kb, Nb = b.shape
    G = offsets.numel() - 1  # groups; with group_mod, group g multiplies by weight block g % group_mod
    assert Kb == K and (G == E if not group_mod else (group_mod == E and G % E == 0))
    N = Nb // 2 if swiglu else Nb
    out = torch.empty((rows, N), dtype=bf16, device=a.device)
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.n, d.k = a.data_ptr(), K, rows, N, K
    d.b[0] = b.data_ptr()
    d.n_seg, d.b_layout, d.num_groups = 1, L.B_GKN, G
    d.group_mod = group_mod
    d.group_offsets = offsets.data_ptr()
    d.epilogue = L.EPI_SWIGLU if swiglu else L.EPI_LINEAR
    d.out[0], d.ldo = out.data_ptr(), N
    if residual is not None:
        assert not swiglu and residual.shape == out.shape
        _chk(residual)
        d.residual, d.ldr = residual.data_ptr(), N
    d.dbg_lbo, d.dbg_sbo, d.dbg_kadv = dbg
    _run_gemm(d, a, "grouped_gemm")
    return out


def grouped_gemm_regions(a_buf: torch.Tensor, b: torch.Tensor, starts: torch.Tensor, counts: torch.Tensor, rows_hint: int,
                         swiglu: bool = False, group_mod: int = 0, out: Optional[torch.Tensor] = None,
                         out_group_base: Optional[torch.Tensor] = None, out_group_row0: Optional[torch.Tensor] = None,
                         ldo: Optional[int] = None) -> Optional[torch.Tensor]:
    """Grouped GEMM over FIXED-CAPACITY row regions (expert parallelism, csrc/ep.cu): group g = rows
    [starts[g], starts[g] + counts[g]) of `a_buf`, multiplied by weight block g % group_mod (group_mod > 0) or g // -group_mod (< 0).  `counts` may be written by peer
    GPUs (it is read on the device at launch).  rows_hint = expected total rows (tile-shape heuristics only).
    With out_group_base / out_group_row0 the rows of group g are stored at (bf16*)out_group_base[g] + (out_group_row0[g] + r)*ldo
    — e.g. straight into the source rank's combine buffer over NVLink — and nothing is returned."""
    _chk(a_buf), _chk(b), _chk(starts, torch.int32, align=4), _chk(counts, torch.int32, align=4)
    cap_rows, K = a_buf.shape
    E, Kb, Nb = b.shape
    G = starts.numel()
    assert Kb == K and counts.numel() == G and (G == E if not group_mod else ((group_mod == E and G % E == 0) if group_mod > 0 else G == E * -group_mod))
    N = Nb // 2 if swiglu else Nb
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.n, d.k = a_buf.data_ptr(), K, max(1, min(rows_hint, cap_rows)), N, K
    d.a_rows = cap_rows
    d.b[0] = b.data_ptr()
    d.n_seg, d.b_layout, d.num_groups = 1, L.B_GKN, G
    d.group_mod = group_mod
    d.group_offsets, d.group_counts = starts.data_ptr(), counts.data_ptr()
    d.epilogue = L.EPI_SWIGLU if swiglu else L.EPI_LINEAR
    if out_group_base is not None:
        assert not swiglu and out_group_row0 is not None and ldo is not None
        _chk(out_group_base, torch.int64, align=8), _chk(out_group_row0, torch.int32, align=4)
        d.out_group_base, d.out_group_row0 = out_group_base.data_ptr(), out_group_row0.data_ptr()
        d.out[0], d.ldo = a_buf.data_ptr(), ldo      # out[0] is never dereferenced on this path (must be non-NULL)
        ret = None
    else:
        if out is None:
            out = torch.empty((cap_rows, N), dtype=bf16, device=a_buf.device)
        _chk(out)
        assert out.shape == (cap_rows, N)
        d.out[0], d.ldo = out.data_ptr(), N
        ret = out
    _run_gemm(d, a_buf, "grouped_gemm")
    return ret


def grouped_gemm_nt(a: torch.Tensor, b: torch.Tensor, offsets: torch.Tensor, group_mod: int = 0,
                    residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Data-gradient of the grouped GEMM: out[rows of e] = a[rows of e] @ b[e].T (+ residual) with b [E, N_out, K]
    (K contiguous) — i.e. the forward weight [E, in, out] used transposed, read in place (ARIA_B_GNK)."""
    _chk(a), _chk(b), _chk(offsets, torch.int32)
    rows, K = a.shape
    E, N, Kb = b.shape
    G = offsets.numel() - 1
    assert Kb == K and (G == E if not group_mod else (group_mod == E and G % E == 0))
    out = torch.empty((rows, N), dtype=bf16, device=a.device)
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.n, d.k = a.data_ptr(), a.stride(0), rows, N, K
    d.b[0] = b.data_ptr()
    d.n_seg, d.b_layout, d.num_groups = 1, L.B_GNK, G
    d.group_mod = group_mod
    d.group_offsets = offsets.data_ptr()
    d.epilogue = L.EPI_LINEAR
    d.out[0], d.ldo = out.data_ptr(), N
    if residual is not None:
        assert residual.shape == out.shape
        _chk(residual)
        d.residual, d.ldr = residual.data_ptr(), N
    _run_gemm(d, a, "grouped_gemm_nt")
    return out


def matmul_kn(a: torch.Tensor, w_kn: torch.Tensor, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """a [M, K] (row stride may exceed K) @ w_kn [K, N] (N contiguous) (+ residual): dense data-gradients, where the
    nn.Linear weight [out, in] = [K, N] is consumed in place through the MN-major B path."""
    if not (a.is_cuda and a.dtype == bf16 and a.stride(1) == 1 and a.data_ptr() % 16 == 0):
        raise RuntimeError("matmul_kn: a must be CUDA bf16 with contiguous rows")
    _chk(w_kn)
    M, K = a.shape
    Kw, N = w_kn.shape
    assert K == Kw
    out = torch.empty((M, N), dtype=bf16, device=a.device)
    off = torch.tensor([0, M], dtype=torch.int32, device=a.device)
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.n, d.k = a.data_ptr(), a.stride(0), M, N, K
    d.b[0] = w_kn.data_ptr()
    d.n_seg, d.b_layout, d.num_groups = 1, L.B_GKN, 1
    d.group_offsets = off.data_ptr()
    d.epilogue = L.EPI_LINEAR
    if residual is not None:
        d.residual, d.ldr = _chk(residual).data_ptr(), N
    d.out[0], d.ldo = out.data_ptr(), N
    _run_gemm(d, a, "matmul_kn")
    return out


def grouped_wgrad(a: torch.Tensor, b: torch.Tensor, offsets: torch.Tensor, num_sources: int = 1) -> torch.Tensor:
    """out[g] = a[rows of g].T @ b[rows of g]; a [rows, Md], b [rows, Nd] (row strides allowed), offsets [G+1] int32 with
    16-aligned entries -> out [G, Md, Nd] bf16 (fp32 accumulation in TMEM).  num_sources=S: offsets [S*G+1] over
    (source, g) row groups, out[g] sums over the sources."""
    for t in (a, b):
        if not (t.is_cuda and t.dtype == bf16 and t.stride(1) == 1 and t.data_ptr() % 16 == 0):
            raise RuntimeError("grouped_wgrad: operands must be CUDA bf16 with contiguous rows")
    _chk(offsets, torch.int32)
    rows, Md = a.shape
    Nd = b.shape[1]
    G = (offsets.numel() - 1) // num_sources
    assert G * num_sources + 1 == offsets.numel()
    out = torch.empty((G, Md, Nd), dtype=bf16, device=a.device)
    with torch.cuda.device(a.device):
        L.check(L.load().aria_grouped_wgrad(_p(a), a.stride(0), _p(b), b.stride(0), _p(out), _p(offsets), rows, Md, Nd, G,
                                            num_sources, _stream(a)), "grouped_wgrad")
    return out


def swiglu_fwd(h1: torch.Tensor) -> torch.Tensor:
    _chk(h1)
    rows, I2 = h1.shape
    h = torch.empty((rows, I2 // 2), dtype=bf16, device=h1.device)
    with torch.cuda.device(h1.device):
        L.check(L.load().aria_swiglu_fwd(_p(h1), _p(h), rows, I2 // 2, _stream(h1)), "swiglu_fwd")
    return h


def swiglu_bwd(h1: torch.Tensor, dh: torch.Tensor) -> torch.Tensor:
    _chk(h1), _chk(dh)
    rows, I2 = h1.shape
    dh1 = torch.empty_like(h1)
    with torch.cuda.device(h1.device):
        L.check(L.load().aria_swiglu_bwd(_p(h1), _p(dh), _p(dh1), rows, I2 // 2, _stream(h1)), "swiglu_bwd")
    return dh1


def combine_bwd(dout: torch.Tensor, y: torch.Tensor, dest_row: torch.Tensor, scores: torch.Tensor):
    """-> (dy [rows(y), d] bf16 with pad rows zero, dscores [T, k] fp32)."""
    _chk(dout), _chk(y), _chk(dest_row, torch.int32), _chk(scores)
    T, k = scores.shape
    dy = torch.zeros_like(y)
    ds = torch.empty((T, k), dtype=torch.float32, device=y.device)
    with torch.cuda.device(y.device):
        L.check(L.load().aria_combine_bwd(_p(dout), _p(y), _p(dest_row), _p(scores), _p(dy), _p(ds), T, y.shape[1], k,
                                          _stream(y)), "combine_bwd")
    return dy, ds


def router_bwd(dscores: torch.Tensor, scores: torch.Tensor, top_idx: torch.Tensor, E: int) -> torch.Tensor:
    _chk(dscores, torch.float32), _chk(scores), _chk(top_idx, torch.int32)
    T, k = scores.shape
    dl = torch.empty((T, E), dtype=bf16, device=scores.device)
    with torch.cuda.device(scores.device):
        L.check(L.load().aria_router_bwd(_p(dscores), _p(scores), _p(top_idx), _p(dl), T, E, k, _stream(scores)), "router_bwd")
    return dl


def router_aux_loss(logits: torch.Tensor, counts: torch.Tensor, k: int, z_coeff: float, aux_coeff: float) -> torch.Tensor:
    """[z_loss, aux_loss] (fp32) of the training-mode router (moe_lm.py:128-166); values are for logging only."""
    _chk(logits), _chk(counts, torch.int32)
    T, E = logits.shape
    lib = L.load()
    nbytes = lib.aria_router_aux_workspace_bytes(E)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=logits.device)
    out = torch.empty(2, dtype=torch.float32, device=logits.device)
    with torch.cuda.device(logits.device):
        L.check(lib.aria_router_aux_loss(_p(logits), _p(counts), _p(out), T, E, k, z_coeff, aux_coeff, _p(ws), nbytes,
                                         _stream(logits)), "router_aux_loss")
    return out


def router_aux_bwd(logits: torch.Tensor, counts: torch.Tensor, dlogits: torch.Tensor, k: int, z_coeff: float, aux_coeff: float,
                   loss_scale: float = 1.0) -> torch.Tensor:
    """dlogits += loss_scale * d(z_loss + aux_loss)/d(logits)  (MoEAuxLossAutoScaler.backward, moe_lm.py:103-117), in place."""
    _chk(logits), _chk(counts, torch.int32), _chk(dlogits)
    T, E = logits.shape
    with torch.cuda.device(logits.device):
        L.check(L.load().aria_router_aux_bwd(_p(logits), _p(counts), _p(dlogits), T, E, k, z_coeff, aux_coeff, loss_scale,
                                             _stream(logits)), "router_aux_bwd")
    return dlogits


def qkv_heads(x: torch.Tensor, weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]],
              outs: Sequence[torch.Tensor], head_dim: int, rows_per_batch: int, pos0: int = 0, rope_mask: int = 0,
              rope_cos: Optional[torch.Tensor] = None, rope_sin: Optional[torch.Tensor] = None,
              position_ids: Optional[torch.Tensor] = None):
    """Fused q/k/v projections: x [B*T, K] @ W_s.T (+bias) (+RoPE) scattered into head-major buffers
    outs[s] [B, H, T_max, head_ld] at token offset pos0 (HF KV-cache layout)."""
    _chk(x)
    K = x.shape[-1]
    x2 = x.reshape(-1, K)
    d = L.GemmDesc()
    d.a, d.lda, d.m, d.k = x2.data_ptr(), K, x2.shape[0], K
    d.n = weights[0].shape[0]
    d.n_seg, d.b_layout, d.num_groups = len(weights), L.B_NK, 1
    d.epilogue = L.EPI_HEADS
    o0 = outs[0]
    for s, (w, b, o) in enumerate(zip(weights, biases, outs)):
        _chk(w), _chk(o)
        assert w.shape[0] == d.n and o.shape[1:] == o0.shape[1:] and o.stride() == o0.stride()
        d.b[s] = w.data_ptr()
        d.out[s] = o.data_ptr()
        if b is not None:
            d.bias[s] = _chk(b).data_ptr()
    d.head_dim, d.head_ld = head_dim, o0.shape[-1]
    d.rows_per_batch, d.pos0 = rows_per_batch, pos0
    d.stride_b, d.stride_h = o0.stride(0), o0.stride(1)
    d.rope_mask = rope_mask
    if rope_mask:
        d.rope_cos, d.rope_sin = _chk(rope_cos).data_ptr(), _chk(rope_sin).data_ptr()
    if position_ids is not None:
        d.position_ids = _chk(position_ids, torch.int32).data_ptr()
    _run_gemm(d, x, "qkv_heads")


# ------------------------------------------------------------------------------------------- MoE routing
def router_topk(x: torch.Tensor, w_router: torch.Tensor, k: int):
    _chk(x), _chk(w_router)
    T, dm = x.shape
    E = w_router.shape[0]
    dev = x.device
    logits = torch.empty((T, E), dtype=bf16, device=dev)
    idx = torch.empty((T, k), dtype=torch.int32, device=dev)
    scores = torch.empty((T, k), dtype=bf16, device=dev)
    counts = torch.empty((E,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.load().aria_router_topk(_p(x), _p(w_router), _p(logits), _p(idx), _p(scores), _p(counts), T, dm, E, k,
                                          _stream(x)), "router_topk")
    return scores, idx, counts, logits


def route_from_logits(logits: torch.Tensor, k: int):
    _chk(logits)
    T, E = logits.shape
    dev = logits.device
    idx = torch.empty((T, k), dtype=torch.int32, device=dev)
    scores = torch.empty((T, k), dtype=bf16, device=dev)
    counts = torch.empty((E,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.load().aria_route_from_logits(_p(logits), _p(idx), _p(scores), _p(counts), T, E, k, _stream(logits)),
                "route_from_logits")
    return scores, idx, counts


def route_given_indices(logits: torch.Tensor, top_idx: torch.Tensor):
    """Scores / counts for a GIVEN expert choice (parity / replay hook; see include/aria_b200.h)."""
    _chk(logits), _chk(top_idx, torch.int32)
    T, E = logits.shape
    k = top_idx.shape[1]
    assert top_idx.shape[0] == T
    scores = torch.empty((T, k), dtype=bf16, device=logits.device)
    counts = torch.empty((E,), dtype=torch.int32, device=logits.device)
    with torch.cuda.device(logits.device):
        L.check(L.load().aria_route_given_indices(_p(logits), _p(top_idx), _p(scores), _p(counts), T, E, k, _stream(logits)),
                "route_given_indices")
    return scores, counts


def build_permutation(top_idx: torch.Tensor, counts: torch.Tensor, row_align: int = 1):
    """row_align=16 (training): expert blocks start on multiples of 16 rows; `src` then has T*k + E*15 slots (upper bound
    of the padded row count, the true total is offsets[E]) and pad rows carry -1."""
    _chk(top_idx, torch.int32), _chk(counts, torch.int32)
    T, k = top_idx.shape
    E = counts.numel()
    dev = top_idx.device
    offsets = torch.empty((E + 1,), dtype=torch.int32, device=dev)
    dest = torch.empty((T * k,), dtype=torch.int32, device=dev)
    src = torch.empty((T * k + E * (row_align - 1),), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.load().aria_build_permutation(_p(top_idx), _p(counts), _p(offsets), _p(dest), _p(src), T, E, k, row_align,
                                                _stream(top_idx)), "build_permutation")
    return offsets, dest, src


def permute_rows(x: torch.Tensor, src_token: torch.Tensor) -> torch.Tensor:
    _chk(x), _chk(src_token, torch.int32)
    rows = src_token.numel()
    out = torch.empty((rows, x.shape[1]), dtype=bf16, device=x.device)
    with torch.cuda.device(x.device):
        L.check(L.load().aria_permute_rows(_p(x), _p(src_token), _p(out), rows, x.shape[1], _stream(x)), "permute_rows")
    return out


def permute_rows_to_ptr(x: torch.Tensor, src_token: torch.Tensor, out_ptr: int) -> None:
    """permute_rows writing to a raw device address — e.g. a PEER GPU's arena (aria_b200.peer.PeerArena): the row copy
    kernel then stores over NVLink."""
    _chk(x), _chk(src_token, torch.int32)
    with torch.cuda.device(x.device):
        L.check(L.load().aria_permute_rows(_p(x), _p(src_token), C.c_void_p(out_ptr), src_token.numel(), x.shape[1], _stream(x)),
                "permute_rows")


def unpermute_combine(y: torch.Tensor, dest_row: torch.Tensor, scores: torch.Tensor,
                      shared: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(y), _chk(dest_row, torch.int32), _chk(scores)
    T, k = scores.shape
    out = torch.empty((T, y.shape[1]), dtype=bf16, device=y.device)
    if shared is not None:
        _chk(shared)
    with torch.cuda.device(y.device):
        L.check(L.load().aria_unpermute_combine(_p(y), _p(dest_row), _p(scores), _p(shared), _p(out), T, y.shape[1], k,
                                                _stream(y)), "unpermute_combine")
    return out


def moe_block_fwd(x: torch.Tensor, w_router: torch.Tensor, fc1_w: torch.Tensor, fc2_w: torch.Tensor, gate_w: Optional[torch.Tensor],
                  up_w: Optional[torch.Tensor], down_w: Optional[torch.Tensor], k: int,
                  forced_top_idx: Optional[torch.Tensor] = None, side_stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
    """MoELayer.forward (moe_lm.py:548-577) as one C-ABI call (`aria_moe_block_fwd`): x [T, d] -> [T, d]."""
    _chk(x), _chk(w_router), _chk(fc1_w), _chk(fc2_w)
    T, d = x.shape
    E, I = fc2_w.shape[0], fc2_w.shape[1]
    assert w_router.shape == (E, d) and fc1_w.shape == (E, d, 2 * I) and fc2_w.shape == (E, I, d)
    Is = 0
    if gate_w is not None:
        _chk(gate_w), _chk(up_w), _chk(down_w)
        Is = gate_w.shape[0]
        assert gate_w.shape == (Is, d) and up_w.shape == (Is, d) and down_w.shape == (d, Is)
    if forced_top_idx is not None:
        _chk(forced_top_idx, torch.int32, align=4)
        assert forced_top_idx.shape == (T, k)
    lib = L.load()
    nbytes = lib.aria_moe_block_fwd_workspace_bytes(T, d, E, k, I, Is)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    out = torch.empty((T, d), dtype=bf16, device=x.device)
    with torch.cuda.device(x.device):
        L.check(lib.aria_moe_block_fwd(_p(x), _p(w_router), _p(fc1_w), _p(fc2_w), _p(gate_w), _p(up_w), _p(down_w), _p(out), T, d, E, k,
                                       I, Is, _p(forced_top_idx), _p(ws), nbytes, _stream(x),
                                       C.c_void_p(side_stream.cuda_stream) if side_stream is not None else None), "moe_block_fwd")
    return out


def offsets_from_counts(counts: torch.Tensor) -> torch.Tensor:
    _chk(counts, torch.int64)
    off = torch.empty((counts.numel() + 1,), dtype=torch.int32, device=counts.device)
    with torch.cuda.device(counts.device):
        L.check(L.load().aria_offsets_from_counts(_p(counts), _p(off), counts.numel(), _stream(counts)), "offsets_from_counts")
    return off


# ------------------------------------------------------------------------------------------- row-wise
def rmsnorm(x: torch.Tensor, weight: torch.Tensor, eps: float, residual: Optional[torch.Tensor] = None):
    """Returns norm(x) or, with residual, (norm(x + residual), x + residual)."""
    _chk(x), _chk(weight)
    d = x.shape[-1]
    rows = x.numel() // d
    out = torch.empty_like(x)
    s = torch.empty_like(x) if residual is not None else None
    if residual is not None:
        _chk(residual)
    with torch.cuda.device(x.device):
        L.check(L.load().aria_rmsnorm(_p(x), _p(residual), _p(weight), _p(out), _p(s), rows, d, eps, _stream(x)), "rmsnorm")
    return out if residual is None else (out, s)


def rmsnorm_bwd(x: torch.Tensor, weight: torch.Tensor, dy: torch.Tensor, eps: float, dres: Optional[torch.Tensor] = None):
    """Backward of rmsnorm(x, weight, eps) (no residual): -> (dx (+ dres), dw [d] bf16, deterministic reduction)."""
    _chk(x), _chk(weight), _chk(dy)
    d = x.shape[-1]
    rows = x.numel() // d
    assert dy.shape == x.shape and weight.numel() == d
    if dres is not None:
        _chk(dres)
        assert dres.shape == x.shape
    dx = torch.empty_like(x)
    dw = torch.empty_like(weight)
    lib = L.load()
    nbytes = lib.aria_rmsnorm_bwd_workspace_bytes(rows, d)
    ws = torch.empty((max(nbytes, 16),), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        L.check(lib.aria_rmsnorm_bwd(_p(x), _p(weight), _p(dy), _p(dres), _p(dx), _p(dw), rows, d, eps, _p(ws), ws.numel(),
                                     _stream(x)), "rmsnorm_bwd")
    return dx, dw


def rope_bwd(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, rows_per_batch: int,
             position_ids: Optional[torch.Tensor] = None) -> torch.Tensor:
    """In place on token-major x [..., n_heads*128]: the transpose of rotate-half RoPE (gradient of the rotated q or k).
    Positions: position_ids [rows] int32 when given, else row % rows_per_batch (the HEADS epilogue's convention)."""
    _chk(x), _chk(cos), _chk(sin)
    rows = x.numel() // x.shape[-1]
    assert x.shape[-1] % 128 == 0 and cos.shape[-1] == 128
    if position_ids is not None:
        _chk(position_ids, torch.int32, align=4)
        assert position_ids.numel() == rows
    with torch.cuda.device(x.device):
        L.check(L.load().aria_rope_bwd(_p(x), _p(cos), _p(sin), _p(position_ids), rows, x.shape[-1] // 128, rows_per_batch,
                                       _stream(x)), "rope_bwd")
    return x


def layernorm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float) -> torch.Tensor:
    _chk(x), _chk(weight), _chk(bias)
    d = x.shape[-1]
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        L.check(L.load().aria_layernorm(_p(x), _p(weight), _p(bias), _p(out), x.numel() // d, d, eps, _stream(x)), "layernorm")
    return out


def rope_table(inv_freq: torch.Tensor, n_pos: int):
    _chk(inv_freq, torch.float32)
    hd = inv_freq.numel() * 2
    cos = torch.empty((n_pos, hd), dtype=bf16, device=inv_freq.device)
    sin = torch.empty_like(cos)
    with torch.cuda.device(inv_freq.device):
        L.check(L.load().aria_rope_table(_p(inv_freq), _p(cos), _p(sin), n_pos, hd, _stream(inv_freq)), "rope_table")
    return cos, sin


def embedding(ids: torch.Tensor, table: torch.Tensor) -> torch.Tensor:
    _chk(ids, torch.int64, align=8), _chk(table)      # ids are read element-wise (a [1, 1] slice of a longer id row is fine)
    out = torch.empty((*ids.shape, table.shape[1]), dtype=bf16, device=table.device)
    with torch.cuda.device(table.device):
        L.check(L.load().aria_embedding(_p(ids), _p(table), _p(out), ids.numel(), table.shape[1], _stream(table)), "embedding")
    return out


def merge_image_features(ids: torch.Tensor, image_token: int, features: torch.Tensor, embeds: torch.Tensor,
                         count_out: Optional[torch.Tensor] = None):
    """In place: embeds rows at <|img|> positions <- consecutive rows of features (masked_scatter)."""
    _chk(ids, torch.int64, align=8), _chk(features), _chk(embeds)
    d = embeds.shape[-1]
    with torch.cuda.device(embeds.device):
        L.check(L.load().aria_merge_image_features(_p(ids), image_token, _p(features), _p(embeds), _p(count_out),
                                                   ids.numel(), d, _stream(embeds)), "merge_image_features")
    return embeds


def im2col_patches(pixels: torch.Tensor, patch: int, k_pad: int) -> torch.Tensor:
    _chk(pixels)
    B, Cc, S, S2 = pixels.shape
    assert Cc == 3 and S == S2
    n = (S // patch) ** 2
    out = torch.empty((B * n, k_pad), dtype=bf16, device=pixels.device)
    with torch.cuda.device(pixels.device):
        L.check(L.load().aria_im2col_patches(_p(pixels), _p(out), B, S, patch, k_pad, _stream(pixels)), "im2col_patches")
    return out


def add_pos_embedding(x: torch.Tensor, pos_ids: torch.Tensor, table: torch.Tensor) -> torch.Tensor:
    _chk(x), _chk(pos_ids, torch.int64), _chk(table)
    out = torch.empty_like(x)
    d = x.shape[-1]
    with torch.cuda.device(x.device):
        L.check(L.load().aria_add_pos_embedding(_p(x), _p(pos_ids), _p(table), _p(out), x.numel() // d, d, _stream(x)),
                "add_pos_embedding")
    return out


# ------------------------------------------------------------------------------------------- attention
def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, Tq: int, Tk: int, scale: float, causal: bool,
              out_hd: int = 128, key_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q [B,H,>=Tq,128], k/v [B,H,>=Tk,128] head-major (first Tq/Tk rows used) -> out [B, Tq, H*out_hd].
    Token rows must be 128 contiguous bf16 at a row stride of 128 (a slice q[:, :, pos0:] of a staging buffer is fine)."""
    for t in (q, k, v):
        if not (t.is_cuda and t.dtype == bf16 and t.dim() == 4 and t.stride(-1) == 1 and t.stride(-2) == 128 and t.data_ptr() % 16 == 0):
            raise RuntimeError("attention: q/k/v must be CUDA bf16 [B,H,T,128] with 128-element token rows (16-byte aligned)")
    B, H = q.shape[0], q.shape[1]
    assert q.shape[-1] == 128 and k.shape[-1] == 128 and k.stride() == v.stride()
    assert q.shape[2] >= Tq and k.shape[2] >= Tk
    out = torch.empty((B, Tq, H * out_hd), dtype=bf16, device=q.device)
    if key_mask is not None:
        _chk(key_mask, torch.uint8)
        assert key_mask.shape == (B, Tk)
    lib = L.load()
    ws, ws_bytes = None, 0
    if not causal:  # persistent launch: scratch for the stream-K pieces of the leftover units (see include/aria_b200.h)
        ws_bytes = lib.aria_attention_fwd_workspace_bytes(B, H, Tq, Tk, out_hd, 0)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=q.device)
    with torch.cuda.device(q.device):
        L.check(lib.aria_attention_fwd(_p(q), _p(k), _p(v), _p(out), _p(key_mask), B, H, Tq, Tk, q.stride(0), q.stride(1),
                                       k.stride(0), k.stride(1), out_hd, scale, int(causal), _p(ws), ws_bytes, _stream(q)),
                "attention_fwd")
    return out


def _check_heads(*ts):
    for t in ts:
        if not (t.is_cuda and t.dtype == bf16 and t.dim() == 4 and t.stride(-1) == 1 and t.stride(-2) == 128 and t.shape[-1] == 128
                and t.data_ptr() % 16 == 0):
            raise RuntimeError("attention: q/k/v must be CUDA bf16 [B,H,T,128] with 128-element token rows (16-byte aligned)")


def attention_fwd_lse(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, scale: float,
                      key_mask: Optional[torch.Tensor] = None):
    """Causal self-attention over q/k/v [B,H,T,128] -> (out [B,T,H*128] bf16, lse [B,H,T] fp32 in the log2 domain of
    scale*log2(e)*s, +inf for a row that sees no key).  out equals `attention(..., causal=True)` where that takes the same kernel."""
    _check_heads(q, k, v)
    B, H, T = q.shape[0], q.shape[1], q.shape[2]
    assert k.shape[:3] == (B, H, T) and k.stride() == v.stride()
    out = torch.empty((B, T, H * 128), dtype=bf16, device=q.device)
    lse = torch.empty((B, H, T), dtype=torch.float32, device=q.device)
    if key_mask is not None:
        _chk(key_mask, torch.uint8)
        assert key_mask.shape == (B, T)
    with torch.cuda.device(q.device):
        L.check(L.load().aria_attention_fwd_lse(_p(q), _p(k), _p(v), _p(out), _p(lse), _p(key_mask), B, H, T, q.stride(0), q.stride(1),
                                                k.stride(0), k.stride(1), scale, 128, 1, _stream(q)), "attention_fwd_lse")
    return out, lse


def attention_bwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: torch.Tensor, dout: torch.Tensor, lse: torch.Tensor,
                  scale: float, key_mask: Optional[torch.Tensor] = None):
    """Gradient of causal `attention_fwd_lse`: q/k/v [B,H,T,128] head-major, out / dout [B,T,H*128] token-major, lse [B,H,T]
    -> (dq, dk, dv), each [B,T,H*128] token-major bf16 (gradients w.r.t. the q/k/v the attention consumed)."""
    _check_heads(q, k, v)
    B, H, T = q.shape[0], q.shape[1], q.shape[2]
    assert k.shape[:3] == (B, H, T) and k.stride() == v.stride()
    _chk(out), _chk(dout), _chk(lse, torch.float32)
    assert out.shape == (B, T, H * 128) and dout.shape == out.shape and lse.shape == (B, H, T)
    if key_mask is not None:
        _chk(key_mask, torch.uint8)
        assert key_mask.shape == (B, T)
    dq, dk, dv = (torch.empty_like(out) for _ in range(3))
    lib = L.load()
    nbytes = lib.aria_attention_bwd_workspace_bytes(B, H, T)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=q.device)
    with torch.cuda.device(q.device):
        L.check(lib.aria_attention_bwd(_p(q), _p(k), _p(v), _p(out), _p(dout), _p(lse), _p(dq), _p(dk), _p(dv), _p(key_mask), B, H, T,
                                       q.stride(0), q.stride(1), k.stride(0), k.stride(1), scale, 128, 1, _p(ws), nbytes, _stream(q)),
                "attention_bwd")
    return dq, dk, dv


def attention_v2(q, k, v, Tq, Tk, scale, causal, out_hd=128, key_mask=None):
    """Round-1 kernel (aria_attention_fwd_v2), kept for A/B timing in scripts/ only."""
    B, H = q.shape[0], q.shape[1]
    out = torch.empty((B, Tq, H * out_hd), dtype=bf16, device=q.device)
    with torch.cuda.device(q.device):
        L.check(L.load().aria_attention_fwd_v2(_p(q), _p(k), _p(v), _p(out), _p(key_mask), B, H, Tq, Tk, q.stride(0), q.stride(1),
                                               k.stride(0), k.stride(1), out_hd, scale, int(causal), _stream(q)), "attention_fwd")
    return out


def attention_decode(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, Tk: int, scale: float,
                     key_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q [B,H,128] (any strides with a contiguous last dim, e.g. a row of the q staging buffer), cache k/v
    [B,H,T_max,128] -> out [B, H*128].  key_mask [B, Tk] uint8, 1 = masked out (padded batch)."""
    _chk(k), _chk(v)
    if not (q.is_cuda and q.dtype == bf16 and q.stride(-1) == 1 and q.data_ptr() % 8 == 0):
        raise RuntimeError("attention_decode: q must be a CUDA bf16 tensor with a contiguous last dim")
    B, H = q.shape[0], q.shape[1]
    lib = L.load()
    ws_bytes = lib.aria_attention_decode_workspace_bytes(B, H, Tk)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=q.device)
    out = torch.empty((B, H * 128), dtype=bf16, device=q.device)
    if key_mask is not None:
        _chk(key_mask, torch.uint8)
        assert key_mask.shape == (B, Tk)
    with torch.cuda.device(q.device):
        L.check(lib.aria_attention_decode(_p(q), _p(k), _p(v), _p(out), _p(key_mask), B, H, Tk, q.stride(0), q.stride(1), k.stride(0),
                                          k.stride(1), scale, _p(ws), ws_bytes, _stream(q)), "attention_decode")
    return out
