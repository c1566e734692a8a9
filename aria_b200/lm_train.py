"""Training path of a whole decoder layer: `MoEDecoderLayer` forward + backward over our CUDA kernels.  The reference gets this
backward from autograd through LlamaRMSNorm, apply_rotary_pos_emb, SDPA / eager attention and the nn.Linear projections
(aria/model/moe_lm.py:580-602); here every gradient is an explicit kernel:

    forward:   rmsnorm -> q/k/v GEMM (+RoPE, head-major scatter) -> causal attention (keeps lse) -> o_proj GEMM (+residual)
               -> rmsnorm -> MoE block (moe_train.MoELayerFunction) -> residual add
    backward:  dWo (wgrad), dO = dout @ Wo -> attention backward (Delta, dK/dV, dQ kernels) -> RoPE transpose on dq, dk
               -> dWq/dWk/dWv (wgrad), dh = dq@Wq + dk@Wk + dv@Wv (chained residual epilogues) -> rmsnorm backward with the
               residual-stream gradient added in the same pass

Every norm sits on a residual branch, so `RMSNormFunction` also returns its input as the residual stream: the gradient of
that branch arrives in the norm's own backward and the kernel adds it (no separate accumulation pass).
Gradients are bf16 tensors accumulated in fp32 inside the kernels; all of them are deterministic run to run.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.utils.checkpoint

from . import ops
from .moe_train import moe_layer_train

bf16 = torch.bfloat16
HEAD_DIM = 128


class RMSNormFunction(torch.autograd.Function):
    """(x, weight, eps) -> (rmsnorm(x), x).  The second output is the residual stream; its gradient is added into dx by the
    backward kernel."""

    @staticmethod
    def forward(ctx, x, weight, eps: float):
        y = ops.rmsnorm(x, weight, eps)
        ctx.save_for_backward(x, weight)
        ctx.eps = eps
        return y, x

    @staticmethod
    def backward(ctx, dy, dres):
        x, weight = ctx.saved_tensors
        dx, dw = ops.rmsnorm_bwd(x, weight, dy.contiguous(), ctx.eps, None if dres is None else dres.contiguous())
        return dx, dw, None


class AttentionFunction(torch.autograd.Function):
    """Causal self-attention sub-block without the norm: out = o_proj(attn(rope(h Wq^T), rope(h Wk^T), h Wv^T)) + residual.
    h, residual [B, T, d] with d = n_heads * 128; rope = (cos, sin) tables of aria_rope_table; key_mask [B, T] uint8
    (1 = masked out) or None; position_ids [B*T] int32 or None (then token t of each row sits at position t)."""

    @staticmethod
    def forward(ctx, h, residual, wq, wk, wv, wo, n_heads: int, rope, key_mask=None, position_ids=None):
        B, T, d = h.shape
        if d != n_heads * HEAD_DIM:
            raise RuntimeError(f"attention training path is written for head_dim {HEAD_DIM}")
        q, k, v = (torch.empty((B, n_heads, T, HEAD_DIM), dtype=bf16, device=h.device) for _ in range(3))
        cos, sin = rope
        ops.qkv_heads(h, [wq, wk, wv], [None] * 3, [q, k, v], HEAD_DIM, T, pos0=0, rope_mask=0b011, rope_cos=cos, rope_sin=sin,
                      position_ids=position_ids)
        scale = HEAD_DIM ** -0.5
        o, lse = ops.attention_fwd_lse(q, k, v, scale, key_mask)
        out = ops.linear(o, wo, residual=residual)
        ctx.save_for_backward(h, wq, wk, wv, wo, q, k, v, o, lse)
        ctx.rope, ctx.key_mask, ctx.position_ids, ctx.scale = rope, key_mask, position_ids, scale
        return out

    @staticmethod
    def backward(ctx, dout):
        h, wq, wk, wv, wo, q, k, v, o, lse = ctx.saved_tensors
        B, T, d = h.shape
        M = B * T
        do = dout.reshape(M, d).contiguous()
        dense = torch.tensor([0, M], dtype=torch.int32, device=do.device)  # one "group": dense weight gradients
        d_wo = ops.grouped_wgrad(do, o.view(M, d), dense)[0]                # [d, d] = dout^T o
        d_o = ops.matmul_kn(do, wo).view(B, T, d)                           # dout @ Wo
        dq, dk, dv = ops.attention_bwd(q, k, v, o, d_o, lse, ctx.scale, ctx.key_mask)
        cos, sin = ctx.rope
        ops.rope_bwd(dq, cos, sin, T, ctx.position_ids)
        ops.rope_bwd(dk, cos, sin, T, ctx.position_ids)
        dq, dk, dv = dq.view(M, d), dk.view(M, d), dv.view(M, d)
        h2 = h.reshape(M, d)
        d_wq = ops.grouped_wgrad(dq, h2, dense)[0]
        d_wk = ops.grouped_wgrad(dk, h2, dense)[0]
        d_wv = ops.grouped_wgrad(dv, h2, dense)[0]
        dh = ops.matmul_kn(dq, wq)
        dh = ops.matmul_kn(dk, wk, residual=dh)
        dh = ops.matmul_kn(dv, wv, residual=dh)
        return dh.view(B, T, d), dout, d_wq, d_wk, d_wv, d_wo, None, None, None, None


class ResidualAddFunction(torch.autograd.Function):
    """a + b (bf16, one rounding) on the combine kernel with k = 1 and the identity row map; the gradient passes to both."""

    @staticmethod
    def forward(ctx, a, b):
        shape = a.shape
        a2, b2 = a.reshape(-1, shape[-1]), b.reshape(-1, shape[-1])
        M = a2.shape[0]
        ident = torch.arange(M, dtype=torch.int32, device=a.device)
        ones = torch.ones((M, 1), dtype=bf16, device=a.device)
        return ops.unpermute_combine(a2, ident, ones, b2).view(shape)

    @staticmethod
    def backward(ctx, g):
        return g, g


_ROPE = {}


def rope_tables(theta: float, n_pos: int, device):
    """cos / sin [n_pos, 128] bf16 (LlamaRotaryEmbedding's fp32 inv_freq, aria_rope_table), cached per device and theta."""
    key = (str(device), float(theta))
    t = _ROPE.get(key)
    if t is None or t[0].shape[0] < n_pos:
        inv_freq = 1.0 / (theta ** (torch.arange(0, HEAD_DIM, 2, dtype=torch.int64).float() / HEAD_DIM))
        t = _ROPE[key] = ops.rope_table(inv_freq.to(device), n_pos)
    return t


def decoder_layer_train(layer, hidden_states: torch.Tensor, position_ids: Optional[torch.Tensor] = None,
                        attention_mask: Optional[torch.Tensor] = None, router_losses: bool = False) -> torch.Tensor:
    """Differentiable `MoEDecoderLayer.forward` (moe_lm.py:590-602) for an `aria_b200.moe_lm.MoEDecoderLayer` whose parameters
    require grad: x + attn(rms(x)) -> h + moe(rms(h)), no KV cache.  hidden_states [B, T, d] bf16.
    position_ids [B, T] (default: arange(T) per row, as LlamaModel uses); attention_mask: the HF 2-D mask [B, T], 1 = keep.
    router_losses=True adds the training-mode z-loss / load-balancing gradients (see moe_train.moe_layer_train)."""
    B, T, d = hidden_states.shape
    dev = hidden_states.device
    attn = layer.self_attn
    key_mask = None
    if attention_mask is not None:
        key_mask = (attention_mask.to(dev) == 0).to(torch.uint8).contiguous()
    pos, n_pos = None, T
    if position_ids is not None:
        pos = position_ids.to(device=dev, dtype=torch.int32).reshape(-1).contiguous()
        n_pos = max(T, int(pos.max()) + 1)
    rope = rope_tables(attn.config.rope_theta, n_pos, dev)
    eps1 = layer.input_layernorm.variance_epsilon
    eps2 = layer.post_attention_layernorm.variance_epsilon
    h, x = RMSNormFunction.apply(hidden_states, layer.input_layernorm.weight, eps1)
    x = AttentionFunction.apply(h, x, attn.q_proj.weight, attn.k_proj.weight, attn.v_proj.weight, attn.o_proj.weight,
                                attn.num_heads, rope, key_mask, pos)
    h, x = RMSNormFunction.apply(x, layer.post_attention_layernorm.weight, eps2)
    return ResidualAddFunction.apply(moe_layer_train(layer.mlp, h, router_losses), x)


# ------------------------------------------------------------------------------------------------ whole language model
class EmbeddingFunction(torch.autograd.Function):
    """nn.Embedding on aria_embedding; the backward (aria_embedding_bwd, only when the table requires grad) sums the rows per
    id in position order.  Positions whose id is skip_id get no gradient: they are image tokens, whose embeddings the image
    features replaced (masked_scatter, modeling_aria.py:272-283)."""

    @staticmethod
    def forward(ctx, ids, table, skip_id: Optional[int] = None):
        ids = ids.contiguous()
        ctx.save_for_backward(ids)
        ctx.vocab, ctx.skip_id = table.shape[0], skip_id
        return ops.embedding(ids, table)

    @staticmethod
    def backward(ctx, g):
        if not ctx.needs_input_grad[1]:
            return None, None, None
        (ids,) = ctx.saved_tensors
        return None, ops.embedding_bwd(ids, g.contiguous(), ctx.vocab, ctx.skip_id), None


class _MergeImageFunction(torch.autograd.Function):
    """embeds with the image-token rows replaced by the (constant) image features; the gradient passes through unchanged (the
    embedding backward skips the image-token rows)."""

    @staticmethod
    def forward(ctx, embeds, ids, image_token: int, features):
        out = embeds.clone()
        ops.merge_image_features(ids.reshape(-1).contiguous(), image_token, features.reshape(-1, features.shape[-1]),
                                 out.view(-1, out.shape[-1]))
        return out

    @staticmethod
    def backward(ctx, g):
        return g, None, None, None


class LMHeadCrossEntropyFunction(torch.autograd.Function):
    """(h [M, d], w [V, d], targets [M] int32, < 0 = ignored) -> mean cross-entropy of the bf16 logits h w^T over the valid rows,
    a 0-dim fp32 tensor, through the fused kernels (aria_lm_xent_fwd / _bwd): no [M, V] tensor is ever allocated.  The
    lm_head gradient is skipped when w does not require grad."""

    @staticmethod
    def forward(ctx, h, w, targets):
        loss, lse, n_valid = ops.lm_xent_fwd(h, w, targets)
        ctx.save_for_backward(h, w, targets, lse, n_valid)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        h, w, targets, lse, n_valid = ctx.saved_tensors
        dh, dw = ops.lm_xent_bwd(h, w, targets, lse, n_valid, dloss, need_dw=ctx.needs_input_grad[1])
        return (dh if ctx.needs_input_grad[0] else None), dw, None


def shifted_targets(labels: torch.Tensor, attention_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int32 [B*T] targets of the shifted loss (modeling_aria.py:300-323): position t of row b predicts labels[b, t+1]; it is
    ignored (-1) when attention_mask[b, t+1] == 0, when that label is negative (ignore_index -100) and at the last position.
    Index plumbing on the labels' device, no sync."""
    B, T = labels.shape
    tgt = torch.full((B, T), -1, dtype=torch.int32, device=labels.device)
    if T > 1:
        nxt = labels[:, 1:]
        keep = nxt >= 0
        if attention_mask is not None:
            keep = keep & (attention_mask[:, -(T - 1):].to(labels.device) != 0)
        tgt[:, :-1] = torch.where(keep, nxt, torch.full_like(nxt, -1)).to(torch.int32)
    return tgt.reshape(-1)


def causal_lm_loss(lm, labels: torch.Tensor, input_ids: Optional[torch.Tensor] = None, inputs_embeds: Optional[torch.Tensor] = None,
                   attention_mask: Optional[torch.Tensor] = None, position_ids: Optional[torch.Tensor] = None,
                   router_losses: bool = False, gradient_checkpointing: bool = False,
                   skip_embed_id: Optional[int] = None) -> torch.Tensor:
    """Training loss of an `aria_b200.moe_lm.AriaMoELMForCausalLM` with a grad_fn: embedding -> every decoder layer
    (decoder_layer_train) -> final RMSNorm -> fused lm_head + shifted cross-entropy (the loss of modeling_aria.py:300-323).
    input_ids [B, T] (embedded here; positions whose id is skip_embed_id get no embedding gradient) or inputs_embeds [B, T, d];
    labels [B, T]; attention_mask: the HF 2-D padding mask, 1 = keep; position_ids [B, T] (default: arange per row).
    gradient_checkpointing=True keeps only each layer's input and recomputes the layer in backward
    (torch.utils.checkpoint, use_reentrant=False); every kernel and the routing are deterministic, so the recompute
    reproduces the forward bit for bit."""
    model = lm.model
    if inputs_embeds is None:
        x = EmbeddingFunction.apply(input_ids, model.embed_tokens.weight, skip_embed_id)
    else:
        x = inputs_embeds
    dev = x.device
    if attention_mask is not None:
        attention_mask = attention_mask.to(dev)
    for layer in model.layers:
        if gradient_checkpointing:
            x = torch.utils.checkpoint.checkpoint(decoder_layer_train, layer, x, position_ids, attention_mask, router_losses,
                                                  use_reentrant=False)
        else:
            x = decoder_layer_train(layer, x, position_ids, attention_mask, router_losses)
    h, _ = RMSNormFunction.apply(x, model.norm.weight, model.norm.variance_epsilon)
    d = h.shape[-1]
    targets = shifted_targets(labels.to(dev), attention_mask)
    return LMHeadCrossEntropyFunction.apply(h.reshape(-1, d), lm.lm_head.weight, targets)
