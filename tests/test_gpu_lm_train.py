"""GPU: decoder-layer training path — causal attention backward (tcgen05), the forward's lse, RMSNorm / RoPE backward and the
whole `decoder_layer_train` — against fp32 autograd through the oracle restatement on the same bf16 values.  Tolerance: relative
L2 error 2e-2 per gradient tensor (1e-2 for the row-wise kernels), as in test_gpu_backward.py."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"
SCALE = 128 ** -0.5


def _rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def _qkv(B, H, T, seed, dev="cpu"):
    g = torch.Generator().manual_seed(seed)
    q, k, v = (torch.randn(B, H, T, 128, generator=g).bfloat16() for _ in range(3))
    dout = torch.randn(B, T, H * 128, generator=g).bfloat16()
    return [t.to(dev) for t in (q, k, v, dout)]


def _dead_keys_mask(T, key_mask):
    """[B, 1, T, T] bool: key j is invisible to query i (causal or masked out)."""
    causal = torch.arange(T)[None, :] > torch.arange(T)[:, None]
    dead = causal[None, None]
    if key_mask is not None:
        dead = dead | key_mask.bool().cpu()[:, None, None, :]
    return dead


def _oracle_grads(q, k, v, dout, key_mask=None):
    """fp32 autograd of the oracle's attention_core with its causal mask (plus key padding) -> (out, dq, dk, dv) token-major."""
    from oracle import aria_oracle as O
    B, H, T, _ = q.shape
    q32, k32, v32 = (t.float().requires_grad_(True) for t in (q, k, v))
    if key_mask is None:
        add = O.causal_additive_mask(T, T, torch.float32)
    else:   # one finite fill value: a query row with no visible key stays finite (uniform) instead of NaN
        add = torch.zeros(B, 1, T, T).masked_fill(_dead_keys_mask(T, key_mask), torch.finfo(torch.float32).min)
    with torch.enable_grad():
        o = O.attention_core(q32, k32, v32, SCALE, add)             # [B, T, H, D]
        o.backward(dout.float().view(B, T, H, 128))
    tm = lambda t: t.detach().transpose(1, 2).reshape(B, T, H * 128)   # noqa: E731
    return o.detach().reshape(B, T, H * 128), tm(q32.grad), tm(k32.grad), tm(v32.grad)


def _ours(q, k, v, dout, key_mask=None):
    from aria_b200 import ops
    o, lse = ops.attention_fwd_lse(q, k, v, SCALE, key_mask)
    dq, dk, dv = ops.attention_bwd(q, k, v, o, dout, lse, SCALE, key_mask)
    torch.cuda.synchronize()
    return o, lse, dq, dk, dv


@pytest.mark.parametrize("B,H,T", [(1, 2, 128), (2, 3, 300), (1, 4, 1000)])
def test_attention_backward_vs_oracle_autograd(B, H, T):
    q, k, v, dout = _qkv(B, H, T, seed=T)
    _, want_dq, want_dk, want_dv = _oracle_grads(q, k, v, dout)
    _, _, dq, dk, dv = _ours(*(t.to(DEV) for t in (q, k, v, dout)))
    for name, got, want in (("dq", dq, want_dq), ("dk", dk, want_dk), ("dv", dv, want_dv)):
        assert torch.isfinite(got).all(), name
        assert _rel_l2(got, want) <= 2e-2, (name, _rel_l2(got, want))


@pytest.mark.parametrize("B,H,T", [(1, 20, 2048), (1, 2, 8192)])
def test_attention_backward_long_vs_fp32_torch(B, H, T):
    """Long sequences: the reference is fp32 torch on the GPU, one head at a time."""
    q, k, v, dout = _qkv(B, H, T, seed=7, dev=DEV)
    _, _, dq, dk, dv = _ours(q, k, v, dout)
    causal = torch.ones(T, T, dtype=torch.bool, device=DEV).triu(1)
    for h in range(0, H, max(1, H // 4)):
        qh, kh, vh = (t[0, h].float().requires_grad_(True) for t in (q, k, v))
        with torch.enable_grad():
            s = (qh @ kh.t() * SCALE).masked_fill(causal, float("-inf"))
            o = torch.softmax(s, -1) @ vh
            o.backward(dout[0, :, h * 128:(h + 1) * 128].float())
        for name, got, want in (("dq", dq, qh.grad), ("dk", dk, kh.grad), ("dv", dv, vh.grad)):
            g = got[0, :, h * 128:(h + 1) * 128]
            assert torch.isfinite(g).all(), name
            assert _rel_l2(g, want) <= 2e-2, (h, name, _rel_l2(g, want))


def test_attention_backward_padding():
    """Left padding: row 1 has 37 pad tokens, so its first query rows see no key at all; dout is zero there (ignored labels)."""
    B, H, T, pad = 2, 3, 300, 37
    q, k, v, dout = _qkv(B, H, T, seed=5)
    key_mask = torch.zeros(B, T, dtype=torch.uint8)
    key_mask[1, :pad] = 1
    dout = dout.clone()
    dout[1, :pad] = 0
    _, want_dq, want_dk, want_dv = _oracle_grads(q, k, v, dout, key_mask)
    o, lse, dq, dk, dv = _ours(*(t.to(DEV) for t in (q, k, v, dout)), key_mask=key_mask.to(DEV))
    for t in (o, dq, dk, dv):
        assert torch.isfinite(t).all()
    assert torch.isinf(lse[1, :, :pad]).all() and torch.isfinite(lse[0]).all() and torch.isfinite(lse[1, :, pad:]).all()
    assert float(dk[1, :pad].abs().max()) == 0.0 and float(dv[1, :pad].abs().max()) == 0.0
    for name, got, want in (("dq", dq, want_dq), ("dk", dk, want_dk), ("dv", dv, want_dv)):
        assert _rel_l2(got, want) <= 2e-2, (name, _rel_l2(got, want))


def test_attention_lse_and_forward_identity():
    from aria_b200 import ops
    B, H, T = 2, 3, 300
    q, k, v, _ = _qkv(B, H, T, seed=9)
    _, lse, *_ = _ours(*(t.to(DEV) for t in (q, k, v, torch.zeros(B, T, H * 128).bfloat16())))
    s = (q.float() @ k.float().transpose(2, 3)) * SCALE
    s = s.masked_fill(_dead_keys_mask(T, None), float("-inf"))
    want = torch.logsumexp(s, -1)                                   # natural log
    got = lse.cpu() * math.log(2.0)
    assert float((got - want).abs().max()) <= 1e-3
    # out is bit-identical to the inference forward at a shape where that takes the same kernel
    B, H, T = 1, 20, 2048
    q, k, v, _ = _qkv(B, H, T, seed=10, dev=DEV)
    o_lse, _ = ops.attention_fwd_lse(q, k, v, SCALE)
    o_ref = ops.attention(q, k, v, T, T, SCALE, causal=True)
    assert torch.equal(o_lse, o_ref)


def test_attention_backward_is_deterministic():
    B, H, T = 2, 4, 1000
    q, k, v, dout = _qkv(B, H, T, seed=3, dev=DEV)
    key_mask = torch.zeros(B, T, dtype=torch.uint8, device=DEV)
    key_mask[0, :11] = 1
    a = _ours(q, k, v, dout, key_mask)
    b = _ours(q, k, v, dout, key_mask)
    for x, y in zip(a[2:], b[2:]):
        assert torch.equal(x, y)


@pytest.mark.parametrize("with_dres", [False, True])
def test_rmsnorm_backward_vs_oracle_autograd(with_dres):
    from aria_b200 import ops
    from oracle import aria_oracle as O
    rows, d, eps = 1000, 2560, 1e-6
    g = torch.Generator().manual_seed(1)
    x = torch.randn(rows, d, generator=g).bfloat16()
    w = (1 + 0.1 * torch.randn(d, generator=g)).bfloat16()
    dy = torch.randn(rows, d, generator=g).bfloat16()
    dres = torch.randn(rows, d, generator=g).bfloat16() if with_dres else None
    x32, w32 = x.float().requires_grad_(True), w.float().requires_grad_(True)
    with torch.enable_grad():
        O.rms_norm(x32, w32, eps).backward(dy.float())
    want_dx = x32.grad + (dres.float() if with_dres else 0)
    dx, dw = ops.rmsnorm_bwd(x.to(DEV), w.to(DEV), dy.to(DEV), eps, None if dres is None else dres.to(DEV))
    assert _rel_l2(dx, want_dx) <= 1e-2
    assert _rel_l2(dw, w32.grad) <= 1e-2
    dx2, dw2 = ops.rmsnorm_bwd(x.to(DEV), w.to(DEV), dy.to(DEV), eps, None if dres is None else dres.to(DEV))
    assert torch.equal(dw, dw2) and torch.equal(dx, dx2)


def test_rope_backward_vs_oracle_autograd():
    from aria_b200 import ops
    from oracle import aria_oracle as O
    B, T, H = 2, 200, 3
    g = torch.Generator().manual_seed(2)
    pos = torch.stack([torch.arange(T), torch.randint(0, 4 * T, (T,), generator=g)])      # per-batch positions
    inv_freq = 1.0 / (5e6 ** (torch.arange(0, 128, 2, dtype=torch.int64).float() / 128))
    cos, sin = ops.rope_table(inv_freq.to(DEV), 4 * T)
    dy = torch.randn(B, T, H * 128, generator=g).bfloat16()
    x32 = torch.randn(B, H, T, 128, generator=g).requires_grad_(True)
    c, s = cos.float().cpu()[pos], sin.float().cpu()[pos]          # [B, T, 128]
    with torch.enable_grad():
        y, _ = O.apply_rope(x32, x32.detach(), c, s)
        y.backward(dy.float().view(B, T, H, 128).transpose(1, 2))
    want = x32.grad.transpose(1, 2).reshape(B, T, H * 128)
    got = dy.to(DEV).clone()
    ops.rope_bwd(got, cos, sin, T, pos.to(DEV, torch.int32).reshape(-1).contiguous())
    assert _rel_l2(got, want) <= 1e-2
    # default positions: row % rows_per_batch
    got0 = dy.to(DEV).clone()
    ops.rope_bwd(got0, cos, sin, T)
    got1 = dy.to(DEV).clone()
    ops.rope_bwd(got1, cos, sin, T, torch.arange(T, dtype=torch.int32, device=DEV).repeat(B))
    assert torch.equal(got0, got1)


# ------------------------------------------------------------------------------------------------ decoder layer
_LAYER_NAMES = ["input_layernorm.weight", "post_attention_layernorm.weight", "self_attn.q_proj.weight", "self_attn.k_proj.weight",
                "self_attn.v_proj.weight", "self_attn.o_proj.weight", "mlp.router.weight", "mlp.experts.fc1.weight",
                "mlp.experts.fc2.weight", "mlp.shared_experts.gate_proj.weight", "mlp.shared_experts.up_proj.weight",
                "mlp.shared_experts.down_proj.weight"]


def _layer_cfg(d, H, E, k, I):
    return dict(hidden_size=d, num_attention_heads=H, num_hidden_layers=1, moe_num_experts=E, moe_topk=k, moe_intermediate_size=I,
                moe_num_shared_experts=2, vocab_size=64, rms_norm_eps=1e-5, rope_theta=5e6)


def _layer_state(tc, seed):
    from oracle import configs as C
    sd = C.lm_state(tc, torch.Generator().manual_seed(seed), prefix="")
    p = "model.layers.0."
    return {n[len(p):]: v.bfloat16() for n, v in sd.items() if n.startswith(p)}


def _our_layer(tc, sd):
    from aria_b200 import moe_lm
    layer = moe_lm.MoEDecoderLayer(moe_lm.AriaMoELMConfig(**tc), 0, device=DEV)
    layer.load_state_dict({n: v.to(DEV) for n, v in sd.items()}, strict=True)
    for p_ in layer.parameters():
        p_.requires_grad_(True)
    return layer


def _oracle_layer(x32, sd32, tc, attention_mask):
    """fp32 oracle decoder layer; with a padding mask it is composed from the oracle's pieces with a causal + padding mask."""
    from oracle import aria_oracle as O
    B, T, d = x32.shape
    pos = torch.arange(T)[None].expand(B, T)
    if attention_mask is None:
        out, _ = O.moe_decoder_layer(x32, sd32, "", tc, pos)
        h = O.rms_norm(x32, sd32["input_layernorm.weight"], tc["rms_norm_eps"])
    else:
        H = tc["num_attention_heads"]
        h = O.rms_norm(x32, sd32["input_layernorm.weight"], tc["rms_norm_eps"])
        lin = lambda t, n: torch.nn.functional.linear(t, sd32[f"self_attn.{n}_proj.weight"]).view(B, T, H, 128).transpose(1, 2)  # noqa
        q, k, v = lin(h, "q"), lin(h, "k"), lin(h, "v")
        cos, sin = O.rope_cos_sin(pos, 128, tc["rope_theta"], torch.float32)
        q, k = O.apply_rope(q, k, cos, sin)
        add = torch.zeros(B, 1, T, T).masked_fill(_dead_keys_mask(T, (attention_mask == 0).to(torch.uint8)),
                                                  torch.finfo(torch.float32).min)
        o = O.attention_core(q, k, v, 128 ** -0.5, add).reshape(B, T, d)
        x1 = x32 + torch.nn.functional.linear(o, sd32["self_attn.o_proj.weight"])
        h2 = O.rms_norm(x1, sd32["post_attention_layernorm.weight"], tc["rms_norm_eps"])
        out = x1 + O.moe_layer(h2, sd32, tc["moe_topk"], "mlp.")
    return out, h


def _router_safe(sd32, x32, tc, attention_mask):
    """Tokens whose top-k choice is not a near-tie (same criterion as test_moe_layer_forward_backward_vs_oracle_autograd)."""
    from oracle import aria_oracle as O
    with torch.no_grad():
        B, T, d = x32.shape
        # the router sees rms(x + attn): recompute the oracle's input to the MoE block
        captured = {}
        orig = O.moe_layer

        def spy(h, w, k, prefix="", **kw):
            captured["h"] = h
            return orig(h, w, k, prefix, **kw)
        O.moe_layer = spy
        try:
            _oracle_layer(x32, sd32, tc, attention_mask)
        finally:
            O.moe_layer = orig
        lg = O.router_gating(captured["h"].reshape(-1, d), sd32["mlp.router.weight"]).sort(1, descending=True).values
    k = tc["moe_topk"]
    return (lg[:, k - 1] - lg[:, k]) / lg.abs().amax(1) > 2 ** -6


@pytest.mark.parametrize("masked", [False, True])
def test_decoder_layer_train_vs_oracle_autograd(masked):
    from aria_b200 import lm_train
    B, T = 2, 160
    tc = _layer_cfg(256, 2, 8, 2, 128)
    sd = _layer_state(tc, seed=21)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, T, 256, generator=g).bfloat16()
    gout = torch.randn(B, T, 256, generator=g).bfloat16()
    attention_mask = None
    if masked:
        attention_mask = torch.ones(B, T, dtype=torch.int64)
        attention_mask[1, :37] = 0
        gout[1, :37] = 0
    sd32 = {n: v.float().requires_grad_(True) for n, v in sd.items()}
    # A router near-tie flips a token's expert choice under bf16 rounding and moves whole rows of gradient.  With 320 random
    # tokens some always are near-ties, so the input rows of such tokens are redrawn (from the same seeded generator) until
    # none is left; attention mixes tokens, hence the loop.  The strict bound below then holds for every token.
    for _ in range(20):
        safe = _router_safe(sd32, x.float(), tc, attention_mask)
        if bool(safe.all()):
            break
        bad = ~safe
        x.view(-1, 256)[bad] = torch.randn(int(bad.sum()), 256, generator=g).bfloat16()
    assert bool(safe.all()), int((~safe).sum())
    x32 = x.float().requires_grad_(True)
    with torch.enable_grad():
        want, _ = _oracle_layer(x32, sd32, tc, attention_mask)
        want.backward(gout.float())
    layer = _our_layer(tc, sd)
    xg = x.to(DEV).requires_grad_(True)
    with torch.enable_grad():
        got = lm_train.decoder_layer_train(layer, xg, attention_mask=None if attention_mask is None else attention_mask.to(DEV))
        got.backward(gout.to(DEV))
    keep = slice(None) if not masked else (attention_mask.bool()[..., None].expand(B, T, 256))
    assert _rel_l2(got.detach().cpu()[keep], want.detach()[keep]) <= 2e-2
    assert _rel_l2(xg.grad, x32.grad) <= 2e-2
    params = dict(layer.named_parameters())
    assert sorted(params) == sorted(_LAYER_NAMES)
    for n in _LAYER_NAMES:
        assert params[n].grad is not None, n
        assert _rel_l2(params[n].grad, sd32[n].grad) <= 2e-2, (n, _rel_l2(params[n].grad, sd32[n].grad))


def test_decoder_layer_train_is_deterministic():
    from aria_b200 import lm_train
    B, T = 2, 160
    tc = _layer_cfg(256, 2, 8, 2, 128)
    layer = _our_layer(tc, _layer_state(tc, seed=21))
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, T, 256, generator=g).bfloat16().to(DEV)
    gout = torch.randn(B, T, 256, generator=g).bfloat16().to(DEV)
    mask = torch.ones(B, T, dtype=torch.int64, device=DEV)
    mask[0, :9] = 0
    runs = []
    for _ in range(2):
        layer.zero_grad(set_to_none=True)
        xg = x.clone().requires_grad_(True)
        with torch.enable_grad():
            lm_train.decoder_layer_train(layer, xg, attention_mask=mask).backward(gout)
        runs.append([xg.grad.clone()] + [p_.grad.clone() for p_ in layer.parameters()])
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_attention_block_full_width_vs_oracle():
    """The attention sub-block at the real width (d=2560, H=20, T=2048): input and q/k/v/o weight gradients."""
    from aria_b200 import lm_train
    from oracle import aria_oracle as O
    B, T, H, d = 1, 2048, 20, 2560
    g = torch.Generator().manual_seed(8)
    w = {n: (torch.randn(d, d, generator=g) * 0.02).bfloat16() for n in ("q", "k", "v", "o")}
    h = torch.randn(B, T, d, generator=g).bfloat16()
    gout = torch.randn(B, T, d, generator=g).bfloat16()
    theta = 5e6
    # reference on the GPU in fp32 (the oracle's functions are device-agnostic)
    w32 = {n: t.to(DEV).float().requires_grad_(True) for n, t in w.items()}
    h32 = h.to(DEV).float().requires_grad_(True)
    with torch.enable_grad():
        lin = lambda t, n: torch.nn.functional.linear(t, w32[n]).view(B, T, H, 128).transpose(1, 2)  # noqa: E731
        q, k, v = lin(h32, "q"), lin(h32, "k"), lin(h32, "v")
        cos, sin = O.rope_cos_sin(torch.arange(T)[None], 128, theta, torch.float32)
        q, k = O.apply_rope(q, k, cos.to(DEV), sin.to(DEV))
        causal = torch.ones(T, T, dtype=torch.bool, device=DEV).triu(1)
        s = (q @ k.transpose(2, 3) * SCALE).masked_fill(causal, float("-inf"))
        o = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B, T, d)
        want = torch.nn.functional.linear(o, w32["o"])
        want.backward(gout.to(DEV).float())
    wg = {n: t.to(DEV).requires_grad_(True) for n, t in w.items()}
    hg = h.to(DEV).requires_grad_(True)
    res = torch.zeros(B, T, d, dtype=torch.bfloat16, device=DEV)
    rope = lm_train.rope_tables(theta, T, DEV)
    with torch.enable_grad():
        got = lm_train.AttentionFunction.apply(hg, res, wg["q"], wg["k"], wg["v"], wg["o"], H, rope, None, None)
        got.backward(gout.to(DEV))
    assert _rel_l2(got.detach(), want.detach()) <= 2e-2
    assert _rel_l2(hg.grad, h32.grad) <= 2e-2
    for n in ("q", "k", "v", "o"):
        assert _rel_l2(wg[n].grad, w32[n].grad) <= 2e-2, (n, _rel_l2(wg[n].grad, w32[n].grad))


def test_decoder_layer_full_width_gradients_are_finite():
    from aria_b200 import lm_train
    B, T = 1, 2048
    tc = _layer_cfg(2560, 20, 64, 6, 1664)
    layer = _our_layer(tc, _layer_state(tc, seed=1))
    g = torch.Generator().manual_seed(2)
    x = torch.randn(B, T, 2560, generator=g).bfloat16().to(DEV).requires_grad_(True)
    with torch.enable_grad():
        out = lm_train.decoder_layer_train(layer, x)
        out.backward(torch.randn(B, T, 2560, generator=g).bfloat16().to(DEV))
    assert torch.isfinite(out).all() and torch.isfinite(x.grad).all()
    for n, p_ in layer.named_parameters():
        assert p_.grad is not None and torch.isfinite(p_.grad).all(), n
