"""CPU: the oracle restatement (oracle/aria_oracle.py) reproduces the golden vectors that
oracle/make_golden.py captured from the UNMODIFIED reference modules (tests/golden/*.pt)."""
import os

import pytest
import torch

from oracle import aria_oracle as O
from oracle import configs as C

GOLD = os.path.join(os.path.dirname(__file__), "golden")
torch.set_grad_enabled(False)


def _load(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


@pytest.mark.parametrize("tag,dtype,tol", [("fp32", torch.float32, 1e-6), ("bf16", torch.bfloat16, 0.0)])
def test_moe_layer_cfg1(tag, dtype, tol):
    """BASELINE.json configs[0]: d=256, 8 experts, top-2, every intermediate of MoELayer.forward."""
    g = _load(f"moe_layer_cfg1_{tag}.pt")
    gen = torch.Generator().manual_seed(g["seed"])
    sd = C.moe_layer_state(C.TINY["text_config"], gen)
    sd = {k: v.to(dtype) for k, v in sd.items()}
    assert C.state_checksum(sd) == pytest.approx(g["checksum"], rel=1e-9), "seeded weights drifted"
    out, p = O.moe_layer(g["x"], sd, 2, return_parts=True)
    # expert sets are identical (no ties in this fixture); order within a row follows the logits
    assert torch.equal(p["top_idx"].sort(1).values, g["top_idx"].sort(1).values)
    assert torch.equal(p["counts"], g["counts"].to(torch.int64))
    # align score columns by expert id before comparing
    o = torch.argsort(p["top_idx"], 1)
    go = torch.argsort(g["top_idx"], 1)
    assert (p["scores"].gather(1, o).float() - g["scores"].gather(1, go).float()).abs().max() <= tol
    assert (p["expert_out"].float() - g["expert_out"].float()).abs().max() <= tol * 10
    assert torch.equal(p["permuted"], g["permuted"])
    assert (p["shared"].float() - g["shared"].float()).abs().max() <= tol * 10
    assert (out.float() - g["out"].float()).abs().max() <= tol * 10


@pytest.mark.parametrize("tag,dtype,tol", [("fp32", torch.float32, 1e-6), ("bf16", torch.bfloat16, 0.0)])
def test_moe_layer_training_mode_gradients(tag, dtype, tol):
    """Training-mode routing (z-loss + load-balancing loss through MoEAuxLossAutoScaler, moe_lm.py:84-166, 203-241, with a
    loss scale of 8): every parameter gradient of the unmodified reference, captured by oracle/make_golden.py."""
    g = _load(f"moe_layer_train_{tag}.pt")
    gen = torch.Generator().manual_seed(g["seed"])
    sd = C.moe_layer_state(g["text_config"], gen)
    sd["router.weight"] = sd["router.weight"] * 20
    sd = {k: v.to(dtype) for k, v in sd.items()}
    assert C.state_checksum(sd) == pytest.approx(g["checksum"], rel=1e-9), "seeded weights drifted"
    w = {n: v.clone().requires_grad_(True) for n, v in sd.items()}
    x = g["x"].clone().requires_grad_(True)
    O._LossGradInjector.scale = g["loss_scale"]
    try:
        with torch.enable_grad():
            out = O.moe_layer(x, w, g["text_config"]["moe_topk"], loss_coeffs=(g["z_coeff"], g["aux_coeff"]))
            out.backward(g["dout"])
    finally:
        O._LossGradInjector.scale = 1.0
    assert (out.detach().float() - g["out"].float()).abs().max() <= tol * 10
    for n, want in g["grads"].items():       # strided sample of each gradient (oracle/make_golden.py: strided_sample)
        scale = max(1.0, float(want.float().abs().max()))
        got = w[n].grad.reshape(-1)[::g["grad_strides"][n]]
        assert (got.float() - want.float()).abs().max() <= tol * scale, n
    # dx sums three autograd branches; bf16 accumulation order is an engine detail -> ulp-level tolerance there
    xtol = 1e-6 if dtype == torch.float32 else 1e-2
    assert (x.grad.float() - g["dx"].float()).abs().max() <= xtol * max(1.0, float(g["dx"].float().abs().max()))
    # the losses really contribute: the router gradient differs from the eval-mode one
    w0 = {n: v.clone().requires_grad_(True) for n, v in sd.items()}
    with torch.enable_grad():
        O.moe_layer(g["x"].clone(), w0, g["text_config"]["moe_topk"]).backward(g["dout"])
    d_router = w0["router.weight"].grad.reshape(-1)[::g["grad_strides"]["router.weight"]]
    assert (d_router.float() - g["grads"]["router.weight"].float()).abs().max() > 1e-3


@pytest.mark.parametrize("tag,tol", [("fp32", 1e-6), ("bf16", 0.0)])
def test_lora_grouped_gemm_golden(tag, tol):
    """aria/lora/layers.py:125-140 forward and the adapter gradients, captured from the unmodified reference layer."""
    g = _load(f"lora_grouped_gemm_{tag}.pt")
    a, b, x = (g[k].clone().requires_grad_(True) for k in ("a", "b", "x"))
    with torch.enable_grad():
        out = O.grouped_gemm_lora(x, g["w"], a, b, g["counts"], g["lora_alpha"] / g["r"])
        out.backward(g["dy"])
    assert (out.detach().float() - g["out"].float()).abs().max() <= tol
    assert (a.grad.float() - g["d_a"].float()).abs().max() <= tol * max(1.0, float(g["d_a"].float().abs().max()))
    assert (b.grad.float() - g["d_b"].float()).abs().max() <= tol * max(1.0, float(g["d_b"].float().abs().max()))
    xtol = 1e-6 if tag == "fp32" else 1e-2
    assert (x.grad.float() - g["dx"].float()).abs().max() <= xtol * float(g["dx"].float().abs().max())


@pytest.mark.parametrize("tag,dtype,tol", [("fp32", torch.float32, 5e-6), ("bf16", torch.bfloat16, 0.0)])
@pytest.mark.parametrize("masked", ["full", "masked"])
def test_aria_tiny_forward(tag, dtype, tol, masked):
    """ViT -> projector -> merge -> 2-layer MoE LM on the tiny config, incl. a padded pixel_mask."""
    g = _load(f"aria_tiny_{tag}_{masked}.pt")
    cfg = C.TINY
    sd = C.aria_state(cfg, seed=g["seed"], dtype=dtype)
    assert C.state_checksum(sd) == pytest.approx(g["checksum"], rel=1e-9), "seeded weights drifted"
    vit, mask = O.vit_forward(g["pixel_values"], g["pixel_mask"], sd, cfg["vision_config"])
    assert (vit.float() - g["vit"].float()).abs().max() <= tol
    if g["pixel_mask"] is not None:
        assert torch.equal(mask, g["image_attn_mask"])
    proj = O.projector_forward(vit, mask if g["pixel_mask"] is not None else None, sd, cfg["projector"])
    assert (proj.float() - g["projector"].float()).abs().max() <= tol
    logits, _ = O.aria_forward(g["input_ids"], g["pixel_values"], g["pixel_mask"], sd, cfg)
    assert (logits.float() - g["logits"].float()).abs().max() <= tol


def test_image_token_mismatch_raises():
    """modeling_aria.py:268-271: ValueError when <|img|> slots != projector outputs."""
    g = _load("aria_tiny_fp32_full.pt")
    sd = C.aria_state(C.TINY, seed=0)
    ids = g["input_ids"].clone()
    ids[0, 5] = 11  # drop one image slot
    with pytest.raises(ValueError):
        O.aria_forward(ids, g["pixel_values"], None, sd, C.TINY)


def test_topk_tie_rule():
    """Tie rule stated in the oracle header: lowest expert index wins."""
    logits = torch.tensor([[1.0, 3.0, 3.0, 0.5, 3.0, 2.0]], dtype=torch.bfloat16)
    _, idx = O.topk_lowest_index(logits, 2)
    assert idx.tolist() == [[1, 2]]
    s, i, c = O.router_routing(logits, 4)
    assert i.tolist() == [[1, 2, 4, 5]] and c.tolist() == [0, 1, 1, 0, 1, 1]


def test_kv_cache_decode_matches_prefill():
    """Decode with a KV cache reproduces the last prefill position (oracle self-consistency)."""
    cfg = C.TINY
    sd = C.aria_state(cfg, seed=3)
    g = torch.Generator().manual_seed(5)
    ids = torch.randint(10, 512, (1, 12), generator=g)
    import torch.nn.functional as F

    emb = F.embedding(ids, sd["language_model.model.embed_tokens.weight"])
    full, _ = O.lm_forward(emb, sd, cfg["text_config"])
    _, past = O.lm_forward(emb[:, :-1], sd, cfg["text_config"])
    step, _ = O.lm_forward(emb[:, -1:], sd, cfg["text_config"], past=past)
    assert (full[:, -1] - step[:, 0]).abs().max() < 2e-5
