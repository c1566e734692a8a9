"""TEST INFRASTRUCTURE — generate tests/golden/*.pt by running the UNMODIFIED reference modules
(loaded by oracle/ref_loader.py; ARIA_REFERENCE_ROOT names a checkout of rhymes-ai/Aria) on CPU with seeded random weights.

    ARIA_REFERENCE_ROOT=<Aria checkout> python oracle/make_golden.py
Each fixture stores inputs, the reference outputs (and MoE intermediates), and the weight checksum;
weights are re-created from the seed by oracle/configs.py.  Large gradients are stored as a strided sample (`flat[::stride]`,
stride stored beside them; see strided_sample) so that the fixtures stay small.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import aria_oracle as O  # noqa: E402
from oracle import configs as C  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
GRAD_SAMPLE = 4096


def strided_sample(t, n=GRAD_SAMPLE):
    """(flat[::stride], stride) with stride the smallest that leaves at most n elements; tests compare the same positions."""
    stride = -(-t.numel() // n)
    return t.detach().reshape(-1)[::stride].clone(), stride


def build_reference_model(ref, cfg, sd, dtype):
    tc, vc = cfg["text_config"], cfg["vision_config"]
    text = ref.moe_lm.AriaMoELMConfig(
        hidden_size=tc["hidden_size"], num_attention_heads=tc["num_attention_heads"],
        num_key_value_heads=tc["num_attention_heads"], num_hidden_layers=tc["num_hidden_layers"],
        moe_num_experts=tc["moe_num_experts"], moe_topk=tc["moe_topk"],
        moe_intermediate_size=tc["moe_intermediate_size"], moe_num_shared_experts=tc["moe_num_shared_experts"],
        vocab_size=tc["vocab_size"], rms_norm_eps=tc["rms_norm_eps"], rope_theta=tc["rope_theta"],
        intermediate_size=tc["moe_intermediate_size"], max_position_embeddings=4096,
        rope_parameters={"rope_type": "default", "rope_theta": tc["rope_theta"]},
    )
    text._attn_implementation = "eager"
    vis = ref.vision_encoder.AriaVisionConfig(
        hidden_size=vc["hidden_size"], num_attention_heads=vc["num_attention_heads"],
        num_hidden_layers=vc["num_hidden_layers"], intermediate_size=vc["intermediate_size"],
        patch_size=vc["patch_size"], image_size=vc["image_size"], layer_norm_eps=vc["layer_norm_eps"],
        hidden_act="gelu_pytorch_tanh",
    )
    vis._attn_implementation = "eager"
    acfg = ref.configuration_aria.AriaConfig(
        vision_config=vis, text_config=text,
        projector_patch_to_query_dict=cfg["projector"]["patch_to_query_dict"],
        image_token_index=cfg["image_token_index"], attn_implementation="eager", pad_token_id=0,
    )
    model = ref.modeling_aria.AriaForConditionalGeneration(acfg)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    # vision post_layernorm is an IdentityOp in the reference (no params); everything else must match.
    assert not unexpected, unexpected
    assert not [m for m in missing if "rotary" not in m and "inv_freq" not in m], missing
    # `from_pretrained(torch_dtype=bf16)` leaves the fp32 RoPE inv_freq buffer alone; a blanket
    # `.to(bf16)` would round it (harness artefact, not reference behaviour) — so restore it.
    rot = model.language_model.model.rotary_emb
    inv = rot.inv_freq.clone()
    model = model.to(dtype).eval()
    rot.inv_freq = inv
    if hasattr(rot, "original_inv_freq"):
        rot.original_inv_freq = inv.clone()
    return model


def make_inputs(cfg, seed, dtype, n_text=24, masked=False):
    g = torch.Generator().manual_seed(seed)
    vc = cfg["vision_config"]
    S = vc["image_size"]
    N = (S // vc["patch_size"]) ** 2
    Q = cfg["projector"]["patch_to_query_dict"][N]
    V = cfg["text_config"]["vocab_size"]
    pixel_values = torch.randn(1, 3, S, S, generator=g).to(dtype)
    text = torch.randint(10, V, (n_text,), generator=g)
    ids = torch.cat([text[:4], torch.full((Q,), cfg["image_token_index"]), text[4:]])[None]
    pixel_mask = None
    if masked:
        pixel_mask = torch.ones(1, S, S, dtype=torch.bool)
        pixel_mask[:, :, S - 2 * vc["patch_size"]:] = False  # right two patch columns padded
    return ids, pixel_values, pixel_mask


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = load_reference()
    torch.set_grad_enabled(False)
    cfg = C.TINY
    report = []

    # ---- (1) BASELINE cfg 1: one MoELayer, d=256, E=8, k=2, I=512; x [2,16,256]; fp32 and bf16 ----
    for dtype, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        gen = torch.Generator().manual_seed(1)
        sd = C.moe_layer_state(cfg["text_config"], gen)
        x = torch.randn(2, 16, 256, generator=gen)
        sd = {k: v.to(dtype) for k, v in sd.items()}
        x = x.to(dtype)
        tcfg = ref.moe_lm.AriaMoELMConfig(hidden_size=256, moe_num_experts=8, moe_topk=2,
                                          moe_intermediate_size=512, moe_num_shared_experts=2)
        layer = ref.moe_lm.MoELayer(tcfg)
        layer.load_state_dict(sd, strict=True)
        layer = layer.to(dtype).eval()
        # intermediates straight from the reference sub-modules (moe_lm.py:565-576)
        scores, idx, counts = layer.router(x)
        perm = layer.token_dispatcher.token_permutation(x, idx)
        eo = layer.experts(perm, counts)
        comb = layer.token_dispatcher.token_unpermutation(eo, scores)
        shared = layer.shared_experts(x)
        out = layer(x)
        o_out, parts = O.moe_layer(x, sd, 2, return_parts=True)
        same_sets = bool((idx.sort(1).values == parts["top_idx"].sort(1).values).all())
        err = float((out.float() - o_out.float()).abs().max())
        report.append(f"moe_layer {tag}: oracle-vs-reference max abs err {err:.3e}, same expert sets {same_sets}")
        torch.save(dict(x=x, scores=scores, top_idx=idx, counts=counts, permuted=perm, expert_out=eo,
                        combined=comb, shared=shared, out=out, checksum=C.state_checksum(sd), seed=1),
                   os.path.join(OUT, f"moe_layer_cfg1_{tag}.pt"))

    # ---- (1b) training-mode routing: the same layer in .train(), forward + backward with the z-loss / load-balancing loss
    # side effects (moe_lm.py:84-166, 203-241) and a non-unit MoEAuxLossAutoScaler scale; reference gradients are the golden
    for dtype, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        gen = torch.Generator().manual_seed(3)
        ttc = dict(hidden_size=128, moe_num_experts=8, moe_topk=2, moe_intermediate_size=64, moe_num_shared_experts=2)
        sd = C.moe_layer_state(ttc, gen)                    # small layer: the fixture stores a sample of every parameter gradient
        sd["router.weight"] = sd["router.weight"] * 20      # spread the logits so the loss terms are well above rounding noise
        x = torch.randn(2, 16, 128, generator=gen)
        dout = torch.randn(2, 16, 128, generator=gen)
        sd = {k: v.to(dtype) for k, v in sd.items()}
        x, dout = x.to(dtype), dout.to(dtype)
        z_c, aux_c, scale = 0.5, 2.0, 8.0
        tcfg = ref.moe_lm.AriaMoELMConfig(moe_z_loss_coeff=z_c, moe_aux_loss_coeff=aux_c, **ttc)
        with torch.enable_grad():
            layer = ref.moe_lm.MoELayer(tcfg)
            layer.load_state_dict(sd, strict=True)
            layer = layer.to(dtype).train()
            ref.moe_lm.MoEAuxLossAutoScaler.set_loss_scale(torch.tensor(scale))
            try:
                xr = x.clone().requires_grad_(True)
                out = layer(xr)
                out.backward(dout)
            finally:
                ref.moe_lm.MoEAuxLossAutoScaler.set_loss_scale(torch.tensor(1.0))
            grads = {n: strided_sample(p.grad) for n, p in layer.named_parameters()}
            w = {n: v.clone().requires_grad_(True) for n, v in sd.items()}
            xo = x.clone().requires_grad_(True)
            O._LossGradInjector.scale = scale
            try:
                O.moe_layer(xo, w, 2, loss_coeffs=(z_c, aux_c)).backward(dout)
            finally:
                O._LossGradInjector.scale = 1.0
        err = max(float((g.float() - w[n].grad.reshape(-1)[::st].float()).abs().max()) for n, (g, st) in grads.items())
        report.append(f"moe_layer train-mode grads {tag}: oracle-vs-reference max abs err over parameter grads {err:.3e}")
        torch.save(dict(x=x, dout=dout, out=out.detach(), grads={n: g for n, (g, _) in grads.items()},
                        grad_strides={n: st for n, (_, st) in grads.items()}, dx=xr.grad.detach(), z_coeff=z_c, aux_coeff=aux_c,
                        loss_scale=scale, checksum=C.state_checksum(sd), seed=3, text_config=ttc),
                   os.path.join(OUT, f"moe_layer_train_{tag}.pt"))

    # ---- (1c) LoRA on the grouped expert GEMM: the unmodified aria/lora/layers.py under the peft stand-in of ref_loader ----
    from oracle.ref_loader import load_reference_lora
    lora_mod = load_reference_lora()
    for dtype, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        gen = torch.Generator().manual_seed(4)
        E, K, N, r, alpha = 4, 128, 192, 8, 32
        counts = torch.tensor([32, 0, 80, 16])                        # 16-row aligned groups, one empty
        rows = int(counts.sum())
        w = (torch.randn(E, K, N, generator=gen) * 0.05).to(dtype)
        a = (torch.randn(E, K, r, generator=gen) * 0.05).to(dtype)
        b = (torch.randn(E, r, N, generator=gen) * 0.05).to(dtype)
        x = torch.randn(rows, K, generator=gen).to(dtype)
        dy = torch.randn(rows, N, generator=gen).to(dtype)
        with torch.enable_grad():
            base = ref.moe_lm.GroupedGEMM(K, N, E)
            layer = lora_mod.GroupedGemmLoraLayer(base, "default", r=r, lora_alpha=alpha).to(dtype)
            with torch.no_grad():
                base.weight.copy_(w)
                layer.lora_A["default"].weight.copy_(a)
                layer.lora_B["default"].weight.copy_(b)
            xr = x.clone().requires_grad_(True)
            out = layer(xr, counts)
            out.backward(dy)
        o_out = O.grouped_gemm_lora(x, w, a, b, counts, alpha / r)
        err = float((out.detach().float() - o_out.float()).abs().max())
        report.append(f"lora grouped gemm {tag}: oracle-vs-reference max abs err {err:.3e}")
        torch.save(dict(x=x, dy=dy, w=w, a=a, b=b, counts=counts, r=r, lora_alpha=alpha, out=out.detach(),
                        d_a=layer.lora_A["default"].weight.grad.detach(), d_b=layer.lora_B["default"].weight.grad.detach(),
                        dx=xr.grad.detach()),
                   os.path.join(OUT, f"lora_grouped_gemm_{tag}.pt"))

    # ---- (2) tiny full model: ViT + projector + merge + 2-layer MoE LM ----
    for dtype, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        sd = C.aria_state(cfg, seed=0, dtype=dtype)
        model = build_reference_model(ref, cfg, sd, dtype)
        for masked in (False, True):
            ids, pv, pm = make_inputs(cfg, seed=2, dtype=dtype, masked=masked)
            vit_out, img_mask = model.vision_tower(pv, pixel_mask=pm)
            vit_h = vit_out.last_hidden_state
            proj = model.multi_modal_projector(vit_h, attn_mask=img_mask)
            out = model(input_ids=ids, pixel_values=pv, pixel_mask=pm, use_cache=False)
            logits = out.logits
            o_vit, o_mask = O.vit_forward(pv, pm, sd, cfg["vision_config"])
            o_proj = O.projector_forward(o_vit, o_mask if pm is not None else None, sd, cfg["projector"])
            o_logits, _ = O.aria_forward(ids, pv, pm, sd, cfg)
            e1 = float((vit_h.float() - o_vit.float()).abs().max())
            e2 = float((proj.float() - o_proj.float()).abs().max())
            e3 = float((logits.float() - o_logits.float()).abs().max())
            report.append(f"aria tiny {tag} masked={masked}: vit {e1:.3e} proj {e2:.3e} logits {e3:.3e} "
                          f"(|logits| max {float(logits.float().abs().max()):.3f})")
            torch.save(dict(input_ids=ids, pixel_values=pv, pixel_mask=pm, vit=vit_h, image_attn_mask=img_mask,
                            projector=proj, logits=logits, checksum=C.state_checksum(sd), seed=0),
                       os.path.join(OUT, f"aria_tiny_{tag}_{'masked' if masked else 'full'}.pt"))

    # ---- (3) the cases of tests/test_oracle_vs_reference.py: same seeds and shapes as the tests, reference outputs only ----
    live = {}
    for dtype, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        for T, E, k in ((1, 8, 2), (7, 8, 2), (64, 16, 6), (33, 64, 6)):
            tc = dict(hidden_size=128, moe_num_experts=E, moe_topk=k, moe_intermediate_size=64, moe_num_shared_experts=2)
            gen = torch.Generator().manual_seed(T * 131 + E)
            sd = {n: v.to(dtype) for n, v in C.moe_layer_state(tc, gen).items()}
            x = torch.randn(1, T, 128, generator=gen).to(dtype)
            layer = ref.moe_lm.MoELayer(ref.moe_lm.AriaMoELMConfig(**tc))
            layer.load_state_dict(sd, strict=True)
            layer = layer.to(dtype).eval()
            _, ridx, _ = layer.router(x)
            live[f"{tag}_T{T}_E{E}_k{k}"] = dict(out=layer(x), top_idx=ridx, checksum=C.state_checksum(sd),
                                                 x_checksum=float(x.double().sum()))
    torch.save(live, os.path.join(OUT, "moe_layer_live.pt"))

    train_live = {}
    for dtype, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        T, E, k, d = 48, 16, 4, 128
        tc = dict(hidden_size=d, moe_num_experts=E, moe_topk=k, moe_intermediate_size=64, moe_num_shared_experts=2,
                  moe_z_loss_coeff=0.5, moe_aux_loss_coeff=2.0)
        gen = torch.Generator().manual_seed(5)
        sd = {n: v.to(dtype) for n, v in C.moe_layer_state(tc, gen).items()}
        sd["router.weight"] = (sd["router.weight"].float() * 20).to(dtype)
        x0 = torch.randn(1, T, d, generator=gen).to(dtype)
        dout = torch.randn(1, T, d, generator=gen).to(dtype)
        fix = dict(checksum=C.state_checksum(sd), x_checksum=float(x0.double().sum()) + float(dout.double().sum()))
        for scale in (1.0, 64.0):
            with torch.enable_grad():
                layer = ref.moe_lm.MoELayer(ref.moe_lm.AriaMoELMConfig(**tc))
                layer.load_state_dict(sd, strict=True)
                layer = layer.to(dtype).train()
                ref.moe_lm.MoEAuxLossAutoScaler.set_loss_scale(torch.tensor(scale))
                try:
                    xr = x0.clone().requires_grad_(True)
                    layer(xr).backward(dout)
                finally:
                    ref.moe_lm.MoEAuxLossAutoScaler.set_loss_scale(torch.tensor(1.0))
            grads = {n: strided_sample(p.grad, 1024) for n, p in layer.named_parameters()}
            fix[scale] = dict(grads={n: g for n, (g, _) in grads.items()}, grad_strides={n: st for n, (_, st) in grads.items()},
                              grad_absmax={n: float(p.grad.float().abs().max()) for n, p in layer.named_parameters()},
                              dx=xr.grad.detach())
        train_live[tag] = fix
    torch.save(train_live, os.path.join(OUT, "moe_layer_train_live.pt"))

    lora_live = {}
    for dtype, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        g = torch.Generator().manual_seed(4)
        E, K, N, r, alpha = 4, 64, 96, 8, 32
        counts = torch.tensor([16, 0, 40, 24])
        rows = int(counts.sum())
        w = (torch.randn(E, K, N, generator=g) * 0.05).to(dtype)
        a = (torch.randn(E, K, r, generator=g) * 0.05).to(dtype)
        b = (torch.randn(E, r, N, generator=g) * 0.05).to(dtype)
        x0 = torch.randn(rows, K, generator=g).to(dtype)
        dy = torch.randn(rows, N, generator=g).to(dtype)
        with torch.enable_grad():
            base = ref.moe_lm.GroupedGEMM(K, N, E)
            layer = lora_mod.GroupedGemmLoraLayer(base, "default", r=r, lora_alpha=alpha).to(dtype)
            with torch.no_grad():
                base.weight.copy_(w)
                layer.lora_A["default"].weight.copy_(a)
                layer.lora_B["default"].weight.copy_(b)
            xr = x0.clone().requires_grad_(True)
            out = layer(xr, counts)
            out.backward(dy)
        fix = dict(x_checksum=float(x0.double().sum()), scaling=layer.scaling["default"], out=out.detach(),
                   d_a=layer.lora_A["default"].weight.grad.detach(), d_b=layer.lora_B["default"].weight.grad.detach(),
                   dx=xr.grad.detach())
        if dtype == torch.float32:
            with torch.no_grad():
                layer.merge()
                merged_weight, stride = strided_sample(base.weight)
                fix.update(merged_out=layer(x0, counts), merged_weight=merged_weight, merged_weight_stride=stride)
        lora_live[tag] = fix
    torch.save(lora_live, os.path.join(OUT, "lora_layer_live.pt"))
    print("\n".join(report))
    with open(os.path.join(OUT, "REPORT.txt"), "w") as f:
        f.write("oracle/make_golden.py — oracle restatement vs unmodified reference, at generation time\n")
        f.write("\n".join(report) + "\n")


if __name__ == "__main__":
    main()
