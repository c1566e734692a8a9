"""Forward + backward of one full-width decoder layer (d=2560, H=20, E=64, top-6, I=1664, two shared experts) at the training
recipe's batch (B=8, T=2048), CUDA events after warm-up, split into its parts: the attention sub-block (q/k/v GEMM + RoPE,
attention, o_proj, and their backward), the two RMSNorms (forward + backward each), the MoE block (moe_train.MoELayerFunction)
and the residual add; then the whole `lm_train.decoder_layer_train`.

    python scripts/bench_decoder_train.py [--out FILE.json] [--B 8] [--T 2048] [--iters 5]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from aria_b200 import lm_train, moe_lm, moe_train  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def timed(fn, iters, reset):
    for _ in range(2):
        reset()
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        reset()   # gradients written, not accumulated (no extra add in the timed window)
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3   # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--B", type=int, default=8)
    ap.add_argument("--T", type=int, default=2048)
    ap.add_argument("--iters", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_decoder_train.py needs a CUDA device")
    B, T, d, H = a.B, a.T, 2560, 20
    cfg = moe_lm.AriaMoELMConfig(hidden_size=d, num_attention_heads=H, num_hidden_layers=1, moe_intermediate_size=1664,
                                 moe_num_experts=64, moe_topk=6, moe_num_shared_experts=2, rms_norm_eps=1e-5, rope_theta=5e6)
    layer = moe_lm.MoEDecoderLayer(cfg, 0, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    with torch.no_grad():
        for n, p in layer.named_parameters():
            if n.endswith("layernorm.weight"):
                p.copy_(1 + 0.1 * torch.randn(p.shape, device="cuda", generator=g))
            else:
                p.copy_(0.02 * torch.randn(p.shape, device="cuda", generator=g))
            p.requires_grad_(True)
    x = torch.randn(B, T, d, device="cuda", generator=g).bfloat16().requires_grad_(True)
    gout = torch.randn(B, T, d, device="cuda", generator=g).bfloat16()
    at = layer.self_attn
    rope = lm_train.rope_tables(cfg.rope_theta, T, "cuda")
    h = torch.randn(B, T, d, device="cuda", generator=g).bfloat16().requires_grad_(True)
    res = torch.randn(B, T, d, device="cuda", generator=g).bfloat16().requires_grad_(True)

    def attention():
        out = lm_train.AttentionFunction.apply(h, res, at.q_proj.weight, at.k_proj.weight, at.v_proj.weight, at.o_proj.weight, H,
                                               rope, None, None)
        out.backward(gout)

    def norm():
        y, r = lm_train.RMSNormFunction.apply(x, layer.input_layernorm.weight, cfg.rms_norm_eps)
        torch.autograd.backward([y, r], [gout, gout])

    def moe():
        moe_train.moe_layer_train(layer.mlp, h).backward(gout)

    def residual_add():
        lm_train.ResidualAddFunction.apply(h, res).backward(gout)

    def reset():
        layer.zero_grad(set_to_none=True)
        x.grad = h.grad = res.grad = None

    def whole():
        lm_train.decoder_layer_train(layer, x).backward(gout)

    info = dict(card=card(), torch=torch.__version__, B=B, T=T, d=d, H=H, E=64, k=6, I=1664)
    print(info, flush=True)
    with torch.enable_grad():
        parts = dict(attention_us=timed(attention, a.iters, reset), norm_us=timed(norm, a.iters, reset), moe_us=timed(moe, a.iters, reset),
                     residual_add_us=timed(residual_add, a.iters, reset))
        parts["norms_us"] = 2 * parts.pop("norm_us")
        parts["layer_us"] = timed(whole, a.iters, reset)
    parts["sum_of_parts_us"] = parts["attention_us"] + parts["norms_us"] + parts["moe_us"] + parts["residual_add_us"]
    for n in ("attention_us", "norms_us", "moe_us", "residual_add_us"):
        parts[n.replace("_us", "_share")] = parts[n] / parts["sum_of_parts_us"]
    info.update(parts)
    info["card_after"] = card()
    print(json.dumps(parts, indent=1), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
