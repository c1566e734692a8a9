"""Whole-model training measurements on one GPU, CUDA events after warm-up (median, min and max over the timed iterations):

  1. the fused lm_head + cross-entropy at the recipe shape (M = B*T = 16384 rows, V = 100352, d = 2560): forward, backward,
     a plain `ops.linear` lm_head of the same shape (the forward's GEMM without the stats epilogue), algorithmic TF/s
     (2*M*V*d per GEMM: 1 in the forward, 3 in the backward) and the peak memory growth of forward + backward, against
     `ops.linear` + `F.cross_entropy(logits.float())` with autograd through the loss on the same shape;
  2. one training step (forward + backward, no optimizer) of the 28-layer, 25.3 B Aria language model at B = 8, T = 2048,
     random init, with per-layer gradient checkpointing: step time, tokens/s, peak memory; then whether the same step
     fits without checkpointing.

    python scripts/bench_lm_train.py [--out FILE.json] [--iters 10] [--steps 3] [--skip-model]"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from aria_b200 import configs, lm_train, moe_lm, ops  # noqa: E402
from aria_b200.modeling_aria import init_random_  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def timed(fn, iters, warmup=2):
    """-> (median, min, max) milliseconds of fn over `iters` event-timed calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return dict(median_ms=statistics.median(ts), min_ms=min(ts), max_ms=max(ts), n=iters)


def peak_growth(fn):
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def bench_loss(iters):
    M, V, d = 16384, 100352, 2560
    g = torch.Generator(device="cuda").manual_seed(0)
    h = torch.randn(M, d, device="cuda", generator=g).bfloat16()
    w = (torch.randn(V, d, device="cuda", generator=g) * d ** -0.5).bfloat16()
    t = torch.randint(0, V, (M,), device="cuda", generator=g).to(torch.int32)
    st = {}

    def fwd():
        st["f"] = ops.lm_xent_fwd(h, w, t)

    def bwd():
        loss, lse, nv = st["f"]
        ops.lm_xent_bwd(h, w, t, lse, nv, torch.ones(1, device="cuda"))

    def plain():
        ops.linear(h, w)

    fwd()
    r = dict(M=M, V=V, d=d, fwd=timed(fwd, iters), bwd=timed(bwd, iters), linear_lm_head=timed(plain, iters))
    flop = 2.0 * M * V * d
    r["fwd_tflops"] = flop / (r["fwd"]["median_ms"] * 1e-3) / 1e12
    r["bwd_tflops"] = 3 * flop / (r["bwd"]["median_ms"] * 1e-3) / 1e12
    r["linear_tflops"] = flop / (r["linear_lm_head"]["median_ms"] * 1e-3) / 1e12
    r["stats_epilogue_overhead"] = r["fwd"]["median_ms"] / r["linear_lm_head"]["median_ms"] - 1
    del st["f"]

    hg, wg = h.clone().requires_grad_(True), w.clone().requires_grad_(True)

    def fused_step():
        with torch.enable_grad():
            lm_train.LMHeadCrossEntropyFunction.apply(hg, wg, t).backward()
        hg.grad = wg.grad = None   # the peak still counts them: subtracted below

    def unfused_step():
        with torch.enable_grad():
            z = ops.linear(hg, wg).requires_grad_(True)
            F.cross_entropy(z.float(), t.long()).backward()

    grads = (hg.numel() + wg.numel()) * 2
    r["fused_peak_growth_bytes_beyond_grads"] = peak_growth(fused_step) - grads
    r["unfused_peak_growth_bytes"] = peak_growth(unfused_step)
    return r


def bench_model(steps):
    tc = dict(configs.ARIA_25B["text_config"])
    cfg = moe_lm.AriaMoELMConfig(**tc)
    lm = moe_lm.AriaMoELMForCausalLM(cfg, device="cuda")
    with torch.no_grad():
        init_random_(lm, seed=0)
    for p in lm.parameters():
        p.requires_grad_(True)
    n_params = sum(p.numel() for p in lm.parameters())
    B, T = 8, 2048
    g = torch.Generator(device="cuda").manual_seed(1)
    ids = torch.randint(0, cfg.vocab_size, (B, T), device="cuda", generator=g)

    def step(ckpt):
        lm.zero_grad(set_to_none=False)
        with torch.enable_grad():
            loss = lm_train.causal_lm_loss(lm, ids, input_ids=ids, gradient_checkpointing=ckpt)
            loss.backward()
        return loss

    r = dict(params=n_params, B=B, T=T, layers=cfg.num_hidden_layers)
    step(True)      # warm-up; allocates the gradients
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t = timed(lambda: step(True), steps, warmup=0)
    r["ckpt_step"] = t
    r["ckpt_tokens_per_s"] = B * T / (t["median_ms"] * 1e-3)
    r["ckpt_peak_bytes"] = torch.cuda.max_memory_allocated()
    r["loss"] = float(step(True).detach())
    try:
        torch.cuda.reset_peak_memory_stats()
        t0 = time.time()
        step(False)
        torch.cuda.synchronize()
        r["no_ckpt_fits"] = True
        r["no_ckpt_step_s_first"] = time.time() - t0
        r["no_ckpt_peak_bytes"] = torch.cuda.max_memory_allocated()
    except torch.cuda.OutOfMemoryError as e:
        r["no_ckpt_fits"] = False
        r["no_ckpt_error"] = str(e).splitlines()[0][:200]
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--skip-model", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lm_train.py needs a CUDA device")
    info = dict(card=card(), torch=torch.__version__)
    print(info, flush=True)
    info["lm_head_loss"] = bench_loss(a.iters)
    print(json.dumps(info["lm_head_loss"], indent=1), flush=True)
    gc.collect()
    torch.cuda.empty_cache()
    if not a.skip_model:
        info["model_step"] = bench_model(a.steps)
        print(json.dumps(info["model_step"], indent=1), flush=True)
    info["card_after"] = card()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
