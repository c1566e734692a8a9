"""Timing of the causal attention training kernels (CUDA events, after warm-up): aria_attention_fwd against
aria_attention_fwd_lse (the same kernel plus the lse store; launched alternately, several rounds, so that the spread shows), and
aria_attention_bwd (Delta + dK/dV + dQ kernels).  Three input sets rotate; at every shape they exceed the 126 MB L2 together.

    python scripts/bench_attn_bwd.py [--out FILE.json] [--quick]

FLOPs: the causal forward needs 4*B*H*128*T(T+1)/2 (QK^T and PV over the visible pairs); the backward 2.5x that (five
GEMMs: S, dP, dV, dK, dQ — "algorithmic"), and this implementation executes seven (the dQ kernel recomputes S and dP —
"executed").  Shares are given against the data-sheet dense BF16 rate (2250 TF/s at 1000 W) and against 1480 TF/s, the
sustained rate this project measured for its GEMMs on a B200."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from aria_b200 import ops  # noqa: E402

PEAK_SHEET, PEAK_SUSTAINED = 2250.0, 1480.0   # TF/s
SCALE = 128 ** -0.5


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def events_time(fn, sets, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(*sets[i % len(sets)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3   # us


def run(B, H, T, iters, rounds, nsets=3):
    g = torch.Generator(device="cuda").manual_seed(0)
    sets = []
    for _ in range(nsets):
        q, k, v = (torch.randn(B, H, T, 128, device="cuda", generator=g).bfloat16() for _ in range(3))
        dout = torch.randn(B, T, H * 128, device="cuda", generator=g).bfloat16()
        o, lse = ops.attention_fwd_lse(q, k, v, SCALE)
        sets.append((q, k, v, dout, o, lse))
    fwd = lambda q, k, v, *_: ops.attention(q, k, v, T, T, SCALE, causal=True)          # noqa: E731
    fwd_lse = lambda q, k, v, *_: ops.attention_fwd_lse(q, k, v, SCALE)                 # noqa: E731
    bwd = lambda q, k, v, dout, o, lse: ops.attention_bwd(q, k, v, o, dout, lse, SCALE)  # noqa: E731
    for f in (fwd, fwd_lse, bwd):      # warm-up: module load, smem opt-in, every input set
        for s in sets:
            f(*s)
    torch.cuda.synchronize()
    t_fwd, t_lse, t_bwd = [], [], []
    for _ in range(rounds):            # alternate the two forwards: a drift in clocks hits both
        t_fwd.append(events_time(fwd, sets, iters))
        t_lse.append(events_time(fwd_lse, sets, iters))
        t_bwd.append(events_time(bwd, sets, iters))
    fl_fwd = 4.0 * B * H * 128 * T * (T + 1) / 2
    fl_alg, fl_exec = 2.5 * fl_fwd, 3.5 * fl_fwd
    tb = min(t_bwd)
    res = dict(B=B, H=H, T=T, iters=iters, rounds=rounds,
               fwd_us=t_fwd, fwd_lse_us=t_lse, bwd_us=t_bwd,
               fwd_lse_over_fwd=min(t_lse) / min(t_fwd),
               fwd_tflops=fl_fwd / min(t_fwd) / 1e6,
               bwd_tflops_algorithmic=fl_alg / tb / 1e6, bwd_tflops_executed=fl_exec / tb / 1e6)
    res["bwd_share_sheet_algorithmic"] = res["bwd_tflops_algorithmic"] / PEAK_SHEET
    res["bwd_share_sustained_algorithmic"] = res["bwd_tflops_algorithmic"] / PEAK_SUSTAINED
    res["bwd_share_sheet_executed"] = res["bwd_tflops_executed"] / PEAK_SHEET
    res["bwd_share_sustained_executed"] = res["bwd_tflops_executed"] / PEAK_SUSTAINED
    print(f"B={B} H={H} T={T}: fwd {min(t_fwd):9.1f} us (spread {max(t_fwd) - min(t_fwd):6.1f}) | fwd_lse {min(t_lse):9.1f} us "
          f"(spread {max(t_lse) - min(t_lse):6.1f}) ratio {res['fwd_lse_over_fwd']:.3f} | bwd {tb:9.1f} us = "
          f"{res['bwd_tflops_algorithmic']:6.1f} TF/s algorithmic ({res['bwd_share_sheet_algorithmic']:.2f} of 2250, "
          f"{res['bwd_share_sustained_algorithmic']:.2f} of 1480), {res['bwd_tflops_executed']:6.1f} TF/s executed "
          f"({res['bwd_share_sheet_executed']:.2f} / {res['bwd_share_sustained_executed']:.2f})", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="recipe shape only, few iterations")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attn_bwd.py needs a CUDA device")
    info = dict(card=card(), torch=torch.__version__)
    print(info, flush=True)
    shapes = [(8, 20, 2048, 20, 5), (1, 20, 8192, 20, 5), (1, 20, 32768, 3, 3)]
    if a.quick:
        shapes = [(8, 20, 2048, 5, 2)]
    info["results"] = [run(B, H, T, it, rd) for B, H, T, it, rd in shapes]
    info["card_after"] = card()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
