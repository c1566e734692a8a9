#!/usr/bin/env python
"""bench.py — Aria-25.3B bf16 prefill tokens/s on B200 (BASELINE.json metric), one process per GPU.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the UNMODIFIED reference's CPU forward on the host cores (oracle/_ref)
    python bench.py --workload cfg3|cfg4|cfg5 # the other BASELINE.json configs (decode, 64K prefill, EP fwd+bwd unit)
    python bench.py --dump-outputs DIR        # also write what the last timed step computed as DIR/<name>.npy (float32)

Default workload (BASELINE.json configs[1], SURVEY.md §8d cfg 2): random-init Aria-25.3B (seed 0), one synthetic
980x980 image (4900 patches -> 256 image tokens) + 512 random text tokens => T = 768 prefill tokens,
num_logits_to_keep=1, batch 1, no KV cache in.  A "step" = one AriaForConditionalGeneration.forward() per rank.

Printed JSON (rank 0, one line):
  value        whole-job tokens/s with inputs already resident in HBM (CUDA events, max over ranks)
  e2e          same metric through the public API with HOST (pinned) buffers: H2D of the step's inputs and D2H of its
               result inside the timed region, every step
  kernels      per-kernel table of the step (CUDA events around every C-ABI call of K eager steps): launches/step,
               ms/step, share of the step, algorithmic FLOPs and bytes per launch, the roofline that bounds it (the slower
               of FLOPs / measured bf16 peak and bytes / measured HBM peak) and the fraction of it achieved
  roofline     the DOMINANT kernel of that table (largest share of the step), in the contract's format
  cpu_baseline the unmodified reference (kind "reference"; oracle port if it is not staged) timed on the host cores on a
               bounded sample of the same workload
--dump-outputs DIR writes, after the timed steps, the arrays the timed path returned in its last step (rank 0): the logits for
cfg2/3/4; dx and every weight gradient for cfg5.  Every input is seeded, so two builds run with the same arguments can be
compared array by array.  An array of more than DUMP_BUDGET / 4 / (number of arrays) elements is replaced by a fixed, seeded
sample of its elements (same positions in every run), so that a dump stays within DUMP_BUDGET bytes.
Multi-GPU (--gpus N > 1): every rank prefills its own request (weak scaling) and the routed experts of every MoE layer are
SHARDED over the ranks — token rows travel over NVLink peer memory (aria_b200/expert_parallel.py); `--multi replicas` runs N
independent replicas instead (no data-path collective).  See DESIGN.md §5.
"""
import argparse
import collections
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_TEXT, T_IMG = 512, 256
T_TOTAL = T_TEXT + T_IMG
DUMP_BUDGET = 64 << 20      # bytes written by --dump-outputs
METRICS = {
    "cfg2": "Aria-25.3B bf16 prefill tokens/sec",
    "cfg3": "Aria-25.3B bf16 decode tokens/sec (batch 32, 2K KV cache)",
    "cfg4": "Aria-25.3B bf16 64K-context prefill tokens/sec",
    "cfg5": "Aria-25.3B MoE layer expert-parallel forward+backward tokens/sec",
}
WORKLOADS = {
    "cfg2": ("cfg2: Aria-25.3B, one 980px image (4900 patches -> 256 image tokens) + 512 text tokens, T=768 prefill, "
             "batch 1, num_logits_to_keep=1, random-init weights"),
    "cfg3": "cfg3: Aria-25.3B decode step, batch 32 against a 2048-token KV cache (28 layers), random-init weights",
    "cfg4": ("cfg4: Aria-25.3B 64K-context video prefill: 32 synthetic 980px frames (8192 image tokens) + 57344 text tokens, "
             "T=65536, batch 1, num_logits_to_keep=1"),
    "cfg5": ("cfg5: ONE full-width MoELayer (d=2560, E=64, k=6, I=1664) forward+backward, 8192 tokens per rank, experts "
             "sharded over the ranks (token all-to-all), eval-mode routing (aux/z losses off)"),
}


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        return self.summarise(self.rows)

    @staticmethod
    def summarise(rows):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ per-kernel table
def op_work(name, a, k):
    """(label, algorithmic FLOPs, algorithmic bytes) of one C-ABI call, from its argument shapes (SURVEY §8d formulas).
    Bytes = every operand read once + the result written once (bf16), weights of ALL experts for a grouped GEMM."""
    bf = 2

    def rows(x):
        return x.numel() // x.shape[-1]

    if name == "linear":
        x, w = a[0], a[1]
        M, (N, K) = rows(x), w.shape
        res = k.get("residual", a[4] if len(a) > 4 else None)
        return f"linear[{M}x{N}x{K}]", 2 * M * N * K, bf * (M * K + N * K + M * N * (2 if res is not None else 1))
    if name == "linear_swiglu":
        x, w = a[0], a[1]
        M, (N, K) = rows(x), w.shape
        return f"linear_swiglu[{M}x2x{N}x{K}]", 4 * M * N * K, bf * (M * K + 2 * N * K + M * N)
    if name in ("linear_multi", "qkv_heads"):
        x, ws = a[0], a[1]
        M, (N, K), S = rows(x), ws[0].shape, len(ws)
        return f"{name}[{M}x{S}x{N}x{K}]", 2 * M * N * K * S, bf * (M * K + S * N * K + S * M * N)
    if name in ("grouped_gemm", "grouped_gemm_nt"):
        x, w = a[0], a[1]
        R, K = x.shape
        E = w.shape[0]
        Nb = w.shape[2] if name == "grouped_gemm" else w.shape[1]
        sw = bool(k.get("swiglu", a[3] if len(a) > 3 and name == "grouped_gemm" else False))
        No = Nb // 2 if sw else Nb
        return (f"{name}{'_swiglu' if sw else ''}[{R}rows,E{E},{K}->{Nb}]", 2 * R * K * Nb, bf * (E * K * Nb + R * K + R * No))
    if name == "grouped_gemm_regions":   # expert parallelism: rows_hint rows spread over fixed-capacity regions, THIS rank's experts
        x, w, rh = a[0], a[1], a[4]
        K, E, Nb = x.shape[1], w.shape[0], w.shape[2]
        sw = bool(k.get("swiglu", False))
        No = Nb // 2 if sw else Nb
        return (f"grouped_gemm_regions{'_swiglu' if sw else ''}[~{rh}rows,E{E}local,{K}->{Nb}]", 2 * rh * K * Nb,
                bf * (E * K * Nb + rh * K + rh * No))
    if name == "grouped_wgrad":
        x, y = a[0], a[1]
        R, Md, Nd = x.shape[0], x.shape[1], y.shape[1]
        G = (a[2].numel() - 1) // k.get("num_sources", 1)
        return f"grouped_wgrad[{R}rows,G{G},{Md}x{Nd}]", 2 * R * Md * Nd, bf * (R * Md + R * Nd + G * Md * Nd)
    if name == "attention":
        q, Tq, Tk, causal = a[0], a[3], a[4], a[6] if len(a) > 6 else k.get("causal")
        hd = k.get("out_hd", a[7] if len(a) > 7 else 128)
        B, H = q.shape[0], q.shape[1]
        pairs = Tq * Tk - (Tq * (Tq - 1) // 2 if causal else 0)
        return (f"attention[{'causal' if causal else 'full'},B{B}xH{H},Tq{Tq},Tk{Tk},hd{hd}]", 4 * B * H * pairs * hd,
                bf * B * H * hd * (2 * Tq + 2 * Tk))
    if name == "attention_decode":
        q, Tk = a[0], a[3]
        B, H = q.shape[0], q.shape[1]
        return f"attention_decode[B{B}xH{H},Tk{Tk}]", 4 * B * H * Tk * 128, bf * B * H * 128 * (2 * Tk + 2)
    if name in ("rmsnorm", "layernorm"):
        x = a[0]
        res = name == "rmsnorm" and (k.get("residual", a[3] if len(a) > 3 else None) is not None)
        return f"{name}[{rows(x)}x{x.shape[-1]}{'+res' if res else ''}]", 0, bf * x.numel() * (4 if res else 2)
    if name == "router_topk":
        x, w = a[0], a[1]
        return f"router_topk[{x.shape[0]}x{w.shape[0]}x{w.shape[1]}]", 2 * x.shape[0] * w.numel(), bf * (x.numel() + w.numel())
    if name == "permute_rows":
        return f"permute_rows[{a[1].numel()}x{a[0].shape[1]}]", 0, bf * 2 * a[1].numel() * a[0].shape[1]
    if name == "unpermute_combine":
        y, sc = a[0], a[2]
        T, kk = sc.shape
        sh = k.get("shared", a[3] if len(a) > 3 else None)
        return f"unpermute_combine[{T}x{kk}x{y.shape[1]}]", 0, bf * T * y.shape[1] * (kk + 1 + (1 if sh is not None else 0))
    if name == "build_permutation":
        return f"build_permutation[{a[0].numel()}]", 0, 4 * 3 * a[0].numel()
    if name in ("embedding", "add_pos_embedding", "im2col_patches", "merge_image_features", "swiglu_fwd", "swiglu_bwd"):
        t = a[2] if name == "merge_image_features" else a[0]
        return f"{name}", 0, bf * 2 * t.numel()
    return name, 0, 0


class KernelTable:
    """CUDA events around every `aria_b200.ops` call (the C-ABI entries) of the eager steps run while `on`."""

    def __init__(self, torch, ops):
        self.torch, self.ops = torch, ops
        self.names = [n for n in dir(ops) if callable(getattr(ops, n)) and not n.startswith("_")
                      and getattr(getattr(ops, n), "__module__", "") == ops.__name__]
        self.orig = {n: getattr(ops, n) for n in self.names}
        self.events = []
        self.depth = 0

    def _wrap(self, n, f):
        def w(*a, **k):
            if self.depth:
                return f(*a, **k)
            self.depth += 1
            e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
            try:
                label, fl, by = op_work(n, a, k)
            except Exception:
                label, fl, by = n, 0, 0
            e0.record()
            try:
                r = f(*a, **k)
            finally:
                e1.record()
                self.depth -= 1
            self.events.append((label, fl, by, e0, e1))
            return r
        return w

    def __enter__(self):
        for n in self.names:
            setattr(self.ops, n, self._wrap(n, self.orig[n]))
        # events time what runs between them ON ONE STREAM: the shared-expert branch, which the product runs on a side stream
        # in parallel with the routed experts (moe_lm.shared_expert_overlapped), is run in line during this pass - otherwise
        # its two GEMMs would be charged with the expert GEMMs they overlap (seen in profiles/r02_bench_a.json: a 13 GFLOP
        # GEMM "taking" 219 us)
        self._side = os.environ.get("ARIA_MOE_SIDE_STREAM")
        os.environ["ARIA_MOE_SIDE_STREAM"] = "0"
        # ... and the MoE block runs kernel by kernel (one ops call each) instead of through aria_moe_block_fwd
        self._blk = os.environ.get("ARIA_MOE_BLOCK")
        os.environ["ARIA_MOE_BLOCK"] = "0"
        return self

    def __exit__(self, *exc):
        for n in self.names:
            setattr(self.ops, n, self.orig[n])
        if self._side is None:
            os.environ.pop("ARIA_MOE_SIDE_STREAM", None)
        else:
            os.environ["ARIA_MOE_SIDE_STREAM"] = self._side
        if self._blk is None:
            os.environ.pop("ARIA_MOE_BLOCK", None)
        else:
            os.environ["ARIA_MOE_BLOCK"] = self._blk

    def table(self, steps, step_ms, peaks, sustained=True, top=14):
        pk_tf = peaks["bf16_tflops_sustained" if sustained and "bf16_tflops_sustained" in peaks else "bf16_tflops"]
        pk_bw = peaks["hbm_gbs"]
        agg = collections.OrderedDict()
        for label, fl, by, e0, e1 in self.events:
            c = agg.setdefault(label, [0, 0.0, fl, by])
            c[0] += 1
            c[1] += e0.elapsed_time(e1)
        rows = []
        for label, (n, ms, fl, by) in agg.items():
            avg_ms = ms / n
            t_tensor, t_hbm = fl / (pk_tf * 1e12) * 1e3, by / (pk_bw * 1e9) * 1e3     # ms at the measured peaks
            bound = "tensor" if t_tensor >= t_hbm else "hbm"
            achieved = (fl / avg_ms / 1e9) if bound == "tensor" else (by / avg_ms / 1e6)   # TFLOP/s | GB/s
            peak = pk_tf if bound == "tensor" else pk_bw
            rows.append({"kernel": label, "launches_per_step": n / steps, "ms_per_step": ms / steps, "avg_launch_us": avg_ms * 1e3,
                         "share": ms / steps / step_ms, "bound": bound, "flops_per_launch": fl, "bytes_per_launch": by,
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                         "frac": achieved / peak if peak else None})
        rows.sort(key=lambda r: -r["ms_per_step"])
        other = rows[top:]
        out = rows[:top]
        if other:
            out.append({"kernel": f"other ({len(other)} kernels)", "launches_per_step": sum(r["launches_per_step"] for r in other),
                        "ms_per_step": sum(r["ms_per_step"] for r in other), "share": sum(r["share"] for r in other)})
        return out


def _traffic_for(label):
    """DRAM bytes per launch of that kernel from a committed `ncu --set full` capture (profiles/kernel_traffic.json:
    {label prefix: {"dram_bytes_read": .., "dram_bytes_write": .., "source": ..}}), else None."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
    except Exception:
        return None
    for prefix, v in tab.items():
        if label.startswith(prefix):
            return v["dram_bytes_read"] + v["dram_bytes_write"]
    return None


# ------------------------------------------------------------------------------------------------ CPU reference leg
def _host_cores():
    try:
        import psutil
        return psutil.cpu_count(logical=False) or os.cpu_count()
    except Exception:
        return os.cpu_count()


class CpuReferenceCfg2:
    """The UNMODIFIED reference (`aria/model/*.py` through oracle/ref_loader.py: /root/reference or the byte-for-byte staging in
    oracle/_ref) on the host CPU, bf16, all physical cores.  Bounded sample of cfg 2: the reference's own
    `AriaForConditionalGeneration.forward()` on the full-size inputs (980 px image, T=768) of a FULL-WIDTH model with ONE ViT
    layer and ONE MoE decoder layer; wall-clock hooks on those two layer modules give the per-layer cost, and the 27-/28-layer
    figure is that forward + 26 x vit_layer + 27 x lm_layer (identical layers, identical shapes) — stated as extrapolated.
    Falls back to the oracle port (kind "port") when the reference files are not staged."""

    def __init__(self, threads=None):
        import torch
        from oracle import configs as C
        from oracle import ref_loader

        self.threads = threads or _host_cores()
        torch.set_num_threads(self.threads)
        self.cfg = C.with_layers(C.ARIA_25B, lm_layers=1, vit_layers=1)
        gen = torch.Generator().manual_seed(0)
        sd = {}
        sd.update(C.vit_state(self.cfg["vision_config"], gen))
        sd.update(C.projector_state(self.cfg["projector"], gen))
        sd.update(C.lm_state(self.cfg["text_config"], gen))
        self.pv = torch.randn(1, 3, 980, 980, generator=gen).bfloat16()
        text = torch.randint(10, self.cfg["text_config"]["vocab_size"], (T_TEXT,), generator=gen)
        self.ids = torch.cat([text[:16], torch.full((T_IMG,), self.cfg["image_token_index"]), text[16:]])[None]
        self.kind = "reference" if ref_loader.reference_available() else "port"
        self.layer_t = {}
        if self.kind == "reference":
            from oracle.make_golden import build_reference_model
            ref = ref_loader.load_reference()
            self.model = build_reference_model(ref, self.cfg, sd, torch.bfloat16)
            self.where = ref_loader.REF_ROOT
            vit_layer = self.model.vision_tower.vision_model.encoder.layers[0]
            lm_layer = self.model.language_model.model.layers[0]
            for tag, mod in (("vit", vit_layer), ("lm", lm_layer)):
                mod.register_forward_pre_hook(lambda m, a, tag=tag: self.layer_t.__setitem__(tag + "_t0", time.perf_counter()))
                mod.register_forward_hook(lambda m, a, o, tag=tag: self.layer_t.__setitem__(tag, time.perf_counter() - self.layer_t[tag + "_t0"]))
        else:
            self.sd = {k: v.bfloat16() for k, v in sd.items()}

    def sample(self):
        import torch
        with torch.no_grad():
            t0 = time.perf_counter()
            if self.kind == "reference":
                # (transformers 5.5 renamed the LM's `num_logits_to_keep`; the reference's keyword is swallowed there, so its
                # lm_head runs over all 768 positions: +0.4 of 12.7 TFLOP, left as is — the reference is not edited)
                self.model(input_ids=self.ids, pixel_values=self.pv, pixel_mask=torch.ones(1, 980, 980, dtype=torch.bool),
                           num_logits_to_keep=1)
                vit_layer, lm_layer = self.layer_t["vit"], self.layer_t["lm"]
            else:
                from oracle import aria_oracle as O
                tv = time.perf_counter()
                x = O.vit_embeddings(self.pv, torch.ones(1, 70, 70, dtype=torch.bool), self.sd, self.cfg["vision_config"],
                                     "vision_tower.vision_model.")
                t1 = time.perf_counter()
                O.vit_encoder_layer(x, self.sd, "vision_tower.vision_model.encoder.layers.0.", self.cfg["vision_config"], None)
                vit_layer = time.perf_counter() - t1
                t1 = time.perf_counter()
                O.aria_forward(self.ids, self.pv, None, self.sd, self.cfg, num_logits_to_keep=1)
                lm_layer = max(1e-9, (time.perf_counter() - t1) - (t1 - tv) - vit_layer)   # whole forward minus the ViT part
            fwd = time.perf_counter() - t0
        total = fwd + 26 * vit_layer + 27 * lm_layer
        what = ("unmodified reference classes (" + self.where + ")") if self.kind == "reference" else "oracle port (oracle/aria_oracle.py)"
        return {"value": T_TOTAL / total, "unit": "tokens/s", "cores": self.threads, "kind": self.kind, "extrapolated": True,
                "sample_wall_s": fwd,
                "sample": (f"{what}, bf16, host CPU: one real AriaForConditionalGeneration.forward() on the cfg-2 inputs (980px image, "
                           f"T=768, num_logits_to_keep=1) of a FULL-WIDTH model with 1 ViT layer + 1 MoE decoder layer = {fwd:.2f}s, of "
                           f"which vit_layer={vit_layer:.3f}s lm_layer={lm_layer:.3f}s (hooks); 27/28-layer time EXTRAPOLATED = forward + "
                           f"26 x vit_layer + 27 x lm_layer = {total:.1f}s")}


class CpuReferenceCfg5:
    """cfg 5 unit on the host: the reference `MoELayer` (full width, all 64 experts on one host) forward + backward through
    torch autograd on a bounded sample of 1024 tokens (the unit is linear in tokens; the GPU arm runs 8192 per rank)."""

    TOK = 1024

    def __init__(self, threads=None):
        import torch
        from oracle import configs as C
        from oracle import ref_loader
        self.threads = threads or _host_cores()
        torch.set_num_threads(self.threads)
        tc = C.ARIA_25B["text_config"]
        gen = torch.Generator().manual_seed(0)
        sd = {k: v.bfloat16() for k, v in C.moe_layer_state(tc, gen).items()}
        self.x = torch.randn(1, self.TOK, tc["hidden_size"], generator=gen).bfloat16().requires_grad_(True)
        self.go = torch.randn(1, self.TOK, tc["hidden_size"], generator=gen).bfloat16()
        self.kind = "reference" if ref_loader.reference_available() else "port"
        self.k = tc["moe_topk"]
        if self.kind == "reference":
            ref = ref_loader.load_reference()
            cfg = ref.moe_lm.AriaMoELMConfig(hidden_size=tc["hidden_size"], num_attention_heads=tc["num_attention_heads"],
                                             moe_num_experts=tc["moe_num_experts"], moe_topk=tc["moe_topk"],
                                             moe_intermediate_size=tc["moe_intermediate_size"], moe_num_shared_experts=2,
                                             intermediate_size=tc["moe_intermediate_size"])
            self.layer = ref.moe_lm.MoELayer(cfg).to(torch.bfloat16).eval()     # eval-mode routing, as the GPU arm
            self.layer.load_state_dict(sd, strict=True)
            self.params = list(self.layer.parameters())
        else:
            self.sd = {k: v.requires_grad_(True) for k, v in sd.items()}
            self.params = list(self.sd.values())

    def sample(self):
        import torch
        for p in self.params + [self.x]:
            p.grad = None
        t0 = time.perf_counter()
        with torch.enable_grad():
            if self.kind == "reference":
                y = self.layer(self.x)
            else:
                from oracle import aria_oracle as O
                y = O.moe_layer(self.x, self.sd, self.k)
            y.backward(self.go)
        dt = time.perf_counter() - t0
        return {"value": self.TOK / dt, "unit": "tokens/s", "cores": self.threads, "kind": self.kind, "extrapolated": False,
                "sample_wall_s": dt,
                "sample": f"reference MoELayer fwd+bwd (torch autograd, bf16, host CPU) on {self.TOK} tokens = {dt:.2f}s"}


def make_cpu_reference(workload):
    if workload == "cfg5":
        return CpuReferenceCfg5()
    if workload == "cfg2":
        return CpuReferenceCfg2()
    return None


def run_reference(args, rank):
    if rank != 0:
        return
    ref = make_cpu_reference(args.workload)
    if ref is None:
        print(json.dumps({"impl": "reference", "metric": METRICS[args.workload],
                          "unavailable": f"no bounded CPU sample defined for {args.workload} (cfg2 and cfg5 have one)"}), flush=True)
        return
    for _ in range(min(args.warmup, 1)):          # one warm-up sample is enough on the CPU (page-in, oneDNN primitive cache)
        ref.sample()
    vals = [ref.sample() for _ in range(args.steps)]
    v = statistics.median([x["value"] for x in vals])
    last = vals[-1]
    toks = T_TOTAL if args.workload == "cfg2" else CpuReferenceCfg5.TOK
    line = {"metric": METRICS[args.workload], "value": v, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": min(args.warmup, 1), "ms_per_step": 1000.0 * toks / v, "sample_wall_ms_per_step": 1000.0 * last["sample_wall_s"],
            "extrapolated": last["extrapolated"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOADS[args.workload], "global_batch": 1, "seq_len": toks, "parallelism": "host CPU"},
            "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU workloads
class Cfg2Prefill:
    """One image + 512 text tokens per rank; CUDA-graph replay of the public forward()."""

    tokens_per_step = T_TOTAL

    def __init__(self, torch, dev, rank, world, multi):
        from aria_b200 import configs as C
        from aria_b200.modeling_aria import AriaConfig, AriaForConditionalGeneration, GraphedPrefill, init_random_
        self.torch, self.world, self.multi = torch, world, multi
        cfg = C.ARIA_25B
        self.model = model = AriaForConditionalGeneration(AriaConfig.from_dict(cfg), device=dev)
        init_random_(model, seed=0)
        self.n_params = sum(p.numel() for p in model.parameters())
        self.ep = None
        if multi == "ep":
            self.ep = model.enable_expert_parallel(T_TOTAL)
        g = torch.Generator().manual_seed(1234 + rank)
        self.pv_host = torch.randn(1, 3, 980, 980, generator=g).bfloat16().pin_memory()
        text = torch.randint(10, cfg["text_config"]["vocab_size"], (T_TEXT,), generator=g)
        self.ids_host = torch.cat([text[:16], torch.full((T_IMG,), cfg["image_token_index"]), text[16:]])[None].contiguous().pin_memory()
        self.logits_host = torch.empty(1, 1, cfg["text_config"]["vocab_size"], dtype=torch.bfloat16).pin_memory()
        self.pv_dev, self.ids_dev = self.pv_host.to(dev), self.ids_host.to(dev)
        self.graphed = GraphedPrefill(model, self.ids_host, self.pv_host, num_logits_to_keep=1)
        self.h2d = self.pv_host.numel() * 2 + self.ids_host.numel() * 8
        self.d2h = self.logits_host.numel() * 2
        self.launch_mode = "CUDA graph replay of the eager forward (same kernels)"
        self.l2 = "per-step working set = 50.6 GB of weights >> 126 MB L2, no flush needed"

    def step_eager(self):
        return self.model(self.ids_dev, self.pv_dev, None, num_logits_to_keep=1, input_ids_host=self.ids_host).logits

    def step_resident(self):
        return self.graphed.replay()

    def step_e2e(self):
        out = self.graphed(self.ids_host, self.pv_host)        # H2D of ids + pixels from pinned host memory, then replay
        self.logits_host.copy_(out, non_blocking=False)        # D2H read of the step's result (synchronises)
        return self.logits_host

    def outputs(self, out):
        return {"logits": out}

    def parallelism(self):
        if self.world == 1:
            return "single GPU"
        if self.multi == "ep":
            return (f"dp{self.world} x ep{self.world}: every rank prefills its own request; routed experts sharded over the ranks, "
                    f"token rows exchanged over NVLink peer memory by our kernels (per MoE layer: dispatch + combine)")
        return f"replicas x{self.world} (no data-path collective)"

    def extra(self):
        if self.ep is None:
            return {}
        tc = self.model.config.text_config
        # rows leaving a rank per direction per layer: k*T*(W-1)/W of 5120 B each (SURVEY §8e), twice (dispatch + combine)
        per_dir = T_TOTAL * tc.moe_topk * (self.world - 1) / self.world * tc.hidden_size * 2
        return {"nvlink": {"bytes_per_rank_per_layer_per_direction": per_dir, "exchanges_per_layer": 2,
                           "bytes_per_rank_per_step": 2 * per_dir * tc.num_hidden_layers,
                           "peak_gbs_per_direction": 770.0, "peak_source": "measured peer copy (B200_PROFILING.md)"}}


class Cfg3Decode:
    tokens_per_step = 32

    def __init__(self, torch, dev, rank, world, multi):
        from aria_b200 import configs as C
        from aria_b200.modeling_aria import AriaConfig, AriaForConditionalGeneration, init_random_
        self.torch = torch
        B, self.Tkv = 32, 2048
        cfg = C.with_layers(C.ARIA_25B, None, 1)
        self.model = AriaForConditionalGeneration(AriaConfig.from_dict(cfg), device=dev)
        init_random_(self.model, 0)
        self.n_params = sum(p.numel() for p in self.model.parameters())
        self.cache = self.model.language_model.new_cache(B, self.Tkv + 8, dev)
        gkv = torch.Generator(device=dev).manual_seed(78 + rank)
        for t in self.cache.k + self.cache.v:
            t.normal_(generator=gkv)
        g = torch.Generator().manual_seed(77 + rank)
        self.ids_host = torch.randint(10, 100352, (B, 1), generator=g).pin_memory()
        self.ids = self.ids_host.to(dev)
        self.logits_host = torch.empty(B, 1, 100352, dtype=torch.bfloat16).pin_memory()
        self.step_eager()
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            self.step_eager()
        torch.cuda.current_stream(dev).wait_stream(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = self.step_eager()
        self.h2d, self.d2h = self.ids_host.numel() * 8, self.logits_host.numel() * 2
        self.launch_mode = "CUDA graph replay of the eager decode step"
        self.l2 = "per-step working set = ~66 GB (weights of the experts hit + 18.8 GB KV) >> 126 MB L2"
        self.world, self.multi = world, multi

    def step_eager(self):
        self.cache.seq_len = self.Tkv - 1     # the new token lands at position Tkv-1 -> attention over Tkv keys
        return self.model(self.ids, past_key_values=self.cache, num_logits_to_keep=1).logits

    def step_resident(self):
        self.graph.replay()
        return self.out

    def step_e2e(self):
        self.ids.copy_(self.ids_host, non_blocking=True)
        self.graph.replay()
        self.logits_host.copy_(self.out)
        return self.logits_host

    def outputs(self, out):
        return {"logits": out}

    def parallelism(self):
        return "single GPU" if self.world == 1 else f"replicas x{self.world} (no data-path collective)"

    def extra(self):
        return {}


class Cfg4LongPrefill:
    tokens_per_step = 65536

    def __init__(self, torch, dev, rank, world, multi):
        from aria_b200 import configs as C
        from aria_b200.modeling_aria import AriaConfig, AriaForConditionalGeneration, init_random_
        self.torch = torch
        T, frames = self.tokens_per_step, 32
        cfg = C.ARIA_25B
        self.model = AriaForConditionalGeneration(AriaConfig.from_dict(cfg), device=dev)
        init_random_(self.model, 0)
        self.n_params = sum(p.numel() for p in self.model.parameters())
        g = torch.Generator().manual_seed(99 + rank)
        ids = torch.randint(10, 100352, (1, T), generator=g)
        ids[0, 64:64 + 256 * frames] = cfg["image_token_index"]
        self.ids_host = ids.pin_memory()
        self.pv_host = torch.randn(frames, 3, 980, 980, generator=g).bfloat16().pin_memory()
        self.ids, self.pv = self.ids_host.to(dev), self.pv_host.to(dev)
        self.logits_host = torch.empty(1, 1, 100352, dtype=torch.bfloat16).pin_memory()
        self.h2d, self.d2h = self.pv_host.numel() * 2 + self.ids_host.numel() * 8, self.logits_host.numel() * 2
        self.launch_mode = "eager launches (a 64K prefill is ~1.5 s of GPU work; launch overhead is negligible)"
        self.l2 = "working set (50.6 GB weights, 18.8 GB KV, activations) >> 126 MB L2"
        self.world, self.multi = world, multi

    def step_eager(self):
        return self.model(self.ids, self.pv, None, num_logits_to_keep=1, input_ids_host=self.ids_host).logits

    step_resident = step_eager

    def step_e2e(self):
        out = self.model(self.ids_host, self.pv_host, None, num_logits_to_keep=1).logits
        self.logits_host.copy_(out)
        return self.logits_host

    def outputs(self, out):
        return {"logits": out}

    def parallelism(self):
        return "single GPU" if self.world == 1 else f"replicas x{self.world} (no data-path collective)"

    def extra(self):
        return {}


class Cfg5EpTrain:
    tokens_per_step = 8192

    def __init__(self, torch, dev, rank, world, multi):
        import torch.distributed as dist
        from aria_b200.expert_parallel import ep_moe_layer_train
        self.torch, self.world, self.fn = torch, world, ep_moe_layer_train
        if not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29544")
            dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
        d, E, self.k, I, T = 2560, 64, 6, 1664, self.tokens_per_step
        g = torch.Generator(device=dev).manual_seed(7)

        def rnd(*s):
            return (torch.randn(*s, generator=g, device=dev) * 0.02).bfloat16().requires_grad_(True)

        self.w = {"router.weight": rnd(E, d), "experts.fc1.weight": rnd(E // world, d, 2 * I),
                  "experts.fc2.weight": rnd(E // world, I, d), "shared_experts.gate_proj.weight": rnd(2 * I, d),
                  "shared_experts.up_proj.weight": rnd(2 * I, d), "shared_experts.down_proj.weight": rnd(d, 2 * I)}
        self.n_params = sum(p.numel() for p in self.w.values())
        gx = torch.Generator().manual_seed(100 + rank)
        self.x_host = torch.randn(T, d, generator=gx).bfloat16().pin_memory()
        self.go_host = torch.randn(T, d, generator=gx).bfloat16().pin_memory()
        self.x = self.x_host.to(dev).requires_grad_(True)
        self.go = self.go_host.to(dev)
        self.dx_host = torch.empty(T, d, dtype=torch.bfloat16).pin_memory()
        self.h2d, self.d2h = 2 * self.x_host.numel() * 2, self.dx_host.numel() * 2
        self.launch_mode = "eager launches through torch.autograd.Function (explicit backward over our kernels)"
        self.l2 = "per-step working set = 1.7 GB of weights + 0.6 GB of activations >> 126 MB L2"

    def step_eager(self):
        torch = self.torch
        with torch.enable_grad():
            for p in list(self.w.values()) + [self.x]:
                p.grad = None
            self.fn(self.x, self.w, self.k).backward(self.go)
        return self.x.grad

    step_resident = step_eager

    def step_e2e(self):
        with self.torch.no_grad():
            self.x.copy_(self.x_host, non_blocking=True)
            self.go.copy_(self.go_host, non_blocking=True)
        self.dx_host.copy_(self.step_eager())
        return self.dx_host

    def outputs(self, out):
        return {"dx": out, **{"d_" + n.replace(".", "_"): p.grad for n, p in self.w.items()}}

    def parallelism(self):
        return (f"ep{self.world}: tokens data-parallel (8192 per rank), routed experts sharded, token all-to-all each way in forward and "
                f"backward") if self.world > 1 else "single GPU (all 64 experts local)"

    def extra(self):
        if self.world == 1:
            return {}
        per_dir = 8192 * 6 * (self.world - 1) / self.world * 2560 * 2
        return {"nvlink": {"bytes_per_rank_per_layer_per_direction": per_dir, "exchanges_per_layer": 4,
                           "peak_gbs_per_direction": 770.0, "peak_source": "measured peer copy (B200_PROFILING.md)"}}


GPU_WORKLOADS = {"cfg2": Cfg2Prefill, "cfg3": Cfg3Decode, "cfg4": Cfg4LongPrefill, "cfg5": Cfg5EpTrain}


def dump_outputs(outs, out_dir):
    """float32 copies of the tensors in `outs` as out_dir/<name>.npy, within DUMP_BUDGET bytes in all: a tensor of more than
    its share of the budget is written as a seeded sample of its elements (flattened; the same positions in every run)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = (DUMP_BUDGET // len(outs) - 1024) // 4       # 1 KB per file for the .npy header
    for name, t in outs.items():
        t = t.detach()
        if t.numel() > cap:
            idx = torch.randint(t.numel(), (cap,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_aria(args, rank, local_rank, world):
    import torch

    from aria_b200 import _lib as L
    from aria_b200 import ops

    L.load()  # fail loudly if the CUDA extension is missing
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    torch.set_grad_enabled(False)
    # N > 1: experts sharded over the ranks by default (the real exchange step of the path, SURVEY §8e)
    multi = "single" if world == 1 else (args.multi or os.environ.get("ARIA_BENCH_MULTI") or ("ep" if args.workload in ("cfg2", "cfg5") else "replicas"))
    wl = GPU_WORKLOADS[args.workload](torch, dev, rank, world, multi)
    steps, warmup = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        """(ms per call, what the last call returned) over n calls"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / n, out

    for _ in range(warmup):
        wl.step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = L.launch_count
    wl.step_eager()       # kernels per step (counted on one eager step; the graph replays exactly these launches)
    launches_per_step = L.launch_count - l0
    ms, out = timed(wl.step_resident, steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(wl.outputs(out), args.dump_outputs)

    # per-kernel table: CUDA events around every C-ABI call of K eager steps (events cannot be recorded inside a graph replay)
    kernels, ms_eager = None, None
    if not args.no_kernel_table:
        with KernelTable(torch, ops) as kt:
            ms_eager, _ = timed(wl.step_eager, steps)
        peaks, peak_src = _peaks()
        kernels = kt.table(steps, ms_eager, peaks)

    for _ in range(2):
        wl.step_e2e()
    ms_e2e, _ = timed(wl.step_e2e, steps)
    clocks = sampler.stop()

    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        return
    peaks, peak_src = _peaks()
    tok = wl.tokens_per_step
    line = {"metric": METRICS[args.workload], "value": world * tok / (ms * 1e-3), "unit": "tokens/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload], "global_batch": world, "seq_len": tok,
                       "parallelism": wl.parallelism(), "params": wl.n_params, "l2": wl.l2},
            "e2e": {"value": world * tok / (ms_e2e * 1e-3), "unit": "tokens/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": wl.h2d, "d2h_bytes_per_step": wl.d2h},
            "gpu_launches": launches_per_step * steps, "launches_per_step": launches_per_step, "launch_mode": wl.launch_mode,
            "clocks": clocks, "impl": "aria_b200"}
    line.update(wl.extra())
    if "nvlink" in line and world > 1:
        nv = line["nvlink"]
        if "bytes_per_rank_per_step" in nv:
            nv["achieved_gbs_per_direction_if_serial"] = nv["bytes_per_rank_per_step"] / 2 / (ms * 1e-3) / 1e9
    if kernels:
        dom = kernels[0]
        line["kernels"] = kernels
        line["eager_ms_per_step"] = ms_eager
        line["roofline"] = {"bound": dom["bound"], "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": dom["peak"],
                            "unit": dom["unit"], "frac": dom["frac"], "traffic": _traffic_for(dom["kernel"]),
                            "peak_source": peak_src + ("; bf16 = sustained figure (kernel timed inside a long step)" if dom["bound"] == "tensor" else ""),
                            "flops_per_launch": dom["flops_per_launch"], "bytes_per_launch": dom["bytes_per_launch"],
                            "avg_launch_ms": dom["avg_launch_us"] / 1e3, "launches_timed": int(round(dom["launches_per_step"] * steps)),
                            "share_of_step": dom["share"], "selected_by": "largest share of the eager step (per-kernel table in `kernels`)"}
    if world == 1 and not args.no_cpu_baseline:
        try:
            ref = make_cpu_reference(args.workload)
            if ref is not None:
                ref.sample()  # warm-up
                s = ref.sample()
                line["cpu_baseline"] = {k: s[k] for k in ("value", "unit", "cores", "kind", "sample", "extrapolated")}
        except Exception as ex:  # the GPU measurement stands on its own; say why the CPU leg is missing
            line["cpu_baseline"] = {"value": None, "error": f"{type(ex).__name__}: {ex}"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="aria", choices=["aria", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--multi", default=None, choices=["ep", "replicas"],
                    help="N > 1: shard the routed experts over the ranks (default for cfg2/cfg5) or run independent replicas")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-table", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "aria":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl aria)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_aria(args, rank, local_rank, world)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
