"""CPU: host-side pieces of bench.py that the driver's contract depends on (clock sampling / throttle-reason parsing, peak
lookup, argument defaults).  The timed paths themselves need a GPU."""
import importlib.util
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["bench_under_test"] = mod
    spec.loader.exec_module(mod)
    return mod


def test_clock_sampler_parses_nvidia_smi_rows():
    b = _bench()
    s = b.ClockSampler(0)
    s.proc = type("P", (), {"terminate": lambda self: None, "wait": lambda self, timeout=None: 0, "kill": lambda self: None})()
    s.rows = ["1965, 1965, 650.1, Not Active, Not Active, Not Active, Active",
              "1800, 1965, 900.0, Not Active, Not Active, Not Active, Active",
              "1700, 1965, 910.0, Not Active, Not Active, Not Active, Not Active",
              "garbage line",
              "[N/A], 1965, 1, Not Active, Not Active, Not Active, Not Active"]
    out = s.stop()
    assert out["sm_mhz"] == 1800 and out["sm_max_mhz"] == 1965 and out["samples"] == 3
    assert out["reasons"] == ["sw_power_cap"]
    s.rows = ["1965, 1965, 650.1, Active, Not Active, Active, Not Active"]
    assert s.stop()["reasons"] == ["hw_slowdown", "sw_thermal_slowdown"]


def test_clock_sampler_without_nvidia_smi_reports_it():
    b = _bench()
    s = b.ClockSampler(0)
    assert s.stop()["reasons"] == ["nvidia-smi unavailable"]


def test_peaks_come_from_the_driver_file_or_the_documented_fallback():
    b = _bench()
    peaks, source = b._peaks()
    assert peaks["hbm_gbs"] > 1000 and peaks["bf16_tflops"] > 500
    assert source.startswith("measured") == os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json"))


def test_workload_is_baseline_cfg2():
    b = _bench()
    assert b.T_TOTAL == 768 and "cfg2" in b.WORKLOADS["cfg2"] and b.METRICS["cfg2"] == "Aria-25.3B bf16 prefill tokens/sec"
    assert set(b.GPU_WORKLOADS) == {"cfg2", "cfg3", "cfg4", "cfg5"}


def test_op_work_models_match_survey_8d():
    """Algorithmic FLOPs / bytes the per-kernel table divides by (SURVEY.md §8d): checked on the cfg-2 shapes."""
    import torch
    b = _bench()
    meta = lambda *s, dt=torch.bfloat16: torch.empty(*s, dtype=dt, device="meta")   # noqa: E731
    # fc1 grouped GEMM + SwiGLU at 768 tokens: 6*768 rows x [64, 2560, 3328]
    lab, fl, by = b.op_work("grouped_gemm", (meta(4608, 2560), meta(64, 2560, 3328), meta(65, dt=torch.int32)), {"swiglu": True})
    assert "swiglu" in lab and fl == 2 * 4608 * 2560 * 3328
    assert by == 2 * (64 * 2560 * 3328 + 4608 * 2560 + 4608 * 1664) == 1129447424          # the number VERDICT r1 recomputed
    # ViT attention, one layer: 4 * 16 * 4900^2 * 72 FLOP
    q = meta(1, 16, 4900, 128)
    lab, fl, by = b.op_work("attention", (q, q, q, 4900, 4900, 0.1, False), {"out_hd": 72})
    assert fl == 4 * 16 * 4900 * 4900 * 72 and "hd72" in lab
    # causal LM attention: 5120 * T^2 per layer up to the diagonal term
    q = meta(1, 20, 768, 128)
    _, fl, _ = b.op_work("attention", (q, q, q, 768, 768, 0.1, True), {})
    assert abs(fl / (5120 * 768 * 768) - 1) < 2e-3
    _, fl, by = b.op_work("linear", (meta(768, 2560), meta(2560, 2560)), {})
    assert fl == 2 * 768 * 2560 * 2560 and by == 2 * (768 * 2560 * 2 + 2560 * 2560)
    # expert parallelism: the fc1 GEMM of ONE rank of 8 (8 local experts, rows of all ranks in fixed-capacity regions)
    lab, fl, by = b.op_work("grouped_gemm_regions", (meta(64 * 784, 2560), meta(8, 2560, 3328), meta(64, dt=torch.int32),
                                                     meta(64, dt=torch.int32), 4608), {"swiglu": True, "group_mod": -8})
    assert "E8local" in lab and fl == 2 * 4608 * 2560 * 3328 and by == 2 * (8 * 2560 * 3328 + 4608 * 2560 + 4608 * 1664)


def test_kernel_table_picks_the_dominant_kernel_by_share():
    b = _bench()

    class Ev:
        def __init__(self, t):
            self.t = t

        def elapsed_time(self, other):
            return other.t - self.t

    kt = b.KernelTable.__new__(b.KernelTable)
    kt.events = [("attention[x]", 110.6e9, 1e6, Ev(0.0), Ev(0.2)), ("gemm[y]", 1e6, 1.1e9, Ev(0.0), Ev(0.15)),
                 ("attention[x]", 110.6e9, 1e6, Ev(1.0), Ev(1.2))]
    rows = kt.table(1, 1.0, {"hbm_gbs": 6484.6, "bf16_tflops": 1739.4, "bf16_tflops_sustained": 1480.4})
    assert rows[0]["kernel"] == "attention[x]" and rows[0]["bound"] == "tensor" and abs(rows[0]["share"] - 0.4) < 1e-9
    assert abs(rows[0]["achieved"] - 553.0) < 1.0 and abs(rows[0]["frac"] - 553.0 / 1480.4) < 1e-3
    assert rows[1]["bound"] == "hbm" and abs(rows[1]["achieved"] - 1.1e9 / 0.15 / 1e6) < 1e-6


def test_dominant_kernels_have_committed_dram_traffic():
    """`roofline.traffic` comes from committed ncu captures (profiles/kernel_traffic.json): present for the two kernels that can be the
    largest share of the cfg-2 step, and within 1.6x of their algorithmic bytes (no wasted re-reads)."""
    b = _bench()
    t_attn = b._traffic_for("attention[full,B1xH16,Tq4900,Tk4900,hd72]")
    t_fc1 = b._traffic_for("grouped_gemm_swiglu[4608rows,E64,2560->3328]")
    assert t_attn and t_fc1 and b._traffic_for("no_such_kernel[1]") is None
    assert 45158400 <= t_attn <= 1.6 * 45158400          # q, k, v, out of 16 heads x 4900 x 72 (+ stream-K pieces)
    assert 1129447424 * 0.98 <= t_fc1 <= 1.05 * 1129447424


def test_dump_outputs_stays_within_budget_and_samples_the_same_positions(tmp_path):
    import numpy as np
    import torch
    b = _bench()
    b.DUMP_BUDGET = 1 << 16
    big = torch.randn(100000, generator=torch.Generator().manual_seed(1))
    outs = {"logits": torch.arange(6.0).reshape(2, 3).bfloat16(), "dx": big}
    for run in ("a", "b"):
        b.dump_outputs(outs, str(tmp_path / run))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= b.DUMP_BUDGET
    small = np.load(tmp_path / "a" / "logits.npy")
    assert small.dtype == np.float32 and small.shape == (2, 3) and (small == np.arange(6.0).reshape(2, 3)).all()
    sample_a, sample_b = np.load(tmp_path / "a" / "dx.npy"), np.load(tmp_path / "b" / "dx.npy")
    assert sample_a.dtype == np.float32 and 0 < sample_a.size < big.numel()
    assert (sample_a == sample_b).all() and np.isin(sample_a, big.numpy()).all()
