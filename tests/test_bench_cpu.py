"""Host logic of bench.py (no GPU, no heavy compute): algorithmic FLOP table vs the conv / GEMM / attention inventory of
the native UNet, synthetic-input invariants (SURVEY.md section 8d), the CPU-sample picker, the per-family roofline
arithmetic, and the schema of the `--impl reference` JSON line with the oracle's compute stubbed out."""
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_flop_table_matches_survey_and_scales_with_area():
    t = bench.TFLOP_PER_PAIR
    assert t[128] == pytest.approx(13.524) and t[96] == pytest.approx(7.284) and t[64] == pytest.approx(3.179)   # SURVEY 8d
    # convolutions and projections scale with the area, self-attention with its square: the per-area cost must rise
    assert t[64] / 64 ** 2 < t[96] / 96 ** 2 < t[128] / 128 ** 2
    assert t[32] == pytest.approx(t[128] / 16) and t[48] == pytest.approx(t[128] * (48 / 128) ** 2)   # CPU-sample estimates


def test_synth_inputs_are_rank_and_slot_invariant():
    """One CPU generator per image (utils.py:86-87 semantics): candidate i is the same noise wherever it is generated."""
    from imagharmony_b200.config import SDXL_BASE as cfg
    a = bench.synth_inputs(cfg, 2, 8, 20, rank=0)
    b = bench.synth_inputs(cfg, 1, 8, 20, rank=1)            # rank 1 with n = 1 draws seed 1001 = rank 0's second image
    assert a[0].shape == (2, 4, 8, 8) and a[0].dtype == torch.float16
    assert torch.equal(a[0][1:], b[0])
    assert a[1].shape == (2, 77 + cfg.num_ip_tokens, cfg.cross_attention_dim) and a[3].shape == (2, cfg.pooled_embed_dim)
    assert a[5].tolist() == [[64.0, 64.0, 0.0, 0.0, 64.0, 64.0]] * 2
    from imagharmony_b200.scheduler import EulerDiscreteScheduler
    ins = EulerDiscreteScheduler().set_timesteps(20).init_noise_sigma
    raw = torch.randn((1, 4, 8, 8), generator=torch.Generator("cpu").manual_seed(1000))
    assert torch.equal(a[0][:1], (raw * ins).half())


def test_workload_string_names_the_configuration():
    s = bench.workload_string(1024, 50, 4)
    assert "1024x1024" in s and "50-step" in s and "4 image(s)/GPU (UNet batch 8)" in s


class _FakeOracle:
    threads = 3

    def __init__(self, seconds_256):
        self.t = seconds_256
        self.calls = []

    def forward_seconds(self, lat):
        self.calls.append(lat)
        return self.t

    def timed_steps(self, lat, steps, warm):
        return 2.0 * steps


def test_pick_cpu_sample_respects_the_budget():
    # one 256^2 forward takes 1 s -> 512^2 ~ 3.76 s, 384^2 ~ 2.25 s per step
    lat, est = bench.pick_cpu_sample(_FakeOracle(1.0), steps=20, warm=5, budget_s=170)
    assert lat == 64 and est == pytest.approx(bench.TFLOP_PER_PAIR[64] / bench.TFLOP_PER_PAIR[32])
    lat, _ = bench.pick_cpu_sample(_FakeOracle(1.0), steps=20, warm=5, budget_s=60)
    assert lat == 48
    o = _FakeOracle(10.0)
    lat, est = bench.pick_cpu_sample(o, steps=20, warm=5, budget_s=60)
    assert lat == 32 and est == pytest.approx(10.0)           # never below 256^2, even over budget
    assert o.calls == [32, 32]                                # one untimed warm-up forward, one calibration forward


def test_family_roofline_arithmetic():
    pk = {"tflops_burst": 1700.0, "tflops_sustained": 1400.0, "hbm_gbs": 6500.0, "source": "test"}
    agg = {"gemm": {"ms": 10.0, "flops": 7.0e12, "bytes": 0.0, "launch_groups": 300},
           "groupnorm": {"ms": 1.0, "flops": 0.0, "bytes": 3.25e9, "launch_groups": 46},
           "attn_self": {"ms": 4.0, "flops": 1.4e12, "bytes": 0.0, "launch_groups": 70}}
    r = bench.family_roofline(agg, pk, step_ms_graph=12.0)
    assert r["family"] == "gemm" and r["bound"] == "tensor" and r["unit"] == "TFLOP/s"      # time-dominant family first
    assert r["achieved"] == pytest.approx(700.0) and r["peak"] == 1400.0 and r["frac"] == pytest.approx(0.5)
    assert r["share_of_step"] == pytest.approx(10.0 / 15.0, abs=1e-4)
    assert r["frac_if_scaled_to_graph_time"] == pytest.approx(0.5 * 15.0 / 12.0)
    g = r["families"]["groupnorm"]
    assert g["bound"] == "hbm" and g["achieved"] == pytest.approx(3250.0) and g["frac"] == pytest.approx(0.5)
    assert list(r["families"]) == ["gemm", "attn_self", "groupnorm"]
    if os.path.exists(bench.TRAFFIC_FILE):                    # the committed ncu capture supplies roofline.traffic
        assert r["traffic"] is None or r["traffic"] > 0


def test_peaks_come_from_the_driver_file_when_present():
    pk = bench.peaks()
    assert pk["tflops_sustained"] <= pk["tflops_burst"] and pk["hbm_gbs"] > 1000
    if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
        assert pk["source"].startswith("measured")


def test_dump_outputs_writes_float32_and_samples_past_the_budget(tmp_path, monkeypatch):
    """`--dump-outputs`: DIR/<name>.npy in float32, whole when it fits; past the budget a seeded sample that is the same
    on every call."""
    import numpy as np
    x = torch.randn(2, 4, 8, 8, generator=torch.Generator("cpu").manual_seed(5)).half()
    bench.dump_outputs(str(tmp_path / "d"), {"latents": x})
    a = np.load(tmp_path / "d" / "latents.npy")
    assert a.dtype == np.float32 and a.shape == (2, 4, 8, 8) and np.array_equal(a, x.float().numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100 * 4)
    bench.dump_outputs(str(tmp_path / "s1"), {"latents": x})
    bench.dump_outputs(str(tmp_path / "s2"), {"latents": x})
    s1, s2 = np.load(tmp_path / "s1" / "latents.npy"), np.load(tmp_path / "s2" / "latents.npy")
    assert s1.dtype == np.float32 and s1.shape == (100,) and np.array_equal(s1, s2)
    assert np.isin(s1, x.float().numpy().reshape(-1)).all()


def test_reference_arm_line_schema(monkeypatch, capsys):
    """`bench.py --impl reference`: one JSON line with the contract's keys; rank != 0 prints nothing."""
    monkeypatch.setattr(bench, "CpuOracle", lambda: _FakeOracle(0.5))
    args = type("A", (), {"steps": 4, "warmup": 1, "gpus": 1, "res": 1024, "images": 1})()
    monkeypatch.setenv("RANK", "1")
    bench.run_reference_arm(args)
    assert capsys.readouterr().out == ""
    monkeypatch.setenv("RANK", "0")
    bench.run_reference_arm(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["unit"] == "denoise-steps/s"
    assert line["steps"] == 4 and line["warmup"] == 1 and line["value"] == pytest.approx(4 / 8.0)
    assert line["ms_per_step"] == pytest.approx(2000.0) and line["vs_baseline"] is None and line["higher_is_better"] is True
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 3 and cb["value"] == line["value"] and cb["sample_res"] == 512
    assert line["e2e"] == {"value": line["value"], "unit": "denoise-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]
