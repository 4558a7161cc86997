#!/usr/bin/env python
"""bench.py -- denoise-steps/s of the SDXL + IMAGHarmony hot path (BASELINE.json metric) on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--images n] [--res 1024]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: UNet forward on the CFG pair(s) + CFG combine + Euler update
(custom_pipelines.py:325-363) at 1024x1024 (latent 128x128), random-init SDXL-base weights, synthetic embeddings.
  value : whole-job denoise-steps/s with inputs resident in HBM (K CUDA-graph replays timed with CUDA events; with
          N > 1 ranks the timed region also contains the path's only collective: the PNS tail = score of each rank's
          final latents -> all_gather of the fp32 scores -> argmax -> broadcast of the winning latent)
  e2e   : same metric through the public call `DenoiseEngine.run(...)` with pinned HOST inputs and a host read of the
          final latents inside the timed region
  roofline : per kernel FAMILY (plain GEMM, GEGLU GEMM, implicit-GEMM conv, self-attention, decoupled cross-attention,
          GroupNorm, pointwise) time share and achieved rate measured live -- one denoise step with a CUDA-event pair
          around every launch, queued behind a spin kernel so the GPU runs them back to back; the headline fields are
          those of the TIME-DOMINANT family
  gpu_eager_baseline : the oracle UNet (reference processors + restated diffusers UNet) in torch-eager fp16 and
          graph-replayed on the same GPU in the same run -- the stand-in for "the reference GPU diffusers path"
  c1_512 : BASELINE config 1 shape (512^2, 1 image) on the native path, the shape the CPU arm times
  cpu_baseline : the CPU oracle (a port of the reference's PyTorch path) on the host cores, bounded sample
  pns (N > 1) : BASELINE config 4 shape -- 4 candidates per GPU, K steps each, H2D + denoise + score + all_gather +
          winner broadcast, wall clock max over ranks, against the bar 1.1 x 4 x (single-candidate time)
`--dump-outputs DIR` writes the final latents of the timed steps (what `DenoiseEngine.run` returns) to DIR/latents.npy
(DIR/latents_rank<r>.npy with N > 1 ranks) in float32: weights and inputs are seeded, so two builds run with the same
arguments can be compared output for output.
`--impl reference` times the CPU path alone (rank 0 only): every step is one REAL denoise step (UNet on the CFG pair +
CFG + Euler) of the oracle at the largest of 512^2 / 384^2 / 256^2 that keeps the K + W steps within the time budget.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "denoise-steps/s @1024^2 SDXL (UNet + CFG + Euler step, IMAGHarmony IP cross-attention)"
# algorithmic FLOPs of one UNet forward per CFG pair (SURVEY.md section 8d / BASELINE.md section 3)
TFLOP_PER_PAIR = {32: 13.524 / 16.0, 48: 13.524 * (48 / 128.0) ** 2, 64: 3.179, 96: 7.284, 128: 13.524}
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the time-dominant family's most frequent instantiation,
# from the committed `ncu --set full` capture (bench.py cannot run ncu on itself): see roofline.traffic_source
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r2_traffic.json")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_burst": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm_gbs": d["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _loop(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def synth_inputs(cfg, n: int, lat: int, T: int, rank: int):
    """SURVEY.md section 8d synthetic inputs: per-image CPU generators (rank/slot invariant), N(0,1) embeddings."""
    from imagharmony_b200.scheduler import EulerDiscreteScheduler
    ins = EulerDiscreteScheduler().set_timesteps(T).init_noise_sigma
    seeds = [1000 + rank * n + i for i in range(n)]
    lat_parts = [torch.randn((1, 4, lat, lat), generator=torch.Generator("cpu").manual_seed(s)) for s in seeds]
    latents = (torch.cat(lat_parts) * ins).half()
    g = torch.Generator("cpu").manual_seed(1234)
    L = 77 + cfg.num_ip_tokens
    pos = torch.randn(n, L, cfg.cross_attention_dim, generator=g).half()
    neg = torch.randn(n, L, cfg.cross_attention_dim, generator=g).half()
    pooled = torch.randn(n, cfg.pooled_embed_dim, generator=g).half()
    npooled = torch.randn(n, cfg.pooled_embed_dim, generator=g).half()
    res = lat * 8.0
    tid = torch.tensor([[res, res, 0.0, 0.0, res, res]] * n)
    return latents, pos, neg, pooled, npooled, tid


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict) -> None:
    """DIR/<name>.npy in float32.  An array larger than the 64 MB budget is written as a fixed, seeded sample of its
    flattened elements (the same positions on every run), so the dump stays comparable at any batch or resolution."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    keep = DUMP_LIMIT_BYTES // 4 // max(len(arrays), 1)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > keep:
            idx = torch.randperm(a.numel(), generator=torch.Generator("cpu").manual_seed(0))[:keep].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(directory, f"{name}.npy"), a.numpy())


def workload_string(res: int, steps: int, images: int) -> str:
    """The one workload both arms report (BASELINE config 2 by default)."""
    return (f"single {res}x{res} edit per GPU, {steps}-step Euler schedule, {images} image(s)/GPU (UNet batch "
            f"{2 * images}), SDXL-base UNet random-init, 77+4 tokens, guidance 5.0, IP scale 1.0")


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (a port of the reference's PyTorch path) on the host cores
# ---------------------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Physical cores this process may use.  torchrun exports OMP_NUM_THREADS=1 for N > 1 ranks: the CPU arm sets its
    thread count explicitly instead of inheriting that."""
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or (os.cpu_count() or 1)
    except Exception:
        phys = max(1, (os.cpu_count() or 2) // 2)
    try:
        phys = min(phys, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return max(1, phys)


class CpuOracle:
    """The CPU fp32 oracle UNet with a fast deterministic fill (timing only)."""

    def __init__(self):
        from imagharmony_b200.config import SDXL_BASE as cfg
        from oracle import adapter_ref as A
        from oracle.unet_ref import UNetRef
        self.cfg = cfg
        self.threads = host_threads()
        torch.set_num_threads(self.threads)
        torch.set_flush_denormal(True)
        with torch.device("meta"):
            m = UNetRef(cfg)
        m = m.to_empty(device="cpu")
        # tile one small random block instead of drawing 2.6 G numbers
        block = (torch.rand(1 << 20, generator=torch.Generator("cpu").manual_seed(0)) * 2 - 1) * 0.02

        def fill(p):
            if p.dim() == 1:
                p.fill_(0.5)
            else:
                flat = p.view(-1)
                reps = (flat.numel() + block.numel() - 1) // block.numel()
                flat.copy_(block.repeat(reps)[: flat.numel()])
        with torch.no_grad():
            for p in m.parameters():
                fill(p)
        with torch.device("meta"):
            A.install_processors(m, cfg)
        for pr in m.attn_processors.values():
            if hasattr(pr, "to_k_ip"):
                pr.to_empty(device="cpu")
                with torch.no_grad():
                    for q in pr.parameters():
                        fill(q)
        self.model = m.eval()

    def inputs(self, lat: int, T: int):
        latents, pos, neg, pooled, npooled, tid = synth_inputs(self.cfg, 1, lat, T, 0)
        return latents.float(), pos.float(), neg.float(), pooled.float(), npooled.float(), tid

    def forward_seconds(self, lat: int) -> float:
        x, pos, neg, pooled, npooled, tid = self.inputs(lat, 4)
        with torch.no_grad():
            t0 = time.time()
            self.model(torch.cat([x, x]), 500.0, torch.cat([neg, pos]), torch.cat([npooled, pooled]), torch.cat([tid, tid]))
            return time.time() - t0

    def timed_steps(self, lat: int, steps: int, warm: int):
        """`warm` + `steps` REAL denoise steps (UNet on the CFG pair + CFG + Euler, oracle/scheduler_ref.denoise_loop) of one
        image at latent size `lat`; returns the seconds of the last `steps` steps."""
        from oracle.scheduler_ref import denoise_loop
        T = steps + warm
        x, pos, neg, pooled, npooled, tid = self.inputs(lat, T)
        marks = []
        fn = lambda s, t, e, te, ti: self.model(s, t, e, te, ti)  # noqa: E731
        t_begin = time.time()
        with torch.no_grad():
            denoise_loop(fn, x, pos, neg, pooled, npooled, tid, T, guidance_scale=5.0,
                         callback=lambda i, t, lt: marks.append(time.time()))
        start = marks[warm - 1] if warm > 0 else t_begin
        return marks[-1] - start


def pick_cpu_sample(oracle: CpuOracle, steps: int, warm: int, budget_s: float):
    """Largest of 512^2 (BASELINE config 1) / 384^2 / 256^2 whose `steps + warm` denoise steps fit the budget, judged from
    one calibration forward at 256^2 scaled by the algorithmic FLOP ratio."""
    oracle.forward_seconds(32)                 # oneDNN primitive creation for the weights happens here, untimed
    t256 = oracle.forward_seconds(32)
    for lat in (64, 48, 32):
        est = t256 * TFLOP_PER_PAIR[lat] / TFLOP_PER_PAIR[32]
        if est * (steps + warm) <= budget_s or lat == 32:
            return lat, est
    return 32, t256


def cpu_sample_text(oracle: CpuOracle, lat: int, steps: int, warm: int) -> str:
    return (f"CPU oracle (port of the reference PyTorch path, fp32, {oracle.threads} threads = physical cores of "
            f"{os.cpu_count()} logical CPUs): {steps} timed + {warm} warm-up REAL denoise steps (UNet on the CFG pair + CFG + "
            f"Euler) of one image at {lat * 8}x{lat * 8} -- the value is steps/s AT THAT SIZE (BASELINE config 1 shape when "
            f"512^2), not scaled to 1024^2; algorithmic FLOP ratio to 1024^2 = {TFLOP_PER_PAIR[128] / TFLOP_PER_PAIR[lat]:.2f}x")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = max(1, args.steps), max(0, args.warmup)
    oracle = CpuOracle()
    lat, _ = pick_cpu_sample(oracle, K, W, budget_s=float(os.environ.get("IH_CPU_BUDGET_S", "170")))
    sec = oracle.timed_steps(lat, K, W)
    value = K / sec
    sample = cpu_sample_text(oracle, lat, K, W)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "denoise-steps/s", "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": sec / K * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.res, K, args.images),
                       "note": "same workload as the native arm; each CPU step is a bounded sample of it (see cpu_baseline.sample)"},
            "cpu_baseline": {"value": value, "unit": "denoise-steps/s", "cores": oracle.threads, "kind": "port",
                             "sample": sample, "sample_res": lat * 8,
                             "value_scaled_to_1024": value * TFLOP_PER_PAIR[lat] / TFLOP_PER_PAIR[128]},
            "e2e": {"value": value, "unit": "denoise-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# native arm
# ---------------------------------------------------------------------------------------------------------------
def build_native(cfg, device):
    from imagharmony_b200.unet import UNet2DConditionModel
    from imagharmony_b200.weights import random_state_dict, shapes_of
    with torch.device("meta"):
        shapes = shapes_of(UNet2DConditionModel(cfg))
    sd = random_state_dict(shapes, seed=0, device=device)          # generated on the GPU: 2.6 B parameters
    unet = UNet2DConditionModel.from_state_dict(cfg, sd, device=device)
    procs = torch.nn.ModuleList(unet.attn_processors.values())
    procs.load_state_dict(random_state_dict(shapes_of(procs), seed=1, device=device))
    unet.finalize()
    return unet


class FamilyTimer:
    """CUDA-event pair around every launch of one eager denoise step, grouped by kernel family.

    The whole step is queued behind a ~100 ms spin kernel so the GPU executes the launches back to back (no host
    launch gaps inside the event pairs).  Events between launches suppress the PDL overlap a graph replay enjoys, so
    the SUM is a little above the graph-replayed step; shares and per-family rates are what this is for."""

    FAMILIES = {
        "gemm": "plain tcgen05 GEMM: gemm_f16_kernel<BN,STAGES,0,PAIR> mode 0 (q|k|v, to_q, to_out, FF-out, proj_in/out, shortcuts)",
        "gemm_geglu": "GEGLU tcgen05 GEMM: gemm_f16_kernel<256,*,1,*> (FF GEGLU-in)",
        "conv3x3": "implicit-GEMM 3x3 conv: gemm_f16_kernel<...> mode 1 (ResBlock convs, resamplers, conv_out)",
        "attn_self": "self-attention: attn2_f16_kernel (+ attn_combine_kernel)",
        "attn_cross": "decoupled text+IP cross-attention: attnx_f16_kernel",
        "groupnorm": "GroupNorm(+SiLU): gn_stats_kernel + gn_apply_kernel",
        "pointwise": "time embeddings, layout glue, upsample, concat, CFG + Euler",
    }

    def __init__(self):
        self.records = []      # (family, flops, bytes, ev0, ev1, shape label)
        self.active = False    # True only inside DenoiseEngine._step: the once-per-call K/V projections are not a step
        self.shapes = {}       # shape label -> [calls, ms, flops]  (IH_BENCH_SHAPES=1 dumps it to gpurun_out/)

    def _wrap(self, ops, name, classify):
        orig = getattr(ops, name)

        def wrapped(*a, **k):
            if not self.active:
                return orig(*a, **k)
            fam, flops, nbytes = classify(*a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = orig(*a, **k)
            e1.record()
            label = name + ":" + "x".join(str(int(v)) for v in (list(a[0].shape) + list(a[1].shape)) if v) if name in ("linear", "conv3x3") \
                else name + ":" + "x".join(str(v) for v in a[3:7]) if name == "attention" else name
            self.records.append((fam, flops, nbytes, e0, e1, label))
            return out
        setattr(ops, name, wrapped)
        return orig

    def measure(self, eng, run_args):
        from imagharmony_b200 import ops

        def c_linear(x, w, bias=None, **k):
            M, K = x.shape
            N = w.shape[0]
            return ("gemm_geglu" if k.get("geglu") else "gemm"), 2.0 * M * N * K, 2.0 * (M * K + N * K + M * N)

        def c_conv(x, w, bias=None, **k):
            B, H, W, Cin = x.shape
            s = k.get("stride", 1)
            Cout = w.shape[0]
            px = B * (H // s) * (W // s)
            csc = w.shape[1] - 9 * Cin                  # fused 1x1 shortcut columns (ResBlock conv2)
            return "conv3x3", (18.0 * Cin + 2.0 * csc) * Cout * px, 2.0 * (B * H * W * (Cin + csc) + px * Cout + w.shape[1] * Cout)

        def c_attn(q, k_, v, B, H, Nq, Nk, **k):
            return ("attn_self" if Nk > 128 else "attn_cross"), 4.0 * B * H * Nq * Nk * 64, 2.0 * 64 * B * H * (2 * Nq + 2 * Nk)

        def c_gn(x0, gamma, beta, **k):
            n = x0.numel() + (k["x1"].numel() if k.get("x1") is not None else 0)
            return "groupnorm", 0.0, 3.0 * 2 * n      # read twice (statistics, apply) + write once

        def c_other(*a, **k):
            return "pointwise", 0.0, 0.0
        table = {"linear": c_linear, "conv3x3": c_conv, "attention": c_attn, "groupnorm": c_gn}
        for name in ("linear_small", "sinusoid", "upsample2x", "concat_channels", "im2col3x3_nchw", "nhwc_to_nchw",
                     "euler_step", "layernorm", "add_bcast"):
            table[name] = c_other
        saved = {name: self._wrap(ops, name, fn) for name, fn in table.items()}
        use_graph = eng.use_cuda_graph
        orig_step = eng._step

        def step(*a, **k):
            self.active = True
            try:
                return orig_step(*a, **k)
            finally:
                self.active = False
        eng._step = step
        try:
            eng.use_cuda_graph = False
            eng.run(*run_args, stop_after=1)            # eager warm-up (kernel attributes, descriptor cache)
            torch.cuda.synchronize()
            self.records.clear()
            torch.cuda._sleep(int(2.5e8))               # ~125 ms head start for the host to queue the whole step
            eng.run(*run_args, stop_after=1)
            torch.cuda.synchronize()
        finally:
            eng.use_cuda_graph = use_graph
            del eng._step                               # back to the class method
            for name, fn in saved.items():
                setattr(ops, name, fn)
        agg = {}
        for fam, flops, nbytes, e0, e1, label in self.records:
            a = agg.setdefault(fam, {"launch_groups": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            ms = e0.elapsed_time(e1)
            a["launch_groups"] += 1
            a["ms"] += ms
            a["flops"] += flops
            a["bytes"] += nbytes
            sh = self.shapes.setdefault(fam + " " + label, [0, 0.0, 0.0])
            sh[0] += 1
            sh[1] += ms
            sh[2] += flops
        if os.environ.get("IH_BENCH_SHAPES", "0") == "1":
            rows = sorted(self.shapes.items(), key=lambda kv: -kv[1][1])
            os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
            with open(os.path.join(ROOT, "gpurun_out", "bench_shapes.md"), "w") as f:
                f.write("| family op:shape (x rows x cols | w) | calls | total ms | avg us | TFLOP/s |\n|---|---:|---:|---:|---:|\n")
                for k, (n, ms, fl) in rows:
                    f.write(f"| {k} | {n} | {ms:.3f} | {ms / n * 1e3:.1f} | {fl / (ms * 1e-3) / 1e12 if fl else 0:.0f} |\n")
        return agg


def family_roofline(agg, pk, step_ms_graph):
    total = sum(a["ms"] for a in agg.values()) or 1.0
    fams = {}
    for fam, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        row = {"kernel": FamilyTimer.FAMILIES.get(fam, fam), "calls": a["launch_groups"], "ms": round(a["ms"], 4),
               "share": round(a["ms"] / total, 4)}
        if a["flops"] > 0:
            row.update(bound="tensor", achieved=a["flops"] / (a["ms"] * 1e-3) / 1e12, unit="TFLOP/s")
            row["frac"] = row["achieved"] / pk["tflops_sustained"]
        elif a["bytes"] > 0:
            row.update(bound="hbm", achieved=a["bytes"] / (a["ms"] * 1e-3) / 1e9, unit="GB/s")
            row["frac"] = row["achieved"] / pk["hbm_gbs"]
        fams[fam] = row
    dom = next(iter(fams))
    d = fams[dom]
    traffic, tsrc = None, "no ncu capture committed for this family yet (profiles/r2_traffic.json absent)"
    if os.path.exists(TRAFFIC_FILE):
        try:
            tj = json.load(open(TRAFFIC_FILE))
            if dom in tj:
                traffic, tsrc = tj[dom]["dram_bytes_per_launch"], tj[dom]["source"]
        except Exception as ex:  # pragma: no cover
            tsrc = f"unreadable {TRAFFIC_FILE}: {ex}"
    return {"bound": d.get("bound", "tensor"), "kernel": d["kernel"], "family": dom, "achieved": d.get("achieved"),
            "peak": pk["tflops_sustained"] if d.get("bound") == "tensor" else pk["hbm_gbs"], "unit": d.get("unit"),
            "frac": d.get("frac"), "share_of_step": d["share"], "traffic": traffic, "traffic_source": tsrc,
            "event_ms_total": total, "graph_ms_per_step": step_ms_graph,
            "frac_if_scaled_to_graph_time": (d.get("frac") * total / step_ms_graph) if d.get("frac") else None,
            "peak_source": pk["source"] + "; sustained figure: the families are timed inside a full step",
            "how": "one eager denoise step, CUDA-event pair around every launch, queued behind a spin kernel; achieved = "
                   "family algorithmic FLOPs (bytes for GroupNorm) / family time; sum of event times "
                   f"{total:.2f} ms vs {step_ms_graph:.2f} ms graph-replayed (event pairs add idle time per launch and suppress PDL "
                   "overlap, so `achieved` / `frac` are LOWER bounds; `frac_if_scaled_to_graph_time` spreads the graph-replayed "
                   "step time over the families by their event-time shares)",
            "families": fams}


def gpu_eager_baseline(cfg, lat: int, n: int, iters: int = 5):
    """The oracle UNet (reference processors + restated diffusers UNet) in torch-eager fp16 on this GPU, and the same
    replayed as a CUDA graph: the stand-in for "the reference GPU diffusers path" (cuDNN / cuBLAS / torch SDPA)."""
    from oracle import adapter_ref as A
    from oracle.unet_ref import UNetRef
    torch.backends.cuda.matmul.allow_tf32 = True
    with torch.device("meta"):
        m = UNetRef(cfg)
    m = m.to_empty(device="cuda").half()
    with torch.no_grad():
        for p in m.parameters():
            if p.dim() == 1:
                p.fill_(0.5)
            else:
                p.uniform_(-0.02, 0.02)
    with torch.device("cuda"):
        A.install_processors(m, cfg, dtype=torch.float16)
    m.eval()
    B = 2 * n
    res = lat * 8.0
    x = torch.randn(B, 4, lat, lat, device="cuda").half()
    ehs = torch.randn(B, 81, cfg.cross_attention_dim, device="cuda").half()
    te = torch.randn(B, cfg.pooled_embed_dim, device="cuda").half()
    tid = torch.tensor([[res, res, 0, 0, res, res]] * B, device="cuda", dtype=torch.float32)
    out = {"what": "oracle UNet forward (reference processors + restated diffusers UNet), torch fp16 on the same GPU; one "
                   "forward per denoise step (CFG combine + Euler not included: they favour this baseline)",
           "unet_batch": B, "res": int(res), "torch": torch.__version__}
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(2):
            m(x, 500.0, ehs, te, tid)
        torch.cuda.synchronize()
        s.record()
        for _ in range(iters):
            m(x, 500.0, ehs, te, tid)
        e.record()
        torch.cuda.synchronize()
        out["eager_ms_per_step"] = s.elapsed_time(e) / iters
        try:
            tt = torch.full((B,), 500.0, device="cuda")
            g = torch.cuda.CUDAGraph()
            st = torch.cuda.Stream()
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                m(x, tt, ehs, te, tid)
            torch.cuda.current_stream().wait_stream(st)
            with torch.cuda.graph(g):
                m(x, tt, ehs, te, tid)
            g.replay()
            torch.cuda.synchronize()
            s.record()
            for _ in range(iters):
                g.replay()
            e.record()
            torch.cuda.synchronize()
            out["graph_ms_per_step"] = s.elapsed_time(e) / iters
            del g
        except Exception as ex:  # pragma: no cover
            out["graph_ms_per_step"] = None
            out["graph_error"] = str(ex)[:200]
    del m
    torch.cuda.empty_cache()
    return out


def build_clip_judge(device):
    """The PNS judge north_star names ("allgather of CLIP scores"): candidate latents -> native VAE decoder -> device-side
    resize / normalise / patchify -> ViT-bigG/14 vision tower -> cosine with the bigG text embedding of the prompt.  Real
    architectures (SDXL VAE, OpenCLIP bigG towers), random-init weights generated on the GPU, identical on every rank."""
    from imagharmony_b200.clip import ClipScorer, ClipTextTower, ClipTowerConfig, ClipVisionTower, tower_param_shapes
    from imagharmony_b200.config import SDXL_VAE
    from imagharmony_b200.vae import AutoencoderKLDecoder
    from imagharmony_b200.weights import random_state_dict, shapes_of
    vcfg = ClipTowerConfig(hidden_size=1664, intermediate_size=8192, num_hidden_layers=48, num_attention_heads=16,
                           hidden_act="gelu", projection_dim=1280, image_size=224, patch_size=14)
    tcfg = ClipTowerConfig(hidden_size=1280, intermediate_size=5120, num_hidden_layers=32, num_attention_heads=20,
                           hidden_act="gelu", projection_dim=1280, vocab_size=49408, eos_token_id=49407)
    vision = ClipVisionTower(vcfg, random_state_dict(tower_param_shapes(vcfg, "vision"), 31, device=device), device=device)
    text = ClipTextTower(tcfg, random_state_dict(tower_param_shapes(tcfg, "text"), 32, device=device), device=device)
    with torch.device("meta"):
        vshapes = shapes_of(AutoencoderKLDecoder(SDXL_VAE))
    vae = AutoencoderKLDecoder.from_state_dict(SDXL_VAE, random_state_dict(vshapes, 33, device=device), device=device)
    scorer = ClipScorer(vision, text, decode=vae.decode)
    ids = torch.full((1, 77), 49407, dtype=torch.int64)
    ids[0, 0] = 49406
    ids[0, 1:9] = torch.tensor([320, 1125, 539, 5567, 15, 2533, 3027, 267])      # a fixed synthetic prompt (no vocabulary offline)
    scorer.set_prompt(input_ids=ids)
    return scorer


def pns_block(args, eng, cfg, lat, K, rank, world, device, dist, single_step_ms):
    """BASELINE config 4 shape at this world size: 4 candidate noises per GPU, K steps each, one batch per rank:
    H2D -> K graph replays -> score -> all_gather -> argmax -> winner broadcast; wall clock, max over ranks."""
    from imagharmony_b200.pns import LinearProbeScorer, pns_select
    from imagharmony_b200.scheduler import EulerDiscreteScheduler
    per = 4
    N = per * world
    seeds = [5000 + i for i in range(N)]
    ins = EulerDiscreteScheduler().set_timesteps(K).init_noise_sigma
    _, pos1, neg1, pooled1, npooled1, tid1 = synth_inputs(cfg, 1, lat, K, 0)
    rep = lambda t, b: t.repeat(b, *([1] * (t.dim() - 1))).pin_memory()  # noqa: E731

    def run_candidates(batch_seeds):
        b = len(batch_seeds)
        lat0 = torch.cat([torch.randn((1, 4, lat, lat), generator=torch.Generator("cpu").manual_seed(s))
                          for s in batch_seeds]) * ins
        return eng.run(lat0.half().pin_memory(), rep(pos1, b), rep(neg1, b), rep(pooled1, b), rep(npooled1, b),
                       rep(tid1, b), K, guidance_scale=5.0, ip_scale=1.0)
    scorer = build_clip_judge(device) if args.pns_judge == "clip" else LinearProbeScorer(4 * lat * lat, seed=99, device=device)
    eng.run(*[t.pin_memory() for t in synth_inputs(cfg, per, lat, K, rank)], K, stop_after=2)     # capture batch-8 graph
    scorer(torch.zeros((per, 4, lat, lat), dtype=torch.float16, device=device))                   # warm the judge
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = pns_select(run_candidates, seeds, scorer, dist=dist, max_batch=per)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    tt = torch.tensor([wall], device=device, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    wall = float(tt[0])
    single = single_step_ms * 1e-3 * K
    bar = 1.1 * single * N / world
    return {"candidates": N, "per_gpu": per, "steps": K, "wall_s": wall, "edits_per_s": N / wall,
            "single_candidate_s": single, "bar_s": bar, "within_bar": wall <= bar, "best_seed": res.best_seed,
            "collective": "all_gather of N fp32 scores + broadcast of the winning latent (NCCL)",
            "scorer": scorer.describe()}


def run_pns(args, eng, cfg, lat, K, W, rank, world, device, dist):
    """`--pns N`: PNS N candidates: shard seeds over ranks, K-step trajectories in batches, score, all_gather, argmax."""
    from imagharmony_b200.pns import LinearProbeScorer, pns_select, pns_two_phase, shard_seeds
    from imagharmony_b200.scheduler import EulerDiscreteScheduler
    N = args.pns
    seeds = [5000 + i for i in range(N)]
    ins = EulerDiscreteScheduler().set_timesteps(K).init_noise_sigma
    _, pos1, neg1, pooled1, npooled1, tid1 = synth_inputs(cfg, 1, lat, K, 0)

    P = max(0, min(args.pns_preview, K))               # two-phase PNS: P preview steps for everyone, K - P for the winner
    rep = lambda t, b: t.repeat(b, *([1] * (t.dim() - 1))).pin_memory()  # noqa: E731

    def run_candidates(batch_seeds):
        b = len(batch_seeds)
        lat0 = torch.cat([torch.randn((1, 4, lat, lat), generator=torch.Generator("cpu").manual_seed(s))
                          for s in batch_seeds]) * ins
        return eng.run(lat0.half().pin_memory(), rep(pos1, b), rep(neg1, b), rep(pooled1, b), rep(npooled1, b),
                       rep(tid1, b), K, guidance_scale=5.0, ip_scale=1.0, stop_after=(P if P else None))

    def run_rest(preview):
        return eng.run(preview, rep(pos1, 1), rep(neg1, 1), rep(pooled1, 1), rep(npooled1, 1), rep(tid1, 1), K,
                       guidance_scale=5.0, ip_scale=1.0, start_step=P)

    scorer = build_clip_judge(device) if args.pns_judge == "clip" else LinearProbeScorer(4 * lat * lat, seed=99, device=device)
    scorer(torch.zeros((1, 4, lat, lat), dtype=torch.float16, device=device))          # warm the judge
    mine = shard_seeds(seeds, rank, world)
    if mine:                                           # warm-up: capture the graphs for this rank's batch sizes
        for bsz in sorted({min(args.pns_batch, len(mine)), len(mine) % args.pns_batch or args.pns_batch} | ({1} if P else set())):
            eng.run(*[t.pin_memory() for t in synth_inputs(cfg, bsz, lat, K, rank)], K, stop_after=W)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if P:
        res = pns_two_phase(run_candidates, run_rest, seeds, scorer, dist=dist, max_batch=args.pns_batch)
    else:
        res = pns_select(run_candidates, seeds, scorer, dist=dist, max_batch=args.pns_batch)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if dist is not None:
        tt = torch.tensor([wall], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        wall = float(tt[0])
    if rank == 0:
        steps_done = N * (P if P else K) + (K - P if P else 0)     # trajectory steps actually executed for the result
        line = {"metric": METRIC + " -- PNS", "value": steps_done / wall, "unit": "denoise-steps/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": wall / K * 1e3, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                "config": {"workload": f"PNS N={N} candidate noises, {args.res}x{args.res}, "
                                       + (f"{P} preview steps each + {K - P} steps for the winner, " if P else f"{K} steps each, ") +
                                       f"{args.pns_batch} candidates per batch, score = {scorer.describe()}, "
                                       f"all_gather of N fp32 scores + broadcast of the winner",
                           "pns_edits_per_s": N / wall, "pns_wall_s": wall, "best_seed": res.best_seed},
                "e2e": {"value": steps_done / wall, "unit": "denoise-steps/s",
                        "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
                        "note": "PNS wall clock includes H2D of every candidate batch and the score gather"},
                "gpu_launches": int(eng.last_launches_per_step * K * ((len(mine) + args.pns_batch - 1) // args.pns_batch))}
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--images", type=int, default=1, help="images (noise candidates) per GPU; UNet batch = 2x (CFG)")
    ap.add_argument("--res", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-families", action="store_true", help="skip the per-family roofline pass")
    ap.add_argument("--pns", type=int, default=0,
                    help="PNS mode: N candidate noises in total, sharded over the ranks (BASELINE config 4: N=32 on 8 GPUs)")
    ap.add_argument("--pns-batch", type=int, default=4, help="candidates denoised together per rank (UNet batch 2x)")
    ap.add_argument("--pns-judge", default="clip", choices=["clip", "probe"],
                    help="judge of the N > 1 `pns` block: native CLIP image-text cosine on decoded candidates (random-init "
                         "bigG towers + SDXL VAE) or the synthetic linear probe of the latent")
    ap.add_argument("--pns-preview", type=int, default=0,
                    help="two-phase PNS: preview steps per candidate before the judge; the winner alone runs the rest")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the final latents of the timed steps to DIR/latents.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.pns > 0):
        ap.error("--dump-outputs records the timed denoise steps of the native path; not with --impl reference or --pns")

    if args.impl == "reference":
        run_reference_arm(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)

    from imagharmony_b200 import ops
    from imagharmony_b200.config import SDXL_BASE as cfg
    from imagharmony_b200.denoise import DenoiseEngine
    from imagharmony_b200.pns import LinearProbeScorer, pns_select

    K, W, n = args.steps, max(args.warmup, 3), args.images
    lat = args.res // 8
    unet = build_native(cfg, device)
    eng = DenoiseEngine(unet, use_cuda_graph=True)
    if args.pns > 0:
        run_pns(args, eng, cfg, lat, K, W, rank, world, device, dist)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return
    run_args = [t.pin_memory() for t in synth_inputs(cfg, n, lat, K, rank)] + [K]
    latents = run_args[0]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up: W steps through the public call (captures the graph, fills caches) -------------------------------
    ops.launch_count_reset()
    eng.run(*run_args, guidance_scale=5.0, ip_scale=1.0, stop_after=W)
    torch.cuda.synchronize()
    launches_per_step = eng.last_launches_per_step

    # ---- device-resident timing: K graph replays (+ the PNS tail when N > 1), CUDA events, max over ranks ----------
    st = eng._buffers(n, lat, lat, run_args[1].shape[1])
    timesteps, sigmas, _ = eng.tables(K)
    graph = next(iter(eng._graphs.values()))[0]
    scorer = LinearProbeScorer(4 * lat * lat, seed=99, device=device)
    seeds_all = list(range(world * n))
    if world > 1:                                           # warm the collective path (NCCL communicator set-up)
        pns_select(lambda s: st["latents"], seeds_all, scorer, dist=dist, max_batch=n)
    st["latents"].copy_(latents)
    st["step"].zero_()
    ops.scale_model_input(st["latents"], st["model_in"], sigmas, st["step"])
    barrier()
    ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    tail = None
    with ClockSampler(local_rank) as clocks:
        ev0.record()
        for _ in range(K):
            graph.replay()
        ev1.record()
        if world > 1:
            tail = pns_select(lambda s: st["latents"], seeds_all, scorer, dist=dist, max_batch=n)
        ev2.record()
        barrier()
    dev_s = ev0.elapsed_time(ev2) * 1e-3
    tail_ms = ev1.elapsed_time(ev2)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latents" if world == 1 else f"latents_rank{rank}": st["latents"]})

    # ---- end to end through the public API: pinned host inputs -> H2D -> K steps -> D2H of the result -------------
    barrier()
    t0 = time.perf_counter()
    out = eng.run(*run_args, guidance_scale=5.0, ip_scale=1.0)
    host_out = out.to("cpu", non_blocking=False)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert torch.isfinite(host_out.float()).all(), "non-finite latents"
    h2d = sum(t.numel() * t.element_size() for t in run_args[:6]) + run_args[5].numel() * run_args[5].element_size()
    d2h = host_out.numel() * host_out.element_size()

    if dist is not None:
        tt = torch.tensor([dev_s, e2e_s, tail_ms], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_s, e2e_s, tail_ms = float(tt[0]), float(tt[1]), float(tt[2])
    step_ms = dev_s / K * 1e3

    pns = None
    if world > 1:
        pns = pns_block(args, eng, cfg, lat, K, rank, world, device, dist, step_ms)

    if rank == 0:
        pk = peaks()
        step_tflop = TFLOP_PER_PAIR.get(lat, 13.524 * (lat / 128.0) ** 2) * n
        line = {
            "metric": METRIC, "value": world * n * K / dev_s, "unit": "denoise-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": workload_string(args.res, K, n),
                       "l2": "per-step working set (5.2 GB weights) exceeds L2; inputs larger than L2",
                       "step_tflop_algorithmic": step_tflop,
                       "step_tflops_achieved": step_tflop * K / dev_s,
                       "step_frac_of_sustained_peak": step_tflop * K / dev_s / pk["tflops_sustained"],
                       "cuda_graph": True,
                       "timed_region": "K graph replays" + (
                           f" + PNS tail (score -> all_gather of {world * n} fp32 -> argmax -> winner broadcast, "
                           f"{tail_ms:.3f} ms)" if world > 1 else "")},
            "e2e": {"value": world * n * K / e2e_s, "unit": "denoise-steps/s", "h2d_bytes_per_step": h2d / K,
                    "d2h_bytes_per_step": d2h / K, "note": "copies happen once per K-step call; bytes amortised per step"},
            "gpu_launches": int(launches_per_step * K + (2 if world > 1 else 0)),
            "clocks": clocks.summary(),
        }
        if pns is not None:
            line["pns"] = pns
        if not args.no_families:
            try:
                agg = FamilyTimer().measure(eng, run_args)
                line["roofline"] = family_roofline(agg, pk, step_ms)
            except Exception as ex:  # pragma: no cover
                line["roofline"] = {"bound": "tensor", "achieved": None, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
                                    "frac": None, "traffic": None, "error": str(ex)[:300]}
        if world == 1:
            # BASELINE config 1 shape on the native path (what the CPU arm times): 512^2, one image
            try:
                a512 = [t.pin_memory() for t in synth_inputs(cfg, 1, 64, K, 0)] + [K]
                eng.run(*a512, stop_after=W)
                s5 = eng._buffers(1, 64, 64, a512[1].shape[1])
                g5 = next(v[0] for k, v in eng._graphs.items() if k[:3] == (1, 64, 64))
                s5["step"].zero_()
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(K):
                    g5.replay()
                b.record()
                torch.cuda.synchronize()
                ms5 = a.elapsed_time(b) / K
                line["c1_512"] = {"workload": "single 512x512 edit, UNet batch 2 (BASELINE config 1 shape), graph-replayed",
                                  "value": 1e3 / ms5, "unit": "denoise-steps/s", "ms_per_step": ms5,
                                  "step_tflops_achieved": TFLOP_PER_PAIR[64] / (ms5 * 1e-3)}
            except Exception as ex:  # pragma: no cover
                line["c1_512"] = {"error": str(ex)[:300]}
            if not args.no_eager_baseline:
                try:
                    line["gpu_eager_baseline"] = gpu_eager_baseline(cfg, lat, n)
                    gb = line["gpu_eager_baseline"]
                    gb["native_ms_per_step"] = step_ms
                    gb["speedup_vs_eager"] = gb["eager_ms_per_step"] / step_ms
                    if gb.get("graph_ms_per_step"):
                        gb["speedup_vs_graph_replayed"] = gb["graph_ms_per_step"] / step_ms
                except Exception as ex:  # pragma: no cover
                    line["gpu_eager_baseline"] = {"error": str(ex)[:300]}
            if not args.no_cpu_baseline:
                try:
                    oracle = CpuOracle()
                    lat_c, _ = pick_cpu_sample(oracle, 2, 1, budget_s=30.0)
                    sec = oracle.timed_steps(lat_c, 2, 1)
                    v = 2 / sec
                    line["cpu_baseline"] = {"value": v, "unit": "denoise-steps/s", "cores": oracle.threads, "kind": "port",
                                            "sample": cpu_sample_text(oracle, lat_c, 2, 1), "sample_res": lat_c * 8,
                                            "value_scaled_to_1024": v * TFLOP_PER_PAIR[lat_c] / TFLOP_PER_PAIR[128]}
                except Exception as ex:  # pragma: no cover
                    line["cpu_baseline"] = {"value": None, "unit": "denoise-steps/s", "cores": host_threads(),
                                            "kind": "port", "sample": f"failed: {ex}"}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
