#!/usr/bin/env python
"""Benchmark of the Aurora forward hot path (BASELINE.json: forecast-steps/sec on the 0.25-degree
721x1440x13-level configuration, B = 1, history 2; 1.3 B-parameter `Aurora`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

* `--impl ours` (default): one "step" = one `Aurora.forward` through the sm_100a kernels.
    value : steps/s with the input Batch already resident in HBM (CUDA events, max over ranks)
    e2e   : steps/s through the public API starting from PINNED HOST tensors, H2D of every input field
            and D2H of the whole prediction inside the timed region
    roofline     : dominant kernel (tcgen05 GEMM): algorithmic FLOPs / CUDA-event time per launch vs the
                   measured cuBLAS bf16 peak of MEASURED_PEAKS.json; plus the attention and adaLN kernels
    cpu_baseline : the CPU oracle port timed on this box's host cores on a bounded sample (N = 1 only)
* `--impl reference`: the reference algorithm's CPU implementation (oracle port; the Python reference
  itself cannot travel to the GPU box) on the host cores, each step a bounded sample extrapolated by
  algorithmic FLOPs.
* N > 1: the forward pass does not need a collective for independent forecasts, so by default each rank runs
  its own replica of the workload ("weak" scaling, no data-path collective).  `--parallelism latshard` instead
  shards ONE forecast over the N GPUs by latitude band with an NCCL halo exchange per Swin block ("strong").

Synthetic data (ERA5-shaped, `loc + scale * N(0,1)` per variable / level) and random weights with the
reference's zero-initialised tensors re-drawn (otherwise every Swin block is an identity).
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from datetime import datetime
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

LEVELS13 = (50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000)

WORKLOADS = {
    # name: (model class, H, W, levels, description)
    "aurora-0.25deg-721x1440x13L": ("Aurora", 721, 1440, LEVELS13),
    "aurora-small-0.25deg-721x1440x13L": ("AuroraSmallPretrained", 721, 1440, LEVELS13),
    "aurora-small-17x32x4L": ("AuroraSmallPretrained", 17, 32, (100, 250, 500, 850)),
    "aurora-highres-0.1deg-1801x3600x13L": ("AuroraHighRes", 1801, 3600, LEVELS13),
    "aurora-airpollution-0.4deg-451x900x13L": ("AuroraAirPollution", 451, 900, LEVELS13),
    "aurora-wave-0.25deg-721x1440x13L": ("AuroraWave", 721, 1440, LEVELS13),
}
DEFAULT_WORKLOAD = "aurora-0.25deg-721x1440x13L"

# Algorithmic work of one forward step (SURVEY.md section 8(d) / App. B), 2 flops per MAC.
ALGO_TFLOP = {"aurora-0.25deg-721x1440x13L": 96.8, "aurora-highres-0.1deg-1801x3600x13L": 91.7,
              "aurora-airpollution-0.4deg-451x900x13L": 69.2, "aurora-wave-0.25deg-721x1440x13L": 96.8,
              "aurora-small-0.25deg-721x1440x13L": 12.6, "aurora-small-17x32x4L": 0.004}


def peaks() -> dict:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------
# synthetic inputs / weights
# ------------------------------------------------------------------------------------------------
def make_host_batch(cfg, h, w, levels, pinned: bool, seed: int = 0):
    """Physically scaled synthetic Batch on the host (optionally pinned)."""
    from aurora_b200 import Batch, Metadata
    from aurora_b200.stats import atmos_stats_of, surf_stats_of

    g = torch.Generator().manual_seed(seed)

    def alloc(shape):
        t = torch.empty(shape, dtype=torch.float32, pin_memory=pinned)
        t.normal_(generator=g)
        return t

    surf = {}
    surf_names = cfg.surf_vars
    wave = any(k.endswith("_density") for k in surf_names)
    if wave:  # AuroraWave takes the raw HRES-WAM names; absent wave components are NaN (here: a band of "land")
        surf_names = tuple(dict.fromkeys(k.removesuffix("_density").removesuffix("_sin").removesuffix("_cos")
                                         for k in surf_names))
    for k in surf_names:
        loc, sc = surf_stats_of(k)
        surf[k] = alloc((1, 2, h, w)).mul_(sc).add_(loc)
        if wave and k not in ("2t", "10u", "10v", "msl", "wind"):
            surf[k].abs_().clamp_(min=0.05)
            surf[k][..., :, : w // 4] = float("nan")
    static = {}
    for k in cfg.static_vars:
        loc, sc = surf_stats_of(k)
        static[k] = alloc((h, w)).mul_(sc).add_(loc)
        if k in ("wmb", "lat_mask"):
            static[k].copy_((static[k] > -1.0).float())
    atmos = {}
    for k in cfg.atmos_vars:
        locs, scs = atmos_stats_of(k, levels)
        t = alloc((1, 2, len(levels), h, w))
        t.mul_(torch.tensor(scs)[None, None, :, None, None]).add_(torch.tensor(locs)[None, None, :, None, None])
        atmos[k] = t
    meta = Metadata(lat=torch.linspace(90, -90, h), lon=torch.linspace(0, 360, w + 1)[:-1],
                    time=(datetime(2020, 6, 1, 12, 0),), atmos_levels=tuple(levels))
    return Batch(surf, static, atmos, meta)


def randomise_parameters_(model, seed: int = 0) -> None:
    """Random weights on the device: N(0, 0.02) matrices, the reference's zero-initialised adaLN
    modulation / LoRA-B / biases re-drawn so that every block contributes (timing is weight-independent)."""
    g = torch.Generator(device=next(model.parameters()).device).manual_seed(seed)
    for name, p in model.named_parameters():
        if name.endswith("norm.weight") or name.endswith(".2.weight") and p.dim() == 1 or name.endswith(".3.weight"):
            p.data.fill_(1.0)
        elif "ln_modulation" in name:
            p.data.normal_(0.0, 0.1, generator=g)
        elif p.dim() == 1:
            p.data.normal_(0.0, 0.02, generator=g)
        elif "token_embeds.weights" in name:
            p.data.uniform_(-0.1, 0.1, generator=g)
        else:
            p.data.normal_(0.0, 0.02, generator=g)
    for name, p in model.named_parameters():
        if p.dim() == 1 and ("surf_norm.weight" in name or name.endswith("norm.weight")):
            p.data.fill_(1.0)


DUMP_MAX_BYTES = 64 * 10**6  # --dump-outputs: all .npy files together stay below this


def dump_outputs(pred, out_dir: str) -> None:
    """Write the prediction `pred` as float32 `out_dir/<group>_<name>.npy` (group: surf, static, atmos).  When all
    fields together would exceed DUMP_MAX_BYTES, every field keeps the same share of its values, flattened, at sorted
    flat indices drawn from one generator seeded with 0 in field order: two builds given the same arguments dump the
    same points."""
    import numpy as np

    fields = {f"{grp}_{k}": v.detach() for grp, d in (("surf", pred.surf_vars), ("static", pred.static_vars),
                                                       ("atmos", pred.atmos_vars)) for k, v in d.items()}
    budget = DUMP_MAX_BYTES // 4 - 1024 * len(fields)  # float32 values; 4 KiB per file left for the .npy header
    share = min(1.0, budget / sum(v.numel() for v in fields.values()))
    g = torch.Generator().manual_seed(0)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, v in fields.items():
        if share < 1.0:
            idx = torch.randint(v.numel(), (int(v.numel() * share),), generator=g).unique()
            v = v.reshape(-1)[idx.to(v.device)]
        np.save(out / f"{name}.npy", v.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self) -> dict:
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = []
        for i, nm in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
            if any(r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------
# Reference legs: the UNMODIFIED reference (oracle/_ref, see oracle/build_ref.py) on the host cores and on the GPU
# ------------------------------------------------------------------------------------------------
CPU_THREADS_CAP = 32  # PyTorch's CPU kernels stop scaling on many-core hosts (128 threads measured 2.8x SLOWER than 32)
SAMPLE_LAT_DIV = 3    # the bounded sample keeps the first 1/3 of the latitude rows of every U-Net stage (fixed)


def host_threads() -> int:
    return max(1, min(CPU_THREADS_CAP, os.cpu_count() or 1))


def build_reference(workload: str, device: str, autocast: bool, seed: int = 0):
    """The unmodified reference model of this workload with the same random parameters the `ours` arm uses."""
    from oracle import ref

    cls, h, w, levels = WORKLOADS[workload]
    model = ref.build_model(cls, device=device, autocast=autocast)
    randomise_parameters_(model, seed=seed)
    return model


def reference_sample_fn(model, workload: str):
    """One bounded-sample "step" of the reference's CPU path: the reference's OWN modules with their own weights —
    the second (shifted-window) Swin3DTransformerBlock of every encoder stage on the first 1/SAMPLE_LAT_DIV of the
    stage's latitude rows (whole window rows), plus the Perceiver decoder's MLP on the same fraction of its rows.
    The sample is the same whatever --steps is."""
    cls, h, w, levels = WORKLOADS[workload]
    p = model.patch_size
    res0 = (4, (h - h % p) // p, w // p)
    g = torch.Generator().manual_seed(0)
    dev = next(model.parameters()).device
    c = torch.randn(1, model.backbone.time_mlp[0].in_features, generator=g).to(dev)
    items = []
    res = res0
    for i, layer in enumerate(model.backbone.encoder_layers):
        blk = layer.blocks[min(1, len(layer.blocks) - 1)]
        wh = blk.window_size[1]
        rows = max(wh, (res[1] // SAMPLE_LAT_DIV + wh - 1) // wh * wh) if res[1] > wh else res[1]
        r = (res[0], min(rows, res[1]), res[2])
        x = torch.randn(1, r[0] * r[1] * r[2], blk.dim, generator=g).to(dev)
        items.append((blk, x, r))
        res = (res[0], (res[1] + res[1] % 2) // 2, (res[2] + res[2] % 2) // 2)
    mlp = model.decoder.level_decoder.layers[0][1]
    e = mlp.net[0].in_features
    rows = max(1024, len(levels) * res0[1] * res0[2] // (4 * SAMPLE_LAT_DIV))
    xm = torch.randn(1, rows, e, generator=g).to(dev)

    def step() -> float:
        t0 = time.perf_counter()
        with torch.inference_mode():
            for blk, x, r in items:
                blk(x, c, r, rollout_step=0)
            mlp(xm)
        return time.perf_counter() - t0

    desc = ("reference modules on a bounded sample: shifted Swin3DTransformerBlock of every encoder stage on "
            + ", ".join(f"{r}" for _, _, r in items) + f" tokens + Perceiver-decoder MLP on {rows} rows, fp32")
    return step, desc


def reference_cpu_measure(workload: str, n_warm: int, n_timed: int) -> dict:
    """The reference's CPU path on this box's host cores: ONE complete `Aurora.forward` of the real reference on the
    workload (timed, after the samples have warmed oneDNN up), and `n_timed` bounded-sample steps.  The samples are
    scaled to whole steps by the factor measured in this very run (complete forward / median sample), not by FLOPs."""
    from oracle import ref

    threads = host_threads()
    torch.set_num_threads(threads)
    cls, h, w, levels = WORKLOADS[workload]
    model = build_reference(workload, "cpu", autocast=False)
    step, desc = reference_sample_fn(model, workload)
    for _ in range(max(1, n_warm)):
        step()
    batch = ref.to_ref_batch(make_host_batch(_our_config(workload), h, w, levels, pinned=False))
    t0 = time.perf_counter()
    with torch.inference_mode():
        model.forward(batch)
    t_full = time.perf_counter() - t0
    del batch
    times = [step() for _ in range(max(1, n_timed))]
    med = statistics.median(times)
    scale = t_full / med
    return {
        "value": len(times) / (sum(times) * scale), "unit": "forecast-steps/s", "cores": threads, "kind": "reference",
        "complete_forward_seconds": t_full, "sample_seconds_median": med, "sample_seconds_min": min(times),
        "sample_seconds_max": max(times), "samples": len(times), "sample_scale": scale,
        "sample": f"unmodified reference (oracle/_ref) {cls}, fp32, {threads} host threads of {os.cpu_count()}: one COMPLETE "
                  f"forward on the {h}x{w}x{len(levels)}L batch = {t_full:.1f} s; steps = {desc}; each sample "
                  f"({med:.2f} s median) is scaled to a whole step by the factor complete/median = {scale:.1f} measured in "
                  f"this run",
        "_times": times,
    }


def port_cpu_measure(workload: str, n_timed: int) -> dict:
    """Fallback when oracle/_ref did not travel: the oracle PORT (oracle/aurora_oracle.py) on the same fixed sample
    geometry, scaled to a step by algorithmic FLOPs (no complete forward: kind "port")."""
    from oracle import aurora_oracle as O
    import aurora_b200 as ab

    threads = host_threads()
    torch.set_num_threads(threads)
    cls, h, w, levels = WORKLOADS[workload]
    cfg = getattr(ab, cls)(_init="empty").config
    cfg = type(cfg)(**{**cfg.__dict__, "use_lora": False})
    p = cfg.patch_size
    res = (cfg.latent_levels, (h - h % p) // p, w // p)
    g = torch.Generator().manual_seed(0)
    c = torch.randn(1, cfg.embed_dim, generator=g)
    items, flops = [], 0.0
    for i in range(len(cfg.encoder_depths)):
        wh = cfg.window_size[1]
        r = (res[0], min(res[1], max(wh, (res[1] // SAMPLE_LAT_DIV + wh - 1) // wh * wh)), res[2])
        d, heads = cfg.embed_dim * 2**i, cfg.encoder_num_heads[i]
        sd = {"blk." + k: v for k, v in {
            "norm1.ln_modulation.1.weight": torch.randn(2 * d, cfg.embed_dim, generator=g) * 0.02,
            "norm1.ln_modulation.1.bias": torch.randn(2 * d, generator=g) * 0.1,
            "norm2.ln_modulation.1.weight": torch.randn(2 * d, cfg.embed_dim, generator=g) * 0.02,
            "norm2.ln_modulation.1.bias": torch.randn(2 * d, generator=g) * 0.1,
            "attn.qkv.weight": torch.randn(3 * d, d, generator=g) * 0.02, "attn.qkv.bias": torch.randn(3 * d, generator=g) * 0.02,
            "attn.proj.weight": torch.randn(d, d, generator=g) * 0.02, "attn.proj.bias": torch.randn(d, generator=g) * 0.02,
            "mlp.fc1.weight": torch.randn(4 * d, d, generator=g) * 0.02, "mlp.fc1.bias": torch.randn(4 * d, generator=g) * 0.02,
            "mlp.fc2.weight": torch.randn(d, 4 * d, generator=g) * 0.02, "mlp.fc2.bias": torch.randn(d, generator=g) * 0.02,
        }.items()}
        l = r[0] * r[1] * r[2]
        items.append((sd, torch.randn(1, l, d, generator=g), r, heads))
        flops += 24.0 * l * d * d + 4.0 * l * 144 * d
        res = (res[0], (res[1] + res[1] % 2) // 2, (res[2] + res[2] % 2) // 2)

    def step():
        t0 = time.perf_counter()
        with torch.inference_mode():
            for sd, x, r, heads in items:
                O.swin_block(sd, "blk", x, c, r, heads, True, cfg, 0)
        return time.perf_counter() - t0

    step()
    times = [step() for _ in range(max(1, n_timed))]
    med = statistics.median(times)
    scale = ALGO_TFLOP[workload] * 1e12 / flops
    return {"value": len(times) / (sum(times) * scale), "unit": "forecast-steps/s", "cores": threads, "kind": "port",
            "sample_seconds_median": med, "samples": len(times), "sample_scale": scale,
            "sample": f"oracle PORT (oracle/_ref missing): one shifted Swin block per stage on 1/{SAMPLE_LAT_DIV} of the "
                      f"latitude rows, fp32, {threads} threads; scaled to a step by algorithmic FLOPs x{scale:.1f}",
            "_times": times}


def cpu_measure(workload: str, n_warm: int, n_timed: int) -> dict:
    from oracle import ref

    if ref.available():
        return reference_cpu_measure(workload, n_warm, n_timed)
    return port_cpu_measure(workload, n_timed)


def gpu_reference_measure(workload: str, dev_batch, device) -> dict:
    """The unmodified reference on the SAME GPU (`model.cuda()`), fp32 (its default) and `autocast=True` (bf16 backbone,
    the reference's own reduced-precision recipe): the denominator of north_star's ">= 10x the reference single-GPU
    PyTorch forward".  Batch resident on the device, CUDA events, 1 warm-up + 3 timed forwards, median."""
    from oracle import ref

    out = {"tf32_matmul_allowed": bool(torch.backends.cuda.matmul.allow_tf32),
           "sdpa": {"flash": torch.backends.cuda.flash_sdp_enabled(), "mem_efficient": torch.backends.cuda.mem_efficient_sdp_enabled(),
                    "math": torch.backends.cuda.math_sdp_enabled(),
                    "note": "the float window mask makes the flash backend ineligible in shifted blocks (SURVEY K2)"},
           "torch": torch.__version__}
    rb = ref.to_ref_batch(dev_batch)
    for tag, autocast in (("fp32", False), ("autocast_bf16", True)):
        try:
            model = build_reference(workload, device, autocast=autocast)
            with torch.inference_mode():
                model.forward(rb)
                torch.cuda.synchronize()
                ts = []
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    model.forward(rb)
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
            out[tag] = {"ms_per_step": statistics.median(ts), "value": 1000.0 / statistics.median(ts),
                        "unit": "forecast-steps/s", "ms_all": ts,
                        "peak_mem_gb": torch.cuda.max_memory_allocated() / 2**30}
            del model
        except Exception as e:  # e.g. out of memory on a smaller part: report, do not fail the bench
            out[tag] = {"error": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.empty_cache()
    return out


def _our_config(workload: str):
    import aurora_b200 as ab

    return getattr(ab, WORKLOADS[workload][0])(_init="empty").config


def gemm_traffic(workload: str, launches: int, algo_bytes: float) -> dict:
    """`traffic` of the roofline object: DRAM bytes (read + write) per GEMM launch from the committed ncu pass
    over one step of this workload (profiles/gemm_traffic.json, written by tools/ncu_traffic.py from the ncu CSV;
    bench.py cannot run ncu itself), next to the compulsory bytes per launch counted from the launch arguments."""
    out = {"traffic": None, "algorithmic_bytes": algo_bytes / launches if launches else None}
    f = ROOT / "profiles" / "gemm_traffic.json"
    if f.exists():
        rec = json.loads(f.read_text()).get(workload)
        if rec:
            out["traffic"] = rec["dram_bytes_per_launch"]
            out["traffic_source"] = rec["source"]
    return out


# ------------------------------------------------------------------------------------------------
def resolve_parallelism(workload: str, gpus: int, mode: str) -> str:
    """`auto`: one forecast latitude-sharded over the GPUs whenever the workload's token grid can be split (bands must be
    multiples of 4 token rows so that the U-Net's 2x2 patch merges stay inside a band); otherwise independent replicas."""
    if gpus <= 1:
        return "single GPU"
    if mode == "replicas":
        return "replicas"
    from aurora_b200 import sharding

    cfg = _our_config(workload)
    _, h, _, _ = WORKLOADS[workload]
    try:
        sharding.plan_slabs((h - h % cfg.patch_size) // cfg.patch_size, len(cfg.encoder_depths), gpus)
    except (NotImplementedError, ValueError):
        if mode == "latshard":
            raise
        return "replicas"
    return "latshard"


def workload_config(workload: str, gpus: int = 1, mode: str = "auto") -> dict:
    """`config`: identical in both arms for the same command line (the driver compares it between the arms)."""
    cls, h, w, levels = WORKLOADS[workload]
    par = resolve_parallelism(workload, gpus, mode)
    return {"workload": workload, "model_class": cls, "grid": f"{h}x{w}", "levels": len(levels), "batch": 1,
            "history": 2, "algorithmic_tflop_per_step": ALGO_TFLOP[workload],
            "parallelism": {"single GPU": "single GPU", "replicas": f"replicas x{gpus} (one forecast per GPU)",
                            "latshard": f"one forecast latitude-sharded over {gpus} GPUs"}[par],
            "l2": "inputs and activations are GBs per step (>> 126 MB L2): no explicit flush between iterations"}


def run_reference_arm(args) -> None:
    """`--impl reference`: the reference's own CPU implementation on the host cores (rank 0 only).  W + K steps, each
    the SAME bounded sample (independent of K), plus one complete forward that calibrates sample -> step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m = cpu_measure(args.workload, args.warmup, args.steps)
    times = m.pop("_times")
    v = m["value"]
    line = {
        "impl": "reference", "metric": "forecast-steps/sec", "value": v, "unit": "forecast-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        # wall time of one timed (bounded-sample) step; a whole forecast step is `sample_scale` times that
        "ms_per_step": 1000.0 * sum(times) / len(times), "ms_per_whole_step": 1000.0 / v,
        "sample_scale": m.get("sample_scale"),
        "higher_is_better": True,
        "scaling": "strong" if resolve_parallelism(args.workload, args.gpus, args.parallelism) == "latshard" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, args.gpus, args.parallelism),
        "cpu_baseline": m,
        "e2e": {"value": v, "unit": "forecast-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--parallelism", default="auto", choices=["auto", "replicas", "latshard"],
                    help="N > 1: ONE forecast sharded by latitude over the N GPUs with a halo exchange per Swin block "
                         "(latshard; `auto` picks it whenever N > 1) or independent forecasts per GPU (replicas)")
    ap.add_argument("--halo", default="peer", choices=["peer", "nccl"],
                    help="latshard halo exchange: kernels writing straight into the neighbours' memory over NVLink inside "
                         "the step's CUDA graph (peer), or NCCL send/recv between graph segments (nccl)")
    ap.add_argument("--cuda-graph", dest="cuda_graph", action="store_true", default=None,
                    help="replay the step from a captured CUDA graph (default: on for latshard, off otherwise)")
    ap.add_argument("--no-cuda-graph", dest="cuda_graph", action="store_false")
    ap.add_argument("--no-gpu-reference", action="store_true",
                    help="skip timing the unmodified reference on the same GPU (N = 1 only)")
    ap.add_argument("--rollout", type=int, default=0, metavar="N",
                    help="also time one N-step autoregressive rollout (BASELINE configs[2]: 40) and add a `rollout` object")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the prediction of the last one as DIR/<group>_<name>.npy "
                         "(float32, a fixed sample when over 64 MB; rank 0's, i.e. its latitude band when sharded)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 1:
        args.warmup = 1

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import aurora_b200 as ab
    from aurora_b200 import cabi

    from aurora_b200 import dist as abd
    import torch.distributed as dist

    rank, world, local_rank = abd.env_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = abd.init_process_group("nccl", dev)

    cls, h, w, levels = WORKLOADS[args.workload]
    model = getattr(ab, cls)(_init="empty", autocast=True).to(dev).eval()
    randomise_parameters_(model, seed=rank)
    cfg = model.config
    host_batch = make_host_batch(cfg, h, w, levels, pinned=True, seed=rank)
    dev_batch = host_batch.to(dev)
    h2d_bytes = sum(v.numel() * 4 for d in (host_batch.surf_vars, host_batch.static_vars, host_batch.atmos_vars)
                    for v in d.values())

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    latshard = distributed and resolve_parallelism(args.workload, world, args.parallelism) == "latshard"
    if args.cuda_graph is None:
        args.cuda_graph = latshard
    model.use_cuda_graph = bool(args.cuda_graph)
    plain_forward = model.forward
    if latshard:
        model.halo_mode = args.halo
        model.forward = lambda b: plain_forward(b, sharded=True)  # noqa: E731

    # ---- warm-up (packs weights, allocates workspace, caches encodings) ----
    for _ in range(args.warmup):
        pred = model.forward(dev_batch)
    d2h_bytes = sum(v.numel() * 4 for d in (pred.surf_vars, pred.atmos_vars) for v in d.values())
    if latshard:  # every rank uploads only its own latitude band of the (cropped) fields
        band_rows = next(iter(pred.surf_vars.values())).shape[-2]
        h2d_bytes = h2d_bytes // h * band_rows
    host_out = {k: torch.empty(v.shape, dtype=torch.float32, pin_memory=True)
                for d in (pred.surf_vars, pred.atmos_vars) for k, v in d.items()}

    # ---- device-resident throughput ----
    barrier()
    launches0 = cabi.launch_count()
    replayed0 = model._engine.replayed_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clk = ClockSampler(local_rank)   # samples through BOTH timed regions (device-resident and end-to-end)
    clk.__enter__()
    e0.record()
    for _ in range(args.steps):
        pred = model.forward(dev_batch)
    e1.record()
    barrier()
    # kernels launched by this library in the timed region: eager launches + those replayed from captured graphs
    launches = (cabi.launch_count() - launches0) + (model._engine.replayed_launches - replayed0)
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(pred, args.dump_outputs)

    # ---- end to end through the public API from pinned host memory ----
    e2e_ms = None
    if not args.no_e2e:
        d2h_stream = torch.cuda.Stream(device=dev)

        def e2e_step():
            p = model.forward(host_batch)     # the public call on HOST tensors: H2D of every field happens inside
                                              # (pinned source -> copy stream, overlaps the previous step's kernels)
            # D2H of the whole prediction into pinned host buffers, like a consumer that streams results out: on its own
            # stream behind an event, so that the read-back of step n runs under the kernels of step n + 1 (the
            # predictions are fresh tensors every step; record_stream keeps the allocator from recycling them early)
            done = torch.cuda.Event()
            done.record()
            d2h_stream.wait_event(done)
            with torch.cuda.stream(d2h_stream):
                for grp in (p.surf_vars, p.atmos_vars):
                    for k, v in grp.items():
                        host_out[k].copy_(v, non_blocking=True)
                        v.record_stream(d2h_stream)
            return p
        e2e_step()
        barrier()
        e0.record()
        for _ in range(args.steps):
            e2e_step()
        e1.record()
        barrier()
        e2e_ms = e0.elapsed_time(e1) / args.steps
    clk.__exit__()
    clocks = clk.summary()

    # ---- autoregressive rollout (rollout.py:14-49): state stays on the device, every prediction is yielded ----
    rollout_info = None
    if args.rollout > 0 and not latshard:
        def run_rollout(n):
            last = None
            for p in ab.rollout(model, host_batch, steps=n):   # initial H2D inside; the caller keeps only the last step
                last = p
            return last
        # warm-up: steps 0, 1 and >= 2 have different graph signatures (the positive-variable clamp starts at step 2,
        # `from_second` LoRA at step 1): three steps capture every graph a long roll-out replays
        run_rollout(min(args.rollout, 3))
        barrier()
        e0.record()
        run_rollout(args.rollout)
        e1.record()
        barrier()
        r_ms = e0.elapsed_time(e1)
        rollout_info = {"steps": args.rollout, "ms_total": r_ms, "ms_per_step": r_ms / args.rollout,
                        "value": world * 1000.0 * args.rollout / r_ms, "unit": "forecast-steps/s",
                        "note": "aurora_b200.rollout from a pinned host batch; history slide and predictions on the device"}

    # ---- N > 1, sharded: the same box running N independent forecasts instead (secondary number) ----
    replicas_info = None
    if latshard:
        model.use_cuda_graph = False
        k = max(2, args.steps // 2)
        plain_forward(dev_batch)
        barrier()
        e0.record()
        for _ in range(k):
            plain_forward(dev_batch)
        e1.record()
        barrier()
        r_ms = abd.max_over_ranks([e0.elapsed_time(e1) / k], device=dev)[0]
        replicas_info = {"value": world * 1000.0 / r_ms, "unit": "forecast-steps/s", "ms_per_step": r_ms, "steps": k,
                         "note": f"{world} independent forecasts, one per GPU, no data-path collective (weak scaling)"}
        model.use_cuda_graph = bool(args.cuda_graph)

    # ---- per-kernel timing for the roofline (one instrumented step; CUDA events around each launch) ----
    cabi.PROFILE = {}
    model.use_cuda_graph = False
    model.forward(dev_batch)
    torch.cuda.synchronize()
    prof = cabi.PROFILE
    cabi.PROFILE = None
    pk = peaks()

    def agg(name):
        rows = prof.get(name, [])
        t = sum(a.elapsed_time(b) for a, b, _, _ in rows) / 1e3
        return len(rows), t, sum(r[2] for r in rows), sum(r[3] for r in rows)

    n_g, t_g, f_g, b_g = agg("gemm")
    n_a, t_a, f_a, b_a = agg("window_attention")
    n_l, t_l, _, b_l = agg("ln_mod_residual")
    n_hp, t_hp, _, b_hp = agg("halo_push")
    n_hw, t_hw, _, _ = agg("halo_wait")
    peak_tf = pk["bf16_tflops_sustained"] or pk["bf16_tflops"]
    roofline = {
        "kernel": "gemm_bf16_tn_kernel (tcgen05)", "bound": "tensor",
        "achieved": f_g / t_g / 1e12 if t_g else None, "peak": peak_tf, "unit": "TFLOP/s",
        "frac": (f_g / t_g / 1e12) / peak_tf if t_g else None,
        **gemm_traffic(args.workload, n_g, b_g),
        "peak_source": pk["source"] + " (sustained figure: kernel timed inside a long step)",
        "launches_per_step": n_g, "seconds_per_step": t_g, "share_of_step": t_g / (ms / 1e3),
        "others": {
            "window_attention": {
                "bound": "hbm", "launches_per_step": n_a, "seconds_per_step": t_a, "share_of_step": t_a / (ms / 1e3),
                "achieved_gbs": b_a / t_a / 1e9 if t_a else None, "hbm_peak_gbs": pk["hbm_gbs"],
                "frac_hbm": (b_a / t_a / 1e9) / pk["hbm_gbs"] if t_a else None,
                "achieved_tflops": f_a / t_a / 1e12 if t_a else None,
                "frac_tensor": (f_a / t_a / 1e12) / pk["bf16_tflops"] if t_a else None,
                # stand-alone roofline of this kernel: min(tensor peak, HBM peak x 72 FLOP/B) (SURVEY 8d)
                "standalone_roofline_tflops": min(pk["bf16_tflops"], pk["hbm_gbs"] * (f_a / b_a) / 1e3) if b_a else None,
                "frac_standalone_roofline": ((f_a / t_a / 1e12) / min(pk["bf16_tflops"], pk["hbm_gbs"] * (f_a / b_a) / 1e3)
                                             if t_a and b_a else None),
            },
            "ln_mod_residual": {
                "bound": "hbm", "launches_per_step": n_l, "seconds_per_step": t_l, "share_of_step": t_l / (ms / 1e3),
                "achieved_gbs": b_l / t_l / 1e9 if t_l else None,
                "frac_hbm": (b_l / t_l / 1e9) / pk["hbm_gbs"] if t_l else None,
            },
        },
    }
    if n_hp:
        roofline["others"]["halo_exchange"] = {
            "bound": "nvlink", "exchanges_per_step": n_hp, "push_seconds_per_step": t_hp,
            "push_achieved_gbs": b_hp / t_hp / 1e9 if t_hp else None, "nvlink_peak_gbs_per_direction": 900.0,
            "bytes_sent_per_exchange": b_hp / n_hp, "wait_seconds_per_step": t_hw,
            "note": "rank 0, one eager instrumented step: push = stores into both neighbours' memory over NVLink; the wait "
                    "for the neighbours' rows happens inside the attention kernel (its loaders spin on the flags before the "
                    "first foreign row), so it is part of window_attention's time; wait_seconds_per_step is the stand-alone "
                    "wait kernel, no longer launched"}

    # ---- max over ranks (times); bytes moved are summed over ranks for a sharded forecast ----
    if distributed:
        mx = abd.max_over_ranks([ms, e2e_ms or 0.0], device=dev)
        ms, e2e_ms = mx[0], (mx[1] if e2e_ms is not None else None)
        if latshard:
            t = torch.tensor([float(h2d_bytes), float(d2h_bytes)], dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            h2d_bytes, d2h_bytes = int(t[0].item()), int(t[1].item())

    if rank == 0:
        cpu = gpu_ref = None
        if world == 1 and not args.no_gpu_reference:
            from oracle import ref as _ref

            if _ref.available():
                gpu_ref = gpu_reference_measure(args.workload, dev_batch, dev)
                if "fp32" in gpu_ref and "ms_per_step" in gpu_ref["fp32"]:
                    for tag in ("fp32", "autocast_bf16"):
                        if "ms_per_step" in gpu_ref.get(tag, {}):
                            gpu_ref[tag]["ours_over_reference"] = gpu_ref[tag]["ms_per_step"] / ms
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_measure(args.workload, 1, 3)
            cpu.pop("_times", None)
        algo_tflop = ALGO_TFLOP[args.workload]
        line = {
            "metric": "forecast-steps/sec", "value": (1 if latshard else world) * 1000.0 / ms, "unit": "forecast-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong" if latshard else "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args.workload, world, args.parallelism),
            "details": {
                "parameters_m": round(sum(p.numel() for p in model.parameters()) / 1e6, 1),
                "precision": "bf16 operands in the Swin backbone, fp16 operands in encoder/decoder, fp32 accumulate/"
                             "residual/LN/softmax",
                "parallelism": ((f"one forecast latitude-sharded over {world} GPUs, halo exchange per Swin block "
                                 f"({'peer-memory kernels over NVLink inside the CUDA graph' if args.halo == 'peer' else 'NCCL send/recv'})")
                                if latshard else f"replicas x{world}") if world > 1 else "single GPU",
                "cuda_graph": bool(args.cuda_graph),
            },
            "model_tflops_achieved": algo_tflop / (ms / 1e3),
            "clocks": clocks,
            "gpu_launches": launches,
            "e2e": None if e2e_ms is None else {
                "value": (1 if latshard else world) * 1000.0 / e2e_ms, "unit": "forecast-steps/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": h2d_bytes * (1 if latshard else world),
                "d2h_bytes_per_step": d2h_bytes * (1 if latshard else world),
            },
            "roofline": roofline,
            "cpu_baseline": cpu,
            "gpu_reference": gpu_ref,
        }
        if replicas_info is not None:
            line["replicas"] = replicas_info
        if rollout_info is not None:
            if distributed:
                rollout_info["note"] += " (rank 0's time)"
            line["rollout"] = rollout_info
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
