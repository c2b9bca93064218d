#!/usr/bin/env python
"""Benchmark of the gecco sampling hot path (BASELINE.json: point clouds/sec, 2048 points, full EDM sampler).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config {1,2,3,4}] [--impl {b200,reference,reference-cuda}]
                    [--dump-outputs DIR]

Workloads (BASELINE.json `configs`, SURVEY.md §8d); `--config 2` is the default and the N = 1 headline:
  1  ShapeNet-PointFlow unconditional: LinearLift + GaussianReparam, 4 clouds per GPU (the reference's CPU-runnable case)
  2  ShapeNet-vol image-conditional: RayNetwork + GaussianReparam, ConvNeXt-T conditioner, 3x137x137 images, 64 clouds per GPU
  3  Taskonomy-style conditional: RayNetwork + UVLReparam, 3x256x256 images, 64 clouds per GPU (the multi-GPU config)
  4  conditional upsampling 2048 -> 16384 points (config-3 model, 5 substeps), 8 clouds per GPU
One "step" = one `Diffusion.sample_stochastic` (configs 1-3) or `Diffusion.upsample` (config 4) call on the batch:
conditioner once + 64 stochastic EDM steps (127 denoiser evaluations; config 4: 64 full + 635 cached evaluations).

Own arm: `value` has the context resident in HBM; `e2e` starts from pinned host images / cameras and ends with the
sampled clouds back on the host.  Under torchrun every rank samples its own clouds (weak scaling, no data-path
collective) and the per-rank results are all-gathered INSIDE the timed region (the "final gather" of north_star);
time = max over ranks.  `roofline` is quoted on the kernel class with the largest share of the step, timed with CUDA
events on the launching stream by the engine's per-kernel-class profiler.
`--impl reference`: the CPU restatement of the reference (oracle/gecco_oracle.py; the Python reference itself cannot
travel to the GPU box) on the host cores, on a bounded sample of the same workload.
`--impl reference-cuda`: the same restatement as plain PyTorch eager on the B200 (cuBLAS / SDPA / native group-norm and
grid-sampler kernels), fp32 and bf16 autocast: the library path a gecco-torch user has today (BASELINE.md §4).
`--dump-outputs DIR`: the result of the last timed step, `samples.npy` (configs 1-4, float64 data-space clouds) or
`loss.npy` + `parameters.npy` (config 5, the updated flat fp32 weights, sampled to fit 64 MB).  Inputs and weights are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

POINTS = 2048
NUM_STEPS = 64
EVALS = 2 * NUM_STEPS - 1
C_, I_, L_, CTX_ = 384, 64, 6, 672
# algorithmic FLOPs of one denoiser evaluation per cloud (BASELINE.md §3)
FLOP_UNCOND = L_ * (16 * POINTS * C_ * C_ + 8 * POINTS * I_ * C_ + 14 * I_ * C_ * C_) + 4 * 3 * POINTS * C_       # 32.209 G
FLOP_COND = FLOP_UNCOND + 2 * POINTS * CTX_ * C_                                                                   # 33.266 G
UPS_N, UPS_SUBSTEPS = 16384, 5
FLOP_CACHED_16K = L_ * (12 * UPS_N * C_ * C_ + 4 * UPS_N * I_ * C_ + 4 * I_ * C_ * C_) + 2 * UPS_N * CTX_ * C_ + 4 * 3 * UPS_N * C_

CONFIGS = {
    1: dict(name="ShapeNet-PointFlow unconditional (LinearLift+SetTransformer L6 C384 I64 H8, GaussianReparam)", kind="uncond",
            reparam="gaussian", mean=[0.0, 0.01, 0.05], sigma=[0.11, 0.04, 0.17], sigma_max=165.0, clouds=4, image=None, K=None,
            flop_per_cloud=EVALS * FLOP_UNCOND),
    2: dict(name="ShapeNet-vol image-conditional (RayNetwork+SetTransformer L6 C384 I64 H8, GaussianReparam, ConvNeXt-T conditioner)",
            kind="cond", reparam="gaussian", mean=[0.0, 0.0, 1.0], sigma=[0.15, 0.15, 0.15], sigma_max=165.0, clouds=64, image=137,
            K=[[1.0859, 0.0, 0.4964], [0.0, 1.0859, 0.4964], [0.0, 0.0, 1.0]], flop_per_cloud=EVALS * FLOP_COND),
    3: dict(name="Taskonomy-style conditional (RayNetwork+SetTransformer L6 C384 I64 H8, UVLReparam, ConvNeXt-T conditioner)",
            kind="cond", reparam="uvl", mean=[0.0, 0.0, 1.38], sigma=[0.56, 0.60, 0.49], sigma_max=180.0, clouds=64, image=256,
            K=[[1.2, 0.0, 0.5], [0.0, 1.2, 0.5], [0.0, 0.0, 1.0]], flop_per_cloud=EVALS * FLOP_COND),
    4: dict(name="conditional upsampling 2048 -> 16384 points (config-3 model, 5 substeps, cached inducer states)",
            kind="cond", reparam="uvl", mean=[0.0, 0.0, 1.38], sigma=[0.56, 0.60, 0.49], sigma_max=180.0, clouds=8, image=256,
            K=[[1.2, 0.0, 0.5], [0.0, 1.2, 0.5], [0.0, 0.0, 1.0]],
            flop_per_cloud=NUM_STEPS * FLOP_COND + (NUM_STEPS * UPS_SUBSTEPS * 2 - UPS_SUBSTEPS) * FLOP_CACHED_16K),
    5: dict(name="EDM training step (denoising loss, forward + backward, gradient all-reduce, fused Adam + EMA) on the config-2 model",
            kind="cond", reparam="gaussian", mean=[0.0, 0.0, 1.0], sigma=[0.15, 0.15, 0.15], sigma_max=165.0, clouds=32, image=137,
            K=[[1.0859, 0.0, 0.4964], [0.0, 1.0859, 0.4964], [0.0, 0.0, 1.0]], flop_per_cloud=3 * FLOP_COND),
}


def workload_text(c: dict, clouds: int) -> str:
    img = "" if c["image"] is None else f", synthetic 3x{c['image']}x{c['image']} images + cameras"
    if c is CONFIGS[5]:
        return (f"{c['name']}, {POINTS} points{img}, {clouds} clouds per GPU and step, bf16 GEMM operands / fp32 accumulation, "
                f"master weights and optimiser state, random-init weights")
    if c is CONFIGS[4]:
        return (f"{c['name']}{img}, {clouds} clouds per GPU, {NUM_STEPS} steps x {UPS_SUBSTEPS} substeps "
                f"({NUM_STEPS} full + {NUM_STEPS * UPS_SUBSTEPS * 2 - UPS_SUBSTEPS} cached evaluations), random-init weights")
    return (f"{c['name']}, {POINTS} points{img}, {clouds} clouds per GPU, {NUM_STEPS}-step stochastic EDM sampler "
            f"({EVALS} denoiser evaluations), random-init weights")


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return dict(hbm=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


DUMP_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict) -> None:
    """Writes every array as <directory>/<name>.npy, float64 kept and anything else as float32, DUMP_BYTES in all.  An
    array over its equal share keeps a fixed, seeded sample of its rows (dim 0, in order), so that two builds run with
    the same arguments write the same positions and can be compared output for output."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096  # room for the .npy header
    for name, t in arrays.items():
        t = t.detach().cpu().reshape(t.shape if t.dim() else (1,))
        t = t if t.dtype == torch.float64 else t.float()
        rows = max(1, share // (t[0].numel() * t.element_size()))
        if rows < t.shape[0]:
            t = t[torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values]
        np.save(os.path.join(directory, name + ".npy"), t.numpy())


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ own arm
def build_model(device, cfg: dict | None = None):
    import gecco_b200 as G
    from gecco_b200.models import ConvNeXtExtractor, GaussianActivation, LinearLift, RayNetwork, SetTransformer
    from gecco_b200.reparam import GaussianReparam, UVLReparam

    c = cfg or CONFIGS[2]
    torch.manual_seed(0)
    m, s = torch.tensor(c["mean"]), torch.tensor(c["sigma"])
    rp = GaussianReparam(m, s) if c["reparam"] == "gaussian" else UVLReparam(m, s)
    st = SetTransformer(n_layers=L_, num_inducers=I_, feature_dim=C_, t_embed_dim=1, num_heads=8, activation=GaussianActivation)
    if c["kind"] == "uncond":
        net, cond = LinearLift(inner=st, feature_dim=C_), G.IdleConditioner()
    else:
        net, cond = RayNetwork(backbone=st, reparam=rp, context_dims=(96, 192, 384)), ConvNeXtExtractor(pretrained=False)
    model = G.Diffusion(backbone=G.EDMPrecond(model=net), conditioner=cond, reparam=rp,
                        loss=G.EDMLoss(schedule=G.LogUniformSchedule(max=c["sigma_max"])))
    return model.to(device).eval()


# which roofline binds a kernel class: the one that gives the larger minimum time for its algorithmic work
def class_roofline(p: dict, pk: dict) -> dict:
    t = p["ms"] * 1e-3
    tf = p["flops"] / t / 1e12 if t > 0 else 0.0
    gbs = p["bytes"] / t / 1e9 if t > 0 else 0.0
    tensor_bound = p["flops"] / (pk["tf_sustained"] * 1e12) >= p["bytes"] / (pk["hbm"] * 1e9)
    if tensor_bound:
        return dict(bound="tensor", achieved=tf, peak=pk["tf_sustained"], unit="TFLOP/s", frac=tf / pk["tf_sustained"],
                    other={"hbm_gbs": gbs, "hbm_frac": gbs / pk["hbm"]})
    return dict(bound="hbm", achieved=gbs, peak=pk["hbm"], unit="GB/s", frac=gbs / pk["hbm"],
                other={"tensor_tflops": tf, "tensor_frac": tf / pk["tf_sustained"]})


KERNEL_OF_CLASS = {
    "gemm_kv_q": "gemm_pair_kernel (tcgen05 cta_group::2): k|v|q projection, M = clouds*2048, N = 1152, K = 384",
    "gemm_mlp_up_act": "gemm_pair_kernel (tcgen05 cta_group::2): MLP up-projection + Gaussian activation, N = 768, K = 384",
    "gemm_mlp_down": "gemm_tc_kernel (tcgen05): MLP down-projection + residual + AdaGN statistics, N = 384, K = 768",
    "gemm_unpool_out": "gemm_pair_kernel (tcgen05 cta_group::2): unpool out-projection + residual + AdaGN statistics, N = 384, K = 384",
    "gemm_img_proj": "gemm_tc_kernel (tcgen05): image-feature projection + xyz embedding, N = 384, K = 672",
    "pool_attention": "pool_tc_kernel (tcgen05): points -> inducers attention core",
    "unpool_attention": "unpool_tc_kernel (tcgen05): inducers -> points attention core",
    "inducer_chain": "inducer-side chain (out_proj, AdaGN, MLP, AdaGN, k/v in-projection)",
    "fold_adagn": "fold_adagn_fast_kernel: AdaGN folded into per-cloud projection weights",
    "mlp_fused": "mlp_pair_kernel (tcgen05 cta_group::2): AdaGN -> GEMM -> Gaussian activation -> GEMM -> + residual, hidden row block parked in L2",
    "lookup": "lookup kernel (projective bilinear gather)", "head_edm_step": "head_kernel: output head + EDM sampler update",
}


def run_own(args):
    import torch.distributed as dist

    import gecco_b200 as G
    from gecco_b200 import engine as E
    from gecco_b200 import parallel as P

    cfg = CONFIGS[args.config]
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    model = build_model(device, cfg)
    B = args.clouds or cfg["clouds"]
    cond = cfg["kind"] == "cond"
    g = torch.Generator("cpu").manual_seed(123 + rank)
    images_h = K_h = ctx_d = None
    if cond:
        images_h = torch.rand(B, 3, cfg["image"], cfg["image"], generator=g).pin_memory()
        K_h = torch.tensor(cfg["K"]).expand(B, 3, 3).contiguous().pin_memory()
        ctx_d = G.Context3d(image=images_h.to(device), K=K_h.to(device))
    n_out = UPS_N if args.config == 4 else POINTS
    out_h = torch.empty(B, n_out, 3, dtype=torch.float64).pin_memory()
    rng = torch.Generator(device).manual_seed(42 + rank)
    seed_h = seed_d = None
    if args.config == 4:  # in-frustum seed cloud (SURVEY.md §8d): diffusion-space normal draws mapped to data space
        seed_d = model.reparam.diffusion_to_data(torch.randn(B, POINTS, 3, generator=g).to(device), ctx_d).float()
        seed_h = seed_d.cpu().pin_memory()

    def call(ctx, seed):
        if args.config == 4:
            return model.upsample(seed, n_new=UPS_N, context=ctx, num_substeps=UPS_SUBSTEPS, rng=rng)
        return model.sample_stochastic((B, POINTS, 3), ctx, rng=rng)

    def finish(out):
        return P.gather_clouds(out) if world > 1 else out  # the only collective of sampling (north_star "final gather")

    def step_resident():
        return finish(call(ctx_d, seed_d))

    def step_e2e():
        ctx = None
        if cond:
            ctx = G.Context3d(image=images_h.to(device, non_blocking=True), K=K_h.to(device, non_blocking=True))
        seed = None if seed_h is None else seed_h.to(device, non_blocking=True)
        out = call(ctx, seed)
        out_h.copy_(out, non_blocking=True)
        return finish(out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return ms.item(), out

    for _ in range(args.warmup):
        out = step_resident()
    assert torch.isfinite(out).all() or args.config in (3, 4), "non-finite samples"  # random-init UVL saturates tanh/exp
    eng = E.engine_for(*model._network())
    clocks = ClockSampler(local) if rank == 0 else None
    E.launch_count(reset=True)
    ms, out = timed(step_resident, args.steps)
    launches = E.launch_count(reset=True)
    graph_status = eng.graph_status()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"samples": out})
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    clk = clocks.stop() if clocks else None

    # host time to enqueue one step (no synchronisation inside): if it approaches ms_per_step the run is launch-bound
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step_resident()
    host_ms = (time.perf_counter() - t0) * 1e3
    torch.cuda.synchronize()

    # per-kernel-class device time of one more step, CUDA events on the launching stream (eager launches: a graph
    # replay cannot carry per-launch events)
    E.profile_start()
    step_resident()
    prof = E.profile_stop()
    total_prof_ms = sum(p["ms"] for p in prof)
    gemm = [p for p in prof if p["name"].startswith("gemm_") or p["name"].endswith("_fused")]
    gemm_ms, gemm_flops = sum(p["ms"] for p in gemm), sum(p["flops"] for p in gemm)
    pk = peaks()
    dom = max(prof, key=lambda p: p["ms"])  # the kernel class with the largest share of the step
    look = next((p for p in prof if p["name"] == "lookup"), None)

    if rank == 0:
        clouds = world * B * args.steps
        value = clouds / (ms * 1e-3)
        traffic = {}
        tfile = ROOT / "profiles" / "roofline_traffic.json"
        if tfile.exists():
            traffic = json.loads(tfile.read_text())
        roof = class_roofline(dom, pk)
        whole_tf = B * cfg["flop_per_cloud"] * args.steps / (ms * 1e-3) / 1e12
        line = {
            "metric": "point clouds/sec (2048 pts, full EDM sampler)", "value": value, "unit": "clouds/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_text(cfg, B), "baseline_config": args.config, "clouds_per_gpu": B, "points": n_out,
                       "num_steps": NUM_STEPS,
                       "l2": "no flush needed: every evaluation streams a >600 MB working set per GPU (L2 is 126 MB)"
                             if B >= 16 else "small batch: the working set of one evaluation fits L2 (as it does in production use of this config)",
                       "parallelism": f"dp{world} (independent clouds, no data-path collective"
                                      + (", final all-gather of the samples inside the timed region)" if world > 1 else ")")},
            "e2e": {"value": clouds / (ms_e2e * 1e-3), "unit": "clouds/s",
                    "h2d_bytes_per_step": (0 if images_h is None else images_h.numel() * 4 + K_h.numel() * 4)
                                          + (0 if seed_h is None else seed_h.numel() * 4),
                    "d2h_bytes_per_step": out_h.numel() * 8},
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_ms,
            "cuda_graph": {0: "off (eager launches)", 1: "captured", 2: "replayed", -1: "capture failed: eager"}.get(graph_status, graph_status),
            "clocks": clk,
            "roofline": {**{k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac")},
                         "traffic": traffic.get(dom["name"] + "_dram_bytes_per_launch"),
                         "kernel_class": dom["name"], "kernel": KERNEL_OF_CLASS.get(dom["name"], dom["name"]),
                         "algorithmic": "FLOPs 2*M*N*K (+ attention 4*M*I*C) and compulsory HBM bytes per launch as listed in DESIGN.md §4",
                         "other_roofline": roof["other"],
                         "launches_timed": dom["launches"], "us_per_launch": dom["ms"] * 1e3 / dom["launches"],
                         "share_of_step": dom["ms"] / total_prof_ms if total_prof_ms else None,
                         "all_tcgen05_gemms": {"tflops": gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None,
                                               "frac_of_tensor_peak": gemm_flops / (gemm_ms * 1e-3) / 1e12 / pk["tf_sustained"] if gemm_ms else None,
                                               "share_of_step": gemm_ms / total_prof_ms if total_prof_ms else None},
                         "peak_source": pk["source"] + ", sustained bf16 / copy bandwidth (kernel timed inside a long step)",
                         "whole_path_tflops": world * whole_tf,
                         "whole_path_frac_of_tensor_peak": whole_tf / pk["tf_sustained"],
                         "lookup_hbm": None if look is None else {
                             "achieved_gbs": look["bytes"] / (look["ms"] * 1e-3) / 1e9, "peak_gbs": pk["hbm"],
                             "frac": look["bytes"] / (look["ms"] * 1e-3) / 1e9 / pk["hbm"],
                             "kernel": "projective lookup (lookup.cu); algorithmic bytes = pyramid + bf16 output + coordinates per launch",
                             "us_per_launch": look["ms"] * 1e3 / look["launches"],
                             "traffic": traffic.get("lookup_dram_bytes_per_launch")}},
            "kernel_classes": [{"name": p["name"], "launches": p["launches"], "ms": round(p["ms"], 3),
                                "tflops": round(p["flops"] / (p["ms"] * 1e-3) / 1e12, 1) if p["ms"] > 0 else None,
                                "gbs": round(p["bytes"] / (p["ms"] * 1e-3) / 1e9, 1) if p["ms"] > 0 else None} for p in prof],
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = oracle_reference(cfg, budget_s=25.0)
            if args.config != 4:
                try:
                    line["library_baseline"] = oracle_reference_cuda(cfg, device)
                except Exception as exc:  # the library arm is context, never a reason to lose the bench line
                    line["library_baseline"] = {"unavailable": repr(exc)[:200]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ config 5: training step
def run_train(args):
    """BASELINE config 5: one optimisation step = EDM loss forward + backward, bucketed gradient all-reduce (NCCL) overlapped
    with backward, fused Adam + EMA; `value` with the batch resident, `e2e` from pinned host batches to the host loss."""
    import torch.distributed as dist

    import gecco_b200 as G
    from gecco_b200 import training as T

    cfg = CONFIGS[5]
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    model = build_model(device, cfg)
    B = args.clouds or cfg["clouds"]
    g = torch.Generator("cpu").manual_seed(123 + rank)
    images_h = torch.rand(B, 3, cfg["image"], cfg["image"], generator=g).pin_memory()
    K_h = torch.tensor(cfg["K"]).expand(B, 3, 3).contiguous().pin_memory()
    ctx_d = G.Context3d(image=images_h.to(device), K=K_h.to(device))
    data_d = model.reparam.diffusion_to_data(torch.randn(B, POINTS, 3, generator=g).to(device), ctx_d).float()
    data_h = data_d.cpu().pin_memory()
    trainer = T.Trainer(model, lr=1e-4, graph=os.environ.get("GECCO_TRAIN_GRAPH", "1") != "0")
    torch.manual_seed(1 + rank)

    def step_resident():
        return trainer.step((data_d, ctx_d))

    def step_e2e():
        ctx = G.Context3d(image=images_h.to(device, non_blocking=True), K=K_h.to(device, non_blocking=True))
        return trainer.step((data_h.to(device, non_blocking=True), ctx)).item()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return ms.item(), out

    for _ in range(args.warmup):
        loss = step_resident()
    assert torch.isfinite(loss), "non-finite training loss"
    from gecco_b200 import engine as E

    clocks = ClockSampler(local) if rank == 0 else None
    E.launch_count(reset=True)
    ms, loss = timed(step_resident, args.steps)
    launches = E.launch_count(reset=True)
    if trainer.graph_mode:  # the captured forward + backward replays its library kernels without passing the C ABI again
        launches += trainer.graph_library_launches * args.steps
    if args.dump_outputs and rank == 0:  # the step returns the loss; the updated weights are the rest of its result
        dump_outputs(args.dump_outputs, {"loss": loss, "parameters": trainer.state.p})
    ms_e2e, _ = timed(step_e2e, args.steps)
    clk = clocks.stop() if clocks else None
    mem_gb = torch.cuda.max_memory_allocated(device) / 2**30
    # the library arm: the same step with every projection on torch's own kernels (GECCO_TRAIN_TC=0) and the normalisations /
    # activations through torch's own autograd ops (GECCO_TRAIN_FUSED=0)
    lib_ms = None
    if world == 1 and not args.no_cpu_baseline:
        prev_fused = os.environ.get("GECCO_TRAIN_FUSED")
        os.environ["GECCO_TRAIN_TC"] = "0"
        os.environ["GECCO_TRAIN_FUSED"] = "0"
        try:
            lib_trainer = T.Trainer(model, lr=1e-4, graph=trainer.graph_mode)  # its own capture, with the library projections
            step_lib = lambda: lib_trainer.step((data_d, ctx_d))
            for _ in range(2):
                step_lib()
            lib_ms, _ = timed(step_lib, args.steps)
        finally:
            os.environ.pop("GECCO_TRAIN_TC", None)
            os.environ.pop("GECCO_TRAIN_FUSED", None)
            if prev_fused is not None:
                os.environ["GECCO_TRAIN_FUSED"] = prev_fused
    if rank == 0:
        pk = peaks()
        clouds = world * B * args.steps
        tf = B * cfg["flop_per_cloud"] * args.steps / (ms * 1e-3) / 1e12
        line = {
            "metric": "training clouds/sec (2048 pts, EDM loss fwd+bwd, gradient all-reduce, Adam+EMA)", "value": clouds / (ms * 1e-3),
            "unit": "clouds/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_text(cfg, B), "baseline_config": 5, "clouds_per_gpu": B, "points": POINTS,
                       "l2": "no flush needed: one step streams tens of GB of activations per GPU",
                       "precision": "bf16 operands / fp32 accumulate, residual stream, statistics and master weights; the ConvNeXt "
                                    "conditioner under bf16 autocast (the reference trains with precision='16-mixed'), "
                                    "GECCO_TRAIN_COND_AUTOCAST=0 for fp32",
                       "parallelism": f"dp{world} (batch sharded on dim 0; gradient all-reduce in "
                                      f"{len(trainer.reducer.buckets)} buckets overlapped with backward)"},
            "e2e": {"value": clouds / (ms_e2e * 1e-3), "unit": "clouds/s",
                    "h2d_bytes_per_step": images_h.numel() * 4 + K_h.numel() * 4 + data_h.numel() * 4, "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches), "cuda_graph": "replayed" if trainer.graph_mode else "off (eager autograd)", "loss": float(loss), "peak_memory_gb": mem_gb, "clocks": clk,
            "parameters": trainer.state.numel,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": tf / pk["tf_sustained"],
                         "traffic": None, "kernel": "whole training step (3 x the forward FLOPs of BASELINE.md §3 per cloud)",
                         "peak_source": pk["source"]},
            "library_baseline": None if lib_ms is None else {
                "value": clouds / (lib_ms * 1e-3), "unit": "clouds/s", "kind": "the same step with every projection on torch / cuBLAS "
                "kernels (bf16 autocast-equivalent operands), same process", "ms_per_step": lib_ms / args.steps},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ reference arms
def _oracle_setup(cfg: dict, B: int, device="cpu"):
    from oracle import gecco_oracle as O
    from tests import synth
    import torchvision.models as tvm

    ocfg = O.OracleConfig(kind=cfg["kind"], reparam=cfg["reparam"], sigma_max=cfg["sigma_max"])
    sd = {k: v.to(device) for k, v in synth.full_state_dict(cfg["kind"], cfg["reparam"], cfg["mean"], cfg["sigma"], 1234).items()}
    if cfg["kind"] != "cond":
        return O, ocfg, sd, (lambda: None), None
    torch.manual_seed(0)
    feats_net = tvm.convnext_tiny(weights=None).features[:6].eval().to(device)  # stages 0-2 (models/feature_pyramid.py:46-53)
    img = torch.rand(B, 3, cfg["image"], cfg["image"], generator=torch.Generator().manual_seed(123)).to(device)
    K = torch.tensor(cfg["K"]).expand(B, 3, 3).contiguous().to(device)

    def pyramid():
        with torch.no_grad():
            x, out = img, []
            for i in range(0, 6, 2):
                x = feats_net[i + 1](feats_net[i](x))
                out.append(x)
        return out

    return O, ocfg, sd, pyramid, K


def oracle_reference(cfg: dict, budget_s: float, steps: int = 1, warmup: int = 0) -> dict:
    """The oracle restatement of the reference path on the host cores, bounded sample of the bench workload: 4 clouds
    (the batch BASELINE.json states for the reference's CPU-runnable case), sampler shortened to fit the budget."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B = 4 if cfg is not CONFIGS[4] else 1
    O, ocfg, sd, pyramid, K = _oracle_setup(cfg, B)
    feats = pyramid()
    if cfg is CONFIGS[4]:
        seed = O.diffusion_to_data(ocfg, sd, torch.randn(B, POINTS, 3), K)
        t0 = time.perf_counter()
        O.upsample(ocfg, sd, seed, n_new=UPS_N, features=feats, K=K, seed=7, num_substeps=UPS_SUBSTEPS, num_steps=2)
        t = time.perf_counter() - t0
        evals_done = 2 * FLOP_COND + (2 * UPS_SUBSTEPS * 2 - UPS_SUBSTEPS) * FLOP_CACHED_16K
        scale = cfg["flop_per_cloud"] / evals_done
        return {"value": B / (t * scale), "unit": "clouds/s", "cores": cores, "kind": "port", "seconds_per_call": t,
                "sample": f"{B} cloud, 2 of {NUM_STEPS} steps x {UPS_SUBSTEPS} substeps, extrapolated x{scale:.1f} by FLOPs, fp32 torch CPU, {t:.1f} s"}
    x = torch.randn(B, POINTS, 3)
    sg = torch.full((B,), 1.0)
    with torch.no_grad():
        O.denoise(ocfg, sd, x, sg, feats, K)
        t0 = time.perf_counter()
        O.denoise(ocfg, sd, x, sg, feats, K)
        t_eval = time.perf_counter() - t0
    n_steps = NUM_STEPS
    total_calls = steps + warmup
    while n_steps > 2 and total_calls * (2 * n_steps - 1) * t_eval > budget_s:
        n_steps //= 2
    times = []
    for i in range(total_calls):
        t0 = time.perf_counter()
        feats = pyramid()
        O.sample_stochastic(ocfg, sd, (B, POINTS, 3), feats, K, rng=torch.Generator().manual_seed(42), num_steps=n_steps)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    scale = EVALS / (2 * n_steps - 1)  # extrapolation to the full 127 evaluations when the sample was shortened
    return {"value": B / (t * scale), "unit": "clouds/s", "cores": cores, "kind": "port",
            "sample": (f"{B} clouds x {POINTS} points, conditioner + {n_steps}-step sampler ({2 * n_steps - 1} evaluations"
                       + ("" if n_steps == NUM_STEPS else f", extrapolated x{scale:.2f} to {EVALS}") + f"), fp32 torch CPU, {t:.1f} s per call"),
            "seconds_per_call": t}


def oracle_reference_cuda(cfg: dict, device, clouds: int = 16, n_steps: int = 4) -> dict:
    """The same restatement as PyTorch eager ON THE B200 (cuBLAS, SDPA, native group-norm / grid-sampler): the library
    path of a gecco-torch user (BASELINE.md §4).  Bounded sample: `clouds` clouds, an n_steps sampler extrapolated to 127
    evaluations; fp32 (TF32 off, like torch's default) and bf16 autocast (the reference trains / samples in 16-bit)."""
    O, ocfg, sd, pyramid, K = _oracle_setup(cfg, clouds, device)
    scale = EVALS / (2 * n_steps - 1)
    out = {"unit": "clouds/s", "kind": "port on cuda (PyTorch eager, library kernels)",
           "sample": f"{clouds} clouds x {POINTS} points, conditioner + {n_steps}-step sampler, extrapolated x{scale:.1f} to {EVALS} evaluations"}

    def run():
        feats = pyramid()
        return O.sample_stochastic_device(ocfg, sd, (clouds, POINTS, 3), feats, K, device=device, num_steps=n_steps)

    for name, ctxm in (("fp32", torch.autocast("cuda", enabled=False)), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
        with ctxm, torch.no_grad():
            run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            torch.cuda.synchronize()
        out[name] = clouds / (e0.elapsed_time(e1) * 1e-3 * scale)
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    world = int(os.environ.get("WORLD_SIZE", 1))
    common = {"impl": "reference", "metric": "point clouds/sec (2048 pts, full EDM sampler)", "unit": "clouds/s", "n_gpus": world,
              "steps": steps, "warmup": warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic"}
    if args.impl == "reference-cuda":
        lib = oracle_reference_cuda(cfg, torch.device("cuda", 0))
        print(json.dumps({**common, "value": lib["bf16_autocast"], "dtype": "bf16", "library_baseline": lib,
                          "config": {"workload": workload_text(cfg, 16), "baseline_config": args.config,
                                     "note": "restatement of the reference path as PyTorch eager on the B200 (library kernels), bf16 autocast"},
                          "e2e": {"value": lib["bf16_autocast"], "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    base = oracle_reference(cfg, budget_s=150.0, steps=steps, warmup=warmup)
    line = {**common, "value": base["value"], "ms_per_step": base["seconds_per_call"] * 1e3, "dtype": "f32",
            "config": {"workload": workload_text(cfg, args.clouds or cfg["clouds"]), "baseline_config": args.config,
                       "note": "CPU restatement of the reference path (oracle port) on the host cores"},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cuda"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("GECCO_BENCH_CONFIG", "2")), choices=sorted(CONFIGS))
    ap.add_argument("--clouds", type=int, default=0, help="clouds per GPU (default: the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (at most 64 MB "
                         "in all; a larger output is replaced by a fixed, seeded sample of its rows)")
    args = ap.parse_args()
    if args.impl != "b200":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of --impl b200")
        run_reference(args)
        return
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; gecco_b200 has no CPU path (use --impl reference for the CPU baseline)")
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.gpus != world and world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr",
               "127.0.0.1", "--master-port", "29531", __file__, "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup",
               str(args.warmup), "--config", str(args.config), "--clouds", str(args.clouds)] \
            + (["--no-cpu-baseline"] if args.no_cpu_baseline else []) \
            + (["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else [])
        raise SystemExit(subprocess.call(cmd))
    if args.config == 5:
        return run_train(args)
    run_own(args)


if __name__ == "__main__":
    main()
