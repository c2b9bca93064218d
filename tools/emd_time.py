"""Timing of the approximate EMD kernel (csrc/emd.cu) on the EMD sample-quality benchmark, with its MUFU / issue bound and the
library arm.  Usage: python tools/emd_time.py [--gen 512] [--ref 512] [--points 2048] [--reps 2] [--lib-pairs 64]

The default size is a ShapeNet category's test split under PointFlow's protocol (a few hundred shapes) on both sides:
512 + 512 clouds of 2048 points, 785,408 ordered cloud pairs.  Reports, in one run on one GPU:
  - the card name and its power limit (nvidia-smi query);
  - time of the three launches of sample_metrics(distance="emd") (S_g x S_g and S_r x S_r as ordered self matrices,
    S_r x S_g all pairs) and point-pair evaluations per second (20 O(N^2) sweeps per cloud pair), and sample_metrics end
    to end;
  - the instruction mix of the kernel's five inner loops per lane and point pair (cuobjdump -sass of the built library);
    the issue rates of MUFU.EX2 / MUFU.SQRT / FFMA measured with micro-kernels compiled by nvcc into a temporary
    directory; from the two the bound of every sweep (the larger of its issue time at the FFMA rate and its MUFU time at
    the measured MUFU rates) and the kernel's fraction of the sum;
  - the library arm: the same algorithm as batched fp32 torch on the GPU (torch_approxmatch: one exp and one product
    with the distances over [pairs, N, N] per level, every sum a batched matrix-vector product, no match matrix) on
    --lib-pairs cloud pairs, extrapolated by pair count, with its max relative difference to the kernel.
Writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import re
import shutil
import subprocess
import sys
import tempfile
from collections import Counter
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

# O(N^2) sweeps of one cloud pair per inner-loop kind (csrc/emd.cu): pass 1 of level 7, the fused row sweep of levels 7..0,
# the fused row sweep of level -1, the level-0 row sweep, the column sweeps of levels 7..-1 (level 0's is O(N))
SWEEPS = {"row_first": 1, "row_fused": 8, "row_fused_last": 1, "row_final": 1, "column": 9}

MICRO_SRC = r"""
#include <cuda_runtime.h>
// 8 independent chains per thread, 8 instructions of the measured kind per loop iteration
__global__ void k_ex2(float* out, int iters) {
  float acc[8];
  for (int k = 0; k < 8; ++k) acc[k] = threadIdx.x * 1e-4f + k * 0.1f;
#pragma unroll 16
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(acc[k]) : "f"(-acc[k]));
  float s = 0.f; for (int k = 0; k < 8; ++k) s += acc[k];
  if (s == 12345.f) out[0] = s;
}
__global__ void k_sqrt(float* out, int iters) {
  float acc[8];
  for (int k = 0; k < 8; ++k) acc[k] = threadIdx.x * 1e-3f + k + 2.f;
#pragma unroll 16
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) asm volatile("sqrt.approx.ftz.f32 %0, %1;" : "=f"(acc[k]) : "f"(acc[k]));
  float s = 0.f; for (int k = 0; k < 8; ++k) s += acc[k];
  if (s == 12345.f) out[0] = s;
}
__global__ void k_ffma(float* out, int iters) {
  float acc[8]; const float b = 0.999f, c = 1e-3f;
  for (int k = 0; k < 8; ++k) acc[k] = threadIdx.x * 1e-3f + k;
#pragma unroll 16
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = fmaf(acc[k], b, c);
  float s = 0.f; for (int k = 0; k < 8; ++k) s += acc[k];
  if (s == 12345.f) out[0] = s;
}
extern "C" int micro_launch(int which, float* out, int iters, int blocks, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (which == 0) k_ex2<<<blocks, 256, 0, s>>>(out, iters);
  else if (which == 1) k_sqrt<<<blocks, 256, 0, s>>>(out, iters);
  else k_ffma<<<blocks, 256, 0, s>>>(out, iters);
  return (int)cudaGetLastError();
}
"""
MICRO_KINDS = ["MUFU.EX2", "MUFU.SQRT", "FFMA"]


def card_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0), "sm_count": torch.cuda.get_device_properties(0).multi_processor_count}
    smi = shutil.which("nvidia-smi")
    if smi:
        r = subprocess.run([smi, "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
        info["nvidia_smi"] = r.stdout.strip() or r.stderr.strip()
    else:
        info["nvidia_smi"] = "not available"
    return info


def _events_ms(fn, reps: int) -> list[float]:
    out = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        out.append(s.elapsed_time(e))
    return out


def rows_per_thread(n: int) -> int:
    """The kernel instantiation the launcher picks for n points (csrc/emd.cu: smallest power of two with 256 R >= n)."""
    r = 1
    while r < 16 and 256 * r < n:
        r *= 2
    return r


def inner_loop_mix(lib_path: Path, r: int) -> dict | None:
    """Opcode counts per lane and point pair of the five inner loops of emd_kernel<r> (the innermost backward branches
    whose body holds a MUFU), classified by their MUFU / FMUL / FFMA content.  None when cuobjdump is missing or a loop
    is not found."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(tool).exists():
        return None
    sass = subprocess.run([tool, "-sass", str(lib_path)], capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    body = next((f for f in funcs if f"emd_kernelILi{r}E" in f.split("\n", 1)[0]), None)
    if body is None:
        return None
    ins = []
    for line in body.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(@!?U?P[0-9T]\s+)?([A-Z0-9_]+)(\.[A-Z0-9_.]+)?\s*(.*?);", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(3), m.group(3) + (m.group(4) or ""), m.group(5)))
    loops = []
    for addr, op, _, rest in ins:
        t = re.search(r"(0x[0-9a-f]+)\s*$", rest.strip())  # "BRA 0x..." and "BRA.U UP1, 0x..."
        if op == "BRA" and t and int(t.group(1), 16) < addr:
            loops.append((int(t.group(1), 16), addr))
    mixes = {}
    for lo, hi in loops:
        if any(lo < l2 and h2 < hi for l2, h2 in loops if (l2, h2) != (lo, hi)):
            continue  # not innermost
        c = Counter(x[2] for x in ins if lo <= x[0] <= hi and x[1] != "NOP")
        ex2, sq = c["MUFU.EX2"], c["MUFU.SQRT"]
        if ex2 == 0 and sq == 0:
            continue
        pairs = max(ex2, sq)  # one MUFU of each present kind per point pair
        if ex2 and sq:
            kind = "row_fused" if c["FMUL"] >= 3 * pairs else "row_fused_last"
        elif sq:
            kind = "row_final"
        else:
            kind = "column" if c["FFMA"] >= 2.5 * pairs else "row_first"
        if kind in mixes:  # a remainder copy of the same loop: keep the unrolled one
            if mixes[kind]["pairs_per_iteration"] >= pairs:
                continue
        mixes[kind] = {"pairs_per_iteration": pairs, "instructions": sum(c.values()),
                       "per_pair": {k: v / pairs for k, v in c.most_common()}}
    if set(mixes) != set(SWEEPS):
        return None
    return mixes


def torch_approxmatch(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """EMD(x[i], y[i]) for x, y [p, N, 3], written as a torch user would batch it: d2 from coordinate differences, per
    level one exp and one product with the distances, the five sums as batched matrix-vector products (w is never formed:
    sum_l w[k,l] = ratioL[k] (e ratioR)[k] and sum_l w[k,l] dist[k,l] = ratioL[k] ((e * dist) ratioR)[k])."""
    d2 = (x[:, :, None, :] - y[:, None, :, :]).pow(2).sum(-1)
    dist = d2.sqrt()
    p, n = x.shape[:2]
    rem_l = torch.ones(p, n, device=x.device)
    rem_r = torch.ones(p, n, device=x.device)
    cost = torch.zeros(p, device=x.device)
    mv = lambda m, v: torch.bmm(m, v[:, :, None])[:, :, 0]   # sum over the last index
    vm = lambda v, m: torch.bmm(v[:, None, :], m)[:, 0, :]   # sum over the middle index
    for level in [-(4.0 ** j) for j in range(7, -2, -1)] + [0.0]:
        e = torch.exp(d2 * level)
        ratio_l = rem_l / (1e-9 + mv(e, rem_r))
        sumr = rem_r * vm(ratio_l, e)
        ratio_r = torch.clamp(rem_r / (sumr + 1e-9), max=1.0) * rem_r
        rem_r = (rem_r - sumr).clamp_min(0.0)
        cost += (ratio_l * mv(e * dist, ratio_r)).sum(1)
        rem_l = (rem_l - ratio_l * mv(e, ratio_r)).clamp_min(0.0)
    return cost / n


def micro_rates(tmp: Path, sm: int) -> dict:
    """Issue rate of each micro-kernel in warp instructions per second on the whole GPU."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src, so = tmp / "micro.cu", tmp / "libmicro.so"
    src.write_text(MICRO_SRC)
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared", "-Xcompiler", "-fPIC", "-o",
                    str(so), str(src)], check=True)
    lib = C.CDLL(str(so))
    lib.micro_launch.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    out = torch.zeros(1, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    blocks = sm * 8
    rates = {}
    for k, name in enumerate(MICRO_KINDS):
        iters = 1 << 16 if name == "FFMA" else 1 << 13
        run = lambda: lib.micro_launch(k, C.c_void_p(out.data_ptr()), iters, blocks, stream)
        assert run() == 0
        torch.cuda.synchronize()
        ms = min(_events_ms(run, 5))
        warp_instr = blocks * 8 * iters * 8.0
        rates[name] = warp_instr / (ms * 1e-3)
    return rates


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gen", type=int, default=512)
    ap.add_argument("--ref", type=int, default=512)
    ap.add_argument("--points", type=int, default=2048)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--lib-pairs", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("emd_time: needs a CUDA device")

    from gecco_b200 import _abi
    from gecco_b200.metrics import _launch, emd_matrix, sample_metrics
    torch.backends.cuda.matmul.allow_tf32 = False  # the library arm stays fp32

    res = {"card": card_info()}
    mg, mr, n = args.gen, args.ref, args.points
    g = torch.Generator(device="cuda").manual_seed(0)
    gen = torch.randn(mg, n, 3, device="cuda", generator=g)
    ref = torch.randn(mr, n, 3, device="cuda", generator=g) * 0.9 + 0.05
    d_gg = torch.empty(mg, mg, device="cuda")
    d_rr = torch.empty(mr, mr, device="cuda")
    d_rg = torch.empty(mr, mg, device="cuda")

    def three():
        _launch("gecco_emd", gen, None, _abi.CHAMFER_SELF, d_gg)
        _launch("gecco_emd", ref, None, _abi.CHAMFER_SELF, d_rr)
        _launch("gecco_emd", ref, gen, _abi.CHAMFER_ALL, d_rg)

    emd_matrix(gen[:4], ref[:4])  # module load, shared-memory attribute
    torch.cuda.synchronize()
    ms = _events_ms(three, args.reps)
    cloud_pairs = mg * (mg - 1) + mr * (mr - 1) + mg * mr
    sweeps = sum(SWEEPS.values())
    evaluations = cloud_pairs * n * n * sweeps
    t = min(ms) * 1e-3
    res["benchmark"] = {"gen": mg, "ref": mr, "points": n, "cloud_pairs": cloud_pairs, "sweeps_per_pair": sweeps,
                        "point_pair_evaluations": evaluations, "ms": [round(x, 1) for x in ms],
                        "point_pair_evaluations_per_s": evaluations / t}
    ms_e2e = _events_ms(lambda: sample_metrics(gen, ref, distance="emd"), 1)
    res["benchmark"]["sample_metrics_e2e_ms"] = [round(x, 1) for x in ms_e2e]

    r = rows_per_thread(n)
    mix = inner_loop_mix(_abi.lib_path(), r)
    res["inner_loops"] = {"rows_per_thread": r, "mix": mix}
    with tempfile.TemporaryDirectory() as tmp:
        rates = micro_rates(Path(tmp), res["card"]["sm_count"])
    res["issue_rates_warp_instr_per_s"] = rates
    if mix is not None:
        # per sweep: the larger of (all instructions at the FFMA rate: one warp instruction per scheduler and cycle) and
        # (its MUFU instructions at their measured rates); a warp instruction covers 32 lane-pairs
        per_kind = {}
        total = 0.0
        for kind, count in SWEEPS.items():
            pp = mix[kind]["per_pair"]
            issue = sum(pp.values()) / rates["FFMA"]
            mufu = pp.get("MUFU.EX2", 0.0) / rates["MUFU.EX2"] + pp.get("MUFU.SQRT", 0.0) / rates["MUFU.SQRT"]
            s = cloud_pairs * n * n / 32 * count * max(issue, mufu)
            per_kind[kind] = {"bound_ms": s * 1e3, "bound_by": "issue" if issue >= mufu else "MUFU",
                              "instr_per_pair": sum(pp.values())}
            total += s
        res["bound"] = {"ms": total * 1e3, "fraction_of_bound": total / t, "per_sweep": per_kind}

    # library arm: the three-pass statement in fp32 torch, batched over a subset of pairs, extrapolated by pair count
    p = min(args.lib_pairs, mg, mr)
    x, y = ref[:p], gen[:p]
    lib_arm = lambda: torch_approxmatch(x, y)
    lib_arm()
    torch.cuda.synchronize()
    lms = min(_events_ms(lib_arm, 2))
    ours = emd_matrix(x, y).diagonal()
    res["library_arm"] = {"pairs_timed": p, "ms": lms, "extrapolated_s": lms * 1e-3 / p * cloud_pairs,
                          "speedup_of_kernel": lms * 1e-3 / p * cloud_pairs / t,
                          "max_rel_diff_vs_kernel": ((lib_arm() - ours).abs() / ours).max().item()}
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()
