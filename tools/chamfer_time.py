"""Timing of the Chamfer kernel (csrc/chamfer.cu) on the sample-quality benchmark, with its instruction-issue bound and the
library arm.  Usage: python tools/chamfer_time.py [--gen 1024] [--ref 1024] [--points 2048] [--reps 3] [--lib-pairs 64]

Reports, in one run on one GPU:
  - the card name and its power limit (nvidia-smi query);
  - time, point pairs/s and bytes read for the three matrix launches of sample_metrics (S_g x S_g and S_r x S_r as self
    matrices, each unordered pair once; S_g x S_r all pairs), and sample_metrics end to end;
  - the instruction mix of the kernel's inner loop per lane and point pair (cuobjdump -sass of the built library), the
    issue rates of FFMA2 / FADD2 / FMNMX3 / FFMA measured with micro-kernels compiled by nvcc into a temporary directory,
    and from the two the issue-bound time of the benchmark and the kernel's fraction of it;
  - the library arm: torch.cdist + amin in fp32 on --lib-pairs cloud pairs, extrapolated by pair count.
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

# Per lane and inner-loop step: 8 rows x 2 columns (csrc/chamfer.cu ROWS_PER_LANE, two columns per packed unit).
PAIRS_PER_STEP = 16

MICRO_SRC = r"""
#include <cuda_runtime.h>
__device__ __forceinline__ float min3f(float a, float b, float c) {
  float d; asm volatile("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c)); return d;
}
// 8 independent chains per thread, 8 instructions of the measured kind per loop iteration
__global__ void k_ffma2(float* out, int iters) {
  float2 acc[8]; const float2 b = make_float2(0.999f, 0.998f), c = make_float2(1e-3f, 2e-3f);
  for (int k = 0; k < 8; ++k) acc[k] = make_float2(threadIdx.x * 1e-3f + k, k);
#pragma unroll 16
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = __ffma2_rn(acc[k], b, c);
  float s = 0.f; for (int k = 0; k < 8; ++k) s += acc[k].x + acc[k].y;
  if (s == 12345.f) out[0] = s;
}
__global__ void k_fadd2(float* out, int iters) {
  float2 acc[8]; const float2 b = make_float2(1e-7f, 2e-7f);
  for (int k = 0; k < 8; ++k) acc[k] = make_float2(threadIdx.x * 1e-3f + k, k);
#pragma unroll 16
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = __fadd2_rn(acc[k], b);
  float s = 0.f; for (int k = 0; k < 8; ++k) s += acc[k].x + acc[k].y;
  if (s == 12345.f) out[0] = s;
}
__global__ void k_fmnmx3(float* out, int iters) {
  float acc[8], v[8]; const float y = threadIdx.x * 1e-3f + 0.5f;
  for (int k = 0; k < 8; ++k) acc[k] = 100.f + k, v[k] = threadIdx.x * 1e-3f + k;
#pragma unroll 16
  for (int i = 0; i < iters; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = min3f(acc[k], v[k], y);
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
  if (which == 0) k_ffma2<<<blocks, 256, 0, s>>>(out, iters);
  else if (which == 1) k_fadd2<<<blocks, 256, 0, s>>>(out, iters);
  else if (which == 2) k_fmnmx3<<<blocks, 256, 0, s>>>(out, iters);
  else k_ffma<<<blocks, 256, 0, s>>>(out, iters);
  return (int)cudaGetLastError();
}
"""
MICRO_KINDS = ["FFMA2", "FADD2", "FMNMX3", "FFMA"]


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


def inner_loop_mix(lib_path: Path) -> dict | None:
    """Opcode counts of the chamfer kernel's inner loop (the backward branch whose body holds the FFMA2s), per lane and
    point pair.  None when cuobjdump is missing or the loop is not found."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(tool).exists():
        return None
    sass = subprocess.run([tool, "-sass", str(lib_path)], capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    body = next((f for f in funcs if "chamfer_kernel" in f.split("\n", 1)[0]), None)
    if body is None:
        return None
    ins = []
    for line in body.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(@!?U?P[0-9T]\s+)?([A-Z0-9_]+)(\.[A-Z0-9_.]+)?\s*(.*?);", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(3), m.group(3) + (m.group(4) or ""), m.group(5)))
    best = None
    for addr, op, _, rest in ins:
        t = re.match(r"(0x[0-9a-f]+)", rest.strip())
        if op == "BRA" and t and int(t.group(1), 16) < addr:
            lo = int(t.group(1), 16)
            loop = [x for x in ins if lo <= x[0] <= addr]
            n = sum(1 for x in loop if x[1] == "FFMA2")
            if best is None or n > best[0]:
                best = (n, loop)
    if best is None or best[0] == 0:
        return None
    loop = best[1]
    counts = Counter(x[1] for x in loop if x[1] not in ("NOP",))
    # the loop body holds unroll x 8 x 3 FFMA2 (three per row and step); divergence fall-backs (BRA.DIV targets) are
    # outside it
    steps = counts["FFMA2"] / (3 * 8)
    pairs = steps * PAIRS_PER_STEP
    return {"steps_per_iteration": steps, "pairs_per_iteration": pairs, "instructions": sum(counts.values()),
            "per_pair": {k: v / pairs for k, v in counts.most_common()}}


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
    blocks, iters = sm * 8, 1 << 16
    rates = {}
    for k, name in enumerate(MICRO_KINDS):
        run = lambda: lib.micro_launch(k, C.c_void_p(out.data_ptr()), iters, blocks, stream)
        assert run() == 0
        torch.cuda.synchronize()
        ms = min(_events_ms(run, 5))
        warp_instr = blocks * 8 * iters * 8.0
        rates[name] = warp_instr / (ms * 1e-3)
    return rates


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gen", type=int, default=1024)
    ap.add_argument("--ref", type=int, default=1024)
    ap.add_argument("--points", type=int, default=2048)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lib-pairs", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("chamfer_time: needs a CUDA device")

    from gecco_b200 import _abi
    from gecco_b200.metrics import _launch, chamfer_matrix, sample_metrics

    res = {"card": card_info()}
    mg, mr, n = args.gen, args.ref, args.points
    g = torch.Generator(device="cuda").manual_seed(0)
    gen = torch.randn(mg, n, 3, device="cuda", generator=g)
    ref = torch.randn(mr, n, 3, device="cuda", generator=g) * 0.9 + 0.05
    d_gg = torch.empty(mg, mg, device="cuda")
    d_rr = torch.empty(mr, mr, device="cuda")
    d_gr = torch.empty(mg, mr, device="cuda")

    def three():
        _launch(gen, None, _abi.CHAMFER_SELF, d_gg)
        _launch(ref, None, _abi.CHAMFER_SELF, d_rr)
        _launch(gen, ref, _abi.CHAMFER_ALL, d_gr)

    chamfer_matrix(gen[:8], ref[:8])  # module load, shared-memory attribute
    torch.cuda.synchronize()
    ms = _events_ms(three, args.reps)
    cloud_pairs = mg * (mg - 1) // 2 + mr * (mr - 1) // 2 + mg * mr
    point_pairs = cloud_pairs * n * n
    t = min(ms) * 1e-3
    # each block reads both clouds while staging them and the first cloud once more for its bounding box
    bytes_read = cloud_pairs * 3 * n * 12
    res["benchmark"] = {"gen": mg, "ref": mr, "points": n, "cloud_pairs": cloud_pairs, "point_pairs": point_pairs,
                        "ms": [round(x, 2) for x in ms], "point_pairs_per_s": point_pairs / t,
                        "gb_read_by_blocks": bytes_read / 1e9, "gb_unique_points": (mg + mr) * n * 12 / 1e9}
    ms_e2e = _events_ms(lambda: sample_metrics(gen, ref), 2)
    res["benchmark"]["sample_metrics_e2e_ms"] = [round(x, 2) for x in ms_e2e]

    mix = inner_loop_mix(_abi.lib_path())
    res["inner_loop"] = mix
    with tempfile.TemporaryDirectory() as tmp:
        rates = micro_rates(Path(tmp), res["card"]["sm_count"])
    res["issue_rates_warp_instr_per_s"] = rates
    if mix is not None:
        # per opcode: its measured rate when a micro-kernel covers it, otherwise the FFMA rate (one warp instruction per
        # scheduler and cycle, the issue limit): an optimistic bound
        per_pair_s = sum(cnt / rates.get(op, rates["FFMA"]) for op, cnt in mix["per_pair"].items())
        lane_pairs = point_pairs  # one lane-pair per point pair; a warp instruction covers 32 lanes
        t_bound = lane_pairs / 32 * per_pair_s
        res["issue_bound"] = {"ms": t_bound * 1e3, "fraction_of_bound": t_bound / t,
                              "instr_per_pair": sum(mix["per_pair"].values())}

    # library arm: cdist + amin on a subset of pairs, extrapolated by pair count
    p = min(args.lib_pairs, mg, mr)
    x, y = gen[:p], ref[:p]

    def lib_arm():
        d = torch.cdist(x, y)
        return d.amin(2).pow(2).mean(1) + d.amin(1).pow(2).mean(1)

    lib_arm()
    torch.cuda.synchronize()
    lms = min(_events_ms(lib_arm, 3))
    ours = chamfer_matrix(x, y).diagonal()
    res["library_arm"] = {"pairs_timed": p, "ms": lms, "extrapolated_s": lms * 1e-3 / p * cloud_pairs,
                          "speedup_of_kernel": lms * 1e-3 / p * cloud_pairs / t,
                          "max_rel_diff_vs_kernel": ((lib_arm() - ours).abs() / ours).max().item()}
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()
