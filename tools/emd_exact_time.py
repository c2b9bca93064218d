"""Timing of the exact EMD kernel (csrc/emd_exact.cu), against scipy's assignment on the host CPU.
Usage: python tools/emd_exact_time.py [--window 1.0] [--scipy-pairs 16]

Workloads (Gaussian clouds, the second set scaled by 0.9 and shifted by 0.05):
  (a) 1024 PAIRED pairs of 2048 points;
  (b) the three matrices of sample_metrics(distance="emd_exact") at 128 + 128 clouds of 2048 points: two SELF launches
      (8128 pairs each) and one ALL launch (16384 pairs);
  (c) 64 PAIRED pairs of 4096 points.
Reports, in one run on one GPU:
  - the card name and its power limit (nvidia-smi query);
  - per workload: gecco_emd_exact alone (inputs cast and every output allocated once, outside the window): one warm-up
    call, then calls repeated over a window of at least --window seconds; ms per call and cloud pairs/s;
  - scipy's cdist + linear_sum_assignment (float64, one thread of the host CPU) on the first --scipy-pairs pairs of (a):
    pairs/s, the CPU model, and the largest relative difference between the kernel's value and scipy's.
Writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import platform
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from chamfer_time import _events_ms, card_info  # noqa: E402


def _cpu_model() -> str:
    try:
        for line in Path("/proc/cpuinfo").read_text().splitlines():
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor() or "unknown"


def _window(fn, window_s: float) -> dict:
    """One warm-up call (timed), then ceil(window_s / its time) calls in one timed window."""
    first = _events_ms(fn, 1)[0]
    reps = max(1, math.ceil(window_s * 1e3 / max(first, 1e-3)))

    def loop():
        for _ in range(reps):
            fn()

    ms = _events_ms(loop, 1)[0]
    return {"warmup_ms": round(first, 2), "reps": reps, "window_ms": round(ms, 1), "ms_per_call": ms / reps}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--scipy-pairs", type=int, default=16)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("emd_exact_time: needs a CUDA device")

    from gecco_b200 import _abi
    from gecco_b200.ops import _lib_for, _stream
    from oracle import emd_exact_oracle as XO

    res = {"card": card_info()}
    g = torch.Generator(device="cuda").manual_seed(0)

    def clouds(m, n):
        return torch.randn(m, n, 3, device="cuda", generator=g)

    def launcher(a, b, mode, out, lower=None, match=None):
        lib = _lib_for(a)
        ea = _abi.EmdExactArgs()
        ea.a, ea.ma, ea.na = a.data_ptr(), a.shape[0], a.shape[1]
        if b is not None:
            ea.b, ea.mb, ea.nb = b.data_ptr(), b.shape[0], b.shape[1]
        ea.mode, ea.out = mode, out.data_ptr()
        ea.lower = lower.data_ptr() if lower is not None else None
        ea.match = match.data_ptr() if match is not None else None
        stream = _stream(a)
        return lambda: _abi.check(lib.gecco_emd_exact(C.byref(ea), stream))

    # (a), (c): PAIRED with lower bound and permutation
    for name, (pairs, n) in {"a": (1024, 2048), "c": (64, 4096)}.items():
        x, y = clouds(pairs, n), clouds(pairs, n) * 0.9 + 0.05
        out, lower = torch.empty(pairs, device="cuda"), torch.empty(pairs, device="cuda")
        match = torch.empty(pairs, n, device="cuda", dtype=torch.int32)
        t = _window(launcher(x, y, _abi.CHAMFER_PAIRED, out, lower, match), args.window)
        gap = ((out - lower) / out).max().item()
        res[name] = dict(t, pairs=pairs, points=n, pairs_per_s=pairs / (t["ms_per_call"] * 1e-3),
                         nan_pairs=int(torch.isnan(out).sum()), max_certified_rel_gap=gap)
        if name == "a":
            k = args.scipy_pairs
            xs, ys = x[:k].double().cpu().numpy(), y[:k].double().cpu().numpy()
            t0 = time.perf_counter()
            want = np.array([XO.lsa(xs[i], ys[i])[0] for i in range(k)])
            dt = time.perf_counter() - t0
            got = out[:k].double().cpu().numpy()
            res["scipy_host"] = {"pairs": k, "points": n, "s": dt, "pairs_per_s": k / dt, "cpu": _cpu_model(),
                                 "max_rel_diff_kernel_vs_scipy": float(np.abs(got - want).max() / want.min())}
        del x, y, out, lower, match
        torch.cuda.empty_cache()

    # (b): the three matrices of sample_metrics(distance="emd_exact")
    m, n = 128, 2048
    s_g, s_r = clouds(m, n), clouds(m, n) * 0.9 + 0.05
    d_gg, d_rr, d_gr = (torch.empty(m, m, device="cuda") for _ in range(3))
    calls = [launcher(s_g, None, _abi.CHAMFER_SELF, d_gg), launcher(s_r, None, _abi.CHAMFER_SELF, d_rr),
             launcher(s_g, s_r, _abi.CHAMFER_ALL, d_gr)]
    pairs = 2 * m * (m - 1) // 2 + m * m
    t = _window(lambda: [c() for c in calls], args.window)
    res["b"] = dict(t, clouds=f"{m} + {m}", points=n, pairs=pairs, pairs_per_s=pairs / (t["ms_per_call"] * 1e-3),
                    nan_entries=int(sum(torch.isnan(d).sum() for d in (d_gg, d_rr, d_gr))))
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()
