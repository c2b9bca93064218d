"""Timing of the nearest-neighbour kernel (csrc/nearest.cu) on the conditional-reconstruction workloads, against
gecco_chamfer PAIRED and a torch arm.  Usage: python tools/nearest_time.py [--window 1.0]

Workloads (paired clouds, x -> y and y -> x):
  (a) 64 pairs of 2048 x 2048: config 2's batch of single-view reconstructions against targets of the same size;
  (b) 8 pairs of 16384 x 65536: config 4's upsampled output against a dense stand-in target.
Reports, in one run on one GPU:
  - the card name and its power limit (nvidia-smi query);
  - per workload: time per call of gecco_nearest alone (memset, centre, search, finish; inputs cast and every buffer
    allocated once, outside the window) repeated over a window of at least --window seconds, point pairs/s, the same
    for gecco_chamfer PAIRED (one block per pair, through metrics._launch with a preallocated output) on the same
    clouds, a chunked fp32 torch.cdist + min / argmin arm, and, labelled separately, the Python call
    nearest_neighbours end to end (input checks with a host synchronise, allocations, index widening);
  - the search loop's SASS mix per lane and point pair (cuobjdump of the built library) and the issue-bound time from
    the FFMA2 / FADD2 / FMNMX3 / FFMA issue rates measured by chamfer_time's micro-kernels.
Writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from chamfer_time import _events_ms, card_info, inner_loop_mix, micro_rates  # noqa: E402

WORKLOADS = {"a": (64, 2048, 2048), "b": (8, 16384, 65536)}


def _window(fn, window_s: float) -> dict:
    """Per-call ms of fn over a window of at least window_s seconds (after one warm-up call), 3 windows."""
    fn()
    torch.cuda.synchronize()
    one = min(_events_ms(fn, 3)) * 1e-3
    reps = max(1, math.ceil(window_s / max(one, 1e-6)))

    def loop():
        for _ in range(reps):
            fn()

    ms = _events_ms(loop, 3)
    return {"reps": reps, "window_ms": [round(x, 1) for x in ms], "ms_per_call": min(ms) / reps}


def torch_arm(x: torch.Tensor, y: torch.Tensor, rows: int = 2048):
    """fp32 torch.cdist + min / argmin, chunked over rows of x so that the distance block stays at rows x Ny."""
    b, nx, ny = x.shape[0], x.shape[1], y.shape[1]
    d_xy = torch.empty(b, nx, device=x.device)
    i_xy = torch.empty(b, nx, device=x.device, dtype=torch.int64)
    d_yx = torch.full((b, ny), float("inf"), device=x.device)
    i_yx = torch.zeros(b, ny, device=x.device, dtype=torch.int64)
    for r0 in range(0, nx, rows):
        d = torch.cdist(x[:, r0:r0 + rows], y).pow_(2)
        d_xy[:, r0:r0 + rows], i_xy[:, r0:r0 + rows] = d.min(2)
        v, i = d.min(1)
        better = v < d_yx
        d_yx = torch.where(better, v, d_yx)
        i_yx = torch.where(better, i + r0, i_yx)
    return d_xy, i_xy, d_yx, i_yx


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nearest_time: needs a CUDA device")

    from gecco_b200 import _abi
    from gecco_b200.metrics import _launch, nearest_neighbours
    from gecco_b200.ops import _lib_for, _stream
    torch.backends.cuda.matmul.allow_tf32 = False  # the torch arm stays fp32

    res = {"card": card_info()}
    mix = inner_loop_mix(_abi.lib_path(), "nearest_kernel")
    res["inner_loop"] = mix
    with tempfile.TemporaryDirectory() as tmp:
        rates = micro_rates(Path(tmp), res["card"]["sm_count"])
    res["issue_rates_warp_instr_per_s"] = rates
    # per opcode: its measured rate when a micro-kernel covers it, otherwise the FFMA rate (the issue limit)
    per_pair_s = None if mix is None else sum(c / rates.get(op, rates["FFMA"]) for op, c in mix["per_pair"].items())
    if mix is not None:
        res["issue_slots_per_pair"] = per_pair_s * rates["FFMA"]

    g = torch.Generator(device="cuda").manual_seed(0)
    for name, (b, nx, ny) in WORKLOADS.items():
        x = torch.randn(b, nx, 3, device="cuda", generator=g)
        y = torch.randn(b, ny, 3, device="cuda", generator=g) * 0.9 + 0.05
        pairs = b * nx * ny
        w = {"pairs": b, "nx": nx, "ny": ny, "point_pairs": pairs}
        lib = _lib_for(x)
        nbytes = lib.gecco_nearest_scratch_bytes(b, nx, ny)
        bufs = [torch.empty(b, nx, device="cuda"), torch.empty(b, nx, device="cuda", dtype=torch.int32),
                torch.empty(b, ny, device="cuda"), torch.empty(b, ny, device="cuda", dtype=torch.int32),
                torch.empty((nbytes + 7) // 8, device="cuda", dtype=torch.int64)]
        na = _abi.NearestArgs()
        na.x, na.y, na.clouds, na.nx, na.ny = x.data_ptr(), y.data_ptr(), b, nx, ny
        na.dist_xy, na.idx_xy, na.dist_yx, na.idx_yx, na.scratch = (t.data_ptr() for t in bufs)
        na.scratch_bytes = nbytes
        stream = _stream(x)
        t = _window(lambda: _abi.check(lib.gecco_nearest(C.byref(na), stream)), args.window)
        w["nearest"] = dict(t, point_pairs_per_s=pairs / (t["ms_per_call"] * 1e-3))
        if per_pair_s is not None:
            bound_ms = pairs / 32 * per_pair_s * 1e3
            w["nearest"]["issue_bound_ms"] = bound_ms
            w["nearest"]["fraction_of_bound"] = bound_ms / t["ms_per_call"]
        cd_out = torch.empty(b, device="cuda")
        t = _window(lambda: _launch("gecco_chamfer", x, y, _abi.CHAMFER_PAIRED, cd_out), args.window)
        w["chamfer_paired"] = dict(t, point_pairs_per_s=pairs / (t["ms_per_call"] * 1e-3))
        t = _window(lambda: nearest_neighbours(x, y), args.window)
        w["nearest_neighbours_python_call"] = t
        t = _window(lambda: torch_arm(x, y), args.window)
        w["torch_cdist_arm"] = dict(t, point_pairs_per_s=pairs / (t["ms_per_call"] * 1e-3))
        w["nearest_speedup_vs_chamfer"] = w["chamfer_paired"]["ms_per_call"] / w["nearest"]["ms_per_call"]
        w["nearest_speedup_vs_torch"] = w["torch_cdist_arm"]["ms_per_call"] / w["nearest"]["ms_per_call"]
        nn = nearest_neighbours(x, y)
        assert torch.equal(nn.dist_xy, bufs[0]) and torch.equal(nn.idx_yx, bufs[3].long())  # the timed launch's result
        ref = torch_arm(x, y)
        w["index_agreement_with_torch_arm"] = [(nn.idx_xy == ref[1]).double().mean().item(),
                                               (nn.idx_yx == ref[3]).double().mean().item()]
        res[name] = w
        del x, y, nn, ref, bufs
        torch.cuda.empty_cache()
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()
