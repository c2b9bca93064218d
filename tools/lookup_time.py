"""Stand-alone timing of the projective lookup at the bench shape (64 clouds x 2048 points, 137^2 and 256^2 pyramids):
legacy global-gather kernel (GECCO_LOOKUP_SLICES=0) against the shared-memory staged kernel at several slice counts.
Reports achieved GB/s on the compulsory traffic (pyramid once + bf16 output once + coordinates)."""
import os, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch
from gecco_b200 import ops

dev = torch.device("cuda:0")
B, N = 64, 2048
flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)


def t_us(fn, n=20, cold=False):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(n):
        if cold:
            flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot * 1000 / n


xin = torch.randn(B, N, 3, device=dev)
sig = torch.full((B,), 2.0, device=dev)
K = torch.tensor([[1.0859, 0, 0.4964], [0, 1.0859, 0.4964], [0, 0, 1]], device=dev).expand(B, 3, 3).contiguous()
lo = torch.empty(B * N, 672, device=dev, dtype=torch.bfloat16)
lst = torch.zeros(B, 16, 2, dtype=torch.float64, device=dev)
for name, sizes, variants in (("137^2", (34, 17, 8), ("0", "2", "4")), ("256^2", (64, 32, 16), ("0", "12"))):
    levels = [torch.randn(B, s, s, c, device=dev).bfloat16() for s, c in zip(sizes, (96, 192, 384))]
    nbytes = sum(l.numel() * 2 for l in levels) + lo.numel() * 2 + xin.numel() * 4
    for v in variants:
        os.environ["GECCO_LOOKUP_SLICES"] = v
        fn = lambda: ops.lookup(xin, levels, K, reparam_kind=1, mean=[0, 0, 1], sigma_r=[0.15] * 3, sigma=sig, rows_per_cloud=N,
                                out_bf16=lo, stats=lst)
        hot, cold = t_us(fn), t_us(fn, cold=True)
        print(f"lookup {name} slices={v:>3s}: hot L2 {hot:7.1f} us ({nbytes / hot / 1e3:7.1f} GB/s)   cold L2 {cold:7.1f} us ({nbytes / cold / 1e3:7.1f} GB/s)")
