"""CPU-side checks of the per-point reconstruction metrics: the float64 nearest-neighbour oracle against explicit loops,
the F-score restatement on hand-computed cases, and every input check of nearest_neighbours / reconstruction_metrics
and of the C entry point, which all refuse before any launch."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from gecco_b200 import _abi
from gecco_b200.metrics import NEAREST_MAX_POINTS, nearest_neighbours, reconstruction_metrics
from oracle import nearest_oracle as NO


def _loops(x, y):
    """Nearest neighbours of one pair by explicit Python loops over float lists; lowest index on ties."""
    def nn(a, b):
        d_out, i_out = [], []
        for p in a:
            best, arg = math.inf, -1
            for j, q in enumerate(b):
                d = sum((pk - qk) ** 2 for pk, qk in zip(p, q))
                if d < best:
                    best, arg = d, j
            d_out.append(best)
            i_out.append(arg)
        return d_out, i_out

    a, b = x.tolist(), y.tolist()
    return nn(a, b) + nn(b, a)


@pytest.mark.parametrize("nx,ny", [(1, 1), (1, 7), (7, 1), (13, 29), (40, 9)])
def test_oracle_matches_loops(nx, ny):
    g = torch.Generator().manual_seed(nx * 100 + ny)
    x = torch.randn(3, nx, 3, generator=g, dtype=torch.float64)
    y = torch.randn(3, ny, 3, generator=g, dtype=torch.float64)
    if ny > 3:
        y[:, 3] = y[:, 1]          # duplicate: the lower index must win
    if ny > 2 and nx > 2:
        x[:, 2] = y[:, 2]          # coincident: distance exactly 0
    got = NO.nearest_f64(x, y, chunk_elems=16 * 3)  # several row chunks
    for b in range(3):
        d_xy, i_xy, d_yx, i_yx = _loops(x[b], y[b])
        assert got[1][b].tolist() == i_xy and got[3][b].tolist() == i_yx
        np.testing.assert_allclose(got[0][b].numpy(), d_xy, rtol=1e-12, atol=0)
        np.testing.assert_allclose(got[2][b].numpy(), d_yx, rtol=1e-12, atol=0)
    if ny > 3:
        assert not (got[1] == 3).any()
    if ny > 2 and nx > 2:
        assert torch.all(got[0][:, 2] == 0)


def test_oracle_second_neighbour():
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 11, 3, generator=g, dtype=torch.float64)
    y = torch.randn(2, 17, 3, generator=g, dtype=torch.float64)
    d_xy, _, d_yx, _, s_xy, s_yx = NO.nearest_f64(x, y, chunk_elems=4 * 17 * 3, second=True)
    full = (x[:, :, None, :] - y[:, None, :, :]).pow(2).sum(-1)
    assert torch.equal(s_xy, full.sort(2).values[:, :, 1]) and torch.equal(d_xy, full.amin(2))
    assert torch.equal(s_yx, full.sort(1).values[:, 1, :]) and torch.equal(d_yx, full.amin(1))
    one = NO.nearest_f64(x[:, :1], y[:, :1], second=True)
    assert torch.all(one[4] == math.inf) and torch.all(one[5] == math.inf)


def test_fscore_hand_cases():
    # perfect match: every distance 0
    p, r, f = NO.fscore_np(np.zeros((1, 5)), np.zeros((1, 4)), [0.01])
    assert p.tolist() == [[1.0]] and r.tolist() == [[1.0]] and f.tolist() == [[1.0]]
    # disjoint clouds: no point within tau in either direction; F is 0, not NaN
    p, r, f = NO.fscore_np(np.full((2, 3), 4.0), np.full((2, 6), 9.0), [0.1, 1.0])
    assert np.all(p == 0) and np.all(r == 0) and np.all(f == 0) and not np.isnan(f).any()
    # asymmetric: 2 of 3 predicted points within tau = 0.5, 1 of 2 target points; the threshold test is strict
    p, r, f = NO.fscore_np([[0.0, 0.1, 0.25]], [[0.0, 1.0]], [0.5, 1.0])
    assert p[0, 0] == pytest.approx(2 / 3) and r[0, 0] == 0.5 and f[0, 0] == pytest.approx(4 / 7)
    assert p[0, 1] == 1.0 and r[0, 1] == 0.5 and f[0, 1] == pytest.approx(2 / 3)


def test_entry_points_check_their_input():
    x = torch.randn(3, 16, 3, dtype=torch.float64)
    with pytest.raises(_abi.GeccoError):        # CPU tensors: there is no CPU path
        nearest_neighbours(x, x)
    with pytest.raises(_abi.GeccoError):
        reconstruction_metrics(x, x, [0.01])
    with pytest.raises(ValueError, match="same number of clouds"):
        nearest_neighbours(x, torch.randn(2, 16, 3))
    with pytest.raises(ValueError, match="same number of clouds"):
        reconstruction_metrics(x, torch.randn(4, 9, 3), [0.01])
    with pytest.raises(ValueError, match="one device"):
        nearest_neighbours(x, torch.empty(3, 16, 3, device="meta"))
    bad = x.clone()
    bad[1, 3, 2] = float("nan")
    bad[2, 0, 0] = float("inf")
    with pytest.raises(ValueError, match=r"2 cloud\(s\) with non-finite points \(indices 1, 2\)"):
        nearest_neighbours(bad, x)
    with pytest.raises(ValueError, match="shape"):
        nearest_neighbours(x[0], x[0])
    with pytest.raises(ValueError, match="at least one point"):
        nearest_neighbours(x[:, :0], x)
    with pytest.raises(TypeError):
        nearest_neighbours(x.long(), x)
    with pytest.raises(TypeError):
        nearest_neighbours(x.tolist(), x)
    huge = torch.zeros(1, 1, 3).expand(1, NEAREST_MAX_POINTS + 1, 3)
    with pytest.raises(ValueError, match="at most 16777216"):
        nearest_neighbours(huge, torch.zeros(1, 5, 3))
    for th in ([], (), [0.0], [-0.01], [float("nan")], [float("inf")], [0.01, 0.0], "0.01", 0.01, None, [True],
               ["0.01"], torch.tensor(0.01), np.array([]), np.array([[0.01]]), np.array([0.01, -1.0])):
        with pytest.raises(ValueError, match="thresholds"):
            reconstruction_metrics(x, x, th)
    # accepted threshold forms get past the threshold check to the CPU-tensor refusal
    for th in ([0.01], (0.005, 0.02), torch.tensor([0.01, 0.02]), np.linspace(0.005, 0.02, 4), np.float32([0.01])):
        with pytest.raises(_abi.GeccoError):
            reconstruction_metrics(x, x, th)


def test_c_entry_point_refuses_bad_arguments():
    lib = _abi.load()
    assert lib.gecco_nearest_scratch_bytes(3, 5, 7) == 8 * 3 * (5 + 7 + 2)
    assert lib.gecco_nearest_scratch_bytes(-1, 5, 7) == -1
    fake = 1 << 20  # never dereferenced: every case below is refused before any device work

    def call(clouds, nx, ny, scratch_bytes=None, scratch=fake):
        a = _abi.NearestArgs()
        a.x = a.y = a.dist_xy = a.idx_xy = a.dist_yx = a.idx_yx = fake
        a.scratch = scratch
        a.clouds, a.nx, a.ny = clouds, nx, ny
        a.scratch_bytes = lib.gecco_nearest_scratch_bytes(clouds, nx, ny) if scratch_bytes is None else scratch_bytes
        rc = lib.gecco_nearest(C.byref(a), None)
        return rc, lib.gecco_last_error().decode()

    for clouds, nx, ny in [(1, 0, 5), (1, 5, 0), (1, NEAREST_MAX_POINTS + 1, 5), (2, 5, NEAREST_MAX_POINTS + 1)]:
        rc, msg = call(clouds, nx, ny)
        assert rc == -1 and "1 to 16777216 points" in msg
    rc, msg = call(-1, 5, 5, scratch_bytes=0)
    assert rc == -1 and "negative cloud count" in msg
    rc, msg = call(2, 5, 5, scratch_bytes=8 * 2 * 12 - 8)
    assert rc == -1 and "scratch" in msg
    rc, msg = call(2, 5, 5, scratch=fake + 8)
    assert rc == -1 and "16-byte aligned" in msg
    rc, msg = call(2, 5, 5, scratch=0)
    assert rc == -1 and "null argument" in msg
