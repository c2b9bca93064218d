"""CPU checks of the exact earth mover's distance: the assignment oracle (oracle/emd_exact_oracle.py) against brute force
on tiny clouds, properties of the definition (symmetry, permutations, the bound from the approximate EMD), and every
input check of optimal_matching / emd_exact_matrix / sample_metrics and of the C entry point, which all refuse before
any launch."""
import ctypes as C

import numpy as np
import pytest
import torch

from gecco_b200 import _abi
from gecco_b200.metrics import EMD_MAX_POINTS, emd_exact_matrix, optimal_matching, sample_metrics
from oracle import emd_exact_oracle as XO
from oracle import emd_oracle as EO


@pytest.mark.parametrize("n", [1, 2, 3, 5, 7])
@pytest.mark.parametrize("kind", ["random", "tied"])
def test_lsa_equals_brute_force(n, kind):
    rng = np.random.default_rng(n * 10 + (kind == "tied"))
    for _ in range(4):
        if kind == "random":
            x, y = rng.normal(size=(n, 3)), rng.normal(size=(n, 3)) * 0.7 + 0.2
        else:  # points on a coarse lattice, repeated points: many equal costs and several optimal permutations
            x = rng.integers(0, 2, size=(n, 3)).astype(np.float64)
            y = rng.integers(0, 2, size=(n, 3)).astype(np.float64)
        got, sigma = XO.lsa(x, y)
        want, perm = XO.brute_force(x, y)
        assert got == pytest.approx(want, rel=1e-12, abs=1e-15)
        assert sorted(sigma.tolist()) == list(range(n))
        assert np.linalg.norm(x - y[sigma], axis=1).mean() == pytest.approx(got, rel=1e-12, abs=1e-15)
        assert np.linalg.norm(x - y[list(perm)], axis=1).mean() == pytest.approx(want, rel=1e-12, abs=1e-15)


def test_single_point_and_identity():
    x, y = np.array([[0.0, 1.0, 2.0]]), np.array([[3.0, 5.0, 2.0]])
    assert XO.lsa(x, y)[0] == 5.0
    rng = np.random.default_rng(1)
    z = rng.normal(size=(30, 3))
    cost, sigma = XO.lsa(z, z[::-1])
    assert cost == 0.0 and np.array_equal(sigma, np.arange(30)[::-1])


def test_symmetric_and_permutation_invariant():
    rng = np.random.default_rng(2)
    x, y = rng.normal(size=(64, 3)), rng.normal(size=(64, 3)) * 0.8 + 0.3
    base = XO.lsa(x, y)[0]
    assert XO.lsa(y, x)[0] == pytest.approx(base, rel=1e-12)
    assert XO.lsa(x[rng.permutation(64)], y)[0] == pytest.approx(base, rel=1e-12)
    assert XO.lsa(x, y[rng.permutation(64)])[0] == pytest.approx(base, rel=1e-12)
    m = XO.emd_exact_matrix_f64(np.stack([x, y, x[::-1]]))
    assert np.array_equal(m, m.T) and np.all(np.diag(m) == 0) and m[0, 2] == 0.0
    assert m[0, 1] == pytest.approx(base, rel=1e-12)


@pytest.mark.parametrize("seed,n,scale,shift", [(0, 64, 1.0, 0.2), (1, 200, 1.0, 0.2), (2, 256, 0.05, 0.0),
                                                (3, 96, 0.5, 10.0)])
def test_below_the_approximate_emd(seed, n, scale, shift):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(2, n, 3, generator=g, dtype=torch.float64) * scale
    b = torch.randn(2, n, 3, generator=g, dtype=torch.float64) * scale * 0.8 + shift
    approx = EO.emd_matrix_f64(a, b)
    exact = XO.emd_exact_matrix_f64(a, b)
    assert (exact <= approx.numpy() * (1 + 1e-12)).all()
    assert (exact < approx.numpy()).any()  # the approximate matching is not optimal on these clouds


def test_entry_points_check_their_input():
    x = torch.randn(3, 16, 3, dtype=torch.float64)
    with pytest.raises(_abi.GeccoError):        # CPU tensors: there is no CPU path
        optimal_matching(x, x)
    with pytest.raises(_abi.GeccoError):
        emd_exact_matrix(x)
    with pytest.raises(_abi.GeccoError):
        emd_exact_matrix(x, x)
    with pytest.raises(_abi.GeccoError):
        sample_metrics(x, x, distance="emd_exact")
    with pytest.raises(ValueError, match="same number of clouds"):
        optimal_matching(x, torch.randn(2, 16, 3))
    with pytest.raises(ValueError, match="one device"):
        optimal_matching(x, torch.empty(3, 16, 3, device="meta"))
    bad = x.clone()
    bad[1, 3, 2] = float("nan")
    bad[2, 0, 0] = float("inf")
    with pytest.raises(ValueError, match=r"2 cloud\(s\) with non-finite points \(indices 1, 2\)"):
        optimal_matching(bad, x)
    with pytest.raises(ValueError, match=r"indices 1, 2"):
        emd_exact_matrix(bad)
    for f in (lambda: optimal_matching(x, torch.randn(3, 15, 3)), lambda: emd_exact_matrix(x, torch.randn(2, 17, 3)),
              lambda: sample_metrics(x, torch.randn(2, 17, 3), distance="emd_exact")):
        with pytest.raises(ValueError, match="equal point counts"):
            f()
    big = torch.zeros(2, EMD_MAX_POINTS + 1, 3)
    with pytest.raises(ValueError, match="at most 4096"):
        optimal_matching(big, big)
    with pytest.raises(ValueError, match="at most 4096"):
        emd_exact_matrix(big)
    with pytest.raises(ValueError, match="shape"):
        optimal_matching(x[0], x[0])
    with pytest.raises(ValueError, match="at least one point"):
        emd_exact_matrix(x[:, :0])
    with pytest.raises(TypeError):
        optimal_matching(x.long(), x.long())
    with pytest.raises(TypeError):
        optimal_matching(x.tolist(), x)
    with pytest.raises(ValueError, match="distance must be"):
        sample_metrics(x, x, distance="emd_approx")


def test_c_entry_point_refuses_bad_arguments():
    lib = _abi.load()
    fake = 1 << 20  # never dereferenced: every case below is refused before any device work

    def call(mode=_abi.CHAMFER_ALL, ma=2, na=5, mb=2, nb=5, a=fake, b=fake, out=fake, lower=fake, match=None):
        args = _abi.EmdExactArgs()
        args.a, args.ma, args.na = a, ma, na
        args.b, args.mb, args.nb = b, mb, nb
        args.mode, args.out, args.lower, args.match = mode, out, lower, match
        rc = lib.gecco_emd_exact(C.byref(args), None)
        return rc, lib.gecco_last_error().decode()

    for na in (0, -1, EMD_MAX_POINTS + 1):
        rc, msg = call(na=na, nb=na)
        assert rc == -1 and "1 to 4096 points" in msg, msg
    rc, msg = call(na=5, nb=6)
    assert rc == -1 and "equal point counts" in msg
    rc, msg = call(mode=_abi.CHAMFER_PAIRED, na=5, nb=6, match=fake)
    assert rc == -1 and "equal point counts" in msg
    rc, msg = call(mode=3)
    assert rc == -1 and "unknown mode" in msg
    rc, msg = call(mode=-1)
    assert rc == -1 and "unknown mode" in msg
    for mode in (_abi.CHAMFER_ALL, _abi.CHAMFER_SELF):
        rc, msg = call(mode=mode, match=fake)
        assert rc == -1 and "match" in msg
    rc, msg = call(mode=_abi.CHAMFER_PAIRED, ma=2, mb=3)
    assert rc == -1 and "as many clouds" in msg
    rc, msg = call(ma=-1)
    assert rc == -1 and "negative cloud count" in msg
    rc, msg = call(mode=_abi.CHAMFER_SELF, b=fake + 64)
    assert rc == -1 and "self mode" in msg
    rc, msg = call(out=None)
    assert rc == -1 and "null argument" in msg
    rc, msg = call(b=None)
    assert rc == -1 and "null argument" in msg
    rc = lib.gecco_emd_exact(None, None)
    assert rc == -1 and "null args" in lib.gecco_last_error().decode()
    # nothing to compute: accepted without touching the device
    assert call(ma=0, mb=4)[0] == 0
    assert call(mode=_abi.CHAMFER_PAIRED, ma=0, mb=0, match=fake)[0] == 0
