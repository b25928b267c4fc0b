"""CPU: the host side of temperature scaling. helpers.temperature_grid's grid and its argument checks, and
helpers.temperature_from_sums on fp64 sums computed in numpy from synthetic pooled probabilities and labels: the fitted
temperature against scipy's minimiser of the exact objective, the bounds, the degenerate inputs and the constructor and
setter checks of SpctEnsemble's temperature."""
import math

import numpy as np
import pytest

NEG_LOG_FLT_MIN = -math.log(np.finfo(np.float32).tiny)


def synthetic(n, k, sharpen, seed, zeros=0.0):
    """(p̄ [n,k] fp64, labels [n]): labels drawn from softmax(z), p̄ = softmax(sharpen * z), so the calibrating
    temperature is about `sharpen`; a fraction `zeros` of the entries of p̄ set to 0 (renormalised)."""
    rng = np.random.default_rng(seed)
    z = rng.normal(size=(n, k)) * 2.0
    q = np.exp(z - z.max(1, keepdims=True))
    q /= q.sum(1, keepdims=True)
    y = (rng.random((n, 1)) > np.cumsum(q, 1)).sum(1).clip(max=k - 1)
    p = np.exp(sharpen * (z - z.max(1, keepdims=True)))
    if zeros:
        p[rng.random(p.shape) < zeros] = 0.0
        p[np.arange(n), p.argmax(1)] = np.maximum(p.max(1), 1e-3)
    p /= p.sum(1, keepdims=True)
    return p, y


def objective(beta, p, y):
    """Per-voxel f(β) = log sum_{c: p_c > 0} p_c^β - β log p_y and f'(β), fp64; -log FLT_MIN and 0 when p_y = 0."""
    with np.errstate(divide="ignore"):
        lg = np.log(p)
    pos = p > 0
    m = np.where(pos, lg, -np.inf).max(1, keepdims=True)
    e = np.where(pos, np.exp(beta * (np.where(pos, lg, 0.0) - m)), 0.0)
    s = e.sum(1)
    ly = lg[np.arange(len(y)), y]
    zero = p[np.arange(len(y)), y] == 0
    f = np.where(zero, NEG_LOG_FLT_MIN, beta * m[:, 0] + np.log(s) - beta * np.where(zero, 0.0, ly))
    d = np.where(zero, 0.0, (e * np.where(pos, lg, 0.0)).sum(1) / s - np.where(zero, 0.0, ly))
    return f, d


def grid_sums(betas, p, y):
    out = np.zeros((2, betas.size))
    for g, b in enumerate(betas):
        f, d = objective(b, p, y)
        out[0, g], out[1, g] = f.sum(), d.sum()
    return out


def scipy_temperature(p, y, t_max):
    from scipy.optimize import minimize_scalar
    r = minimize_scalar(lambda b: objective(b, p, y)[0].mean(), bounds=(1.0 / t_max, t_max), method="bounded",
                        options={"xatol": 1e-10})
    return 1.0 / r.x, r.fun


def test_grid():
    from innovative3D.helpers import temperature_grid
    b = temperature_grid(8.0, 33)
    assert b.size == 33 and b[16] == 1.0 and np.all(np.diff(b) > 0)
    assert abs(b[0] - 1 / 8) <= 1e-7 and abs(b[-1] - 8) <= 1e-6
    assert np.array_equal(b, b.astype(np.float32).astype(np.float64))           # the values the kernel evaluates
    np.testing.assert_allclose(b[1:] / b[:-1], 8.0 ** (1 / 16), rtol=1e-6)      # geometric
    assert temperature_grid(2.0, 5)[2] == 1.0 and temperature_grid(30.0, 63).size == 63


@pytest.mark.parametrize("points", [4, 6, 3, 1, 65, 64, 33.5, True])
def test_grid_rejects_points(points):
    from innovative3D.helpers import temperature_grid
    with pytest.raises(ValueError, match="points"):
        temperature_grid(8.0, points)


@pytest.mark.parametrize("t_max", [1.0, 0.5, -2.0, float("inf"), float("nan")])
def test_grid_rejects_t_max(t_max):
    from innovative3D.helpers import temperature_grid
    with pytest.raises(ValueError, match="t_max"):
        temperature_grid(t_max, 33)


@pytest.mark.parametrize("t_max,points,rtol", [(8.0, 33, 1e-4), (4.0, 21, 1e-4), (8.0, 63, 1e-4), (16.0, 45, 1e-4),
                                              (3.0, 9, 1e-3)])
@pytest.mark.parametrize("sharpen,k,zeros", [(2.0, 5, 0.0), (0.6, 13, 0.0), (1.3, 2, 0.0), (2.5, 16, 0.2)])
def test_temperature_matches_scipy(t_max, points, rtol, sharpen, k, zeros):
    """The interpolated minimiser is within 1e-4 relative of scipy's on the exact objective for grids whose points are
    at most 14 % apart (1e-3 on the coarse 9-point grid over [1/3, 3], 32 % apart: the cubic's error grows with the
    spacing); the reported, interpolated nll within a tenth of that of the objective there; nll_at_1 is the untempered nll."""
    from innovative3D.helpers import temperature_from_sums, temperature_grid
    p, y = synthetic(20000, k, sharpen, seed=int(10 * sharpen) + k, zeros=zeros)
    if zeros:   # voxels whose label has p̄_y = 0 contribute the constant -log FLT_MIN
        assert (p[np.arange(len(y)), y] == 0).any()
    betas = temperature_grid(t_max, points)
    res = temperature_from_sums(betas, grid_sums(betas, p, y), len(y))
    t_ref, nll_ref = scipy_temperature(p, y, t_max)
    assert not res["at_bound"], res["grid"]["dnll"]
    assert abs(res["temperature"] / t_ref - 1) <= rtol, (res["temperature"], t_ref)
    assert abs(res["nll"] - nll_ref) <= rtol / 10 * max(1.0, nll_ref)
    assert abs(res["nll_at_1"] - objective(1.0, p, y)[0].mean()) <= 1e-12
    assert res["counted"] == len(y) and res["grid"]["nll"].size == points
    np.testing.assert_allclose(res["grid"]["temperature"], 1.0 / betas)


def test_at_bound_both_sides():
    """Overconfident beyond t_max: T̂ = t_max (β at the smallest grid value); underconfident beyond 1/t_max:
    T̂ = 1/t_max. at_bound in both cases, and not otherwise."""
    from innovative3D.helpers import temperature_from_sums, temperature_grid
    betas = temperature_grid(2.0, 9)
    p, y = synthetic(5000, 5, 6.0, seed=1)                # wants T near 6
    r = temperature_from_sums(betas, grid_sums(betas, p, y), len(y))
    assert r["at_bound"] and r["temperature"] == pytest.approx(2.0, rel=1e-6)
    assert np.all(r["grid"]["dnll"] > 0)
    p, y = synthetic(5000, 5, 0.15, seed=2)               # wants T near 0.15
    r = temperature_from_sums(betas, grid_sums(betas, p, y), len(y))
    assert r["at_bound"] and r["temperature"] == pytest.approx(0.5, rel=1e-6)
    assert np.all(r["grid"]["dnll"] < 0)
    assert r["nll"] == r["grid"]["nll"][-1]
    p, y = synthetic(5000, 5, 1.5, seed=3)
    assert not temperature_from_sums(betas, grid_sums(betas, p, y), len(y))["at_bound"]


def test_secant_fallback_and_exact_zero():
    """A linear slope with a flat nll (no cubic minimum inside) falls back to the secant root of f'; a grid point with
    f' = 0 exactly is the answer."""
    from innovative3D.helpers import temperature_from_sums
    betas = np.array([0.5, 1.0, 2.0])
    r = temperature_from_sums(betas, np.array([[3.0, 3.0, 3.0], [-1.0, 1.0, 3.0]]), 1)
    assert 0.5 <= 1 / r["temperature"] <= 1.0 and not r["at_bound"]
    r = temperature_from_sums(betas, np.array([[3.0, 2.0, 3.0], [-1.0, 0.0, 3.0]]), 1)
    assert r["temperature"] == 1.0
    # a quadratic nll: the Hermite cubic is exact, its minimiser is the vertex
    f = lambda b: (b - 0.8) ** 2          # noqa: E731
    r = temperature_from_sums(betas, np.array([[f(b) for b in betas], [2 * (b - 0.8) for b in betas]]) * 7, 7)
    assert r["temperature"] == pytest.approx(1 / 0.8, rel=1e-12) and r["nll"] == pytest.approx(0.0, abs=1e-12)


def test_rejects_no_counted_voxel_and_bad_inputs():
    from innovative3D.helpers import temperature_from_sums, temperature_grid
    betas = temperature_grid(8.0, 33)
    with pytest.raises(ValueError, match="no counted voxel"):
        temperature_from_sums(betas, np.zeros((2, 33)), 0)
    with pytest.raises(ValueError, match="sums"):
        temperature_from_sums(betas, np.zeros((2, 31)), 5)
    with pytest.raises(ValueError, match="ascending"):
        temperature_from_sums(betas[::-1], np.zeros((2, 33)), 5)


def test_ensemble_temperature_checks():
    """The temperature must be positive and finite, in the constructor and the setter (no GPU needed: the members are
    CPU cores)."""
    import torch
    from innovative3D import config as C
    from innovative3D import models
    torch.manual_seed(0)
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]()
    ens = models.SpctEnsemble([lit])
    assert ens.temperature == 1.0
    ens.temperature = 2.5
    assert ens.temperature == 2.5
    assert models.SpctEnsemble([lit], temperature=0.7).temperature == 0.7
    for bad in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError, match="temperature"):
            models.SpctEnsemble([lit], temperature=bad)
        with pytest.raises(ValueError, match="temperature"):
            ens.temperature = bad
    assert ens.temperature == 2.5
