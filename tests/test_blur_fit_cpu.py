"""Fitting the blur stops, host side: a float64 restatement of the blur's derivative in its sigma map (used by the GPU tests as
the reference for rdc_gaussian_blur_sigma_adjoint), checked against central differences of the restated blur; the projected
gradient minimiser behind api.fit_blur; and the argument checks of both new entry points that need no device.

With the taps [f, l] of taps_for(sigma_p) held fixed, a pass Y(p) = sum_k g(k) X(clamp(p + k)) / a is smooth in sigma_p:
g(k) = exp(-k^2 / s^2), s = sigma_p + 1e-6, g'(k) = g(k) 2 k^2 / s^3 and dY(p)/dsigma_p = sum_k g'(k) (X(clamp(p + k)) - Y(p)) / a.
The blur D = V(H(S)) reads sigma_p in both passes at p, so sigma_p moves T(p) and, on the band, D(p).
"""
import ctypes
import itertools

import numpy as np
import pytest

from raytracingdiffusioncurves_b200 import api
from test_blur_adjoint_cpu import SIGMA_CASES, sigma_case, taps

RDC_E_INVALID = -1


def pass_matrices(first, last, sigma, n, absolute=False):
    """One pass along a line of n pixels with taps [first, last] (frozen) and float64 weights of `sigma`:
    m[p, clamp(p + k)] += g_p(k) / a_p, dm[p] the derivative of row p in sigma_p, reads[p] the sources row p reads.
    absolute: dm's two parts added by magnitude instead of subtracted."""
    m = np.zeros((n, n))
    dm = np.zeros((n, n))
    reads = np.zeros((n, n), bool)
    for p in range(n):
        if first[p] > last[p]:
            continue
        k = np.arange(first[p], last[p] + 1)
        s = float(sigma[p]) + 1e-6
        g = np.exp(-(k * k) / (s * s))
        gp = g * 2.0 * (k * k) / (s * s * s)
        a, ap = g.sum(), gp.sum()
        cols = np.clip(p + k, 0, n - 1)
        np.add.at(m[p], cols, g / a)
        np.add.at(dm[p], cols, gp / a + (1.0 if absolute else -1.0) * g * ap / (a * a))
        reads[p, cols] = True
    return m, dm, reads


def restated_passes(sigma, source, sigma_eval=None, absolute=False):
    """Both passes over every row, taps of `sigma` (float32, as the kernels see it), weights of sigma_eval (default: sigma)
    in float64. Returns T, dT/dsigma, D, dD/dsigma (float64 [h, w, 4]), the column matrices of V and the NaN mask of D
    (a pixel without taps, or one that reads a NaN). absolute: the sums of the magnitudes of their terms instead (a scale for
    fp32 rounding)."""
    sigma = np.asarray(sigma, np.float32)
    h, w = sigma.shape
    first, last, _ = taps(sigma)
    dead = first > last
    se = np.asarray(sigma if sigma_eval is None else sigma_eval, np.float64)
    src = np.asarray(source, np.float64)
    src_nan = np.isnan(src).any(-1)
    src = np.nan_to_num(src)
    if absolute:
        src = np.abs(src)
    t, dt, t_nan = np.zeros((h, w, 4)), np.zeros((h, w, 4)), np.zeros((h, w), bool)
    for y in range(h):
        m, dm, reads = pass_matrices(first[y], last[y], se[y], w, absolute)
        t[y], dt[y] = m @ src[y], dm @ src[y]
        t_nan[y] = dead[y] | (reads & src_nan[y]).any(1)
    d, dd, d_nan, vm = np.zeros((h, w, 4)), np.zeros((h, w, 4)), np.zeros((h, w), bool), []
    for x in range(w):
        m, dm, reads = pass_matrices(first[:, x], last[:, x], se[:, x], h, absolute)
        d[:, x], dd[:, x] = m @ t[:, x], dm @ t[:, x]
        d_nan[:, x] = dead[:, x] | (reads & t_nan[:, x]).any(1)
        vm.append(m)
    return t, dt, d, dd, vm, d_nan


def masked_dot(f, x):
    """sum <f, x> over channels whose factor is nonzero (a zero factor adds nothing, even against a NaN)"""
    return np.where(f != 0.0, f * np.where(f != 0.0, x, 0.0), 0.0).sum(-1)


def restated_sigma_adjoint(sigma, source, grad, row_begin=0, row_end=None, absolute=False):
    """float64 [h, w]: sum over band pixels p of <grad[p], d D[p] / d sigma[q]> for every q, taps frozen; grad is [h, w, 4]
    and only its band rows are read. The vertical term on the band, plus the horizontal term through V's transpose.
    absolute: the same sums of absolute values, a bound for the rounding of an fp32 evaluation."""
    h, w = np.asarray(sigma).shape
    row_end = h if row_end is None else row_end
    t, dt, d, dd, vm, _ = restated_passes(sigma, source, absolute=absolute)
    g = np.zeros((h, w, 4))
    g[row_begin:row_end] = np.asarray(grad, np.float64)[row_begin:row_end]
    if absolute:
        g = np.abs(g)
    out = masked_dot(g, dd)
    g_t = np.stack([vm[x].T @ g[:, x] for x in range(w)], axis=1)  # the gradient in T
    return out + masked_dot(g_t, dt)


def frozen_objective_rows(sigma, source, grad, sigma_eval):
    """per row y: sum_x <grad, D(sigma_eval)> with the taps of `sigma`; grad is zero where D is NaN"""
    _, _, d, _, _, _ = restated_passes(sigma, source, sigma_eval)
    return masked_dot(np.asarray(grad, np.float64), d).sum(1)


def random_case(case, h, w, seed):
    """sigma map, source and a gradient that is zero where the blurred frame is NaN (and in a few single channels)"""
    rng = np.random.default_rng(seed)
    sigma = sigma_case(case, h, w, seed=seed)
    source = rng.random((h, w, 4)).astype(np.float32)
    grad = rng.standard_normal((h, w, 4)).astype(np.float32)
    grad[rng.random((h, w, 4)) < 0.1] = 0.0
    grad[restated_passes(sigma, source)[5]] = 0.0
    return sigma, source, grad


def bands(h):
    return [(b, e) for b in range(h) for e in range(b + 1, h + 1)]


@pytest.mark.parametrize("case", SIGMA_CASES)
@pytest.mark.parametrize("h,w", [(1, 1), (1, 17), (17, 1), (13, 9)])
def test_restated_sigma_derivative_matches_central_differences(case, h, w):
    sigma, source, grad = random_case(case, h, w, seed=h * 100 + w)
    se = sigma.astype(np.float64)
    # rows of the frozen objective under sigma_q +- step, for every q: any band's difference is a sum of rows
    plus, minus, steps = {}, {}, {}
    first, last, _ = taps(sigma)
    for y, x in itertools.product(range(h), range(w)):
        if first[y, x] > last[y, x]:
            continue
        steps[y, x] = step = 1e-5 * max(1.0, abs(se[y, x]))
        for store, sign in ((plus, 1.0), (minus, -1.0)):
            s = se.copy()
            s[y, x] += sign * step
            store[y, x] = frozen_objective_rows(sigma, source, grad, s)
    for b, e in bands(h):
        got = restated_sigma_adjoint(sigma, source, grad, b, e)
        want = np.zeros((h, w))
        for q, step in steps.items():
            want[q] = (plus[q][b:e].sum() - minus[q][b:e].sum()) / (2 * step)
        assert np.all(np.isfinite(got))
        scale = np.abs(want).max()
        # the differences' own rounding, eps |F| / step, is the floor where the derivative is 0 (a 1x1 buffer is the identity)
        floor = 100 * 2.2e-16 * np.abs(grad[b:e]).sum() / 1e-5
        assert np.abs(got - want).max() <= 1e-8 * scale + floor, (b, e, np.abs(got - want).max(), scale)
        if case == "zero":
            assert not np.any(got)  # one tap, k = 0: g'(0) = 0


def test_restatement_is_zero_beyond_the_reach():
    sigma, source, grad = random_case("mixed", 40, 5, seed=11)
    reach = int(np.ceil(3 * np.nanmax(sigma)))
    got = restated_sigma_adjoint(sigma, source, grad, 20, 22)
    assert not np.any(got[:20 - reach]) and not np.any(got[22 + reach:])


# ---- projected_descent ----

def bounded_least_squares(seed, n=6, m=12):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((m, n))
    b = rng.standard_normal(m) + a @ np.where(rng.random(n) < 0.5, -1.0, 1.0)  # a solution with some bounds active
    lower = np.where(rng.random(n) < 0.5, 0.0, -0.25)

    def f_and_grad(x):
        r = a @ x - b
        return 0.5 * float(r @ r), a.T @ r

    return a, b, lower, f_and_grad


def brute_force_active_set(a, b, lower):
    """the minimiser over x >= lower, by enumerating which bounds are active"""
    n = a.shape[1]
    best = None
    for active in itertools.product([False, True], repeat=n):
        act = np.array(active)
        x = np.where(act, lower, 0.0)
        free = ~act
        if free.any():
            x[free] = np.linalg.lstsq(a[:, free], b - a[:, act] @ lower[act], rcond=None)[0]
        if np.all(x >= lower - 1e-12):
            r = a @ x - b
            if best is None or r @ r < best[0]:
                best = (r @ r, x)
    return best[1]


@pytest.mark.parametrize("seed", range(5))
def test_projected_descent_reaches_the_bounded_least_squares_solution(seed):
    a, b, lower, f_and_grad = bounded_least_squares(seed)
    want = brute_force_active_set(a, b, lower)
    assert np.any(np.isclose(want, lower)), "the case should have an active bound"
    x, objectives = api.projected_descent(f_and_grad, np.ones(a.shape[1]), lower, 500)
    assert np.allclose(x, want, atol=1e-7), (x, want)


@pytest.mark.parametrize("seed", range(5))
def test_projected_descent_never_raises_the_objective_and_stays_feasible(seed):
    a, b, lower, f_and_grad = bounded_least_squares(seed)
    seen = []

    def recording(x):
        seen.append(x.copy())
        return f_and_grad(x)

    x, objectives = api.projected_descent(recording, np.full(a.shape[1], 3.0), lower, 60)
    assert len(objectives) >= 2
    assert all(b <= a for a, b in zip(objectives, objectives[1:]))
    assert all(np.all(s >= lower) for s in seen) and np.all(x >= lower)


def test_projected_descent_returns_a_stationary_start_unchanged():
    calls = []

    def flat(x):
        calls.append(1)
        return 1.5, np.zeros_like(x)

    x0 = np.array([0.25, 2.0, 0.0])
    x, objectives = api.projected_descent(flat, x0, np.zeros(3), 10)
    assert np.array_equal(x, x0) and objectives == [1.5] and len(calls) == 1
    # a gradient that only pushes into active bounds is stationary too
    x, objectives = api.projected_descent(lambda x: (0.0, np.array([0.0, 0.0, 1.0])), x0, np.zeros(3), 10)
    assert np.array_equal(x, x0) and objectives == [0.0]


def test_projected_descent_rejects_steps_to_nan():
    def f_and_grad(x):
        if x[0] < 0.5:
            return float("nan"), np.full_like(x, np.nan)
        return 0.5 * float((x[0] - 0.4) ** 2), np.array([x[0] - 0.4])

    x, objectives = api.projected_descent(f_and_grad, np.array([2.0]), np.zeros(1), 50)
    assert x[0] >= 0.5 and np.all(np.isfinite(objectives)) and all(b <= a for a, b in zip(objectives, objectives[1:]))


# ---- argument checks ----

def test_sigma_adjoint_rejects_bad_arguments_without_a_device():
    buf = ctypes.c_void_p(16)
    f = api.lib.rdc_gaussian_blur_sigma_adjoint

    def rejected(*args):
        assert f(*args) == RDC_E_INVALID
        assert "blur sigma adjoint" in api.last_error()

    ok = [buf, buf, buf, buf, buf, 8, 6, 0, 6, None, None]
    for i in range(5):  # null grad_sigma, grad_dest, source, sigma, scratch
        args = list(ok)
        args[i] = None
        rejected(*args)
    for w, h, b, e in [(0, 6, 0, 6), (8, 0, 0, 1), (-1, 6, 0, 6), (8, 6, -1, 6), (8, 6, 0, 7), (8, 6, 3, 3), (8, 6, 4, 2)]:
        rejected(buf, buf, buf, buf, buf, w, h, b, e, None, None)
    with pytest.raises(api.RdcError):
        api.gaussian_blur_sigma_adjoint(16, 16, 16, 16, 16, 8, 6, 5, 2)


def test_render_blur_adjoint_rejects_null_arguments_without_a_device():
    p = api.default_frame_params(16, 16, 8)
    buf = ctypes.c_void_p(1)
    f = api.lib.rdc_render_blur_adjoint
    assert f(None, ctypes.byref(p), buf, buf, None) == RDC_E_INVALID
    assert "null scene" in api.last_error()
    assert f(buf, None, buf, buf, None) == RDC_E_INVALID
    assert "null params" in api.last_error()
    assert f(buf, ctypes.byref(p), None, buf, None) == RDC_E_INVALID
    assert "null sigma_grad" in api.last_error()
    assert f(buf, ctypes.byref(p), buf, None, None) == RDC_E_INVALID
    assert "null output array" in api.last_error()
