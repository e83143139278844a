"""The transpose of the variable-sigma blur, host side: a float64 restatement of the blur as a matrix (used by the GPU tests
as the explicit B), checked against the CPU oracle's blur, and the argument checks of rdc_gaussian_blur_adjoint that need
no device.

The blur of a buffer of `height` rows, band [row_begin, row_end): pixel p has the taps [f, l] of taps_for(sigma_p) (csrc/blur.cu)
and weights g(k) = exp(-k^2 / (sigma_p + 1e-6)^2), a_p = sum g. The horizontal pass T = Hm S over every row, the vertical pass
D = V T on the band, both clamp-to-edge and renormalised by a of the pixel written. A pixel without taps (NaN sigma, sigma
<= -1/3) has a NaN output; in the matrix its row is zero, which is the transpose's convention (it contributes nothing).
"""
import ctypes

import numpy as np
import pytest

from raytracingdiffusioncurves_b200 import api

RDC_E_INVALID = -1
MAX_TAPS = 16384


def taps(sigma):
    """taps_for in fp32: (first, last, sig_square) per pixel; first > last where the pixel has no taps."""
    s = np.asarray(sigma, np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        k_size = np.float32(2) * np.ceil(np.float32(3) * s) + np.float32(1)
        lo = np.clip(-k_size / np.float32(2), -MAX_TAPS, MAX_TAPS)
        hi = np.clip(k_size / np.float32(2), -MAX_TAPS, MAX_TAPS)
        first = np.where(np.isnan(k_size), 0, np.trunc(np.nan_to_num(lo))).astype(np.int64)
        last = np.where(np.isnan(k_size), -1, np.floor(np.nan_to_num(hi))).astype(np.int64)
    sig_square = ((s + np.float32(1e-6)) * (s + np.float32(1e-6))).astype(np.float64)
    return first, last, sig_square


def line_matrix(first, last, sig_square, n):
    """One pass along a line of n pixels: M[p, clamp(p + k)] += g_p(k) / a_p, and which source each output reads at all."""
    m = np.zeros((n, n))
    reads = np.zeros((n, n), bool)
    for p in range(n):
        if first[p] > last[p]:
            continue
        k = np.arange(first[p], last[p] + 1)
        g = np.exp(-(k * k) / sig_square[p])
        cols = np.clip(p + k, 0, n - 1)
        np.add.at(m[p], cols, g / g.sum())
        reads[p, cols] = True
    return m, reads


def blur_matrix(sigma, row_begin=0, row_end=None):
    """B: float64 [(row_end - row_begin) * W, height * W], source pixels row-major; and the mask of band pixels whose
    forward output is NaN (no taps, or a tap on a horizontal-pass pixel without taps)."""
    sigma = np.asarray(sigma, np.float32)
    h, w = sigma.shape
    row_end = h if row_end is None else row_end
    first, last, sq = taps(sigma)
    dead = first > last
    hm = np.zeros((h * w, h * w))
    for y in range(h):
        hm[y * w:(y + 1) * w, y * w:(y + 1) * w] = line_matrix(first[y], last[y], sq[y], w)[0]
    v = np.zeros(((row_end - row_begin) * w, h * w))
    nan = np.zeros((row_end - row_begin) * w, bool)
    for x in range(w):
        m, reads = line_matrix(first[:, x], last[:, x], sq[:, x], h)
        for y in range(row_begin, row_end):
            v[(y - row_begin) * w + x, x::w] = m[y]
            nan[(y - row_begin) * w + x] = dead[y, x] or bool((reads[y] & dead[:, x]).any())
    return v @ hm, nan


def apply(b, image):
    """B applied to a float [height, W, 4] image: float64 [rows * W, 4]."""
    return b @ np.asarray(image, np.float64).reshape(-1, 4)


def sigma_case(case, h, w, seed=0):
    """Sigma maps of the tests: zero, mixed (zeros, tiny sigmas whose outer taps underflow, up to 6), large (reach beyond
    the buffer), NaN and negative (one tap, or none at all) entries."""
    rng = np.random.default_rng(seed)
    mixed = (rng.random((h, w)) * 6.0).astype(np.float32)
    mixed[mixed < 1.5] = 0.0
    mixed[rng.random((h, w)) < 0.1] = 0.01
    if case == "zero":
        return np.zeros((h, w), np.float32)
    if case == "mixed":
        return mixed
    if case == "large":
        return (20.0 + rng.random((h, w)) * 40.0).astype(np.float32)
    if case == "nan":
        mixed[rng.random((h, w)) < 0.15] = np.nan
        return mixed
    if case == "negative":
        pick = rng.random((h, w))
        mixed[pick < 0.3] = -0.2   # k_size 1: one tap
        mixed[pick < 0.2] = -0.5   # no taps
        mixed[pick < 0.1] = -3.0
        return mixed
    raise ValueError(case)


SIGMA_CASES = ["zero", "mixed", "large", "nan", "negative"]


@pytest.mark.parametrize("case", SIGMA_CASES)
@pytest.mark.parametrize("h,w", [(1, 1), (1, 17), (17, 1), (13, 9), (23, 31)])
def test_restatement_matches_the_oracle_blur(port_oracle, case, h, w):
    sigma = sigma_case(case, h, w, seed=h * 100 + w)
    image = np.random.default_rng(7).random((h, w, 4), dtype=np.float32)
    want = port_oracle.blur(image, sigma).reshape(-1, 4)
    b, nan = blur_matrix(sigma)
    got = apply(b, image)
    assert np.array_equal(np.isnan(want).any(-1), nan)
    assert np.array_equal(np.isnan(want).all(-1), nan)
    bound = np.abs(b) @ np.abs(image.reshape(-1, 4).astype(np.float64))
    err = np.abs(got[~nan] - want[~nan])
    assert np.all(err <= 3e-5 * bound[~nan] + 1e-30), err.max()
    # every row of a pixel with taps sums to one: the blur is a weighted mean
    assert np.allclose(b[~nan].sum(1), 1.0, atol=1e-12)


def test_restatement_band_rows_are_the_full_blur_rows():
    sigma = sigma_case("mixed", 11, 7, seed=3)
    full, nan = blur_matrix(sigma)
    band, band_nan = blur_matrix(sigma, 4, 6)
    assert np.array_equal(band, full[4 * 7:6 * 7]) and np.array_equal(band_nan, nan[4 * 7:6 * 7])


def test_taps_follow_the_kernel():
    first, last, _ = taps(np.array([0.0, 0.01, 1.0, 2.5, -0.2, -1 / 3, -0.5, np.nan, 1e9, np.inf], np.float32))
    assert list(zip(first, last)) == [(0, 0), (-1, 1), (-3, 3), (-8, 8), (0, 0), (0, -1), (0, -1), (0, -1),
                                      (-MAX_TAPS, MAX_TAPS), (-MAX_TAPS, MAX_TAPS)]


def test_adjoint_rejects_bad_arguments_without_a_device():
    buf = ctypes.c_void_p(16)
    f = api.lib.rdc_gaussian_blur_adjoint

    def rejected(*args):
        assert f(*args) == RDC_E_INVALID
        assert "blur adjoint" in api.last_error()

    ok = [buf, buf, buf, buf, 8, 6, 0, 6, None, None]
    for i in range(4):  # null grad_source, grad_dest, sigma, scratch
        args = list(ok)
        args[i] = None
        rejected(*args)
    for w, h, b, e in [(0, 6, 0, 6), (8, 0, 0, 1), (-1, 6, 0, 6), (8, 6, -1, 6), (8, 6, 0, 7), (8, 6, 3, 3), (8, 6, 4, 2)]:
        rejected(buf, buf, buf, buf, w, h, b, e, None, None)
    with pytest.raises(api.RdcError):
        api.gaussian_blur_adjoint(16, 16, 16, 16, 8, 6, 5, 2)
