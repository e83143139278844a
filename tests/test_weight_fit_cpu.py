"""Fitting the weight and exponent stops, host side: the argument checks of rdc_render_weight_adjoint that need no device, and
the unknowns of api.fit_weights (api.weight_unknowns): which entries are unknowns, the log mapping of the weights, the bounds,
the gradient's chain rule, and that everything else keeps the scene's values.
"""
import ctypes

import numpy as np

from raytracingdiffusioncurves_b200 import api

RDC_E_INVALID = -1


def test_render_weight_adjoint_rejects_null_arguments_without_a_device():
    p = api.default_frame_params(16, 16, 8)
    buf = ctypes.c_void_p(1)
    f = api.lib.rdc_render_weight_adjoint

    def rejected(args, words):
        assert f(*args) == RDC_E_INVALID
        assert words in api.last_error(), api.last_error()

    rejected((None, ctypes.byref(p), buf, buf, buf, buf, None), "null scene")
    rejected((buf, None, buf, buf, buf, buf, None), "null params")
    rejected((buf, ctypes.byref(p), buf, buf, None, buf, None), "null output array")
    rejected((buf, ctypes.byref(p), buf, buf, buf, None, None), "null output array")
    rejected((buf, ctypes.byref(p), None, None, buf, buf, None), "null image_grad and sigma_grad")


def scene_like(n_weight, n_degree, seed=0):
    """the weight and exponent entries of a HostScene.to_numpy() dictionary: real stops, one padding entry, sentinels"""
    rng = np.random.default_rng(seed)
    weight = np.concatenate([rng.uniform(0.2, 3.0, n_weight), [0.0, 0.0, 0.0]]).astype(np.float32)
    degree = np.concatenate([rng.uniform(0.0, 2.0, n_degree), [0.0, 0.0]]).astype(np.float32)
    weight[n_weight + 1:] = np.float32(7.5)  # sentinels with a value of their own, to see that they are kept
    degree[n_degree:] = np.float32(-4.25)
    return {"n_weight": n_weight, "weight": weight, "n_weight_degree": n_degree, "weight_degree": degree}


def test_weight_unknowns_round_trip():
    d = scene_like(7, 5)
    x0, lower, stops, chain = api.weight_unknowns(d)
    assert x0.dtype == np.float64 and x0.shape == (12,) and lower.shape == (12,)
    weight, degree = stops(x0)
    assert weight.dtype == np.float32 and degree.dtype == np.float32
    assert np.array_equal(weight, d["weight"]) and np.array_equal(degree, d["weight_degree"])
    assert np.allclose(x0[:7], np.log(d["weight"][:7].astype(np.float64)), rtol=0, atol=1e-15)
    assert np.array_equal(x0[7:], d["weight_degree"][:5].astype(np.float64))


def test_weight_unknowns_keep_zero_weights_padding_and_sentinels():
    d = scene_like(6, 4, seed=1)
    d["weight"][1] = 0.0
    d["weight"][4] = -0.5
    x0, lower, stops, chain = api.weight_unknowns(d)
    assert x0.shape == (4 + 4,)  # stops 1 and 4 are not unknowns
    x = x0 + np.random.default_rng(2).uniform(-1.0, 1.0, x0.shape)
    weight, degree = stops(x)
    free = [0, 2, 3, 5]
    assert np.array_equal(weight[[1, 4]], d["weight"][[1, 4]])
    assert np.array_equal(weight[6:], d["weight"][6:]) and np.array_equal(degree[4:], d["weight_degree"][4:])
    assert np.allclose(weight[free], np.exp(x[:4]), rtol=1e-7) and np.all(weight[free] > 0)
    assert np.array_equal(degree[:4], x[4:].astype(np.float32))


def test_weight_unknowns_bounds():
    d = scene_like(3, 4, seed=3)
    d["weight_degree"][:4] = np.float32([0.5, -0.25, 0.0, 2.0])
    x0, lower, stops, chain = api.weight_unknowns(d)
    assert np.all(np.isneginf(lower[:3]))
    assert np.array_equal(lower[3:], [0.0, -0.25, 0.0, 0.0])  # min(0, start): an exponent below 0 may stay where it is
    assert np.all(x0 >= lower)


def test_weight_unknowns_chain_rule():
    """the gradient in the logs is weight * dL/dweight, the exponents' passes through; entries that are not unknowns drop"""
    d = scene_like(5, 3, seed=4)
    d["weight"][2] = 0.0
    x0, lower, stops, chain = api.weight_unknowns(d)
    rng = np.random.default_rng(5)
    gw, ge = rng.standard_normal(d["weight"].shape), rng.standard_normal(d["weight_degree"].shape)
    x = x0 + 0.3
    got = chain(x, gw, ge)
    free = [0, 1, 3, 4]
    weight = stops(x)[0]
    assert np.allclose(got[:4], weight[free].astype(np.float64) * gw[free], rtol=1e-15)
    assert np.array_equal(got[4:], ge[:3])
    # against central differences of a loss that is linear in the two arrays
    def loss(x):
        w, e = stops(x)
        return float(w.astype(np.float64) @ gw + e.astype(np.float64) @ ge)
    for j in range(x.size):
        v = np.zeros_like(x)
        v[j] = 1e-3
        fd = (loss(x + v) - loss(x - v)) / 2e-3
        assert abs(fd - got[j]) <= 1e-4 * max(1.0, abs(got[j])), (j, fd, got[j])
