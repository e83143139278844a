"""The host side of the colour fit: api.cgls against numpy's least squares, api.fit_stops (masking, fixed padding) through
a dense stand-in for render and its transpose, and the argument checks of rdc_render_color_adjoint that need no device."""
import ctypes

import numpy as np
import pytest

from raytracingdiffusioncurves_b200 import api

RDC_E_INVALID = -1


def test_cgls_matches_lstsq_numpy():
    rng = np.random.default_rng(1)
    a = rng.standard_normal((80, 14))
    b = rng.standard_normal(80)
    x0 = rng.standard_normal(14)
    x, res = api.cgls(lambda p: a @ p, lambda r: a.T @ r, b, x0, 30)
    want = np.linalg.lstsq(a, b, rcond=None)[0]
    assert np.allclose(x, want, rtol=1e-9, atol=1e-9)
    assert res[0] == pytest.approx(np.linalg.norm(b - a @ x0))
    assert all(r1 <= r0 * (1 + 1e-12) for r0, r1 in zip(res, res[1:]))
    assert res[-1] == pytest.approx(np.linalg.norm(b - a @ want), rel=1e-9)


def test_cgls_rank_deficient_and_torch():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(2)
    a = rng.standard_normal((40, 6)) @ rng.standard_normal((6, 10))  # rank 6 of 10 columns
    b = rng.standard_normal(40)
    at, bt = torch.from_numpy(a), torch.from_numpy(b)
    x, res = api.cgls(lambda p: at @ p, lambda r: at.T @ r, bt, torch.zeros(10, dtype=torch.float64), 20)
    want = np.linalg.lstsq(a, b, rcond=None)[0]  # minimum norm: CGLS from 0 stays in the row space
    assert isinstance(x, torch.Tensor) and x.dtype == torch.float64
    assert np.allclose(x.numpy(), want, rtol=1e-8, atol=1e-8)
    assert len(res) <= 21


def fake_scene(rng, nl=4, nr=3):
    length = max(nl, nr) + 2
    d = {"n_color_left": nl, "n_color_right": nr,
         "color_left": rng.random((length, 3)).astype(np.float32), "color_right": rng.random((length, 3)).astype(np.float32),
         "color_left_u": np.zeros(length, np.float32), "color_right_u": np.zeros(length, np.float32)}
    return d, length


class DenseOperator:
    """render = M @ (left, right) per channel, with NaN at the pixels no ray hits; adjoint = its transpose there."""

    def __init__(self, rng, rows, w, length):
        self.rows, self.w = rows, w
        self.m = rng.standard_normal((rows * w, 2 * length))
        self.dead = rng.random(rows * w) < 0.15

    def render(self, left, right):
        x = np.concatenate([left, right]).astype(np.float64)  # [2L, 3]
        img = self.m @ x
        img[self.dead] = np.nan
        out = np.ones((self.rows * self.w, 4), np.float32)
        out[:, :3] = img
        return out.reshape(self.rows, self.w, 4)

    def adjoint(self, g):
        g3 = g[..., :3].reshape(-1, 3).astype(np.float64)
        g3[self.dead] = 0.0
        t = self.m.T @ g3
        half = t.shape[0] // 2
        return t[:half], t[half:]


def test_fit_stops_masks_and_keeps_padding():
    rng = np.random.default_rng(3)
    d, length = fake_scene(rng)
    nl, nr = d["n_color_left"], d["n_color_right"]
    rows, w = 7, 9
    op = DenseOperator(rng, rows, w, length)
    target = rng.random((rows, w, 4)).astype(np.float32)
    target[2, 3, 1] = np.nan  # a masked target pixel
    fitted, res = api.fit_stops(d, target, op.render, op.adjoint, 60)

    # padding entries and sentinels keep their values
    assert np.array_equal(fitted["color_left"][nl:], d["color_left"][nl:])
    assert np.array_equal(fitted["color_right"][nr:], d["color_right"][nr:])
    assert fitted["color_left"].dtype == np.float32
    # the input is not modified
    assert fitted["color_left"] is not d["color_left"]

    # the restricted least-squares problem, solved directly: unknowns = real stops, the fixed entries are a constant
    keep = ~(op.dead | np.isnan(target[..., :3]).reshape(-1, 3).any(-1))
    cols = list(range(nl)) + [length + j for j in range(nr)]
    fixed = [j for j in range(2 * length) if j not in cols]
    x_all = np.concatenate([d["color_left"], d["color_right"]]).astype(np.float64)
    b = target[..., :3].reshape(-1, 3).astype(np.float64) - op.m[:, fixed] @ x_all[fixed]
    want = np.linalg.lstsq(op.m[keep][:, cols], b[keep], rcond=None)[0]  # [nl + nr, 3]
    got = np.concatenate([fitted["color_left"][:nl], fitted["color_right"][:nr]])
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5)
    assert all(r1 <= r0 * (1 + 1e-9) for r0, r1 in zip(res, res[1:]))
    best = np.linalg.norm(op.m[keep][:, cols] @ want - b[keep])
    assert res[-1] == pytest.approx(best, rel=1e-5)


def test_fit_stops_masked_pixels_do_not_matter():
    rng = np.random.default_rng(4)
    d, length = fake_scene(rng, 3, 5)
    rows, w = 6, 8
    op = DenseOperator(rng, rows, w, length)
    target = rng.random((rows, w, 3)).astype(np.float32)
    target[0, :2] = np.nan
    a, _ = api.fit_stops(d, target, op.render, op.adjoint, 40)
    other = target.copy()
    other.reshape(-1, 3)[op.dead] = 1e6  # pixels no ray hits: whatever the target says there is ignored
    b, _ = api.fit_stops(d, other, op.render, op.adjoint, 40)
    assert np.array_equal(a["color_left"], b["color_left"]) and np.array_equal(a["color_right"], b["color_right"])


def test_adjoint_rejects_null_arguments_without_a_device():
    p = api.default_frame_params(16, 16, 8)
    buf = ctypes.c_void_p(1)
    assert api.lib.rdc_render_color_adjoint(None, ctypes.byref(p), buf, buf, buf, None) == RDC_E_INVALID
    assert "null scene" in api.last_error()
    assert api.lib.rdc_render_color_adjoint(buf, None, buf, buf, buf, None) == RDC_E_INVALID
    assert "null params" in api.last_error()
