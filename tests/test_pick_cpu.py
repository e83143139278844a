"""Picking without a device: the pixel -> scene point mapping of rdc_view_pixel_to_scene, bit for bit against a float32
restatement of the render's ray origin plus half a pixel, and the argument checks of rdc_scene_pick / _pick_frame."""
import ctypes as C
import math

import numpy as np
import pytest

from raytracingdiffusioncurves_b200 import api

RDC_E_INVALID = -1


def centre(width, height, zoom, off_x, off_y, orzan, ix, iy):
    """render.cu origin_x / origin_y (unsigned arithmetic, then a signed cast) + 0.5 * zoom, one float32 rounding per op."""
    f = np.float32

    def signed(v):  # uint32 wrap-around, then the signed cast
        v %= 1 << 32
        return v - (1 << 32) if v >= 1 << 31 else v

    cx = signed(ix - width // 2)
    cy = signed((height - iy) - height // 2) if orzan else signed(iy - height // 2)
    z = f(zoom)
    x = f(f(f(cx) * z) + f(off_x))
    y = f(f(f(cy) * z) + f(off_y))
    return f(x + f(f(0.5) * z)), f(y + f(f(0.5) * z))


VIEWS = [
    (1920, 1080, 512 / 1080, 0.0, 0.0),
    (17, 5, 1.0, 0.0, 0.0),
    (1, 1, 3.0, 10.0, -4.0),
    (33, 18, -2.5, 123.25, -77.5),   # negative zoom
    (64, 63, 0.0, 5.0, 6.0),         # zoom 0: every pixel is the offset
    (3840, 2160, 0.1234567, -1e4, 2.5e3),
]


@pytest.mark.parametrize("orzan", [0, 1])
@pytest.mark.parametrize("view", VIEWS, ids=lambda v: f"{v[0]}x{v[1]}@{v[2]:g}")
def test_pixel_to_scene_is_the_render_origin_plus_half_a_pixel(view, orzan):
    w, h, zoom, ox, oy = view
    p = api.default_frame_params(w, h, 8, zoom_factor=zoom, offset_x=ox, offset_y=oy, use_diffusion_curve_save=orzan)
    rng = np.random.default_rng(w * 7 + h)
    pix = {(0, 0), (w - 1, h - 1), (w // 2, h // 2), (w // 2 - 1 if w > 1 else 0, h - 1)}
    pix |= {(int(rng.integers(w)), int(rng.integers(h))) for _ in range(40)}
    for ix, iy in sorted(pix):
        x, y = api.view_pixel_to_scene(p, ix, iy)
        wx, wy = centre(w, h, zoom, ox, oy, orzan, ix, iy)
        assert np.float32(x).view(np.uint32) == wx.view(np.uint32), (ix, iy, x, wx)
        assert np.float32(y).view(np.uint32) == wy.view(np.uint32), (ix, iy, y, wy)


def test_pixel_to_scene_rejects_pixels_outside_the_frame():
    p = api.default_frame_params(16, 9, 8)
    x, y = C.c_float(), C.c_float()
    assert api.lib.rdc_view_pixel_to_scene(C.byref(p), 16, 0, C.byref(x), C.byref(y)) == RDC_E_INVALID
    assert "outside" in api.last_error()
    assert api.lib.rdc_view_pixel_to_scene(C.byref(p), 0, 9, C.byref(x), C.byref(y)) == RDC_E_INVALID
    assert api.lib.rdc_view_pixel_to_scene(None, 0, 0, C.byref(x), C.byref(y)) == RDC_E_INVALID
    assert "null" in api.last_error()
    assert api.lib.rdc_view_pixel_to_scene(C.byref(p), 0, 0, None, C.byref(y)) == RDC_E_INVALID


def test_pick_record_layout():
    assert api.PICK_DTYPE.itemsize == 32
    assert list(api.PICK_DTYPE.names) == ["chord", "segment", "curve", "flags", "u", "distance", "x", "y"]


BUF = C.create_string_buffer(64)  # stands for a device buffer: every call below is rejected before touching it
PTR = C.cast(BUF, C.c_void_p)


@pytest.mark.parametrize("args,word", [
    ((None, PTR, 4, math.inf, 1, None, None, None), "out"),
    ((None, None, 4, math.inf, 1, PTR, None, None), "points"),
    ((None, PTR, 4, math.nan, 1, PTR, None, None), "max_distance"),
    ((None, PTR, 4, 0.0, 1, PTR, None, None), "max_distance"),
    ((None, PTR, 4, -1.0, 1, PTR, None, None), "max_distance"),
    ((None, PTR, 4, math.inf, 1, PTR, None, None), "scene"),
    ((None, None, 0, 5.0, 1, PTR, None, None), "scene"),
])
def test_pick_validation(args, word):
    assert api.lib.rdc_scene_pick(*args) == RDC_E_INVALID
    assert word in api.last_error()


def frame(**kw):
    return api.default_frame_params(40, 30, 8, **kw)


@pytest.mark.parametrize("params,md,out,word", [
    (None, math.inf, PTR, "params"),
    (frame(), math.inf, None, "out"),
    (frame(), math.nan, PTR, "max_distance"),
    (frame(), -2.0, PTR, "max_distance"),
    (frame(row_begin=7, row_end=7), math.inf, PTR, "band"),
    (frame(row_begin=8, row_end=7), math.inf, PTR, "band"),
    (frame(row_end=31), math.inf, PTR, "band"),
    (api.default_frame_params(0, 30, 8), math.inf, PTR, "band"),
    (frame(strip_stride=2), math.inf, PTR, "strip"),
    (frame(), math.inf, PTR, "scene"),
], ids=["params", "out", "nan", "negative", "empty", "inverted", "beyond", "no-width", "strips", "scene"])
def test_pick_frame_validation(params, md, out, word):
    assert api.lib.rdc_scene_pick_frame(None, C.byref(params) if params is not None else None, md, out, None, None) == RDC_E_INVALID
    assert word in api.last_error()
