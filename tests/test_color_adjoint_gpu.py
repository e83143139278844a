"""rdc_render_color_adjoint: the transpose of the render in the colour stops, and the least-squares colour fit on top.

The image rdc_render writes is linear in the colour values (fixed frame parameters): image = A x. The adjoint must be A's
transpose: against A's columns built through the product's own forward path (update_stops + render), by the dot-product
test on every bundled scene and route, across bands, traversals and streams. api.fit_colors must then reach the colours
that made a target, and the least-squares optimum of a target they did not make.
"""
import os

import numpy as np
import pytest

from helpers import scene_ids
from test_scene_update_gpu import SYNTH_PORTALS, synth_portals_xml

pytestmark = pytest.mark.gpu

RDC_E_INVALID = -1


@pytest.fixture(scope="module")
def api():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from raytracingdiffusioncurves_b200 import api as _api

    return _api


def stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


@pytest.fixture(scope="module")
def scene_dict(api, xml_dir, tmp_path_factory):
    """(name, orzan) -> the ingested arrays as numpy (HostScene.to_numpy), each read once."""
    synth = str(tmp_path_factory.mktemp("adjoint") / "synth_portals.xml")
    with open(synth, "w") as fh:
        fh.write(synth_portals_xml(api))
    cache = {}

    def get(name, orzan=True):
        if (name, orzan) not in cache:
            opts = api.default_ingest_options(use_diffusion_curve_save=int(orzan))
            if name == "synth100k":
                host = api.HostScene.from_xml_text(api.synth_xml(100000, 8192, 8192), opts)
            else:
                host = api.HostScene.from_xml_file(synth if name == SYNTH_PORTALS else os.path.join(xml_dir, name), opts)
            cache[(name, orzan)] = host.to_numpy()
        return cache[(name, orzan)]

    return get


def build(api, d, on=None):
    return api.Scene(api.arrays_from_numpy(d), None, stream() if on is None else on)


def params_for(api, d, w, h, n, **kw):
    kw.setdefault("zoom_factor", d["image_height"] / h)
    kw.setdefault("max_trace_depth", 0)
    return api.default_frame_params(w, h, n, **kw)


def render(api, scene, p):
    import torch

    rows = p.row_end - p.row_begin
    image = torch.empty((rows, p.image_width, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, p.image_width), dtype=torch.float32, device="cuda")
    scene.render(p, image.data_ptr(), sigma.data_ptr(), stream())
    torch.cuda.synchronize()
    return image.cpu().numpy()


def adjoint(api, scene, d, p, y, on=None):
    """A^T y for y float [rows, W, 3]: (left, right) float64 [L, 3]."""
    import torch

    g = torch.zeros((y.shape[0], y.shape[1], 4), dtype=torch.float32, device="cuda")
    g[..., :3] = torch.from_numpy(np.ascontiguousarray(y, np.float32)).cuda()
    left = torch.full(d["color_left"].shape, 7.0, dtype=torch.float64, device="cuda")  # overwritten by the call
    right = torch.full(d["color_right"].shape, 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    scene.color_adjoint(p, g.data_ptr(), left.data_ptr(), right.data_ptr(), stream() if on is None else on)
    torch.cuda.synchronize()
    return left.cpu().numpy(), right.cpu().numpy()


def with_colours(d, left, right):
    e = dict(d)
    e["color_left"], e["color_right"] = np.asarray(left, np.float32), np.asarray(right, np.float32)
    return e


def apply_a(api, scene, d, p, left, right):
    """A x through the forward path: new colour values on the handle, then a render (NaN pixels -> 0)."""
    scene.update_stops(api.arrays_from_numpy(with_colours(d, left, right)), stream())
    return render(api, scene, p)[..., :3]


def dot_test(api, d, p, seed=0, scene=None, tol=1e-5):
    rng = np.random.default_rng(seed)
    scene = scene or build(api, d)
    rows = p.row_end - p.row_begin
    y = rng.random((rows, p.image_width, 3)) + 0.1
    left, right = rng.random(d["color_left"].shape) + 0.1, rng.random(d["color_right"].shape) + 0.1
    img = apply_a(api, scene, d, p, left, right)
    lhs = float(np.nansum(img.astype(np.float64) * y.astype(np.float32)))
    gl, gr = adjoint(api, scene, d, p, y)
    rhs = float((gl * left.astype(np.float32)).sum() + (gr * right.astype(np.float32)).sum())
    assert np.isfinite(lhs) and np.isfinite(rhs)
    assert abs(lhs - rhs) <= tol * max(abs(lhs), 1e-30) or lhs == rhs == 0.0, (lhs, rhs)
    return lhs


# ---------------------------------------------------------------------------------------------------------------------
# 1. against the explicit matrix
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["arch.xml", "circles.xml", "weight_demo.xml", "test5.xml", "DiffusionCurvePack/face.xml"])
def test_adjoint_equals_explicit_transpose(api, scene_dict, name):
    d = scene_dict(name)
    p = params_for(api, d, 48, 40, 16)
    scene = build(api, d)
    length = d["color_left"].shape[0]
    cols = {}  # (family, stop) -> column [pixels, 3]: a colour channel only ever sees its own channel
    for fam in (0, 1):
        for j0 in range(0, length, 3):
            stops = [min(j0 + c, length - 1) for c in range(3)]
            x = [np.zeros((length, 3)), np.zeros((length, 3))]
            for c, j in enumerate(stops):
                x[fam][j, c] = 1.0
            img = apply_a(api, scene, d, p, *x)
            for c, j in enumerate(stops):
                cols[(fam, j)] = img[..., c].reshape(-1)
    nan = np.isnan(next(iter(cols.values())))
    a = np.stack([np.where(nan, 0.0, cols[(f, j)]) for f in (0, 1) for j in range(length)], axis=1).astype(np.float64)
    assert np.isfinite(a).all()
    rng = np.random.default_rng(1)
    for _ in range(3):
        y = rng.standard_normal((p.image_height, p.image_width, 3)).astype(np.float32)
        gl, gr = adjoint(api, scene, d, p, y)
        got = np.concatenate([gl, gr])  # [2L, 3]
        y3 = y.reshape(-1, 3).astype(np.float64)
        want = a.T @ y3
        bound = np.abs(a).T @ np.abs(y3)
        assert np.all(np.abs(got - want) <= 1e-5 * bound + 1e-12), np.max(np.abs(got - want) - 1e-5 * bound)


# ---------------------------------------------------------------------------------------------------------------------
# 2. dot-product test
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", scene_ids())
def test_dot_product_every_scene(api, scene_dict, name):
    d = scene_dict(name)
    dot_test(api, d, params_for(api, d, 64, 48, 32))


def test_dot_product_synthetic_portals(api, scene_dict):
    d = scene_dict(SYNTH_PORTALS)
    dot_test(api, d, params_for(api, d, 96, 96, 16))


def test_dot_product_100k_band(api, scene_dict):
    d = scene_dict("synth100k")
    p = params_for(api, d, 2048, 2048, 64, row_begin=1001, row_end=1034)
    scene = build(api, d)
    assert scene.launch_plan(p).mode == api.MODE_LOCAL
    dot_test(api, d, p, scene=scene)


LADY = "DiffusionCurvePack/lady_bug.xml"


@pytest.mark.parametrize("route,name,mode", [(1, LADY, 0), (0, "arch.xml", 1), (3, LADY, 3), (2, LADY, 2)],
                         ids=["tree", "whole-scene-table", "cut-table", "local-table"])
def test_dot_product_routes(api, scene_dict, route, name, mode):
    d = scene_dict(name)
    view = dict(zoom_factor=1.0, offset_x=-30.0, offset_y=20.0) if name == LADY else {}
    p = params_for(api, d, 128, 96, 64, route=route, **view)
    scene = build(api, d)
    assert scene.launch_plan(p).mode == mode  # the render really takes that route
    dot_test(api, d, p, scene=scene)


@pytest.mark.parametrize("case", ["aa_off", "orzan_off", "fractional_n", "n_below_8", "zoom_pan", "far_view", "brute"])
def test_dot_product_params(api, scene_dict, case):
    orzan = case != "orzan_off"
    d = scene_dict("DiffusionCurvePack/face.xml", orzan)
    kw = {"aa_off": dict(use_aa=0), "orzan_off": dict(use_diffusion_curve_save=0), "zoom_pan": dict(zoom_factor=2.5, offset_x=-40.0, offset_y=65.0),
          "far_view": dict(offset_x=1e5, offset_y=-1e5), "brute": dict(traversal=api.TRAVERSAL_BRUTE_FORCE)}.get(case, {})
    n = {"fractional_n": 12.5, "n_below_8": 5}.get(case, 24)
    p = params_for(api, d, 56, 44, n, frame=3, seed=9, **kw)
    assert dot_test(api, d, p) > 0.0  # (from far away the scene still fills some directions of every pixel)


# ---------------------------------------------------------------------------------------------------------------------
# 3. bands, traversals, repeats
# ---------------------------------------------------------------------------------------------------------------------
def close(a, b, rel=1e-12):
    a, b = np.concatenate(a), np.concatenate(b)
    assert np.isfinite(a).all() and np.isfinite(b).all()
    assert np.abs(a - b).max() <= rel * np.abs(a).max(), np.abs(a - b).max() / np.abs(a).max()


@pytest.mark.parametrize("name", ["arch.xml", "DiffusionCurvePack/lady_bug.xml"])
def test_bands_traversals_repeats(api, scene_dict, name):
    d = scene_dict(name)
    w, h = 72, 41
    p = params_for(api, d, w, h, 32)
    scene = build(api, d)
    y = np.random.default_rng(2).random((h, w, 3)) + 0.1
    whole = adjoint(api, scene, d, p, y)
    split = 17  # an odd row: the tile row 16-19 is cut in two
    top = adjoint(api, scene, d, params_for(api, d, w, h, 32, row_begin=0, row_end=split), y[:split])
    bottom = adjoint(api, scene, d, params_for(api, d, w, h, 32, row_begin=split, row_end=h), y[split:])
    close(whole, (top[0] + bottom[0], top[1] + bottom[1]))
    close(whole, adjoint(api, scene, d, params_for(api, d, w, h, 32, traversal=api.TRAVERSAL_BRUTE_FORCE), y))
    close(whole, adjoint(api, scene, d, p, y))
    assert np.abs(np.concatenate(whole)).max() > 0


# ---------------------------------------------------------------------------------------------------------------------
# 4. stream order after rdc_scene_update_stops
# ---------------------------------------------------------------------------------------------------------------------
def test_order_after_update_on_another_stream(api, scene_dict):
    import torch

    d = scene_dict("DiffusionCurvePack/lady_bug.xml")
    p = params_for(api, d, 96, 64, 32)
    e = dict(d)
    for fam in ("color_left", "color_right"):  # move every inner colour stop of every curve 30 % toward the next one
        u = d[fam + "_u"].copy()
        for start, count in d[fam + "_index"]:
            for j in range(start + 1, start + count - 1):
                u[j] += np.float32(0.3) * (u[j + 1] - u[j])
        assert not np.array_equal(u, d[fam + "_u"])
        e[fam + "_u"] = u
    y = np.random.default_rng(3).random((64, 96, 3)) + 0.1
    fresh = adjoint(api, build(api, e), e, p, y)

    scene = build(api, d)
    adjoint(api, scene, d, p, y)  # the handle has launched before
    g = torch.zeros((64, 96, 4), dtype=torch.float32, device="cuda")
    g[..., :3] = torch.from_numpy(y.astype(np.float32)).cuda()
    left = torch.empty(d["color_left"].shape, dtype=torch.float64, device="cuda")
    right = torch.empty_like(left)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    scene.update_stops(api.arrays_from_numpy(e), sa.cuda_stream)
    scene.color_adjoint(p, g.data_ptr(), left.data_ptr(), right.data_ptr(), sb.cuda_stream)  # no host wait in between
    sb.synchronize()
    close(fresh, (left.cpu().numpy(), right.cpu().numpy()))


# ---------------------------------------------------------------------------------------------------------------------
# 5. rejections
# ---------------------------------------------------------------------------------------------------------------------
def test_rejections(api, scene_dict):
    import torch

    d = scene_dict("PortalDemo.xml")
    scene = build(api, d)
    g = torch.zeros((40, 48, 4), dtype=torch.float32, device="cuda")
    out = torch.zeros(d["color_left"].shape, dtype=torch.float64, device="cuda")
    gp, op = g.data_ptr(), out.data_ptr()

    def rejected(p, gptr=gp, lptr=op, rptr=op, words=()):
        with pytest.raises(api.RdcError) as ei:
            scene.color_adjoint(p, gptr, lptr, rptr, stream())
        assert ei.value.code == RDC_E_INVALID
        msg = str(ei.value)
        for word in words:
            assert word in msg, msg

    rejected(params_for(api, d, 48, 40, 8, max_trace_depth=2), words=("portals",))
    rejected(params_for(api, d, 48, 40, 8, strip_stride=2), words=("strips",))
    rejected(params_for(api, d, 48, 40, 8), gptr=0, words=("image_grad",))
    rejected(params_for(api, d, 48, 40, 8), lptr=0, words=("output",))
    rejected(params_for(api, d, 48, 40, 8), rptr=0, words=("output",))
    rejected(params_for(api, d, 48, 40, 0.5), words=("rays per pixel",))
    rejected(params_for(api, d, 48, 40, 8, row_begin=30, row_end=20), words=("band",))
    scene.color_adjoint(params_for(api, d, 48, 40, 8), gp, op, op, stream())  # depth 0 is accepted
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 6. the fit
# ---------------------------------------------------------------------------------------------------------------------
def masked_residual(a, b):
    m = ~(np.isnan(a[..., :3]).any(-1) | np.isnan(b[..., :3]).any(-1))
    return float(np.linalg.norm((a[..., :3] - b[..., :3])[m].astype(np.float64))), m


def grey(d):
    e = dict(d)
    for fam in ("color_left", "color_right"):
        c = d[fam].copy()
        c[: d["n_" + fam]] = 0.5
        e[fam] = c
    return e


@pytest.mark.parametrize("name", ["arch.xml", "weight_demo.xml"])
def test_fit_reaches_the_colours_of_the_target(api, scene_dict, name):
    d = scene_dict(name)
    p = params_for(api, d, 64, 48, 32)
    target = render(api, build(api, d), p)
    start = grey(d)
    scene = build(api, start)
    fitted, res = api.fit_colors(scene, start, p, target, 40)
    assert len(res) >= 2 and res[-1] < res[0]
    assert all(r1 <= r0 for r0, r1 in zip(res, res[1:])), res
    got = render(api, scene, p)  # the handle holds the fitted stops
    again = render(api, build(api, fitted), p)
    assert np.array_equal(np.isnan(got), np.isnan(again)) and np.allclose(np.nan_to_num(got), np.nan_to_num(again), atol=1e-6)
    err, m = masked_residual(got, target)
    mse = err ** 2 / (3 * m.sum())
    psnr = 10 * np.log10(1.0 / max(mse, 1e-30))
    assert psnr >= 60.0, (psnr, res)
    # padding entries and sentinels are untouched
    for fam in ("color_left", "color_right"):
        n = d["n_" + fam]
        assert np.array_equal(fitted[fam][n:], start[fam][n:])


@pytest.mark.parametrize("name", ["arch.xml", "weight_demo.xml"])
def test_fit_is_the_least_squares_optimum_of_a_noisy_target(api, scene_dict, name):
    d = scene_dict(name)
    p = params_for(api, d, 64, 48, 32)
    target = render(api, build(api, d), params_for(api, d, 64, 48, 32, frame=7))  # other rays: not in A's range
    truth, _ = masked_residual(render(api, build(api, d), p), target)
    start = grey(d)
    scene = build(api, start)
    fitted, res = api.fit_colors(scene, start, p, target, 60)
    fit, _ = masked_residual(render(api, scene, p), target)
    assert truth > 0.0
    assert fit <= 1.001 * truth, (fit, truth, res[-3:])
