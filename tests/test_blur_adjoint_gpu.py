"""rdc_gaussian_blur_adjoint: the transpose of the variable-sigma blur, alone and composed with the colour adjoint.

For a fixed sigma map the blur is linear in the image, dest = B source. The adjoint must be B's transpose: against the
float64 restatement of B (tests/test_blur_adjoint_cpu.py), itself checked column by column against the product's own
rdc_gaussian_blur, on every band; by the dot-product test on the real sigma maps of the bundled scenes; and in its
structure (band rows, scratch, in place, repeats, reach, the all-zero flag). Composed with rdc_render_color_adjoint it is
the transpose of the blurred frame rdc_render_frame_to_host writes, and api.fit_colors(use_blur=True) fits that frame.
"""
import os

import numpy as np
import pytest

from test_blur_adjoint_cpu import SIGMA_CASES, blur_matrix, sigma_case, taps
from test_color_adjoint_gpu import build, grey, masked_residual, params_for, with_colours

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from raytracingdiffusioncurves_b200 import api as _api

    return _api


@pytest.fixture(scope="module")
def scene_dict(api, xml_dir):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = api.HostScene.from_xml_file(os.path.join(xml_dir, name)).to_numpy()
        return cache[name]

    return get


def stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def blur(api, image, sigma, band, flag=None):
    """rdc_gaussian_blur of a device image [height, W, 4] on band rows: float32 [rows, W, 4] (band-local)."""
    import torch

    h, w = sigma.shape
    dest = torch.full_like(image, np.nan)
    scratch = torch.empty_like(image)
    api.gaussian_blur(dest.data_ptr(), image.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, h, band[0], band[1],
                      0 if flag is None else flag.data_ptr(), stream())
    return dest[band[0]:band[1]]


def blur_adjoint(api, grad, sigma, band, flag=None, out=None, scratch=None):
    """rdc_gaussian_blur_adjoint of a device gradient [height, W, 4] (rows outside band unread): [height, W, 4]."""
    import torch

    h, w = sigma.shape
    out = torch.full_like(grad, 7.0) if out is None else out
    scratch = torch.empty((h * w + 1, 4), dtype=torch.float32, device="cuda") if scratch is None else scratch
    api.gaussian_blur_adjoint(out.data_ptr(), grad.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, h, band[0], band[1],
                              0 if flag is None else flag.data_ptr(), stream())
    return out


# ---------------------------------------------------------------------------------------------------------------------
# 1. against the explicit matrix
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", SIGMA_CASES)
@pytest.mark.parametrize("h,w", [(1, 1), (1, 17), (17, 1), (13, 9)])
def test_adjoint_equals_explicit_transpose(api, case, h, w):
    import torch

    sigma_np = sigma_case(case, h, w, seed=h * 100 + w + 1)
    sigma = cuda(sigma_np)
    full, nan = blur_matrix(sigma_np)
    # B column by column from the product's forward on unit images (a channel only ever sees its own channel)
    columns = []
    for j in range(h * w):
        unit = torch.zeros((h, w, 4), dtype=torch.float32, device="cuda")
        unit.view(-1, 4)[j] = 1.0
        columns.append(blur(api, unit, sigma, (0, h)).reshape(-1, 4))
    product = torch.stack(columns, 1).cpu().numpy().astype(np.float64)  # [pixels, pixels, 4]
    assert all(np.array_equal(product[..., c], product[..., 0], equal_nan=True) for c in range(4))
    product = product[..., 0]
    assert np.array_equal(np.isnan(product).any(1), nan)
    assert np.all(np.abs(product[~nan] - full[~nan]) <= 3e-6), np.abs(product[~nan] - full[~nan]).max()

    rng = np.random.default_rng(h + w)
    for b in range(h):
        for e in range(b + 1, h + 1):
            g = rng.standard_normal((h, w, 4)).astype(np.float32)
            g[:b] = np.nan  # rows outside the band are never read
            g[e:] = np.nan
            got = blur_adjoint(api, cuda(g), sigma, (b, e)).cpu().numpy().reshape(-1, 4)
            band = full[b * w:e * w]
            gb = g[b:e].reshape(-1, 4).astype(np.float64)
            want = band.T @ gb
            bound = np.abs(band).T @ np.abs(gb)
            assert np.isfinite(got).all(), (b, e)
            assert np.all(np.abs(got - want) <= 3e-5 * bound + 1e-30), (b, e, np.abs(got - want).max())


# ---------------------------------------------------------------------------------------------------------------------
# 2. dot-product test on the real sigma maps
# ---------------------------------------------------------------------------------------------------------------------
def scene_sigma(api, d, w, h, rpp=4):
    """The blur map and max_sigma flag rdc_render writes for the whole scene in a w x h view."""
    import torch

    scene = build(api, d)
    p = params_for(api, d, w, h, rpp)
    flag = torch.zeros((1,), dtype=torch.float32, device="cuda")
    p.max_sigma = flag.data_ptr()
    image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
    scene.render(p, image.data_ptr(), sigma.data_ptr(), stream())
    torch.cuda.synchronize()
    return sigma, flag


BLUR_SCENES = ["DiffusionCurvePack/" + n for n in ("behindthecurtain.xml", "dolphin.xml", "drape.xml", "face.xml", "fille.xml",
                                                   "lady_bug.xml", "lady_bug1024.xml", "zephyr.xml")]


def test_blur_scenes_are_the_bundled_scenes_with_blur(api, xml_dir):
    from helpers import all_scene_files

    with_blur = sorted(os.path.relpath(f, xml_dir) for f in all_scene_files() if api.HostScene.from_xml_file(f).max_blur() > 0)
    assert with_blur == BLUR_SCENES


@pytest.mark.parametrize("name", BLUR_SCENES)
def test_dot_product_real_sigma_maps_1080p(api, scene_dict, name):
    import torch

    w, h = 1920, 1080
    sigma, flag = scene_sigma(api, scene_dict(name), w, h)
    assert flag.item() > 0
    gen = torch.Generator(device="cuda").manual_seed(5)
    s = torch.rand((h, w, 4), device="cuda", generator=gen) + 0.1
    for band in [(0, h), (333, 778), (0, 1), (h - 1, h), (517, 518)]:
        g = torch.rand((h, w, 4), device="cuda", generator=gen) + 0.1
        d = blur(api, s, sigma, band, flag)
        nan = torch.isnan(d)
        g[band[0]:band[1]][nan] = 0.0  # pixels the forward leaves NaN are outside the fit (fit_stops masks them the same way)
        g[:band[0]] = np.nan
        g[band[1]:] = np.nan
        adj = blur_adjoint(api, g, sigma, band, flag)
        assert bool(torch.isfinite(adj).all())
        lhs = float((torch.nan_to_num(d).double() * g[band[0]:band[1]].double()).sum())
        rhs = float((s.double() * adj.double()).sum())
        assert abs(lhs - rhs) <= 1e-5 * abs(lhs), (band, lhs, rhs)


# ---------------------------------------------------------------------------------------------------------------------
# 3. structure
# ---------------------------------------------------------------------------------------------------------------------
def test_scratch_in_place_repeats_and_reach(api, scene_dict):
    import torch

    h, w = 300, 257
    sigma_full, flag = scene_sigma(api, scene_dict("DiffusionCurvePack/fille.xml"), w, h)
    sigma = sigma_full.clone()
    sigma[:140] = torch.clamp(sigma[:140], max=2.0)  # rows around the band: reach ceil(3 * 2) = 6 ...
    sigma[160:] = torch.clamp(sigma[160:], max=2.0)
    sigma[140:160] = torch.clamp(sigma[140:160], max=1.3)  # ... the band's own pixels: 4
    sigma[10, 10], sigma[150, 100] = 2.0, 1.3
    band = (149, 153)
    first, last, _ = taps(sigma.cpu().numpy())
    reach = int(np.max(np.where(first <= last, last, 0)))
    assert reach == 6
    g = torch.randn((h, w, 4), device="cuda")
    g[:band[0]] = np.nan
    g[band[1]:] = np.nan

    scratch = torch.zeros((h * w + 1, 4), device="cuda")
    ref = blur_adjoint(api, g, sigma, band, flag, scratch=scratch).clone()
    assert bool(torch.isfinite(ref).all())
    nz = ref.abs().amax(dim=(1, 2)) > 0
    rows = torch.nonzero(nz).flatten().cpu().numpy()
    # the vertical pass of the band reaches 4 rows, the horizontal pass stays in its row
    assert rows.min() >= band[0] - 4 and rows.max() < band[1] + 4 and len(rows) > band[1] - band[0]
    assert bool((ref[: band[0] - reach] == 0).all()) and bool((ref[band[1] + reach:] == 0).all())

    nan_scratch = torch.full((h * w + 1, 4), np.nan, device="cuda")
    assert torch.equal(blur_adjoint(api, g, sigma, band, flag, scratch=nan_scratch), ref)
    for _ in range(3):
        assert torch.equal(blur_adjoint(api, g, sigma, band, flag), ref)
    inplace = g.clone()
    blur_adjoint(api, inplace, sigma, band, flag, out=inplace)
    assert torch.equal(inplace, ref)

    # the full fille sigma map, in place against out of place, and repeats, bit for bit
    g2 = torch.randn((h, w, 4), device="cuda")
    ref2 = blur_adjoint(api, g2, sigma_full, (0, h), flag).clone()
    assert torch.equal(blur_adjoint(api, g2, sigma_full, (0, h), flag), ref2)
    inplace = g2.clone()
    blur_adjoint(api, inplace, sigma_full, (0, h), flag, out=inplace)
    assert torch.equal(inplace, ref2)


def test_all_zero_flag_is_the_identity_on_the_band(api, scene_dict):
    import torch

    h, w = 96, 128
    sigma, flag = scene_sigma(api, scene_dict("arch.xml"), w, h)
    assert flag.item() == 0.0
    g = torch.randn((h, w, 4), device="cuda")
    for band in [(0, h), (31, 58)]:
        out = blur_adjoint(api, g, sigma, band, flag)
        assert torch.equal(out[band[0]:band[1]], g[band[0]:band[1]])
        assert bool((out[:band[0]] == 0).all()) and bool((out[band[1]:] == 0).all())
        inplace = g.clone()
        blur_adjoint(api, inplace, sigma, band, flag, out=inplace)
        assert torch.equal(inplace, out)


def test_rejections(api):
    import torch

    buf = torch.zeros((4, 4, 4), device="cuda")
    sig = torch.zeros((4, 4), device="cuda")
    p = buf.data_ptr()
    for args in [(p, p, sig.data_ptr(), 0, 4, 4, 0, 4), (p, p, sig.data_ptr(), p, 4, 4, 2, 2), (p, p, 0, p, 4, 4, 0, 4)]:
        with pytest.raises(api.RdcError) as ei:
            api.gaussian_blur_adjoint(*args)
        assert "blur adjoint" in str(ei.value)


# ---------------------------------------------------------------------------------------------------------------------
# 4. composed with the render: the blurred frame
# ---------------------------------------------------------------------------------------------------------------------
def frame_to_host(api, scene, p):
    import torch

    rows = p.row_end - p.row_begin
    host = torch.empty((rows, p.image_width, 4), dtype=torch.float32).pin_memory()
    scene.render_frame_to_host(p, True, host.data_ptr(), stream())
    return host.numpy().copy()


@pytest.mark.parametrize("name", ["DiffusionCurvePack/face.xml", "DiffusionCurvePack/fille.xml",
                                  "DiffusionCurvePack/lady_bug.xml", "DiffusionCurvePack/dolphin.xml"])
@pytest.mark.parametrize("band", [None, (0, 37), (29, 72)], ids=["frame", "top", "bottom"])
def test_dot_product_blurred_frame(api, scene_dict, name, band):
    d = scene_dict(name)
    w, h = 96, 72
    kw = {} if band is None else dict(row_begin=band[0], row_end=band[1])
    p = params_for(api, d, w, h, 32, **kw)
    rows = p.row_end - p.row_begin
    scene = build(api, d)
    rng = np.random.default_rng(11)
    e = with_colours(d, rng.random(d["color_left"].shape) + 0.1, rng.random(d["color_right"].shape) + 0.1)
    left, right = e["color_left"], e["color_right"]
    render, adjoint = api._color_operator(scene, d, p, True, stream())
    fit_image = render(left, right).cpu().numpy()  # puts x on the handle; its blur map is what the adjoint uses
    img = frame_to_host(api, scene, p)  # B A x, from the product's frame path
    assert np.array_equal(fit_image.view(np.uint32), img.view(np.uint32))
    img = img[..., :3]
    y = (rng.random((rows, w, 3)) + 0.1).astype(np.float32)
    y[np.isnan(img).any(-1)] = 0.0
    lhs = float(np.nansum(img.astype(np.float64) * y))
    g = np.zeros((rows, w, 4), np.float32)
    g[..., :3] = y
    gl, gr = adjoint(cuda(g))  # A^T B^T y
    rhs = float((gl * left).sum() + (gr * right).sum())
    assert np.isfinite(lhs) and np.isfinite(rhs) and lhs > 0
    assert abs(lhs - rhs) <= 1e-5 * abs(lhs), (lhs, rhs)


@pytest.mark.parametrize("name", ["DiffusionCurvePack/face.xml", "DiffusionCurvePack/fille.xml"])
def test_fit_blurred_target_from_grey(api, scene_dict, name):
    d = scene_dict(name)
    p = params_for(api, d, 64, 48, 32)
    target = frame_to_host(api, build(api, d), p)
    start = grey(d)
    scene = build(api, start)
    fitted, res = api.fit_colors(scene, start, p, target, 250, use_blur=True)
    assert all(r1 <= r0 for r0, r1 in zip(res, res[1:])), res
    got = frame_to_host(api, scene, p)  # the handle holds the fitted stops
    err, m = masked_residual(got, target)
    psnr = 10 * np.log10(1.0 / max(err ** 2 / (3 * m.sum()), 1e-30))
    assert psnr >= 60.0, (psnr, res[-3:])
    # the fit's own forward on the fitted stops is the frame rdc_render_frame_to_host writes, bit for bit
    render, _ = api._color_operator(scene, start, p, True, stream())
    fit_image = render(fitted["color_left"], fitted["color_right"]).cpu().numpy()
    assert np.array_equal(fit_image.view(np.uint32), frame_to_host(api, scene, p).view(np.uint32))
    # fitting the unblurred image to the same target cannot reach it
    plain_fitted, plain_res = api.fit_colors(build(api, start), start, p, target, 80)
    plain, _ = masked_residual(frame_to_host(api, build(api, plain_fitted), p), target)
    assert res[-1] < plain_res[-1] and err < plain, (res[-1], plain_res[-1], err, plain)


@pytest.mark.parametrize("name", ["DiffusionCurvePack/face.xml", "DiffusionCurvePack/fille.xml"])
def test_fit_blurred_target_of_other_rays(api, scene_dict, name):
    d = scene_dict(name)
    p = params_for(api, d, 64, 48, 32)
    target = frame_to_host(api, build(api, d), params_for(api, d, 64, 48, 32, frame=7))  # other rays: not in the range
    truth, _ = masked_residual(frame_to_host(api, build(api, d), p), target)
    start = grey(d)
    scene = build(api, start)
    api.fit_colors(scene, start, p, target, 250, use_blur=True)
    fit, _ = masked_residual(frame_to_host(api, scene, p), target)
    assert truth > 0.0
    assert fit <= 1.001 * truth, (fit, truth)
