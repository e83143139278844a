"""Fitting the blur stops: rdc_gaussian_blur_sigma_adjoint (the blur's derivative in its sigma map), rdc_render_blur_adjoint
(the render's transpose in the blur values) and api.fit_blur on top.

The sigma derivative must equal the float64 restatement of tests/test_blur_fit_cpu.py (itself checked against central
differences), on small buffers for every band and on crops of the bundled scenes' real sigma maps, with its structure (rows
beyond the reach, the all-zero flag, repeats, NaN pixels). The blur map is linear in the blur values, sigma = A_b x, and the
blur-value adjoint must be A_b's transpose: against explicit columns, by the dot-product test on every scene and route,
across bands, traversals and streams. Chained, they are the gradient of a loss on the blurred frame, and fit_blur must
recover the blur stops of a target.
"""
import numpy as np
import pytest

from helpers import scene_ids
from test_blur_adjoint_cpu import SIGMA_CASES
from test_blur_adjoint_gpu import BLUR_SCENES, blur, cuda, scene_sigma
from test_blur_fit_cpu import bands, frozen_objective_rows, random_case, restated_passes, restated_sigma_adjoint
from test_color_adjoint_gpu import api, build, close, params_for, scene_dict, stream  # noqa: F401 (fixtures)
from test_scene_update_gpu import SYNTH_PORTALS

pytestmark = pytest.mark.gpu

RDC_E_INVALID = -1


def sigma_adjoint(api, grad, source, sigma, band, flag=None, out=None, scratch=None):
    """rdc_gaussian_blur_sigma_adjoint on device buffers ([height, W, 4] gradient and source, [height, W] sigma): [height, W]."""
    import torch

    h, w = sigma.shape
    out = torch.full_like(sigma, 7.0) if out is None else out
    scratch = torch.full((2 * h * w + 1, 4), np.nan, dtype=torch.float32, device="cuda") if scratch is None else scratch
    api.gaussian_blur_sigma_adjoint(out.data_ptr(), grad.data_ptr(), source.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w,
                                    h, band[0], band[1], 0 if flag is None else flag.data_ptr(), stream())
    torch.cuda.synchronize()
    return out


def band_grad(rng, h, w, band, d_nan):
    """a random gradient on the band, zero where the blurred frame is NaN and in a few single channels, NaN off the band
    (never read)"""
    g = rng.standard_normal((h, w, 4)).astype(np.float32)
    g[rng.random((h, w, 4)) < 0.1] = 0.0
    g[d_nan] = 0.0
    g[:band[0]] = np.nan
    g[band[1]:] = np.nan
    return g


def check_against_restatement(got, sigma, source, g, band, tol=1e-5):
    want = restated_sigma_adjoint(sigma, source, g, *band)
    bound = restated_sigma_adjoint(sigma, source, g, *band, absolute=True)
    assert np.isfinite(got).all(), band
    err = np.abs(got - want)
    assert np.all(err <= tol * bound + 1e-30), (band, err.max(), np.abs(want).max())
    return want


# ---------------------------------------------------------------------------------------------------------------------
# 1. the sigma derivative against the restatement
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", SIGMA_CASES)
@pytest.mark.parametrize("h,w", [(1, 1), (1, 17), (17, 1), (13, 9)])
def test_sigma_adjoint_equals_restatement(api, case, h, w):
    sigma, source, _ = random_case(case, h, w, seed=h * 100 + w + 2)
    d_nan = restated_passes(sigma, source)[5]
    reach = int(np.ceil(3 * np.nanmax(sigma))) if np.any(sigma > -1 / 3) else 0
    rng = np.random.default_rng(h + w)
    s_dev, src_dev = cuda(sigma), cuda(source)
    for b, e in bands(h):
        g = band_grad(rng, h, w, (b, e), d_nan)
        got = sigma_adjoint(api, cuda(g), src_dev, s_dev, (b, e)).cpu().numpy().astype(np.float64)
        check_against_restatement(got, sigma, source, g, (b, e))
        assert not np.any(got[:max(0, b - reach)]) and not np.any(got[e + reach:])  # rows beyond the reach: exactly 0
        if case == "zero":
            assert not np.any(got)


def test_sigma_adjoint_structure(api, scene_dict):
    """all-zero flag, repeats, rows beyond the reach, and NaN pixels of the source"""
    import torch

    h, w = 120, 97
    sigma, flag = scene_sigma(api, scene_dict("DiffusionCurvePack/fille.xml"), w, h)
    assert flag.item() > 0
    reach = int(np.ceil(3 * float(torch.nan_to_num(sigma).max())))  # (pixels no ray hits have a NaN sigma)
    gen = torch.Generator(device="cuda").manual_seed(3)
    source = torch.rand((h, w, 4), device="cuda", generator=gen)
    band = (51, 58)
    g = torch.randn((h, w, 4), device="cuda", generator=gen)
    g[band[0]:band[1]][torch.isnan(blur(api, source, sigma, band, flag))] = 0.0
    first = sigma_adjoint(api, g, source, sigma, band, flag)
    again = sigma_adjoint(api, g, source, sigma, band, flag)
    assert torch.equal(first, again)  # no atomics: the same bits
    assert bool(torch.isfinite(first).all()) and float(first.abs().max()) > 0
    assert not bool(first[:max(0, band[0] - reach)].any()) and not bool(first[band[1] + reach:].any())
    zero = torch.zeros((1,), dtype=torch.float32, device="cuda")
    assert not bool(sigma_adjoint(api, g, source, sigma, band, zero).any())  # max_sigma 0: 0 everywhere

    # NaN pixels in the source: the blurred frame is NaN around them; with the gradient zeroed there, the result is finite
    nan_source = source.clone()
    nan_source[40:45, 30:33] = np.nan
    nan_source[55, 60] = np.nan
    d = torch.full_like(source, np.nan)
    scratch = torch.empty_like(source)
    api.gaussian_blur(d.data_ptr(), nan_source.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, h, band[0], band[1],
                      flag.data_ptr(), stream())
    torch.cuda.synchronize()
    dead = torch.isnan(d[band[0]:band[1]])
    assert bool(dead.any()) and not bool(dead.all())
    g2 = g.clone()
    g2[band[0]:band[1]][dead] = 0.0
    got = sigma_adjoint(api, g2, nan_source, sigma, band, flag)
    assert bool(torch.isfinite(got).all()) and float(got.abs().max()) > 0


def crop_case(api, scene_dict, name, ch=40, cw=56):
    """a crop of the scene's 1080p sigma map around its largest sigma, the rendered image there as source"""
    import torch

    d = scene_dict(name)
    w, h = 1920, 1080
    scene = build(api, d)
    p = params_for(api, d, w, h, 4)
    image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
    scene.render(p, image.data_ptr(), sigma.data_ptr(), stream())
    torch.cuda.synchronize()
    s = sigma.cpu().numpy()
    # centred where the blur is large and the image varies (on a flat colour the derivative is 0 throughout)
    lum = np.nan_to_num(image.cpu().numpy()[..., :3].sum(-1))
    gy, gx = np.gradient(lum)
    y, x = np.unravel_index(np.argmax(np.nan_to_num(s) * np.hypot(gx, gy)), s.shape)
    y0, x0 = min(max(0, y - ch // 2), h - ch), min(max(0, x - cw // 2), w - cw)
    return s[y0:y0 + ch, x0:x0 + cw].copy(), image.cpu().numpy()[y0:y0 + ch, x0:x0 + cw].copy()


@pytest.mark.parametrize("name", BLUR_SCENES)
def test_sigma_adjoint_on_real_sigma_maps(api, scene_dict, name):
    sigma, source = crop_case(api, scene_dict, name)
    h, w = sigma.shape
    assert np.nanmax(sigma) > 0
    d_nan = restated_passes(sigma, source)[5]
    rng = np.random.default_rng(7)
    s_dev, src_dev = cuda(sigma), cuda(source)
    for band in [(0, h), (7, 26), (0, 1), (h - 1, h), (19, 20)]:
        g = band_grad(rng, h, w, band, d_nan)
        got = sigma_adjoint(api, cuda(g), src_dev, s_dev, band).cpu().numpy().astype(np.float64)
        check_against_restatement(got, sigma, source, g, band)
        # the directional derivative of sum <G, blur(S, sigma + t v)> at t = 0, taps frozen, by central differences of the
        # float64 restated blur
        v = rng.standard_normal((h, w))
        g0 = np.where(np.isnan(g), 0.0, g)
        step = 1e-5
        fd = (frozen_objective_rows(sigma, source, g0, sigma + step * v).sum()
              - frozen_objective_rows(sigma, source, g0, sigma - step * v).sum()) / (2 * step)
        bound = float(np.abs(restated_sigma_adjoint(sigma, source, g, *band, absolute=True)).ravel() @ np.abs(v).ravel())
        floor = 100 * 2.2e-16 * float(np.abs(g0).sum() * np.nanmax(np.abs(source))) / step  # the differences' own rounding
        assert abs(float(got.ravel() @ v.ravel()) - fd) <= 1e-5 * bound + floor, (band, float(got.ravel() @ v.ravel()), fd)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the render's transpose in the blur values
# ---------------------------------------------------------------------------------------------------------------------
def blur_map(api, scene, p):
    import torch

    rows = p.row_end - p.row_begin
    image = torch.empty((rows, p.image_width, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, p.image_width), dtype=torch.float32, device="cuda")
    scene.render(p, image.data_ptr(), sigma.data_ptr(), stream())
    torch.cuda.synchronize()
    return sigma.cpu().numpy()


def with_blur(d, x):
    e = dict(d)
    e["blur"] = np.asarray(x, np.float32)
    return e


def apply_ab(api, scene, d, p, x):
    """A_b x through the forward path: new blur values on the handle, then the render's blur map"""
    scene.update_stops(api.arrays_from_numpy(with_blur(d, x)), stream())
    return blur_map(api, scene, p)


def blur_adjoint(api, scene, d, p, y, on=None):
    """A_b^T y for y float [rows, W]: float64 [n_blur + 2]"""
    import torch

    g = torch.from_numpy(np.ascontiguousarray(y, np.float32)).cuda()
    out = torch.full(d["blur"].shape, 7.0, dtype=torch.float64, device="cuda")  # overwritten by the call
    torch.cuda.synchronize()
    scene.blur_adjoint(p, g.data_ptr(), out.data_ptr(), stream() if on is None else on)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def dot_test(api, d, p, seed=0, scene=None, tol=1e-5):
    rng = np.random.default_rng(seed)
    scene = scene or build(api, d)
    rows = p.row_end - p.row_begin
    y = rng.random((rows, p.image_width)) + 0.1
    x = rng.random(d["blur"].shape) + 0.1
    s = apply_ab(api, scene, d, p, x)
    lhs = float(np.nansum(s.astype(np.float64) * y.astype(np.float32)))
    rhs = float((blur_adjoint(api, scene, d, p, y) * x.astype(np.float32)).sum())
    assert np.isfinite(lhs) and np.isfinite(rhs)
    assert abs(lhs - rhs) <= tol * max(abs(lhs), 1e-30) or lhs == rhs == 0.0, (lhs, rhs)
    return lhs


@pytest.mark.parametrize("name", ["arch.xml", "weight_demo.xml", "test5.xml", "DiffusionCurvePack/face.xml",
                                  "DiffusionCurvePack/lady_bug.xml"])
def test_blur_adjoint_equals_explicit_transpose(api, scene_dict, name):
    d = scene_dict(name)
    p = params_for(api, d, 48, 40, 16)
    scene = build(api, d)
    length = d["blur"].shape[0]
    cols = []
    for j in range(length):
        x = np.zeros(length)
        x[j] = 1.0
        cols.append(apply_ab(api, scene, d, p, x).reshape(-1))
    nan = np.isnan(cols[0])
    a = np.stack([np.where(nan, 0.0, c) for c in cols], axis=1).astype(np.float64)
    assert np.isfinite(a).all() and np.abs(a).max() > 0
    rng = np.random.default_rng(1)
    for _ in range(3):
        y = rng.standard_normal((p.image_height, p.image_width)).astype(np.float32)
        got = blur_adjoint(api, scene, d, p, y)
        y1 = y.reshape(-1).astype(np.float64)
        want = a.T @ y1
        bound = np.abs(a).T @ np.abs(y1)
        assert np.all(np.abs(got - want) <= 1e-5 * bound + 1e-12), np.max(np.abs(got - want) - 1e-5 * bound)


@pytest.mark.parametrize("name", scene_ids())
def test_blur_dot_product_every_scene(api, scene_dict, name):
    d = scene_dict(name)
    dot_test(api, d, params_for(api, d, 64, 48, 32))


def test_blur_dot_product_synthetic_portals(api, scene_dict):
    d = scene_dict(SYNTH_PORTALS)
    dot_test(api, d, params_for(api, d, 96, 96, 16))


def test_blur_dot_product_100k_band(api, scene_dict):
    d = scene_dict("synth100k")
    p = params_for(api, d, 2048, 2048, 64, row_begin=1001, row_end=1034)
    scene = build(api, d)
    assert scene.launch_plan(p).mode == api.MODE_LOCAL
    dot_test(api, d, p, scene=scene)


LADY = "DiffusionCurvePack/lady_bug.xml"


@pytest.mark.parametrize("route,name,mode", [(1, LADY, 0), (0, "arch.xml", 1), (3, LADY, 3), (2, LADY, 2)],
                         ids=["tree", "whole-scene-table", "cut-table", "local-table"])
def test_blur_dot_product_routes(api, scene_dict, route, name, mode):
    d = scene_dict(name)
    view = dict(zoom_factor=1.0, offset_x=-30.0, offset_y=20.0) if name == LADY else {}
    p = params_for(api, d, 128, 96, 64, route=route, **view)
    scene = build(api, d)
    assert scene.launch_plan(p).mode == mode
    dot_test(api, d, p, scene=scene)


@pytest.mark.parametrize("name", ["arch.xml", "DiffusionCurvePack/lady_bug.xml"])
def test_blur_bands_traversals_repeats(api, scene_dict, name):
    d = scene_dict(name)
    w, h = 72, 41
    p = params_for(api, d, w, h, 32)
    scene = build(api, d)
    y = np.random.default_rng(2).random((h, w)) + 0.1
    whole = blur_adjoint(api, scene, d, p, y)
    split = 17
    top = blur_adjoint(api, scene, d, params_for(api, d, w, h, 32, row_begin=0, row_end=split), y[:split])
    bottom = blur_adjoint(api, scene, d, params_for(api, d, w, h, 32, row_begin=split, row_end=h), y[split:])
    close([whole], [top + bottom])
    close([whole], [blur_adjoint(api, scene, d, params_for(api, d, w, h, 32, traversal=api.TRAVERSAL_BRUTE_FORCE), y)])
    close([whole], [blur_adjoint(api, scene, d, p, y)])
    assert np.abs(whole).max() > 0


def test_blur_order_after_update_on_another_stream(api, scene_dict):
    import torch

    d = scene_dict("DiffusionCurvePack/lady_bug.xml")
    p = params_for(api, d, 96, 64, 32)
    e = dict(d)
    u = d["blur_u"].copy()  # move every inner blur stop of every curve 30 % toward the next one
    for start, count in d["blur_index"]:
        for j in range(start + 1, start + count - 1):
            u[j] += np.float32(0.3) * (u[j + 1] - u[j])
    assert not np.array_equal(u, d["blur_u"])
    e["blur_u"] = u
    y = np.random.default_rng(3).random((64, 96)) + 0.1
    fresh = blur_adjoint(api, build(api, e), e, p, y)

    scene = build(api, d)
    blur_adjoint(api, scene, d, p, y)  # the handle has launched before
    g = torch.from_numpy(y.astype(np.float32)).cuda()
    out = torch.empty(d["blur"].shape, dtype=torch.float64, device="cuda")
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    scene.update_stops(api.arrays_from_numpy(e), sa.cuda_stream)
    scene.blur_adjoint(p, g.data_ptr(), out.data_ptr(), sb.cuda_stream)  # no host wait in between
    sb.synchronize()
    close([fresh], [out.cpu().numpy()])


def test_blur_adjoint_rejections(api, scene_dict):
    import torch

    d = scene_dict("PortalDemo.xml")
    scene = build(api, d)
    g = torch.zeros((40, 48), dtype=torch.float32, device="cuda")
    out = torch.zeros(d["blur"].shape, dtype=torch.float64, device="cuda")
    gp, op = g.data_ptr(), out.data_ptr()

    def rejected(p, gptr=gp, optr=op, words=()):
        with pytest.raises(api.RdcError) as ei:
            scene.blur_adjoint(p, gptr, optr, stream())
        assert ei.value.code == RDC_E_INVALID
        msg = str(ei.value)
        for word in words:
            assert word in msg, msg

    rejected(params_for(api, d, 48, 40, 8, max_trace_depth=2), words=("portals", "blur"))
    rejected(params_for(api, d, 48, 40, 8, strip_stride=2), words=("strips",))
    rejected(params_for(api, d, 48, 40, 8), gptr=0, words=("sigma_grad",))
    rejected(params_for(api, d, 48, 40, 8), optr=0, words=("output",))
    rejected(params_for(api, d, 48, 40, 0.5), words=("rays per pixel",))
    scene.blur_adjoint(params_for(api, d, 48, 40, 8), gp, op, stream())  # depth 0 is accepted
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 3. end to end: the gradient of a loss on the blurred frame in the blur values
# ---------------------------------------------------------------------------------------------------------------------
def blurred_frame_and_gradient(api, scene, d, p, x, target):
    """(1/2 ||blurred - target||^2, its gradient in the blur values) for blur values x (full array), float64"""
    import torch

    rows, w = p.row_end - p.row_begin, p.image_width
    scene.update_stops(api.arrays_from_numpy(with_blur(d, x)), stream())
    flag = torch.zeros((1,), dtype=torch.float32, device="cuda")
    bp = api.FrameParams.from_buffer_copy(p)
    bp.max_sigma = flag.data_ptr()
    image = torch.empty((rows, w, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, w), dtype=torch.float32, device="cuda")
    scene.render(bp, image.data_ptr(), sigma.data_ptr(), stream())
    frame = blur(api, image, sigma, (0, rows), flag)
    r = frame[..., :3].double() - target
    assert bool(torch.isfinite(r).all())
    g = torch.zeros_like(image)
    g[..., :3] = r.float()
    grad_sigma = sigma_adjoint(api, g, image, sigma, (0, rows), flag)
    out = torch.empty(d["blur"].shape, dtype=torch.float64, device="cuda")
    scene.blur_adjoint(p, grad_sigma.data_ptr(), out.data_ptr(), stream())
    torch.cuda.synchronize()
    return 0.5 * float((r * r).sum()), out.cpu().numpy()


@pytest.mark.parametrize("name", ["DiffusionCurvePack/face.xml", "DiffusionCurvePack/fille.xml", "DiffusionCurvePack/lady_bug.xml",
                                  "DiffusionCurvePack/dolphin.xml"])
def test_chained_gradient_matches_central_differences(api, scene_dict, name):
    """Central differences through the fp32 render and blur are a sanity check, not an exact one. Inside the difference
    step some pixels' ceil(3 sigma) steps, and there the blur jumps (the new edge taps weigh up to e^-9 of the centre tap);
    and the objective carries the fp32 rounding of every pixel, which the difference divides by the step. Hence 1e-3
    relative, a step of 1e-2 px per unit of direction (at 1e-3 the rounding alone moved the differences by about 0.008 on
    all four scenes), and directions whose entries have the gradient's signs and random sizes: with random signs the
    derivative along the direction can cancel to a value the rounding then dominates (0.47 on dolphin.xml)."""
    import torch

    d = scene_dict(name)
    p = params_for(api, d, 96, 80, 32, zoom_factor=d["image_height"] / 80 / 2.0, offset_x=10.0, offset_y=-15.0)
    scene = build(api, d)
    nb = int(d["n_blur"])
    rng = np.random.default_rng(4)
    x = d["blur"].astype(np.float64).copy()
    x[:nb] = x[:nb] * 0.7 + 1.0  # every stop away from 0, where the gradient vanishes
    target = torch.rand((80, 96, 3), dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    _, grad = blurred_frame_and_gradient(api, scene, d, p, x, target)
    for _ in range(3):
        v = np.zeros_like(x)
        v[:nb] = np.sign(grad[:nb]) * rng.uniform(0.1, 1.0, nb)
        step = 1e-2
        fp, _ = blurred_frame_and_gradient(api, scene, d, p, x + step * v, target)
        fm, _ = blurred_frame_and_gradient(api, scene, d, p, x - step * v, target)
        fd = (fp - fm) / (2 * step)
        an = float(grad @ v)
        print(f"chained gradient {name}: directional derivative {an:.6g}, central difference {fd:.6g}, "
              f"relative difference {abs(fd - an) / abs(an):.2e}")
        assert abs(fd - an) <= 1e-3 * abs(an), (fd, an)


# ---------------------------------------------------------------------------------------------------------------------
# 4. fit_blur
# ---------------------------------------------------------------------------------------------------------------------
def blurred_target(api, scene, p):
    rows, w = p.row_end - p.row_begin, p.image_width
    host = np.empty((rows, w, 4), np.float32)
    scene.render_frame_to_host(p, True, host.ctypes.data, stream())
    return host


def masked_psnr(a, b):
    m = ~(np.isnan(a[..., :3]).any(-1) | np.isnan(b[..., :3]).any(-1))
    mse = float(((a[..., :3][m].astype(np.float64) - b[..., :3][m]) ** 2).mean())
    return 10 * np.log10(1.0 / mse) if mse > 0 else np.inf


def fit_view(api, d):
    return params_for(api, d, 256, 256, 64)


@pytest.mark.parametrize("start", ["half", "one_px"])
@pytest.mark.parametrize("name", ["DiffusionCurvePack/face.xml", "DiffusionCurvePack/lady_bug.xml"])
def test_fit_blur_recovers_the_blur_of_the_target(api, scene_dict, name, start):
    d = scene_dict(name)
    p = fit_view(api, d)
    scene = build(api, d)
    target = blurred_target(api, scene, p)  # the scene's own blur stops, the same rays
    nb = int(d["n_blur"])
    s = d["blur"].copy()
    s[:nb] = s[:nb] * np.float32(0.5) if start == "half" else np.float32(1.0)
    start_d = with_blur(d, s)
    scene.update_stops(api.arrays_from_numpy(start_d), stream())
    before = masked_psnr(blurred_target(api, scene, p), target)
    fitted, objectives = api.fit_blur(scene, start_d, p, target, iterations=60)
    after = masked_psnr(blurred_target(api, scene, p), target)  # the handle holds the fitted stops
    print(f"fit_blur {name} from {start}: {before:.2f} dB -> {after:.2f} dB in {len(objectives) - 1} iterations")
    assert all(b <= a for a, b in zip(objectives, objectives[1:]))
    assert objectives[-1] < objectives[0]
    assert np.array_equal(fitted["blur"][nb:], d["blur"][nb:]) and np.all(fitted["blur"][:nb] >= 0)
    assert after >= 40.0, (before, after)


def test_alternating_colour_and_blur_fits_recover_both(api, scene_dict):
    d = scene_dict("DiffusionCurvePack/face.xml")
    p = fit_view(api, d)
    nb = int(d["n_blur"])
    changed = dict(d)
    changed["color_left"] = (d["color_left"] * np.float32(0.7) + np.float32(0.15)).astype(np.float32)
    changed["color_right"] = (d["color_right"] * np.float32(0.7) + np.float32(0.1)).astype(np.float32)
    b = d["blur"].copy()
    b[:nb] = b[:nb] * np.float32(1.6) + np.float32(0.5)
    changed["blur"] = b
    scene = build(api, changed)
    target = blurred_target(api, scene, p)
    scene.update_stops(api.arrays_from_numpy(d), stream())
    current = d
    before = masked_psnr(blurred_target(api, scene, p), target)
    for _ in range(4):
        current, _ = api.fit_colors(scene, current, p, target, iterations=30, use_blur=True)
        current, _ = api.fit_blur(scene, current, p, target, iterations=30)
    after = masked_psnr(blurred_target(api, scene, p), target)
    print(f"alternating fit on face.xml: {before:.2f} dB -> {after:.2f} dB")
    assert after >= 40.0, (before, after)
