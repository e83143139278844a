"""Fitting the weight and exponent stops: rdc_render_weight_adjoint (the derivative of the render's image and blur map in
those stops, as a vector-Jacobian product) and api.fit_weights on top.

The frame does not change when every weight is scaled by one factor, so sum_k weight[k] grad_weight[k] = 0 for any gradient:
checked on every scene and route. The derivative must agree with central differences through update_stops + rdc_render, per
entry and along directions, and, chained through the blur's two adjoints, with central differences of a loss on the blurred
frame. It must be the same across bands, traversals, repeats and streams, and fit_weights must recover the weights and
exponents of a target.
"""
import numpy as np
import pytest

from helpers import scene_ids
from test_blur_adjoint_gpu import blur
from test_blur_fit_gpu import blurred_target, fit_view, masked_psnr, sigma_adjoint
from test_color_adjoint_gpu import api, build, close, params_for, scene_dict, stream  # noqa: F401 (fixtures)
from test_scene_update_gpu import SYNTH_PORTALS

pytestmark = pytest.mark.gpu

RDC_E_INVALID = -1
LADY = "DiffusionCurvePack/lady_bug.xml"


def with_weights(d, weight, degree):
    e = dict(d)
    e["weight"], e["weight_degree"] = np.asarray(weight, np.float32), np.asarray(degree, np.float32)
    return e


def moved(d, seed):
    """the scene's stops moved off their defaults (all weights 1 and exponents 0.5 on most scenes): real weights times a
    factor in [0.5, 2], real exponents plus [0, 0.5]"""
    rng = np.random.default_rng(seed)
    nw, ne = int(d["n_weight"]), int(d["n_weight_degree"])
    w, e = d["weight"].copy(), d["weight_degree"].copy()
    w[:nw] *= np.exp2(rng.uniform(-1.0, 1.0, nw)).astype(np.float32)
    e[:ne] += rng.uniform(0.0, 0.5, ne).astype(np.float32)
    return w, e


def frame(api, scene, d, p, weight, degree):
    """(image [rows, W, 3], blur map [rows, W]) in float64 for the given weight and exponent arrays"""
    import torch

    scene.update_stops(api.arrays_from_numpy(with_weights(d, weight, degree)), stream())
    rows = p.row_end - p.row_begin
    image = torch.empty((rows, p.image_width, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, p.image_width), dtype=torch.float32, device="cuda")
    scene.render(p, image.data_ptr(), sigma.data_ptr(), stream())
    torch.cuda.synchronize()
    return image.cpu().numpy()[..., :3].astype(np.float64), sigma.cpu().numpy().astype(np.float64)


def weight_adjoint(api, scene, d, p, y, ys, on=None):
    """the gradient for an image gradient y [rows, W, 3] and a sigma gradient ys [rows, W] (either None): float64 arrays
    laid out like d's weight and weight_degree"""
    import torch

    gp = sp = 0
    if y is not None:
        g = torch.zeros((y.shape[0], y.shape[1], 4), dtype=torch.float32, device="cuda")
        g[..., :3] = torch.from_numpy(np.ascontiguousarray(y, np.float32)).cuda()
        gp = g.data_ptr()
    if ys is not None:
        s = torch.from_numpy(np.ascontiguousarray(ys, np.float32)).cuda()
        sp = s.data_ptr()
    gw = torch.full(d["weight"].shape, 7.0, dtype=torch.float64, device="cuda")  # overwritten by the call
    ge = torch.full(d["weight_degree"].shape, 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    scene.weight_adjoint(p, gp, sp, gw.data_ptr(), ge.data_ptr(), stream() if on is None else on)
    torch.cuda.synchronize()
    return gw.cpu().numpy(), ge.cpu().numpy()


def random_gradients(rng, p):
    rows = p.row_end - p.row_begin
    return (rng.standard_normal((rows, p.image_width, 3)).astype(np.float32),
            rng.standard_normal((rows, p.image_width)).astype(np.float32))


# ---------------------------------------------------------------------------------------------------------------------
# 1. homogeneity: scaling every weight leaves the frame unchanged
# ---------------------------------------------------------------------------------------------------------------------
def homogeneity(api, d, p, seed=0, scene=None):
    rng = np.random.default_rng(seed)
    scene = scene or build(api, d)
    w, e = moved(d, seed)
    scene.update_stops(api.arrays_from_numpy(with_weights(d, w, e)), stream())
    y, ys = random_gradients(rng, p)
    gw, ge = weight_adjoint(api, scene, d, p, y, ys)
    assert np.isfinite(gw).all() and np.isfinite(ge).all()
    terms = w.astype(np.float64) * gw
    assert np.abs(terms).sum() > 0 and np.abs(ge).sum() > 0, "the gradient should not vanish"
    assert abs(terms.sum()) <= 1e-5 * np.abs(terms).sum(), (terms.sum(), np.abs(terms).sum())
    return terms


@pytest.mark.parametrize("name", scene_ids())
def test_homogeneity_every_scene(api, scene_dict, name):
    d = scene_dict(name)
    homogeneity(api, d, params_for(api, d, 64, 48, 32))


def test_homogeneity_synthetic_portals(api, scene_dict):
    d = scene_dict(SYNTH_PORTALS)
    homogeneity(api, d, params_for(api, d, 96, 96, 16))


def test_homogeneity_100k_band(api, scene_dict):
    d = scene_dict("synth100k")
    p = params_for(api, d, 2048, 2048, 64, row_begin=1001, row_end=1034)
    scene = build(api, d)
    assert scene.launch_plan(p).mode == api.MODE_LOCAL
    homogeneity(api, d, p, scene=scene)


@pytest.mark.parametrize("route,name,mode", [(1, LADY, 0), (0, "arch.xml", 1), (3, LADY, 3), (2, LADY, 2)],
                         ids=["tree", "whole-scene-table", "cut-table", "local-table"])
def test_homogeneity_routes(api, scene_dict, route, name, mode):
    d = scene_dict(name)
    view = dict(zoom_factor=1.0, offset_x=-30.0, offset_y=20.0) if name == LADY else {}
    p = params_for(api, d, 128, 96, 64, route=route, **view)
    scene = build(api, d)
    assert scene.launch_plan(p).mode == mode
    homogeneity(api, d, p, scene=scene)


# ---------------------------------------------------------------------------------------------------------------------
# 2. against central differences through update_stops + rdc_render
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["weight_demo.xml", "arch.xml"])
def test_every_entry_matches_central_differences(api, scene_dict, name):
    """Nothing steps as the weights and exponents move (the hits stay), so the differences see the smooth map; their error
    is the fp32 rounding of the pixels a stop moves, over the step, and the step's h^2 term."""
    d = scene_dict(name)
    p = params_for(api, d, 48, 40, 16)
    scene = build(api, d)
    w, e = moved(d, 1)
    y, ys = random_gradients(np.random.default_rng(2), p)
    scene.update_stops(api.arrays_from_numpy(with_weights(d, w, e)), stream())
    gw, ge = weight_adjoint(api, scene, d, p, y, ys)
    img0, sig0 = frame(api, scene, d, p, w, e)
    live = ~(np.isnan(img0).any(-1) | np.isnan(sig0))
    yd, ysd = y.astype(np.float64), ys.astype(np.float64)
    worst = 0.0
    for fam, x, got in (("weight", w, gw), ("weight_degree", e, ge)):
        for k in range(x.shape[0]):
            h = 1e-3 * max(abs(float(x[k])), 1.0) if fam == "weight" else 1e-3
            xp, xm = x.copy(), x.copy()
            xp[k] += np.float32(h)
            xm[k] -= np.float32(h)
            step = float(xp[k]) - float(xm[k])  # the float32 step actually taken
            args = (xp, e) if fam == "weight" else (w, xp)
            ip, sp = frame(api, scene, d, p, *args)
            args = (xm, e) if fam == "weight" else (w, xm)
            im, sm = frame(api, scene, d, p, *args)
            ji, js = (ip - im) / step, (sp - sm) / step  # the column of the Jacobian
            ji, js = np.where(live[..., None], ji, 0.0), np.where(live, js, 0.0)
            fd = float((yd * ji).sum() + (ysd * js).sum())
            bound = float((np.abs(yd) * np.abs(ji)).sum() + (np.abs(ysd) * np.abs(js)).sum())
            # the rounding of the moved pixels' fp32 values, over the step
            moved_px = live & ((ip != im).any(-1) | (sp != sm))
            floor = 4 * 6e-8 * float((np.abs(yd) * np.abs(img0)).sum(-1)[moved_px].sum()
                                     + (np.abs(ysd) * np.abs(sig0))[moved_px].sum()) / step
            err = abs(float(got[k]) - fd)
            worst = max(worst, err / max(bound, 1e-300))
            assert err <= 1e-3 * bound + floor, (fam, k, float(got[k]), fd, bound, floor)
    print(f"per-entry derivative {name}: largest difference {worst:.2e} of the entry's bound")


@pytest.mark.parametrize("family", ["weight", "weight_degree"])
@pytest.mark.parametrize("name", ["weight_demo.xml", "arch.xml", LADY, "DiffusionCurvePack/face.xml",
                                  "DiffusionCurvePack/dolphin.xml"])
def test_directional_derivative_matches_central_differences(api, scene_dict, name, family):
    """Directions have the gradient's signs and random sizes (test_chained_gradient_matches_central_differences of
    test_blur_fit_gpu.py says why): along them the derivative is a sum of terms of one sign and cannot cancel to rounding."""
    d = scene_dict(name)
    p = params_for(api, d, 96, 80, 32, zoom_factor=d["image_height"] / 80 / 2.0, offset_x=10.0, offset_y=-15.0)
    scene = build(api, d)
    w, e = moved(d, 3)
    rng = np.random.default_rng(4)
    y, ys = random_gradients(rng, p)
    scene.update_stops(api.arrays_from_numpy(with_weights(d, w, e)), stream())
    gw, ge = weight_adjoint(api, scene, d, p, y, ys)
    yd, ysd = y.astype(np.float64), ys.astype(np.float64)
    n = int(d["n_" + family])
    x, g = (w, gw) if family == "weight" else (e, ge)
    for _ in range(2):
        v = np.zeros(x.shape)
        v[:n] = np.sign(g[:n]) * rng.uniform(0.1, 1.0, n) * (x[:n] if family == "weight" else 1.0)
        h = 1e-3

        def at(t):
            xt = (x + t * v).astype(np.float32)
            return frame(api, scene, d, p, xt, e) if family == "weight" else frame(api, scene, d, p, w, xt)

        (ip, sp), (im, sm) = at(h), at(-h)
        live = ~(np.isnan(ip).any(-1) | np.isnan(sp) | np.isnan(im).any(-1) | np.isnan(sm))
        fd = float((np.where(live[..., None], yd * (ip - im), 0.0)).sum() + np.where(live, ysd * (sp - sm), 0.0).sum()) / (2 * h)
        an = float(g @ v)
        print(f"directional derivative {name} {family}: {an:.6g}, central difference {fd:.6g}, relative difference "
              f"{abs(fd - an) / abs(an):.2e}")
        assert abs(fd - an) <= 1e-3 * abs(an), (fd, an)


# ---------------------------------------------------------------------------------------------------------------------
# 3. through the blur
# ---------------------------------------------------------------------------------------------------------------------
def blurred_loss_and_gradient(api, scene, d, p, w, e, target):
    """(1/2 ||blurred - target||^2, its gradient in the weight and exponent arrays), float64: blur adjoint and sigma adjoint
    of the residual, then the weight adjoint with both"""
    import torch

    rows, wd = p.row_end - p.row_begin, p.image_width
    scene.update_stops(api.arrays_from_numpy(with_weights(d, w, e)), stream())
    flag = torch.zeros((1,), dtype=torch.float32, device="cuda")
    bp = api.FrameParams.from_buffer_copy(p)
    bp.max_sigma = flag.data_ptr()
    image = torch.empty((rows, wd, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, wd), dtype=torch.float32, device="cuda")
    scene.render(bp, image.data_ptr(), sigma.data_ptr(), stream())
    out = blur(api, image, sigma, (0, rows), flag)
    r = out[..., :3].double() - target
    assert bool(torch.isfinite(r).all())
    g = torch.zeros_like(image)
    g[..., :3] = r.float()
    grad_sigma = sigma_adjoint(api, g, image, sigma, (0, rows), flag)
    grad_image = torch.empty_like(image)
    scratch = torch.empty((rows * wd + 1, 4), dtype=torch.float32, device="cuda")
    api.gaussian_blur_adjoint(grad_image.data_ptr(), g.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), wd, rows, 0, rows,
                              flag.data_ptr(), stream())
    gw = torch.empty(d["weight"].shape, dtype=torch.float64, device="cuda")
    ge = torch.empty(d["weight_degree"].shape, dtype=torch.float64, device="cuda")
    scene.weight_adjoint(p, grad_image.data_ptr(), grad_sigma.data_ptr(), gw.data_ptr(), ge.data_ptr(), stream())
    torch.cuda.synchronize()
    return 0.5 * float((r * r).sum()), gw.cpu().numpy(), ge.cpu().numpy()


@pytest.mark.parametrize("name", ["DiffusionCurvePack/face.xml", "DiffusionCurvePack/fille.xml", LADY,
                                  "DiffusionCurvePack/dolphin.xml"])
def test_chained_gradient_through_the_blur(api, scene_dict, name):
    """As in test_blur_fit_gpu.py: through the blur a pixel's ceil(3 sigma) can step inside the difference step, so the bar
    is 1e-3 with directions that carry the gradient's signs."""
    import torch

    d = scene_dict(name)
    p = params_for(api, d, 96, 80, 32, zoom_factor=d["image_height"] / 80 / 2.0, offset_x=10.0, offset_y=-15.0)
    scene = build(api, d)
    w, e = moved(d, 5)
    rng = np.random.default_rng(6)
    target = torch.rand((80, 96, 3), dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    _, gw, ge = blurred_loss_and_gradient(api, scene, d, p, w, e, target)
    for family in ("weight", "weight_degree"):
        n = int(d["n_" + family])
        x, g = (w, gw) if family == "weight" else (e, ge)
        v = np.zeros(x.shape)
        v[:n] = np.sign(g[:n]) * rng.uniform(0.1, 1.0, n) * (x[:n] if family == "weight" else 1.0)
        h = 1e-3

        def at(t):
            xt = (x + t * v).astype(np.float32)
            args = (xt, e) if family == "weight" else (w, xt)
            return blurred_loss_and_gradient(api, scene, d, p, *args, target)[0]

        fd = (at(h) - at(-h)) / (2 * h)
        an = float(g @ v)
        print(f"chained gradient {name} {family}: directional derivative {an:.6g}, central difference {fd:.6g}, "
              f"relative difference {abs(fd - an) / abs(an):.2e}")
        assert abs(fd - an) <= 1e-3 * abs(an), (fd, an)


# ---------------------------------------------------------------------------------------------------------------------
# 4. bands, traversals, repeats, streams
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["arch.xml", LADY])
def test_bands_traversals_repeats(api, scene_dict, name):
    d = scene_dict(name)
    wd, h = 72, 41
    p = params_for(api, d, wd, h, 32)
    scene = build(api, d)
    w, e = moved(d, 7)
    scene.update_stops(api.arrays_from_numpy(with_weights(d, w, e)), stream())
    y, ys = random_gradients(np.random.default_rng(8), p)
    whole = weight_adjoint(api, scene, d, p, y, ys)
    split = 17  # an odd row: the tile row 16-19 is cut in two
    top = weight_adjoint(api, scene, d, params_for(api, d, wd, h, 32, row_begin=0, row_end=split), y[:split], ys[:split])
    bottom = weight_adjoint(api, scene, d, params_for(api, d, wd, h, 32, row_begin=split, row_end=h), y[split:], ys[split:])
    close(whole, (top[0] + bottom[0], top[1] + bottom[1]))
    close(whole, weight_adjoint(api, scene, d, params_for(api, d, wd, h, 32, traversal=api.TRAVERSAL_BRUTE_FORCE), y, ys))
    close(whole, weight_adjoint(api, scene, d, p, y, ys))
    assert np.abs(np.concatenate(whole)).max() > 0
    # a null gradient is a zero one
    zero_sigma = weight_adjoint(api, scene, d, p, y, np.zeros_like(ys))
    close(zero_sigma, weight_adjoint(api, scene, d, p, y, None))
    zero_image = weight_adjoint(api, scene, d, p, np.zeros_like(y), ys)
    close(zero_image, weight_adjoint(api, scene, d, p, None, ys))


def test_order_after_update_on_another_stream(api, scene_dict):
    import torch

    d = scene_dict(LADY)
    p = params_for(api, d, 96, 64, 32)
    w, e = moved(d, 9)
    changed = with_weights(d, w, e)
    y, ys = random_gradients(np.random.default_rng(10), p)
    fresh = weight_adjoint(api, build(api, changed), changed, p, y, ys)

    scene = build(api, d)
    weight_adjoint(api, scene, d, p, y, ys)  # the handle has launched before
    g = torch.zeros((64, 96, 4), dtype=torch.float32, device="cuda")
    g[..., :3] = torch.from_numpy(y).cuda()
    s = torch.from_numpy(ys).cuda()
    gw = torch.empty(d["weight"].shape, dtype=torch.float64, device="cuda")
    ge = torch.empty(d["weight_degree"].shape, dtype=torch.float64, device="cuda")
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    scene.update_stops(api.arrays_from_numpy(changed), sa.cuda_stream)
    scene.weight_adjoint(p, g.data_ptr(), s.data_ptr(), gw.data_ptr(), ge.data_ptr(), sb.cuda_stream)  # no host wait
    sb.synchronize()
    close(fresh, (gw.cpu().numpy(), ge.cpu().numpy()))


# ---------------------------------------------------------------------------------------------------------------------
# 5. rejections
# ---------------------------------------------------------------------------------------------------------------------
def test_rejections(api, scene_dict):
    import torch

    d = scene_dict("PortalDemo.xml")
    scene = build(api, d)
    g = torch.zeros((40, 48, 4), dtype=torch.float32, device="cuda")
    s = torch.zeros((40, 48), dtype=torch.float32, device="cuda")
    out = torch.zeros(d["weight"].shape, dtype=torch.float64, device="cuda")
    gp, sp, op = g.data_ptr(), s.data_ptr(), out.data_ptr()

    def rejected(p, gptr=gp, sptr=sp, wptr=op, eptr=op, words=()):
        with pytest.raises(api.RdcError) as ei:
            scene.weight_adjoint(p, gptr, sptr, wptr, eptr, stream())
        assert ei.value.code == RDC_E_INVALID
        msg = str(ei.value)
        for word in words:
            assert word in msg, msg

    rejected(params_for(api, d, 48, 40, 8, max_trace_depth=2), words=("portals", "weight"))
    rejected(params_for(api, d, 48, 40, 8, strip_stride=2), words=("strips",))
    rejected(params_for(api, d, 48, 40, 8), gptr=0, sptr=0, words=("image_grad and sigma_grad",))
    rejected(params_for(api, d, 48, 40, 8), wptr=0, words=("output",))
    rejected(params_for(api, d, 48, 40, 8), eptr=0, words=("output",))
    rejected(params_for(api, d, 48, 40, 0.5), words=("rays per pixel",))
    scene.weight_adjoint(params_for(api, d, 48, 40, 8), gp, sp, op, op, stream())  # depth 0 is accepted
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 6. fit_weights
# ---------------------------------------------------------------------------------------------------------------------
def unblurred_target(api, scene, p):
    rows, w = p.row_end - p.row_begin, p.image_width
    host = np.empty((rows, w, 4), np.float32)
    scene.render_frame_to_host(p, False, host.ctypes.data, stream())
    return host


def changed_weights(d, seed):
    """the start of the fits: weights times a seeded factor in [0.5, 2], exponents + 0.3"""
    rng = np.random.default_rng(seed)
    nw, ne = int(d["n_weight"]), int(d["n_weight_degree"])
    w, e = d["weight"].copy(), d["weight_degree"].copy()
    w[:nw] *= np.exp2(rng.uniform(-1.0, 1.0, nw)).astype(np.float32)
    e[:ne] += np.float32(0.3)
    return with_weights(d, w, e)


@pytest.mark.parametrize("name,use_blur", [("weight_demo.xml", False), (LADY, False), ("DiffusionCurvePack/face.xml", True)])
def test_fit_weights_recovers_the_target(api, scene_dict, name, use_blur):
    d = scene_dict(name)
    p = fit_view(api, d)
    scene = build(api, d)
    shot = blurred_target if use_blur else unblurred_target
    target = shot(api, scene, p)  # the scene's own stops, the same rays
    start = changed_weights(d, 11)
    scene.update_stops(api.arrays_from_numpy(start), stream())
    before = masked_psnr(shot(api, scene, p), target)
    fitted, objectives = api.fit_weights(scene, start, p, target, iterations=60, use_blur=use_blur)
    after = masked_psnr(shot(api, scene, p), target)  # the handle holds the fitted stops
    print(f"fit_weights {name} use_blur={use_blur}: {before:.2f} dB -> {after:.2f} dB in {len(objectives) - 1} iterations")
    assert all(b <= a for a, b in zip(objectives, objectives[1:]))
    assert objectives[-1] < objectives[0]
    nw, ne = int(d["n_weight"]), int(d["n_weight_degree"])
    assert np.array_equal(fitted["weight"][nw:], start["weight"][nw:])
    assert np.array_equal(fitted["weight_degree"][ne:], start["weight_degree"][ne:])
    assert np.all(fitted["weight"][:nw] > 0)
    for k in ("color_left", "color_right", "blur", "weight_u", "weight_degree_u"):
        assert np.array_equal(fitted[k], start[k])
    assert after >= 40.0, (before, after)


def test_alternating_colour_blur_and_weight_fits(api, scene_dict):
    d = scene_dict("DiffusionCurvePack/face.xml")
    p = fit_view(api, d)
    nb = int(d["n_blur"])
    changed = changed_weights(d, 12)
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
        current, _ = api.fit_weights(scene, current, p, target, iterations=30, use_blur=True)
    after = masked_psnr(blurred_target(api, scene, p), target)
    print(f"alternating colour, blur and weight fits on face.xml: {before:.2f} dB -> {after:.2f} dB")
    assert after >= 40.0, (before, after)
