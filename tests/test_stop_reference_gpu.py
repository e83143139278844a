"""The render and its three stop adjoints, entry by entry, against the float64 reference of tests/stop_reference.py.

Each case renders with hit ids and first asserts that they equal the chord ids of the oracle's ray records bit for bit: the
reference then restates the kernel's own rays. From there every pixel of the frame and every entry of the colour, blur,
weight and exponent adjoints must lie within tau * bound of the reference (bound: stop_reference's magnitudes, the sum
over the rays of the absolute values each term is made of).

Error model, in units of u = 2^-24 (the fp32 unit roundoff), for one ray's term relative to its magnitude:
* the stop lerps: a few roundings each, and the ratio's __fdividef (rdc_ratio, at most 2 ulp): 16 covers every lerp,
  product and sum of a term together;
* rdc_weight_falloff: exp2f(-e log2f(t)) is off by about 2 |e ln t| u (measured 1.9 |e ln t| u at e = 3.7, rdc_math.h), and
  the lerped e by a few u of |e|, which t^-e turns into |ln t| times that: 10 max |e| |ln t| covers both, for the weight in
  a term and for each weight in W and K;
* the fp32 sum of W over the pixel's n rays in ray order (the frame and the colour and blur adjoints): (n - 1) u of the sum
  of the magnitudes. The weight adjoint sums W and K in fp64 and has no such term.
So tau = u (16 + 10 L + n) for the frame, the colour and the blur adjoint, and u (16 + 10 L) for the weight and exponent
adjoints, with L = max over the case's rays of |e| |ln t|: 3e-6 + 6e-8 n for the default exponent at t ~ 100, up to ~4e-5
for exponent 3.7 at t ~ 1e-5 or 1e5. The worst err / bound of each family is printed per case and for the whole module.
"""
import math

import numpy as np
import pytest

import stop_reference as sr
from helpers import copy_params, scene_ids
from oracle import pyoracle as po
from test_color_adjoint_gpu import adjoint as color_adjoint
from test_color_adjoint_gpu import api, build, params_for, scene_dict, stream  # noqa: F401 (fixtures)
from test_scene_update_gpu import SYNTH_PORTALS
from test_stop_reference_cpu import EDGE_VIEWS, edge_scene_xml, gradients
from test_weight_fit_gpu import moved, weight_adjoint, with_weights

pytestmark = pytest.mark.gpu

LADY = "DiffusionCurvePack/lady_bug.xml"
FAMILIES = ("forward", "colour", "blur", "weight", "exponent")
WORST = {f: 0.0 for f in FAMILIES}  # over the module, printed at its end


@pytest.fixture(scope="module", autouse=True)
def worst_summary():
    yield
    print("\nstop reference, worst err / bound over the module: "
          + ", ".join(f"{f} {WORST[f]:.2e}" for f in FAMILIES))


@pytest.fixture(scope="module")
def edge_dict(api):
    opts = api.default_ingest_options(use_diffusion_curve_save=1)
    return api.HostScene.from_xml_text(edge_scene_xml().encode(), opts).to_numpy()


def tau(family, n, elnt):
    t = sr.U * (16 + 10 * elnt)
    return t + sr.U * n if family in ("forward", "colour", "blur") else t


def render_with_hits(api, scene, p):
    import torch

    rows, n_iter = p.row_end - p.row_begin, int(math.ceil(p.number_of_rays_per_pixel))
    image = torch.empty((rows, p.image_width, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, p.image_width), dtype=torch.float32, device="cuda")
    hits = torch.empty((rows, p.image_width, n_iter), dtype=torch.int32, device="cuda")
    q = api.FrameParams.from_buffer_copy(p)
    q.hit_ids = hits.data_ptr()
    scene.render(q, image.data_ptr(), sigma.data_ptr(), stream())
    torch.cuda.synchronize()
    return image.cpu().numpy(), sigma.cpu().numpy(), hits.cpu().numpy().view(np.uint32)


def blur_adjoint(api, scene, d, p, gs):
    import torch

    g = torch.from_numpy(np.ascontiguousarray(gs, np.float32)).cuda()
    out = torch.full(d["blur"].shape, 7.0, dtype=torch.float64, device="cuda")  # overwritten by the call
    torch.cuda.synchronize()
    scene.blur_adjoint(p, g.data_ptr(), out.data_ptr(), stream())
    torch.cuda.synchronize()
    return out.cpu().numpy()


def within(family, got, want, bound, t, label):
    """every entry within t * bound (NaN nowhere); returns the worst err / bound"""
    assert np.isfinite(got).all(), f"{label} {family}: non-finite entries"
    err = np.abs(got - want)
    bad = err > t * bound + 1e-30
    assert not bad.any(), (f"{label} {family}: {int(bad.sum())} entries outside tau * bound; worst err / bound "
                           f"{float((err / np.maximum(bound, 1e-300)).max()):.3e}, tau {t:.2e}")
    ratio = float((err / np.where(bound > 0, bound, np.inf)).max(initial=0.0))
    WORST[family] = max(WORST[family], ratio)
    return ratio


def check(api, d, p, label, search="grid", families=True, zeros=True, seed=0):
    """hits bit-equal to the records, then the frame and (with `families`) the four adjoints against the reference"""
    scene = build(api, d)
    image, sigma, hits = render_with_hits(api, scene, p)
    q = copy_params(p, po.FrameParams)
    q.hit_ids = q.max_sigma = q.stats = None
    rec = po.Oracle("port").ray_records(d, q, search=search)
    assert np.array_equal(hits, rec["id"]), f"{label}: {int((hits != rec['id']).sum())} hit ids differ from the records"
    fr = sr.frame(d, rec)
    n, L = rec.shape[-1], fr["elnt"]
    assert np.array_equal(np.isnan(image[..., :3]).any(-1), fr["nan"]) and np.array_equal(np.isnan(sigma), fr["nan"]), \
        f"{label}: NaN pixels differ"
    live = ~fr["nan"]
    assert live.any(), f"{label}: every pixel is NaN"
    worst = {"forward": max(
        within("forward", image[..., :3].astype(np.float64)[live], fr["image"][live], fr["image_scale"][live],
               tau("forward", n, L), label),
        within("forward", sigma.astype(np.float64)[live], fr["blur"][live], fr["blur_scale"][live], tau("forward", n, L), label))}
    if families:
        G, gs = gradients(np.random.default_rng(seed), rec, zeros)
        want, bound = sr.vjp(d, rec, G, gs)
        left, right = color_adjoint(api, scene, d, p, G)
        worst["colour"] = within("colour", np.concatenate([left, right]), np.concatenate([want["color_left"], want["color_right"]]),
                                 np.concatenate([bound["color_left"], bound["color_right"]]), tau("colour", n, L), label)
        worst["blur"] = within("blur", blur_adjoint(api, scene, d, p, gs), want["blur"], bound["blur"], tau("blur", n, L), label)
        gw, ge = weight_adjoint(api, scene, d, p, G, gs)
        worst["weight"] = within("weight", gw, want["weight"], bound["weight"], tau("weight", n, L), label)
        worst["exponent"] = within("exponent", ge, want["weight_degree"], bound["weight_degree"], tau("exponent", n, L), label)
        assert np.abs(gw).sum() > 0 and np.abs(ge).sum() > 0, f"{label}: the weight adjoint vanishes"
    print(f"{label}: hits {int((rec['id'] != sr.MISS).sum())} of {rec.size} rays, max |e ln t| {L:.1f}, tau(weight) "
          f"{tau('weight', n, L):.1e}; worst err / bound " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    return rec


def stops(d, which, seed=1):
    return d if which == "ingested" else with_weights(d, *moved(d, seed))


STOPS = ["ingested", "moved"]


# ---------------------------------------------------------------------------------------------------------------------
# bundled scenes, the synthetic portal scene, the 100 k-curve scene
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", STOPS)
@pytest.mark.parametrize("name", scene_ids())
def test_every_scene(api, scene_dict, name, which):
    d = stops(scene_dict(name), which)
    check(api, d, params_for(api, d, 48, 40, 16), f"{name} {which}", zeros=which == "moved")


@pytest.mark.parametrize("which", STOPS)
def test_synthetic_portals_depth_0(api, scene_dict, which):
    d = stops(scene_dict(SYNTH_PORTALS), which)
    check(api, d, params_for(api, d, 96, 96, 16), f"synthetic portals {which}")


def test_100k_band(api, scene_dict):
    d = stops(scene_dict("synth100k"), "moved")
    p = params_for(api, d, 2048, 2048, 64, row_begin=1001, row_end=1010)
    check(api, d, p, "100k band", search="grid")


# ---------------------------------------------------------------------------------------------------------------------
# bands, single rows, frame options, traversals, routes, many rays per pixel
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows", [(0, 41), (13, 30), (17, 18), (40, 41)], ids=["whole", "band-13-30", "row-17", "row-40"])
@pytest.mark.parametrize("name", ["arch.xml", LADY])
def test_bands_and_rows(api, scene_dict, name, rows):
    d = stops(scene_dict(name), "moved", 2)
    check(api, d, params_for(api, d, 72, 41, 32, row_begin=rows[0], row_end=rows[1]), f"{name} rows {rows}")


PARAM_CASES = ["aa_off", "orzan_off", "fractional_n", "n_below_8", "zoom_pan", "far_view", "brute"]


@pytest.mark.parametrize("which", STOPS)
@pytest.mark.parametrize("case", PARAM_CASES)
def test_frame_options(api, scene_dict, case, which):
    orzan = case != "orzan_off"
    d = stops(scene_dict("DiffusionCurvePack/face.xml", orzan), which, 3)
    kw = {"aa_off": dict(use_aa=0), "orzan_off": dict(use_diffusion_curve_save=0), "zoom_pan": dict(zoom_factor=2.5, offset_x=-40.0, offset_y=65.0),
          "far_view": dict(offset_x=1e5, offset_y=-1e5), "brute": dict(traversal=api.TRAVERSAL_BRUTE_FORCE)}.get(case, {})
    n = {"fractional_n": 12.5, "n_below_8": 5}.get(case, 24)
    check(api, d, params_for(api, d, 56, 44, n, frame=3, seed=9, **kw), f"face.xml {case} {which}")


@pytest.mark.parametrize("route,name,mode", [(1, LADY, 0), (0, "arch.xml", 1), (3, LADY, 3), (2, LADY, 2)],
                         ids=["tree", "whole-scene-table", "cut-table", "local-table"])
def test_routes_forward(api, scene_dict, route, name, mode):
    d = stops(scene_dict(name), "moved", 4)
    view = dict(zoom_factor=1.0, offset_x=-30.0, offset_y=20.0) if name == LADY else {}
    p = params_for(api, d, 128, 96, 64, route=route, **view)
    assert build(api, d).launch_plan(p).mode == mode  # the render really takes that route
    check(api, d, p, f"{name} route {route}", families=False)


@pytest.mark.parametrize("n", [1000, 4096])
@pytest.mark.parametrize("name", ["weight_demo.xml", LADY])
def test_many_rays_per_pixel(api, scene_dict, name, n):
    """n (- 1) u of W's fp32 sum dominates tau here"""
    d = stops(scene_dict(name), "moved", 5)
    check(api, d, params_for(api, d, 64, 48, n, row_begin=22, row_end=26), f"{name} n={n}")


# ---------------------------------------------------------------------------------------------------------------------
# the generated edge scene (tests/test_stop_reference_cpu.py: edge_curves)
# ---------------------------------------------------------------------------------------------------------------------
EDGE_CASES = dict(EDGE_VIEWS, far=(64, 64, 32, dict(zoom_factor=8.0, offset_x=6e4, offset_y=-8e4)))


@pytest.mark.parametrize("which", STOPS)
@pytest.mark.parametrize("view", sorted(EDGE_CASES))
def test_edge_scene(api, edge_dict, view, which):
    d = stops(edge_dict, which, 6)
    w, h, n, kw = EDGE_CASES[view]
    rec = check(api, d, params_for(api, d, w, h, n, **kw), f"edges {view} {which}", zeros=view != "whole")
    if view == "box":
        assert sr.frame(d, rec)["nan"].any(), "the box's pixels should be NaN"
