"""The float64 reference of tests/stop_reference.py checked against itself and the CPU oracle, without a device.

* Its frame equals oracle.render, NaN pattern included. The oracle shades in fp32: each ray's lerps (a few roundings each,
  the ratio an exact IEEE division), libm powf for t^-e, whose error grows with |e ln t| through the rounding of e, and the
  ray-order sums of n terms ((n - 1) u of the summed magnitudes), then one division. So per pixel and channel
  |oracle - ref| <= u (n + 16 + 10 max |e| |ln t|) scale, scale = (sum |w| |c| + |P| sum |w|) / |W| (stop_reference.frame).
* Its weight and exponent VJPs equal the complex-step derivatives of its own frame, entry by entry, and its colour and blur
  VJPs equal the transposes of explicit float64 matrices built column by column from its frame.
* The scale identity sum_k weight[k] grad_weight[k] = 0 holds to float64 rounding.

The scenes are bundled ones and the generated edge scenes below, which the device tests (tests/test_stop_reference_gpu.py)
use too; the last test here checks that they exercise what they are built for.
"""
import os

import numpy as np
import pytest

import stop_reference as sr
from helpers import curve_xml, scene_xml, straight
from oracle import pyoracle as po

# ---------------------------------------------------------------------------------------------------------------------
# generated edge scenes (CurveSetXML; coordinates in the file's 512 x 512 frame)
# ---------------------------------------------------------------------------------------------------------------------
POLY_Y, POLY_X0, POLY_STEP, POLY_SEGMENTS = 300, 100, 60, 5  # the polyline: straight segments of 60, integer vertices
POLY_WEIGHTS = [(0, 0.0), (10, 0.0), (15, 2.5), (20, 1e-3), (30, 1e3), (35, 1.0), (50, 4.0)]  # weight 0 on segment 0
POLY_EXPONENTS = [(0, -1.0), (5, 0.0), (12.5, 0.5), (20, 0.5), (25, 0.9), (40, 2.0), (45, 3.7), (50, 3.7)]
CONSTANT_EXPONENTS = [-1.0, 0.0, 0.5, 0.9, 2.0, 3.7]
SPREAD_WEIGHTS = [1e-3, 1e-2, 1.0, 30.0, 1e3, 0.5]
ARC = [(120.0, 420.0), (120.0, 500.0), (240.0, 500.0), (240.0, 420.0)]  # one curved segment of several chords


def polyline(y, x0, step, segments):
    pts = [(x0, y)]
    for k in range(segments):
        pts += straight(x0 + step * k, y, x0 + step * (k + 1), y)[1:]
    return pts


def box(x0, y0, side):
    """a closed square as one curve of four straight segments"""
    corners = [(x0, y0), (x0 + side, y0), (x0 + side, y0 + side), (x0, y0 + side), (x0, y0)]
    pts = [corners[0]]
    for a, b in zip(corners, corners[1:]):
        pts += straight(*a, *b)[1:]
    return pts


def edge_curves(arc_chords):
    """Weight and exponent stops at different u; stops at segment boundaries (integer u) on a polyline whose vertices the
    rays of an integer view meet exactly; weight 0 on part of a shaded curve; a closed box of weight 0 (the pixels inside
    it are NaN); exponents -1, 0, 0.5, 0.9, 2, 3.7; weights from 1e-3 to 1e3; and a curved segment of `arc_chords` chords
    with a weight stop at every chord end k/K and more exponent stops in one segment than any walk hint skips."""
    curves = [curve_xml(polyline(POLY_Y, POLY_X0, POLY_STEP, POLY_SEGMENTS), (200, 40, 90), POLY_WEIGHTS, POLY_EXPONENTS)]
    ends = [(10.0 * k / arc_chords, 1.0 + 0.5 * (k % 3)) for k in range(arc_chords + 1)]
    many = [(0.7 * k, 0.3 + 0.25 * (k % 5)) for k in range(15)]
    curves.append(curve_xml(ARC, (30, 220, 120), ends, many))
    curves.append(curve_xml(box(380, 380, 90), (90, 90, 250), [(0, 0.0), (40, 0.0)]))
    for k, (e, w) in enumerate(zip(CONSTANT_EXPONENTS, SPREAD_WEIGHTS)):  # single segments last: walks past a curve's
        x = 40 + 40 * k                                                    # own list stay inside the file's lists
        curves.append(curve_xml(straight(x, 20, x + 30, 200), (40 * k, 250 - 40 * k, 128), [(0, w), (10, w)], [(0, e), (10, e)]))
    return curves


def arc_chords():
    """chords of the arc's one segment (the flatness rule of rdc_chord_count, via the oracle)"""
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "arc.xml")
        with open(path, "w") as fh:
            fh.write(scene_xml([curve_xml(ARC)]))
        _, ids = po.Oracle("port").chords(po.ingest_xml(path, True))
    return int(ids[0, 2])


def edge_scene_xml():
    return scene_xml(edge_curves(arc_chords()))


# views of the edge scene: (w, h, n, frame parameters); scene coordinates are the file's minus 256, axes swapped
POLY_SCENE_X = POLY_Y - 256  # the polyline is the line x = 44 of the scene, its vertices at y = -156 + 60 k
EDGE_VIEWS = {
    "whole": (64, 64, 32, dict(zoom_factor=8.0)),
    # use_aa 0, zoom 1, integer offsets: ray 0 of every pixel runs along +x from an integer origin, through the polyline's
    # vertices at y = -96 and -36 (curve_u exactly 1 and 2 on the stops there)
    "vertices": (32, 64, 8, dict(zoom_factor=1.0, offset_x=0.0, offset_y=-66.0, use_aa=0)),
    # origins 1e-4 from the polyline: t from about 1e-5 on, |ln t| up to about 11
    "tiny": (16, 16, 16, dict(zoom_factor=1e-5, offset_x=POLY_SCENE_X - 1.5e-4, offset_y=4.0)),
    "box": (32, 32, 16, dict(zoom_factor=4.0, offset_x=425.0 - 256, offset_y=425.0 - 256)),
}


@pytest.fixture(scope="module")
def edge_scene(tmp_path_factory):
    path = tmp_path_factory.mktemp("stop_reference") / "edges.xml"
    path.write_text(edge_scene_xml())
    return str(path)


def records(oracle, d, w, h, n, **view):
    view.setdefault("max_trace_depth", 0)
    p = po.make_params(w, h, n, **view)
    return oracle.ray_records(d, p), p


# ---------------------------------------------------------------------------------------------------------------------
# 1. the frame against the oracle
# ---------------------------------------------------------------------------------------------------------------------
FRAME_SCENES = ["weight_demo.xml", "arch.xml", "PortalDemo.xml", "DiffusionCurvePack/lady_bug.xml",
                "DiffusionCurvePack/face.xml", "circles.xml"]


def check_frame_against_oracle(oracle, d, p, rec):
    img, blur, hits = oracle.render(d, p, want_hits=True, search="grid")
    assert np.array_equal(hits, rec["id"]), "the records are not the render's rays"
    fr = sr.frame(d, rec)
    assert np.array_equal(np.isnan(img[..., :3]).any(-1), fr["nan"]) and np.array_equal(np.isnan(blur), fr["nan"])
    live = ~fr["nan"]
    tau = sr.U * (rec.shape[-1] + 16 + 10 * fr["elnt"])
    e_img = np.abs(img[..., :3].astype(np.float64) - fr["image"])[live]
    e_blur = np.abs(blur.astype(np.float64) - fr["blur"])[live]
    assert np.all(e_img <= tau * fr["image_scale"][live] + 1e-30), (e_img / fr["image_scale"][live]).max()
    assert np.all(e_blur <= tau * fr["blur_scale"][live] + 1e-30), (e_blur / fr["blur_scale"][live]).max()
    return fr


@pytest.mark.parametrize("name", FRAME_SCENES)
def test_frame_equals_the_oracle(port_oracle, xml_dir, name):
    d = po.ingest_xml(os.path.join(xml_dir, name), True)
    rec, p = records(port_oracle, d, 48, 40, 16, zoom_factor=d["image_height"] / 40)
    fr = check_frame_against_oracle(port_oracle, d, p, rec)
    assert (~fr["nan"]).sum() > 0


@pytest.mark.parametrize("view", sorted(EDGE_VIEWS))
def test_frame_equals_the_oracle_edge_scene(port_oracle, edge_scene, view):
    d = po.ingest_xml(edge_scene, True)
    w, h, n, kw = EDGE_VIEWS[view]
    rec, p = records(port_oracle, d, w, h, n, **kw)
    check_frame_against_oracle(port_oracle, d, p, rec)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the VJPs against the reference's own derivatives
# ---------------------------------------------------------------------------------------------------------------------
def gradients(rng, rec, zeros=True):
    """G [rows, W, 3] and g_sigma [rows, W], float32; with `zeros` the green channel, g_sigma on every other row and all of
    G on every third column are zero"""
    rows, w, _ = rec.shape
    G = rng.standard_normal((rows, w, 3)).astype(np.float32)
    gs = rng.standard_normal((rows, w)).astype(np.float32)
    if zeros:
        G[..., 1] = 0.0
        G[:, ::3] = 0.0
        gs[::2] = 0.0
    return G, gs


def moved(d, seed):
    """weights times [0.5, 2], exponents plus [0, 0.5], as test_weight_fit_gpu.moved"""
    rng = np.random.default_rng(seed)
    e = dict(d)
    nw, ne = int(d["n_weight"]), int(d["n_weight_degree"])
    e["weight"], e["weight_degree"] = d["weight"].copy(), d["weight_degree"].copy()
    e["weight"][:nw] *= np.exp2(rng.uniform(-1.0, 1.0, nw)).astype(np.float32)
    e["weight_degree"][:ne] += rng.uniform(0.0, 0.5, ne).astype(np.float32)
    return e


def vjp_cases(xml_dir, edge_scene):
    out = []
    for name in ("weight_demo.xml", "arch.xml"):
        d = po.ingest_xml(os.path.join(xml_dir, name), True)
        out.append((name, moved(d, 1), (24, 20, 8, dict(zoom_factor=d["image_height"] / 20))))
    d = po.ingest_xml(edge_scene, True)
    for view in ("whole", "tiny", "box"):
        w, h, n, kw = EDGE_VIEWS[view]
        out.append(("edges-" + view, d, (w // 2, h // 2, n // 2, dict(kw, zoom_factor=kw["zoom_factor"] * 2))))
    return out


def test_weight_and_exponent_vjps_equal_complex_step_derivatives(port_oracle, xml_dir, edge_scene):
    """Entry by entry against the derivative of stop_reference.loss by a complex step, Im L(x + i h e_k) / h with h = 1e-30:
    a difference quotient without the cancellation of real differences, so it holds at float64 rounding whatever the
    scales (a weight of 0 beside weights of 1e-11 in one pixel, a weight of 1e-3 beside one of 1e3 in another). The NaN
    pixels stay those of the unmoved stops: a step off a weight of 0 would bring the pixels of the weight-0 box to life,
    outside the derivative."""
    rng = np.random.default_rng(0)
    h = 1e-30
    for cid, d, (w, ht, n, kw) in vjp_cases(xml_dir, edge_scene):
        rec, _ = records(port_oracle, d, w, ht, n, **kw)
        R = sr.Rays(d, rec)
        G, gs = gradients(rng, rec)
        grads, bounds = sr.vjp(d, R, G, gs)
        live = ~sr.frame(d, R)["nan"]
        for fam in ("weight", "weight_degree"):
            x = d[fam].astype(np.complex128)
            touched = np.nonzero(bounds[fam])[0]
            assert len(touched) > 0, (cid, fam)
            for k in touched:
                xk = x.copy()
                xk[k] += 1j * h
                cs = sr.loss(d, R, G, gs, {fam: xk}, live).imag / h
                assert abs(cs - grads[fam][k]) <= 1e-12 * bounds[fam][k], (cid, fam, k, cs, grads[fam][k], bounds[fam][k])


def test_colour_and_blur_vjps_are_explicit_transposes(port_oracle, xml_dir, edge_scene):
    """A and A_b column by column: the reference frame with one stop value 1 and the rest 0 (weights as they are)."""
    rng = np.random.default_rng(1)
    for cid, d, (w, h, n, kw) in vjp_cases(xml_dir, edge_scene):
        rec, _ = records(port_oracle, d, w, h, n, **kw)
        R = sr.Rays(d, rec)
        G, gs = gradients(rng, rec)
        grads, _ = sr.vjp(d, R, G, gs)
        live = ~sr.frame(d, R)["nan"]
        Gl, gsl = G.astype(np.float64)[live], gs.astype(np.float64)[live]
        zero = {fam: np.zeros(d[fam].shape) for fam in ("color_left", "color_right", "blur")}
        for fam in ("color_left", "color_right"):
            want = np.zeros(d[fam].shape)
            for j in range(d[fam].shape[0]):
                x = np.zeros(d[fam].shape)
                x[j] = 1.0  # stop j in all three channels: a channel only sees its own
                col = sr.frame(d, R, dict(zero, **{fam: x}))["image"][live]
                want[j] = (col * Gl).sum(0)
            assert np.allclose(grads[fam], want, rtol=1e-12, atol=1e-12 * np.abs(want).max()), (cid, fam)
        want = np.zeros(d["blur"].shape)
        for j in range(d["blur"].shape[0]):
            x = np.zeros(d["blur"].shape)
            x[j] = 1.0
            want[j] = (sr.frame(d, R, dict(zero, blur=x))["blur"][live] * gsl).sum()
        assert np.allclose(grads["blur"], want, rtol=1e-12, atol=1e-12 * np.abs(want).max()), cid


def test_scale_identity(port_oracle, xml_dir, edge_scene):
    rng = np.random.default_rng(2)
    for cid, d, (w, h, n, kw) in vjp_cases(xml_dir, edge_scene):
        rec, _ = records(port_oracle, d, w, h, n, **kw)
        G, gs = gradients(rng, rec)
        grads, bounds = sr.vjp(d, rec, G, gs)
        terms = d["weight"].astype(np.float64) * grads["weight"]
        scale = (np.abs(d["weight"].astype(np.float64)) * bounds["weight"]).sum()  # sum over the rays of |w| |s - K| / W
        assert np.abs(terms).sum() > 0, cid
        assert abs(terms.sum()) <= 1e-13 * scale, (cid, terms.sum(), scale)


# ---------------------------------------------------------------------------------------------------------------------
# 3. the edge scene exercises what it is built for
# ---------------------------------------------------------------------------------------------------------------------
def test_edge_scene_is_what_it_claims(port_oracle, edge_scene):
    d = po.ingest_xml(edge_scene, True)
    # weight and exponent stops at different u; more exponent stops in the arc's one segment than the hint skips
    assert not np.array_equal(d["weight_u"][:d["n_weight"]], d["weight_degree_u"][:d["n_weight_degree"]])
    K = arc_chords()
    assert K >= 4
    arc_w = d["weight_u"][d["weight_index"][1, 0]:][:d["weight_index"][1, 1]]
    chord_ends = np.float32(np.arange(K + 1)) / np.float32(K)
    assert np.isin(chord_ends, arc_w).sum() >= K // 2  # most chord ends k/K are weight stops, bit for bit
    assert d["weight_degree_index"][1, 1] >= 15
    fams = {}
    for view, (w, h, n, kw) in EDGE_VIEWS.items():
        rec, _ = records(port_oracle, d, w, h, n, **kw)
        R = sr.Rays(d, rec)
        s = sr.shade(d, R)
        fr = sr.frame(d, R)
        fams[view] = (rec, R, s, fr)
    # exact hits on the polyline's vertices, where a weight stop sits at the same u
    rec, R, s, fr = fams["vertices"]
    flat = rec.reshape(-1)
    hit = (flat["id"] != sr.MISS) & (flat["curve"] == 0)
    assert np.isin(flat["curve_u"][hit], np.float32([1.0, 2.0])).sum() >= 2
    # weight 0 on a shaded ray whose pixel is live; every weight from 1e-3 to 1e3 and every exponent shades some ray
    rec, R, s, fr = fams["whole"]
    live = ~fr["nan"].reshape(-1)[R.pixel]
    assert ((s["w"] == 0) & live).any()
    assert np.isin(np.float32(SPREAD_WEIGHTS), s["m"].astype(np.float32)).all()
    assert np.isin(np.float32(CONSTANT_EXPONENTS), s["e"].astype(np.float32)).all()
    # pixels inside the box are NaN
    assert fams["box"][3]["nan"].any() and not fams["box"][3]["nan"].all()
    # tiny t
    rec, R, s, fr = fams["tiny"]
    assert R.t.min() < 1e-4 and fr["elnt"] > 8
