"""First hits where the culling margins are thinnest: every route against the brute-force kernel and the CPU oracle.

The tree, the whole-scene table, the cut table and the local table skip boxes by a slab test of padded boxes, which is
only allowed to skip a box that cannot hold the winning chord (DESIGN.md section 4). The rounding of that test and of the
chord test grows with the ray origins' coordinates, so the cases here look at the scenes from 1e3 to 1e6 units away (by
offset and by zoom), at rays laid exactly along chords and box edges, at ties built on purpose, and at degenerate trees.
The reference is the brute-force kernel (RDC_TRAVERSAL_BRUTE_FORCE tests every chord for every ray) over frames with a
floor on the number of hits, so that an all-miss view cannot pass, and the port oracle on one band of each case.
"""
import os

import numpy as np
import pytest

from helpers import GpuRenderer, compare_images, copy_params, curve_xml, dust_curves, scene_xml, straight
from oracle import pyoracle as po
from raytracingdiffusioncurves_b200.api import (MODE_CUT, MODE_LOCAL, MODE_TABLE, MODE_TREE, ROUTE_AUTO, ROUTE_LOCAL_TABLE,
                                                ROUTE_TREE, TRAVERSAL_BRUTE_FORCE, TREE_MORTON, TREE_SAH)

pytestmark = pytest.mark.gpu

MISS = -1  # hit ids are read as int32
RGB_TOL = 1e-4


def grid_curves():
    """Axis-aligned and diagonal straight curves with every vertex on integer coordinates (spans divisible by 3, so the
    inner control points are integers too): with use_aa 0, integer zoom and integer offsets the rays start on integer
    coordinates and ray 0 runs along (1, 0), i.e. exactly along the horizontal chords and through their end points."""
    out = []
    for k in range(12):
        y = 96 + 27 * k
        out.append(curve_xml(straight(60 + 6 * k, y, 240 + 9 * k, y), (20 * k, 40, 200)))     # horizontal
        out.append(curve_xml(straight(300 + 15 * k, 60, 300 + 15 * k, 420), (200, 20 * k, 40)))  # vertical
        out.append(curve_xml(straight(30 + 24 * k, 450, 60 + 24 * k, 480), (40, 200, 20 * k)))  # diagonal
    return out


def tie_curves(base, reverse):
    """`base` with its first curve repeated before and after it in the file: exact ties (the smaller chord id must win),
    or, reversed, a copy whose chords meet the rays within an ulp of the original's."""
    first = base[0]
    if reverse:
        import re

        pts = re.findall(r"<control_point [^>]*/>", first)
        first = first.replace("".join(pts), "".join(reversed(pts)))
    return [first] + base + [first]


def generated(name):
    arch = [curve_xml(straight(100 + 3 * k, 100, 160 + 3 * k, 400 - 6 * k)) for k in range(20)]
    return {
        "dust.xml": lambda: dust_curves(),
        "grid.xml": grid_curves,
        "one_chord.xml": lambda: [curve_xml(straight(200, 180, 290, 330))],
        "zero_length.xml": lambda: dust_curves(600)[:300] + [curve_xml([(256.0, 256.0)] * 4)] + dust_curves(600)[300:],
        "identical.xml": lambda: [curve_xml(straight(150, 200, 330, 290))] * 300 + [curve_xml(straight(40, 40, 470, 60))],
        "runs64.xml": lambda: dust_curves(64, seed=3),
        "runs65.xml": lambda: dust_curves(65, seed=3),
        "ties_exact.xml": lambda: tie_curves(arch, False),
        "ties_near.xml": lambda: tie_curves(arch, True),
        "ties_exact_dust.xml": lambda: tie_curves(grid_curves() + dust_curves(400), False),
        "ties_near_dust.xml": lambda: tie_curves(grid_curves() + dust_curves(400), True),
    }[name]()


@pytest.fixture(scope="module")
def api():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from raytracingdiffusioncurves_b200 import api as _api

    return _api


class Scenes:
    def __init__(self, xml_dir, tmp_dir):
        self.xml_dir, self.tmp_dir = xml_dir, tmp_dir
        self._gpu, self._dicts = {}, {}

    def path(self, name):
        p = os.path.join(self.xml_dir, name)
        if os.path.exists(p):
            return p
        p = os.path.join(self.tmp_dir, name)
        if not os.path.exists(p):
            with open(p, "w") as fh:
                fh.write(scene_xml(generated(name)))
        return p

    def gpu(self, api, name, **accel):
        key = (name, tuple(sorted(accel.items())))
        if key not in self._gpu:
            self._gpu[key] = GpuRenderer(self.path(name), accel=api.default_accel_options(**accel) if accel else None)
        return self._gpu[key]

    def dict(self, name):
        if name not in self._dicts:
            self._dicts[name] = po.ingest_xml(self.path(name), True)
        return self._dicts[name]


@pytest.fixture(scope="module")
def scenes(xml_dir, tmp_path_factory):
    return Scenes(xml_dir, str(tmp_path_factory.mktemp("margins")))


def params(api, w, h, n, **kw):
    return copy_params(po.make_params(w, h, n, **kw), api.FrameParams)


def trace(r, p):
    """One launch; hit ids (int32) and image stay on the device."""
    import torch

    rows, n_iter = p.row_end - p.row_begin, int(np.ceil(p.number_of_rays_per_pixel))
    image = torch.empty((rows, p.image_width, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, p.image_width), dtype=torch.float32, device="cuda")
    hits = torch.empty((rows, p.image_width, n_iter), dtype=torch.int32, device="cuda")
    p.hit_ids, p.max_sigma, p.stats = hits.data_ptr(), None, None
    r.scene.render(p, image.data_ptr(), sigma.data_ptr(), torch.cuda.current_stream().cuda_stream)
    return hits, image


def bands_from_centre(h, band):
    starts = list(range(0, h, band))
    return sorted(starts, key=lambda b: abs(b + band / 2 - h / 2))


def against_brute_force(api, r, w, h, n, route, mode, floor, band, **view):
    """Bands of the frame, nearest the centre first, until the brute force has `floor` hits: LBVH hit ids against the
    brute force's, NaN pattern and RGB within RGB_TOL. Returns (differing rays, hits, rays)."""
    import torch

    differing = hits = rays = 0
    for b in bands_from_centre(h, band):
        e = min(h, b + band)
        p = params(api, w, h, n, route=route, row_begin=b, row_end=e, **view)
        assert r.scene.launch_plan(p).mode == mode, (route, r.scene.launch_plan(p).mode)
        got, gimg = trace(r, p)
        want, wimg = trace(r, params(api, w, h, n, traversal=TRAVERSAL_BRUTE_FORCE, row_begin=b, row_end=e, **view))
        torch.cuda.synchronize()
        differing += int((got != want).sum())
        hits += int((want != MISS).sum())
        rays += want.numel()
        gn, wn = torch.isnan(gimg[..., :3]), torch.isnan(wimg[..., :3])
        assert torch.equal(gn, wn) or differing > 0, f"rows [{b}, {e}): NaN (all-miss) pixels differ"
        d = float((gimg[..., :3] - wimg[..., :3]).abs()[~wn].max()) if (~wn).any() and not differing else 0.0
        assert d <= RGB_TOL or differing > 0, f"rows [{b}, {e}): max |rgb diff| {d}"
        if hits >= floor:
            break
    return differing, hits, rays


def against_oracle(api, scenes, r, name, w, h, n, route, rows, accel=None, **view):
    b, e = rows
    oimg, _, ohits = po.Oracle("port").render(scenes.dict(name), po.make_params(w, h, n, row_begin=b, row_end=e, **view),
                                              accel=accel, want_hits=True, search="grid")
    hits, image = trace(r, params(api, w, h, n, route=route, row_begin=b, row_end=e, **view))
    got = hits.cpu().numpy().view(np.uint32)
    assert np.array_equal(got, ohits), f"{int((got != ohits).sum())} of {got.size} hit ids differ from the oracle"
    compare_images(image.cpu().numpy(), oimg, RGB_TOL)
    return int((ohits != 0xFFFFFFFF).sum())


# ---------------------------------------------------------------------------------------------------------------------
# A. far views
# ---------------------------------------------------------------------------------------------------------------------
# (id, scene, accel options, route, expected mode, max_trace_depth)
FAR_CASES = [
    ("arch-table", "arch.xml", {}, ROUTE_AUTO, MODE_TABLE, 2),
    ("arch-table-width0", "arch.xml", dict(curve_width=0.0), ROUTE_AUTO, MODE_TABLE, 2),
    ("arch-tree-morton", "arch.xml", dict(tree=TREE_MORTON), ROUTE_TREE, MODE_TREE, 2),
    ("lady_bug-cut", "DiffusionCurvePack/lady_bug.xml", {}, ROUTE_AUTO, MODE_CUT, 2),
    ("lady_bug-cut-width0", "DiffusionCurvePack/lady_bug.xml", dict(curve_width=0.0), ROUTE_AUTO, MODE_CUT, 2),
    ("dust-cut", "dust.xml", {}, ROUTE_AUTO, MODE_CUT, 2),
    ("dust-cut-width0", "dust.xml", dict(curve_width=0.0), ROUTE_AUTO, MODE_CUT, 2),
    ("dust-local", "dust.xml", {}, ROUTE_LOCAL_TABLE, MODE_LOCAL, 2),
    ("dust-tree-sah", "dust.xml", dict(tree=TREE_SAH), ROUTE_TREE, MODE_TREE, 2),
    ("dust-tree-morton-width0", "dust.xml", dict(tree=TREE_MORTON, curve_width=0.0), ROUTE_TREE, MODE_TREE, 2),
    ("portal-d2", "PortalDemo.xml", {}, ROUTE_AUTO, MODE_TABLE, 2),
    ("portal-d31", "PortalDemo.xml", {}, ROUTE_TREE, MODE_TREE, 31),
]
DISTANCES = [1e3, 1e4, 1e5, 1e6]
FLOOR = 100_000  # brute-force hits a case must see
# offset: the frame's origins ~R from the scene in direction (0.6, 0.8), zoom 1; every row sees the scene alike
OFFSET_FRAME = (512, 32768, 256, 256)  # width, height, rays per pixel, rows per band
# zoom: the scene at the centre of a 4096 x 4096 frame whose edges lie R away; the centre rows hold most hits
ZOOM_FRAME = (4096, 4096, 128, 64)


def far_view(kind, R):
    if kind == "offset":
        return dict(zoom_factor=1.0, offset_x=0.6 * R, offset_y=0.8 * R), OFFSET_FRAME
    return dict(zoom_factor=R / 2048), ZOOM_FRAME


FAR_VIEWS = [(k, R) for k in ("offset", "zoom") for R in DISTANCES]


@pytest.mark.parametrize("view", FAR_VIEWS, ids=[f"{k}-{R:.0e}" for k, R in FAR_VIEWS])
@pytest.mark.parametrize("case", FAR_CASES, ids=[c[0] for c in FAR_CASES])
def test_far_view_against_brute_force(case, view, api, scenes):
    cid, name, accel, route, mode, depth = case
    kind, R = view
    v, (w, h, n, band) = far_view(kind, R)
    if mode == MODE_LOCAL and kind == "zoom":
        pytest.skip("a zoomed-out tile meets more runs than the local table holds: the route is the tree")
    r = scenes.gpu(api, name, **accel)
    differing, hits, rays = against_brute_force(api, r, w, h, n, route, mode, FLOOR, band, max_trace_depth=depth, **v)
    print(f"{cid} {kind} R={R:.0e}: {differing} differing rays, {hits} hits of {rays} rays")
    assert hits >= FLOOR, f"only {hits} hits in {rays} rays"
    assert differing == 0, f"{differing} rays differ from the brute force ({hits} hits of {rays} rays)"
    # one band against the oracle: the centre rows of the frame
    acc = po.make_accel(**{k: v for k, v in accel.items() if k == "curve_width"}) if "curve_width" in accel else None
    c = h // 2
    against_oracle(api, scenes, r, name, w, h, n if kind == "zoom" else 64, route, (c, c + 2), accel=acc,
                   max_trace_depth=depth, **v)


@pytest.mark.parametrize("R", [1e5, 1e6])
@pytest.mark.parametrize("name", ["arch.xml", "dust.xml"])
def test_far_view_adjoints_against_brute_force(name, R, api, scenes):
    """color_adjoint and blur_adjoint trace with closest_chord: at a far view the tree and the brute force give the same."""
    import torch

    r = scenes.gpu(api, name)
    d = r.host.to_numpy()
    w, h, n = 512, 512, 256
    rng = np.random.default_rng(1)
    g = torch.from_numpy(rng.random((h, w, 4), dtype=np.float32)).cuda()
    sg = torch.from_numpy(rng.random((h, w), dtype=np.float32)).cuda()
    out = {}
    for trav in (0, TRAVERSAL_BRUTE_FORCE):
        p = api.default_frame_params(w, h, n, zoom_factor=1.0, offset_x=0.6 * R, offset_y=0.8 * R, max_trace_depth=0,
                                     traversal=trav)
        left = torch.zeros(d["color_left"].shape, dtype=torch.float64, device="cuda")
        right = torch.zeros(d["color_right"].shape, dtype=torch.float64, device="cuda")
        blur = torch.zeros(d["blur"].shape, dtype=torch.float64, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        r.scene.color_adjoint(p, g.data_ptr(), left.data_ptr(), right.data_ptr(), s)
        r.scene.blur_adjoint(p, sg.data_ptr(), blur.data_ptr(), s)
        torch.cuda.synchronize()
        out[trav] = [a.cpu().numpy() for a in (left, right, blur)]
    assert np.abs(out[0][0]).sum() > 0, "the view sees nothing"
    for a, b in zip(out[0], out[TRAVERSAL_BRUTE_FORCE]):
        np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-12)


# ---------------------------------------------------------------------------------------------------------------------
# B, C. grazing rays, ties built on purpose, degenerate trees
# ---------------------------------------------------------------------------------------------------------------------
# (id, scene, accel options, [(route, expected mode)], view, frame (w, h, n), hit floor)
INT_VIEW = dict(zoom_factor=2.0, offset_x=-6.0, offset_y=10.0, use_aa=0)  # exact origins, ray 0 along (1, 0)
ROUTES_SMALL = [(ROUTE_AUTO, MODE_TABLE), (ROUTE_TREE, MODE_TREE), (ROUTE_LOCAL_TABLE, MODE_LOCAL)]
ROUTES_LARGE = [(ROUTE_AUTO, MODE_CUT), (ROUTE_TREE, MODE_TREE), (ROUTE_LOCAL_TABLE, MODE_LOCAL)]
EDGE_CASES = [
    ("grid-grazing", "grid.xml", {}, ROUTES_SMALL, INT_VIEW, (256, 256, 64), 100_000),
    ("grid-grazing-width0", "grid.xml", dict(curve_width=0.0), ROUTES_SMALL, INT_VIEW, (256, 256, 64), 100_000),
    ("grid-grazing-zoom1", "grid.xml", {}, ROUTES_SMALL, dict(zoom_factor=1.0, offset_x=3.0, offset_y=-4.0, use_aa=0),
     (512, 512, 16), 100_000),
    ("ties-exact", "ties_exact.xml", {}, ROUTES_SMALL, dict(zoom_factor=2.0), (256, 256, 64), 100_000),
    ("ties-near", "ties_near.xml", {}, ROUTES_SMALL, dict(zoom_factor=2.0), (256, 256, 64), 100_000),
    ("ties-exact-cut", "ties_exact_dust.xml", {}, ROUTES_LARGE, INT_VIEW, (256, 256, 64), 100_000),
    ("ties-near-cut", "ties_near_dust.xml", {}, ROUTES_LARGE, INT_VIEW, (256, 256, 64), 100_000),
    ("one-chord", "one_chord.xml", {}, ROUTES_SMALL, dict(zoom_factor=2.0), (256, 256, 64), 50_000),
    ("one-chord-far", "one_chord.xml", {}, ROUTES_SMALL, dict(zoom_factor=1.0, offset_x=6e4, offset_y=-8e4), (512, 4096, 256),
     10_000),
    ("zero-length", "zero_length.xml", {}, [(ROUTE_AUTO, MODE_CUT), (ROUTE_TREE, MODE_TREE)], dict(zoom_factor=2.0),
     (256, 256, 64), 100_000),
    ("identical-morton", "identical.xml", dict(tree=TREE_MORTON), [(ROUTE_TREE, MODE_TREE)], dict(zoom_factor=2.0), (256, 256, 64),
     100_000),
    ("identical-sah", "identical.xml", dict(tree=TREE_SAH), [(ROUTE_AUTO, MODE_CUT), (ROUTE_TREE, MODE_TREE)], dict(zoom_factor=2.0),
     (256, 256, 64), 100_000),
    ("runs64", "runs64.xml", {}, ROUTES_SMALL, dict(zoom_factor=2.0), (256, 256, 256), 20_000),
    ("runs65", "runs65.xml", {}, ROUTES_LARGE, dict(zoom_factor=2.0), (256, 256, 256), 20_000),
]


@pytest.mark.parametrize("case", EDGE_CASES, ids=[c[0] for c in EDGE_CASES])
def test_edge_scenes_against_brute_force_and_oracle(case, api, scenes):
    cid, name, accel, routes, view, (w, h, n), floor = case
    r = scenes.gpu(api, name, **accel)
    acc = po.make_accel(curve_width=accel["curve_width"]) if "curve_width" in accel else None
    for route, mode in routes:
        differing, hits, rays = against_brute_force(api, r, w, h, n, route, mode, floor, 64, **view)
        print(f"{cid} route {route}: {differing} differing rays, {hits} hits of {rays} rays")
        assert hits >= floor, f"only {hits} hits in {rays} rays"
        assert differing == 0, f"route {route}: {differing} rays differ from the brute force"
        c = h // 2
        assert against_oracle(api, scenes, r, name, w, h, n, route, (c - 2, c + 2), accel=acc, **view) > 0


def test_generated_scenes_are_what_they_claim(api, scenes):
    """Run counts and trees behind the edge cases: one run, 64 and 65 runs (the whole-scene table's limit), one chord per
    dust segment, a zero-length segment that still makes a chord."""
    assert scenes.gpu(api, "one_chord.xml").scene.stats.n_runs == 1
    assert scenes.gpu(api, "runs64.xml").scene.stats.n_runs == 64
    assert scenes.gpu(api, "runs65.xml").scene.stats.n_runs == 65
    dust = scenes.gpu(api, "dust.xml").scene.stats
    assert dust.n_chords == dust.n_runs == 3000
    assert scenes.gpu(api, "zero_length.xml").scene.stats.n_chords == 601
    assert scenes.gpu(api, "identical.xml", tree=TREE_SAH).scene.stats.n_runs == 301


@pytest.mark.parametrize("view", [dict(zoom_factor=2.0), dict(zoom_factor=1.0, offset_x=6e4, offset_y=-8e4)], ids=["near", "far"])
def test_one_run_tree_tests_each_chord_once(view, api, scenes):
    """A scene of one run has a root with one child: the tree route tests the run once per traced ray, never twice."""
    r = scenes.gpu(api, "one_chord.xml")
    p = params(api, 64, 64, 64, route=ROUTE_TREE, **view)
    out = r.render(p, want_hits=True, want_stats=True)
    rays, nodes, chords = out["stats"][:3]
    assert rays > 0
    assert chords == rays, f"{chords} chords tested for {rays} traced rays"
    plain = r.render(params(api, 64, 64, 64, route=ROUTE_TREE, traversal=TRAVERSAL_BRUTE_FORCE, **view), want_hits=True)
    assert np.array_equal(out["hits"], plain["hits"])
