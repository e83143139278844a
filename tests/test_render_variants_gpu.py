"""Every built variant of the render kernel against the CPU oracle, at the ray-count, tile and band edges where a kernel
goes wrong.

`k_render` is built as 21 kernels: mode (tree, whole-scene run table, local run table, cut table) x scene staging (shared or
global memory) x portal-capable x counting build, with the whole-scene table only staged in shared memory and the counting
build only portal-capable. rdc_scene_launch_plan reports which one a launch would use; the variant matrix below reaches
each of them once, and a plain check keeps the matrix complete. The other sections vary what the kernels compute with: the
number of rays per pixel against the units a tile's rays are dealt to, frame shapes against the 8x4 tiles and the 8-row
strips, shading records against stop-list walks, routes, leaf-run lengths and chord options, and the state a handle keeps
from one launch to the next.
"""
import os
import re

import numpy as np
import pytest

from helpers import GpuRenderer, bits, compare_images, copy_params
from oracle import pyoracle as po
from raytracingdiffusioncurves_b200.api import (MODE_CUT, MODE_LOCAL, MODE_TABLE, MODE_TREE, ROUTE_AUTO, ROUTE_LOCAL_TABLE,
                                                ROUTE_TREE)

gpu = pytest.mark.gpu

RGB_TOL = 1e-4  # absolute, fp32: the parity tolerance against the oracle
UNITS_TOL = 2e-6  # frames that differ only in how a pixel's rays are grouped into partial sums
MISS = 0xFFFFFFFF
STRIP_ROWS = 8  # RDC_STRIP_ROWS
SYNTH_PORTALS = "synth_portals"  # 1500 one-segment curves, every tenth pair joined by a portal


def variant_index(mode, smem, portals, stats):
    return ((mode * 2 + smem) * 2 + portals) * 2 + stats


def built_variants():
    """The kernels the library builds: the whole-scene table only with shared-memory staging, the counting build only
    on the portal-capable kernel."""
    return {(m, s, p, c) for m in (MODE_TREE, MODE_TABLE, MODE_LOCAL, MODE_CUT) for s in (0, 1) for p in (0, 1) for c in (0, 1)
            if not (m == MODE_TABLE and not s) and not (c and not p)}


@pytest.fixture(scope="module")
def api():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from raytracingdiffusioncurves_b200 import api as _api

    return _api


def synth_portals_xml(api) -> str:
    """The synthetic scene of test_parity_gpu.test_local_run_table_with_portals: curves 10k and 10k+1 are a portal pair."""
    xml = api.synth_xml(1500, 512, 512).decode()
    count = [0]

    def connect(m):
        c = count[0]
        count[0] += 1
        if c % 10 == 0:
            return f'<curve connects="{c + 1}" '
        if c % 10 == 1:
            return f'<curve connects="{c - 1}" '
        return m.group(0)

    return re.sub(r"<curve ", connect, xml)


class Scenes:
    """Scene files by name, their oracle ingest, GPU handles per accel options and oracle frames, each made once."""

    def __init__(self, api, oracle, xml_dir, tmp_dir):
        self.api, self.oracle, self.xml_dir = api, oracle, xml_dir
        synth = os.path.join(tmp_dir, "synth_portals.xml")
        with open(synth, "w") as fh:
            fh.write(synth_portals_xml(api))
        self.synth = synth
        self._dicts, self._gpu, self._frames = {}, {}, {}

    def path(self, name):
        return self.synth if name == SYNTH_PORTALS else os.path.join(self.xml_dir, name)

    def dict(self, name):
        if name not in self._dicts:
            self._dicts[name] = po.ingest_xml(self.path(name), True)
        return self._dicts[name]

    def gpu(self, name, **accel):
        key = (name, tuple(sorted(accel.items())))
        if key not in self._gpu:
            self._gpu[key] = GpuRenderer(self.path(name), accel=self.api.default_accel_options(**accel) if accel else None)
        return self._gpu[key]

    def fresh(self, name, **accel):
        return GpuRenderer(self.path(name), accel=self.api.default_accel_options(**accel) if accel else None)

    def frame(self, name, w, h, n, chords=None, **view):
        """The oracle's whole frame (image, blur map, hits); bands are rows of it. Route, units, strips and the counting
        build are the product's business and never change the oracle's answer. `chords`: make_accel keywords."""
        view = {k: v for k, v in view.items() if k not in ("route", "units_per_tile", "row_begin", "row_end")}
        key = (name, w, h, n, tuple(sorted((chords or {}).items())), tuple(sorted(view.items())))
        if key not in self._frames:
            accel = po.make_accel(**chords) if chords else None
            self._frames[key] = self.oracle.render(self.dict(name), po.make_params(w, h, n, **view), accel=accel, want_hits=True,
                                                   search="grid")
        return self._frames[key]


@pytest.fixture(scope="module")
def scenes(api, port_oracle, xml_dir, tmp_path_factory):
    return Scenes(api, port_oracle, xml_dir, str(tmp_path_factory.mktemp("variants")))


def params(api, w, h, n, **kw):
    return copy_params(po.make_params(w, h, n, **kw), api.FrameParams)


def plan_of(r, p, stats=False):
    """The hook's plan for `p`, with a counting buffer when `stats` (the hook only looks at whether there is one)."""
    import torch

    q = copy_params(p, type(p))
    buf = torch.zeros((9,), dtype=torch.int64, device="cuda") if stats else None
    q.stats = buf.data_ptr() if stats else None
    return r.scene.launch_plan(q)


def check_against_oracle(out, want, rows=slice(None)):
    """Hits bit-exact; RGB within RGB_TOL; the blur map's NaN pattern and values like test_render_parity_small."""
    oimg, oblur, ohits = (a[rows] for a in want)
    assert np.array_equal(out["hits"], ohits), f"{int((out['hits'] != ohits).sum())} hit ids differ from the oracle"
    compare_images(out["image"], oimg, RGB_TOL)
    assert np.array_equal(np.isnan(out["blur_map"]), np.isnan(oblur))
    m = ~np.isnan(oblur)
    assert np.max(np.abs(out["blur_map"][m] - oblur[m]), initial=0) <= 1e-4 * max(1.0, float(np.nanmax(oblur, initial=0)))


def assert_same_bits(a, b, what=""):
    for key in ("image", "blur_map", "hits"):
        if a[key] is not None and b[key] is not None:
            assert np.array_equal(bits(a[key]), bits(b[key])), f"{what}: {key} differs"


def assert_close_units(a, b, what=""):
    """Same hits and NaN pattern, RGB and blur within UNITS_TOL: the same samples summed in another grouping."""
    assert np.array_equal(a["hits"], b["hits"]), what
    for key, sl in (("image", np.s_[..., :3]), ("blur_map", np.s_[...])):
        x, y = a[key][sl], b[key][sl]
        assert np.array_equal(np.isnan(x), np.isnan(y)), f"{what}: {key} NaN pattern"
        m = ~np.isnan(x)
        d = float(np.max(np.abs(x[m] - y[m]), initial=0))
        assert d <= UNITS_TOL * max(1.0, float(np.max(np.abs(y[m]), initial=0))), f"{what}: {key} differs by {d}"


# ---------------------------------------------------------------------------------------------------------------------
# A. the variant matrix: one case per built kernel
# ---------------------------------------------------------------------------------------------------------------------
# (id, scene, accel options, view, counting build, expected (mode, smem, portals))
FIT = dict(zoom_factor=512 / 18)  # a bundled scene's 512-pixel height in an 18-row frame
LADY_FIT = dict(zoom_factor=10.0)
MATRIX = [
    ("tree-smem", "arch.xml", {}, dict(FIT, route=ROUTE_TREE), False, (MODE_TREE, 1, 0)),
    ("tree-smem-portals-d2", "PortalDemo.xml", {}, dict(FIT, route=ROUTE_TREE, max_trace_depth=2), False, (MODE_TREE, 1, 1)),
    ("tree-smem-counting", "arch.xml", {}, dict(FIT, route=ROUTE_TREE), True, (MODE_TREE, 1, 1)),
    ("tree-global", "DiffusionCurvePack/lady_bug.xml", {}, dict(LADY_FIT, route=ROUTE_TREE), False, (MODE_TREE, 0, 0)),
    ("tree-global-portals-d31", SYNTH_PORTALS, {}, dict(zoom_factor=1.0, offset_x=20.0, offset_y=-30.0, route=ROUTE_TREE,
                                                        max_trace_depth=31), False, (MODE_TREE, 0, 1)),
    ("tree-global-counting", SYNTH_PORTALS, {}, dict(zoom_factor=1.0, offset_x=20.0, offset_y=-30.0, route=ROUTE_TREE),
     True, (MODE_TREE, 0, 1)),
    ("table-smem", "arch.xml", {}, dict(FIT), False, (MODE_TABLE, 1, 0)),
    ("table-smem-portals-d31", "PortalDemo.xml", {}, dict(FIT, max_trace_depth=31), False, (MODE_TABLE, 1, 1)),
    ("table-smem-counting", "test3.xml", {}, dict(FIT), True, (MODE_TABLE, 1, 1)),
    ("local-smem", "test4.xml", {}, dict(zoom_factor=1.0, route=ROUTE_LOCAL_TABLE), False, (MODE_LOCAL, 1, 0)),
    ("local-smem-portals-d0", "PortalDemo.xml", {}, dict(zoom_factor=1.0, offset_x=-40.0, offset_y=25.0, route=ROUTE_LOCAL_TABLE,
                                                         max_trace_depth=0), False, (MODE_LOCAL, 1, 1)),
    ("local-smem-counting", "test5.xml", {}, dict(zoom_factor=1.0, route=ROUTE_LOCAL_TABLE), True, (MODE_LOCAL, 1, 1)),
    ("local-global", "DiffusionCurvePack/dolphin.xml", {}, dict(zoom_factor=0.5, offset_x=60.0, offset_y=-40.0,
                                                                route=ROUTE_LOCAL_TABLE), False, (MODE_LOCAL, 0, 0)),
    ("local-global-portals-d2", SYNTH_PORTALS, {}, dict(zoom_factor=1.0, offset_x=20.0, offset_y=-30.0, route=ROUTE_LOCAL_TABLE,
                                                        max_trace_depth=2), False, (MODE_LOCAL, 0, 1)),
    ("local-global-counting", "DiffusionCurvePack/lady_bug.xml", {}, dict(zoom_factor=1.0, offset_x=-30.0, offset_y=20.0,
                                                                          route=ROUTE_LOCAL_TABLE), True, (MODE_LOCAL, 0, 1)),
    ("cut-smem", "test4.xml", {}, dict(FIT), False, (MODE_CUT, 1, 0)),
    ("cut-smem-portals-d2", "PortalDemo.xml", dict(run_length=2), dict(FIT, max_trace_depth=2), False, (MODE_CUT, 1, 1)),
    ("cut-smem-counting", "test4.xml", {}, dict(zoom_factor=3.0, offset_x=10.0, offset_y=-5.0), True, (MODE_CUT, 1, 1)),
    ("cut-global", "DiffusionCurvePack/lady_bug.xml", {}, dict(LADY_FIT), False, (MODE_CUT, 0, 0)),
    ("cut-global-portals-d0", SYNTH_PORTALS, {}, dict(zoom_factor=1.0, offset_x=20.0, offset_y=-30.0, max_trace_depth=0),
     False, (MODE_CUT, 0, 1)),
    ("cut-global-counting", "DiffusionCurvePack/lady_bug.xml", {}, dict(zoom_factor=3.0, offset_x=-30.0, offset_y=20.0), True,
     (MODE_CUT, 0, 1)),
]
MATRIX_FRAME = (27, 18, 64)  # neither dimension a multiple of the 8x4 tile
_matrix_ran, _matrix_checked = set(), set()  # case ids started; kernels whose case passed


def test_matrix_covers_every_built_kernel_once():
    expected = [(*case[5], int(case[4])) for case in MATRIX]
    assert len(expected) == len(set(expected)), "two cases aim at the same kernel"
    assert set(expected) == built_variants(), f"missing {built_variants() - set(expected)}, not built {set(expected) - built_variants()}"
    assert len(built_variants()) == 21


@gpu
@pytest.mark.parametrize("case", MATRIX, ids=[c[0] for c in MATRIX])
def test_variant_matrix(case, api, scenes):
    cid, name, accel, view, stats, (mode, smem, portals) = case
    _matrix_ran.add(cid)
    w, h, n = MATRIX_FRAME
    r = scenes.gpu(name, **accel)
    p = params(api, w, h, n, **view)
    plan = plan_of(r, p, stats)
    got = (plan.mode, plan.smem, plan.portals, plan.stats)
    assert got == (mode, smem, portals, int(stats)), f"{cid}: the hook reports (mode, smem, portals, stats) = {got}"
    assert plan.built == 1 and plan.variant == variant_index(mode, smem, portals, int(stats))
    want = scenes.frame(name, w, h, n, **view)
    out = r.render(params(api, w, h, n, **view), want_hits=True, want_stats=stats)
    check_against_oracle(out, want)
    has_portals = r.scene.stats.has_portals
    if stats:
        plain = r.render(params(api, w, h, n, **view), want_hits=True)
        assert_same_bits(out, plain, "counting build against the plain build")
        primary_hits = int((want[2] != MISS).sum())
        shaded, deferred = out["stats"][3], out["stats"][4]
        if has_portals:
            assert shaded >= primary_hits
        else:
            assert shaded == primary_hits, f"{shaded} hits shaded, the oracle has {primary_hits} primary hits"
        if mode != MODE_LOCAL:
            assert deferred == 0
    # pinned units: the frame in two bands split at an odd row equals the whole frame bit for bit
    whole = r.render(params(api, w, h, n, units_per_tile=2, **view), want_hits=True, want_stats=stats)
    check_against_oracle(whole, want)
    parts = [r.render(params(api, w, h, n, units_per_tile=2, row_begin=b, row_end=e, **view), want_hits=True, want_stats=stats)
             for b, e in ((0, 7), (7, h))]
    joined = {k: np.concatenate([q[k] for q in parts]) for k in ("image", "blur_map", "hits")}
    assert_same_bits(joined, whole, "two bands against the whole frame")
    _matrix_checked.add((mode, smem, portals, int(stats)))


@gpu
def test_every_built_kernel_was_launched_and_checked():
    """Placed after the matrix in this file, so pytest runs it after the cases: 21 of 21 kernels launched and checked.
    Skipped when not every case of the matrix ran before it (a selection of tests)."""
    if len(_matrix_ran) < len(MATRIX):
        pytest.skip(f"only {len(_matrix_ran)} of the {len(MATRIX)} matrix cases ran")
    missing = built_variants() - _matrix_checked
    print(f"{len(_matrix_checked)}/{len(built_variants())} built kernels launched and checked")
    assert not missing, f"not checked: {sorted(missing)}"


# ---------------------------------------------------------------------------------------------------------------------
# B. ray-index edges: rays per pixel against units per tile
# ---------------------------------------------------------------------------------------------------------------------
RAY_COUNTS = [8, 9, 31, 33, 63, 65, 129, 257, 513, 1000]
RAY_SCENES = {  # scene -> (view, [(route, mode)])
    "arch.xml": (dict(zoom_factor=512 / 9), [(ROUTE_AUTO, MODE_TABLE), (ROUTE_TREE, MODE_TREE)]),
    "test4.xml": (dict(zoom_factor=1.0), [(ROUTE_AUTO, MODE_CUT), (ROUTE_LOCAL_TABLE, MODE_LOCAL)]),
    "DiffusionCurvePack/lady_bug.xml": (dict(zoom_factor=1.0, offset_x=-30.0, offset_y=20.0), [(ROUTE_AUTO, MODE_CUT), (ROUTE_LOCAL_TABLE, MODE_LOCAL),
                                                                                                (ROUTE_TREE, MODE_TREE)]),
}


def expected_units(requested, n, mode):
    """The documented reduction: at least 16 rays per unit of a tile, 64 on the local run table."""
    split = requested
    while split > 1 and n < (64 if mode == MODE_LOCAL else 16) * split:
        split //= 2
    return split


@gpu
@pytest.mark.parametrize("n", RAY_COUNTS)
@pytest.mark.parametrize("name", list(RAY_SCENES), ids=[s.split("/")[-1] for s in RAY_SCENES])
def test_ray_counts_against_units_per_tile(name, n, api, scenes):
    """13x9 frames, whole and as the band [3, 9): every route's hits equal the oracle's whatever the units per tile, and
    frames that differ only in units agree within UNITS_TOL. Chunks of 32 ray iterations per unit end at every offset."""
    view, routes = RAY_SCENES[name]
    w, h = 13, 9
    want = scenes.frame(name, w, h, n, **view)
    r = scenes.gpu(name)
    for route, mode in routes:
        for rows in ((0, h), (3, 9)):
            outs = []
            for units in (1, 2, 4, 8):
                p = params(api, w, h, n, route=route, units_per_tile=units, row_begin=rows[0], row_end=rows[1], **view)
                plan = plan_of(r, p)
                assert plan.mode == mode, (route, plan.mode)
                assert plan.units_per_tile == expected_units(units, n, mode), (route, units, plan.units_per_tile)
                out = r.render(p, want_hits=True)
                check_against_oracle(out, want, slice(*rows))
                outs.append(out)
            for units, out in zip((2, 4, 8), outs[1:]):
                assert_close_units(out, outs[0], f"route {route} rows {rows}: {units} units against 1")


# ---------------------------------------------------------------------------------------------------------------------
# C. frame-shape edges, in every mode
# ---------------------------------------------------------------------------------------------------------------------
SHAPE_MODES = [("table", "arch.xml", ROUTE_AUTO, MODE_TABLE), ("tree", "arch.xml", ROUTE_TREE, MODE_TREE),
               ("cut", "test4.xml", ROUTE_AUTO, MODE_CUT), ("local", "test4.xml", ROUTE_LOCAL_TABLE, MODE_LOCAL)]


def shape_view(name, h):
    return dict(zoom_factor=512 / max(h, 9)) if name == "arch.xml" else dict(zoom_factor=1.0, offset_x=5.0, offset_y=-3.0)


def reassemble_strips(parts, band_rows, stride):
    """The band's rows in order from the packed outputs of offsets 0..stride-1 (distributed.StripPlan's indexing)."""
    rows = []
    for t in range(-(-band_rows // STRIP_ROWS)):
        k = t // stride
        rows.append(parts[t % stride][k * STRIP_ROWS:k * STRIP_ROWS + min(STRIP_ROWS, band_rows - t * STRIP_ROWS)])
    return np.concatenate(rows)


@gpu
@pytest.mark.parametrize("mode_case", SHAPE_MODES, ids=[m[0] for m in SHAPE_MODES])
def test_frame_shapes(mode_case, api, scenes):
    _, name, route, mode = mode_case
    n = 24
    r = scenes.gpu(name)
    # tiny frames: a tile hangs over the right and the bottom edge, or the frame is a single pixel row or column
    for w in (1, 5, 9, 17):
        for h in (1, 3, 5):
            view = shape_view(name, h)
            p = params(api, w, h, n, route=route, **view)
            assert plan_of(r, p).mode == mode, (w, h)
            check_against_oracle(r.render(p, want_hits=True), scenes.frame(name, w, h, n, **view))
    # single-row bands at odd rows (row_skew 1 and 3)
    w, h = 17, 11
    view = shape_view(name, h)
    want = scenes.frame(name, w, h, n, **view)
    for b in (1, 3, 5, 9):
        check_against_oracle(r.render(params(api, w, h, n, route=route, row_begin=b, row_end=b + 1, **view), want_hits=True), want,
                             slice(b, b + 1))
    # strips of 8 rows dealt to 3 ranks over the band [5, 47), reassembled: the band rendered in one call
    w, h, b, e = 20, 50, 5, 47
    view = shape_view(name, h)
    want = scenes.frame(name, w, h, n, **view)
    band = r.render(params(api, w, h, n, route=route, units_per_tile=1, row_begin=b, row_end=e, **view), want_hits=True)
    check_against_oracle(band, want, slice(b, e))
    parts = [r.render(params(api, w, h, n, route=route, units_per_tile=1, row_begin=b, row_end=e, strip_stride=3, strip_offset=o,
                             **view), want_hits=True) for o in range(3)]
    joined = {k: reassemble_strips([q[k] for q in parts], e - b, 3) for k in ("image", "blur_map", "hits")}
    if mode == MODE_LOCAL:  # a strip's tiles start at its own first row, so the table (and which rays it defers) may differ
        assert_close_units(joined, band, "strips against the band")
    else:
        assert_same_bits(joined, band, "strips against the band")
    check_against_oracle(joined, want, slice(b, e))
    # an offset past the band's last strip: nothing to render, the buffers stay as they were
    import torch

    image = torch.full((STRIP_ROWS, w, 4), float("nan"), dtype=torch.float32, device="cuda")
    sigma = torch.full((STRIP_ROWS, w), float("nan"), dtype=torch.float32, device="cuda")
    p = params(api, w, h, n, route=route, row_begin=b, row_end=e, strip_stride=8, strip_offset=7, **view)
    r.scene.render(p, image.data_ptr(), sigma.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.isnan(image).all() and torch.isnan(sigma).all()
    # the scene far outside the frame: every ray misses
    w, h = 9, 5
    far = dict(zoom_factor=1.0, offset_x=1e8, offset_y=-1e8)
    want = scenes.frame(name, w, h, n, **far)
    assert (want[2] == MISS).all() and np.isnan(want[0][..., :3]).all()
    check_against_oracle(r.render(params(api, w, h, n, route=route, **far), want_hits=True), want)
    # zoom 0 (every pixel at one origin) and a negative zoom (a mirrored view)
    for zoom in (0.0, -1.5):
        z = dict(zoom_factor=zoom, offset_x=7.0, offset_y=3.0)
        p = params(api, w, h, n, route=route, **z)
        assert plan_of(r, p).mode == mode, zoom
        check_against_oracle(r.render(p, want_hits=True), scenes.frame(name, w, h, n, **z))


# ---------------------------------------------------------------------------------------------------------------------
# D. equalities the code states
# ---------------------------------------------------------------------------------------------------------------------
RECORD_MODES = [("table", "arch.xml", dict(zoom_factor=512 / 18), ROUTE_AUTO, MODE_TABLE),
                ("tree", "DiffusionCurvePack/lady_bug.xml", dict(zoom_factor=10.0), ROUTE_TREE, MODE_TREE),
                ("cut", "DiffusionCurvePack/lady_bug.xml", dict(zoom_factor=10.0), ROUTE_AUTO, MODE_CUT),
                ("local", "test4.xml", dict(zoom_factor=1.0), ROUTE_LOCAL_TABLE, MODE_LOCAL)]


@gpu
@pytest.mark.parametrize("mode_case", RECORD_MODES, ids=[m[0] for m in RECORD_MODES])
def test_shading_records_equal_stop_list_walks(mode_case, api, scenes):
    _, name, view, route, mode = mode_case
    w, h, n = 27, 18, 64
    records = scenes.gpu(name)
    walks = scenes.gpu(name, shading_records=-1)
    p = params(api, w, h, n, route=route, **view)
    assert plan_of(records, p).mode == mode and plan_of(walks, p).mode == mode
    a = records.render(params(api, w, h, n, route=route, **view), want_hits=True)
    b = walks.render(params(api, w, h, n, route=route, **view), want_hits=True)
    check_against_oracle(a, scenes.frame(name, w, h, n, **view))
    assert_same_bits(a, b, "shading records against stop-list walks")


ROUTE_SCENES = [("arch.xml", dict(zoom_factor=512 / 18), MODE_TABLE), ("test3.xml", dict(zoom_factor=512 / 18), None),
                ("test4.xml", dict(zoom_factor=1.0), MODE_CUT), ("DiffusionCurvePack/lady_bug.xml", dict(zoom_factor=1.0, offset_x=-30.0,
                                                                                                   offset_y=20.0), MODE_CUT)]


@gpu
@pytest.mark.parametrize("route_case", ROUTE_SCENES, ids=[c[0].split("/")[-1] for c in ROUTE_SCENES])
def test_routes_give_the_same_frame(route_case, api, scenes):
    """Units pinned: the tree, the whole-scene table and the cut table give the same bits; the local run table the same
    hits and pixels within UNITS_TOL (it adds the samples of the rays it defers to the tree at the end)."""
    name, view, auto_mode = route_case
    w, h, n = 27, 18, 128
    r = scenes.gpu(name)
    frames = {}
    for route in (ROUTE_TREE, ROUTE_AUTO, ROUTE_LOCAL_TABLE):
        p = params(api, w, h, n, route=route, units_per_tile=2, **view)
        frames[route] = (plan_of(r, p).mode, r.render(p, want_hits=True))
    check_against_oracle(frames[ROUTE_TREE][1], scenes.frame(name, w, h, n, **view))
    if auto_mode is not None:
        assert frames[ROUTE_AUTO][0] == auto_mode
    assert frames[ROUTE_TREE][0] == MODE_TREE and frames[ROUTE_LOCAL_TABLE][0] in (MODE_LOCAL, MODE_TREE)
    assert_same_bits(frames[ROUTE_AUTO][1], frames[ROUTE_TREE][1], f"route {frames[ROUTE_AUTO][0]} against the tree")
    assert_close_units(frames[ROUTE_LOCAL_TABLE][1], frames[ROUTE_TREE][1], "local run table against the tree")


@gpu
@pytest.mark.parametrize("name", ["test4.xml", "PortalDemo.xml"])
def test_run_length_does_not_change_the_frame(name, api, scenes):
    """Leaf runs of 1..8 chords, or chosen from the density (0): other trees over the same chords, the same frame."""
    w, h, n = 27, 18, 32
    view = dict(zoom_factor=512 / h, route=ROUTE_TREE)
    want = scenes.frame(name, w, h, n, **view)
    first = None
    for run_length in range(9):
        out = scenes.fresh(name, run_length=run_length).render(params(api, w, h, n, **view), want_hits=True)
        check_against_oracle(out, want)
        if first is None:
            first = out
        else:
            assert_same_bits(out, first, f"run_length {run_length} against 0")


# ---------------------------------------------------------------------------------------------------------------------
# E. chord options against the oracle
# ---------------------------------------------------------------------------------------------------------------------
CHORD_OPTIONS = [dict(flatness_tolerance=0.01), dict(flatness_tolerance=0.5), dict(curve_width=0.0), dict(curve_width=0.05),
                 dict(max_chords_per_segment=1), dict(max_chords_per_segment=3)]


@gpu
@pytest.mark.parametrize("opts", CHORD_OPTIONS, ids=[f"{k}={v}" for o in CHORD_OPTIONS for k, v in o.items()])
@pytest.mark.parametrize("name", ["test4.xml", "PortalDemo.xml", "DiffusionCurvePack/lady_bug.xml"],
                         ids=["test4", "PortalDemo", "lady_bug"])
def test_chord_options(name, opts, api, scenes):
    r = scenes.fresh(name, **opts)
    geom, ids = r.scene.chords()
    ogeom, oids = scenes.oracle.chords(scenes.dict(name), po.make_accel(**opts))
    assert np.array_equal(ids, oids)
    assert np.array_equal(bits(geom), bits(ogeom))
    w, h, n = 27, 18, 32
    for view in (dict(zoom_factor=512 / h), dict(zoom_factor=1.0, offset_x=-30.0, offset_y=20.0, route=ROUTE_LOCAL_TABLE)):
        out = r.render(params(api, w, h, n, **view), want_hits=True)
        check_against_oracle(out, scenes.frame(name, w, h, n, chords=opts, **view))


# ---------------------------------------------------------------------------------------------------------------------
# F. what a handle keeps between launches
# ---------------------------------------------------------------------------------------------------------------------
def handle_sequence(name, h, view):
    """Unlike launches in a row on one handle: (what, launches as keyword sets, counting build, expected (mode, units, group)).
    The first launch combines two units in global memory; a later one needs more partial sums and grows them; group mode
    and the global-memory combine alternate; the rays per pixel change; the first launch ends the sequence again."""
    first = ("tree 65 rays, 2 units", [dict(view, n=65, route=ROUTE_TREE, units_per_tile=2)], False, (MODE_TREE, 2, 0))
    mode = MODE_TABLE if name == "arch.xml" else MODE_CUT
    if mode == MODE_TABLE:
        grow = ("tree 65 rays, 4 units", [dict(view, n=65, route=ROUTE_TREE, units_per_tile=4)], False, (MODE_TREE, 4, 0))
    else:
        grow = ("local 513 rays, 8 units", [dict(view, n=513, route=ROUTE_LOCAL_TABLE, units_per_tile=8)], False, (MODE_LOCAL, 8, 0))
    return [
        first,
        grow,
        ("9 rays", [dict(view, n=9)], False, (mode, 1, 0)),
        ("129 rays, 8 units, bands", [dict(view, n=129, units_per_tile=8, row_begin=0, row_end=5),
                                      dict(view, n=129, units_per_tile=8, row_begin=5, row_end=h)], False, (mode, 8, 8)),
        ("counting build", [dict(view, n=64)], True, (mode, None, None)),
        ("strips", [dict(view, n=64, units_per_tile=2, strip_stride=2, strip_offset=o) for o in (0, 1)], False, (mode, 2, 2)),
        ("9 rays, again", [dict(view, n=9)], False, (mode, 1, 0)),
        (first[0] + ", again",) + first[1:],
    ]


HANDLE_SCENES = [("arch.xml", dict(zoom_factor=512 / 14)), ("test4.xml", dict(zoom_factor=1.0, offset_x=5.0, offset_y=-3.0))]


@gpu
@pytest.mark.parametrize("name,view", HANDLE_SCENES, ids=[c[0] for c in HANDLE_SCENES])
def test_handle_state_between_launches(name, view, api, scenes):
    """One handle renders a sequence of unlike launches (handle_sequence); each equals the same launch on a fresh handle,
    bit for bit. Covers the base-direction table (new rays per pixel), the partial sums growing, the tile arrival counters
    rewinding, and switching between group mode and the global-memory combine, on the whole-scene table (arch.xml) and on
    the cut and local tables (test4.xml)."""
    w, h = 21, 14
    steps = handle_sequence(name, h, view)

    def launch(r, kw, stats):
        kw = dict(kw)
        n = kw.pop("n")
        p = params(api, w, h, n, **kw)
        plan, out = plan_of(r, p, stats), r.render(p, want_hits=True, want_stats=stats)
        if p.strip_stride > 1:  # only the strips of this offset are written, packed from the first row
            rows = sum(min(STRIP_ROWS, h - t * STRIP_ROWS) for t in range(-(-h // STRIP_ROWS)) if t % p.strip_stride == p.strip_offset)
            out = {k: out[k][:rows] for k in ("image", "blur_map", "hits")}
        return plan, out

    shared = scenes.fresh(name)
    for what, launches, stats, (mode, units, group) in steps:
        for kw in launches:
            plan, got = launch(shared, kw, stats)
            assert plan.mode == mode, what
            if units is not None:
                assert (plan.units_per_tile, plan.group) == (units, group), what
            _, want = launch(scenes.fresh(name), kw, stats)
            assert_same_bits(got, want, what)
