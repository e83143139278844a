"""rdc_scene_pick / rdc_scene_pick_frame: the nearest chord to a point, against a float32 numpy brute force over the chords.

The pick is the lexicographic minimum of (d2, chord id) over the chords within max_distance, with d2, the fraction s and
the nearest point c computed exactly as rdc_point_chord computes them, so every field is compared bit for bit: whichever
tree the scene was built with and however long its leaf runs are, the tree walk must find what the brute force finds.
"""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from helpers import XML_DIR, bits, scene_ids

pytestmark = pytest.mark.gpu

F = np.float32
INF = math.inf
NAN_BITS = 0x7FFFFFFF
FAMILIES = ("color_left", "color_right", "blur", "weight", "weight_degree")
SYNTH_PORTALS = "synth_portals"
SYNTH_100K = "synth_100k"


@pytest.fixture(scope="module")
def api():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from raytracingdiffusioncurves_b200 import api as _api

    return _api


def stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def synth_portals_xml(api) -> str:
    """1500 one-segment curves of the synthetic generator; curves 10k and 10k+1 are a portal pair."""
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


_HOSTS = {}


def host_scene(api, name):
    """Scene name -> (HostScene, numpy arrays), each ingested once."""
    if name not in _HOSTS:
        if name == SYNTH_PORTALS:
            h = api.HostScene.from_xml_text(synth_portals_xml(api).encode())
        elif name == SYNTH_100K:
            h = api.HostScene.from_xml_text(api.synth_xml(100000, 8192, 8192))
        else:
            h = api.HostScene.from_xml_file(os.path.join(XML_DIR, name))
        _HOSTS[name] = (h, h.to_numpy())
    return _HOSTS[name]


def build(api, arrays, **opts):
    return api.Scene(arrays, api.default_accel_options(**opts), stream())


# ---------------------------------------------------------------------------------------------------------------------
# the product's answers
# ---------------------------------------------------------------------------------------------------------------------
def buffers(pts, with_stops):
    """Device copies of the points and room for the answers (ready when this returns)."""
    import torch

    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 2)
    n = len(pts)
    d_pts = torch.from_numpy(pts).cuda()
    out = torch.empty((max(n, 1), 32), dtype=torch.uint8, device="cuda")
    stops = torch.empty((max(n, 1), 3, 4), dtype=torch.float32, device="cuda") if with_stops else None
    torch.cuda.synchronize()
    return out, stops, d_pts


def pick(api, scene, pts, md=INF, orzan=1, with_stops=False, on=None, bufs=None):
    """Picks `pts`; with `bufs` (buffers()) it only enqueues and returns them for fetch()."""
    res = bufs if bufs is not None else buffers(pts, with_stops)
    out, stops, d_pts = res
    n = len(np.asarray(pts).reshape(-1, 2))
    scene.pick(d_pts.data_ptr(), n, out.data_ptr(), stops.data_ptr() if stops is not None else 0, md, orzan,
               stream() if on is None else on)
    return res if bufs is not None else fetch(api, res, n)


def fetch(api, res, n):
    import torch

    out, stops, _ = res
    torch.cuda.synchronize()
    got = out.cpu().numpy().view(api.PICK_DTYPE).reshape(-1)[:n]
    return (got, stops.cpu().numpy()[:n]) if stops is not None else got


def pick_frame(api, scene, p, md=INF, with_stops=False):
    import torch

    n = (p.row_end - p.row_begin) * p.image_width
    out = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    stops = torch.empty((n, 3, 4), dtype=torch.float32, device="cuda") if with_stops else None
    scene.pick_frame(p, out.data_ptr(), stops.data_ptr() if with_stops else 0, md, stream())
    return fetch(api, (out, stops, None), n)


# ---------------------------------------------------------------------------------------------------------------------
# the reference: float32 brute force with the (d2, id) rule, one rounding per operation like rdc_point_chord
# ---------------------------------------------------------------------------------------------------------------------
def nearest(geom, pts, md2):
    """Index of the nearest chord (-1: none with d2 <= md2), and its s, c and d2, for every point."""
    ax, ay, bx, by = (geom[:, i].astype(F) for i in range(4))
    ex, ey = bx - ax, by - ay
    ee = ex * ex + ey * ey
    n = len(pts)
    idx = np.full(n, -1, np.int64)
    out_s, out_x, out_y, out_d2 = (np.zeros(n, F) for _ in range(4))
    chunk = max(1, (1 << 22) // max(len(geom), 1))
    with np.errstate(all="ignore"):
        for lo in range(0, n, chunk):
            px = pts[lo:lo + chunk, 0:1].astype(F)
            py = pts[lo:lo + chunk, 1:2].astype(F)
            wx, wy = px - ax, py - ay
            s = np.where(ee > 0, (wx * ex + wy * ey) / np.where(ee > 0, ee, F(1)), F(0)).astype(F)
            s = np.minimum(np.maximum(s, F(0)), F(1))
            x = ax + s * ex
            y = ay + s * ey
            dx, dy = px - x, py - y
            d2 = dx * dx + dy * dy
            d2m = np.where(d2 <= md2, d2, F(np.inf))
            j = np.argmin(d2m, axis=1)  # first minimum: the smallest id among equal d2
            r = np.arange(len(j))
            ok = d2[r, j] <= md2
            idx[lo:lo + chunk] = np.where(ok, j, -1)
            out_s[lo:lo + chunk], out_x[lo:lo + chunk], out_y[lo:lo + chunk], out_d2[lo:lo + chunk] = s[r, j], x[r, j], y[r, j], d2[r, j]
    finite = np.isfinite(pts).all(axis=1)
    idx[~finite] = -1
    return idx, out_s, out_x, out_y, out_d2


def spline_normal(t, v):
    """rdc_spline_normal in float32, operation for operation. v: [n, 4, 2]."""
    t = t.astype(F)
    d3 = F(3) * t * t
    d0 = F(-3) * t * t + F(6) * t - F(3)
    d1 = F(9) * t * t - F(12) * t
    d2 = F(-9) * t * t + F(6) * t + F(3)
    sixth = F(1) / F(6)
    nx = sixth * (d3 * v[:, 3, 1] + v[:, 0, 1] * d0 + v[:, 1, 1] * d1 + v[:, 2, 1] * d2)
    ny = -sixth * (d3 * v[:, 3, 0] + v[:, 0, 0] * d0 + v[:, 1, 0] * d1 + v[:, 2, 0] * d2)
    return nx, ny


def is_right(u, dx, dy, v, orzan):
    """rdc_is_ray_right: ((n . D) <= 0) != orzan."""
    nx, ny = spline_normal(u, v)
    return ((nx * dx + ny * dy) <= F(0)) != bool(orzan)


def brute(d, geom, ids, pts, md=INF, orzan=1):
    """What rdc_scene_pick must return for every point, as a PICK_DTYPE array."""
    from raytracingdiffusioncurves_b200 import api

    pts = np.asarray(pts, F).reshape(-1, 2)
    md2 = F(F(md) * F(md))
    idx, s, x, y, d2 = nearest(geom, pts, md2)
    hit = idx >= 0
    j = np.where(hit, idx, 0)
    seg = ids[j, 0]
    k, K = ids[j, 1], ids[j, 2]
    u = ((k.astype(F) + s) / K.astype(F)).astype(F)
    ordinal = d["curve_index"][seg]
    curve = d["curve_map"][seg]
    v = d["vertices"][:, :2][d["segment_indices"][seg][:, None] + np.arange(4)].astype(F)
    with np.errstate(all="ignore"):
        right = is_right(u, (x - pts[:, 0]).astype(F), (y - pts[:, 1]).astype(F), v, orzan)
    flags = right.astype(np.uint32) * np.uint32(1) | (d["curve_connect"][curve] >= 0).astype(np.uint32) * np.uint32(2)
    out = np.zeros(len(pts), api.PICK_DTYPE)
    nan = np.uint32(NAN_BITS).view(F)
    none = np.uint32(0xFFFFFFFF)
    out["chord"] = np.where(hit, j, none)
    out["segment"] = np.where(hit, seg, none)
    out["curve"] = np.where(hit, curve, none)
    out["flags"] = np.where(hit, flags, 0)
    out["u"] = np.where(hit, (u + ordinal.astype(F)).astype(F), nan)
    out["distance"] = np.where(hit, np.sqrt(d2).astype(F), F(np.inf))
    out["x"] = np.where(hit, x, nan)
    out["y"] = np.where(hit, y, nan)
    return out


def assert_same_picks(got, want, what=""):
    for f in ("chord", "segment", "curve", "flags"):
        bad = np.nonzero(got[f] != want[f])[0]
        assert len(bad) == 0, f"{what}: {f} differs at {len(bad)} points, first {bad[0]}: {got[bad[0]]} vs {want[bad[0]]}"
    for f in ("u", "distance", "x", "y"):
        g, w = got[f], want[f]
        same = (bits(g) == bits(w)) | (np.isnan(g) & np.isnan(w))
        bad = np.nonzero(~same)[0]
        assert len(bad) == 0, f"{what}: {f} bits differ at {len(bad)} points, first {bad[0]}: {got[bad[0]]} vs {want[bad[0]]}"


def probe_points(geom, d, count, seed):
    """Random points in the scene box +- a margin, chord end points and midpoints (distance 0), points far outside."""
    rng = np.random.default_rng(seed)
    lo = np.minimum(geom[:, :2].min(axis=0), geom[:, 2:].min(axis=0))
    hi = np.maximum(geom[:, :2].max(axis=0), geom[:, 2:].max(axis=0))
    ext = np.maximum(hi - lo, 1.0)
    n_rand, n_end, n_mid, n_far = count // 2, count // 5, count // 5, count - count // 2 - 2 * (count // 5)
    rand = lo - 0.1 * ext + rng.random((n_rand, 2)) * 1.2 * ext
    pick_c = rng.integers(0, len(geom), n_end + n_mid)
    ends = np.where(rng.random((n_end, 1)) < 0.5, geom[pick_c[:n_end], :2], geom[pick_c[:n_end], 2:])
    mids = (geom[pick_c[n_end:], :2] + geom[pick_c[n_end:], 2:]) * F(0.5)
    ang = rng.random(n_far) * 2 * np.pi
    far = (lo + hi) / 2 + np.stack([np.cos(ang), np.sin(ang)], 1) * ext.max() * rng.uniform(3, 1000, (n_far, 1))
    return np.concatenate([rand, ends, mids, far]).astype(F)


_BRUTE = {}

BUILDS = [("sah-rl1", dict(tree=2, run_length=1)), ("sah-rl8", dict(tree=2, run_length=8)),
          ("morton-rl1", dict(tree=1, run_length=1)), ("morton-rl8", dict(tree=1, run_length=8))]


@pytest.mark.parametrize("name", scene_ids() + [SYNTH_PORTALS])
def test_pick_equals_the_brute_force(name, api):
    host, d = host_scene(api, name)
    first = None
    for label, opts in BUILDS:
        scene = build(api, host.arrays, **opts)
        geom, ids = scene.chords()
        if first is None:
            first = (geom, ids)
            pts = probe_points(geom, d, 4096, seed=len(geom))
            want = brute(d, geom, ids, pts)
        else:  # the chords do not depend on the tree or the run length
            assert np.array_equal(bits(geom), bits(first[0])) and np.array_equal(ids, first[1])
        got = pick(api, scene, pts)
        assert_same_picks(got, want, f"{name} {label}")
        assert (got["chord"] != api.PICK_NONE).all()
        scene.close()


def test_pick_on_the_100k_curve_scene_with_points_on_padded_box_edges(api):
    host, d = host_scene(api, SYNTH_100K)
    rng = np.random.default_rng(3)
    for label, opts in [BUILDS[1], BUILDS[3]]:
        scene = build(api, host.arrays, **opts)
        geom, ids = scene.chords()
        pad = F(scene.stats.pad)
        # runs of 8 chords of one segment (k // 8) and their padded boxes, as the build makes them
        key = ids[:, 0].astype(np.int64) * 4096 + ids[:, 1] // 8
        order = np.argsort(key, kind="stable")
        starts = np.r_[0, np.nonzero(np.diff(key[order]))[0] + 1]
        xs = np.minimum(geom[order, 0], geom[order, 2]), np.maximum(geom[order, 0], geom[order, 2])
        ys = np.minimum(geom[order, 1], geom[order, 3]), np.maximum(geom[order, 1], geom[order, 3])
        runs = rng.choice(len(starts), 80, replace=False)
        x0 = np.minimum.reduceat(xs[0], starts)[runs] - pad
        x1 = np.maximum.reduceat(xs[1], starts)[runs] + pad
        y0 = np.minimum.reduceat(ys[0], starts)[runs] - pad
        y1 = np.maximum.reduceat(ys[1], starts)[runs] + pad
        t = rng.random(80).astype(F)
        edges = np.concatenate([np.stack([x0, y0 + t * (y1 - y0)], 1), np.stack([x1, y0 + t * (y1 - y0)], 1),
                                np.stack([x0 + t * (x1 - x0), y0], 1), np.stack([x0 + t * (x1 - x0), y1], 1),
                                np.stack([x0, y0], 1), np.stack([x1, y1], 1)]).astype(F)
        pts = np.concatenate([edges, probe_points(geom, d, 200, seed=9)])
        assert_same_picks(pick(api, scene, pts), brute(d, geom, ids, pts), f"100k {label}")
        scene.close()


TIE_XML = """<!DOCTYPE CurveSetXML>
<curve_set image_width="512" image_height="512" nb_curves="2" >
{curves}
</curve_set>
"""
TIE_CURVE = """ <curve nb_control_points="4" nb_left_colors="2" nb_right_colors="2" nb_blur_points="2" lifetime="32" use_endcap="false" >
  <control_points_set>{points}</control_points_set>
  <left_colors_set><left_color G="0" R="0" globalID="0" B="255" /><left_color G="0" R="0" globalID="10" B="255" /></left_colors_set>
  <right_colors_set><right_color G="0" R="255" globalID="0" B="0" /><right_color G="0" R="255" globalID="10" B="0" /></right_colors_set>
  <blur_points_set><best_scale value="0" globalID="0" /><best_scale value="0" globalID="10" /></blur_points_set>
  <weight_set><weight globalID="0" w="1" /><weight globalID="10" w="1" /></weight_set>
  <weight_degree_set><weight_degree globalID="0" w="0.5" /><weight_degree globalID="10" w="0.5" /></weight_degree_set>
 </curve>"""


def test_ties_go_to_the_smaller_chord_id(api):
    """Two curves mirrored about the scene's y = 0 (XML x = 256 in an Orzan save): negation commutes with rounding, so
    their chords are exact mirror images and a point on y = 0 is equally far from both. Shared end points tie too."""
    ys = [(100, 60), (200, 75), (300, 40), (400, 70)]  # (XML y -> scene x, XML x offset from 256 -> scene y)
    curves = []
    for sign in (1, -1):
        pts = "".join(f'<control_point y="{a}" x="{256 + sign * b}" />' for a, b in ys)
        curves.append(TIE_CURVE.format(points=pts))
    host = api.HostScene.from_xml_text(TIE_XML.format(curves="\n".join(curves)).encode())
    d = host.to_numpy()
    for label, opts in BUILDS:
        scene = build(api, host.arrays, **opts)
        geom, ids = scene.chords()
        seg_curve = d["curve_map"][ids[:, 0]]
        a = np.nonzero(seg_curve == 0)[0]
        b = np.nonzero(seg_curve == 1)[0]
        assert len(a) == len(b) and np.array_equal(bits(geom[a][:, [0, 2]]), bits(geom[b][:, [0, 2]]))
        assert np.array_equal(bits(geom[a][:, [1, 3]]), bits(-geom[b][:, [1, 3]]))
        xs = np.linspace(geom[:, [0, 2]].min() + 1, geom[:, [0, 2]].max() - 1, 101, dtype=F)
        mirror = np.stack([xs, np.zeros_like(xs)], 1)
        shared = geom[a[:-1], 2:4]  # end of chord k = start of chord k + 1
        pts = np.concatenate([mirror, shared]).astype(F)
        got = pick(api, scene, pts)
        want = brute(d, geom, ids, pts)
        assert_same_picks(got, want, f"ties {label}")
        assert (d["curve_map"][got["segment"][:len(xs)]] == 0).all(), "a tie between the two curves went to the larger id"
        # the brute force really sees a tie: the mirrored chord is exactly as far
        _, _, _, _, d2a = nearest(geom[b], mirror, F(np.inf))
        assert np.array_equal(bits(d2a), bits(nearest(geom[a], mirror, F(np.inf))[4]))
        # at a shared end point chord k + 1 has d2 = 0 and chord k has d2 = 0 too where a + (b - a) rounds to b: a tie
        d2k = np.array([nearest(geom[c:c + 1], shared[i:i + 1], F(np.inf))[4][0] for i, c in enumerate(a[:-1])], F)
        tied = d2k == 0
        assert tied.sum() >= len(tied) // 2
        assert np.array_equal(got["chord"][len(xs):][tied], a[:-1][tied]), "a shared end point went to the later chord"
        assert (got["distance"][len(xs):] == 0).all()
        scene.close()


def test_max_distance_and_non_finite_points(api):
    host, d = host_scene(api, "arch.xml")
    scene = build(api, host.arrays)
    geom, ids = scene.chords()
    pts = probe_points(geom, d, 2048, seed=1)
    bad = np.array([[np.nan, 0], [0, np.nan], [np.inf, 0], [0, -np.inf], [np.nan, np.inf]], F)
    pts = np.concatenate([pts, bad])
    for md in (0.5, 3.0, 40.0, INF):
        got = pick(api, scene, pts, md=md)
        want = brute(d, geom, ids, pts, md=md)
        assert_same_picks(got, want, f"max_distance {md}")
        if md != INF:
            assert (got["chord"] == api.PICK_NONE).any() and (got["chord"] != api.PICK_NONE).any()
        miss = got[got["chord"] == api.PICK_NONE]
        assert (miss["segment"] == api.PICK_NONE).all() and (miss["curve"] == api.PICK_NONE).all() and (miss["flags"] == 0).all()
        assert np.isinf(miss["distance"]).all() and np.isnan(miss["u"]).all() and np.isnan(miss["x"]).all() and np.isnan(miss["y"]).all()
        assert (got["chord"][-len(bad):] == api.PICK_NONE).all()
    got, stops = pick(api, scene, bad, with_stops=True)
    assert np.isnan(stops).all()
    assert pick(api, scene, np.zeros((0, 2), F)).shape == (0,)


def centres(api, p):
    """rdc_view_pixel_to_scene for every pixel of the band, restated in float32 (tests/test_pick_cpu.py pins it)."""
    w, h = p.image_width, p.image_height
    ix = np.arange(w, dtype=np.int64)
    iy = np.arange(p.row_begin, p.row_end, dtype=np.int64)

    def signed(v):
        return ((v % (1 << 32)) ^ (1 << 31)) - (1 << 31)

    cx = signed(ix - w // 2)
    cy = signed((h - iy) - h // 2) if p.use_diffusion_curve_save else signed(iy - h // 2)
    z = F(p.zoom_factor)
    x = (cx.astype(F) * z + F(p.offset_x)).astype(F) + F(0.5) * z
    y = (cy.astype(F) * z + F(p.offset_y)).astype(F) + F(0.5) * z
    gx, gy = np.meshgrid(x.astype(F), y.astype(F))
    pts = np.stack([gx, gy], -1).reshape(-1, 2).astype(F)
    for k in (0, len(pts) - 1, len(pts) // 3):  # the restatement is the library's mapping
        r, c = divmod(k, w)
        assert tuple(F(v) for v in api.view_pixel_to_scene(p, c, p.row_begin + r)) == tuple(pts[k])
    return pts


@pytest.mark.parametrize("orzan", [1, 0])
def test_pick_frame_equals_pick_on_the_pixel_centres(api, orzan):
    opts = api.default_ingest_options(use_diffusion_curve_save=orzan)
    host = api.HostScene.from_xml_file(os.path.join(XML_DIR, "arch.xml"), opts)
    scene = build(api, host.arrays)
    views = [api.default_frame_params(1920, 1080, 8, zoom_factor=512 / 1080),                          # headline view
             api.default_frame_params(320, 200, 8, zoom_factor=0.02, offset_x=-128, offset_y=0),        # close-up
             api.default_frame_params(64, 48, 8, zoom_factor=3.0, offset_x=5e4, offset_y=-3e4),          # far away
             api.default_frame_params(1, 1, 8), api.default_frame_params(17, 5, 8, zoom_factor=31.0)]
    for p in views:
        p.use_diffusion_curve_save = orzan
        for md in (INF, 6.0):
            got, stops = pick_frame(api, scene, p, md=md, with_stops=True)
            want, want_stops = pick(api, scene, centres(api, p), md=md, orzan=orzan, with_stops=True)
            assert_same_picks(got, want, f"frame {p.image_width}x{p.image_height} md {md}")
            assert np.array_equal(bits(stops), bits(want_stops))
    # an odd band reassembled into the whole frame
    p = api.default_frame_params(203, 77, 8, zoom_factor=3.1, use_diffusion_curve_save=orzan)
    whole = pick_frame(api, scene, p)
    parts = []
    for b, e in ((0, 13), (13, 40), (40, 77)):
        p.row_begin, p.row_end = b, e
        parts.append(pick_frame(api, scene, p))
    assert np.array_equal(np.concatenate(parts).view(np.uint8), whole.view(np.uint8))
    p.row_begin, p.row_end, p.strip_stride = 0, 77, 2
    with pytest.raises(api.RdcError, match="strip"):
        pick_frame(api, scene, p)


# ---------------------------------------------------------------------------------------------------------------------
# side and stops
# ---------------------------------------------------------------------------------------------------------------------
def interp64(index, us, vals, curve, u):
    """DeviceCode.cu:36-44 in float64: linear walk from the curve's first stop, strict '<'."""
    start, count = (int(v) for v in index[curve])
    ind = start
    while ind < start + count and us[ind + 1] < u:
        ind += 1
    with np.errstate(all="ignore"):
        ratio = (np.float64(u) - us[ind]) / (np.float64(us[ind + 1]) - us[ind])
        return (1 - ratio) * vals[ind].astype(np.float64) + ratio * vals[ind + 1].astype(np.float64)


def stops64(d, got):
    out = np.full((len(got), 3, 4), np.nan)
    for i, g in enumerate(got):
        if g["chord"] == 0xFFFFFFFF:
            continue
        c, u = int(g["curve"]), g["u"]
        out[i, 0, :3] = interp64(d["color_left_index"], d["color_left_u"], d["color_left"], c, u)
        out[i, 1, :3] = interp64(d["color_right_index"], d["color_right_u"], d["color_right"], c, u)
        out[i, 0, 3] = interp64(d["blur_index"], d["blur_u"], d["blur"], c, u)
        out[i, 1, 3] = interp64(d["weight_index"], d["weight_u"], d["weight"], c, u)
        out[i, 2, 0] = interp64(d["weight_degree_index"], d["weight_degree_u"], d["weight_degree"], c, u)
        out[i, 2, 1:] = 0
    return out


@pytest.mark.parametrize("name", ["arch.xml", "DiffusionCurvePack/lady_bug.xml", "PortalDemo.xml", "weight_demo.xml", SYNTH_PORTALS])
@pytest.mark.parametrize("records", [0, -1], ids=["records", "walks"])
def test_side_and_stops_at_the_pick(name, records, api):
    host, d = host_scene(api, name)
    scene = build(api, host.arrays, shading_records=records)
    geom, ids = scene.chords()
    pts = probe_points(geom, d, 1500, seed=17)
    for orzan in (1, 0):
        got, stops = pick(api, scene, pts, orzan=orzan, with_stops=True)
        assert_same_picks(got, brute(d, geom, ids, pts, orzan=orzan), f"{name} orzan {orzan}")
        # the side rule at distance 0 (D = 0): right without the Orzan orientation, left with it
        zero = got["distance"] == 0
        assert zero.any()
        assert ((got["flags"][zero] & api.PICK_RIGHT) != 0).all() == (orzan == 0)
        assert ((got["flags"][zero] & api.PICK_RIGHT) == 0).all() == (orzan == 1)
        np.testing.assert_allclose(stops, stops64(d, got), rtol=1e-6, atol=1e-6, equal_nan=True, err_msg=f"{name} orzan {orzan}")
    if d["curve_connect"].max() >= 0:
        assert (got["flags"] & api.PICK_PORTAL).any()


def edited(api, d, seed):
    """Every stop value replaced, counts and parameters kept."""
    rng = np.random.default_rng(seed)
    e = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in d.items()}
    for fam in FAMILIES:
        n = e["n_" + fam]
        e[fam][:n] = rng.random(e[fam][:n].shape).astype(F) * (4 if fam == "blur" else 1)
    return e


def test_pick_is_ordered_like_a_launch_across_streams(api):
    import torch

    host, d = host_scene(api, "DiffusionCurvePack/lady_bug.xml")
    d_new = edited(api, d, 5)
    a_old, a_new = api.arrays_from_numpy(d), api.arrays_from_numpy(d_new)
    fresh_old, fresh_new = build(api, a_old), build(api, a_new)
    geom, _ = fresh_old.chords()
    pts = probe_points(geom, d, 1024, seed=2)
    want_old = pick(api, fresh_old, pts, with_stops=True)
    want_new = pick(api, fresh_new, pts, with_stops=True)
    assert not np.array_equal(want_old[1], want_new[1])

    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    scene = build(api, a_old)
    torch.cuda.synchronize()
    # before the update, on another stream than the update's: the old stops; after it, without a host wait: the new ones
    bufs = [buffers(pts, True) for _ in range(3)]
    before = pick(api, scene, pts, on=s2.cuda_stream, bufs=bufs[0])
    scene.update_stops(a_new, s1.cuda_stream)
    after = pick(api, scene, pts, on=s2.cuda_stream, bufs=bufs[1])
    back = pick(api, scene, pts, on=s1.cuda_stream, bufs=bufs[2])
    for res, want in ((before, want_old), (after, want_new), (back, want_new)):
        got, stops = fetch(api, res, len(pts))
        assert_same_picks(got, want[0])
        assert np.array_equal(bits(stops), bits(want[1]))

    # the handle's renders after picks equal the renders of a fresh handle
    p = api.default_frame_params(96, 64, 32, zoom_factor=d["image_height"] / 64)
    frames = []
    bufs = buffers(pts, False)
    for sc in (scene, fresh_new):
        image = torch.empty((64, 96, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((64, 96), dtype=torch.float32, device="cuda")
        pick(api, sc, pts, on=s2.cuda_stream, bufs=bufs)
        sc.render(p, image.data_ptr(), sigma.data_ptr(), s1.cuda_stream)
        torch.cuda.synchronize()
        frames.append((image.cpu().numpy(), sigma.cpu().numpy()))
    assert np.array_equal(bits(frames[0][0]), bits(frames[1][0])) and np.array_equal(bits(frames[0][1]), bits(frames[1][1]))


def test_pick_argument_errors_on_a_real_handle(api):
    host, _ = host_scene(api, "arch.xml")
    scene = build(api, host.arrays)
    p = api.default_frame_params(16, 16, 8, row_begin=4, row_end=4)
    with pytest.raises(api.RdcError, match="band"):
        scene.pick_frame(p, 16, 0, INF, stream())
    with pytest.raises(api.RdcError, match="max_distance"):
        scene.pick(16, 1, 16, 0, 0.0, 1, stream())
    scene.pick(0, 0, 16, 0, INF, 1, stream())  # n == 0: nothing enqueued, nothing read
    assert api.lib.rdc_scene_pick(scene.handle, None, 1, INF, 1, C.c_void_p(16), None, None) == -1
