"""The slab test's margin against the ray origins' rounding, restated in numpy float32 (no GPU).

render.cu culls a run when the fused slab test of its padded box (slab_ray / slab_enter) says the ray cannot meet the box
before the best hit so far. That is exact only if the box of the chord the brute force hits always passes. The rounding
of the fused test, of rcp.approx and of the chord test's p - o grows with the ORIGIN's coordinates, so a view far from a
small scene can push the hit outside the padded box as the slab test sees it. Here rays from 1e3 to 1e6 units away are
aimed at the end points of straight chords (each chord its own run, so the end points are box corners), the port oracle
finds their first hits by brute force, and the restated slab test is asked whether the hit chord's box passes:

* with the padding alone (curve_width + 4e-6 x extent) it rejects some hit boxes at 1e6, which shows the sweep can see
  the problem;
* with the boxes widened by the launch's w = max(0, 16 x 2^-23 x M - pad) (render.cu slab_widening) it rejects none,
  for every curve_width including 0, with rcp.approx bracketed by the neighbours of the IEEE reciprocal.
"""
import os

import numpy as np
import pytest

from helpers import dust_curves, scene_xml
from oracle import pyoracle as po

f32 = np.float32
SLACK = f32(1.000002)  # RDC_CULL_SLACK
DISTANCES = [1e3, 1e4, 1e5, 1e6]
MISS = 0xFFFFFFFF


def fma32(a, b, c):
    """fmaf through float64: the product of two float32 values is exact there, one rounding to float32 after the add."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(f32)


def slab_rcp_candidates(d):
    """rcp.approx.ftz.f32 of |d| clamped away from 0: within 1 ulp of the IEEE reciprocal, so either neighbour of it."""
    a = np.where(np.abs(d) < f32(1e-30), np.copysign(f32(1e-30), d), d).astype(f32)
    r = (f32(1) / a).astype(f32)
    return [np.nextafter(r, f32(-np.inf)), r, np.nextafter(r, f32(np.inf))]


def slab_passes(o, d, box, t_hit, w):
    """slab_ray + slab_enter of render.cu on the box widened by w (render.cu k_widen_boxes) and the cull condition
    tn <= te && tn <= t * RDC_CULL_SLACK, for every pair of reciprocal candidates; True where all of them let the box
    through."""
    ox, oy, dx, dy = o[:, 0], o[:, 1], d[:, 0], d[:, 1]
    x0, y0 = (box[:, 0] - w).astype(f32), (box[:, 1] - w).astype(f32)
    x1, y1 = (box[:, 2] + w).astype(f32), (box[:, 3] + w).astype(f32)
    ok = np.ones(len(o), bool)
    for idx in slab_rcp_candidates(dx):
        nox = -(ox * idx).astype(f32)
        tx1, tx2 = fma32(x0, idx, nox), fma32(x1, idx, nox)
        for idy in slab_rcp_candidates(dy):
            noy = -(oy * idy).astype(f32)
            ty1, ty2 = fma32(y0, idy, noy), fma32(y1, idy, noy)
            te = np.minimum(np.maximum(tx1, tx2), np.maximum(ty1, ty2))
            tn = np.maximum(np.maximum(np.minimum(tx1, tx2), np.minimum(ty1, ty2)), f32(0))
            ok &= (tn <= te) & (tn <= (t_hit * SLACK).astype(f32))
    return ok


def widening(o, pad):
    """render.cu slab_widening with M = the ray's own largest origin coordinate (the smallest M a launch can have)."""
    m = np.max(np.abs(o.astype(np.float64)), axis=1)
    w = 16.0 * 2.0 ** -23 * m * (1.0 + 1e-6) - float(pad)
    return np.where(w > 0, w, 0).astype(f32)


@pytest.fixture(scope="module")
def sweep(port_oracle, tmp_path_factory):
    """Rays aimed at (and a hair beside) every chord end point of 1500 straight segments from each distance, their
    brute-force first hits, and the chords."""
    path = os.path.join(str(tmp_path_factory.mktemp("margins")), "dust.xml")
    with open(path, "w") as fh:
        fh.write(scene_xml(dust_curves(1500, seed=11)))
    scene = po.ingest_xml(path, True)
    geom, _ = port_oracle.chords(scene)
    assert len(geom) == 1500  # one chord, hence one run, per segment
    rng = np.random.default_rng(3)
    ends = np.concatenate([geom[:, 0:2], geom[:, 2:4]]).astype(np.float64)
    out = {}
    for R in DISTANCES:
        rays = []
        for _ in range(8):
            ang = rng.uniform(0, 2 * np.pi, len(ends))
            u = np.stack([np.cos(ang), np.sin(ang)], 1)
            aim = ends + rng.normal(0, 1e-3, ends.shape) * rng.integers(0, 2, (len(ends), 1))
            o = (aim + R * u).astype(f32)
            d = -u
            d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32)
            rays.append(np.concatenate([o, d], 1))
        rays = np.concatenate(rays).astype(f32)
        ids, t, _ = port_oracle.trace_rays(scene, rays, search="grid")
        out[R] = (rays, ids, t)
    extent = f32(np.max(np.abs(scene["vertices"][:, :2])))
    return geom, extent, out


def hit_boxes(geom, ids, pad):
    g = geom[ids]
    lo = np.minimum(g[:, 0:2], g[:, 2:4])
    hi = np.maximum(g[:, 0:2], g[:, 2:4])
    return np.concatenate([(lo - pad).astype(f32), (hi + pad).astype(f32)], 1)  # (xmin, ymin, xmax, ymax)


def rejected(sweep, curve_width, new_rule):
    """Hit boxes the restated slab test rejects, per distance."""
    geom, extent, rays_by_r = sweep
    pad = f32(f32(curve_width) + f32(f32(4e-6) * extent))
    counts = {}
    for R, (rays, ids, t) in rays_by_r.items():
        hit = ids != MISS
        assert hit.sum() > 0.5 * len(ids), f"R={R}: only {hit.sum()} of {len(ids)} rays hit"
        o, d = rays[hit, 0:2], rays[hit, 2:4]
        w = widening(o, pad) if new_rule else np.zeros(len(o), f32)
        counts[R] = int((~slab_passes(o, d, hit_boxes(geom, ids[hit], pad), t[hit], w)).sum())
    return counts


def test_padding_alone_rejects_hits_far_away(sweep):
    counts = rejected(sweep, 1e-3, new_rule=False)
    print(f"hit boxes rejected by the padding alone, by distance: {counts}")
    assert counts[1e3] == 0
    assert counts[1e6] > 0, "the sweep cannot see the problem it is meant to catch"


@pytest.mark.parametrize("curve_width", [1e-3, 0.0, 0.05])
def test_widened_boxes_reject_no_hit(sweep, curve_width):
    counts = rejected(sweep, curve_width, new_rule=True)
    assert all(c == 0 for c in counts.values()), f"hit boxes rejected with the widening, by distance: {counts}"


def test_no_widening_near_the_scene():
    """Views near the scene keep the plain padded test (w = 0): the headline frame (arch.xml, extent ~135, 1920 x 1080 at
    zoom 512/1080) and any origin within twice the extent for curve_width 0."""
    extent = 135.0
    for cw in (1e-3, 0.0):
        pad = f32(f32(cw) + f32(f32(4e-6) * f32(extent)))
        headline_m = (0.5 * 1920 + 2) * 512 / 1080
        assert widening(np.array([[headline_m, 0.0]], f32), pad)[0] == 0 or cw == 0.0
        assert widening(np.array([[2 * extent, 0.0]], f32), pad)[0] == 0
