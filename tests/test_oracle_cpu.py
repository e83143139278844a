"""Pins the CPU oracle.

 * oracle/_ref (the reference's own DeviceCode.cu compiled for the host) must reproduce the committed
   golden vectors it generated, and the restated port must equal them BIT FOR BIT — hits, image, blur map.
 * analytic scenes: a pixel far on one side of a near-straight curve converges to that side's colour.
 * blur restatement: sigma 0 is the identity, constant sigma keeps a constant image, weights follow
   exp(-k^2/sigma^2) (helperKernels.cu:79).
"""
import os

import numpy as np
import pytest

from helpers import DIFFERENT_VIEW, bits, reference_checks, seeded_blur_input, sha_bits
from oracle import pyoracle as po

CASES = ["arch", "portal", "lady_bug", "weight_demo", "drape"]


def load_case(golden_dir, xml_dir, name):
    z = np.load(os.path.join(golden_dir, f"render_{name}.npz"))
    w, h, n, zoom = z["meta"]
    scene = po.ingest_xml(os.path.join(xml_dir, str(z["scene_file"])), True)
    params = po.make_params(int(w), int(h), float(n), zoom_factor=float(zoom))
    return z, scene, params


@pytest.mark.parametrize("name", CASES)
def test_port_equals_reference_golden_bit_for_bit(name, golden_dir, xml_dir, port_oracle):
    z, scene, params = load_case(golden_dir, xml_dir, name)
    image, blur, hits = port_oracle.render(scene, params, want_hits=True)
    assert np.array_equal(hits, z["hits"])
    assert np.array_equal(bits(image), bits(z["image"]))
    assert np.array_equal(bits(blur), bits(z["blur_map"]))


@pytest.mark.parametrize("name", CASES[:3])
def test_reference_build_reproduces_its_golden(name, golden_dir, xml_dir, ref_oracle):
    z, scene, params = load_case(golden_dir, xml_dir, name)
    image, blur, hits = ref_oracle.render(scene, params, want_hits=True)
    assert np.array_equal(hits, z["hits"])
    assert np.array_equal(bits(image), bits(z["image"]))


def test_port_equals_reference_on_a_different_view(xml_dir, port_oracle):
    """Against the reference's render of the view stored as sha256 of its bits (tests/golden/make_golden.py), and live
    where oracle/_ref is built."""
    name, (w, h, n), kw = DIFFERENT_VIEW
    scene = po.ingest_xml(os.path.join(xml_dir, name), True)
    params = po.make_params(w, h, n, **kw)
    a = port_oracle.render(scene, params, want_hits=True)
    want = reference_checks()["different_view"]
    assert sha_bits(a[2]) == want["hits"]
    assert sha_bits(a[0]) == want["image"] and sha_bits(a[1]) == want["blur_map"]
    if po.Oracle.reference_available():
        b = po.Oracle("reference").render(scene, params, want_hits=True)
        assert np.array_equal(a[2], b[2])
        assert np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(bits(a[1]), bits(b[1]))


def test_reference_build_rejects_other_switches(xml_dir, ref_oracle):
    scene = po.ingest_xml(os.path.join(xml_dir, "arch.xml"), True)
    with pytest.raises(RuntimeError):
        ref_oracle.render(scene, po.make_params(8, 8, 8, use_aa=0))


def test_band_rendering_is_partition_invariant(xml_dir, port_oracle):
    scene = po.ingest_xml(os.path.join(xml_dir, "arch.xml"), True)
    full = port_oracle.render(scene, po.make_params(24, 20, 16, zoom_factor=20.0), want_hits=True)
    top = port_oracle.render(scene, po.make_params(24, 20, 16, zoom_factor=20.0, row_begin=0, row_end=7), want_hits=True)
    rest = port_oracle.render(scene, po.make_params(24, 20, 16, zoom_factor=20.0, row_begin=7, row_end=20), want_hits=True)
    for k in range(3):
        assert np.array_equal(bits(np.concatenate([top[k], rest[k]])), bits(full[k]))


def test_line_scene_converges_to_side_colours(xml_dir, port_oracle):
    """test.xml is one near-straight curve: every ray that hits it from one side sees that side's stops."""
    scene = po.ingest_xml(os.path.join(xml_dir, "test.xml"), False)
    params = po.make_params(512, 512, 64, use_diffusion_curve_save=0)
    geom, _ = port_oracle.chords(scene)
    y_mid = float(np.mean(geom[:, [1, 3]]))
    row_above = int(np.clip(256 + y_mid - 60, 0, 511))
    row_below = int(np.clip(256 + y_mid + 60, 0, 511))
    above = port_oracle.render(scene, po.make_params(512, 512, 64, use_diffusion_curve_save=0, row_begin=row_above,
                                                     row_end=row_above + 1))[0][0, 200:312, :3]
    below = port_oracle.render(scene, po.make_params(512, 512, 64, use_diffusion_curve_save=0, row_begin=row_below,
                                                     row_end=row_below + 1))[0][0, 200:312, :3]
    left = scene["color_left"][: scene["n_color_left"]]
    right = scene["color_right"][: scene["n_color_right"]]
    lo = np.minimum(left.min(0), right.min(0)) - 1e-6
    hi = np.maximum(left.max(0), right.max(0)) + 1e-6
    for img in (above, below):
        m = ~np.isnan(img[:, 0])
        assert m.any() and np.all(img[m] >= lo) and np.all(img[m] <= hi)
    # the two sides differ wherever the stop lists do
    if not np.allclose(left.mean(0), right.mean(0)):
        assert not np.allclose(np.nanmean(above, 0), np.nanmean(below, 0), atol=1e-3)
    del params


def test_all_miss_pixels_are_nan(xml_dir, port_oracle):
    scene = po.ingest_xml(os.path.join(xml_dir, "arch.xml"), True)
    # far away, looking at nothing: offset the view by 10^6 pixels and use 2 rays
    image, blur, hits = port_oracle.render(scene, po.make_params(4, 4, 2, offset_x=1e6, offset_y=1e6, use_aa=0), want_hits=True)
    m = np.all(hits == 0xFFFFFFFF, axis=-1)
    assert m.any()
    assert np.all(np.isnan(image[m][:, :3])) and np.all(np.isnan(blur[m]))


def test_blur_restatement_properties(port_oracle):
    rng = np.random.default_rng(0)
    img = rng.random((12, 17, 4), dtype=np.float32)
    assert np.array_equal(port_oracle.blur(img, np.zeros((12, 17), np.float32)), img)
    const = np.full((9, 9, 4), 0.25, np.float32)
    out = port_oracle.blur(const, np.full((9, 9), 2.0, np.float32))
    np.testing.assert_allclose(out, 0.25, rtol=1e-6)
    # impulse response along a row: weights exp(-k^2/sigma^2), support ceil(3 sigma)
    imp = np.zeros((1, 31, 4), np.float32)
    imp[0, 15] = 1.0
    sigma = 1.5
    out = port_oracle.blur(imp, np.full((1, 31), sigma, np.float32))[0, :, 0]
    k = np.arange(-5, 6)
    wts = np.exp(-(k * k) / (sigma + 1e-6) ** 2)
    expect = np.zeros(31)
    expect[10:21] = wts / wts.sum()
    np.testing.assert_allclose(out, expect, atol=1e-6)
    assert out[9] == 0 and out[21] == 0


GRID_VIEWS = [("arch.xml", 64, 48, 32, 512 / 48, 0.0, 0.0, 2), ("PortalDemo.xml", 64, 48, 24, 512 / 48, 0.0, 0.0, 31),
              ("DiffusionCurvePack/dolphin.xml", 48, 36, 16, 0.5, 60.0, -40.0, 2),
              ("DiffusionCurvePack/dolphin.xml", 40, 30, 8, 633 / 30, 0.0, 0.0, 2),
              ("DiffusionCurvePack/roses_spirales.xml", 40, 30, 16, 0.75, 0.0, 0.0, 2),
              ("DiffusionCurvePack/lady_bug.xml", 40, 30, 16, 4.0, -30.0, 20.0, 2)]


@pytest.mark.parametrize("name,w,h,n,zoom,off_x,off_y,depth", GRID_VIEWS, ids=[f"{v[0].split('/')[-1]}@{v[4]:.2f}" for v in GRID_VIEWS])
def test_grid_search_equals_brute_force(name, w, h, n, zoom, off_x, off_y, depth, xml_dir, port_oracle):
    """The uniform grid (oracle_common.h) only narrows which chords a ray is tested against: same closest hit,
    same image, bit for bit, as testing every chord — which is what lets the full-size parity tests use it."""
    scene = po.ingest_xml(os.path.join(xml_dir, name), True)
    p = po.make_params(w, h, n, zoom_factor=zoom, offset_x=off_x, offset_y=off_y, max_trace_depth=depth)
    a = port_oracle.render(scene, p, want_hits=True, search="brute")
    b = port_oracle.render(scene, p, want_hits=True, search="grid")
    assert np.array_equal(a[2], b[2])
    assert np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(bits(a[1]), bits(b[1]))
    assert (a[2] != 0xFFFFFFFF).any()


def test_grid_search_equals_brute_force_reference_build(xml_dir, ref_oracle):
    scene = po.ingest_xml(os.path.join(xml_dir, "DiffusionCurvePack/zephyr.xml"), True)
    p = po.make_params(40, 30, 16, zoom_factor=2.0, offset_x=10.0, offset_y=5.0)
    a = ref_oracle.render(scene, p, want_hits=True, search="brute")
    b = ref_oracle.render(scene, p, want_hits=True, search="grid")
    assert np.array_equal(a[2], b[2]) and np.array_equal(bits(a[0]), bits(b[0]))


def test_port_blur_equals_the_reference_own_kernels():
    """a12 pinned by the reference's code: gaussHorizontal / gaussVertical (helperKernels.cu:48-134) cut out of the file and
    compiled for the host (oracle/ref_extract.sh); the restated blur equals them bit for bit, sigma 0 and NaN included.
    Their output is stored as sha256 of its bits (tests/golden/make_golden.py); live where oracle/_ref is built."""
    image, sigma = seeded_blur_input()  # its NaN pixel is an all-miss pixel (DeviceCode.cu:176-181): spreads like in the reference
    want = reference_checks()["blur_seeded"]
    assert [sha_bits(image), sha_bits(sigma)] == [want["input_image"], want["input_sigma"]], "the seeded input changed"
    got = po.Oracle("port").blur(image, sigma, threads=2)
    assert sha_bits(got) == want["blurred"]
    got_big = po.Oracle("port").blur(image, np.full_like(sigma, 16.0))
    assert sha_bits(got_big) == want["blurred_sigma16"]
    if po.ref_extracts_available():
        assert np.array_equal(bits(got), bits(po.ref_blur(image, sigma, threads=3)))
        assert np.array_equal(bits(got_big), bits(po.ref_blur(image, np.full_like(sigma, 16.0))))
