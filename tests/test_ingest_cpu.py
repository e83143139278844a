"""Host logic: XML loader + ingest (no GPU). Checks the product's C++ ingest against
   (1) the reference's rapidxml element tree (golden hashes, and live when oracle/_ref exists),
   (2) the oracle's independent Python restatement of optixHello.cpp:212-515,
   (3) the worked example of SURVEY.md Appendix B.4."""
import hashlib
import json
import os

import numpy as np
import pytest

from helpers import all_scene_files, assert_scene_equal, ingest_digest, reference_checks, scene_ids, sha_bits, XML_DIR
from oracle import pyoracle as po
from raytracingdiffusioncurves_b200 import api


@pytest.mark.parametrize("path", all_scene_files(), ids=scene_ids())
def test_element_tree_matches_rapidxml_golden(path, golden_dir):
    with open(os.path.join(golden_dir, "xml_dump_sha256.json")) as fh:
        golden = json.load(fh)
    got = hashlib.sha256(api.xml_dump(path).encode()).hexdigest()
    assert got == golden[os.path.relpath(path, XML_DIR)]


@pytest.mark.parametrize("path", all_scene_files()[:6], ids=scene_ids()[:6])
def test_element_tree_matches_rapidxml_live(path):
    if not os.path.exists(po.REF_XML_DUMP):
        pytest.skip("oracle/_ref/ref_xml_dump not built")
    assert api.xml_dump(path) == po.ref_xml_dump(path)


@pytest.mark.parametrize("orzan", [True, False], ids=["orzan", "native"])
@pytest.mark.parametrize("path", all_scene_files(), ids=scene_ids())
def test_ingest_matches_oracle(path, orzan):
    got = api.HostScene.from_xml_file(path, api.default_ingest_options(use_diffusion_curve_save=int(orzan))).to_numpy()
    want = po.ingest_xml(path, orzan)
    assert_scene_equal(got, want)


def test_ingest_knobs_reach_the_arrays(xml_dir):
    path = os.path.join(xml_dir, "line.xml")  # end-capped, no weight_degree_set
    opts = api.default_ingest_options(endcap_size=12.0, default_weight_degree=0.75)
    got = api.HostScene.from_xml_file(path, opts).to_numpy()
    want = po.ingest_xml(path, True, default_weight_degree=0.75, endcap_size=12.0)
    assert_scene_equal(got, want)
    base = po.ingest_xml(path, True)
    assert not np.array_equal(base["vertices"], want["vertices"])
    assert np.all(want["weight_degree"][: want["n_weight_degree"]] == 0.75)


def test_arch_known_answers(xml_dir):
    """SURVEY.md Appendix B.4."""
    s = api.HostScene.from_xml_file(os.path.join(xml_dir, "arch.xml")).to_numpy()
    assert (s["image_width"], s["image_height"]) == (512, 512)
    assert s["segment_indices"].tolist() == [0, 4, 8]
    assert s["curve_map"].tolist() == [0, 0, 0]
    assert s["curve_index"].tolist() == [0, 1, 2]
    assert s["curve_map_inverse"].tolist() == [0]
    assert s["curve_connect"].tolist() == [-1]
    assert s["vertices"].shape == (12, 3)
    np.testing.assert_array_equal(s["vertices"][4:8, :2], [[384, 1408], [-384, -128], [384, -128], [-384, 1408]])
    b = s["vertices"][4:8, :2]
    np.testing.assert_allclose((b[0] + 4 * b[1] + b[2]) / 6, [-128, 128])
    np.testing.assert_allclose(s["color_left_u"][:9], [0, 1, 1, 1.3, 1.7, 2, 2, 2, 3], rtol=1e-6)
    assert s["color_left_index"].tolist() == [[0, 9]] and s["color_right_index"].tolist() == [[0, 9]]
    np.testing.assert_array_equal(s["blur_u"][:4], [0, 1, 3, 3])
    np.testing.assert_array_equal(s["blur"][:4], 0)
    np.testing.assert_allclose(s["weight_u"][:7], [0, 1, 1.3, 1.5, 1.7, 2, 3], rtol=1e-6)
    np.testing.assert_array_equal(s["weight"][:7], 1)
    np.testing.assert_array_equal(s["weight_degree_u"][:4], [0, 1, 2, 3])
    np.testing.assert_array_equal(s["weight_degree"][:4], 0.5)
    np.testing.assert_array_equal(s["color_left"][2], [1, 0, 0])  # R=0 G=0 B=255 stored as (B,G,R)
    # the stop walk over-reads: every u array ends in two +INF sentinels
    for fam in ("color_left", "color_right", "blur", "weight", "weight_degree"):
        assert np.all(np.isinf(s[fam + "_u"][-2:]))
    # start cap hugs the first control point
    cap = s["vertices"][0:4, :2]
    assert np.all(np.abs((cap[0] + 4 * cap[1] + cap[2]) / 6 - [-128, 128]) < 1e-3)


def test_portal_demo_structure(xml_dir):
    s = api.HostScene.from_xml_file(os.path.join(xml_dir, "PortalDemo.xml")).to_numpy()
    assert s["curve_connect"].tolist() == [-1, -1, 3, 2, 4]
    assert s["curve_map_inverse"].tolist() == [0, 1, 2, 3, 4]
    assert s["weight"][s["weight_index"][1, 0]] == 0  # absorbing wall


def test_error_behaviour(tmp_path):
    with pytest.raises(api.RdcError) as e:
        api.HostScene.from_xml_file(str(tmp_path / "missing.xml"))
    assert e.value.code == -3  # RDC_E_IO
    bad = tmp_path / "bad.xml"
    bad.write_text("<curve_set image_width='4' image_height='4'><curve></curve_set>")
    with pytest.raises(api.RdcError) as e:
        api.HostScene.from_xml_file(str(bad))
    assert e.value.code == -2  # RDC_E_PARSE
    three = tmp_path / "three.xml"
    three.write_text(
        "<curve_set image_width='4' image_height='4'><curve><control_points_set>"
        "<control_point x='0' y='0'/><control_point x='1' y='0'/><control_point x='2' y='0'/>"
        "</control_points_set></curve></curve_set>")
    with pytest.raises(api.RdcError) as e:
        api.HostScene.from_xml_file(str(three))
    assert e.value.code == -2 and "3k+1" in str(e.value)
    empty = tmp_path / "empty.xml"
    empty.write_text("<!DOCTYPE CurveSetXML><curve_set image_width='4' image_height='4'></curve_set>")
    with pytest.raises(api.RdcError):
        api.HostScene.from_xml_file(str(empty))


def test_synthetic_scene_is_deterministic_and_loads():
    a = api.synth_xml(200, 1024, 1024)
    b = api.synth_xml(200, 1024, 1024)
    assert a == b and a != api.synth_xml(200, 1024, 1024, seed=1)
    s = api.HostScene.from_xml_text(a).to_numpy()
    assert len(s["curve_connect"]) == 200 and len(s["segment_indices"]) == 200
    assert s["n_weight"] == 400 and np.all(s["weight"][:400] == 1)


def test_image_to_rgba8_follows_the_screenshot_convention():
    img = np.zeros((2, 3, 4), np.float32)
    img[0, 0] = [0.5, 2.0, np.nan, 1.0]
    img[1, 2] = [1.0, 0.25, -1.0, 1.0]
    out = api.image_to_rgba8(img, flip=False)
    assert out[0, 0].tolist() == [127, 255, 0, 255] and out[1, 2].tolist() == [255, 63, 0, 255]
    assert np.array_equal(api.image_to_rgba8(img, flip=True), out[::-1])


def test_scene_cache_round_trip(xml_dir, tmp_path):
    for name in ("arch.xml", "PortalDemo.xml", "DiffusionCurvePack/dolphin.xml"):
        a = api.HostScene.from_xml_file(os.path.join(xml_dir, name))
        path = str(tmp_path / "scene.rdc")
        a.save(path)
        b = api.HostScene.from_cache(path)
        assert_scene_equal(a.to_numpy(), b.to_numpy())
    bad = tmp_path / "bad.rdc"
    bad.write_bytes(b"not a cache at all")
    with pytest.raises(api.RdcError) as e:
        api.HostScene.from_cache(str(bad))
    assert e.value.code == -2
    with pytest.raises(api.RdcError) as e:
        api.HostScene.from_cache(str(tmp_path / "missing.rdc"))
    assert e.value.code == -3


def test_xml_tree_edge_cases(tmp_path):
    """The in-place parser: entities decoded where they stand, both quote styles, empty elements, everything that is
    not an element skipped (the nodes rapidxml's parse<0> does not create), errors with a line number."""
    doc = tmp_path / "edge.xml"
    doc.write_bytes(
        b"\xef\xbb\xbf<?xml version='1.0'?>\n<!DOCTYPE a [ <!ENTITY x 'y'> ]>\n<!-- c <b/> -->\n"
        b"<a k=\"1 &amp; 2\" q='say &quot;hi&quot; &#65;&#x42;&#xe9; &unknown; &lt;&gt;&apos;'>text <![CDATA[ <z/> ]]>\n"
        b" <b/><b x = \"2\" />\n <c>\n  <d name=\"it's\"></d>\n </c>\n</a>\n<trailing/>\n")
    assert api.xml_dump(str(doc)) == (
        "a k=1 & 2 q=say \"hi\" ABé &unknown; <>'\n"
        " b\n"
        " b x=2\n"
        " c\n"
        "  d name=it's\n")
    for text, what in (("<a><b></a>", "closes"), ("<a", "unterminated"), ("<a x=1/>", "quoted"), ("<a x='1/>", "unterminated"),
                       ("", "no root"), ("<a>\n\n<b>\n</b>", "line 4"), ("<!-- never closed <a/>", "unterminated"),
                       ("<a>" * 600 + "</a>" * 600, "nested")):
        bad = tmp_path / "bad.xml"
        bad.write_text(text)
        with pytest.raises(api.RdcError) as e:
            api.xml_dump(str(bad))
        assert e.value.code == -2 and what in str(e.value), (text[:20], str(e.value))


def test_numbers_are_read_like_atof(tmp_path):
    """Attribute values go through a fast exact parser with atof as the fallback: same floats either way."""
    def scene(xs):
        pts = "".join(f"<control_point x='{x}' y='{i}'/>" for i, x in enumerate(xs))
        return (f"<curve_set image_width='0' image_height='0'><curve><control_points_set>{pts}</control_points_set>"
                "<left_colors_set><left_color R='1' G='2' B='3' globalID='0'/><left_color R='1' G='2' B='3' globalID='10'/></left_colors_set>"
                "<right_colors_set><right_color R='1' G='2' B='3' globalID='0'/><right_color R='1' G='2' B='3' globalID='10'/></right_colors_set>"
                "<blur_points_set><best_scale value=' 1.5' globalID='0'/><best_scale value='+2.25x' globalID='1e1'/></blur_points_set>"
                "</curve></curve_set>")
    xs = ["0.1", " 7.25", "+3", "1e-3junk"]
    s = api.HostScene.from_xml_text(scene(xs).encode(), api.default_ingest_options(use_diffusion_curve_save=0)).to_numpy()
    want = np.array([np.float32(float(v)) for v in ("0.1", "7.25", "3", "1e-3")], np.float32)
    # Bezier (b0..b3) -> B-spline control points; b0 = (V0 + 4 V1 + V2)/6 recovers the first value
    v = s["vertices"][:4, 0].astype(np.float64)
    bezier = [(v[0] + 4 * v[1] + v[2]) / 6, (2 * v[1] + v[2]) / 3, (v[1] + 2 * v[2]) / 3, (v[1] + 4 * v[2] + v[3]) / 6]
    np.testing.assert_allclose(bezier, want, atol=2e-5)
    assert s["blur"][:2].tolist() == [1.5, 2.25] and s["blur_u"][:2].tolist() == [0.0, 1.0]


@pytest.mark.parametrize("path", all_scene_files(), ids=scene_ids())
def test_product_ingest_equals_the_reference_own_loop(path):
    """a2 pinned by the reference's code: optixHello.cpp:108-117,170-515 and its helpers :1302-1386, cut out of the file where
    it lies and compiled for the host (oracle/ref_extract.sh -> oracle/_ref/libref_ingest.so), run on every bundled XML.
    The product's arrays equal the reference's bit for bit (the product appends +INF sentinels after them). The reference's
    arrays are stored as sha256 of their bits (tests/golden/make_golden.py); where oracle/_ref is built they are also
    computed live and must match what is stored."""
    want = reference_checks()["ingest"][os.path.relpath(path, XML_DIR)]
    mine = api.HostScene.from_xml_file(path).to_numpy()
    assert set(want) == set(mine)
    for k, v in want.items():
        if isinstance(v, dict):
            n = v["shape"][0]
            m = np.ascontiguousarray(mine[k][:n])
            assert [str(m.dtype), list(m.shape)] == [v["dtype"], v["shape"]], k
            assert sha_bits(m) == v["sha256"], k
            if k.endswith("_u"):  # what follows the reference's entries is the two sentinels, nothing else
                assert np.all(np.isinf(mine[k][n:])) and len(mine[k]) >= n + 2
        else:
            assert mine[k] == v, k
    if po.ref_extracts_available():
        assert ingest_digest(po.ref_ingest(path)) == want
