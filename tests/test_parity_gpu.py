"""Parity tests proper: the CUDA path, through the C ABI, against the CPU oracle on the same seeded rays.

Bar (BASELINE.json north_star): first-hit chord index of every primary ray bit-exact, per-pixel RGB
within 1e-4 absolute (fp32), PSNR reported. Chord tables (integer/bit work) are bit-exact.
"""
import os

import numpy as np
import pytest

from helpers import GpuRenderer, bits, compare_images, copy_params
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

RGB_TOL = 1e-4  # absolute, fp32 — the tolerance north_star states


@pytest.fixture(scope="module")
def api():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from raytracingdiffusioncurves_b200 import api as _api

    return _api


def product_params(api, p):
    return copy_params(p, api.FrameParams)


SCENES = ["arch.xml", "arch2.xml", "line.xml", "test.xml", "test2.xml", "test3.xml", "test4.xml", "test5.xml", "circles.xml",
          "endcap.xml", "weight_demo.xml", "PortalDemo.xml", "DiffusionCurvePack/behindthecurtain.xml",
          "DiffusionCurvePack/dolphin.xml", "DiffusionCurvePack/drape.xml", "DiffusionCurvePack/face.xml",
          "DiffusionCurvePack/fille.xml", "DiffusionCurvePack/lady_bug.xml", "DiffusionCurvePack/roses_spirales.xml",
          "DiffusionCurvePack/zephyr.xml"]


@pytest.mark.parametrize("name", SCENES)
def test_chord_tables_bit_exact(name, xml_dir, api, port_oracle):
    path = os.path.join(xml_dir, name)
    r = GpuRenderer(path)
    geom, ids = r.scene.chords()
    ogeom, oids = port_oracle.chords(po.ingest_xml(path, True))
    assert np.array_equal(ids, oids)
    assert np.array_equal(bits(geom), bits(ogeom))
    st = r.scene.stats
    assert st.n_chords == len(ogeom) and st.n_nodes == max(st.n_runs - 1, 1) and st.bvh_depth <= 62
    assert -(-st.n_chords // 8) <= st.n_runs <= st.n_chords


@pytest.mark.parametrize("name", SCENES)
def test_render_parity_small(name, xml_dir, api, port_oracle):
    path = os.path.join(xml_dir, name)
    scene = po.ingest_xml(path, True)
    big = "Pack" in name
    w, h, n = (40, 30, 16) if big else (64, 48, 32)
    zoom = scene["image_height"] / h
    p = po.make_params(w, h, n, zoom_factor=zoom)
    oimg, oblur, ohits = port_oracle.render(scene, p, want_hits=True)
    r = GpuRenderer(path)
    for traversal in (api.TRAVERSAL_LBVH, api.TRAVERSAL_BRUTE_FORCE):
        out = r.render(product_params(api, po.make_params(w, h, n, zoom_factor=zoom, traversal=traversal)), want_hits=True)
        assert np.array_equal(out["hits"], ohits), f"hit indices differ (traversal {traversal})"
        d, psnr = compare_images(out["image"], oimg, RGB_TOL)
        m = ~np.isnan(oblur)
        assert np.array_equal(np.isnan(out["blur_map"]), np.isnan(oblur))
        assert np.max(np.abs(out["blur_map"][m] - oblur[m]), initial=0) <= 1e-4 * max(1.0, float(np.nanmax(oblur, initial=0)))
        print(f"{name}: max|rgb diff| {d:.2e}, psnr {psnr:.1f} dB")


@pytest.mark.parametrize("case", ["arch", "portal", "lady_bug", "weight_demo", "drape"])
def test_render_matches_reference_golden(case, golden_dir, xml_dir, api):
    """Golden vectors produced by the reference's own DeviceCode.cu (tests/golden/make_golden.py)."""
    z = np.load(os.path.join(golden_dir, f"render_{case}.npz"))
    w, h, n, zoom = z["meta"]
    r = GpuRenderer(os.path.join(xml_dir, str(z["scene_file"])))
    out = r.render(api.default_frame_params(int(w), int(h), float(n), zoom_factor=float(zoom)), want_hits=True)
    assert np.array_equal(out["hits"], z["hits"])
    compare_images(out["image"], z["image"], RGB_TOL)


@pytest.mark.parametrize("kw", [dict(use_aa=0), dict(use_diffusion_curve_save=0), dict(frame=7, seed=123),
                                dict(offset_x=31.5, offset_y=-12.25, zoom_factor=3.0), dict(number_of_rays_per_pixel=7.5)],
                         ids=["no_aa", "native", "frame_seed", "pan_zoom", "fractional_rpp"])
def test_switches_and_knobs(kw, xml_dir, api, port_oracle):
    path = os.path.join(xml_dir, "DiffusionCurvePack/lady_bug.xml")
    orzan = kw.get("use_diffusion_curve_save", 1) != 0
    scene = po.ingest_xml(path, orzan)
    base = dict(zoom_factor=10.0)
    base.update(kw)
    n = base.pop("number_of_rays_per_pixel", 24)
    p = po.make_params(48, 40, n, **base)
    oimg, oblur, ohits = port_oracle.render(scene, p, want_hits=True)
    out = GpuRenderer(path, orzan=orzan).render(product_params(api, p), want_hits=True)
    assert np.array_equal(out["hits"], ohits)
    compare_images(out["image"], oimg, RGB_TOL)


@pytest.mark.parametrize("depth", [0, 1, 2, 31])
def test_portals_iterative_retrace(depth, xml_dir, api, port_oracle):
    """config 4: connects attribute; the CUDA loop against the oracle's recursion, up to depth 31."""
    path = os.path.join(xml_dir, "PortalDemo.xml")
    scene = po.ingest_xml(path, True)
    p = po.make_params(96, 54, 32, zoom_factor=512 / 54, max_trace_depth=depth)
    oimg, oblur, ohits = port_oracle.render(scene, p, want_hits=True)
    out = GpuRenderer(path).render(product_params(api, p), want_hits=True)
    assert np.array_equal(out["hits"], ohits)
    compare_images(out["image"], oimg, RGB_TOL)


@pytest.mark.parametrize("name", ["arch.xml", "DiffusionCurvePack/lady_bug.xml"])
def test_units_per_tile_only_moves_the_summation_order(name, xml_dir, api, port_oracle):
    """1, 2, 4 or 8 work units per tile (the library picks one per launch): the same first hits bit for bit, pixels within
    the rounding of a differently ordered sum, each within the parity tolerance of the oracle; pinned, a frame rendered in
    bands equals the one-call frame bit for bit."""
    path = os.path.join(xml_dir, name)
    scene = po.ingest_xml(path, True)
    w, h, n = 64, 48, 128
    zoom = scene["image_height"] / h
    oimg, _, ohits = port_oracle.render(scene, po.make_params(w, h, n, zoom_factor=zoom), want_hits=True, search="grid")
    r = GpuRenderer(path)
    images = []
    for units in (1, 2, 4, 8):
        out = r.render(api.default_frame_params(w, h, n, zoom_factor=zoom, units_per_tile=units), want_hits=True)
        assert np.array_equal(out["hits"], ohits), units
        compare_images(out["image"], oimg, RGB_TOL)
        images.append(out["image"])
        parts = [r.render(api.default_frame_params(w, h, n, zoom_factor=zoom, units_per_tile=units, row_begin=b, row_end=e))["image"]
                 for b, e in ((0, 20), (20, 48))]
        assert np.array_equal(bits(np.concatenate(parts)), bits(out["image"])), units
    for img in images[1:]:
        m = ~np.isnan(images[0])
        assert np.max(np.abs(img[m] - images[0][m])) <= 2e-6
    with pytest.raises(api.RdcError):
        r.render(api.default_frame_params(w, h, n, zoom_factor=zoom, units_per_tile=3))


@pytest.mark.parametrize("name", ["DiffusionCurvePack/lady_bug.xml", "DiffusionCurvePack/dolphin.xml", "PortalDemo.xml", "test2.xml"])
def test_tree_builders_give_the_same_frame(name, xml_dir, api, port_oracle):
    """Morton radix tree (GPU) and binned surface-area-heuristic tree (host): different trees over the same leaves — the same
    first hits and the same pixels bit for bit, on the tree route and on the automatic one, and both equal to the oracle."""
    path = os.path.join(xml_dir, name)
    scene = po.ingest_xml(path, True)
    w, h, n = 72, 52, 16
    zoom = scene["image_height"] / h
    oimg, _, ohits = port_oracle.render(scene, po.make_params(w, h, n, zoom_factor=zoom), want_hits=True, search="grid")
    outs, boxes = {}, {}
    for tree in (api.TREE_MORTON, api.TREE_SAH):
        r = GpuRenderer(path, accel=api.default_accel_options(tree=tree))
        assert r.scene.stats.n_nodes == max(r.scene.stats.n_runs - 1, 1) and 1 <= r.scene.stats.bvh_depth <= 62
        for route in (api.ROUTE_TREE, api.ROUTE_AUTO):
            out = r.render(api.default_frame_params(w, h, n, zoom_factor=zoom, route=route), want_hits=True, want_stats=True)
            assert np.array_equal(out["hits"], ohits), (tree, route)
            plain = r.render(api.default_frame_params(w, h, n, zoom_factor=zoom, route=route), want_hits=True)
            assert np.array_equal(plain["hits"], ohits), (tree, route, "plain build")
            compare_images(out["image"], oimg, RGB_TOL)
            outs[(tree, route)] = out["image"]
            boxes[(tree, route)] = out["stats"][1]
    for route in (api.ROUTE_TREE, api.ROUTE_AUTO):
        assert np.array_equal(bits(outs[(api.TREE_MORTON, route)]), bits(outs[(api.TREE_SAH, route)])), route
    print(f"{name}: boxes tested on the tree route: Morton {boxes[(api.TREE_MORTON, api.ROUTE_TREE)]}, SAH {boxes[(api.TREE_SAH, api.ROUTE_TREE)]}")
    with pytest.raises(api.RdcError):
        GpuRenderer(path, accel=api.default_accel_options(tree=7))


CUT_VIEWS = [("DiffusionCurvePack/lady_bug.xml", 512 / 52, 0.0, 0.0, 16, 2), ("DiffusionCurvePack/lady_bug.xml", 1.0, -30.0, 20.0, 24, 2),
             ("DiffusionCurvePack/face.xml", 0.3, -20.0, 35.0, 40, 2), ("DiffusionCurvePack/dolphin.xml", 633 / 52, 0.0, 0.0, 16, 2),
             ("DiffusionCurvePack/dolphin.xml", 0.5, 60.0, -40.0, 16, 2), ("test4.xml", 512 / 52, 0.0, 0.0, 32, 2),
             ("PortalDemo.xml", 3.0, 10.0, -5.0, 16, 31)]


@pytest.mark.parametrize("name,zoom,off_x,off_y,n,depth", CUT_VIEWS, ids=[f"{v[0].split('/')[-1]}@{v[1]:.2f}" for v in CUT_VIEWS])
def test_cut_table_views(name, zoom, off_x, off_y, n, depth, xml_dir, api, port_oracle):
    """The per-tile table over a 64-entry cut through the tree (mid-size scenes): entries are subtrees or leaves, nearest
    first; every first hit still the oracle's brute-force closest chord, whole frames and frames cut in bands alike."""
    path = os.path.join(xml_dir, name)
    scene = po.ingest_xml(path, True)
    w, h = 72, 52
    kw = dict(zoom_factor=zoom, offset_x=off_x, offset_y=off_y, max_trace_depth=depth)
    oimg, oblur, ohits = port_oracle.render(scene, po.make_params(w, h, n, **kw), want_hits=True, search="grid")
    r = GpuRenderer(path, accel=api.default_accel_options(tree=api.TREE_SAH))
    forced = r.scene.stats.n_runs > 64
    route = api.ROUTE_CUT_TABLE if forced else api.ROUTE_AUTO
    out = r.render(api.default_frame_params(w, h, n, route=route, **kw), want_hits=True)
    assert np.array_equal(out["hits"], ohits)
    compare_images(out["image"], oimg, RGB_TOL)
    counted = r.render(api.default_frame_params(w, h, n, route=route, **kw), want_hits=True, want_stats=True)
    assert np.array_equal(counted["hits"], ohits)
    tree = r.render(api.default_frame_params(w, h, n, route=api.ROUTE_TREE, **kw), want_hits=True, want_stats=True)
    assert np.array_equal(tree["hits"], ohits)
    parts = [r.render(api.default_frame_params(w, h, n, route=route, row_begin=b, row_end=e, **kw))["image"] for b, e in ((0, 20), (20, 52))]
    assert np.array_equal(bits(np.concatenate(parts)), bits(out["image"]))
    print(f"{name} zoom {zoom:.2f}: rays traced {counted['stats'][0]} (tree route {tree['stats'][0]}), boxes {counted['stats'][1]} ({tree['stats'][1]})")


def test_row_bands_concatenate_bit_exactly(xml_dir, api):
    """Partition invariance (SURVEY.md §4.4): 1-GPU image == concatenation of bands, bit for bit."""
    r = GpuRenderer(os.path.join(xml_dir, "DiffusionCurvePack/zephyr.xml"))
    w, h, n = 80, 61, 16
    full = r.render(api.default_frame_params(w, h, n, zoom_factor=512 / h), want_hits=True)
    for world in (2, 3, 8):
        parts = []
        for rank in range(world):
            b, e = api.row_band(h, rank, world)
            parts.append(r.render(api.default_frame_params(w, h, n, zoom_factor=512 / h, row_begin=b, row_end=e), want_hits=True))
        for key in ("image", "blur_map", "hits"):
            assert np.array_equal(bits(np.concatenate([q[key] for q in parts])), bits(full[key])), (world, key)


def test_interleaved_strips_reassemble_bit_exactly(xml_dir, api):
    """The multi-GPU split (8-row strips dealt round-robin) emulated on one GPU: every rank's packed
    strips, put back in order with distributed.StripPlan.source_index, equal the one-call frame."""
    import torch

    from raytracingdiffusioncurves_b200 import distributed as rd

    r = GpuRenderer(os.path.join(xml_dir, "DiffusionCurvePack/zephyr.xml"))
    w, h, n = 72, 83, 8
    full = r.render(api.default_frame_params(w, h, n, zoom_factor=512 / h), want_hits=True)
    for world in (2, 3, 8):
        plan = rd.StripPlan(h, w, world, 0, 0)
        images, sigmas = [], []
        for rank in range(world):
            image = torch.zeros((plan.packed_rows, w, 4), dtype=torch.float32, device="cuda")
            sigma = torch.zeros((plan.packed_rows, w), dtype=torch.float32, device="cuda")
            p = api.default_frame_params(w, h, n, zoom_factor=512 / h, strip_stride=world, strip_offset=rank)
            r.scene.render(p, image.data_ptr(), sigma.data_ptr(), torch.cuda.current_stream().cuda_stream)
            images.append(image)
            sigmas.append(sigma)
        idx = plan.source_index().cuda()
        got = torch.cat(images).index_select(0, idx).cpu().numpy()
        got_sigma = torch.cat(sigmas).index_select(0, idx).cpu().numpy()
        assert np.array_equal(bits(got), bits(full["image"])), world
        assert np.array_equal(bits(got_sigma), bits(full["blur_map"])), world


def test_render_to_frames_places_strips_in_full_frames(xml_dir, api):
    """rdc_render_to_frames (the multi-GPU form): every rank's strips stored straight into two full target frames
    give, together, the one-call frame — bit for bit, in both targets."""
    import torch

    r = GpuRenderer(os.path.join(xml_dir, "DiffusionCurvePack/zephyr.xml"))
    w, h, n = 72, 83, 8
    full = r.render(api.default_frame_params(w, h, n, zoom_factor=512 / h))
    s = torch.cuda.current_stream().cuda_stream
    for world in (2, 3):
        images = [torch.full((h, w, 4), float("nan"), dtype=torch.float32, device="cuda") for _ in range(2)]
        sigmas = [torch.full((h, w), float("nan"), dtype=torch.float32, device="cuda") for _ in range(2)]
        for rank in range(world):
            p = api.default_frame_params(w, h, n, zoom_factor=512 / h, strip_stride=world, strip_offset=rank)
            r.scene.render_to_frames(p, [t.data_ptr() for t in images], [t.data_ptr() for t in sigmas], s)
        torch.cuda.synchronize()
        for t in range(2):
            assert np.array_equal(bits(images[t].cpu().numpy()), bits(full["image"])), (world, t)
            assert np.array_equal(bits(sigmas[t].cpu().numpy()), bits(full["blur_map"])), (world, t)
    with pytest.raises(api.RdcError):
        r.scene.render_to_frames(api.default_frame_params(w, h, n), [0], [0], s)


def test_lbvh_equals_brute_force_at_headline_size(xml_dir, api):
    """Size-independent property at BASELINE's config 2 (arch.xml 1920x1080, 128 rays/pixel):
    the LBVH traversal and the no-tree kernel agree on every one of the 265 M first hits."""
    import torch

    r = GpuRenderer(os.path.join(xml_dir, "arch.xml"))
    w, h, n = 1920, 1080, 128
    sums = []
    for traversal in (api.TRAVERSAL_LBVH, api.TRAVERSAL_BRUTE_FORCE):
        acc = torch.zeros((2,), dtype=torch.int64, device="cuda")
        imgs = []
        for b in range(0, h, 120):  # bands keep the hit buffer at 118 MB
            p = api.default_frame_params(w, h, n, zoom_factor=512 / h, row_begin=b, row_end=b + 120, traversal=traversal)
            hits = torch.empty((120, w, n), dtype=torch.int32, device="cuda")
            image = torch.empty((120, w, 4), dtype=torch.float32, device="cuda")
            sigma = torch.empty((120, w), dtype=torch.float32, device="cuda")
            p.hit_ids = hits.data_ptr()
            r.scene.render(p, image.data_ptr(), sigma.data_ptr(), torch.cuda.current_stream().cuda_stream)
            hv = hits.to(torch.int64) & 0xFFFFFFFF
            pos = torch.arange(hv.numel(), device="cuda", dtype=torch.int64).reshape(hv.shape) + b * w * n
            acc[0] += hv.sum()
            acc[1] += ((hv + 1) * (pos % 1000003)).sum()  # order-sensitive checksum
            imgs.append(image)
        torch.cuda.synchronize()
        sums.append((acc.cpu().tolist(), torch.cat(imgs)))
    assert sums[0][0] == sums[1][0]
    assert torch.equal(sums[0][1].view(torch.int32), sums[1][1].view(torch.int32))


@pytest.mark.parametrize("name", ["DiffusionCurvePack/face.xml", "DiffusionCurvePack/dolphin.xml", "arch.xml"])
def test_blur_parity(name, xml_dir, api, port_oracle):
    path = os.path.join(xml_dir, name)
    scene = po.ingest_xml(path, True)
    w, h, n = 96, 64, 8
    p = po.make_params(w, h, n, zoom_factor=scene["image_height"] / h)
    oimg, oblur, _ = port_oracle.render(scene, p)
    r = GpuRenderer(path)
    out = r.render(product_params(api, p), blur=True)
    # blur the GPU's own render with the oracle's blur: isolates the blur kernels
    want = port_oracle.blur(out["image"], out["blur_map"])[..., :3]  # parity is defined on RGB (.w is never
    got = out["blurred"][..., :3]                                     # written by the reference's raygen)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    m = ~np.isnan(want)
    assert np.max(np.abs(got[m] - want[m]), initial=0) <= 1e-5
    if name == "arch.xml":
        assert out["max_sigma"] == 0.0 and np.array_equal(bits(out["blurred"]), bits(out["image"]))
    else:
        assert out["max_sigma"] > 0.0
        again = r.render(product_params(api, p), blur=True, use_flag=False)
        assert np.array_equal(bits(again["blurred"]), bits(out["blurred"]))
    # end to end against the all-oracle pipeline
    full = port_oracle.blur(oimg, oblur)[..., :3]
    m = ~np.isnan(full) & ~np.isnan(got)
    assert np.max(np.abs(got[m] - full[m]), initial=0) <= 2e-4


def test_blur_against_the_reference_own_kernels(golden_dir, xml_dir, api):
    """k_blur_* against gaussHorizontal / gaussVertical themselves (helperKernels.cu:48-134 compiled for the host by
    oracle/ref_extract.sh), on a rendered frame with the scene's real sigmas: the stored frame and its reference blur
    (tests/golden/make_golden.py), and, where oracle/_ref is built, the GPU's own 200x150 render blurred live."""
    import torch

    z = np.load(os.path.join(golden_dir, "blur_fille.npz"))
    h, w = z["blur_map"].shape
    assert float(z["blur_map"].max()) > 4.0
    src = torch.from_numpy(z["image"]).cuda()
    sigma = torch.from_numpy(z["blur_map"]).cuda()
    dest, scratch = torch.empty_like(src), torch.empty_like(src)
    api.gaussian_blur(dest.data_ptr(), src.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, h, 0, h, 0,
                      torch.cuda.current_stream().cuda_stream)
    got, want = dest.cpu().numpy()[..., :3], z["blurred_rgb"]
    assert np.array_equal(np.isnan(got), np.isnan(want))
    m = ~np.isnan(want)
    assert np.max(np.abs(got[m] - want[m]), initial=0) <= 1e-5
    if not po.ref_extracts_available():
        return
    assert np.array_equal(bits(po.ref_blur(z["image"], z["blur_map"])[..., :3]), bits(want))  # the stored answer is the reference's
    r = GpuRenderer(os.path.join(xml_dir, "DiffusionCurvePack/fille.xml"))
    w, h, n = 200, 150, 8
    out = r.render(api.default_frame_params(w, h, n, zoom_factor=512 / h), blur=True)
    assert out["max_sigma"] > 4.0
    want = po.ref_blur(out["image"], out["blur_map"])[..., :3]
    got = out["blurred"][..., :3]
    assert np.array_equal(np.isnan(got), np.isnan(want))
    m = ~np.isnan(want)
    assert np.max(np.abs(got[m] - want[m]), initial=0) <= 1e-5


def test_banded_blur_equals_full_blur(api):
    """rdc_gaussian_blur_band: horizontal pass only on the band plus the rows its vertical pass can reach."""
    import torch

    h, w = 90, 70
    img = torch.rand((h, w, 4), dtype=torch.float32, device="cuda")
    sigma = torch.rand((h, w), dtype=torch.float32, device="cuda") * 4.0
    sigma[sigma < 1.0] = 0.0
    s = torch.cuda.current_stream().cuda_stream
    full, scratch = torch.zeros_like(img), torch.zeros_like(img)
    api.gaussian_blur(full.data_ptr(), img.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, h, 0, h, 0, s)
    halo = int(np.ceil(3 * 4.0))
    parts = torch.zeros_like(img)
    for b, e in ((0, 31), (31, 60), (60, 90)):
        scratch2 = torch.full_like(img, float("nan"))  # rows outside band + halo must never be read
        api.gaussian_blur_band(parts.data_ptr(), img.data_ptr(), sigma.data_ptr(), scratch2.data_ptr(), w, h, b, e, halo, 0, s)
    torch.cuda.synchronize()
    assert torch.equal(parts.view(torch.int32), full.view(torch.int32))


def test_reference_named_helpers(api):
    import torch

    x = torch.empty(1000, dtype=torch.float32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    api.lib.setFloatDevice(x.data_ptr(), 1000, 1e-3, s)
    api.lib.setupCurand(None, 16, 16, s)
    img = torch.rand((20, 30, 4), dtype=torch.float32, device="cuda")
    sigma = torch.full((20, 30), 1.25, dtype=torch.float32, device="cuda")
    ref = img.clone()
    api.lib.gaussianBlur(img.data_ptr(), img.data_ptr(), sigma.data_ptr(), 30, 20, s)  # in place, as the reference calls it
    torch.cuda.synchronize()
    assert torch.all(x == 1e-3)
    from oracle import pyoracle

    want = pyoracle.Oracle("port").blur(ref.cpu().numpy(), sigma.cpu().numpy())
    assert np.max(np.abs(img.cpu().numpy() - want)) <= 1e-5


def test_frame_to_host_equals_device_path(xml_dir, api):
    import torch

    r = GpuRenderer(os.path.join(xml_dir, "DiffusionCurvePack/fille.xml"))
    w, h, n = 64, 48, 8
    p = api.default_frame_params(w, h, n, zoom_factor=512 / h)
    dev = r.render(p, blur=True)
    host = torch.empty((h, w, 4), dtype=torch.float32).pin_memory()
    p2 = api.default_frame_params(w, h, n, zoom_factor=512 / h)
    r.scene.render_frame_to_host(p2, True, host.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert np.array_equal(bits(host.numpy()), bits(dev["blurred"]))


def test_pipelined_frames_equal_frame_by_frame(xml_dir, api):
    import torch

    r = GpuRenderer(os.path.join(xml_dir, "DiffusionCurvePack/zephyr.xml"))
    w, h, n = 96, 64, 8
    s = torch.cuda.current_stream().cuda_stream
    want = []
    for f in range(4):
        buf = torch.empty((h, w, 4), dtype=torch.float32).pin_memory()
        r.scene.render_frame_to_host(api.default_frame_params(w, h, n, zoom_factor=512 / h, frame=f), True, buf.data_ptr(), s)
        want.append(buf.numpy().copy())
    bufs = [torch.empty((h, w, 4), dtype=torch.float32).pin_memory() for _ in range(4)]
    for f in range(4):
        r.scene.render_frame_to_host_async(api.default_frame_params(w, h, n, zoom_factor=512 / h, frame=f), True, bufs[f].data_ptr(), s)
    r.scene.frame_wait()
    for f in range(4):
        assert np.array_equal(bits(bufs[f].numpy()), bits(want[f])), f
    assert not np.array_equal(bits(want[0]), bits(want[1]))  # frames differ: the frame number keys the generator


def test_bad_arguments_are_reported(xml_dir, api):
    r = GpuRenderer(os.path.join(xml_dir, "arch.xml"))
    import torch

    img = torch.empty((8, 8, 4), device="cuda")
    sig = torch.empty((8, 8), device="cuda")
    for kw in (dict(max_trace_depth=32), dict(row_begin=5, row_end=5), dict(row_end=9), dict(number_of_rays_per_pixel=0.0)):
        with pytest.raises(api.RdcError):
            r.scene.render(api.default_frame_params(8, 8, kw.pop("number_of_rays_per_pixel", 4), **kw), img.data_ptr(), sig.data_ptr())


def test_synthetic_scene_global_memory_path(api, port_oracle, tmp_path):
    """A scene too large for the shared-memory staging path (config 5 in miniature)."""
    xml = api.synth_xml(3000, 1024, 1024)
    f = tmp_path / "synth.xml"
    f.write_bytes(xml)
    scene = po.ingest_xml(str(f), True)
    p = po.make_params(48, 48, 8, zoom_factor=1024 / 48)
    oimg, oblur, ohits = port_oracle.render(scene, p, want_hits=True)
    r = GpuRenderer(str(f))
    assert r.scene.stats.traversal_bytes > 32 * 1024
    out = r.render(product_params(api, p), want_hits=True)
    assert np.array_equal(out["hits"], ohits)
    compare_images(out["image"], oimg, RGB_TOL)


LOCAL_VIEWS = [("DiffusionCurvePack/dolphin.xml", 0.25, 0.0, 0.0, 16), ("DiffusionCurvePack/dolphin.xml", 0.5, 60.0, -40.0, 16),
               ("DiffusionCurvePack/dolphin.xml", 2.0, 0.0, 0.0, 8), ("DiffusionCurvePack/lady_bug.xml", 1.0, -30.0, 20.0, 24),
               ("DiffusionCurvePack/zephyr.xml", 0.125, 10.0, 10.0, 16), ("DiffusionCurvePack/face.xml", 0.3, -20.0, 35.0, 40),
               ("DiffusionCurvePack/roses_spirales.xml", 0.75, 0.0, 0.0, 16)]


@pytest.mark.parametrize("name,zoom,off_x,off_y,n", LOCAL_VIEWS, ids=[f"{v[0].split('/')[-1]}@{v[1]}" for v in LOCAL_VIEWS])
def test_local_run_table_views(name, zoom, off_x, off_y, n, xml_dir, api, port_oracle):
    """Close-up views of the larger scenes through the LOCAL run table (the route of scenes too large for a cut through the
    tree; forced here): primary rays settled by the per-tile table of nearby runs, the rest deferred to the tree — every first
    hit still the oracle's brute-force closest chord."""
    path = os.path.join(xml_dir, name)
    scene = po.ingest_xml(path, True)
    w, h = 72, 52  # not a multiple of the 8x4 tile
    # route: left to itself the library keeps scenes this small on the tree (it is faster there)
    p = po.make_params(w, h, n, zoom_factor=zoom, offset_x=off_x, offset_y=off_y, route=api.ROUTE_LOCAL_TABLE)
    oimg, oblur, ohits = port_oracle.render(scene, p, want_hits=True)
    r = GpuRenderer(path)
    out = r.render(product_params(api, p), want_hits=True)
    assert np.array_equal(out["hits"], ohits)
    compare_images(out["image"], oimg, RGB_TOL)
    brute = r.render(product_params(api, po.make_params(w, h, n, zoom_factor=zoom, offset_x=off_x, offset_y=off_y,
                                                        traversal=api.TRAVERSAL_BRUTE_FORCE)), want_hits=True)
    assert np.array_equal(out["hits"], brute["hits"])
    counted = r.render(product_params(api, p), want_hits=True, want_stats=True)
    assert np.array_equal(counted["hits"], ohits)
    traced, _, _, _, deferred, gathered = counted["stats"]
    print(f"{name} zoom {zoom}: {traced} rays traced, {deferred} deferred to the tree, {gathered} nodes visited by table queries")
    if zoom <= 1.0:
        assert gathered > 0, "the local run table was not used"
        assert deferred < traced


def test_local_run_table_synthetic_close_up(api, port_oracle, tmp_path):
    """Config 5 in miniature at its own scale (one pixel = one scene unit): the local-table path on a dense scene."""
    xml = api.synth_xml(3000, 1024, 1024)
    f = tmp_path / "synth.xml"
    f.write_bytes(xml)
    scene = po.ingest_xml(str(f), True)
    r = GpuRenderer(str(f))
    for off_x, off_y, n in ((0.0, 0.0, 16), (300.0, -250.0, 32), (-480.0, 470.0, 8)):
        p = po.make_params(64, 48, n, zoom_factor=1.0, offset_x=off_x, offset_y=off_y, route=api.ROUTE_LOCAL_TABLE)
        oimg, oblur, ohits = port_oracle.render(scene, p, want_hits=True)
        out = r.render(product_params(api, p), want_hits=True, want_stats=True)
        assert np.array_equal(out["hits"], ohits)
        compare_images(out["image"], oimg, RGB_TOL)
        traced, _, _, _, deferred, gathered = out["stats"]
        assert gathered > 0 and deferred < traced
        plain = r.render(product_params(api, p), want_hits=True)
        assert np.array_equal(plain["hits"], ohits)
        # the same frame in two bands: bit-identical pixels (the table depends on the tile only)
        parts = [r.render(product_params(api, po.make_params(64, 48, n, zoom_factor=1.0, offset_x=off_x, offset_y=off_y,
                                                               route=api.ROUTE_LOCAL_TABLE, row_begin=b, row_end=e)))
                 for b, e in ((0, 16), (16, 48))]
        assert np.array_equal(bits(np.concatenate([q["image"] for q in parts])), bits(plain["image"]))


def test_local_run_table_with_portals(api, port_oracle, tmp_path):
    """The local-table kernel on a scene that has `connects` curves: primary hits settled by the table continue
    through portals on the tree; deferred rays do the same."""
    import re

    xml = api.synth_xml(1500, 512, 512).decode()
    count = [0]

    def connect(m):  # curves 10k <-> 10k+1 become a portal pair (every synthetic curve has one segment)
        c = count[0]
        count[0] += 1
        if c % 10 == 0:
            return f'<curve connects="{c + 1}" '
        if c % 10 == 1:
            return f'<curve connects="{c - 1}" '
        return m.group(0)

    xml = re.sub(r"<curve ", connect, xml)
    f = tmp_path / "synth_portals.xml"
    f.write_text(xml)
    scene = po.ingest_xml(str(f), True)
    assert (scene["curve_connect"] >= 0).sum() == 300
    r = GpuRenderer(str(f))
    for depth in (0, 2, 31):
        p = po.make_params(64, 48, 16, zoom_factor=1.0, offset_x=20.0, offset_y=-30.0, max_trace_depth=depth,
                           route=api.ROUTE_LOCAL_TABLE)
        oimg, oblur, ohits = port_oracle.render(scene, p, want_hits=True)
        out = r.render(product_params(api, p), want_hits=True, want_stats=True)
        assert np.array_equal(out["hits"], ohits)
        compare_images(out["image"], oimg, RGB_TOL)
        assert out["stats"][5] > 0, "the local run table was not used"
        plain = r.render(product_params(api, p), want_hits=True)
        assert np.array_equal(plain["hits"], ohits)
        compare_images(plain["image"], oimg, RGB_TOL)


def test_accumulate_is_a_running_mean(api):
    import torch

    frames = [torch.rand((6, 5, 4), dtype=torch.float32, device="cuda") for _ in range(5)]
    acc = torch.zeros_like(frames[0])
    s = torch.cuda.current_stream().cuda_stream
    for k, f in enumerate(frames):
        assert api.lib.rdc_accumulate(acc.data_ptr(), f.data_ptr(), 30, k, s) == 0
    torch.cuda.synchronize()
    assert torch.allclose(acc, torch.stack(frames).mean(0), atol=1e-6)


def test_optixhello_cli_renders_and_reports(xml_dir, tmp_path):
    """The reference's command line: positional xml (relative to the current directory) and rays per pixel;
    'Setup took' and 'Average frame time' lines (optixHello.cpp:1157,1263)."""
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "raytracingdiffusioncurves_b200", "OptixHello")
    out = tmp_path / "arch.png"
    r = subprocess.run([exe, "tests/golden/xmls/arch.xml", "16", "--width", "160", "--height", "120", "--frames", "2", "--out", str(out)],
                       cwd=root, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Setup took : " in r.stdout and "Average frame time  : " in r.stdout and "frame : 2" in r.stdout
    assert out.read_bytes()[:8] == b"\x89PNG\r\n\x1a\n"
    missing = subprocess.run([exe, "tests/golden/xmls/nope.xml", "16"], cwd=root, capture_output=True, text=True)
    assert missing.returncode == 2 and "cannot open" in missing.stderr
