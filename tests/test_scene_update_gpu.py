"""rdc_scene_update_stops: new stop lists on a built scene, and the stop tables k_stop_tables derives from them.

The stop tables (seg_walk, chord_walk, chord_records: device_scene.h) are pinned to a numpy restatement of the sequential
host loop that built them before they were built on the GPU. An update must leave the handle equal, table for table and
frame for frame, to a fresh build of the edited arrays, on every route, with and without shading records, whatever stream
it is issued on, and a rejected update must leave the handle as it was.
"""
import ctypes
import math
import os

import numpy as np
import pytest

from helpers import bits, compare_images, copy_params, scene_ids
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

FAMILIES = ("color_left", "color_right", "blur", "weight", "weight_degree")
RDC_E_INVALID = -1
SYNTH_PORTALS = "synth_portals"  # 1500 one-segment curves, every tenth pair joined by a portal


@pytest.fixture(scope="module")
def api():
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from raytracingdiffusioncurves_b200 import api as _api

    return _api


def synth_portals_xml(api) -> str:
    """The synthetic portal scene of test_render_variants_gpu: curves 10k and 10k+1 are a portal pair."""
    import re

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


@pytest.fixture(scope="module")
def scene_dicts(api, xml_dir, tmp_path_factory):
    """Scene name -> the ingested arrays as numpy (HostScene.to_numpy), each read once."""
    synth = str(tmp_path_factory.mktemp("update") / "synth_portals.xml")
    with open(synth, "w") as fh:
        fh.write(synth_portals_xml(api))
    cache = {}

    def get(name):
        if name not in cache:
            path = synth if name == SYNTH_PORTALS else os.path.join(xml_dir, name)
            cache[name] = api.HostScene.from_xml_file(path).to_numpy()
        return cache[name]

    return get


def stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def build(api, d, records=True, on=None):
    return api.Scene(api.arrays_from_numpy(d), api.default_accel_options(shading_records=0 if records else -1),
                     stream() if on is None else on)


# ---------------------------------------------------------------------------------------------------------------------
# the sequential host loop that built the stop tables before k_stop_tables, restated in numpy
# ---------------------------------------------------------------------------------------------------------------------
def walk(j, end, us, x):
    """rdc_walk_hint, vectorised: advance each j while j < end and us[j + 1] < x."""
    j = j.copy()
    while True:
        step = j < end
        step[step] = us[j[step] + 1] < x[step]
        if not step.any():
            return j
        j[step] += 1


def host_loop_tables(d, chord_ids, with_records):
    """seg_walk, chord_walk and chord_records as build_scene's host loop made them: per segment, the walks at the ordinal;
    per chord in k order, each walk continued from the previous chord's position to rdc_hit_u(k, K, 0) + ordinal."""
    f32 = np.float32
    nseg = len(d["curve_map"])
    c = d["curve_map"].astype(np.int64)
    ordinal = d["curve_index"]
    o32 = ordinal.astype(f32)
    K = np.bincount(chord_ids[:, 0], minlength=nseg).astype(np.int64)
    base = np.concatenate([[0], np.cumsum(K)])
    n_chords = int(base[-1])
    # walk order: left, right, blur, weight, exponent, portal-left (the right list's range on the left u array)
    idx = [d[f + "_index"] for f in FAMILIES] + [d["color_right_index"]]
    us = [d[f + "_u"] for f in FAMILIES] + [d["color_left_u"]]
    start = [ix[c, 0].astype(np.int64) for ix in idx]
    end = [ix[c, 0].astype(np.int64) + ix[c, 1] for ix in idx]

    seg_walk = np.zeros((nseg, 16), np.uint32)
    for w in range(6):
        col = 2 * w if w < 5 else 12
        seg_walk[:, col] = walk(start[w], end[w], us[w], o32)
        seg_walk[:, col + 1] = end[w]
    seg_walk[:, 10], seg_walk[:, 11] = c, ordinal

    chord_walk = np.zeros((n_chords, 8), np.uint32)
    records = np.zeros((n_chords, 32), np.float32) if with_records else None
    rec_bits = records.view(np.uint32) if with_records else None
    prev = [s.copy() for s in start]
    for k in range(int(K.max())):
        sel = np.nonzero(K > k)[0]
        Kf = K[sel].astype(f32)
        cu_min = (f32(k) + f32(0)) / Kf + o32[sel]
        chord = base[sel] + k
        f = []
        for w in range(6):
            prev[w][sel] = walk(prev[w][sel], end[w][sel], us[w], cu_min)
            f.append(prev[w][sel])
        chord_walk[chord, :6] = np.stack(f, 1)
        if not with_records:
            continue
        cu_max = (f32(k) + f32(1)) / Kf + o32[sel]
        flags = np.zeros(len(sel), np.uint32)
        for w in range(5):
            steps = (f[w] < end[w][sel]) & (us[w][np.minimum(f[w] + 1, len(us[w]) - 1)] < cu_max)
            flags |= np.where(steps, 0, 1 << w).astype(np.uint32)
        for sf, fam in enumerate(("blur", "weight", "weight_degree")):
            j, u, v = f[2 + sf], d[fam + "_u"], d[fam]
            records[chord, 4 * sf:4 * sf + 4] = np.stack([u[j], u[j + 1], v[j], v[j + 1]], 1)
        for side, fam in enumerate(("color_left", "color_right")):
            j, u, v = f[side], d[fam + "_u"], d[fam]
            records[chord, 12 + 8 * side:15 + 8 * side] = v[j]
            records[chord, 15 + 8 * side] = u[j]
            records[chord, 16 + 8 * side:19 + 8 * side] = v[j + 1]
            records[chord, 19 + 8 * side] = u[j + 1]
        cs = c[sel].astype(np.uint32)
        meta_w = (cs & 0x07FFFFFF) | (flags << 27)
        meta_w = np.where((K[sel] > 0xFFFF) | (cs > 0x07FFFFFF), meta_w & 0x07FFFFFF, meta_w)
        rec_bits[chord, 28] = sel
        rec_bits[chord, 29] = ordinal[sel]
        rec_bits[chord, 30] = (np.uint32(k) | (K[sel].astype(np.uint32) << 16)).astype(np.uint32)
        rec_bits[chord, 31] = meta_w
    return {"seg_walk": seg_walk, "chord_walk": chord_walk, "chord_records": records}


def assert_same_tables(got, want, what=""):
    for key in ("seg_walk", "chord_walk", "chord_records"):
        if want[key] is None:
            assert got[key] is None, f"{what}: {key}"
            continue
        g, w = bits(got[key]), bits(want[key])
        assert g.shape == w.shape, f"{what}: {key} shape"
        bad = np.argwhere(g != w)
        assert len(bad) == 0, f"{what}: {key} differs at {len(bad)} words, first [row, word] {bad[:3].tolist()}"


@pytest.mark.parametrize("name", scene_ids() + [SYNTH_PORTALS])
def test_stop_tables_equal_the_host_loop(name, api, scene_dicts):
    d = scene_dicts(name)
    for records in (True, False):
        scene = build(api, d, records)
        _, ids = scene.chords()
        got = scene.stop_tables()
        assert (got["chord_records"] is not None) == records
        assert_same_tables(got, host_loop_tables(d, ids, records), f"{name}, records {records}")


# ---------------------------------------------------------------------------------------------------------------------
# edits of the stop lists
# ---------------------------------------------------------------------------------------------------------------------
def lists_of(d, fam):
    """Per curve: (u, values) of family `fam`."""
    return [(d[fam + "_u"][s:s + n].copy(), d[fam][s:s + n].copy()) for s, n in d[fam + "_index"]]


def with_lists(d, new):
    """A copy of scene `d` whose families are rebuilt from per-curve lists (`new` overrides some), with the sentinels and
    padding of rdc_scene_arrays: +INF parameters and zero values past the end, both colour families max(n) + 2 long."""
    e = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in d.items()}
    lists = {f: new[f] if f in new else lists_of(d, f) for f in FAMILIES}
    n = {f: sum(len(u) for u, _ in lists[f]) for f in FAMILIES}
    colour_len = max(n["color_left"], n["color_right"]) + 2
    for f in FAMILIES:
        colour = f.startswith("color")
        padded = colour_len if colour else n[f] + 2
        u = np.full((padded,), np.inf, np.float32)
        v = np.zeros((padded, 3) if colour else (padded,), np.float32)
        index = np.zeros((len(lists[f]), 2), np.uint32)
        at = 0
        for c, (uu, vv) in enumerate(lists[f]):
            index[c] = (at, len(uu))
            u[at:at + len(uu)] = uu
            v[at:at + len(uu)] = vv
            at += len(uu)
        e["n_" + f], e[f + "_index"], e[f], e[f + "_u"] = n[f], index, v, u
    return e


def new_values(fam, shape, rng):
    if fam.startswith("color"):
        return rng.random(shape, dtype=np.float32)
    lo, hi = {"blur": (0.0, 2.5), "weight": (0.5, 2.0), "weight_degree": (0.2, 1.5)}[fam]
    return rng.uniform(lo, hi, shape).astype(np.float32)


def edit_values(d, rng):
    """Every colour, blur, weight and exponent value replaced; counts and parameters kept."""
    return with_lists(d, {f: [(u, new_values(f, v.shape, rng)) for u, v in lists_of(d, f)] for f in FAMILIES})


def edit_positions(d, rng):
    """Every stop moved along its curve by up to a quarter segment (lists may end up unsorted)."""
    return with_lists(d, {f: [((u + rng.uniform(-0.25, 0.25, u.shape)).astype(np.float32), v) for u, v in lists_of(d, f)]
                          for f in FAMILIES})


def edit_grow(d, rng):
    """A stop added between every two stops of every list (one after a single stop): the lists outgrow the handle."""
    new = {}
    for f in FAMILIES:
        out = []
        for u, v in lists_of(d, f):
            mid_u = (u[:-1] + u[1:]) / 2 if len(u) > 1 else u + np.float32(0.5)
            mid_v = new_values(f, (len(mid_u),) + v.shape[1:], rng)
            uu = np.empty((len(u) + len(mid_u),), np.float32)
            vv = np.empty((len(uu),) + v.shape[1:], np.float32)
            uu[0::2], vv[0::2] = u, v
            uu[1::2], vv[1::2] = mid_u, mid_v
            out.append((uu, vv))
        new[f] = out
    return with_lists(d, new)


def edit_shrink(d, rng):
    """Every other stop removed from lists of two stops or more."""
    return with_lists(d, {f: [(u[::2], v[::2]) if len(u) > 1 else (u, v) for u, v in lists_of(d, f)] for f in FAMILIES})


def edit_single(d, rng):
    """The weight family cut to one stop per curve."""
    return with_lists(d, {"weight": [(u[:1], v[:1]) for u, v in lists_of(d, "weight")]})


def edit_restore(d, rng):
    return d


EDITS = [("values", edit_values), ("positions", edit_positions), ("grow", edit_grow), ("shrink", edit_shrink),
         ("single", edit_single), ("restore", edit_restore)]
EDIT_SCENES = [("arch.xml", 2), ("DiffusionCurvePack/lady_bug.xml", 2), ("PortalDemo.xml", 2), ("PortalDemo.xml", 31),
               ("weight_demo.xml", 2), ("DiffusionCurvePack/fille.xml", 2), (SYNTH_PORTALS, 2)]
EDIT_IDS = [f"{n.split('/')[-1]}-d{depth}" for n, depth in EDIT_SCENES]


# ---------------------------------------------------------------------------------------------------------------------
# frames
# ---------------------------------------------------------------------------------------------------------------------
def render(api, scene, p, on=None, blur=False):
    """One launch into fresh device buffers; returns host copies of image, blur map and hit ids (and the blurred image)."""
    import torch

    rows, w = p.row_end - p.row_begin, p.image_width
    image = torch.empty((rows, w, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((rows, w), dtype=torch.float32, device="cuda")
    hits = torch.empty((rows, w, int(math.ceil(p.number_of_rays_per_pixel))), dtype=torch.int32, device="cuda")
    q = copy_params(p, type(p))
    q.hit_ids = hits.data_ptr()
    st = stream() if on is None else on
    scene.render(q, image.data_ptr(), sigma.data_ptr(), st)
    out = {"image": image, "blur_map": sigma, "hits": hits}
    if blur:
        scratch, blurred = torch.empty_like(image), torch.empty_like(image)
        api.gaussian_blur(blurred.data_ptr(), image.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, rows, 0, rows, 0, st)
        out["blurred"] = blurred
    return out


def to_host(out):
    import torch

    torch.cuda.synchronize()
    return {k: (v.cpu().numpy().view(np.uint32) if k == "hits" else v.cpu().numpy()) for k, v in out.items()}


def assert_same_frame(a, b, what=""):
    for key in a:
        assert np.array_equal(bits(a[key]), bits(b[key])), f"{what}: {key} differs"


W, H, N = 27, 18, 32


def view(api, d, depth, **kw):
    return api.default_frame_params(W, H, N, zoom_factor=d["image_height"] / H, max_trace_depth=depth, **kw)


def route_frames(api, scene, d, depth):
    """The frame on the tree, local-table, cut-table and automatic routes, units per tile pinned."""
    frames = [render(api, scene, view(api, d, depth, route=route, units_per_tile=2))
              for route in (api.ROUTE_TREE, api.ROUTE_LOCAL_TABLE, api.ROUTE_CUT_TABLE, api.ROUTE_AUTO)]
    return [to_host(f) for f in frames]


@pytest.mark.parametrize("name,depth", EDIT_SCENES, ids=EDIT_IDS)
def test_update_equals_a_fresh_build(name, depth, api, scene_dicts):
    d0 = scene_dicts(name)
    rng = np.random.default_rng(7)
    for records in (True, False):
        scene = build(api, d0, records)
        original = route_frames(api, scene, d0, depth)
        capacity = scene.stats.device_bytes
        for what, edit in EDITS:
            d = edit(d0, rng)
            scene.update_stops(api.arrays_from_numpy(d))
            fresh = build(api, d, records)
            tag = f"{name} d{depth} records {records}, edit {what}"
            assert_same_tables(scene.stop_tables(), fresh.stop_tables(), tag)
            got = route_frames(api, scene, d, depth)
            for g, w in zip(got, route_frames(api, fresh, d, depth)):
                assert_same_frame(g, w, tag)
            if what == "grow":
                assert scene.stats.device_bytes > capacity, "the grown lists did not need more room"
            if what == "restore":
                for g, w in zip(got, original):
                    assert_same_frame(g, w, tag + " against the original handle")
            fresh.close()
        scene.close()


def check_against_oracle(out, want, oracle):
    """Hits bit-exact, RGB within 1e-4, the blur map's NaN pattern and values; a blurred frame within 1e-5 of the oracle's
    blur of the same frame."""
    oimg, oblur, ohits = want
    assert np.array_equal(out["hits"], ohits), f"{int((out['hits'] != ohits).sum())} hit ids differ from the oracle"
    compare_images(out["image"], oimg, 1e-4)
    assert np.array_equal(np.isnan(out["blur_map"]), np.isnan(oblur))
    m = ~np.isnan(oblur)
    assert np.max(np.abs(out["blur_map"][m] - oblur[m]), initial=0) <= 1e-4 * max(1.0, float(np.nanmax(oblur, initial=0)))
    if "blurred" in out:
        assert float(np.nanmax(out["blur_map"], initial=0)) > 1.0
        compare_images(out["blurred"], oracle.blur(out["image"], out["blur_map"]), 1e-5)


@pytest.mark.parametrize("name,depth", EDIT_SCENES, ids=EDIT_IDS)
def test_edited_scene_against_the_oracle(name, depth, api, scene_dicts, port_oracle):
    d0 = scene_dicts(name)
    rng = np.random.default_rng(11)
    scene = build(api, d0)
    blur = name.endswith("fille.xml")
    for what, edit in EDITS:
        d = edit(d0, rng)
        scene.update_stops(api.arrays_from_numpy(d))
        p = view(api, d, depth)
        out = to_host(render(api, scene, p, blur=blur))
        want = port_oracle.render(d, copy_params(p, po.FrameParams), want_hits=True, search="grid")
        check_against_oracle(out, want, port_oracle)


# ---------------------------------------------------------------------------------------------------------------------
# stream order without host waits
# ---------------------------------------------------------------------------------------------------------------------
LADY = "DiffusionCurvePack/lady_bug.xml"


def test_update_on_another_stream_is_ordered_like_a_launch(api, scene_dicts):
    import torch

    d0 = scene_dicts(LADY)
    rng = np.random.default_rng(3)
    a, b = torch.cuda.Stream(), torch.cuda.Stream()
    big = api.default_frame_params(256, 256, 128, zoom_factor=2.0)  # long enough for the update to be issued meanwhile
    small = view(api, d0, 2)
    for what, edit in (("fits", edit_values), ("grows", edit_grow)):
        d = edit(d0, rng)
        scene = build(api, d0)
        torch.cuda.synchronize()
        first = render(api, scene, big, a.cuda_stream)
        scene.update_stops(api.arrays_from_numpy(d), b.cuda_stream)
        second = render(api, scene, small, a.cuda_stream)
        first, second = to_host(first), to_host(second)
        old, new = build(api, d0), build(api, d)
        assert_same_frame(first, to_host(render(api, old, big)), f"{what}: the frame before the update")
        assert_same_frame(second, to_host(render(api, new, small)), f"{what}: the frame after the update")


def test_alternating_updates_and_renders(api, scene_dicts):
    """32 updates on one stream and renders on another, no host wait in between. The caller's arrays are one set of numpy
    buffers changed in place after every call, so a frame only comes out right when each update took its own copy."""
    import torch

    d0 = scene_dicts(LADY)
    rng = np.random.default_rng(5)
    versions = [edit_values(d0, rng) for _ in range(32)]
    work = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in d0.items()}
    arrays = api.arrays_from_numpy(work)
    a, b = torch.cuda.Stream(), torch.cuda.Stream()
    scene = build(api, d0)
    p = view(api, d0, 2)
    scene.update_stops(arrays, b.cuda_stream)  # the first update allocates the staging buffer
    torch.cuda.synchronize()
    outs = []
    for v in versions:
        for f in FAMILIES:
            work[f][...] = v[f]
        scene.update_stops(arrays, b.cuda_stream)
        outs.append(render(api, scene, p, a.cuda_stream))
    for f in FAMILIES:
        work[f][...] = 0.0
    for i, (v, out) in enumerate(zip(versions, outs)):
        assert_same_frame(to_host(out), to_host(render(api, build(api, v), p)), f"update {i}")


# ---------------------------------------------------------------------------------------------------------------------
# rejections
# ---------------------------------------------------------------------------------------------------------------------
def test_rejected_update_leaves_the_handle_intact(api, scene_dicts):
    d0 = scene_dicts("PortalDemo.xml")
    scene = build(api, d0)
    p = view(api, d0, 2)
    before = to_host(render(api, scene, p))
    tables = scene.stop_tables()
    good = edit_values(d0, np.random.default_rng(1))

    def attempt(arrays):
        rc = api.lib.rdc_scene_update_stops(scene.handle, ctypes.byref(arrays) if arrays is not None else None, None)
        assert rc == RDC_E_INVALID
        assert api.last_error()
        assert_same_frame(to_host(render(api, scene, p)), before, "after a rejected update")
        assert_same_tables(scene.stop_tables(), tables, "after a rejected update")

    for field in ("n_curves", "n_segments", "n_vertices"):
        arrays = api.arrays_from_numpy(good)
        setattr(arrays, field, getattr(arrays, field) - 1)
        attempt(arrays)
    past = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in good.items()}
    past["blur_index"][-1, 1] += 3  # the last curve's blur stops run past the list
    attempt(api.arrays_from_numpy(past))
    for field in ("color_right_index", "weight", "blur_u"):
        arrays = api.arrays_from_numpy(good)
        setattr(arrays, field, None)
        attempt(arrays)
    attempt(None)
    assert api.lib.rdc_scene_update_stops(None, ctypes.byref(api.arrays_from_numpy(good)), None) == RDC_E_INVALID
    scene.update_stops(api.arrays_from_numpy(good))  # the handle still takes a good update
    assert_same_frame(to_host(render(api, scene, p)), to_host(render(api, build(api, good), p)), "a good update after rejections")


# ---------------------------------------------------------------------------------------------------------------------
# frame-to-host and peer paths
# ---------------------------------------------------------------------------------------------------------------------
def halo_rows(d, depth):
    """ceil(3 * largest blur a frame can hold), from the (edited) blur stops, as HostScene.max_blur and
    rdc_host_scene_halo_rows compute it from a host scene."""
    m = float(d["blur"][:d["n_blur"]].max(initial=0.0))
    if (d["curve_connect"] >= 0).any() and m > 1.0:
        m = m ** (depth + 1)
    return int(math.ceil(3 * max(m, 0.0)))


def test_frame_to_host_sees_the_update(api, scene_dicts):
    import torch

    d0 = scene_dicts(LADY)
    d = edit_values(d0, np.random.default_rng(9))
    p = api.default_frame_params(96, 76, 16, zoom_factor=512 / 76)
    updated = build(api, d0)
    updated.update_stops(api.arrays_from_numpy(d))
    frames = []
    for scene in (updated, build(api, d)):
        host = torch.empty((76, 96, 4), dtype=torch.float32).pin_memory()
        scene.render_frame_to_host(p, True, host.data_ptr(), stream())
        frames.append(host.numpy().copy())
    assert np.array_equal(bits(frames[0]), bits(frames[1]))


def peer_frame(api, d0, d, width, height, world=2):
    """rdc_peer_render_frame over `world` ranks in this process (device rank % device_count), each rank's handle built
    from d0 and updated to d (d0 None: built from d). Returns rank 0's finished frame."""
    import torch

    n_dev = torch.cuda.device_count()
    devices = [r % n_dev for r in range(world)]
    scenes, streams, frames = [], [], []
    for r, dev in enumerate(devices):
        with torch.cuda.device(dev):
            s = torch.cuda.Stream()
            scene = build(api, d if d0 is None else d0, on=s.cuda_stream)
            if d0 is not None:
                scene.update_stops(api.arrays_from_numpy(d), s.cuda_stream)
            streams.append(s)
            scenes.append(scene)
            frames.append(api.PeerFrames(width, height, r, world))
    api.PeerFrames.connect_local(frames)
    p = api.default_frame_params(width, height, 8, zoom_factor=512 / height)
    halo = halo_rows(d, p.max_trace_depth)
    for r, dev in enumerate(devices):
        with torch.cuda.device(dev):
            scenes[r].reserve(p, False, streams[r].cuda_stream)
    ptr = 0
    for r, dev in enumerate(devices):
        with torch.cuda.device(dev):
            got = frames[r].render_frame(scenes[r], p, True, halo, streams[r].cuda_stream)
            ptr = got if r == 0 else ptr
    for dev in set(devices):
        torch.cuda.synchronize(dev)
    for f in frames:
        f.status()
    out = torch.empty((height, width, 4), dtype=torch.float32)
    with torch.cuda.device(devices[0]):
        rc = ctypes.CDLL("libcudart.so").cudaMemcpy(ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(ptr),
                                                    ctypes.c_size_t(out.numel() * 4), 2)
        assert rc == 0
    for f in frames:
        f.close()
    return out.numpy()


def test_peer_frame_sees_the_update(api, scene_dicts):
    """The update raises the blur: the blur's reach (halo_rows) is recomputed from the edited stops."""
    d0 = scene_dicts(LADY)
    d = edit_values(d0, np.random.default_rng(13))
    n = d["n_blur"]
    d["blur"][:n] = d0["blur"][:n] * np.float32(1.5) + np.float32(1.0)
    assert halo_rows(d, 2) > halo_rows(d0, 2)
    got = peer_frame(api, d0, d, 96, 76)
    want = peer_frame(api, None, d, 96, 76)
    assert np.array_equal(bits(got[..., :3]), bits(want[..., :3]))
