"""What a colour edit costs: rdc_scene_update_stops against a rebuild with rdc_accel_build, and one frame for scale.
    python tools/time_update.py                                   # this tree's library
    RDC_B200_LIB=/path/to/parent/librdc_b200.so python tools/time_update.py   # also the other library's build, alternated

Per scene (lady_bug.xml, dolphin.xml, the synthetic 100 k-curve scene of bench.py's config 5):
  - build: rdc_accel_build, host clock around the call (it ends synchronised);
  - update that fits: device events around rdc_scene_update_stops with new values (same counts), and the host time the
    call takes to enqueue; no host synchronisation happens in it, so the enqueue time stays far below a build;
  - update that grows: every stop doubled, on a fresh handle, host clock around the call and a synchronise;
  - one frame, 1920x1080 @128 rays per pixel, device events.
Prints the card's name and power limit first, then one line per scene and one JSON line per scene."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OTHER_LIB = os.environ.pop("RDC_B200_LIB", None)  # this tree's library for the api; the other one is loaded below
import numpy as np  # noqa: E402
import torch  # noqa: E402

from raytracingdiffusioncurves_b200 import api  # noqa: E402

XML = os.path.join(ROOT, "tests", "golden", "xmls")
FAMILIES = ("color_left", "color_right", "blur", "weight", "weight_degree")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()


def new_values(d, seed):
    """Every stop value replaced, counts and parameters kept: an update that fits."""
    rng = np.random.default_rng(seed)
    e = dict(d)
    for f in FAMILIES:
        v = d[f].copy()
        n = d["n_" + f]
        v[:n] = rng.random(v[:n].shape, dtype=np.float32) * (2.0 if f == "blur" else 1.0) + (0.5 if f == "weight" else 0.0)
        e[f] = v
    return e


def doubled(d):
    """Every stop twice: the lists need twice the room, an update that grows."""
    e = dict(d)
    n = {f: 2 * d["n_" + f] for f in FAMILIES}
    colour_len = max(n["color_left"], n["color_right"]) + 2
    for f in FAMILIES:
        colour = f.startswith("color")
        padded = colour_len if colour else n[f] + 2
        u = np.full((padded,), np.inf, np.float32)
        v = np.zeros((padded, 3) if colour else (padded,), np.float32)
        u[:n[f]] = np.repeat(d[f + "_u"][:d["n_" + f]], 2)
        v[:n[f]] = np.repeat(d[f][:d["n_" + f]], 2, axis=0)
        e["n_" + f], e[f + "_u"], e[f], e[f + "_index"] = n[f], u, v, d[f + "_index"] * 2
    return e


def other_builder():
    if not OTHER_LIB:
        return None
    lib = C.CDLL(OTHER_LIB)
    lib.rdc_accel_build.argtypes = [C.POINTER(api.SceneArrays), C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.rdc_accel_build.restype = C.c_int
    lib.rdc_scene_destroy.argtypes = [C.c_void_p]

    def build(arrays, stream):
        h = C.c_void_p()
        t0 = time.perf_counter()
        rc = lib.rdc_accel_build(C.byref(arrays), None, C.c_void_p(stream), C.byref(h))
        torch.cuda.synchronize()
        t = (time.perf_counter() - t0) * 1e3
        assert rc == 0, rc
        lib.rdc_scene_destroy(h)
        return t

    return build


def main():
    torch.cuda.init()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
    print(f"other library: {OTHER_LIB or 'none'}", flush=True)
    other = other_builder()
    scenes = [("lady_bug.xml", os.path.join(XML, "DiffusionCurvePack", "lady_bug.xml")),
              ("dolphin.xml", os.path.join(XML, "DiffusionCurvePack", "dolphin.xml")),
              ("synth100k", api.synth_xml(100000, 8192, 8192))]
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, src in scenes:
        host = api.HostScene.from_xml_text(src) if isinstance(src, bytes) else api.HostScene.from_xml_file(src)
        d = host.to_numpy()
        arrays = api.arrays_from_numpy(d)

        def build():
            t0 = time.perf_counter()
            s = api.Scene(arrays, None, stream)
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3, s

        build()[1].close()  # first build: module load
        if other:
            other(arrays, stream)
        builds, other_builds = [], []
        for _ in range(7):  # the two libraries alternate
            t, s = build()
            builds.append(t)
            s.close()
            if other:
                other_builds.append(other(arrays, stream))

        scene = build()[1]
        edits = [api.arrays_from_numpy(new_values(d, seed)) for seed in range(2)]
        scene.update_stops(edits[0], stream)  # the handle's first update allocates its staging buffer
        torch.cuda.synchronize()
        dev_ms, enqueue_ms = [], []
        for i in range(20):
            start.record()
            t0 = time.perf_counter()
            scene.update_stops(edits[i % 2], stream)
            enqueue_ms.append((time.perf_counter() - t0) * 1e3)
            stop.record()
            torch.cuda.synchronize()
            dev_ms.append(start.elapsed_time(stop))

        grown = api.arrays_from_numpy(doubled(d))
        grow_ms = []
        for _ in range(3):
            s = build()[1]
            t0 = time.perf_counter()
            s.update_stops(grown, stream)
            torch.cuda.synchronize()
            grow_ms.append((time.perf_counter() - t0) * 1e3)
            s.close()

        p = api.default_frame_params(1920, 1080, 128, zoom_factor=d["image_height"] / 1080)
        image = torch.empty((1080, 1920, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((1080, 1920), dtype=torch.float32, device="cuda")
        scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)
        frame_ms = []
        for _ in range(5):
            start.record()
            scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)
            stop.record()
            torch.cuda.synchronize()
            frame_ms.append(start.elapsed_time(stop))

        med = statistics.median
        res = {"scene": name, "chords": scene.stats.n_chords, "curves": scene.stats.n_curves,
               "build_ms": med(builds), "build_ms_min": min(builds),
               "other_build_ms": med(other_builds) if other else None, "other_build_ms_min": min(other_builds) if other else None,
               "update_fits_device_ms": med(dev_ms), "update_fits_enqueue_ms": med(enqueue_ms),
               "update_fits_enqueue_ms_max": max(enqueue_ms), "update_grows_ms": med(grow_ms), "frame_1080p_128_ms": med(frame_ms)}
        other_txt = f" (other library {res['other_build_ms']:.2f} ms)" if other else ""
        print(f"{name}: {res['chords']} chords; build {res['build_ms']:.2f} ms{other_txt}; update that fits "
              f"{res['update_fits_device_ms']:.3f} ms on the device, {res['update_fits_enqueue_ms']:.3f} ms to enqueue; update that "
              f"grows {res['update_grows_ms']:.2f} ms; frame 1080p@128 {res['frame_1080p_128_ms']:.2f} ms", flush=True)
        print(json.dumps(res), flush=True)
        scene.close()


if __name__ == "__main__":
    main()
