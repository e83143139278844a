"""What the colour adjoint costs: rdc_render_color_adjoint (A^T of the frame in the colour stops) next to one rdc_render of
the same view, and the wall time of one iteration of api.fit_colors' loop (update_stops, render, adjoint).
    python tools/time_color_adjoint.py

Views (the zoom is the XML height over the frame height, as in bench.py; max_trace_depth 0):
  - arch.xml and lady_bug.xml at 1920x1080, 128 rays per pixel; dolphin.xml at 3840x2160, 256; the synthetic 100 k-curve
    scene of bench.py's config 5 at 2048x2048, 64.
Per view: device time (CUDA events, L2 not flushed) of the adjoint with a gradient that is nonzero on every pixel and of
one frame, median of 5 launches after a warm-up. Then a fit iteration at 512x512, 128 rays per pixel, on lady_bug.xml: host
clock around update_stops + render + adjoint (the arrays back on the host, as fit_colors has them), median of 20.
Prints the card's name and power limit first, then one line and one JSON line per measurement."""
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from raytracingdiffusioncurves_b200 import api  # noqa: E402

XML = os.path.join(ROOT, "tests", "golden", "xmls")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()


def device_ms(fn, reps, warm=2):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warm):
        fn()
    times = []
    for _ in range(reps):
        start.record()
        fn()
        stop.record()
        torch.cuda.synchronize()
        times.append(start.elapsed_time(stop))
    return statistics.median(times), min(times)


def buffers(d, h, w):
    image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
    grad = torch.rand((h, w, 4), dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(1)) + 0.1
    left = torch.empty(d["color_left"].shape, dtype=torch.float64, device="cuda")
    right = torch.empty(d["color_right"].shape, dtype=torch.float64, device="cuda")
    return image, sigma, grad, left, right


def main():
    torch.cuda.init()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
    views = [("arch.xml", os.path.join(XML, "arch.xml"), 1920, 1080, 128),
             ("lady_bug.xml", os.path.join(XML, "DiffusionCurvePack", "lady_bug.xml"), 1920, 1080, 128),
             ("dolphin.xml", os.path.join(XML, "DiffusionCurvePack", "dolphin.xml"), 3840, 2160, 256),
             ("synth100k", api.synth_xml(100000, 8192, 8192), 2048, 2048, 64)]
    for name, src, w, h, n in views:
        host = api.HostScene.from_xml_text(src) if isinstance(src, bytes) else api.HostScene.from_xml_file(src)
        d = host.to_numpy()
        scene = api.Scene(host.arrays, None, stream)
        p = api.default_frame_params(w, h, n, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
        image, sigma, grad, left, right = buffers(d, h, w)
        scene.reserve(p, False, stream)
        adj = device_ms(lambda: scene.color_adjoint(p, grad.data_ptr(), left.data_ptr(), right.data_ptr(), stream), 5)
        ren = device_ms(lambda: scene.render(p, image.data_ptr(), sigma.data_ptr(), stream), 5)
        res = {"scene": name, "width": w, "height": h, "rays_per_pixel": n, "chords": scene.stats.n_chords,
               "colour_stops": int(d["color_left"].shape[0]), "adjoint_ms": adj[0], "adjoint_ms_min": adj[1],
               "render_ms": ren[0], "render_ms_min": ren[1], "adjoint_over_render": adj[0] / ren[0]}
        print(f"{name} {w}x{h} @{n}: adjoint {adj[0]:.3f} ms (min {adj[1]:.3f}), render {ren[0]:.3f} ms (min {ren[1]:.3f}); "
              f"adjoint = {res['adjoint_over_render']:.2f} frames", flush=True)
        print(json.dumps(res), flush=True)
        scene.close()

    # one iteration of the fit loop at 512x512 on lady_bug.xml
    host = api.HostScene.from_xml_file(os.path.join(XML, "DiffusionCurvePack", "lady_bug.xml"))
    d = host.to_numpy()
    scene = api.Scene(host.arrays, None, stream)
    w = h = 512
    p = api.default_frame_params(w, h, 128, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
    image, sigma, grad, left, right = buffers(d, h, w)
    scene.reserve(p, False, stream)
    rng = np.random.default_rng(0)
    work = dict(d)
    times = []
    for i in range(25):
        work["color_left"] = rng.random(d["color_left"].shape).astype(np.float32)
        work["color_right"] = rng.random(d["color_right"].shape).astype(np.float32)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        scene.update_stops(api.arrays_from_numpy(work), stream)
        scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)
        scene.color_adjoint(p, grad.data_ptr(), left.data_ptr(), right.data_ptr(), stream)
        left.cpu(), right.cpu()
        if i >= 5:
            times.append((time.perf_counter() - t0) * 1e3)
    res = {"scene": "lady_bug.xml", "width": w, "height": h, "rays_per_pixel": 128, "fit_iteration_ms": statistics.median(times),
           "fit_iteration_ms_min": min(times)}
    print(f"fit iteration lady_bug.xml {w}x{h} @128: {res['fit_iteration_ms']:.3f} ms (min {res['fit_iteration_ms_min']:.3f})",
          flush=True)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
