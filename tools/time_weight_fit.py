"""What fitting the weight and exponent stops costs: rdc_render_weight_adjoint next to one frame of the same view, and one
evaluation of api.fit_weights' loop, unblurred and blurred.
    python tools/time_weight_fit.py

Views of the weight adjoint: those of the colour adjoint's table (DESIGN.md §3.5): arch.xml and lady_bug.xml at 1080p @128,
dolphin.xml at 4K @256, the 100 k-curve scene at 2048x2048 @64, whole scene in view, max_trace_depth 0. Device time (CUDA
events, L2 not flushed) of the adjoint with an image and a sigma gradient, next to one rdc_render, median of 5 after a
warm-up. Then fit_weights at 512x512, 128 rays per pixel, on lady_bug.xml from weights times a seeded factor in [0.5, 2] and
exponents + 0.3: host clock around each evaluation (update_stops + render [+ blur] + residual [+ blur adjoint + sigma
derivative] + weight adjoint, the gradient back on the host) over 20 iterations, median; with use_blur False and True.
Prints the card's name, power limit and clock first, then one line and one JSON line per measurement."""
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

from time_color_adjoint import ROOT, card, device_ms

sys.path.insert(0, ROOT)
from raytracingdiffusioncurves_b200 import api  # noqa: E402

XML = os.path.join(ROOT, "tests", "golden", "xmls")


def main():
    torch.cuda.init()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
    gen = torch.Generator("cuda").manual_seed(1)

    views = [("arch.xml", os.path.join(XML, "arch.xml"), 1920, 1080, 128),
             ("lady_bug.xml", os.path.join(XML, "DiffusionCurvePack", "lady_bug.xml"), 1920, 1080, 128),
             ("dolphin.xml", os.path.join(XML, "DiffusionCurvePack", "dolphin.xml"), 3840, 2160, 256),
             ("synth100k", api.synth_xml(100000, 8192, 8192), 2048, 2048, 64)]
    for name, src, w, h, n in views:
        host = api.HostScene.from_xml_text(src) if isinstance(src, bytes) else api.HostScene.from_xml_file(src)
        scene = api.Scene(host.arrays, None, stream)
        p = api.default_frame_params(w, h, n, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
        image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
        grad = torch.rand((h, w, 4), dtype=torch.float32, device="cuda", generator=gen) + 0.1
        grad_sigma = torch.rand((h, w), dtype=torch.float32, device="cuda", generator=gen) + 0.1
        gw = torch.empty((host.arrays.n_weight + 2,), dtype=torch.float64, device="cuda")
        ge = torch.empty((host.arrays.n_weight_degree + 2,), dtype=torch.float64, device="cuda")
        scene.reserve(p, False, stream)
        adj = device_ms(lambda: scene.weight_adjoint(p, grad.data_ptr(), grad_sigma.data_ptr(), gw.data_ptr(), ge.data_ptr(),
                                                     stream), 5)
        ren = device_ms(lambda: scene.render(p, image.data_ptr(), sigma.data_ptr(), stream), 5)
        res = {"scene": name, "width": w, "height": h, "rays_per_pixel": n, "weight_adjoint_ms": adj[0], "frame_ms": ren[0],
               "adjoint_over_frame": adj[0] / ren[0]}
        print(f"{name} {w}x{h} @{n}: weight adjoint {adj[0]:.2f} ms, frame {ren[0]:.2f} ms "
              f"= {res['adjoint_over_frame']:.2f} frames", flush=True)
        print(json.dumps(res), flush=True)
        scene.close()

    # fit_weights at 512x512 @128 on lady_bug.xml: the wall time of each evaluation of the objective and its gradient
    w = h = 512
    host = api.HostScene.from_xml_file(os.path.join(XML, "DiffusionCurvePack", "lady_bug.xml"))
    d = host.to_numpy()
    p = api.default_frame_params(w, h, 128, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
    rng = np.random.default_rng(11)
    start = dict(d)
    start["weight"] = d["weight"].copy()
    start["weight"][:d["n_weight"]] *= np.exp2(rng.uniform(-1.0, 1.0, d["n_weight"])).astype(np.float32)
    start["weight_degree"] = d["weight_degree"].copy()
    start["weight_degree"][:d["n_weight_degree"]] += np.float32(0.3)
    descent = api.projected_descent
    for use_blur in (False, True):
        scene = api.Scene(host.arrays, None, stream)
        target = np.empty((h, w, 4), np.float32)
        scene.render_frame_to_host(p, use_blur, target.ctypes.data, stream)
        times, iterations = [], []

        def timed(f_and_grad, x0, lower, n):
            def f(x):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = f_and_grad(x)
                times.append((time.perf_counter() - t0) * 1e3)
                return out
            x, objectives = descent(f, x0, lower, n)
            iterations.append(len(objectives) - 1)
            return x, objectives

        api.projected_descent = timed
        try:
            t0 = time.perf_counter()
            api.fit_weights(scene, start, p, target, iterations=20, use_blur=use_blur)
            total = (time.perf_counter() - t0) * 1e3
        finally:
            api.projected_descent = descent
        res = {"scene": "lady_bug.xml", "width": w, "height": h, "rays_per_pixel": 128, "use_blur": use_blur,
               "evaluation_ms": statistics.median(times[2:]), "evaluations": len(times), "iterations": iterations[0],
               "fit_ms": total}
        print(f"fit_weights lady_bug.xml {w}x{h} @128 use_blur={use_blur}: one evaluation {res['evaluation_ms']:.3f} ms "
              f"(median); {res['iterations']} iterations, {res['evaluations']} evaluations, {total:.1f} ms in all", flush=True)
        print(json.dumps(res), flush=True)
        scene.close()


if __name__ == "__main__":
    main()
