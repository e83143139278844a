"""What fitting the blur stops costs: rdc_gaussian_blur_sigma_adjoint next to the forward blur and the blur's transpose on
real sigma maps, rdc_render_blur_adjoint next to one frame of the same view, and one evaluation of api.fit_blur's loop.
    python tools/time_blur_fit.py

Sigma maps: the blur map rdc_render writes for face.xml, lady_bug.xml and fille.xml at 1920x1080 (whole scene in view, 32 rays
per pixel, max_trace_depth 0). Per map: device time (CUDA events, L2 not flushed) of the forward blur, its transpose and its
sigma derivative on the whole frame, median of 20 after a warm-up. Views of the blur-value adjoint: those of the colour
adjoint's table (DESIGN.md §3.5), median of 5. Then fit_blur at 512x512, 128 rays per pixel, on lady_bug.xml: host clock
around each evaluation (update_stops + render + blur + residual + sigma derivative + blur-value adjoint, the gradient back on
the host) over 20 iterations, median. Prints the card's name and power limit first, then one line and one JSON line per
measurement."""
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

    w, h = 1920, 1080
    for name in ("face.xml", "lady_bug.xml", "fille.xml"):
        host = api.HostScene.from_xml_file(os.path.join(XML, "DiffusionCurvePack", name))
        scene = api.Scene(host.arrays, None, stream)
        flag = torch.zeros((1,), dtype=torch.float32, device="cuda")
        p = api.default_frame_params(w, h, 32, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
        p.max_sigma = flag.data_ptr()
        image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
        scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)
        dest = torch.empty_like(image)
        grad = torch.rand((h, w, 4), dtype=torch.float32, device="cuda", generator=gen)
        out = torch.empty_like(image)
        grad_sigma = torch.empty_like(sigma)
        scratch = torch.empty((2 * h * w + 1, 4), dtype=torch.float32, device="cuda")
        fwd = device_ms(lambda: api.gaussian_blur(dest.data_ptr(), image.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, h,
                                                  0, h, flag.data_ptr(), stream), 20)
        adj = device_ms(lambda: api.gaussian_blur_adjoint(out.data_ptr(), grad.data_ptr(), sigma.data_ptr(), scratch.data_ptr(),
                                                          w, h, 0, h, flag.data_ptr(), stream), 20)
        sig = device_ms(lambda: api.gaussian_blur_sigma_adjoint(grad_sigma.data_ptr(), grad.data_ptr(), image.data_ptr(),
                                                                sigma.data_ptr(), scratch.data_ptr(), w, h, 0, h, flag.data_ptr(),
                                                                stream), 20)
        res = {"scene": name, "width": w, "height": h, "max_sigma": float(flag.item()),
               "blur_ms": fwd[0], "blur_adjoint_ms": adj[0], "sigma_adjoint_ms": sig[0], "sigma_adjoint_ms_min": sig[1],
               "sigma_adjoint_over_blur": sig[0] / fwd[0]}
        print(f"{name} {w}x{h}: max sigma {res['max_sigma']:.2f}; blur {fwd[0]:.3f} ms, blur adjoint {adj[0]:.3f} ms, "
              f"sigma adjoint {sig[0]:.3f} ms (min {sig[1]:.3f}) = {res['sigma_adjoint_over_blur']:.2f} blurs", flush=True)
        print(json.dumps(res), flush=True)
        scene.close()

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
        grad = torch.rand((h, w), dtype=torch.float32, device="cuda", generator=gen) + 0.1
        out = torch.empty((host.arrays.n_blur + 2,), dtype=torch.float64, device="cuda")
        scene.reserve(p, False, stream)
        adj = device_ms(lambda: scene.blur_adjoint(p, grad.data_ptr(), out.data_ptr(), stream), 5)
        ren = device_ms(lambda: scene.render(p, image.data_ptr(), sigma.data_ptr(), stream), 5)
        res = {"scene": name, "width": w, "height": h, "rays_per_pixel": n, "blur_adjoint_ms": adj[0], "frame_ms": ren[0],
               "adjoint_over_frame": adj[0] / ren[0]}
        print(f"{name} {w}x{h} @{n}: blur-value adjoint {adj[0]:.2f} ms, frame {ren[0]:.2f} ms "
              f"= {res['adjoint_over_frame']:.2f} frames", flush=True)
        print(json.dumps(res), flush=True)
        scene.close()

    # fit_blur at 512x512 @128 on lady_bug.xml: the wall time of each evaluation of the objective and its gradient
    w = h = 512
    host = api.HostScene.from_xml_file(os.path.join(XML, "DiffusionCurvePack", "lady_bug.xml"))
    d = host.to_numpy()
    scene = api.Scene(host.arrays, None, stream)
    p = api.default_frame_params(w, h, 128, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
    target = np.empty((h, w, 4), np.float32)
    scene.render_frame_to_host(p, True, target.ctypes.data, stream)
    start = dict(d)
    start["blur"] = d["blur"] * np.float32(0.5)
    times, iterations = [], []
    descent = api.projected_descent

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
        api.fit_blur(scene, start, p, target, iterations=20)
        total = (time.perf_counter() - t0) * 1e3
    finally:
        api.projected_descent = descent
    res = {"scene": "lady_bug.xml", "width": w, "height": h, "rays_per_pixel": 128, "evaluation_ms": statistics.median(times[2:]),
           "evaluations": len(times), "iterations": iterations[0], "fit_ms": total}
    print(f"fit_blur lady_bug.xml {w}x{h} @128: one evaluation {res['evaluation_ms']:.3f} ms (median); "
          f"{res['iterations']} iterations, {res['evaluations']} evaluations, {total:.1f} ms in all", flush=True)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
