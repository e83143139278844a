"""What the blur's transpose costs: rdc_gaussian_blur_adjoint next to the forward rdc_gaussian_blur on real sigma maps, and
one iteration of api.fit_colors(use_blur=True)'s loop.
    python tools/time_blur_adjoint.py

Sigma maps: the blur map rdc_render writes for face.xml, lady_bug.xml and fille.xml at 1920x1080 (whole scene in view, as in
bench.py; 32 rays per pixel, max_trace_depth 0). Per map: device time (CUDA events, L2 not flushed) of the forward blur and
of its transpose on the whole frame, median of 20 after a warm-up. Then a fit iteration at 512x512, 128 rays per pixel, on
lady_bug.xml: host clock around update_stops + render + blur + blur adjoint + colour adjoint (the arrays back on the host,
as fit_colors has them), median of 20, and the same iteration without the blur. Prints the card's name and power limit
first, then one line and one JSON line per measurement."""
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

XML = os.path.join(ROOT, "tests", "golden", "xmls", "DiffusionCurvePack")


def scene_for(name, w, h, n, stream):
    host = api.HostScene.from_xml_file(os.path.join(XML, name))
    scene = api.Scene(host.arrays, None, stream)
    p = api.default_frame_params(w, h, n, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
    return host, scene, p


def main():
    torch.cuda.init()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
    w, h = 1920, 1080
    for name in ("face.xml", "lady_bug.xml", "fille.xml"):
        host, scene, p = scene_for(name, w, h, 32, stream)
        flag = torch.zeros((1,), dtype=torch.float32, device="cuda")
        p.max_sigma = flag.data_ptr()
        image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
        scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)
        dest = torch.empty_like(image)
        grad = torch.rand((h, w, 4), dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
        out = torch.empty_like(image)
        scratch = torch.empty((h * w + 1, 4), dtype=torch.float32, device="cuda")
        fwd = device_ms(lambda: api.gaussian_blur(dest.data_ptr(), image.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, h,
                                                  0, h, flag.data_ptr(), stream), 20)
        adj = device_ms(lambda: api.gaussian_blur_adjoint(out.data_ptr(), grad.data_ptr(), sigma.data_ptr(), scratch.data_ptr(),
                                                          w, h, 0, h, flag.data_ptr(), stream), 20)
        finite = sigma[torch.isfinite(sigma)]
        res = {"scene": name, "width": w, "height": h, "max_sigma": float(flag.item()),
               "mean_sigma": float(finite.mean()), "reach_rows": int(np.ceil(3 * float(flag.item()))),
               "blur_ms": fwd[0], "blur_ms_min": fwd[1], "adjoint_ms": adj[0], "adjoint_ms_min": adj[1],
               "adjoint_over_blur": adj[0] / fwd[0]}
        print(f"{name} {w}x{h}: max sigma {res['max_sigma']:.2f} (mean {res['mean_sigma']:.2f}); blur {fwd[0]:.3f} ms "
              f"(min {fwd[1]:.3f}), adjoint {adj[0]:.3f} ms (min {adj[1]:.3f}); adjoint = {res['adjoint_over_blur']:.2f} blurs",
              flush=True)
        print(json.dumps(res), flush=True)
        scene.close()

    # one iteration of the blurred fit loop at 512x512 on lady_bug.xml, and the unblurred one for comparison
    w = h = 512
    host, scene, p = scene_for("lady_bug.xml", w, h, 128, stream)
    d = host.to_numpy()
    rng = np.random.default_rng(0)
    grad = torch.rand((h, w, 4), dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    for use_blur in (True, False):
        render, adjoint = api._color_operator(scene, d, p, use_blur, stream)
        times = []
        for i in range(25):
            left = rng.random(d["color_left"].shape).astype(np.float32)
            right = rng.random(d["color_right"].shape).astype(np.float32)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            render(left, right)
            adjoint(grad)
            if i >= 5:
                times.append((time.perf_counter() - t0) * 1e3)
        res = {"scene": "lady_bug.xml", "width": w, "height": h, "rays_per_pixel": 128, "use_blur": use_blur,
               "fit_iteration_ms": statistics.median(times), "fit_iteration_ms_min": min(times)}
        print(f"fit iteration lady_bug.xml {w}x{h} @128, use_blur={use_blur}: {res['fit_iteration_ms']:.3f} ms "
              f"(min {res['fit_iteration_ms_min']:.3f})", flush=True)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
