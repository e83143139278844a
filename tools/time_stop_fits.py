"""What fitting stops to an image costs: the three stop adjoints next to one frame of the same view, the blur, its transpose
and its sigma derivative on real sigma maps, and one iteration or evaluation of each fit's loop.
    python tools/time_stop_fits.py

1. Views (the zoom is the XML height over the frame height, as in bench.py; whole scene in view, max_trace_depth 0):
   arch.xml and lady_bug.xml at 1920x1080, 128 rays per pixel; dolphin.xml at 3840x2160, 256; the synthetic 100 k-curve
   scene of bench.py's config 5 at 2048x2048, 64. Per view: device time (CUDA events, L2 not flushed) of
   rdc_render_color_adjoint, rdc_render_blur_adjoint and rdc_render_weight_adjoint with gradients that are nonzero on every
   pixel (an image and a sigma gradient for the weights), next to one rdc_render, median of 5 launches after a warm-up.
2. Sigma maps: the blur map rdc_render writes for face.xml, lady_bug.xml and fille.xml at 1920x1080 (32 rays per pixel).
   Per map: device time of rdc_gaussian_blur, rdc_gaussian_blur_adjoint and rdc_gaussian_blur_sigma_adjoint on the whole
   frame, median of 20 after a warm-up.
3. Fits at 512x512, 128 rays per pixel, on lady_bug.xml, host clock:
   - colour: one iteration (update_stops + render + adjoint, the arrays back on the host, as fit_colors has them), median
     of 20 after 5; the same through api._color_operator, blurred (+ blur + blur adjoint) and unblurred;
   - fit_blur from half the blur: each evaluation (update_stops + render + blur + residual + sigma derivative + blur-value
     adjoint, the gradient back on the host) over 20 iterations, median;
   - fit_weights from weights times a seeded factor in [0.5, 2] and exponents + 0.3: each evaluation (update_stops +
     render [+ blur] + residual [+ blur adjoint + sigma derivative] + weight adjoint) over 20 iterations, median; with
     use_blur False and True.
Prints the card's name and power limit first, then one line and one JSON line per measurement; lines that would otherwise
look alike carry a "family" key."""
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
PACK = os.path.join(XML, "DiffusionCurvePack")
VIEWS = [("arch.xml", os.path.join(XML, "arch.xml"), 1920, 1080, 128),
         ("lady_bug.xml", os.path.join(PACK, "lady_bug.xml"), 1920, 1080, 128),
         ("dolphin.xml", os.path.join(PACK, "dolphin.xml"), 3840, 2160, 256),
         ("synth100k", None, 2048, 2048, 64)]


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


def report(text, res):
    print(text, flush=True)
    print(json.dumps(res), flush=True)


def seeded(shape, offset=0.0):
    return torch.rand(shape, dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(1)) + offset


def adjoints(stream):
    for name, path, w, h, n in VIEWS:
        host = api.HostScene.from_xml_file(path) if path else api.HostScene.from_xml_text(api.synth_xml(100000, 8192, 8192))
        d = host.to_numpy()
        scene = api.Scene(host.arrays, None, stream)
        p = api.default_frame_params(w, h, n, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
        image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
        grad, grad_sigma = seeded((h, w, 4), 0.1), seeded((h, w), 0.1)
        left = torch.empty(d["color_left"].shape, dtype=torch.float64, device="cuda")
        right = torch.empty(d["color_right"].shape, dtype=torch.float64, device="cuda")
        gb = torch.empty((host.arrays.n_blur + 2,), dtype=torch.float64, device="cuda")
        gw = torch.empty((host.arrays.n_weight + 2,), dtype=torch.float64, device="cuda")
        ge = torch.empty((host.arrays.n_weight_degree + 2,), dtype=torch.float64, device="cuda")
        scene.reserve(p, False, stream)
        ren = device_ms(lambda: scene.render(p, image.data_ptr(), sigma.data_ptr(), stream), 5)
        view = {"scene": name, "width": w, "height": h, "rays_per_pixel": n}
        calls = {"colour": lambda: scene.color_adjoint(p, grad.data_ptr(), left.data_ptr(), right.data_ptr(), stream),
                 "blur": lambda: scene.blur_adjoint(p, grad_sigma.data_ptr(), gb.data_ptr(), stream),
                 "weight": lambda: scene.weight_adjoint(p, grad.data_ptr(), grad_sigma.data_ptr(), gw.data_ptr(), ge.data_ptr(),
                                                        stream)}
        for family, call in calls.items():
            adj = device_ms(call, 5)
            if family == "colour":
                res = {**view, "chords": scene.stats.n_chords, "colour_stops": int(d["color_left"].shape[0]),
                       "adjoint_ms": adj[0], "adjoint_ms_min": adj[1], "render_ms": ren[0], "render_ms_min": ren[1],
                       "adjoint_over_render": adj[0] / ren[0]}
            else:
                res = {**view, f"{family}_adjoint_ms": adj[0], "frame_ms": ren[0], "adjoint_over_frame": adj[0] / ren[0]}
            res["family"] = family
            report(f"{name} {w}x{h} @{n}: {family} adjoint {adj[0]:.3f} ms (min {adj[1]:.3f}), frame {ren[0]:.3f} ms "
                   f"(min {ren[1]:.3f}) = {adj[0] / ren[0]:.2f} frames", res)
        scene.close()


def blur_maps(stream):
    w, h = 1920, 1080
    for name in ("face.xml", "lady_bug.xml", "fille.xml"):
        host = api.HostScene.from_xml_file(os.path.join(PACK, name))
        scene = api.Scene(host.arrays, None, stream)
        flag = torch.zeros((1,), dtype=torch.float32, device="cuda")
        p = api.default_frame_params(w, h, 32, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
        p.max_sigma = flag.data_ptr()
        image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
        scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)
        dest, out, grad = torch.empty_like(image), torch.empty_like(image), seeded((h, w, 4))
        grad_sigma = torch.empty_like(sigma)
        scratch = torch.empty((2 * h * w + 1, 4), dtype=torch.float32, device="cuda")
        band = (w, h, 0, h, flag.data_ptr(), stream)
        fwd = device_ms(lambda: api.gaussian_blur(dest.data_ptr(), image.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), *band),
                        20)
        adj = device_ms(lambda: api.gaussian_blur_adjoint(out.data_ptr(), grad.data_ptr(), sigma.data_ptr(), scratch.data_ptr(),
                                                          *band), 20)
        sig = device_ms(lambda: api.gaussian_blur_sigma_adjoint(grad_sigma.data_ptr(), grad.data_ptr(), image.data_ptr(),
                                                                sigma.data_ptr(), scratch.data_ptr(), *band), 20)
        finite = sigma[torch.isfinite(sigma)]
        res = {"scene": name, "width": w, "height": h, "max_sigma": float(flag.item()), "mean_sigma": float(finite.mean()),
               "reach_rows": int(np.ceil(3 * float(flag.item()))), "blur_ms": fwd[0], "blur_ms_min": fwd[1],
               "adjoint_ms": adj[0], "adjoint_ms_min": adj[1], "adjoint_over_blur": adj[0] / fwd[0],
               "sigma_adjoint_ms": sig[0], "sigma_adjoint_ms_min": sig[1], "sigma_adjoint_over_blur": sig[0] / fwd[0]}
        report(f"{name} {w}x{h}: max sigma {res['max_sigma']:.2f} (mean {res['mean_sigma']:.2f}); blur {fwd[0]:.3f} ms "
               f"(min {fwd[1]:.3f}), adjoint {adj[0]:.3f} ms (min {adj[1]:.3f}) = {res['adjoint_over_blur']:.2f} blurs, "
               f"sigma adjoint {sig[0]:.3f} ms (min {sig[1]:.3f}) = {res['sigma_adjoint_over_blur']:.2f} blurs", res)
        scene.close()


def timed_fit(fit):
    """fit() with api.projected_descent timing each evaluation: (evaluation times in ms, iterations, total ms)"""
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
        fit()
        total = (time.perf_counter() - t0) * 1e3
    finally:
        api.projected_descent = descent
    return times, iterations[0], total


def fits(stream):
    w = h = 512
    host = api.HostScene.from_xml_file(os.path.join(PACK, "lady_bug.xml"))
    d = host.to_numpy()
    p = api.default_frame_params(w, h, 128, zoom_factor=host.arrays.image_height / h, max_trace_depth=0)
    view = {"scene": "lady_bug.xml", "width": w, "height": h, "rays_per_pixel": 128}

    # colour: one iteration of the fit loop, by hand and through the operator fit_colors uses
    scene = api.Scene(host.arrays, None, stream)
    image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
    sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
    grad = seeded((h, w, 4), 0.1)
    left = torch.empty(d["color_left"].shape, dtype=torch.float64, device="cuda")
    right = torch.empty(d["color_right"].shape, dtype=torch.float64, device="cuda")
    scene.reserve(p, False, stream)
    work = dict(d)

    def by_hand(cl, cr):
        work["color_left"], work["color_right"] = cl, cr
        scene.update_stops(api.arrays_from_numpy(work), stream)
        scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)
        scene.color_adjoint(p, grad.data_ptr(), left.data_ptr(), right.data_ptr(), stream)
        left.cpu(), right.cpu()

    grad_op = seeded((h, w, 4))
    for use_blur in (None, True, False):  # None: by hand
        if use_blur is None:
            step = by_hand
        else:
            render, adjoint = api._color_operator(scene, d, p, use_blur, stream)
            step = lambda cl, cr: (render(cl, cr), adjoint(grad_op))  # noqa: E731
        rng = np.random.default_rng(0)
        times = []
        for i in range(25):
            cl = rng.random(d["color_left"].shape).astype(np.float32)
            cr = rng.random(d["color_right"].shape).astype(np.float32)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step(cl, cr)
            if i >= 5:
                times.append((time.perf_counter() - t0) * 1e3)
        res = {"family": "colour", **view, "fit_iteration_ms": statistics.median(times), "fit_iteration_ms_min": min(times)}
        if use_blur is not None:
            res["use_blur"] = use_blur
        report(f"colour fit iteration lady_bug.xml {w}x{h} @128{'' if use_blur is None else f', use_blur={use_blur}'}: "
               f"{res['fit_iteration_ms']:.3f} ms (min {res['fit_iteration_ms_min']:.3f})", res)
    scene.close()

    def fit_line(family, use_blur, fit):
        times, iterations, total = timed_fit(fit)
        res = {"family": family, **view, "evaluation_ms": statistics.median(times[2:]), "evaluations": len(times),
               "iterations": iterations, "fit_ms": total}
        if use_blur is not None:
            res["use_blur"] = use_blur
        report(f"fit_{family} lady_bug.xml {w}x{h} @128{'' if use_blur is None else f' use_blur={use_blur}'}: one evaluation "
               f"{res['evaluation_ms']:.3f} ms (median); {iterations} iterations, {len(times)} evaluations, {total:.1f} ms in all",
               res)

    # fit_blur from half the blur, and fit_weights from perturbed weights and exponents (unblurred and blurred), each on a
    # fresh handle, to the frame of the scene's own stops
    target = np.empty((h, w, 4), np.float32)
    scene = api.Scene(host.arrays, None, stream)
    scene.render_frame_to_host(p, True, target.ctypes.data, stream)
    start = dict(d)
    start["blur"] = d["blur"] * np.float32(0.5)
    fit_line("blur", None, lambda: api.fit_blur(scene, start, p, target, iterations=20))
    scene.close()
    rng = np.random.default_rng(11)
    start = dict(d)
    start["weight"] = d["weight"].copy()
    start["weight"][:d["n_weight"]] *= np.exp2(rng.uniform(-1.0, 1.0, d["n_weight"])).astype(np.float32)
    start["weight_degree"] = d["weight_degree"].copy()
    start["weight_degree"][:d["n_weight_degree"]] += np.float32(0.3)
    for use_blur in (False, True):
        scene = api.Scene(host.arrays, None, stream)
        scene.render_frame_to_host(p, use_blur, target.ctypes.data, stream)
        fit_line("weights", use_blur, lambda: api.fit_weights(scene, start, p, target, iterations=20, use_blur=use_blur))
        scene.close()


def main():
    torch.cuda.init()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
    adjoints(stream)
    blur_maps(stream)
    fits(stream)


if __name__ == "__main__":
    main()
