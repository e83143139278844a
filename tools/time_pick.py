"""What picking costs: rdc_scene_pick_frame (one nearest-chord query per pixel) next to one rdc_render of the same view,
and the host-to-result latency of a single click (rdc_scene_pick with n = 1).
    python tools/time_pick.py

Views (the zoom is the XML height over the frame height, as in bench.py):
  - arch.xml at 1920x1080 (the headline view), lady_bug.xml at 1920x1080, dolphin.xml at 3840x2160,
    the synthetic 100 k-curve scene of bench.py's config 5 at 2048x2048.
Per view: device time (CUDA events, L2 not flushed: the tree stays resident as it does in an editor's frame loop) of
pick_frame without and with the stop values, median of 20 launches after a warm-up, and of one 128-rays-per-pixel frame,
median of 5. Then per scene: a single-point pick, host clock from the call to the end of an event synchronise, median of
200 (points and result buffers are on the device already, as an editor would keep them).
Prints the card's name and power limit first, then one line and one JSON line per view."""
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from raytracingdiffusioncurves_b200 import api  # noqa: E402

XML = os.path.join(ROOT, "tests", "golden", "xmls")
INF = float("inf")


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


def main():
    torch.cuda.init()
    stream = torch.cuda.current_stream().cuda_stream
    print(f"card: {card()}  (name, power limit, max SM clock)", flush=True)
    views = [("arch.xml", os.path.join(XML, "arch.xml"), 1920, 1080),
             ("lady_bug.xml", os.path.join(XML, "DiffusionCurvePack", "lady_bug.xml"), 1920, 1080),
             ("dolphin.xml", os.path.join(XML, "DiffusionCurvePack", "dolphin.xml"), 3840, 2160),
             ("synth100k", api.synth_xml(100000, 8192, 8192), 2048, 2048)]
    for name, src, w, h in views:
        host = api.HostScene.from_xml_text(src) if isinstance(src, bytes) else api.HostScene.from_xml_file(src)
        scene = api.Scene(host.arrays, None, stream)
        p = api.default_frame_params(w, h, 128, zoom_factor=host.arrays.image_height / h, max_trace_depth=2)
        out = torch.empty((h * w, 32), dtype=torch.uint8, device="cuda")
        stops = torch.empty((h * w, 3, 4), dtype=torch.float32, device="cuda")
        pick_ms = device_ms(lambda: scene.pick_frame(p, out.data_ptr(), 0, INF, stream), 20)
        stops_ms = device_ms(lambda: scene.pick_frame(p, out.data_ptr(), stops.data_ptr(), INF, stream), 20)
        image = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
        sigma = torch.empty((h, w), dtype=torch.float32, device="cuda")
        scene.reserve(p, False, stream)
        render_ms = device_ms(lambda: scene.render(p, image.data_ptr(), sigma.data_ptr(), stream), 5)

        # one click: the pixel under the cursor, mapped on the host, picked on the device, result awaited
        x, y = api.view_pixel_to_scene(p, w // 2, h // 2)
        pt = torch.tensor([[x, y]], dtype=torch.float32, device="cuda")
        one = torch.empty((1, 32), dtype=torch.uint8, device="cuda")
        done = torch.cuda.Event()
        torch.cuda.synchronize()
        lat = []
        for i in range(220):
            t0 = time.perf_counter()
            scene.pick(pt.data_ptr(), 1, one.data_ptr(), 0, INF, 1, stream)
            done.record()
            done.synchronize()
            if i >= 20:
                lat.append((time.perf_counter() - t0) * 1e3)
        res = {"scene": name, "width": w, "height": h, "chords": scene.stats.n_chords, "runs": scene.stats.n_runs,
               "pick_frame_ms": pick_ms[0], "pick_frame_ms_min": pick_ms[1],
               "pick_frame_stops_ms": stops_ms[0], "pick_frame_stops_ms_min": stops_ms[1],
               "render_128rpp_ms": render_ms[0], "pick_over_render": pick_ms[0] / render_ms[0],
               "single_pick_latency_ms": statistics.median(lat), "single_pick_latency_ms_p90": sorted(lat)[int(0.9 * len(lat))]}
        print(f"{name} {w}x{h}: {res['chords']} chords; pick_frame {res['pick_frame_ms']:.3f} ms, with stops "
              f"{res['pick_frame_stops_ms']:.3f} ms; render @128 {res['render_128rpp_ms']:.3f} ms "
              f"(pick = {100 * res['pick_over_render']:.1f} % of a frame); one click {res['single_pick_latency_ms']:.3f} ms",
              flush=True)
        print(json.dumps(res), flush=True)
        scene.close()


if __name__ == "__main__":
    main()
