#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native diffusion-curve ray tracer.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one frame of the hot path: ray generation + closest-hit traversal + shading + normalisation
(`rdc_render`) followed by the variable-sigma blur (`rdc_gaussian_blur`), on BASELINE.json's configs[1]:
xmls/arch.xml at 1920x1080, 128 rays per pixel, Orzan flag / blur / per-ray jitter as shipped, denoiser
off. The metric is Grays/s = primary rays per second (W*H*rpp / t_frame / 1e9), whole job.

N > 1: the image is dealt out in 8-row strips, round-robin over the ranks (scene + tree replicated). All of it runs
through the C ABI (csrc/peer.cu; torch.distributed only carries the CUDA IPC handles at set-up, the timing reductions and
host barriers). `value`: the frame reaches rank 0's device through peer memory — the render kernel of every rank stores
its finished pixels straight into rank 0's frame over NVLink, then one barrier kernel; scenes with blur store the rendered
frame into every rank's buffer, every rank blurs one contiguous band and the blur stores it into rank 0's frame
(rdc_peer_render_frame). `e2e`: host consumer — every rank copies its own rows of the finished frame over its own PCIe link
into one pinned host frame shared by all ranks (rdc_peer_frame_to_host). Total work is fixed as N grows ("strong" scaling);
every exchange is inside the timed region. After the headline measurement the same run renders a few frames of
BASELINE.json configs[4] (8192x8192 @512, 100 k synthetic curves) at the same N and reports them under "secondary".

Prints ONE JSON line (rank 0). Nothing here reads /root/reference.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene, width, height, rays per pixel, max trace depth)
    "arch_1080p_128rpp": ("xml:arch.xml", 1920, 1080, 128, 2),            # BASELINE.json configs[1] (headline)
    "arch_512_128rpp": ("xml:arch.xml", 512, 512, 128, 2),                # configs[0]
    "portal_1080p_depth31": ("xml:PortalDemo.xml", 1920, 1080, 128, 31),  # configs[3]
    "ladybug_1080p_128rpp": ("xml:DiffusionCurvePack/lady_bug.xml", 1920, 1080, 128, 2),   # dense bundled scene
    "dolphin_4k_256rpp": ("xml:DiffusionCurvePack/dolphin.xml", 3840, 2160, 256, 2),        # configs[2], largest bundled scene
    "synth100k_8k_512rpp": ("synth:100000:8192", 8192, 8192, 512, 2),     # configs[4]
    "synth100k_2k_64rpp": ("synth:100000:8192", 2048, 2048, 64, 2),       # configs[4] geometry, smaller frame
}
DEFAULT_WORKLOAD = "arch_1080p_128rpp"
XML_DIR = os.path.join(ROOT, "tests", "golden", "xmls")

# SURVEY.md §8(d): algorithmic work per ray, FMA = 2 flops
F_GEN, F_NODE, F_SEG, F_SHADE, F_ACC = 40.0, 30.0, 20.0, 100.0, 10.0

# From the committed `ncu --set full` capture of k_render on the headline workload
# (profiles/r01c_k_render_arch_ncu_summary.txt): DRAM bytes per launch and issue-slot utilisation.
NCU_CAPTURE = {
    # DRAM bytes: ncu pass with the partial sums' lines discarded after use (the shipped default), profiles/r01c_discard_partials.log;
    # before that the same launch wrote 155 MB (profiles/r01c_k_render_arch_ncu_summary.txt, which also holds the issue-slot figure)
    "arch_1080p_128rpp": {"dram_bytes": 3.64e6 + 30.32e6, "issue_active": 0.8130, "source": "profiles/r01c_discard_partials.log, profiles/r01c_k_render_arch_ncu_summary.txt"},
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-secondary", dest="secondary", action="store_false",
                    help="skip the config-5 block (8192x8192 @512 synthetic scene) that follows the headline measurement")
    ap.add_argument("--secondary-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="b200 arm only: after the timed steps, write the finished frame of the last timed step to DIR/frame.npy "
                         "(float32 RGBA; frames over 64 MB: a seeded sample of rows, their indices in DIR/frame_rows.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computed")
    return args


def workload_zoom(spec, height):
    """zoom = xml image height / output height (SURVEY.md Appendix E), without needing the product library."""
    kind, _, rest = spec.partition(":")
    if kind == "synth":
        return float(rest.split(":")[1]) / height
    import re

    with open(os.path.join(XML_DIR, rest), "rb") as fh:
        head = fh.read(4096).decode("utf-8", "replace")
    return float(re.search(r'image_height="(\d+)"', head).group(1)) / height


def scene_source(spec):
    """Returns (kind, payload): ('file', path) or ('text', xml bytes)."""
    kind, _, rest = spec.partition(":")
    if kind == "xml":
        return "file", os.path.join(XML_DIR, rest)
    n, size = rest.split(":")
    from raytracingdiffusioncurves_b200 import api

    return "text", api.synth_xml(int(n), int(size), int(size))


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def workload_config(name, n_gpus):
    """What both arms print under "config": the workload, nothing that varies from run to run."""
    spec, width, height, rpp, depth = WORKLOADS[name]
    return {"workload": name, "scene": spec, "width": width, "height": height, "rays_per_pixel": rpp, "blur": True, "aa": True,
            "orzan": True, "max_trace_depth": depth, "zoom": workload_zoom(spec, height),
            "parallelism": "single GPU" if n_gpus == 1 else f"{RDC_STRIP_ROWS}-row strips dealt round-robin over {n_gpus} GPUs, frame on rank 0",
            "l2": "flushed between timed steps (256 MiB write)"}


RDC_STRIP_ROWS = 8  # include/rdc_b200.h


def host_threads():
    """Host threads the CPU arm may use: the process's affinity mask, NOT OMP_NUM_THREADS (torchrun exports
    OMP_NUM_THREADS=1 to every rank, which would put the CPU arm on one core and inflate every N > 1 ratio)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_oracle_run(kind_pref, scene_spec, width, height, rpp, depth, zoom, target_seconds, whole_frame=False):
    """Times the CPU implementation on a bounded band of the workload (or the whole frame). Returns the cpu_baseline dict."""
    from oracle import pyoracle as po

    kind = kind_pref if (kind_pref == "port" or po.Oracle.reference_available()) else "port"
    if kind == "reference" and depth != 2:  # noqa
        kind = "port"  # the reference build is compiled with MAX_TRACE_DEPTH 2
    oracle = po.Oracle(kind)
    skind, payload = scene_source(scene_spec)
    if skind == "text":
        path = "/tmp/rdc_bench_synth.xml"
        with open(path, "wb") as fh:
            fh.write(payload)
    else:
        path = payload
    scene = po.ingest_xml(path, True)
    mid = height // 2

    def run(rows):
        b = max(0, mid - rows // 2)
        p = po.make_params(width, height, rpp, zoom_factor=zoom, max_trace_depth=depth, row_begin=b, row_end=min(height, b + rows))
        t0 = time.perf_counter()
        oracle.render(scene, p, threads=threads)
        return time.perf_counter() - t0, (p.row_end - p.row_begin)

    threads = host_threads()
    if whole_frame:
        t, rows = run(height)
    else:
        t_probe, rows_probe = run(max(threads, 8))
        rows = int(max(rows_probe, min(height, rows_probe * target_seconds / max(t_probe, 1e-6))))
        t, rows = run(rows)
    rays = float(rows) * width * rpp
    return {
        "value": rays / t / 1e9, "unit": "Grays/s", "cores": threads,
        "kind": "reference" if kind == "reference" else "port",
        "sample": f"{rows} centre rows of the {width}x{height}@{rpp} frame ({rays / 1e6:.1f} M rays, {t:.1f} s), render only, "
                  + ("reference DeviceCode.cu compiled for the host (oracle/_ref)" if kind == "reference"
                     else "restated oracle (oracle/oracle_port.cpp)") + ", brute-force closest hit, OpenMP",
        "ms_per_frame_extrapolated": t / rows * height * 1e3,
    }


def run_reference(args):
    """--impl reference: the reference's own CPU-runnable implementation of the path, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec, width, height, rpp, depth = WORKLOADS[args.workload]
    zoom = workload_zoom(spec, height)
    # a step is one whole frame while that keeps the run within a few minutes (the headline frame takes ~4 s on 16 threads);
    # for the heavier workloads each step is a band of the frame sized from a probe
    per_step_seconds = max(1.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    probe = cpu_oracle_run("reference", spec, width, height, rpp, depth, zoom, 1.0)
    whole = probe["ms_per_frame_extrapolated"] * 1e-3 * (args.steps + args.warmup) <= 240.0
    results = []
    for i in range(args.warmup + args.steps):
        r = cpu_oracle_run("reference", spec, width, height, rpp, depth, zoom, per_step_seconds, whole_frame=whole)
        if i >= args.warmup:
            results.append(r)
    value = sum(r["value"] for r in results) / len(results)
    base = results[-1]
    base["value"] = value
    line = {
        "impl": "reference", "metric": "Grays/s", "value": value, "unit": "Grays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(width) * height * rpp / (value * 1e9) * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "bundled scene file" if spec.startswith("xml:") else "synthetic",
        "config": workload_config(args.workload, args.gpus),
        "details": {"step": "one whole frame on the host cores" if whole else
                    "a bounded band of the frame on the host cores; ms_per_step is the extrapolated full frame",
                    "threads_from": "os.sched_getaffinity (OMP_NUM_THREADS is ignored: torchrun sets it to 1)"},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "Grays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def source_sha16():
    """Hash of the CODE the shipped library is built from (comments and white space stripped: editing a comment does not make a
    profile stale); profiles/r02_ncu_k_render.json records the one its captures were taken with."""
    import hashlib
    import re

    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "raytracingdiffusioncurves_b200", "csrc")
    for f in sorted(os.listdir(csrc)) + ["../../include/rdc_b200.h", "../../include/params.h", "../../Makefile"]:
        path = os.path.join(csrc, f)
        if os.path.isfile(path) and f.endswith((".cu", ".cpp", ".h", "Makefile")):
            text = open(path, "r", errors="replace").read()
            if not f.endswith("Makefile"):
                text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)       # block comments
                text = re.sub(r"(?m)(?<![:\"'])//[^\n]*$", " ", text)    # line comments (not the // of a URL or inside a string start)
            h.update(" ".join(text.split()).encode())
    return h.hexdigest()[:16]


def ncu_capture(workload):
    """Per-launch DRAM bytes and issue-slot utilisation of k_render from the committed ncu capture of the SHIPPED build
    (profiles/r02_ncu_k_render.json, written by tools/ncu_to_json.py from an .ncu-rep; never a constant in this file)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_k_render.json")) as fh:
            doc = json.load(fh)
    except Exception:
        return None
    rec = doc.get("captures", {}).get(workload)
    if not rec:
        return None
    rec = dict(rec)
    rec["source"] = "profiles/r02_ncu_k_render.json"
    rec["captured_with_source_sha16"] = doc.get("source_sha16")
    rec["same_sources_as_this_build"] = doc.get("source_sha16") == source_sha16()
    return rec


class Workload:
    """One bench workload on this rank: scene + tree on the device, frame buffers, and the two per-frame calls
    (device consumer for `value`, host consumer for `e2e`). N > 1 goes through the C ABI's peer frames (csrc/peer.cu)."""

    def __init__(self, name, api, torch, dist, dev, rank, world):
        self.name, self.api, self.torch, self.dist, self.dev, self.rank, self.world = name, api, torch, dist, dev, rank, world
        self.spec, self.width, self.height, self.rpp, self.depth = WORKLOADS[name]
        self.stream = torch.cuda.current_stream().cuda_stream
        kind, payload = scene_source(self.spec)
        self.kind = kind
        t0 = time.perf_counter()
        self.host = api.HostScene.from_xml_file(payload) if kind == "file" else api.HostScene.from_xml_text(payload)
        self.ingest_ms = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        self.scene = api.Scene(self.host.arrays, None, self.stream)
        torch.cuda.synchronize()
        self.build_ms = (time.perf_counter() - t0) * 1e3
        self.zoom = float(self.host.arrays.image_height) / self.height  # SURVEY.md Appendix E
        self.halo = self.host.halo_rows(self.depth)
        self.flag = torch.zeros((1,), dtype=torch.float32, device=dev)
        self.scene.reserve(self.params(0), world == 1, self.stream)
        w, h = self.width, self.height
        if world == 1:
            self.band = torch.empty((h, w, 4), dtype=torch.float32, device=dev)
            self.sigma = torch.empty((h, w), dtype=torch.float32, device=dev)
            self.scratch = torch.empty((h, w, 4), dtype=torch.float32, device=dev)
            self.out = torch.empty((h, w, 4), dtype=torch.float32, device=dev)
            self.exchange = None
            self.launches_per_step = 3
        else:
            # frames shared by the ranks: allocated by the library, IPC handles exchanged over torch.distributed (plumbing)
            self.peers = api.PeerFrames(w, h, rank, world)
            mine = torch.frombuffer(bytearray(self.peers.export_handles()), dtype=torch.uint8).to(dev)
            every = torch.empty((world * api.PEER_HANDLE_BYTES,), dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(every, mine)
            self.peers.connect_ipc(bytes(every.cpu().numpy().tobytes()))
            dist.barrier()
            my_strips = len(range(rank, (h + RDC_STRIP_ROWS - 1) // RDC_STRIP_ROWS, world))
            self.band = torch.empty((max(1, my_strips) * RDC_STRIP_ROWS, w, 4), dtype=torch.float32, device=dev)  # roofline launches
            self.sigma = torch.empty((max(1, my_strips) * RDC_STRIP_ROWS, w), dtype=torch.float32, device=dev)
            self.exchange = ("C ABI peer frames (rdc_peer_render_frame): render kernel stores into the consumers' frames over NVLink, "
                             "barrier kernel on flags in peer memory; CUDA IPC handles exchanged once at set-up")
            self.launches_per_step = 2 + (3 if self.halo > 0 else 0)  # render + barrier [+ 2 blur kernels + barrier]

    def params(self, step, **kw):
        return self.api.default_frame_params(self.width, self.height, self.rpp, zoom_factor=self.zoom, max_trace_depth=self.depth,
                                             frame=step, **kw)

    def frame_step(self, step, wait_event=0):
        """One frame, inputs resident, finished frame on (rank 0's) device."""
        api = self.api
        if self.world == 1:
            self.flag.zero_()
            p = self.params(step)
            p.max_sigma = self.flag.data_ptr()
            self.scene.render(p, self.band.data_ptr(), self.sigma.data_ptr(), self.stream)
            api.gaussian_blur(self.out.data_ptr(), self.band.data_ptr(), self.sigma.data_ptr(), self.scratch.data_ptr(), self.width,
                              self.height, 0, self.height, self.flag.data_ptr(), self.stream)
            return self.out.data_ptr()
        return self.peers.render_frame(self.scene, self.params(step), True, self.halo, self.stream, wait_event)

    def my_share(self, step):
        q = self.params(step)
        if self.world > 1:
            q.strip_stride, q.strip_offset = self.world, self.rank
        return q

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def time_value(self, steps, warmup, flush, sampler=None):
        """Device-timed frames, L2 flushed between them, max over ranks. Returns (ms per step, wall seconds)."""
        torch = self.torch
        for s in range(warmup):
            self.frame_step(s)
        if sampler:
            sampler.start()  # (NVML start-up takes milliseconds and differs from rank to rank: keep it in front of the barrier)
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        self.barrier()  # all ranks enter the timed region together: a rank that came early would count its wait for the others
        wall0 = time.perf_counter()
        for s in range(steps):
            flush.zero_()  # evict L2 between timed iterations (untimed)
            starts[s].record()
            self.last_frame = self.frame_step(warmup + s)
            ends[s].record()
        self.barrier()
        wall = time.perf_counter() - wall0
        if sampler:
            sampler.stop_flag = True
            sampler.join()
        total_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in zip(starts, ends))], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(total_ms, op=self.dist.ReduceOp.MAX)
            self.peers.status()
        return float(total_ms.item()) / steps, wall

    def time_e2e(self, n):
        """The same frames through host buffers: parameters in, finished frame in pinned host memory, every step; the copy of
        one frame overlaps the rendering of the next (two host frames in turn). Returns (seconds per step, description)."""
        torch, api = self.torch, self.api
        w, h = self.width, self.height
        if self.world == 1:
            hosts = [torch.empty((h, w, 4), dtype=torch.float32).pin_memory() for _ in range(2)]
            for s in range(2):
                self.scene.render_frame_to_host(self.params(s), True, hosts[0].data_ptr(), self.stream)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for s in range(n):
                self.scene.render_frame_to_host_async(self.params(1000 + s), True, hosts[s % 2].data_ptr(), self.stream)
            self.scene.frame_wait()
            t = (time.perf_counter() - t0) / n
            t0 = time.perf_counter()
            for s in range(n):
                self.scene.render_frame_to_host(self.params(2000 + s), True, hosts[0].data_ptr(), self.stream)
            t_sync = (time.perf_counter() - t0) / n
            return t, ("rdc_render_frame_to_host_async + rdc_frame_wait (render + blur + copy to pinned host memory, the copy of one "
                       f"frame overlapping the next frame's rendering); frame-by-frame rdc_render_frame_to_host: {t_sync * 1e3:.3f} ms")
        # one host frame all ranks address: POSIX shared memory created by rank 0, pinned in every process
        names = [f"/rdc_bench_{os.getpid()}_{k}" for k in range(2)] if self.rank == 0 else [None, None]
        self.dist.broadcast_object_list(names, src=0)
        nbytes = h * w * 16
        hosts = []
        if self.rank == 0:
            hosts = [api.HostFrame(nm, nbytes, True) for nm in names]
        self.dist.barrier()
        if self.rank != 0:
            hosts = [api.HostFrame(nm, nbytes, False) for nm in names]
        for s in range(2):
            self.peers.frame_to_host(self.scene, self.params(s), True, self.halo, hosts[s % 2].ptr, self.stream)
        self.peers.wait()
        self.barrier()
        t0 = time.perf_counter()
        for s in range(n):
            self.peers.frame_to_host(self.scene, self.params(1000 + s), True, self.halo, hosts[s % 2].ptr, self.stream)
        self.peers.wait()  # this rank's rows of every frame are in host memory
        self.barrier()     # ... and so are everybody else's
        t_local = torch.tensor([(time.perf_counter() - t0) / n], dtype=torch.float64, device=self.dev)
        self.dist.all_reduce(t_local, op=self.dist.ReduceOp.MAX)
        self.e2e_check = None
        if self.rank == 0:  # the assembled host frame is a finished frame: no row was left untouched
            self.e2e_check = bool(np_isfinite_or_nan_rows(hosts[(n - 1) % 2].numpy((h, w, 4))))
        self.dist.barrier()
        for hf in hosts:
            hf.close()
        return float(t_local.item()), ("rdc_peer_frame_to_host + rdc_peer_frames_wait: every rank renders its strips and copies its own rows "
                                       "of the finished frame over its own PCIe link into one pinned host frame shared by all ranks "
                                       "(POSIX shared memory), the copies of one frame overlapping the next frame's rendering")

    def kernel_roofline(self, reps):
        """k_render alone on this rank's share: work per ray from the counting build, time from CUDA events on its stream."""
        torch = self.torch
        stats = torch.zeros((9,), dtype=torch.int64, device=self.dev)
        stats[6:8] = torch.iinfo(torch.int64).max  # the timeline slots take minima
        my_rows = sum(min(RDC_STRIP_ROWS, self.height - t * RDC_STRIP_ROWS)
                      for t in range(self.rank, (self.height + RDC_STRIP_ROWS - 1) // RDC_STRIP_ROWS, self.world)) if self.world > 1 else self.height
        p = self.my_share(0)
        p.stats = stats.data_ptr()
        self.scene.render(p, self.band.data_ptr(), self.sigma.data_ptr(), self.stream)
        torch.cuda.synchronize()
        host_stats = stats.cpu().tolist()
        traced, nodes, chords, shaded, deferred, gathered = [float(x) for x in host_stats[:6]]
        t_start, t_first_idle, t_last = host_stats[6:9]
        nodes += gathered
        rays = float(my_rows) * self.width * self.rpp
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pk = self.my_share(1)
        pk.max_sigma = self.flag.data_ptr()
        k0.record()
        for _ in range(reps):
            self.scene.render(pk, self.band.data_ptr(), self.sigma.data_ptr(), self.stream)
        k1.record()
        torch.cuda.synchronize()
        kernel_ms = k0.elapsed_time(k1) / reps
        per = {"nodes": nodes / rays, "chords": chords / rays, "hits_shaded": shaded / rays, "rays_traced": traced / rays,
               "deferred_to_tree": deferred / rays, "table_query_nodes": gathered / rays}
        f_ray = F_GEN + per["nodes"] * F_NODE + per["chords"] * F_SEG + per["hits_shaded"] * F_SHADE + F_ACC
        b_ray = per["nodes"] * 32.0 + per["chords"] * 32.0  # SURVEY.md 8d: L2-side bytes per ray
        per["counting_build_timeline_ms"] = {"first_warp_out_of_work": (t_first_idle - t_start) * 1e-6, "last_warp_out": (t_last - t_start) * 1e-6}
        return {"rays": rays, "rows": my_rows, "kernel_ms": kernel_ms, "per_ray": per, "flops_per_ray": f_ray, "l2_bytes_per_ray": b_ray}

    def close(self):
        if self.world > 1:
            self.torch.cuda.synchronize()
            self.dist.barrier()
            self.peers.close()


def np_isfinite_or_nan_rows(frame):
    """Every row of an assembled host frame was written: alpha is 1 everywhere (rdc_render writes w = 1; the blur keeps it)."""
    import numpy as np

    a = frame[..., 3]
    return np.all(np.abs(a - 1.0) < 1e-3)


DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(work, out_dir):
    """--dump-outputs: the frame the last timed step left on (rank 0's) device, as the caller of the timed path receives it.
    Frames larger than DUMP_BYTES keep a fixed, seeded sample of whole rows, so runs with the same arguments compare."""
    import numpy as np

    torch = work.torch
    h, w = work.height, work.width

    class DeviceFrame:  # the frame lives in memory the library owns (peer frames for N > 1): viewed, not copied
        __cuda_array_interface__ = {"shape": (h, w, 4), "typestr": "<f4", "data": (work.last_frame, False), "strides": None,
                                    "version": 3}

    frame = torch.as_tensor(DeviceFrame(), device=work.dev)
    os.makedirs(out_dir, exist_ok=True)
    row_bytes = w * 4 * 4
    if h * row_bytes > DUMP_BYTES:
        n_rows = (DUMP_BYTES - 4096) // (row_bytes + 8)  # 4096: room for the two .npy headers
        rows = np.sort(np.random.default_rng(0).choice(h, n_rows, replace=False))
        frame = frame.index_select(0, torch.from_numpy(rows).to(work.dev))
        np.save(os.path.join(out_dir, "frame_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "frame.npy"), frame.cpu().numpy())


def measure_peaks(api, torch, stream, dev):
    """FP32 (dependent FFMA) and L2-read microbenchmarks on this GPU, now."""
    sink = torch.zeros((4,), dtype=torch.float32, device=dev)
    flops = ctypes.c_double()
    api.lib.rdc_microbench_fp32(2048, 2, sink.data_ptr(), ctypes.byref(flops), stream)
    torch.cuda.synchronize()
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0.record()
    api.lib.rdc_microbench_fp32(2048, 10, sink.data_ptr(), ctypes.byref(flops), stream)
    m1.record()
    torch.cuda.synchronize()
    fp32 = flops.value * 10 / (m0.elapsed_time(m1) * 1e-3) / 1e12
    buf = torch.zeros((32 << 20,), dtype=torch.uint8, device=dev)  # 32 MB: stays in L2
    nbytes = ctypes.c_double()
    api.lib.rdc_microbench_l2(buf.data_ptr(), buf.numel(), 4, 1, sink.data_ptr(), ctypes.byref(nbytes), stream)  # warm
    torch.cuda.synchronize()
    m0.record()
    api.lib.rdc_microbench_l2(buf.data_ptr(), buf.numel(), 16, 4, sink.data_ptr(), ctypes.byref(nbytes), stream)
    m1.record()
    torch.cuda.synchronize()
    l2 = nbytes.value * 4 / (m0.elapsed_time(m1) * 1e-3) / 1e9
    return fp32, l2


def roofline_block(work, k, fp32_peak, l2_peak, hbm_peak, single_gpu):
    achieved = k["rays"] * k["flops_per_ray"] / (k["kernel_ms"] * 1e-3) / 1e12
    l2_achieved = k["rays"] * k["l2_bytes_per_ray"] / (k["kernel_ms"] * 1e-3) / 1e9
    alg_bytes = float(k["rows"]) * work.width * 20.0
    cap = ncu_capture(work.name) if single_gpu else None
    return {
        "bound": "fp32", "kernel": "k_render", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak,
        "traffic": cap.get("dram_bytes") if cap else None,
        "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one launch under ncu --set full (profiles/r02_ncu_k_render.json); "
                        "below the algorithmic bytes where the frame the launch writes is still in the 126 MB L2 when it ends",
        "issue_slots": cap,
        "peak_source": "dependent-FFMA microbenchmark (rdc_microbench_fp32) run in this process; MEASURED_PEAKS.json has no FP32 figure",
        "kernel_ms": k["kernel_ms"], "flops_per_ray": k["flops_per_ray"], "per_ray": k["per_ray"],
        "l2": {"applies": work.scene.stats.traversal_bytes > 56 * 1024,  # smaller scenes are staged in shared memory: no L2 traffic to bound
               "bytes_per_ray": k["l2_bytes_per_ray"], "achieved_gbs": l2_achieved, "peak_gbs": l2_peak, "frac": l2_achieved / l2_peak,
               "peak_source": "L2-read microbenchmark (rdc_microbench_l2: 32 MB buffer, ld.global.cg, 128-bit loads) run in this process",
               "note": "SURVEY.md 8d: rays * (boxes + chords) * 32 B / t / L2 peak; the larger of the fp32 and l2 fractions is the binding one. "
                       "An upper bound of the real L2 traffic: table slots' boxes come from shared memory and L1 serves part of the run records"},
        "hbm": {"algorithmic_bytes": alg_bytes, "achieved_gbs": alg_bytes / (k["kernel_ms"] * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                "frac": (alg_bytes / (k["kernel_ms"] * 1e-3) / 1e9 / hbm_peak) if hbm_peak else None,
                "note": "output only (16 B image + 4 B sigma per pixel): the path is not HBM-bound; the partial sums of split work "
                        "units stay in L2 (their lines are discarded once added up, see DESIGN.md 3.1)"},
    }


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from raytracingdiffusioncurves_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    if os.environ.get("NCCL_DEBUG"):
        # NCCL logs to stdout unless told otherwise; stdout carries the one JSON line, so its log (rank counts included) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)  # plumbing only: handle exchange, timing reductions, host barriers
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)  # > 126 MB L2

    work = Workload(args.workload, api, torch, dist, dev, rank, world)
    sampler = ClockSampler(local_rank)
    ms_per_step, wall = work.time_value(args.steps, args.warmup, flush, sampler)
    if args.dump_outputs and rank == 0:
        dump_outputs(work, args.dump_outputs)
    rays_per_frame = float(work.width) * work.height * work.rpp
    value = rays_per_frame / (ms_per_step * 1e-3) / 1e9

    n_e2e = max(3, min(args.steps, 50))
    t_e2e, e2e_api = work.time_e2e(n_e2e)
    e2e = {"value": rays_per_frame / t_e2e / 1e9, "unit": "Grays/s", "ms_per_step": t_e2e * 1e3,
           "h2d_bytes_per_step": ctypes.sizeof(api.FrameParams) * world, "d2h_bytes_per_step": work.height * work.width * 16,
           "steps": n_e2e, "api": e2e_api}
    if world > 1 and rank == 0:
        e2e["host_frame_complete"] = work.e2e_check

    fp32_peak = l2_peak = hbm_peak = None
    roofline = None
    if rank == 0:
        fp32_peak, l2_peak = measure_peaks(api, torch, stream, dev)
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                hbm_peak = json.load(fh).get("hbm_gbs")
        except Exception:
            pass
        roofline = roofline_block(work, work.kernel_roofline(max(5, min(args.steps, 30))), fp32_peak, l2_peak, hbm_peak, world == 1)
    details = {"curves": work.scene.stats.n_curves, "segments": work.scene.stats.n_segments, "chords": work.scene.stats.n_chords,
               "runs": work.scene.stats.n_runs, "bvh_depth": work.scene.stats.bvh_depth, "exchange": work.exchange,
               "setup_ms": {"ingest": work.ingest_ms, "upload_and_tree_build": work.build_ms},
               "wall_ms_per_step_incl_flush": wall / args.steps * 1e3, "source_sha16": source_sha16()}
    launches = work.launches_per_step * args.steps * world
    kind = work.kind
    work.close()

    # ---- secondary: BASELINE.json configs[4], the 8192x8192 @512 synthetic 100 k-curve scene, a few frames at this N ----
    secondary = None
    if args.secondary and args.workload == DEFAULT_WORKLOAD:
        sec = Workload("synth100k_8k_512rpp", api, torch, dist, dev, rank, world)
        sec_ms, _ = sec.time_value(args.secondary_steps, 1, flush)
        sec_rays = float(sec.width) * sec.height * sec.rpp
        if rank == 0:
            k = sec.kernel_roofline(2)
            secondary = {"config": workload_config(sec.name, world), "metric": "Grays/s", "value": sec_rays / (sec_ms * 1e-3) / 1e9,
                         "ms_per_step": sec_ms, "steps": args.secondary_steps, "warmup": 1, "n_gpus": world, "scaling": "strong",
                         "chords": sec.scene.stats.n_chords, "runs": sec.scene.stats.n_runs,
                         "setup_ms": {"ingest": sec.ingest_ms, "upload_and_tree_build": sec.build_ms},
                         "roofline": roofline_block(sec, k, fp32_peak, l2_peak, hbm_peak, world == 1)}
        launches += sec.launches_per_step * (args.secondary_steps + 1) * world
        sec.close()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        spec, width, height, rpp, depth = WORKLOADS[args.workload]
        cpu_baseline = cpu_oracle_run("reference", spec, width, height, rpp, depth, workload_zoom(spec, height), args.cpu_seconds)

    if rank == 0:
        line = {
            "metric": "Grays/s", "value": value, "unit": "Grays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "bundled scene file (tests/golden/xmls)" if kind == "file" else "synthetic (rdc_synth_xml, SplitMix64 0x5EEDC0DE)",
            "config": workload_config(args.workload, world),
            "details": details,
            "clocks": sampler.result(),
            "e2e": e2e,
            "gpu_launches": launches,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
