"""ctypes binding of librdc_b200.so (include/rdc_b200.h) — the host-side mirror used by tests and bench.py.

The reference is a C++ executable, so the product's host code is C++ (csrc/, the ``OptixHello`` program);
this module only marshals pointers. Device memory comes from the caller (torch tensors or raw pointers);
nothing here computes anything and there is no CPU path: if the CUDA library is missing, import fails.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RDC_B200_LIB") or os.path.join(_HERE, "librdc_b200.so")  # override: kernel experiments

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
        "raytracingdiffusioncurves_b200 has no CPU fallback."
    )

_lib = C.CDLL(LIB_PATH)

u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
f32p = C.POINTER(C.c_float)


class IngestOptions(C.Structure):
    _fields_ = [("use_diffusion_curve_save", C.c_int), ("default_weight_degree", C.c_float), ("endcap_size", C.c_float)]


class SceneArrays(C.Structure):
    _fields_ = [
        ("image_width", C.c_int), ("image_height", C.c_int),
        ("n_vertices", C.c_uint32), ("n_segments", C.c_uint32), ("n_curves", C.c_uint32),
        ("vertices", f32p), ("segment_indices", u32p), ("curve_map", u32p), ("curve_index", u32p),
        ("curve_connect", i32p), ("curve_map_inverse", u32p),
        ("n_color_left", C.c_uint32), ("n_color_right", C.c_uint32), ("n_blur", C.c_uint32),
        ("n_weight", C.c_uint32), ("n_weight_degree", C.c_uint32),
        ("color_left_index", u32p), ("color_left", f32p), ("color_left_u", f32p),
        ("color_right_index", u32p), ("color_right", f32p), ("color_right_u", f32p),
        ("blur_index", u32p), ("blur", f32p), ("blur_u", f32p),
        ("weight_index", u32p), ("weight", f32p), ("weight_u", f32p),
        ("weight_degree_index", u32p), ("weight_degree", f32p), ("weight_degree_u", f32p),
    ]


class AccelOptions(C.Structure):
    _fields_ = [("curve_width", C.c_float), ("flatness_tolerance", C.c_float), ("max_chords_per_segment", C.c_int),
                ("run_length", C.c_int), ("shading_records", C.c_int), ("tree", C.c_int)]


class SceneInfo(C.Structure):
    _fields_ = [
        ("n_segments", C.c_uint32), ("n_curves", C.c_uint32), ("n_chords", C.c_uint32), ("n_runs", C.c_uint32),
        ("n_nodes", C.c_uint32), ("bvh_depth", C.c_uint32), ("has_portals", C.c_int), ("device_bytes", C.c_uint64),
        ("traversal_bytes", C.c_uint64), ("pad", C.c_float),
    ]


class FrameParams(C.Structure):
    _fields_ = [
        ("image_width", C.c_uint32), ("image_height", C.c_uint32), ("number_of_rays_per_pixel", C.c_float),
        ("zoom_factor", C.c_float), ("offset_x", C.c_float), ("offset_y", C.c_float),
        ("frame", C.c_uint32), ("seed", C.c_uint32), ("row_begin", C.c_uint32), ("row_end", C.c_uint32),
        ("strip_stride", C.c_uint32), ("strip_offset", C.c_uint32),
        ("use_diffusion_curve_save", C.c_int), ("use_aa", C.c_int), ("max_trace_depth", C.c_int),
        ("traversal", C.c_int), ("hit_ids", C.c_void_p), ("max_sigma", C.c_void_p), ("stats", C.c_void_p),
        ("route", C.c_int), ("units_per_tile", C.c_uint32), ("local_radius", C.c_float),
    ]


class LaunchPlan(C.Structure):
    _fields_ = [
        ("mode", C.c_int), ("smem", C.c_int), ("portals", C.c_int), ("stats", C.c_int), ("variant", C.c_int),
        ("built", C.c_int), ("units_per_tile", C.c_uint32), ("group", C.c_uint32), ("dynamic_smem", C.c_uint64),
    ]


TRAVERSAL_LBVH = 0
TRAVERSAL_BRUTE_FORCE = 1
ROUTE_AUTO, ROUTE_TREE, ROUTE_LOCAL_TABLE, ROUTE_CUT_TABLE = 0, 1, 2, 3
TREE_AUTO, TREE_MORTON, TREE_SAH = 0, 1, 2
MODE_TREE, MODE_TABLE, MODE_LOCAL, MODE_CUT = 0, 1, 2, 3  # rdc_launch_plan::mode
PICK_NONE, PICK_RIGHT, PICK_PORTAL = 0xFFFFFFFF, 1, 2  # rdc_pick::chord for a miss, rdc_pick::flags bits
# struct rdc_pick (32 bytes); stops of a pick are three float4: {left rgb, blur}, {right rgb, weight}, {weight_degree, 0, 0, 0}
PICK_DTYPE = np.dtype([("chord", np.uint32), ("segment", np.uint32), ("curve", np.uint32), ("flags", np.uint32),
                       ("u", np.float32), ("distance", np.float32), ("x", np.float32), ("y", np.float32)])

# every symbol include/rdc_b200.h declares, with its prototype (tests check the library exports them all)
PROTOTYPES = {
    "rdc_default_ingest_options": (None, [C.POINTER(IngestOptions)]),
    "rdc_ingest_xml_file": (C.c_int, [C.c_char_p, C.POINTER(IngestOptions), C.POINTER(C.c_void_p)]),
    "rdc_ingest_xml_memory": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(IngestOptions), C.POINTER(C.c_void_p)]),
    "rdc_host_scene_arrays": (C.c_int, [C.c_void_p, C.POINTER(SceneArrays)]),
    "rdc_host_scene_destroy": (None, [C.c_void_p]),
    "rdc_host_scene_save": (C.c_int, [C.c_void_p, C.c_char_p]),
    "rdc_host_scene_load": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "rdc_xml_dump_file": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "rdc_free": (None, [C.c_void_p]),
    "rdc_default_accel_options": (None, [C.POINTER(AccelOptions)]),
    "rdc_accel_build": (C.c_int, [C.POINTER(SceneArrays), C.POINTER(AccelOptions), C.c_void_p, C.POINTER(C.c_void_p)]),
    "rdc_scene_get_info": (C.c_int, [C.c_void_p, C.POINTER(SceneInfo)]),
    "rdc_scene_download_chords": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "rdc_scene_download_stop_tables": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rdc_scene_update_stops": (C.c_int, [C.c_void_p, C.POINTER(SceneArrays), C.c_void_p]),
    "rdc_scene_destroy": (None, [C.c_void_p]),
    "rdc_default_frame_params": (None, [C.POINTER(FrameParams), C.c_uint32, C.c_uint32, C.c_float]),
    "rdc_scene_reserve": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_int, C.c_void_p]),
    "rdc_scene_launch_plan": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.POINTER(LaunchPlan)]),
    "rdc_render": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "rdc_render_to_frames": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                       C.c_void_p]),
    "rdc_render_color_adjoint": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rdc_render_blur_adjoint": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "rdc_render_weight_adjoint": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]),
    "rdc_scene_pick": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rdc_scene_pick_frame": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rdc_view_pixel_to_scene": (C.c_int, [C.POINTER(FrameParams), C.c_uint32, C.c_uint32, f32p, f32p]),
    "rdc_peer_frames_create": (C.c_int, [C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "rdc_peer_frames_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rdc_peer_frames_connect_ipc": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rdc_peer_frames_connect_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "rdc_peer_frames_destroy": (None, [C.c_void_p]),
    "rdc_peer_barrier": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rdc_peer_status": (C.c_int, [C.c_void_p]),
    "rdc_peer_render_frame": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(FrameParams), C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                        C.POINTER(C.c_void_p)]),
    "rdc_peer_frame_to_host": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(FrameParams), C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rdc_peer_frames_wait": (C.c_int, [C.c_void_p]),
    "rdc_host_frame_open": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "rdc_host_frame_close": (C.c_int, [C.c_char_p, C.c_void_p, C.c_size_t, C.c_int]),
    "rdc_host_scene_halo_rows": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "gaussianBlur": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "setFloatDevice": (None, [C.c_void_p, C.c_uint, C.c_float, C.c_void_p]),
    "setupCurand": (None, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "rdc_gaussian_blur": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p, C.c_void_p]),
    "rdc_gaussian_blur_band": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_void_p, C.c_void_p]),
    "rdc_gaussian_blur_adjoint": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_void_p, C.c_void_p]),
    "rdc_gaussian_blur_sigma_adjoint": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                                  C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "rdc_render_frame_to_host": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_int, C.c_void_p, C.c_void_p]),
    "rdc_render_frame_to_host_async": (C.c_int, [C.c_void_p, C.POINTER(FrameParams), C.c_int, C.c_void_p, C.c_void_p]),
    "rdc_frame_wait": (C.c_int, [C.c_void_p]),
    "rdc_image_to_rgba8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "rdc_write_ppm": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int, C.c_int]),
    "rdc_write_png": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int, C.c_int]),
    "rdc_write_jpg": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "rdc_psnr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "rdc_view_scroll": (None, [C.POINTER(FrameParams), C.c_double]),
    "rdc_view_drag": (None, [C.POINTER(FrameParams), C.c_double, C.c_double]),
    "rdc_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]),
    "rdc_synth_xml": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "rdc_microbench_fp32": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "rdc_microbench_l2": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "rdc_last_error_string": (C.c_char_p, []),
    "rdc_version": (C.c_char_p, []),
}
for _name, (_res, _args) in PROTOTYPES.items():
    _fn = getattr(_lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args

lib = _lib


class RdcError(RuntimeError):
    def __init__(self, code: int, where: str):
        self.code = code
        msg = _lib.rdc_last_error_string().decode("utf-8", "replace")
        super().__init__(f"{where} failed with code {code}: {msg}")


def _check(code: int, where: str) -> None:
    if code != 0:
        raise RdcError(code, where)


def last_error() -> str:
    return _lib.rdc_last_error_string().decode("utf-8", "replace")


def default_ingest_options(**overrides) -> IngestOptions:
    o = IngestOptions()
    _lib.rdc_default_ingest_options(C.byref(o))
    for k, v in overrides.items():
        setattr(o, k, v)
    return o


def default_accel_options(**overrides) -> AccelOptions:
    o = AccelOptions()
    _lib.rdc_default_accel_options(C.byref(o))
    for k, v in overrides.items():
        setattr(o, k, v)
    return o


def default_frame_params(width: int, height: int, rays_per_pixel: float, **overrides) -> FrameParams:
    p = FrameParams()
    _lib.rdc_default_frame_params(C.byref(p), width, height, float(rays_per_pixel))
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


_FAMILIES = ("color_left", "color_right", "blur", "weight", "weight_degree")


class HostScene:
    """Result of the ingest: the structure-of-arrays scene in host memory (reference Params arrays)."""

    def __init__(self, handle: int):
        self._h = C.c_void_p(handle)
        self.arrays = SceneArrays()
        _check(_lib.rdc_host_scene_arrays(self._h, C.byref(self.arrays)), "rdc_host_scene_arrays")

    @classmethod
    def from_xml_file(cls, path: str, options: IngestOptions | None = None) -> "HostScene":
        h = C.c_void_p()
        _check(_lib.rdc_ingest_xml_file(os.fsencode(path), C.byref(options) if options else None, C.byref(h)),
               "rdc_ingest_xml_file")
        return cls(h.value)

    @classmethod
    def from_xml_text(cls, text: bytes, options: IngestOptions | None = None) -> "HostScene":
        h = C.c_void_p()
        _check(_lib.rdc_ingest_xml_memory(text, len(text), C.byref(options) if options else None, C.byref(h)),
               "rdc_ingest_xml_memory")
        return cls(h.value)

    @classmethod
    def from_cache(cls, path: str) -> "HostScene":
        h = C.c_void_p()
        _check(_lib.rdc_host_scene_load(os.fsencode(path), C.byref(h)), "rdc_host_scene_load")
        return cls(h.value)

    def save(self, path: str) -> None:
        _check(_lib.rdc_host_scene_save(self._h, os.fsencode(path)), "rdc_host_scene_save")

    def close(self) -> None:
        if self._h:
            _lib.rdc_host_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def halo_rows(self, max_trace_depth: int = 0) -> int:
        """rdc_host_scene_halo_rows: the blur's reach in rows for any frame of this scene (0: no blur)."""
        out = C.c_int()
        _check(_lib.rdc_host_scene_halo_rows(self._h, max_trace_depth, C.byref(out)), "rdc_host_scene_halo_rows")
        return out.value

    def max_blur(self, max_trace_depth: int = 0) -> float:
        """Upper bound of any blur_map value: sigma is a weighted mean of blur stops; each portal passed
        multiplies it by another stop (DeviceCode.cu:311)."""
        a = self.arrays
        if a.n_blur == 0:
            return 0.0
        m = float(np.ctypeslib.as_array(a.blur, shape=(a.n_blur,)).max())
        portals = bool((np.ctypeslib.as_array(a.curve_connect, shape=(a.n_curves,)) >= 0).any())
        if portals and m > 1.0:
            m = m ** (max_trace_depth + 1)
        return max(m, 0.0)

    def to_numpy(self) -> dict:
        """Copies of every array (sentinels included), keyed like struct Params."""
        a = self.arrays

        def arr(ptr, shape, dtype):
            n = int(np.prod(shape))
            if n == 0:
                return np.zeros(shape, dtype)
            return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True).reshape(shape)

        colour_len = max(a.n_color_left, a.n_color_right) + 2
        out = {
            "image_width": a.image_width, "image_height": a.image_height,
            "vertices": arr(a.vertices, (a.n_vertices, 3), np.float32),
            "segment_indices": arr(a.segment_indices, (a.n_segments,), np.uint32),
            "curve_map": arr(a.curve_map, (a.n_segments,), np.uint32),
            "curve_index": arr(a.curve_index, (a.n_segments,), np.uint32),
            "curve_connect": arr(a.curve_connect, (a.n_curves,), np.int32),
            "curve_map_inverse": arr(a.curve_map_inverse, (a.n_curves,), np.uint32),
        }
        for fam in _FAMILIES:
            n = getattr(a, "n_" + fam)
            padded = colour_len if fam.startswith("color") else n + 2
            stride = 3 if fam.startswith("color") else 1
            out["n_" + fam] = n
            out[fam + "_index"] = arr(getattr(a, fam + "_index"), (a.n_curves, 2), np.uint32)
            out[fam] = arr(getattr(a, fam), (padded, stride) if stride == 3 else (padded,), np.float32)
            out[fam + "_u"] = arr(getattr(a, fam + "_u"), (padded,), np.float32)
        return out


def arrays_from_numpy(d: dict) -> SceneArrays:
    """SceneArrays over a dictionary laid out like HostScene.to_numpy() (its inverse): edit a copy of a scene in numpy
    and pass it to Scene or Scene.update_stops. The structure keeps its arrays alive."""
    keep = {}

    def ptr(name, dtype, ctype):
        arr = np.ascontiguousarray(d[name], dtype)
        keep[name] = arr
        return arr.ctypes.data_as(C.POINTER(ctype))

    a = SceneArrays()
    a.image_width, a.image_height = int(d["image_width"]), int(d["image_height"])
    a.n_vertices = len(d["vertices"])
    a.n_segments = len(d["segment_indices"])
    a.n_curves = len(d["curve_connect"])
    a.vertices = ptr("vertices", np.float32, C.c_float)
    a.segment_indices = ptr("segment_indices", np.uint32, C.c_uint32)
    a.curve_map = ptr("curve_map", np.uint32, C.c_uint32)
    a.curve_index = ptr("curve_index", np.uint32, C.c_uint32)
    a.curve_connect = ptr("curve_connect", np.int32, C.c_int32)
    a.curve_map_inverse = ptr("curve_map_inverse", np.uint32, C.c_uint32)
    for fam in _FAMILIES:
        setattr(a, "n_" + fam, int(d["n_" + fam]))
        setattr(a, fam + "_index", ptr(fam + "_index", np.uint32, C.c_uint32))
        setattr(a, fam, ptr(fam, np.float32, C.c_float))
        setattr(a, fam + "_u", ptr(fam + "_u", np.float32, C.c_float))
    a._keep = keep
    return a


def xml_dump(path: str) -> str:
    p = C.c_void_p()
    _check(_lib.rdc_xml_dump_file(os.fsencode(path), C.byref(p)), "rdc_xml_dump_file")
    try:
        return C.string_at(p).decode("utf-8", "replace")
    finally:
        _lib.rdc_free(p)


def synth_xml(n_curves: int, width: int, height: int, seed: int = 0x5EEDC0DE) -> bytes:
    p = C.c_void_p()
    n = C.c_size_t()
    _check(_lib.rdc_synth_xml(n_curves, width, height, seed, C.byref(p), C.byref(n)), "rdc_synth_xml")
    try:
        return C.string_at(p, n.value)
    finally:
        _lib.rdc_free(p)


@dataclass
class SceneStats:
    n_segments: int
    n_curves: int
    n_chords: int
    n_runs: int
    n_nodes: int
    bvh_depth: int
    has_portals: bool
    device_bytes: int
    traversal_bytes: int
    pad: float


class Scene:
    """Device-resident scene + LBVH (one per device); wraps rdc_accel_build / rdc_render."""

    def __init__(self, arrays: SceneArrays, options: AccelOptions | None = None, stream: int = 0):
        h = C.c_void_p()
        _check(_lib.rdc_accel_build(C.byref(arrays), C.byref(options) if options else None, C.c_void_p(stream), C.byref(h)),
               "rdc_accel_build")
        self._h = h
        self._refresh_stats()
        # build_scene's rule for the per-chord shading records: not turned off, and the table fits 32 MB
        self.has_records = (options.shading_records if options else 0) >= 0 and self.stats.n_chords * 128 <= 32 << 20

    def _refresh_stats(self) -> None:
        info = SceneInfo()
        _check(_lib.rdc_scene_get_info(self._h, C.byref(info)), "rdc_scene_get_info")
        self.stats = SceneStats(info.n_segments, info.n_curves, info.n_chords, info.n_runs, info.n_nodes, info.bvh_depth,
                                bool(info.has_portals), info.device_bytes, info.traversal_bytes, info.pad)

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def close(self) -> None:
        if self._h:
            _lib.rdc_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def chords(self):
        n = self.stats.n_chords
        geom = np.empty((n, 4), np.float32)
        ids = np.empty((n, 3), np.uint32)
        _check(_lib.rdc_scene_download_chords(self._h, geom.ctypes.data, ids.ctypes.data), "rdc_scene_download_chords")
        return geom, ids

    def update_stops(self, arrays: SceneArrays, stream: int = 0) -> None:
        """rdc_scene_update_stops: new colour, blur, weight and exponent stops on the built scene (same geometry)."""
        _check(_lib.rdc_scene_update_stops(self._h, C.byref(arrays), C.c_void_p(stream)), "rdc_scene_update_stops")
        self._refresh_stats()

    def stop_tables(self) -> dict:
        """rdc_scene_download_stop_tables: seg_walk uint32 [n_segments,16], chord_walk uint32 [n_chords,8], chord_records
        float32 [n_chords,32] or None when the scene has no shading records."""
        st = self.stats
        seg_walk = np.empty((st.n_segments, 16), np.uint32)
        chord_walk = np.empty((st.n_chords, 8), np.uint32)
        records = np.empty((st.n_chords, 32), np.float32) if self.has_records else None
        _check(_lib.rdc_scene_download_stop_tables(self._h, seg_walk.ctypes.data, chord_walk.ctypes.data,
                                                   records.ctypes.data if records is not None else None),
               "rdc_scene_download_stop_tables")
        return {"seg_walk": seg_walk, "chord_walk": chord_walk, "chord_records": records}

    def reserve(self, params: FrameParams, host_frames: bool = False, stream: int = 0) -> None:
        """rdc_scene_reserve: allocate the handle's scratch for frames like `params` ahead of the first render."""
        _check(_lib.rdc_scene_reserve(self._h, C.byref(params), int(host_frames), C.c_void_p(stream)), "rdc_scene_reserve")

    def launch_plan(self, params: FrameParams) -> LaunchPlan:
        """rdc_scene_launch_plan: the render kernel variant, units per tile and shared memory rdc_render would use."""
        out = LaunchPlan()
        _check(_lib.rdc_scene_launch_plan(self._h, C.byref(params), C.byref(out)), "rdc_scene_launch_plan")
        return out

    def render(self, params: FrameParams, image_ptr: int, blur_map_ptr: int, stream: int = 0) -> None:
        """Enqueue one frame (rows [row_begin,row_end)) on `stream`. Pointers are device addresses."""
        _check(_lib.rdc_render(self._h, C.byref(params), C.c_void_p(image_ptr), C.c_void_p(blur_map_ptr), C.c_void_p(stream)),
               "rdc_render")

    def render_to_frames(self, params: FrameParams, image_ptrs, blur_map_ptrs, stream: int = 0) -> None:
        """Like render, but every finished pixel is stored at its place in each of the given FULL frames (device
        addresses, peers' memory included): rdc_render_to_frames."""
        n = len(image_ptrs)
        images = (C.c_void_p * n)(*image_ptrs)
        sigmas = (C.c_void_p * n)(*blur_map_ptrs)
        _check(_lib.rdc_render_to_frames(self._h, C.byref(params), n, images, sigmas, C.c_void_p(stream)), "rdc_render_to_frames")

    def color_adjoint(self, params: FrameParams, grad_ptr: int, left_ptr: int, right_ptr: int, stream: int = 0) -> None:
        """rdc_render_color_adjoint: A^T grad, the transpose of render in the colour stops. grad_ptr: device float32 [rows, W, 4]
        (dL/dRGB, band-local like render's image); left_ptr, right_ptr: device float64 [max(n_color_left, n_color_right) + 2, 3],
        overwritten. Enqueue-only."""
        _check(_lib.rdc_render_color_adjoint(self._h, C.byref(params), C.c_void_p(grad_ptr), C.c_void_p(left_ptr),
                                             C.c_void_p(right_ptr), C.c_void_p(stream)), "rdc_render_color_adjoint")

    def blur_adjoint(self, params: FrameParams, grad_ptr: int, out_ptr: int, stream: int = 0) -> None:
        """rdc_render_blur_adjoint: A_b^T grad, the transpose of render's blur map in the blur stops. grad_ptr: device float32
        [rows, W] (band-local); out_ptr: device float64 laid out like the handle's blur array (n_blur + 2)."""
        _check(_lib.rdc_render_blur_adjoint(self._h, C.byref(params), C.c_void_p(grad_ptr), C.c_void_p(out_ptr),
                                            C.c_void_p(stream)), "rdc_render_blur_adjoint")

    def weight_adjoint(self, params: FrameParams, image_grad_ptr: int, sigma_grad_ptr: int, weight_ptr: int, degree_ptr: int,
                       stream: int = 0) -> None:
        """rdc_render_weight_adjoint: the gradient of the render's image and blur map in the weight and exponent stops, for
        a device float4 image gradient and a device float32 sigma gradient ([rows, W], band-local; 0 means zero, not both).
        weight_ptr / degree_ptr: device float64 laid out like the handle's weight (n_weight + 2) and weight_degree
        (n_weight_degree + 2) arrays."""
        _check(_lib.rdc_render_weight_adjoint(self._h, C.byref(params), C.c_void_p(image_grad_ptr), C.c_void_p(sigma_grad_ptr),
                                              C.c_void_p(weight_ptr), C.c_void_p(degree_ptr), C.c_void_p(stream)),
               "rdc_render_weight_adjoint")

    def pick(self, points_ptr: int, n: int, out_ptr: int, stops_ptr: int = 0, max_distance: float = float("inf"),
             use_diffusion_curve_save: int = 1, stream: int = 0) -> None:
        """rdc_scene_pick: the nearest chord to each of n device float2 points, into device records of PICK_DTYPE (and,
        when stops_ptr is given, three float4 of stop values per point). Enqueue-only."""
        _check(_lib.rdc_scene_pick(self._h, C.c_void_p(points_ptr), n, max_distance, int(use_diffusion_curve_save),
                                   C.c_void_p(out_ptr), C.c_void_p(stops_ptr), C.c_void_p(stream)), "rdc_scene_pick")

    def pick_frame(self, params: FrameParams, out_ptr: int, stops_ptr: int = 0, max_distance: float = float("inf"),
                   stream: int = 0) -> None:
        """rdc_scene_pick_frame: one pick per pixel centre of the band of `params` (band-local, like render)."""
        _check(_lib.rdc_scene_pick_frame(self._h, C.byref(params), max_distance, C.c_void_p(out_ptr), C.c_void_p(stops_ptr),
                                         C.c_void_p(stream)), "rdc_scene_pick_frame")

    def render_frame_to_host(self, params: FrameParams, use_blur: bool, host_image_ptr: int, stream: int = 0) -> None:
        _check(_lib.rdc_render_frame_to_host(self._h, C.byref(params), int(use_blur), C.c_void_p(host_image_ptr),
                                             C.c_void_p(stream)), "rdc_render_frame_to_host")


def _scene_async(self, params, use_blur, host_image_ptr, stream=0):
    _check(_lib.rdc_render_frame_to_host_async(self._h, C.byref(params), int(use_blur), C.c_void_p(host_image_ptr), C.c_void_p(stream)),
           "rdc_render_frame_to_host_async")


def _scene_wait(self):
    _check(_lib.rdc_frame_wait(self._h), "rdc_frame_wait")


Scene.render_frame_to_host_async = _scene_async
Scene.frame_wait = _scene_wait


PEER_HANDLE_BYTES = 320  # RDC_PEER_HANDLE_BYTES


class PeerFrames:
    """One rank's view of the frames the GPUs of a box share (rdc_peer_frames_*). Pointer marshalling only."""

    def __init__(self, width: int, height: int, rank: int, world: int):
        h = C.c_void_p()
        _check(_lib.rdc_peer_frames_create(width, height, rank, world, C.byref(h)), "rdc_peer_frames_create")
        self._h, self.rank, self.world, self.width, self.height = h, rank, world, width, height

    def export_handles(self) -> bytes:
        buf = C.create_string_buffer(PEER_HANDLE_BYTES)
        _check(_lib.rdc_peer_frames_export(self._h, buf), "rdc_peer_frames_export")
        return buf.raw

    def connect_ipc(self, all_handles: bytes) -> None:
        assert len(all_handles) == PEER_HANDLE_BYTES * self.world
        _check(_lib.rdc_peer_frames_connect_ipc(self._h, all_handles), "rdc_peer_frames_connect_ipc")

    @staticmethod
    def connect_local(frames) -> None:
        arr = (C.c_void_p * len(frames))(*[f._h for f in frames])
        _check(_lib.rdc_peer_frames_connect_local(arr, len(frames)), "rdc_peer_frames_connect_local")

    def barrier(self, stream: int = 0) -> None:
        _check(_lib.rdc_peer_barrier(self._h, C.c_void_p(stream)), "rdc_peer_barrier")

    def status(self) -> None:
        _check(_lib.rdc_peer_status(self._h), "rdc_peer_status")

    def render_frame(self, scene: "Scene", params: FrameParams, use_blur: bool, halo_rows: int, stream: int = 0,
                     wait_event: int = 0) -> int:
        """Device consumer: returns the device address of the finished frame on rank 0, 0 elsewhere."""
        out = C.c_void_p()
        _check(_lib.rdc_peer_render_frame(scene.handle, self._h, C.byref(params), int(use_blur), halo_rows, C.c_void_p(wait_event),
                                          C.c_void_p(stream), C.byref(out)), "rdc_peer_render_frame")
        return out.value or 0

    def frame_to_host(self, scene: "Scene", params: FrameParams, use_blur: bool, halo_rows: int, host_frame_ptr: int,
                      stream: int = 0) -> None:
        _check(_lib.rdc_peer_frame_to_host(scene.handle, self._h, C.byref(params), int(use_blur), halo_rows,
                                           C.c_void_p(host_frame_ptr), C.c_void_p(stream)), "rdc_peer_frame_to_host")

    def wait(self) -> None:
        _check(_lib.rdc_peer_frames_wait(self._h), "rdc_peer_frames_wait")

    def close(self) -> None:
        if self._h:
            _lib.rdc_peer_frames_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostFrame:
    """A host frame every rank of a box can address: POSIX shared memory, pinned (rdc_host_frame_open)."""

    def __init__(self, name: str, nbytes: int, create: bool):
        p = C.c_void_p()
        _check(_lib.rdc_host_frame_open(name.encode(), nbytes, int(create), C.byref(p)), "rdc_host_frame_open")
        self.name, self.nbytes, self.ptr, self.owner = name, nbytes, p.value, create

    def numpy(self, shape):
        return np.ctypeslib.as_array(C.cast(self.ptr, f32p), shape=(self.nbytes // 4,)).reshape(shape)

    def close(self) -> None:
        if self.ptr:
            _lib.rdc_host_frame_close(self.name.encode(), C.c_void_p(self.ptr), self.nbytes, int(self.owner))
            self.ptr = 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def gaussian_blur(dest_ptr: int, src_ptr: int, sigma_ptr: int, scratch_ptr: int, width: int, height: int,
                  row_begin: int = 0, row_end: int | None = None, max_sigma_ptr: int = 0, stream: int = 0) -> None:
    _check(_lib.rdc_gaussian_blur(C.c_void_p(dest_ptr), C.c_void_p(src_ptr), C.c_void_p(sigma_ptr), C.c_void_p(scratch_ptr),
                                  width, height, row_begin, height if row_end is None else row_end,
                                  C.c_void_p(max_sigma_ptr), C.c_void_p(stream)), "rdc_gaussian_blur")


def gaussian_blur_band(dest_ptr: int, src_ptr: int, sigma_ptr: int, scratch_ptr: int, width: int, height: int,
                       row_begin: int, row_end: int, halo_rows: int, max_sigma_ptr: int = 0, stream: int = 0) -> None:
    _check(_lib.rdc_gaussian_blur_band(C.c_void_p(dest_ptr), C.c_void_p(src_ptr), C.c_void_p(sigma_ptr), C.c_void_p(scratch_ptr),
                                       width, height, row_begin, row_end, halo_rows, C.c_void_p(max_sigma_ptr),
                                       C.c_void_p(stream)), "rdc_gaussian_blur_band")


def gaussian_blur_adjoint(grad_source_ptr: int, grad_dest_ptr: int, sigma_ptr: int, scratch_ptr: int, width: int, height: int,
                          row_begin: int = 0, row_end: int | None = None, max_sigma_ptr: int = 0, stream: int = 0) -> None:
    """rdc_gaussian_blur_adjoint: grad_source (float4, all `height` rows) = the transpose of gaussian_blur with the same sigma,
    band and max_sigma, applied to grad_dest's band rows. scratch: float4[width * height + 1]."""
    _check(_lib.rdc_gaussian_blur_adjoint(C.c_void_p(grad_source_ptr), C.c_void_p(grad_dest_ptr), C.c_void_p(sigma_ptr),
                                          C.c_void_p(scratch_ptr), width, height, row_begin, height if row_end is None else row_end,
                                          C.c_void_p(max_sigma_ptr), C.c_void_p(stream)), "rdc_gaussian_blur_adjoint")


def gaussian_blur_sigma_adjoint(grad_sigma_ptr: int, grad_dest_ptr: int, src_ptr: int, sigma_ptr: int, scratch_ptr: int,
                                width: int, height: int, row_begin: int = 0, row_end: int | None = None, max_sigma_ptr: int = 0,
                                stream: int = 0) -> None:
    """rdc_gaussian_blur_sigma_adjoint: grad_sigma (float, all `height` rows) = the derivative of <grad_dest, gaussian_blur(src,
    sigma)> on the band in each pixel's sigma, taps held fixed. scratch: float4[2 * width * height + 1]."""
    _check(_lib.rdc_gaussian_blur_sigma_adjoint(C.c_void_p(grad_sigma_ptr), C.c_void_p(grad_dest_ptr), C.c_void_p(src_ptr),
                                                C.c_void_p(sigma_ptr), C.c_void_p(scratch_ptr), width, height, row_begin,
                                                height if row_end is None else row_end, C.c_void_p(max_sigma_ptr),
                                                C.c_void_p(stream)), "rdc_gaussian_blur_sigma_adjoint")


def _is_torch(a) -> bool:
    return type(a).__module__.startswith("torch")


def _dot(a, b) -> float:
    return float((a * b).sum())


def cgls(apply_a, apply_at, b, x0, iterations: int):
    """Conjugate gradients on the normal equations (CGLS) for min ||A x - b||, in float64, on numpy arrays or torch tensors.
    apply_a(p) -> A p has the type and shape of b; apply_at(r) -> A^T r those of x0. Returns (x, residuals): residuals[0] is
    ||b - A x0|| and residuals[k] the residual after iteration k. Stops early when A^T r or A p vanishes (x is then a
    least-squares solution, or the step would be undefined), and when a step would raise the residual: in exact arithmetic
    it never does, so that only happens once rounding (fp32 images) dominates the remaining progress; the step is not
    taken, so the residuals returned never increase."""
    if _is_torch(x0):
        import torch

        x = x0.to(dtype=torch.float64, copy=True)
    else:
        x = np.array(x0, np.float64)
    r = b - apply_a(x)
    s = apply_at(r)
    p = s * 1.0
    gamma = _dot(s, s)
    residuals = [_dot(r, r) ** 0.5]
    for _ in range(iterations):
        if gamma == 0.0:
            break
        q = apply_a(p)
        qq = _dot(q, q)
        if qq == 0.0:
            break
        alpha = gamma / qq
        r_next = r - alpha * q
        res_next = _dot(r_next, r_next) ** 0.5
        if res_next > residuals[-1]:
            break
        x = x + alpha * p
        r = r_next
        residuals.append(res_next)
        s = apply_at(r)
        gamma_next = _dot(s, s)
        p = s + (gamma_next / gamma) * p
        gamma = gamma_next
    return x, residuals


def fit_stops(d: dict, target, render, adjoint, iterations: int):
    """The least-squares colour fit behind fit_colors, over any render / adjoint pair (numpy or torch images).
    render(left, right) -> image [rows, W, >=3] for float32 colour arrays laid out like d["color_left"] / d["color_right"];
    adjoint(grad) -> (left, right) float64 arrays of that layout, the transpose of render at the same pixels, for a float32
    grad [rows, W, 4]. Only the real stops (j < n_color_*) are unknowns: padding entries and sentinels keep d's values and
    their gradient is dropped. Pixels that are NaN in the target or in the render have zero residual. The image is affine in
    the unknowns (the fixed entries add a constant), so the fit is CGLS on its linear part: render with zeros in the fixed
    entries. Returns (fitted copy of d, residual norms as cgls returns them)."""
    nl, nr = int(d["n_color_left"]), int(d["n_color_right"])
    base_l = np.asarray(d["color_left"], np.float32)
    base_r = np.asarray(d["color_right"], np.float32)

    def colours(x, fixed):
        x = x.cpu().numpy() if _is_torch(x) else np.asarray(x)
        left = base_l.copy() if fixed else np.zeros_like(base_l)
        right = base_r.copy() if fixed else np.zeros_like(base_r)
        left[:nl] = x[:3 * nl].reshape(nl, 3)
        right[:nr] = x[3 * nl:].reshape(nr, 3)
        return left, right

    torch_images = _is_torch(target)
    if torch_images:
        import torch

        isnan, where = torch.isnan, lambda m, a: torch.where(m, a, torch.zeros_like(a))
        f64 = lambda a: a.to(torch.float64)  # noqa: E731
    else:
        isnan, where = np.isnan, lambda m, a: np.where(m, a, 0.0)
        f64 = lambda a: np.asarray(a, np.float64)  # noqa: E731
    target3 = f64(target[..., :3])
    n = 3 * (nl + nr)
    constant = f64(render(*colours(np.zeros(n), True))[..., :3])  # what the fixed entries alone give
    keep = ~(isnan(constant).any(-1) | isnan(target3).any(-1))[..., None]
    b = where(keep, target3 - constant)

    def apply_a(p):
        return where(keep, f64(render(*colours(p, False))[..., :3]))

    def apply_at(r):
        if torch_images:
            g = torch.zeros(r.shape[:-1] + (4,), dtype=torch.float32, device=r.device)
        else:
            g = np.zeros(r.shape[:-1] + (4,), np.float32)
        g[..., :3] = r
        gl, gr = adjoint(g)
        return np.concatenate([np.asarray(gl, np.float64)[:nl].ravel(), np.asarray(gr, np.float64)[:nr].ravel()])

    x0 = np.concatenate([base_l[:nl].ravel(), base_r[:nr].ravel()]).astype(np.float64)
    x, residuals = cgls(apply_a, apply_at, b, x0, iterations)
    fitted = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in d.items()}
    fitted["color_left"], fitted["color_right"] = colours(x, True)
    return fitted, residuals


class _BandFrame:
    """The band of `params` as the fits see it, built once per (scene, params, use_blur): forward(**stops) puts the stop
    arrays given (HostScene.to_numpy() names) on the handle over `d`'s (update_stops) and renders the band, then, with
    use_blur, blurs it as rdc_render_frame_to_host(use_blur=1) does (the band as a buffer of its own rows, with the render's
    max_sigma flag); it returns the frame, float32 [rows, W, 4]. transpose(g) is the blur's transpose Bᵀ g with the last
    forward's blur map (g itself without the blur) and sigma_adjoint(g) the blurred frame's derivative in that map. Device
    buffers are reused from call to call; `stream` must be torch's current stream."""

    def __init__(self, scene: "Scene", d: dict, params: FrameParams, use_blur: bool, stream: int):
        import torch

        self.scene, self.params, self.use_blur, self.stream = scene, params, use_blur, stream
        self.rows, self.w = params.row_end - params.row_begin, params.image_width
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.image = torch.empty((self.rows, self.w, 4), dtype=torch.float32, device=self.dev)
        self.sigma = torch.empty((self.rows, self.w), dtype=torch.float32, device=self.dev)
        self.work = dict(d)
        if use_blur:
            self.blurred = torch.empty_like(self.image)
            self.grad_image = torch.empty_like(self.image)
            self.grad_sigma = torch.empty_like(self.sigma)
            # the blur's and both derivatives'
            self.scratch = torch.empty((2 * self.rows * self.w + 1, 4), dtype=torch.float32, device=self.dev)
            self.flag = torch.zeros((1,), dtype=torch.float32, device=self.dev)
            self.blur_params = FrameParams.from_buffer_copy(params)
            self.blur_params.max_sigma = self.flag.data_ptr()
        scene.reserve(params, False, stream)

    def _blur_args(self):
        return self.scratch.data_ptr(), self.w, self.rows, 0, self.rows, self.flag.data_ptr(), self.stream

    def forward(self, **stops):
        self.work.update(stops)
        self.scene.update_stops(arrays_from_numpy(self.work), self.stream)
        if not self.use_blur:
            self.scene.render(self.params, self.image.data_ptr(), self.sigma.data_ptr(), self.stream)
            return self.image
        self.flag.zero_()
        self.scene.render(self.blur_params, self.image.data_ptr(), self.sigma.data_ptr(), self.stream)
        gaussian_blur(self.blurred.data_ptr(), self.image.data_ptr(), self.sigma.data_ptr(), *self._blur_args())
        return self.blurred

    def transpose(self, g):
        if not self.use_blur:
            return g
        gaussian_blur_adjoint(self.grad_image.data_ptr(), g.data_ptr(), self.sigma.data_ptr(), *self._blur_args())
        return self.grad_image

    def sigma_adjoint(self, g):
        gaussian_blur_sigma_adjoint(self.grad_sigma.data_ptr(), g.data_ptr(), self.image.data_ptr(), self.sigma.data_ptr(),
                                    *self._blur_args())
        return self.grad_sigma


def _color_operator(scene: "Scene", d: dict, params: FrameParams, use_blur: bool, stream: int):
    """The (render, adjoint) pair fit_colors hands to fit_stops: render(left, right) is _BandFrame.forward with those colour
    values; adjoint(grad) is the blur's transpose with the last render's blur map (colour values never change it), then
    Scene.color_adjoint. `stream` must be torch's current stream."""
    import torch

    frame = _BandFrame(scene, d, params, use_blur, stream)
    grad_left = torch.empty(np.asarray(d["color_left"]).shape, dtype=torch.float64, device=frame.dev)
    grad_right = torch.empty(np.asarray(d["color_right"]).shape, dtype=torch.float64, device=frame.dev)

    def render(left, right):
        return frame.forward(color_left=left, color_right=right)

    def adjoint(g):
        g = frame.transpose(g.contiguous())
        scene.color_adjoint(params, g.data_ptr(), grad_left.data_ptr(), grad_right.data_ptr(), stream)
        return grad_left.cpu().numpy(), grad_right.cpu().numpy()

    return render, adjoint


def fit_colors(scene: "Scene", d: dict, params: FrameParams, target, iterations: int = 40, stream: int | None = None,
               use_blur: bool = False):
    """Colour stops whose render of `params` comes closest to `target` in least squares, for the curves, u lists, weights
    and exponents of `d` (HostScene.to_numpy() layout, the scene `scene` was built from). target: float32 [rows, W, 3|4],
    numpy or torch, the band of `params`; NaN pixels are ignored. A p is Scene.update_stops + Scene.render, A^T r is
    Scene.color_adjoint (fit_stops). use_blur: fit the blurred frame instead, exactly what rdc_render_frame_to_host(params,
    use_blur=1) writes: A p is followed by gaussian_blur with the render's blur map, and A^T r starts with
    gaussian_blur_adjoint. During the fit the handle holds the search directions (zeros in the fixed entries); on return it
    holds the fitted stops. Returns (fitted copy of d, residual norm of every iteration). `stream` must be torch's current
    stream (the default): the residuals are formed there."""
    import torch

    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    render, adjoint = _color_operator(scene, d, params, use_blur, stream)
    target = torch.as_tensor(target, dtype=torch.float32, device=torch.device("cuda", torch.cuda.current_device()))
    fitted, residuals = fit_stops(d, target, render, adjoint, iterations)
    scene.update_stops(arrays_from_numpy(fitted), stream)
    return fitted, residuals


def projected_descent(f_and_grad, x0, lower, iterations: int):
    """Minimise f over x >= lower by projected gradient descent, in float64 on numpy arrays. f_and_grad(x) -> (f, gradient).
    Each iteration steps to P(x - alpha g) (P clips to the bound) with alpha the Barzilai-Borwein length s.s / s.y of the
    last step (the first from the gradient's largest entry), and backtracks along that direction until Armijo's condition
    f(x + t d) <= f(x) + 1e-4 t g.d holds. A trial whose f is NaN or larger is never taken, so the objective never increases.
    Stops early when the projected step is zero (x is stationary: a zero gradient returns the start) or 40 halvings find no
    decrease. Returns (x, objectives): objectives[0] is f at the projected start, objectives[k] f after iteration k."""
    lower = np.asarray(lower, np.float64)
    x = np.maximum(np.array(x0, np.float64), lower)
    f, g = f_and_grad(x)
    g = np.asarray(g, np.float64)
    objectives = [float(f)]
    peak = float(np.abs(g).max()) if g.size else 0.0
    alpha = 1.0 / peak if peak > 0.0 else 1.0
    for _ in range(iterations):
        d = np.maximum(x - alpha * g, lower) - x
        slope = float(g @ d)
        if not np.any(d) or not slope < 0.0:
            break
        t = 1.0
        for _ in range(40):
            x_new = np.maximum(x + t * d, lower)
            f_new, g_new = f_and_grad(x_new)
            if f_new <= f + 1e-4 * t * slope:
                break
            t *= 0.5
        else:
            break
        g_new = np.asarray(g_new, np.float64)
        s, y = x_new - x, g_new - g
        sy = float(s @ y)
        if sy > 0.0:
            alpha = min(max(float(s @ s) / sy, 1e-30), 1e30)
        elif np.any(g_new):  # no curvature along the step: restart from the gradient's scale
            alpha = 1.0 / float(np.abs(g_new).max())
        x, f, g = x_new, f_new, g_new
        objectives.append(float(f))
    return x, objectives


def _fit_band(frame: _BandFrame, d: dict, target, stops, gradient, x0, lower, iterations: int):
    """Minimises 1/2 ||frame.forward(**stops(x)) - target||^2 over x >= lower with projected_descent, then puts the fitted
    stops on the handle. target: float32 [rows, W, 3|4], numpy or torch; pixels NaN in the target or in the start's frame
    are ignored. gradient(x, g) -> the objective's gradient in x for g, float32 [rows, W, 4], whose RGB holds the residual
    (.w zero). A trial whose objective is not finite gets no gradient: projected_descent refuses it without reading one.
    Returns (fitted copy of d, objective of every iteration)."""
    import torch

    target3 = torch.as_tensor(target, dtype=torch.float32, device=frame.dev)[..., :3].to(torch.float64)

    def frame3(x):
        return frame.forward(**stops(x))[..., :3].to(torch.float64)

    keep = ~(torch.isnan(frame3(x0)).any(-1) | torch.isnan(target3).any(-1))[..., None]
    grad_image = torch.zeros_like(frame.image)

    def f_and_grad(x):
        r = torch.where(keep, frame3(x) - target3, torch.zeros((), dtype=torch.float64, device=frame.dev))
        f = 0.5 * float((r * r).sum())
        if not np.isfinite(f):
            return f, np.full_like(x, np.nan)
        grad_image[..., :3] = r
        return f, gradient(x, grad_image)

    x, objectives = projected_descent(f_and_grad, x0, lower, iterations)
    fitted = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in d.items()}
    fitted.update(stops(x))
    frame.scene.update_stops(arrays_from_numpy(fitted), frame.stream)
    return fitted, objectives


def fit_blur(scene: "Scene", d: dict, params: FrameParams, target, iterations: int = 30, stream: int | None = None):
    """Blur stops whose blurred render of `params` comes closest to `target`: minimises 1/2 ||blurred frame - target||^2 over
    the real blur stops (j < n_blur), each >= 0, with the curves, colours, u lists, weights and exponents of `d`
    (HostScene.to_numpy() layout, the scene `scene` was built from) fixed. The blurred frame is exactly what
    rdc_render_frame_to_host(params, use_blur=1) writes. target: float32 [rows, W, 3|4], numpy or torch, the band of
    `params`; pixels NaN in the target or in the blurred frame of the start are ignored. Padding and sentinels keep d's values.
    One evaluation is update_stops, render (with the max_sigma flag), gaussian_blur of the band as its own buffer, the
    residual, gaussian_blur_sigma_adjoint and Scene.blur_adjoint; projected_descent drives them.
    The objective is not convex, and its gradient vanishes as sigma -> 0: the outer taps weigh g'(+-1) = 2 sigma^-3 e^{-1/sigma^2}.
    A stop that starts at 0 stays there, so start from a nonzero blur (a constant 1 px does). The tap count steps where
    ceil(3 sigma) does; the line search absorbs those small jumps. Returns (fitted copy of d, objective of every iteration);
    on return the handle holds the fitted stops. `stream` must be torch's current stream (the default)."""
    import torch

    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    frame = _BandFrame(scene, d, params, True, stream)
    nb = int(d["n_blur"])
    base = np.asarray(d["blur"], np.float32)
    grad_blur = torch.empty(base.shape, dtype=torch.float64, device=frame.dev)

    def stops(x):
        b = base.copy()
        b[:nb] = x
        return {"blur": b}

    def gradient(x, g):
        scene.blur_adjoint(params, frame.sigma_adjoint(g).data_ptr(), grad_blur.data_ptr(), stream)
        return grad_blur[:nb].cpu().numpy()

    return _fit_band(frame, d, target, stops, gradient, base[:nb].astype(np.float64), np.zeros(nb), iterations)


def weight_unknowns(d: dict):
    """The unknowns of fit_weights for a scene laid out like HostScene.to_numpy(): the real weight stops (j < n_weight) that
    are > 0, as log(weight), then the real exponent stops (j < n_weight_degree), raw. Returns (x0, lower, stops, chain):
    x0 the start and lower the bounds (-inf for the logs, min(0, start) for the exponents), float64; stops(x) -> (weight,
    weight_degree), float32 arrays laid out like d's in which every other entry (weights <= 0, padding, sentinels) keeps d's
    value; chain(x, grad_weight, grad_weight_degree) -> the gradient in x of a loss whose gradient in the two arrays is given
    (weight * dL/dweight for the logs). With log weights the weights stay positive, and scaling them all, which leaves the
    frame unchanged, is a shift of the logs that the fit never needs to resolve."""
    nw, ne = int(d["n_weight"]), int(d["n_weight_degree"])
    base_w = np.asarray(d["weight"], np.float32)
    base_e = np.asarray(d["weight_degree"], np.float32)
    free = np.flatnonzero(base_w[:nw] > 0)
    k = free.size
    x0 = np.concatenate([np.log(base_w[free].astype(np.float64)), base_e[:ne].astype(np.float64)])
    lower = np.concatenate([np.full(k, -np.inf), np.minimum(0.0, base_e[:ne].astype(np.float64))])

    def stops(x):
        weight, degree = base_w.copy(), base_e.copy()
        weight[free] = np.exp(x[:k])
        degree[:ne] = x[k:]
        return weight, degree

    def chain(x, grad_weight, grad_degree):
        weight = stops(x)[0][free].astype(np.float64)
        return np.concatenate([weight * np.asarray(grad_weight, np.float64)[free], np.asarray(grad_degree, np.float64)[:ne]])

    return x0, lower, stops, chain


def fit_weights(scene: "Scene", d: dict, params: FrameParams, target, iterations: int = 30, stream: int | None = None,
                use_blur: bool = False):
    """Weight and exponent stops whose render of `params` comes closest to `target`: minimises 1/2 ||frame - target||^2 over
    the unknowns of weight_unknowns(d) with projected_descent, the curves, colours, blur and u lists of `d`
    (HostScene.to_numpy() layout, the scene `scene` was built from) fixed. target: float32 [rows, W, 3|4], numpy or torch,
    the band of `params`; pixels NaN in the target or in the start's frame are ignored, and a step that makes a kept pixel
    NaN (all its weights driven to 0) has a NaN objective, which the line search refuses. One evaluation is update_stops,
    render, the residual and Scene.weight_adjoint with the image gradient. use_blur: fit the blurred frame instead, exactly
    what rdc_render_frame_to_host(params, use_blur=1) writes; the weights move both the image and the blur map, so the
    gradient is gaussian_blur_adjoint and gaussian_blur_sigma_adjoint of the residual, then Scene.weight_adjoint with both.
    Returns (fitted copy of d, objective of every iteration); on return the handle holds the fitted stops. `stream` must be
    torch's current stream (the default)."""
    import torch

    if stream is None:
        stream = torch.cuda.current_stream().cuda_stream
    frame = _BandFrame(scene, d, params, use_blur, stream)
    x0, lower, stops, chain = weight_unknowns(d)
    grad_weight = torch.empty(np.asarray(d["weight"]).shape, dtype=torch.float64, device=frame.dev)
    grad_degree = torch.empty(np.asarray(d["weight_degree"]).shape, dtype=torch.float64, device=frame.dev)

    def gradient(x, g):
        grad_image = frame.transpose(g).data_ptr()
        grad_sigma = frame.sigma_adjoint(g).data_ptr() if use_blur else 0
        scene.weight_adjoint(params, grad_image, grad_sigma, grad_weight.data_ptr(), grad_degree.data_ptr(), stream)
        return chain(x, grad_weight.cpu().numpy(), grad_degree.cpu().numpy())

    return _fit_band(frame, d, target, lambda x: dict(zip(("weight", "weight_degree"), stops(x))), gradient, x0, lower,
                     iterations)


def view_pixel_to_scene(params: FrameParams, ix: int, iy: int) -> tuple[float, float]:
    """rdc_view_pixel_to_scene: the scene point Scene.pick_frame picks for pixel (ix, iy), e.g. under a cursor click."""
    x, y = C.c_float(), C.c_float()
    _check(_lib.rdc_view_pixel_to_scene(C.byref(params), ix, iy, C.byref(x), C.byref(y)), "rdc_view_pixel_to_scene")
    return x.value, y.value


def image_to_rgba8(image: np.ndarray, flip: bool) -> np.ndarray:
    h, w, _ = image.shape
    img = np.ascontiguousarray(image, np.float32)
    out = np.empty((h, w, 4), np.uint8)
    _check(_lib.rdc_image_to_rgba8(img.ctypes.data, w, h, int(flip), out.ctypes.data), "rdc_image_to_rgba8")
    return out


def psnr(a: np.ndarray, b: np.ndarray) -> tuple[float, float]:
    """rdc_psnr on two [H, W, 4] float images: (PSNR in dB, largest absolute RGB difference)."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    assert a.shape == b.shape and a.shape[-1] == 4
    p, m = C.c_double(), C.c_double()
    _check(_lib.rdc_psnr(a.ctypes.data, b.ctypes.data, a.size // 4, C.byref(p), C.byref(m)), "rdc_psnr")
    return p.value, m.value


def row_band(height: int, rank: int, world: int) -> tuple[int, int]:
    """Rows [begin,end) of rank `rank` of `world`: contiguous bands, remainder spread over the first ranks."""
    base, rem = divmod(height, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def cuda_callbacks(scene: "Scene", make_params, stream: int = 0):
    """(render_strips, blur_rows) for distributed.render_frame, bound to the CUDA entry points.
    make_params() -> FrameParams of the frame being rendered (whole image; the strip fields are set here)."""

    def render_strips(image, sigma, stride, offset):
        p = make_params()
        p.strip_stride, p.strip_offset = (stride, offset) if stride > 1 else (0, 0)
        scene.render(p, image.data_ptr(), sigma.data_ptr(), stream)

    def blur_rows(dest, source, sigma, scratch, height, row_begin, row_end, halo):
        dest_ptr = dest if isinstance(dest, int) else dest.data_ptr()  # an address: a frame in a peer's memory
        gaussian_blur_band(dest_ptr, source.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), source.shape[1], height,
                           row_begin, row_end, halo, 0, stream)

    return render_strips, blur_rows
