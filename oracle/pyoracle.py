"""TEST INFRASTRUCTURE — Python face of the CPU oracle.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / ``--impl reference`` legs import this
module. The product package never does.

Two things live here:

* ``ingest_xml`` — an independent restatement of the reference's XML loader (optixHello.cpp:212-515 and
  helpers :1302-1386) in Python: different language, different XML parser (xml.etree) and a literal,
  list-appending transcription of the reference's control flow, so that it checks the product's C++ ingest
  rather than sharing code with it. float32 arithmetic is reproduced with numpy scalars in the reference's
  operand order.
* ``Oracle`` — ctypes binding of ``oracle/_build/liboracle_port.so`` (the restated device logic,
  oracle_port.cpp) and, when present, ``oracle/_ref/libref_oracle.so`` (the reference's own DeviceCode.cu
  compiled for the host, ref_glue.cpp).
"""
from __future__ import annotations

import ctypes as C
import os
import struct
import subprocess
import xml.etree.ElementTree as ET

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_LIB = os.path.join(HERE, "_build", "liboracle_port.so")
REF_LIB = os.path.join(HERE, "_ref", "libref_oracle.so")
REF_XML_DUMP = os.path.join(HERE, "_ref", "ref_xml_dump")
REF_INGEST_LIB = os.path.join(HERE, "_ref", "libref_ingest.so")
REF_BLUR_LIB = os.path.join(HERE, "_ref", "libref_blur.so")

f32 = np.float32


# --------------------------------------------------------------------------------------------------
# ingest (optixHello.cpp:212-515, 1302-1386)
# --------------------------------------------------------------------------------------------------
def _atof(s: str) -> float:
    """C atof: longest numeric prefix, 0.0 if none."""
    s = s.strip()
    import re

    m = re.match(r"[+-]?(\d+\.?\d*([eE][+-]?\d+)?|\.\d+([eE][+-]?\d+)?|inf(inity)?|nan)", s, re.I)
    return float(m.group(0)) if m else 0.0


def _atoi(s: str) -> int:
    import re

    m = re.match(r"\s*[+-]?\d+", s)
    return int(m.group(0)) if m else 0


def _inv_sqrt(number: np.float32) -> np.float32:
    # optixHello.cpp:1372-1386
    x2 = f32(number * f32(0.5))
    i = struct.unpack("<I", struct.pack("<f", float(number)))[0]
    i = (0x5F3759DF - (i >> 1)) & 0xFFFFFFFF
    y = f32(struct.unpack("<f", struct.pack("<I", i))[0])
    return f32(y * f32(f32(1.5) - f32(f32(x2 * y) * y)))


def _bezier_tangent(t, v):
    # optixHello.cpp:1354-1357, float arithmetic, left to right
    t = f32(t)
    a3 = f32(f32(f32(3) * t) * t)
    a0 = f32(f32(f32(f32(f32(-3) * t) * t) + f32(f32(6) * t)) - f32(3))
    a1 = f32(f32(f32(f32(f32(9) * t) * t) - f32(f32(12) * t)) + f32(3))
    a2 = f32(f32(f32(f32(-9) * t) * t) + f32(f32(6) * t))

    def comp(k):
        r = f32(a3 * v[3][k])
        r = f32(r + f32(v[0][k] * a0))
        r = f32(r + f32(v[1][k] * a1))
        r = f32(r + f32(v[2][k] * a2))
        return r

    return comp(0), comp(1)


_M = [[6, -7, 2, 0], [0, 2, -1, 0], [0, -1, 2, 0], [0, 2, -7, 6]]


def _correct_control_points(xy, vertices):
    # optixHello.cpp:1335-1343
    for i in range(4):
        row = []
        for k in (0, 1):
            r = f32(xy[0][k] * f32(_M[i][0]))
            r = f32(r + f32(xy[1][k] * f32(_M[i][1])))
            r = f32(r + f32(xy[2][k] * f32(_M[i][2])))
            r = f32(r + f32(xy[3][k] * f32(_M[i][3])))
            row.append(r)
        vertices.append((row[0], row[1], f32(0)))


def _endcap_points(endpoint, tangent, size: int):
    # optixHello.cpp:1360-1369
    norm = _inv_sqrt(f32(f32(tangent[0] * tangent[0]) + f32(tangent[1] * tangent[1])))
    cos = f32(tangent[1] * norm)
    sin = f32(f32(-tangent[0]) * norm)
    sz = f32(size)
    p1 = (f32(f32(f32(f32(-cos) - sin) * sz) + endpoint[0]), f32(f32(f32(f32(-sin) + cos) * sz) + endpoint[1]))
    p2 = (f32(f32(f32(cos - sin) * sz) + endpoint[0]), f32(f32(f32(sin + cos) * sz) + endpoint[1]))
    return p1, p2


def ingest_xml(path: str, use_diffusion_curve_save: bool = True, default_weight_degree: float = 0.5,
               endcap_size: float = 8.0) -> dict:
    """Returns the same dictionary layout as raytracingdiffusioncurves_b200.api.HostScene.to_numpy()."""
    orzan = bool(use_diffusion_curve_save)
    with open(path, "rb") as fh:
        root = ET.fromstring(fh.read())
    width = _atoi(root.attrib["image_width"])
    height = _atoi(root.attrib["image_height"])
    ax0, ax1 = ("y", "x") if orzan else ("x", "y")

    def point(node):
        return (f32(f32(_atof(node.attrib[ax0])) - f32(width // 2)), f32(f32(_atof(node.attrib[ax1])) - f32(height // 2)))

    vertices, curve_map, curve_map_inverse, curve_index, curve_connect, segment_indices = [], [], [], [], [], []
    fam = {k: {"index": [], "value": [], "u": []} for k in ("color_left", "color_right", "blur", "weight", "weight_degree")}
    current_segment = 0
    n_segments = 0
    totals = {k: 0 for k in fam}

    def stop_u(node, use_endcap):
        return f32(_atof(node.attrib["globalID"]) / float(f32(10.0)) + (1.0 if use_endcap else 0.0))

    for current_curve, curve in enumerate(list(root)):
        current_curve_segment = 0
        nodes = list(curve.find("control_points_set"))
        use_endcap = curve.attrib.get("use_endcap", "") == "true"
        curve_connect.append(int(curve.attrib["connects"]) if "connects" in curve.attrib else -1)
        curve_map_inverse.append(n_segments)

        def add_segment():
            nonlocal current_segment, current_curve_segment
            segment_indices.append(current_segment)
            current_segment += 4
            curve_map.append(current_curve)
            curve_index.append(current_curve_segment)
            current_curve_segment += 1

        if use_endcap:
            first = [point(n) for n in nodes[:4]]
            tan = _bezier_tangent(1e-3, first)
            tan = (f32(-tan[0]), f32(-tan[1]))
            p1, p2 = _endcap_points(first[0], tan, int(endcap_size))
            _correct_control_points([first[0], p1, p2, first[0]], vertices)
            add_segment()
        i = 0
        while i + 1 < len(nodes):  # while (current_node->next_sibling())
            _correct_control_points([point(n) for n in nodes[i:i + 4]], vertices)
            i += 3
            add_segment()
        if use_endcap:
            last4 = [point(n) for n in nodes[-4:]]
            tan = _bezier_tangent(1 - 1e-3, last4)
            p1, p2 = _endcap_points(last4[3], tan, int(endcap_size))
            _correct_control_points([last4[3], p1, p2, last4[3]], vertices)
            add_segment()

        # colours (:333-410)
        L, R = fam["color_left"], fam["color_right"]
        L["index"].append([totals["color_left"], 0])
        zero = (f32(0), f32(0), f32(0))
        if use_endcap:
            R["value"] += [zero, zero]
            L["value"] += [zero, zero]
            R["u"] += [f32(0), f32(1)]
            L["u"] += [f32(0), f32(1)]

        def push_color(node, F):
            c = (f32(f32(_atoi(node.attrib["B" if orzan else "R"])) / f32(255.0)),
                 f32(f32(_atoi(node.attrib["G"])) / f32(255.0)),
                 f32(f32(_atoi(node.attrib["R" if orzan else "B"])) / f32(255.0)))
            F["value"].append(c)
            F["u"].append(stop_u(node, use_endcap))
            F["index"][-1][1] += 1

        for node in list(curve.find("left_colors_set")):
            push_color(node, L)
        R["index"].append([totals["color_right"], 0])
        for node in list(curve.find("right_colors_set")):
            push_color(node, R)
        if orzan:
            close_u = f32(current_curve_segment - (1 if use_endcap else 0))
            R["value"].append(R["value"][-1]); R["index"][-1][1] += 1; R["u"].append(close_u)
            L["value"].append(L["value"][-1]); L["index"][-1][1] += 1; L["u"].append(close_u)
        if use_endcap:
            lx, rx = L["index"][-1][0], R["index"][-1][0]
            L["value"][lx] = L["value"][lx + 2]
            L["value"][lx + 1] = R["value"][rx + 2]
            L["index"][-1][1] += 2
            R["value"][rx] = L["value"][lx + 2]
            R["value"][rx + 1] = R["value"][rx + 2]
            R["index"][-1][1] += 2
            L["value"].append(R["value"][-1])
            L["value"].append(L["value"][len(L["value"]) - 2])
            L["index"][-1][1] += 2
            R["value"].append(R["value"][-1])
            R["value"].append(L["value"][len(L["value"]) - 3])
            R["index"][-1][1] += 2
            R["u"] += [f32(current_curve_segment - 1), f32(current_curve_segment)]
            L["u"] += [f32(current_curve_segment - 1), f32(current_curve_segment)]
        totals["color_left"] += L["index"][-1][1]
        totals["color_right"] += R["index"][-1][1]

        # blur / weight / exponent (:414-511)
        def scalar(name, set_name, attr, default):
            F = fam[name]
            F["index"].append([totals[name], 0])
            set_node = curve.find(set_name)
            if set_node is not None:
                if use_endcap:
                    F["value"].append(f32(0 if default is None or name == "weight" else default))
                    F["u"].append(f32(0))
                    F["index"][-1][1] += 1
                for node in list(set_node):
                    F["value"].append(f32(_atof(node.attrib[attr])))
                    F["u"].append(stop_u(node, use_endcap))
                    F["index"][-1][1] += 1
                if use_endcap:
                    F["value"][F["index"][-1][0]] = F["value"][F["index"][-1][0] + 1]
                    F["value"].append(F["value"][-1])
                    F["u"].append(f32(current_curve_segment))
                    F["index"][-1][1] += 1
            else:
                if default is None:
                    raise ValueError("curve without blur_points_set")
                F["value"] += [f32(default), f32(default)]
                F["u"] += [f32(0), f32(current_curve_segment)]
                F["index"][-1][1] += 2
            totals[name] += F["index"][-1][1]

        scalar("blur", "blur_points_set", "value", None)
        scalar("weight", "weight_set", "w", 1.0)
        scalar("weight_degree", "weight_degree_set", "w", default_weight_degree)
        n_segments += current_curve_segment

    out = {
        "image_width": width, "image_height": height,
        "vertices": np.array(vertices, np.float32).reshape(-1, 3),
        "segment_indices": np.array(segment_indices, np.uint32),
        "curve_map": np.array(curve_map, np.uint32),
        "curve_index": np.array(curve_index, np.uint32),
        "curve_connect": np.array(curve_connect, np.int32),
        "curve_map_inverse": np.array(curve_map_inverse, np.uint32),
    }
    colour_len = max(len(fam["color_left"]["u"]), len(fam["color_right"]["u"])) + 2
    for name, F in fam.items():
        n = len(F["u"])
        padded = colour_len if name.startswith("color") else n + 2
        u = np.full((padded,), np.inf, np.float32)
        u[:n] = np.array(F["u"], np.float32)
        if name.startswith("color"):
            v = np.zeros((padded, 3), np.float32)
            v[:n] = np.array(F["value"], np.float32).reshape(-1, 3)
        else:
            v = np.zeros((padded,), np.float32)
            v[:n] = np.array(F["value"], np.float32)
        out["n_" + name] = n
        out[name + "_index"] = np.array(F["index"], np.uint32).reshape(-1, 2)
        out[name] = v
        out[name + "_u"] = u
    return out


# --------------------------------------------------------------------------------------------------
# ctypes structs (layout of include/rdc_b200.h; declared here so the oracle does not import the product)
# --------------------------------------------------------------------------------------------------
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
f32p = C.POINTER(C.c_float)


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


def arrays_from_dict(d: dict):
    """SceneArrays view over a dictionary of numpy arrays (keeps the arrays alive through the return)."""
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
    for fam in ("color_left", "color_right", "blur", "weight", "weight_degree"):
        setattr(a, "n_" + fam, int(d["n_" + fam]))
        setattr(a, fam + "_index", ptr(fam + "_index", np.uint32, C.c_uint32))
        setattr(a, fam, ptr(fam, np.float32, C.c_float))
        setattr(a, fam + "_u", ptr(fam + "_u", np.float32, C.c_float))
    return a, keep


# oracle_port.cpp RayRecord: what a primary ray decided
RAY_RECORD = np.dtype([("id", np.uint32), ("t", np.float32), ("segment_u", np.float32), ("curve", np.uint32),
                       ("curve_u", np.float32), ("right", np.int32), ("portal", np.int32)])
MISS = 0xFFFFFFFF


def make_params(width, height, rays_per_pixel, **kw) -> FrameParams:
    p = FrameParams()
    p.image_width, p.image_height = width, height
    p.number_of_rays_per_pixel = float(rays_per_pixel)
    p.zoom_factor, p.offset_x, p.offset_y = 1.0, 0.0, 0.0
    p.frame, p.seed = 0, 0
    p.row_begin, p.row_end = 0, height
    p.use_diffusion_curve_save, p.use_aa, p.max_trace_depth = 1, 1, 2
    p.traversal = 0
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def make_accel(curve_width=1e-3, flatness_tolerance=0.05, max_chords_per_segment=1024) -> AccelOptions:
    return AccelOptions(curve_width, flatness_tolerance, max_chords_per_segment, 0, 0, 0)


def build(verbose: bool = False) -> None:
    """Compile the oracle(s): always the port; the _ref pair only where /root/reference exists."""
    r = subprocess.run(["make", "-C", HERE], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout)


class Oracle:
    """kind = 'port' (oracle_port.cpp) or 'reference' (the reference's DeviceCode.cu through oracle/shim)."""

    def __init__(self, kind: str = "port"):
        self.kind = kind
        path = PORT_LIB if kind == "port" else REF_LIB
        if not os.path.exists(path):
            if kind == "port":
                build()
            if not os.path.exists(path):
                raise FileNotFoundError(path)
        self.lib = C.CDLL(path)
        sig = [C.POINTER(SceneArrays), C.POINTER(AccelOptions), C.POINTER(FrameParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        self._render = self.lib.oracle_render if kind == "port" else self.lib.ref_render
        self._render.argtypes = sig
        self._render.restype = C.c_int
        self._threads = self.lib.oracle_threads if kind == "port" else self.lib.ref_threads
        self._threads.restype = C.c_int
        self._set_search = self.lib.oracle_set_search if kind == "port" else self.lib.ref_set_search
        self._set_search.argtypes = [C.c_int]
        if kind == "port":
            self.lib.oracle_chords.argtypes = [C.POINTER(SceneArrays), C.POINTER(AccelOptions), C.c_void_p, C.c_void_p, u32p]
            self.lib.oracle_blur.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]

    @staticmethod
    def reference_available() -> bool:
        return os.path.exists(REF_LIB)

    def threads(self) -> int:
        return int(self._threads())

    def render(self, scene: dict, params: FrameParams, accel: AccelOptions | None = None, want_hits: bool = False,
               threads: int = 0, search: str = "brute"):
        """search: 'brute' tests every chord per ray; 'grid' narrows the candidates with a uniform grid first (same
        closest hit, bit for bit — tests/test_oracle_cpu.py — and the only way through scenes of a million chords)."""
        self._set_search({"brute": 0, "grid": 1}[search])
        accel = accel or make_accel()
        a, keep = arrays_from_dict(scene)
        rows = params.row_end - params.row_begin
        w = params.image_width
        n_iter = int(np.ceil(params.number_of_rays_per_pixel))
        image = np.zeros((rows, w, 4), np.float32)
        blur_map = np.zeros((rows, w), np.float32)
        hits = np.zeros((rows, w, n_iter), np.uint32) if want_hits else None
        rc = self._render(C.byref(a), C.byref(accel), C.byref(params), image.ctypes.data, blur_map.ctypes.data,
                          hits.ctypes.data if want_hits else None, threads)
        if rc != 0:
            raise RuntimeError(f"{self.kind} oracle render returned {rc}")
        del keep
        return image, blur_map, hits

    def ray_records(self, scene: dict, params: FrameParams, accel: AccelOptions | None = None, search: str = "grid",
                    threads: int = 0) -> np.ndarray:
        """The primary rays of the band as render() traces them (Philox draws, rotation, jitter, closest hit): a RAY_RECORD
        array [rows, W, ceil(N)] laid out like render()'s hit ids, with the chord, t, segment_u, curve, curve_u, side and
        whether the curve is a portal. Everything downstream of these decisions (stops, weights, the frame) is left to the
        caller."""
        assert self.kind == "port"
        self._set_search({"brute": 0, "grid": 1}[search])
        accel = accel or make_accel()
        a, keep = arrays_from_dict(scene)
        stride = params.strip_stride if params.strip_stride > 1 else 1
        rows = sum(1 for iy in range(params.row_begin, params.row_end)
                   if ((iy - params.row_begin) // 8) % stride == (params.strip_offset if stride > 1 else 0))
        out = np.zeros((rows, params.image_width, int(np.ceil(params.number_of_rays_per_pixel))), RAY_RECORD)
        self.lib.oracle_ray_records.argtypes = [C.POINTER(SceneArrays), C.POINTER(AccelOptions), C.POINTER(FrameParams),
                                                C.c_void_p, C.c_int]
        rc = self.lib.oracle_ray_records(C.byref(a), C.byref(accel), C.byref(params), out.ctypes.data, threads)
        if rc != 0:
            raise RuntimeError(f"oracle_ray_records returned {rc}")
        del keep
        return out

    def trace_rays(self, scene: dict, rays: np.ndarray, accel: AccelOptions | None = None, search: str = "brute"):
        """Closest hit of n primary rays (rays[n,4] = ox, oy, dx, dy): (chord id, t, segment parameter u)."""
        assert self.kind == "port"
        self._set_search({"brute": 0, "grid": 1}[search])
        accel = accel or make_accel()
        a, keep = arrays_from_dict(scene)
        rays = np.ascontiguousarray(rays, np.float32)
        n = len(rays)
        ids, t, u = np.empty(n, np.uint32), np.empty(n, np.float32), np.empty(n, np.float32)
        self.lib.oracle_trace_rays.argtypes = [C.POINTER(SceneArrays), C.POINTER(AccelOptions), C.c_void_p, C.c_uint32, C.c_void_p,
                                               C.c_void_p, C.c_void_p]
        self.lib.oracle_trace_rays(C.byref(a), C.byref(accel), rays.ctypes.data, n, ids.ctypes.data, t.ctypes.data, u.ctypes.data)
        del keep
        return ids, t, u

    def chords(self, scene: dict, accel: AccelOptions | None = None):
        assert self.kind == "port"
        accel = accel or make_accel()
        a, keep = arrays_from_dict(scene)
        n = C.c_uint32()
        self.lib.oracle_chords(C.byref(a), C.byref(accel), None, None, C.byref(n))
        geom = np.empty((n.value, 4), np.float32)
        ids = np.empty((n.value, 3), np.uint32)
        self.lib.oracle_chords(C.byref(a), C.byref(accel), geom.ctypes.data, ids.ctypes.data, C.byref(n))
        del keep
        return geom, ids

    def blur(self, image: np.ndarray, sigma: np.ndarray, threads: int = 0) -> np.ndarray:
        assert self.kind == "port"
        h, w, _ = image.shape
        src = np.ascontiguousarray(image, np.float32)
        sig = np.ascontiguousarray(sigma, np.float32)
        out = np.empty_like(src)
        self.lib.oracle_blur(out.ctypes.data, src.ctypes.data, sig.ctypes.data, w, h, threads)
        return out


def ref_ingest(path: str) -> dict:
    """The reference's OWN ingest loop (optixHello.cpp:108-117,170-515 and helpers :1302-1386, cut out and compiled for the
    host by oracle/ref_extract.sh) run on `path`. Same dictionary layout as ingest_xml, WITHOUT the +INF sentinels the
    product appends (the reference has none). Compiled with the reference's USE_DIFFUSION_CURVE_SAVE (true)."""
    lib = C.CDLL(REF_INGEST_LIB)
    lib.ref_ingest.argtypes = [C.c_char_p]
    lib.ref_ingest_array.argtypes = [C.c_char_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.ref_ingest_array.restype = C.c_void_p
    if lib.ref_ingest(os.fsencode(path)) != 0:
        raise RuntimeError(f"the reference's ingest failed on {path}")

    def arr(name, dtype, cols):
        n, eb = C.c_size_t(), C.c_size_t()
        ptr = lib.ref_ingest_array(name.encode(), C.byref(n), C.byref(eb))
        assert n.value != 2 ** 64 - 1, name
        if n.value == 0:
            return np.zeros((0, cols) if cols > 1 else (0,), dtype)
        flat = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(n.value * eb.value,)).copy().view(dtype)
        return flat.reshape(n.value, cols) if cols > 1 else flat

    w, h = C.c_int(), C.c_int()
    lib.ref_ingest_size(C.byref(w), C.byref(h))
    out = {"image_width": w.value, "image_height": h.value, "vertices": arr("vertices", np.float32, 3),
           "segment_indices": arr("segmentIndices", np.uint32, 1), "curve_map": arr("curve_map", np.uint32, 1),
           "curve_index": arr("curve_index", np.uint32, 1), "curve_connect": arr("curve_connect", np.int32, 1),
           "curve_map_inverse": arr("curve_map_inverse", np.uint32, 1)}
    for fam in ("color_left", "color_right", "blur", "weight", "weight_degree"):
        out[fam + "_index"] = arr(fam + "_index", np.uint32, 2)
        out[fam] = arr(fam, np.float32, 3 if fam.startswith("color") else 1)
        out[fam + "_u"] = arr(fam + "_u", np.float32, 1)
        out["n_" + fam] = len(out[fam + "_u"])
    return out


def ref_blur(image: np.ndarray, sigma: np.ndarray, threads: int = 0) -> np.ndarray:
    """The reference's OWN gaussHorizontal / gaussVertical (helperKernels.cu:48-134, cut out and compiled for the host by
    oracle/ref_extract.sh), through the launcher sequence of :137-148."""
    lib = C.CDLL(REF_BLUR_LIB)
    lib.ref_blur.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    h, w, _ = image.shape
    src = np.ascontiguousarray(image, np.float32)
    sig = np.ascontiguousarray(sigma, np.float32)
    out = np.empty_like(src)
    lib.ref_blur(out.ctypes.data, src.ctypes.data, sig.ctypes.data, w, h, threads)
    return out


def ref_extracts_available() -> bool:
    return os.path.exists(REF_INGEST_LIB) and os.path.exists(REF_BLUR_LIB)


def ref_xml_dump(path: str) -> str:
    r = subprocess.run([REF_XML_DUMP, path], capture_output=True)
    if r.returncode != 0:
        raise RuntimeError(r.stderr.decode())
    return r.stdout.decode("utf-8", "replace")


def psnr(a: np.ndarray, b: np.ndarray) -> float:
    m = np.isfinite(a) & np.isfinite(b)
    mse = float(np.mean((a[m].astype(np.float64) - b[m].astype(np.float64)) ** 2)) if m.any() else 0.0
    return float("inf") if mse == 0 else 10.0 * np.log10(1.0 / mse)
