"""Builds and calls tests/probes/rdc_math_probe.cu, the test probe for csrc/rdc_math.h.

The probe is compiled with the Makefile's own flags (read from the Makefile, so that a change to them is tested too):
NVFLAGS for the device build, CXXFLAGS with -x c++ for its host twin. Both go to a temporary directory; nothing is
written to the tree.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "probes", "rdc_math_probe.cu")

# name -> (input words per row, output words per row)
SHAPES = {
    "philox": (6, 4), "u01": (1, 1), "sincospi": (1, 2), "sincospi_kernel": (1, 2), "spline": (9, 4),
    "is_ray_right": (12, 1), "interp_from": (3, 2), "walk_hint": (3, 1), "lerp": (3, 2), "chord_count": (10, 1),
    "ray_chord": (9, 3), "chord_hit": (9, 3), "inv_dd": (3, 1), "portal_skip": (2, 2), "safe_inv": (1, 1),
    "slab": (8, 2), "point_chord": (6, 4), "point_box_d2": (6, 1), "pixel_centre": (5, 2), "ratio": (2, 1),
    "weight_falloff": (2, 1), "jitter": (4, 2),
}


def make_variable(name):
    """Value of a Makefile variable, expanded by make itself."""
    r = subprocess.run(["make", "-s", "--no-print-directory", "-C", ROOT, "--eval", f"rdcp-print: ; @echo $({name})", "rdcp-print"],
                       capture_output=True, text=True, check=True)
    return r.stdout.split()


def _compile(cmd, out_dir):
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} failed:\n{r.stdout}\n{r.stderr}")


def build_host(out_dir):
    cxx = shutil.which("g++") or "g++"
    so = os.path.join(out_dir, "rdc_math_probe_host.so")
    _compile([cxx, *make_variable("CXXFLAGS"), "-x", "c++", SRC, "-shared", "-o", so], out_dir)
    return so


def build_device(out_dir):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = os.path.join(out_dir, "rdc_math_probe_device.so")
    _compile([nvcc, *make_variable("NVFLAGS"), SRC, "-shared", "-o", so], out_dir)
    return so


def words(a):
    """float32 or integer array -> uint32 words (floats keep their bit patterns)."""
    a = np.asarray(a)
    if a.dtype == np.float32:
        return a.view(np.uint32)
    if a.dtype.kind == "f":
        return a.astype(np.float32).view(np.uint32)
    return a.astype(np.int64).astype(np.uint32)


def rows(*cols):
    """Columns (each float32 or integer) -> an n x k matrix of uint32 words."""
    n = max(np.size(c) for c in cols)
    return np.stack([np.broadcast_to(words(c), (n,)) for c in cols], 1).copy()


# Ray counts at which the ray directions are checked: every N below the culling threshold of 8, the powers of two and
# their neighbours (where the iterated rotation has the most steps to drift), and the largest N the render accepts.
RAY_COUNTS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 16, 31, 33, 64, 100, 128, 255, 256, 257, 512, 1000, 1024, 4096, 16384, 65536]
# jitter draws: the smallest and largest rdc_u01 values, the middle, and the largest below 1
JITTER_U = [2.0 ** -33, 0.5, 1.0 - 2.0 ** -24, 1.0]


def two_over_n(n):
    """render.cu: a.two_over_n = 2 / p.number_of_rays_per_pixel, in float."""
    return np.float32(2.0) / np.float32(n)


def restate_base_dirs(rs, rc, n):
    """k_base_dirs in float32 numpy: (1,0) rotated i times by [[rc, -rs], [rs, rc]]. Every numpy float32 operation
    rounds once and nothing is contracted, so this repeats the kernel's arithmetic exactly."""
    rs, rc = np.float32(rs), np.float32(rc)
    out = np.empty((n, 2), np.float32)
    x, y = np.float32(1.0), np.float32(0.0)
    for i in range(n):
        out[i] = x, y
        x, y = x * rc - y * rs, x * rs + y * rc
    return out


def restate_jitter(base, js, jc):
    """gen_ray: the base directions rotated by (jc, js), in float32."""
    bx, by = base[:, 0], base[:, 1]
    js, jc = np.float32(js), np.float32(jc)
    return np.stack([bx * jc - by * js, bx * js + by * jc], 1)


class Probe:
    """One build of the probe. `run(name, in_words, aux)` -> uint32 output words [n, k]."""

    def __init__(self, path, device):
        self.lib = ctypes.CDLL(path)
        self.device = device
        for name in list(SHAPES) + ["base_dirs"]:
            f = getattr(self.lib, f"rdcp_{name}")
            f.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
            f.restype = ctypes.c_int

    def _call(self, name, n, inp, n_out_words, aux):
        inp = np.ascontiguousarray(inp, np.uint32)
        aux = None if aux is None else np.ascontiguousarray(aux, np.float32)
        if not self.device:
            out = np.zeros(n_out_words, np.uint32)
            rc = getattr(self.lib, f"rdcp_{name}")(n, inp.ctypes.data, out.ctypes.data, None if aux is None else aux.ctypes.data)
            assert rc == 0
            return out
        import torch

        d_in = torch.from_numpy(inp.view(np.int32).reshape(-1)).cuda()
        d_out = torch.zeros(max(n_out_words, 1), dtype=torch.int32, device="cuda")
        d_aux = None if aux is None else torch.from_numpy(aux.reshape(-1)).cuda()
        torch.cuda.synchronize()
        rc = getattr(self.lib, f"rdcp_{name}")(n, d_in.data_ptr(), d_out.data_ptr(), None if d_aux is None else d_aux.data_ptr())
        torch.cuda.synchronize()
        assert rc == 0, f"rdcp_{name}: cudaError {rc}"
        return d_out.cpu().numpy().view(np.uint32)[:n_out_words]

    def run(self, name, inp, aux=None):
        ni, no = SHAPES[name]
        inp = np.asarray(inp, np.uint32).reshape(-1, ni)
        n = len(inp)
        return self._call(name, n, inp, n * no, aux).reshape(n, no)

    def base_dirs(self, two_over_n, n_iter):
        """Base directions of rays 0..n_iter-1 as float32 [n_iter, 2]."""
        inp = rows(np.float32(two_over_n), n_iter)
        return self._call("base_dirs", 1, inp, 2 * n_iter, None).view(np.float32).reshape(n_iter, 2)
