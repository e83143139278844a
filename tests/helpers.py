"""Shared helpers for the parity tests."""
import glob
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
XML_DIR = os.path.join(ROOT, "tests", "golden", "xmls")

# Inputs of the reference-comparison tests; tests/golden/make_golden.py stores the reference's answers to them.
DIFFERENT_VIEW = ("PortalDemo.xml", (48, 36, 24), dict(zoom_factor=9.0, offset_x=13.0, offset_y=-7.5, frame=3, seed=11))
# fille.xml at the pixel scale of a 200x150 frame: its real sigmas, up to 8.4 output pixels
FILLE_BLUR_VIEW = ("DiffusionCurvePack/fille.xml", (64, 48, 8), dict(zoom_factor=512 / 150))


def seeded_blur_input():
    """37x53 image with one all-miss (NaN) pixel; sigmas up to 6, zero below 1.5."""
    rng = np.random.default_rng(5)
    image = rng.random((37, 53, 4), dtype=np.float32)
    sigma = (rng.random((37, 53), dtype=np.float32) * 6.0).astype(np.float32)
    sigma[sigma < 1.5] = 0.0
    image[3, 4, :3] = np.nan
    return image, sigma


def sha_bits(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def ingest_digest(scene: dict) -> dict:
    """Arrays as dtype, shape and sha256 of their bits; counts as they are."""
    return {k: {"dtype": str(v.dtype), "shape": list(v.shape), "sha256": sha_bits(v)} if isinstance(v, np.ndarray) else int(v)
            for k, v in scene.items()}


def reference_checks() -> dict:
    with open(os.path.join(ROOT, "tests", "golden", "reference_checks.json")) as fh:
        return json.load(fh)


def all_scene_files():
    return sorted(glob.glob(os.path.join(XML_DIR, "*.xml")) + glob.glob(os.path.join(XML_DIR, "*", "*.xml")))


def scene_ids():
    return [os.path.relpath(f, XML_DIR) for f in all_scene_files()]


def bits(a: np.ndarray) -> np.ndarray:
    return a.view(np.uint32) if a.dtype == np.float32 else a


def assert_scene_equal(a: dict, b: dict):
    assert set(a) == set(b)
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert a[k].shape == b[k].shape, k
            assert np.array_equal(bits(a[k]), bits(b[k])), k
        else:
            assert a[k] == b[k], k


def copy_params(src, dst_cls):
    """Copy a FrameParams between the oracle's and the product's ctypes classes (same layout)."""
    dst = dst_cls()
    for name, _ in src._fields_:
        setattr(dst, name, getattr(src, name))
    return dst


class GpuRenderer:
    """Drives the product through its C ABI with torch-owned device buffers."""

    def __init__(self, xml_path, orzan=True, accel=None):
        import torch
        from raytracingdiffusioncurves_b200 import api

        self.torch, self.api = torch, api
        self.host = api.HostScene.from_xml_file(xml_path, api.default_ingest_options(use_diffusion_curve_save=int(orzan)))
        self.scene = api.Scene(self.host.arrays, accel, torch.cuda.current_stream().cuda_stream)

    def render(self, params, want_hits=False, blur=False, use_flag=True, want_stats=False):
        torch, api = self.torch, self.api
        rows = params.row_end - params.row_begin
        w = params.image_width
        n_iter = int(np.ceil(params.number_of_rays_per_pixel))
        dev = torch.device("cuda")
        image = torch.empty((rows, w, 4), dtype=torch.float32, device=dev)
        sigma = torch.empty((rows, w), dtype=torch.float32, device=dev)
        hits = torch.empty((rows, w, n_iter), dtype=torch.int32, device=dev) if want_hits else None
        flag = torch.zeros((1,), dtype=torch.float32, device=dev)
        params.hit_ids = hits.data_ptr() if want_hits else None
        params.max_sigma = flag.data_ptr() if use_flag else None
        stats = torch.zeros((9,), dtype=torch.int64, device=dev) if want_stats else None
        if want_stats:
            stats[6:8] = torch.iinfo(torch.int64).max  # launch timeline slots take minima
        params.stats = stats.data_ptr() if want_stats else None  # selects the counting build of the kernel
        stream = torch.cuda.current_stream().cuda_stream
        self.scene.render(params, image.data_ptr(), sigma.data_ptr(), stream)
        blurred = None
        if blur:
            scratch = torch.empty_like(image)
            blurred = torch.empty_like(image)
            api.gaussian_blur(blurred.data_ptr(), image.data_ptr(), sigma.data_ptr(), scratch.data_ptr(), w, rows, 0, rows,
                              flag.data_ptr() if use_flag else 0, stream)
        torch.cuda.synchronize()
        out = {
            "image": image.cpu().numpy(),
            "blur_map": sigma.cpu().numpy(),
            "hits": hits.cpu().numpy().view(np.uint32) if want_hits else None,
            "blurred": blurred.cpu().numpy() if blur else None,
            "max_sigma": float(flag.item()),
            # rays traced, boxes tested, chords tested, hits shaded, rays deferred to the tree, nodes visited by table queries
            "stats": stats.cpu().tolist()[:6] if want_stats else None,
        }
        return out


def curve_xml(points, colour=(255, 64, 0), weights=None, exponents=None) -> str:
    """One curve of the CurveSetXML format: control points as given, two colour stops per side, blur 0 -> 2. `weights` and
    `exponents`, lists of (globalID, value) (u = globalID / 10), add a weight_set and a weight_degree_set; without them the
    curve takes the ingest's defaults (weight 1, exponent 0.5)."""
    pts = "".join(f'<control_point x="{x:.9g}" y="{y:.9g}" />' for x, y in points)
    r, g, b = colour
    stops = "".join(f'<{set_name}>' + "".join(f'<{tag} globalID="{gid:.9g}" w="{v:.9g}" />' for gid, v in given) + f'</{set_name}>'
                    for set_name, tag, given in (("weight_set", "weight", weights), ("weight_degree_set", "weight_degree", exponents))
                    if given is not None)
    return (f'<curve nb_control_points="{len(points)}"><control_points_set>{pts}</control_points_set>'
            f'<left_colors_set><left_color G="{g}" R="{r}" globalID="0" B="{b}" /><left_color G="{b}" R="{g}" globalID="10" B="{r}" />'
            f'</left_colors_set><right_colors_set><right_color G="{r}" R="{b}" globalID="0" B="{g}" />'
            f'<right_color G="{g}" R="{r}" globalID="10" B="{b}" /></right_colors_set>'
            '<blur_points_set><best_scale value="0" globalID="0" /><best_scale value="2" globalID="10" /></blur_points_set>'
            + stops + '</curve>\n')


def straight(ax, ay, bx, by):
    """Control points of a straight segment from a to b (equally spaced, so its chords are one chord)."""
    return [(ax + (bx - ax) * k / 3.0, ay + (by - ay) * k / 3.0) for k in range(4)]


def scene_xml(curves, size=512) -> str:
    return (f'<!DOCTYPE CurveSetXML>\n<curve_set image_width="{size}" image_height="{size}" nb_curves="{len(curves)}">\n'
            + "".join(curves) + "</curve_set>\n")


def dust_curves(n=3000, seed=7, size=512):
    """n straight segments of length 0.02-0.5 scattered over a size x size box: every segment is its own run, so most hits
    land near a corner of its padded box."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        cx, cy = rng.uniform(4, size - 4, 2)
        half, ang = 0.5 * rng.uniform(0.02, 0.5), rng.uniform(0, np.pi)
        dx, dy = half * np.cos(ang), half * np.sin(ang)
        out.append(curve_xml(straight(cx - dx, cy - dy, cx + dx, cy + dy), (k % 256, (7 * k) % 256, (31 * k) % 256)))
    return out


def compare_images(got, want, tol=1e-4):
    """RGB within tol where both finite; NaN pattern identical. Returns (max abs diff, psnr)."""
    g, w = got[..., :3], want[..., :3]
    assert np.array_equal(np.isnan(g), np.isnan(w)), "NaN (all-miss) pixels differ"
    m = ~np.isnan(w)
    d = float(np.max(np.abs(g[m] - w[m]))) if m.any() else 0.0
    mse = float(np.mean((g[m].astype(np.float64) - w[m].astype(np.float64)) ** 2)) if m.any() else 0.0
    psnr = float("inf") if mse == 0 else 10 * np.log10(1.0 / mse)
    assert d <= tol, f"max |rgb diff| {d} > {tol} (psnr {psnr:.1f} dB)"
    return d, psnr
