"""A float64 restatement of the frame and of the render's stop adjoints, downstream of the rays' decisions.

The decisions of a primary ray (which chord it hits, at which t and u, on which side, whether the curve is a portal) come
from the oracle's own ray loop (pyoracle.Oracle.ray_records), bit for bit the render's. Everything after them is restated
here in float64 from the ingested scene dictionary:

* the stop walks of rdc_interp_from, literally: from the curve's start index, step while the next stop's u is below the
  hit's u (fp32 compares on the fp32 lists, so the indices are the kernel's), ratio (u - lo) / (hi - lo) in float64 (a +INF
  sentinel above gives 0, as in fp32);
* the lerped colour, blur, weight multiplier m and exponent e, f = t^-e, w = m f;
* the frame P = sum w c / W, sigma = sum w b / W, with the NaN pixels decided as the render decides them: the fp32 weights
  summed in ray order are zero;
* the vector-Jacobian products for pixel gradients G (RGB) and g_sigma: colour A^T G into left / right by side, blur
  A_b^T g_sigma, and with s = <G, c> + g_sigma b and K = sum w s / W, (1 - rho_w) f (s - K) / W to weight[iw] (rho_w ... to
  iw + 1) and -(1 - rho_e) w ln t (s - K) / W to weight_degree[ie] (rho_e ... to ie + 1). Portal hits shade nothing.

Beside every output entry it returns a bound: the sum over the rays that reach the entry of the magnitude of the ray's term
before its split into (1 - rho) and rho, with each operand replaced by the sum of the absolute values it is made of (a lerp
(1 - rho) a + rho b by (|a| + |b|)(|1 - rho| + |rho|), s by sum |G| |c| + |g_sigma| |b|, K by sum |w| |s| / |W|). The fp32
rounding of any step of the kernel's computation of a term is a small multiple of the unit roundoff times that magnitude,
cancellation included (s - K, a lerp between stops of opposite sign, rho near 1), so |got - ref| <= tau bound_k holds with a
tau that depends only on the error model (see tests/test_stop_reference_gpu.py).
"""
import numpy as np

MISS = 0xFFFFFFFF
U = 2.0 ** -24  # unit roundoff of float32


def walk(index, us, curve, cu):
    """rdc_interp_from from each curve's first stop: (ind, ratio) per ray; us the fp32 list, cu the rays' fp32 u"""
    start = index[curve, 0].astype(np.int64)
    end = start + index[curve, 1].astype(np.int64)
    ind = start.copy()
    step = (ind < end) & (us[ind + 1] < cu)
    while step.any():
        ind[step] += 1
        step &= ind < end
        step[step] = us[ind[step] + 1] < cu[step]
    lo, hi = us[ind].astype(np.float64), us[ind + 1].astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        ratio = (cu.astype(np.float64) - lo) / (hi - lo)
    return ind, ratio


def lerp(values, ind, ratio):
    """(1 - rho) a + rho b in float64 and its magnitude (|a| + |b|)(|1 - rho| + |rho|); values [n] or [n, 3]"""
    a, b = values[ind], values[ind + 1]
    r = ratio if values.ndim == 1 else ratio[:, None]
    share = np.abs(1 - r) + np.abs(r)
    return a * (1 - r) + b * r, (np.abs(a) + np.abs(b)) * share


class Rays:
    """The shaded primary rays of a band (hits on curves that are not portals) and their stop walks: the part of the frame
    that does not depend on any stop value."""

    def __init__(self, d, records):
        self.rows, self.width, self.n = records.shape
        self.npix = self.rows * self.width
        flat = records.reshape(-1)
        sel = np.nonzero((flat["id"] != MISS) & (flat["portal"] == 0))[0]
        self.pixel, self.ray = sel // self.n, sel % self.n  # ascending: pixel by pixel, each in ray order
        curve, cu = flat["curve"][sel].astype(np.int64), flat["curve_u"][sel]
        self.t = flat["t"][sel].astype(np.float64)
        self.lnt = np.log(self.t)
        self.right = flat["right"][sel] != 0
        self.walks = {fam: walk(d[fam + "_index"], d[fam + "_u"], curve, cu) for fam in ("blur", "weight", "weight_degree")}
        # colours: the side's list and index
        ind, ratio = np.zeros(len(sel), np.int64), np.zeros(len(sel))
        for fam, side in (("color_left", ~self.right), ("color_right", self.right)):
            ind[side], ratio[side] = walk(d[fam + "_index"], d[fam + "_u"], curve[side], cu[side])
        self.walks["color"] = (ind, ratio)

    def sum_pixels(self, v):
        if np.iscomplexobj(v):
            return self.sum_pixels(v.real) + 1j * self.sum_pixels(v.imag)
        return np.bincount(self.pixel, v, self.npix)


def _values(d, values, fam):
    v = np.asarray(values.get(fam, d[fam]) if values else d[fam])
    return v if np.iscomplexobj(v) else v.astype(np.float64)  # complex: for complex-step derivatives


def shade(d, R, values=None):
    """per ray: colour c [n, 3], its magnitude, blur b, its magnitude, m, e (and magnitudes), f, w, w's magnitude"""
    out = {}
    ind, ratio = R.walks["color"]
    cl, cr = _values(d, values, "color_left"), _values(d, values, "color_right")
    c, cbar = np.zeros((len(ind), 3)), np.zeros((len(ind), 3))
    for vals, side in ((cl, ~R.right), (cr, R.right)):
        c[side], cbar[side] = lerp(vals, ind[side], ratio[side])
    out["c"], out["cbar"] = c, cbar
    out["b"], out["bbar"] = lerp(_values(d, values, "blur"), *R.walks["blur"])
    out["m"], out["mbar"] = lerp(_values(d, values, "weight"), *R.walks["weight"])
    out["e"], out["ebar"] = lerp(_values(d, values, "weight_degree"), *R.walks["weight_degree"])
    out["f"] = np.exp(-out["e"] * R.lnt)  # t^-e
    out["w"] = out["m"] * out["f"]
    out["wbar"] = out["mbar"] * out["f"]
    return out


def nan_pixels(R, w):
    """the render's NaN pixels: the fp32 weights, summed in ray order like PixelSums::add, are zero"""
    W32 = np.zeros(R.npix, np.float32)
    w32 = w.real.astype(np.float32)
    for i in range(R.n):
        m = R.ray == i
        W32[R.pixel[m]] = W32[R.pixel[m]] + w32[m]
    return W32 == 0


def frame(d, records_or_rays, values=None):
    """the frame in float64: image [rows, W, 3], blur map [rows, W] (NaN where the render writes NaN), their scales
    (sum |w| |c| + |P| sum |w|) / |W| for the rounding bound, and max over the shaded rays of |e| |ln t| (the growth of the
    device falloff's error); `values` replaces stop value arrays of d (float64 allowed)"""
    R = records_or_rays if isinstance(records_or_rays, Rays) else Rays(d, records_or_rays)
    s = shade(d, R, values)
    W = R.sum_pixels(s["w"])
    Wbar = R.sum_pixels(s["wbar"])
    nan = nan_pixels(R, s["w"])
    with np.errstate(invalid="ignore", divide="ignore"):
        image = np.stack([R.sum_pixels(s["w"] * s["c"][:, k]) for k in range(3)], -1) / W[:, None]
        blur = R.sum_pixels(s["w"] * s["b"]) / W
        image_scale = (np.stack([R.sum_pixels(s["wbar"] * s["cbar"][:, k]) for k in range(3)], -1)
                       + np.abs(image) * Wbar[:, None]) / np.abs(W)[:, None]
        blur_scale = (R.sum_pixels(s["wbar"] * s["bbar"]) + np.abs(blur) * Wbar) / np.abs(W)
    image[nan], blur[nan], image_scale[nan], blur_scale[nan] = np.nan, np.nan, 0.0, 0.0
    live_rays = ~nan[R.pixel]
    shape = (R.rows, R.width)
    return {"image": image.reshape(shape + (3,)), "blur": blur.reshape(shape), "nan": nan.reshape(shape),
            "image_scale": image_scale.reshape(shape + (3,)), "blur_scale": blur_scale.reshape(shape),
            "elnt": float((s["ebar"] * np.abs(R.lnt))[live_rays].max(initial=0.0))}


def vjp(d, records_or_rays, G, g_sigma, values=None):
    """(grads, bounds): dicts over color_left [L, 3], color_right [L, 3], blur, weight, weight_degree laid out like d's value
    arrays, for pixel gradients G [rows, W, 3] and g_sigma [rows, W] (float32 inputs are taken as they are)"""
    R = records_or_rays if isinstance(records_or_rays, Rays) else Rays(d, records_or_rays)
    s = shade(d, R, values)
    W = R.sum_pixels(s["w"])
    live = ~nan_pixels(R, s["w"])
    on = live[R.pixel]
    px = R.pixel[on]
    G = np.asarray(G, np.float64).reshape(-1, 3)[px]
    gs = np.asarray(g_sigma, np.float64).reshape(-1)[px]
    sh = {k: v[on] for k, v in s.items()}
    invW = 1.0 / W[px]
    grads, bounds = {}, {}

    def scatter(name, shape, ind, ratio, term, mag):
        """term (1 - rho) to ind and term rho to ind + 1; mag (|1 - rho| + |rho|) to both; term, mag [n] or [n, k]"""
        n = shape[0]
        k = 1 if len(shape) == 1 else shape[1]
        term, mag = term.reshape(len(ind), k), mag.reshape(len(ind), k)
        r = ratio[:, None]
        share = np.abs(1 - r) + np.abs(r)
        g, b = np.zeros(n * k), np.zeros(n * k)
        for c in range(k):
            for off, part in ((0, 1 - r), (1, r)):
                idx = (ind + off) * k + c
                g += np.bincount(idx, term[:, c] * part[:, 0], n * k)
                b += np.bincount(idx, mag[:, c] * share[:, 0], n * k)
        grads[name], bounds[name] = g.reshape(shape), b.reshape(shape)

    ind, ratio = R.walks["color"]
    ind, ratio, right = ind[on], ratio[on], R.right[on]
    coef, coefbar = sh["w"] * invW, sh["wbar"] * np.abs(invW)
    for fam, side in (("color_left", ~right), ("color_right", right)):
        scatter(fam, d[fam].shape, ind[side], ratio[side], G[side] * coef[side, None],
                np.abs(G[side]) * coefbar[side, None])
    bi, br = (a[on] for a in R.walks["blur"])
    scatter("blur", d["blur"].shape, bi, br, gs * coef, np.abs(gs) * coefbar)

    # a zero gradient component adds nothing, whatever the stop value
    sray = np.where(G != 0, G * sh["c"], 0.0).sum(-1) + np.where(gs != 0, gs * sh["b"], 0.0)
    sbar = (np.abs(G) * sh["cbar"]).sum(-1) + np.abs(gs) * sh["bbar"]
    K = np.bincount(px, sh["w"] * sray, R.npix)[px] * invW
    Kbar = np.bincount(px, sh["wbar"] * sbar, R.npix)[px] * np.abs(invW)
    q, qbar = (sray - K) * invW, (sbar + Kbar) * np.abs(invW)
    wi, wr = (a[on] for a in R.walks["weight"])
    scatter("weight", d["weight"].shape, wi, wr, sh["f"] * q, sh["f"] * qbar)
    ei, er = (a[on] for a in R.walks["weight_degree"])
    lnt = R.lnt[on]
    scatter("weight_degree", d["weight_degree"].shape, ei, er, -sh["w"] * lnt * q, sh["wbar"] * np.abs(lnt) * qbar)
    return grads, bounds


def loss(d, rays, G, g_sigma, values=None, live=None):
    """sum over the live pixels (by default those the frame does not make NaN) of <G, P> + g_sigma sigma, in float64 (or
    complex128 for complex `values`): the scalar whose gradient vjp returns"""
    fr = frame(d, rays, values)
    live = ~fr["nan"] if live is None else live
    return ((np.asarray(G, np.float64)[live] * fr["image"][live]).sum()
            + (np.asarray(g_sigma, np.float64)[live] * fr["blur"][live]).sum())
