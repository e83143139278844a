"""The device build of csrc/rdc_math.h against its host build, and its two documented exceptions against float64.

rdc_math.h promises that nvcc (-fmad=false) and g++ (-ffp-contract=off) builds of it give bit-identical results. The
renders only exercise that through equal hit ids, at the inputs a scene happens to produce. Here the probe in
tests/probes is built both ways with the Makefile's flags and every function the header puts in the bit-exact set runs
on one corpus in both: random values at scene magnitudes, then every argument in turn set to +-0, the smallest and
largest denormals, +-1e-30, +-1e30, +-inf and NaN, and the edge cases of each function. Outputs must agree word for word;
two NaNs agree whatever their payload.

rdc_ratio (__fdividef) and rdc_weight_falloff (rsqrtf, exp2f(log2f)) are outside that set on the device and are
bounded against float64 instead.
"""
import numpy as np
import pytest

import math_probe as mp

pytestmark = pytest.mark.gpu

F32 = np.float32
INF = np.inf
SPECIAL = np.array([0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, -1.1754942e-38, 1e-30, -1e-30, 1e30, -1e30, INF, -INF, np.nan],
                   np.float32)


@pytest.fixture(scope="module")
def probes(tmp_path_factory):
    import torch

    assert torch.cuda.is_available()
    d = str(tmp_path_factory.mktemp("rdc_math_probe"))
    return mp.Probe(mp.build_host(d), device=False), mp.Probe(mp.build_device(d), device=True)


def fw(a):
    return np.asarray(a, np.float32).view(np.uint32)


def with_specials(rng, m, float_cols, per=3, mixed=1024):
    """Rows of m, then for every float column and every special value `per` random rows with that column set to it,
    then `mixed` rows in which every float column is a special value with probability 0.4."""
    parts = [m]
    for j in float_cols:
        for v in SPECIAL:
            r = m[rng.integers(0, len(m), per)].copy()
            r[:, j] = fw(v)
            parts.append(r)
    r = m[rng.integers(0, len(m), mixed)].copy()
    for j in float_cols:
        pick = rng.random(mixed) < 0.4
        r[pick, j] = fw(SPECIAL[rng.integers(0, len(SPECIAL), pick.sum())])
    parts.append(r)
    return np.concatenate(parts)


def coords(rng, n, scale=1000.0):
    return rng.uniform(-scale, scale, n).astype(np.float32)


def unit_dirs(rng, n):
    a = rng.uniform(0, 2 * np.pi, n)
    return np.cos(a).astype(np.float32), np.sin(a).astype(np.float32)


def stop_table(rng):
    """A flat stop table like the ingest's: lists of count+1 stops, each followed by two +INF sentinels. Sorted, with
    repeats, non-monotonic, and holding NaN or inf. Returns (table, [(start, count)])."""
    table, lists = [], []
    for j in range(200):
        count = int(rng.integers(0, 9))
        kind = j % 5
        s = rng.uniform(0, 1, count + 1)
        if kind == 0:
            s = np.sort(s)
        elif kind == 1:
            s = np.sort(np.round(s * 4) / 4)  # repeated stops: zero-width intervals
        elif kind == 3:
            s[rng.integers(0, count + 1)] = rng.choice([np.nan, INF, -INF, -0.0])
        elif kind == 4:
            s = np.sort(s)[::-1]
        lists.append((len(table), count))
        table += list(s) + [INF, INF]
    return np.array(table, np.float32), lists


def corpus(name, rng):
    """name -> (input words, indices of float input columns, indices of float output columns, aux table)."""
    n = 4096
    u = lambda lo, hi: rng.uniform(lo, hi, n).astype(np.float32)  # noqa: E731
    aux = None
    if name == "philox":
        m = rng.integers(0, 2 ** 32, (n, 6), dtype=np.uint64).astype(np.uint32)
        m[:64] = np.array([0, 0xFFFFFFFF], np.uint32)[rng.integers(0, 2, (64, 6))]
        return m, [], [], None
    if name == "u01":
        m = np.concatenate([rng.integers(0, 2 ** 32, n, dtype=np.uint64), [0, 1, 2 ** 24 - 1, 2 ** 24, 2 ** 24 + 1, 0x80000080,
                                                                           0xFFFFFF7F, 0xFFFFFF80, 0xFFFFFFFF]])
        return mp.rows(m), [], [0], None
    if name in ("sincospi", "sincospi_kernel"):
        lim = 4.0 if name == "sincospi" else 0.25
        x = np.concatenate([u(-lim, lim), np.arange(-16, 17) / 4.0 * (lim / 4.0), 2.0 ** np.arange(-149, 127, 0.5)]).astype(np.float32)
        return with_specials(rng, mp.rows(x), [0]), [0], [0, 1], None
    if name == "spline":
        m = mp.rows(np.concatenate([u(0, 1)[: n - 8], F32([0, 1, -0.0, 0.5, 1e-7, 1 - 6e-8, -0.01, 1.01])]),
                    *[coords(rng, n) for _ in range(8)])
        return with_specials(rng, m, range(9)), range(9), range(4), None
    if name == "is_ray_right":
        dx, dy = unit_dirs(rng, n)
        dx[:16], dy[:16] = 0.0, 0.0
        m = mp.rows(u(0, 1), dx, dy, *[coords(rng, n) for _ in range(8)], rng.integers(0, 2, n))
        return with_specials(rng, m, range(11)), range(11), [], None
    if name in ("interp_from", "walk_hint"):
        aux, lists = stop_table(rng)
        pick = rng.integers(0, len(lists), n)
        start = np.array([lists[p][0] for p in pick], np.uint32)
        count = np.array([lists[p][1] for p in pick], np.uint32)
        q = np.where(rng.random(n) < 0.3, aux[start + (rng.integers(0, 1 << 30, n) % (count + 1))], u(-0.2, 1.2))
        if name == "interp_from":  # from the list's start, or from a later index (the walk hint's use)
            first = start + np.where(rng.random(n) < 0.5, 0, rng.integers(0, 1 << 30, n) % (count + 1))
            m = mp.rows(first, start + count, q.astype(np.float32))
            return with_specials(rng, m, [2]), [2], [1], aux
        m = mp.rows(start, count, q.astype(np.float32))
        return with_specials(rng, m, [2]), [2], [], aux
    if name == "lerp":
        m = mp.rows(u(-1, 1), u(-1, 1), np.concatenate([u(-0.1, 1.1)[: n - 4], F32([0, 1, 0.5, -0.0])]))
        return with_specials(rng, m, range(3)), range(3), range(2), None
    if name == "chord_count":
        # nearly straight segments (few chords) and wild ones (kmax), tolerance 0.05 and others
        base = np.stack([coords(rng, n) for _ in range(8)], 1)
        line = np.linspace(0, 1, 4)[None, :, None] * (base[:, None, 2:4] - base[:, None, :2]) + base[:, None, :2]
        straight = (line + rng.normal(0, 0.01, line.shape)).reshape(n, 8).astype(np.float32)
        v = np.where(rng.random((n, 1)) < 0.5, straight, base).astype(np.float32)
        tol = np.where(rng.random(n) < 0.5, F32(0.05), u(1e-3, 10)).astype(np.float32)
        kmax = rng.integers(-2, 80, n)
        m = mp.rows(*v.T, tol, kmax)
        return with_specials(rng, m, range(9)), range(9), [], None
    if name == "ray_chord":
        ox, oy = coords(rng, n), coords(rng, n)
        dx, dy = unit_dirs(rng, n)
        primary = rng.random(n) < 0.5
        dx = np.where(primary, dx, dx * u(0.1, 3)).astype(np.float32)
        dy = np.where(primary, dy, dy * u(0.1, 3)).astype(np.float32)
        inv = np.where(primary, F32(1), F32(1) / (dx * dx + dy * dy)).astype(np.float32)
        ax, ay, bx, by = (coords(rng, n) for _ in range(4))
        e = n // 4  # rays that start on a chord end
        ax[:e], ay[:e] = ox[:e], oy[:e]
        bx[e:2 * e], by[e:2 * e] = ox[e:2 * e], oy[e:2 * e]
        g = slice(2 * e, 3 * e)  # rays that graze: both ends on the ray's supporting line
        s1, s2 = u(-50, 50)[g], u(-50, 50)[g]
        ax[g], ay[g] = ox[g] + s1 * dx[g], oy[g] + s1 * dy[g]
        bx[g], by[g] = ox[g] + s2 * dx[g], oy[g] + s2 * dy[g]
        m = mp.rows(ox, oy, dx, dy, inv, ax, ay, bx, by)
        return with_specials(rng, m, range(9)), range(9), [1, 2], None
    if name == "chord_hit":
        dx, dy = unit_dirs(rng, n)
        w = [coords(rng, n, 100) for _ in range(4)]
        ea, eb = u(-100, 100), u(-100, 100)
        k = n // 8
        ea[:k] = rng.choice(F32([0.0, -0.0]), k)  # a chord end on the ray's line
        eb[k:2 * k] = rng.choice(F32([0.0, -0.0]), k)
        ea[2 * k:3 * k] = rng.choice(F32([0.0, -0.0]), k)
        eb[2 * k:3 * k] = rng.choice(F32([0.0, -0.0]), k)
        eb[3 * k:4 * k] = -ea[3 * k:4 * k]  # opposite signs, equal size
        m = mp.rows(dx, dy, F32(1), *w, ea, eb)
        return with_specials(rng, m, range(9)), range(9), [1, 2], None
    if name == "inv_dd":
        dx, dy = unit_dirs(rng, n)
        m = mp.rows(dx * u(0.01, 100), dy, rng.integers(0, 2, n))
        return with_specials(rng, m, [0, 1]), [0, 1], [0], None
    if name == "portal_skip":
        m = mp.rows(np.concatenate([u(-0.1, 1.1)[: n - 6], F32([0, 1, -0.0, 1 - 6e-8, 0.5, 2.0])]), rng.integers(0, 65, n))
        return with_specials(rng, m, [0]), [0], [], None
    if name == "safe_inv":
        near = (F32(1e-30) * (1 + np.arange(-8, 9) * 2.0 ** -23)).astype(np.float32)
        x = np.concatenate([near, -near, (10.0 ** rng.uniform(-45, 38, n)).astype(np.float32) * rng.choice([-1, 1], n)]).astype(np.float32)
        return with_specials(rng, mp.rows(x), [0]), [0], [0], None
    if name == "slab":
        dx, dy = unit_dirs(rng, n)
        dx[:64], dy[64:128] = 0.0, -0.0
        sinv = lambda d: np.where(np.abs(d) < 1e-30, np.copysign(1e30, d), 1.0 / np.where(np.abs(d) < 1e-30, 1.0, d.astype(np.float64))).astype(np.float32)  # noqa: E731
        x0, x1, y0, y1 = (coords(rng, n) for _ in range(4))
        m = mp.rows(coords(rng, n), coords(rng, n), sinv(dx), sinv(dy), np.minimum(x0, x1), np.minimum(y0, y1), np.maximum(x0, x1),
                    np.maximum(y0, y1))
        return with_specials(rng, m, range(8)), range(8), [0, 1], None
    if name == "point_chord":
        v = [coords(rng, n) for _ in range(6)]
        v[4][:64], v[5][:64] = v[2][:64], v[3][:64]  # degenerate chords
        v[0][64:128], v[1][64:128] = v[2][64:128], v[3][64:128]  # the point on a chord end
        return with_specials(rng, mp.rows(*v), range(6)), range(6), range(4), None
    if name == "point_box_d2":
        v = [coords(rng, n) for _ in range(6)]
        return with_specials(rng, mp.rows(*v), range(6)), range(6), [0], None
    if name == "pixel_centre":
        sizes = np.array([0, 1, 2, 3, 511, 512, 1080, 1920, 4097, 2 ** 31, 2 ** 31 + 1, 0xFFFFFFFF], np.uint64)
        size = sizes[rng.integers(0, len(sizes), n)]
        # indices inside the frame (below size / 2 the unsigned difference wraps), beyond it, and the largest
        idx = np.where(rng.random(n) < 0.8, rng.integers(0, 1 << 62, n).astype(np.uint64) % np.maximum(size, 1),
                       rng.integers(0, 2 ** 32, n, dtype=np.uint64))
        zoom = (u(0.01, 4) * rng.choice([-1, 1], n)).astype(np.float32)
        m = mp.rows(size, zoom, coords(rng, n), rng.integers(0, 2, n), idx)
        return with_specials(rng, m, [1, 2]), [1, 2], [0, 1], None
    if name == "jitter":
        ns = np.array(mp.RAY_COUNTS + [1.5, 7.5, 8.5], np.float32)
        bx, by = unit_dirs(rng, n)
        m = mp.rows(bx, by, mp.two_over_n(ns[rng.integers(0, len(ns), n)]), np.concatenate([F32(mp.JITTER_U), u(0, 1)[4:]]))
        return with_specials(rng, m, range(4)), range(4), [0, 1], None
    raise KeyError(name)


BIT_EXACT = ["philox", "u01", "sincospi", "sincospi_kernel", "spline", "is_ray_right", "interp_from", "walk_hint", "lerp",
             "chord_count", "ray_chord", "chord_hit", "inv_dd", "portal_skip", "safe_inv", "slab", "point_chord", "point_box_d2",
             "pixel_centre", "jitter"]


def mismatches(h, d, float_out):
    same = h == d
    hf, df = h.view(np.float32), d.view(np.float32)
    for j in float_out:
        same[:, j] |= np.isnan(hf[:, j]) & np.isnan(df[:, j])
    return np.nonzero(~same.all(1))[0]


@pytest.mark.parametrize("name", BIT_EXACT)
def test_device_equals_host(probes, name):
    host, dev = probes
    rng = np.random.default_rng(100 + BIT_EXACT.index(name))
    inp, _, float_out, aux = corpus(name, rng)
    h, d = host.run(name, inp, aux), dev.run(name, inp, aux)
    if name == "interp_from":
        # the ratio is rdc_ratio's (__fdividef on the device): checked against the ratio probe on the same operands below
        bad = mismatches(h[:, :1], d[:, :1], [])
    else:
        bad = mismatches(h, d, float_out)
    detail = "\n".join(f"  in {[hex(w) for w in inp[i]]} ({inp[i].view(np.float32)})\n  host {[hex(w) for w in h[i]]} "
                       f"device {[hex(w) for w in d[i]]}" for i in bad[:5])
    assert len(bad) == 0, f"{name}: {len(bad)} of {len(inp)} rows differ between the nvcc and g++ builds:\n{detail}"
    if name == "interp_from":
        idx = d[:, 0].astype(np.int64)
        q = inp[:, 2].view(np.float32)
        num, den = q - aux[idx], aux[idx + 1] - aux[idx]
        want = dev.run("ratio", mp.rows(num, den))[:, 0]
        assert len(mismatches(d[:, 1:2], want[:, None], [0])) == 0


# ------------------------------------------------------------------------------------------------------------------
# Ray directions on the device
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", mp.RAY_COUNTS)
def test_device_ray_directions_equal_restatement(probes, n):
    """The directions test_shared_math_cpu.py checks against render.cu's culling margin are the device's, bit for bit."""
    host, dev = probes
    ton = mp.two_over_n(n)
    rs, rc = dev.run("sincospi", [[ton.view(np.uint32)]])[0].view(np.float32)
    base = mp.restate_base_dirs(rs, rc, n)
    assert np.array_equal(dev.base_dirs(ton, n).view(np.uint32), base.view(np.uint32))
    small = F32(0) <= ton <= F32(0.25)
    for u in mp.JITTER_U:
        js, jc = dev.run("sincospi_kernel" if small else "sincospi", [[(ton * F32(u)).view(np.uint32)]])[0].view(np.float32)
        got = dev.run("jitter", mp.rows(base[:, 0], base[:, 1], ton, F32(u))).view(np.float32)
        assert np.array_equal(got.view(np.uint32), mp.restate_jitter(base, js, jc).view(np.uint32)), f"N={n} u={u}"


# ------------------------------------------------------------------------------------------------------------------
# rdc_ratio: __fdividef on the device
# ------------------------------------------------------------------------------------------------------------------
RATIO_ULP = 2.0


def test_ratio_within_two_ulp(probes):
    host, dev = probes
    rng = np.random.default_rng(7)
    n = 200_000
    den = (2.0 ** rng.uniform(-126, 126, n) * rng.choice([-1, 1], n)).astype(np.float32)
    num = (2.0 ** rng.uniform(-60, 60, n) * rng.choice([-1, 1], n)).astype(np.float32)
    # the render's ratios: (u - lo) / (hi - lo) with stops in [0, 1]
    lo, hi = np.sort(rng.uniform(0, 1, (2, n)).astype(np.float32), 0)
    uu = rng.uniform(0, 1, n).astype(np.float32)
    num, den = np.concatenate([num, uu - lo]), np.concatenate([den, hi - lo])
    den = np.where(np.abs(den) < 2.0 ** -126, F32(2.0 ** -126), den).astype(np.float32)
    exact = num.astype(np.float64) / den.astype(np.float64)
    normal = (np.abs(exact) >= 2.0 ** -126) & (np.abs(exact) < 2.0 ** 127)
    got = dev.run("ratio", mp.rows(num, den))[:, 0].view(np.float32)
    err = np.abs(got.astype(np.float64) - exact) / np.spacing(np.abs(exact).astype(np.float32)).astype(np.float64)
    print(f"rdc_ratio device: worst {err[normal].max():.3f} ulp over {normal.sum()} quotients with |den| in [2^-126, 2^126]")
    assert err[normal].max() <= RATIO_ULP


def test_ratio_outside_the_range(probes):
    """What __fdividef gives where the 2-ulp bound does not hold (recorded in rdc_math.h)."""
    host, dev = probes
    rng = np.random.default_rng(8)
    num = rng.uniform(-10, 10, 1000).astype(np.float32)
    big = (2.0 ** rng.uniform(126.01, 127.99, 1000) * rng.choice([-1, 1], 1000)).astype(np.float32)
    got = dev.run("ratio", mp.rows(num, big))[:, 0].view(np.float32)
    print(f"rdc_ratio device, |den| > 2^126: {np.unique(got)[:8]}")
    assert np.all(got == 0.0)  # host: |num / den| < 2^-122
    tiny = (2.0 ** rng.uniform(-149, -126.01, 1000) * rng.choice([-1, 1], 1000)).astype(np.float32)
    got = dev.run("ratio", mp.rows(num, tiny))[:, 0].view(np.float32)
    want = host.run("ratio", mp.rows(num, tiny))[:, 0].view(np.float32)
    over = np.isinf(want)
    print(f"rdc_ratio device, denormal den: {over.sum()} quotients overflow on the host, {np.isinf(got[~over]).sum()} of the "
          f"others on the device")
    assert over.sum() > 500 and np.array_equal(got[over], want[over])  # overflow: the same infinity
    # zero, infinite and NaN denominators and numerators, and the other special values: as IEEE division
    s = SPECIAL
    a, b = np.repeat(s, len(s)), np.tile(s, len(s))
    got = dev.run("ratio", mp.rows(a, b))[:, 0].view(np.float32)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        want = (a.astype(np.float64) / b.astype(np.float64)).astype(np.float32)
    bad = [f"{x}/{y}={g}" for x, y, g, w in zip(a, b, got, want) if not (g == w or (np.isnan(g) and np.isnan(w)))]
    assert not bad, ", ".join(bad)


# ------------------------------------------------------------------------------------------------------------------
# rdc_weight_falloff: rsqrtf, exp2f(log2f) on the device
# ------------------------------------------------------------------------------------------------------------------
EXPONENTS = [0.0, 0.25, 0.5, 1.0, 2.0, 3.7]


def falloff_bound(e):
    """Relative error bound of the device's t^-e: rsqrtf's 2 ulp, and log2f's error carried through exp2f, which grows
    with the exponent.

    Why this is inside the 1e-4 RGB tolerance: a pixel's colour is a weighted mean m = sum w_k c_k / sum w_k. With every
    w_k off by a factor (1 + d_k), |d_k| <= eps, the mean moves by sum w_k d_k (c_k - m) / sum w_k (1 + d_k), at most
    eps / (1 - eps) * (max c - min c), whatever the ratio of the weights. The bundled scenes' weight stops span 1..20
    (weight_demo.xml) with exponents up to 0.9: eps <= falloff_bound(0.9) = 2.05e-6, so colours in [0, 1] move by 2e-6.
    Even e = 3.7 (7.65e-6) stays thirteen times below 1e-4."""
    return 2.5e-7 + 2e-6 * e


def test_weight_falloff_relative_error(probes):
    host, dev = probes
    t = (10.0 ** np.linspace(-6, 6, 100_001)).astype(np.float32)
    worst = {}
    for e in EXPONENTS:
        got = dev.run("weight_falloff", mp.rows(t, F32(e)))[:, 0].view(np.float32).astype(np.float64)
        want = t.astype(np.float64) ** -e
        rel = np.abs(got - want) / want
        worst[e] = float(rel.max())
    print("rdc_weight_falloff device, worst relative error: " + ", ".join(f"e={e}: {w:.3g}" for e, w in worst.items()))
    for e, w in worst.items():
        assert w <= falloff_bound(e), f"e={e}: {w:.3g} > {falloff_bound(e):.3g}"
