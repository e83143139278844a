"""The host build of csrc/rdc_math.h against references that do not share it: ray generation.

Every oracle includes rdc_math.h, and the reference's DeviceCode.cu is routed into it for curand_uniform and
sincospif, so the parity tests compare the header with itself. Here the host build (the probe in tests/probes, compiled
like the product's host code) meets independent statements of the same operations:

 * Philox4x32-10: Random123's known-answer vectors (kat_vectors, philox4x32 with 10 rounds) and a pure-Python round
   function;
 * rdc_u01: the exact value x 2^-32 + 2^-33, in float64;
 * rdc_sincospi: float64 sin(pi x) and cos(pi x);
 * the ray directions: k_base_dirs and gen_ray's jitter restated in float32 numpy, and the float64 angle of every
   direction against the stratum that render.cu's angular culling assumes it lies in.
"""
import numpy as np
import pytest

import math_probe as mp

F32 = np.float32


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return mp.Probe(mp.build_host(str(tmp_path_factory.mktemp("rdc_math_probe"))), device=False)


def f32(w):
    return np.asarray(w, np.uint32).view(np.float32)


# ------------------------------------------------------------------------------------------------------------------
# Philox4x32-10
# ------------------------------------------------------------------------------------------------------------------
KAT = [  # Random123 kat_vectors: philox4x32 10 rounds, ctr, key -> output
    ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
]


def philox_reference(ctr, key):
    """Philox4x32-10 (Salmon et al. 2011, Random123's philox4x32round / philox4x32bumpkey), vectorised over rows."""
    c = [np.asarray(ctr[:, j], np.uint64) for j in range(4)]
    k0, k1 = np.asarray(key[:, 0], np.uint64), np.asarray(key[:, 1], np.uint64)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & mask, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & mask]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & mask, (k1 + np.uint64(0xBB67AE85)) & mask
    return np.stack(c, 1).astype(np.uint32)


@pytest.mark.parametrize("ctr,key,want", KAT, ids=["zeros", "ones", "pi"])
def test_philox_known_answers(host, ctr, key, want):
    got = host.run("philox", [ctr + key])[0]
    assert [f"{v:08x}" for v in got] == [f"{v:08x}" for v in want]


def test_philox_matches_restatement(host):
    rng = np.random.default_rng(1)
    inp = rng.integers(0, 2 ** 32, size=(100_000, 6), dtype=np.uint64).astype(np.uint32)
    inp[:1000, 2:4] = 0  # the render's counters: (pixel, ray, 0, 0)
    got = host.run("philox", inp)
    want = philox_reference(inp[:, :4], inp[:, 4:])
    bad = np.nonzero((got != want).any(1))[0]
    assert len(bad) == 0, f"{len(bad)} rows differ, first: in {inp[bad[0]]} got {got[bad[0]]} want {want[bad[0]]}"


# ------------------------------------------------------------------------------------------------------------------
# rdc_u01
# ------------------------------------------------------------------------------------------------------------------
def u01_exact(x):
    """x 2^-32 + 2^-33, correctly rounded to float32 (the float64 sum is exact: 34 significant bits)."""
    return (np.asarray(x, np.uint32).astype(np.float64) * 2.0 ** -32 + 2.0 ** -33).astype(np.float32)


def u01_curand(x):
    """curand_uniform's mapping as written, x * 2^-32f + 2^-33f with x converted to float first: float(x) rounds
    to nearest even, then one fused multiply-add (also exact in float64)."""
    xf = np.asarray(x, np.uint32).astype(np.float64).astype(np.float32).astype(np.float64)
    return (xf * 2.0 ** -32 + 2.0 ** -33).astype(np.float32)


U01_EDGES = [0, 1, 2 ** 24 - 1, 2 ** 24, 2 ** 24 + 1, 0x80000080, 0xFFFFFF7F, 0xFFFFFF80, 0xFFFFFFFF]


def test_u01_edges(host):
    x = np.array(U01_EDGES, np.uint32)
    got = f32(host.run("u01", x[:, None])[:, 0])
    assert got[-1] == 1.0  # 0xFFFFFFFF maps to exactly 1
    assert got[0] == F32(2.0 ** -33)
    np.testing.assert_array_equal(got.view(np.uint32), u01_curand(x).view(np.uint32))
    # The correctly rounded value of x 2^-32 + 2^-33, except where float(x) rounds a tie down to even before the
    # multiply-add: 2^24 + 1 (-> 2^24) and 0x80000080 (-> 2^31) come out one ulp low, as curand_uniform does.
    exact = u01_exact(x)
    tie_down = np.isin(x, [2 ** 24 + 1, 0x80000080])
    np.testing.assert_array_equal(got[~tie_down].view(np.uint32), exact[~tie_down].view(np.uint32))
    np.testing.assert_array_equal(got[tie_down].view(np.uint32), exact[tie_down].view(np.uint32) - 1)


def test_u01_random(host):
    rng = np.random.default_rng(2)
    x = np.sort(rng.integers(0, 2 ** 32, size=1_000_000, dtype=np.uint64).astype(np.uint32))
    got = f32(host.run("u01", x[:, None])[:, 0])
    np.testing.assert_array_equal(got.view(np.uint32), u01_curand(x).view(np.uint32))
    assert np.all(got > 0.0) and np.all(got <= 1.0)
    assert np.all(np.diff(got) >= 0.0)  # monotone
    # one ulp from the correctly rounded value at most, and only where float(x) was a tie
    exact = u01_exact(x)
    diff = got.view(np.uint32).astype(np.int64) - exact.view(np.uint32).astype(np.int64)
    assert set(np.unique(diff)) <= {-1, 0}
    xf = x.astype(np.float64).astype(np.float32).astype(np.float64)
    spacing = np.spacing(x.astype(np.float64).astype(np.float32)).astype(np.float64)
    tie = np.abs(x.astype(np.float64) - xf) * 2 == spacing
    assert np.all(tie[diff != 0])


# ------------------------------------------------------------------------------------------------------------------
# rdc_sincospi
# ------------------------------------------------------------------------------------------------------------------
SINCOSPI_ULP = 2.0  # the header's "~2 ulp"
UNIT_ULP = 4.0  # s^2 + c^2 within 4 ulp(1) = 4 * 2^-23 of 1


def ulp_error(got, want):
    """|got - want| in units of the float32 spacing at |want| (float64 want)."""
    sp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    return np.abs(got.astype(np.float64) - want) / sp


def neighbours(x, k=4):
    """float32 x and its neighbours up to k ulp either side."""
    out = [np.asarray(x, np.float32)]
    lo = hi = out[0]
    for _ in range(k):
        lo = np.nextafter(lo, F32(-np.inf))
        hi = np.nextafter(hi, F32(np.inf))
        out += [lo, hi]
    return np.concatenate(out)


def sincospi_inputs():
    rng = np.random.default_rng(3)
    dense = np.linspace(-4.0, 4.0, 400_001).astype(np.float32)
    quarters = neighbours(np.arange(-16, 17) / 4.0)
    tiny = np.concatenate([F32([0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, -1.1754942e-38, 1e-30, -1e-30]),
                           np.logspace(-40, -1, 2000).astype(np.float32)])
    # the render passes two_over_n * u01 with two_over_n = 2 / rays per pixel <= 2, and the base rotation 2 / N
    render = np.concatenate([(mp.two_over_n(n) * F32(np.concatenate([mp.JITTER_U, rng.uniform(0, 1, 64)]))) for n in range(1, 9)]
                            + [mp.two_over_n(np.array(mp.RAY_COUNTS, np.float32))])
    # beyond it: integers and half-integers, where sin and cos are exact, up to the domain's end (2x must not overflow)
    big = np.concatenate([2.0 ** np.arange(2, 127), 2.0 ** np.arange(2, 23) + 0.5, 2.0 ** np.arange(2, 24) + 1.0,
                          [np.nextafter(F32(2.0 ** 127), F32(0))]]).astype(np.float32)
    x = np.concatenate([dense, rng.uniform(-4, 4, 200_000).astype(np.float32), quarters, tiny, -tiny, render, big, -big])
    return x.astype(np.float32)


def sincospi_reference(x):
    """float64 sin(pi x), cos(pi x). x = q/2 + r with |r| <= 1/4 exactly (float64 holds every float32 x - q/2), so the
    quarter turns are exact and only sin, cos of pi r round."""
    x64 = x.astype(np.float64)
    q = np.round(2.0 * x64)
    r = x64 - 0.5 * q
    sr, cr = np.sin(np.pi * r), np.cos(np.pi * r)
    quadrant = np.mod(q, 4.0)
    s = np.select([quadrant == 0, quadrant == 1, quadrant == 2], [sr, cr, -sr], -cr)
    c = np.select([quadrant == 0, quadrant == 1, quadrant == 2], [cr, -sr, -cr], sr)
    return s, c


def test_sincospi_accuracy(host):
    x = sincospi_inputs()
    out = f32(host.run("sincospi", x.view(np.uint32)[:, None]))
    s, c = out[:, 0], out[:, 1]
    ws, wc = sincospi_reference(x)
    es, ec = ulp_error(s, ws), ulp_error(c, wc)
    worst = int(np.argmax(np.maximum(es, ec)))
    print(f"rdc_sincospi host: worst {max(es.max(), ec.max()):.3f} ulp (sin {es.max():.3f}, cos {ec.max():.3f}) at x={x[worst]!r}")
    assert es.max() <= SINCOSPI_ULP and ec.max() <= SINCOSPI_ULP, f"x={x[worst]!r}: sin {s[worst]!r} vs {ws[worst]!r}, cos {c[worst]!r} vs {wc[worst]!r}"
    unit = np.abs(s.astype(np.float64) ** 2 + c.astype(np.float64) ** 2 - 1.0) / 2.0 ** -23
    print(f"rdc_sincospi host: worst |s^2 + c^2 - 1| {unit.max():.3f} ulp(1)")
    assert unit.max() <= UNIT_ULP, f"x={x[np.argmax(unit)]!r}"
    # exact where the answer is exact: integers and half-integers give 0 and +-1
    ints = (x == np.round(x)) | (2 * x == np.round(2 * x))
    assert np.array_equal(s[ints], ws[ints].astype(np.float32)) and np.array_equal(c[ints], wc[ints].astype(np.float32))
    # odd and even: sin(-x) = -sin(x), cos(-x) = cos(x) bit for bit
    neg = f32(host.run("sincospi", (-x).view(np.uint32)[:, None]))
    assert np.array_equal(neg[:, 0], -s) and np.array_equal(neg[:, 1], c)


def test_sincospi_kernel_accuracy(host):
    """The unreduced polynomial, which gen_ray calls directly for N >= 8 (|x| <= 1/4)."""
    x = np.concatenate([np.linspace(-0.25, 0.25, 200_001), neighbours(F32([-0.25, 0.0, 0.25]))]).astype(np.float32)
    out = f32(host.run("sincospi_kernel", x.view(np.uint32)[:, None]))
    ws, wc = sincospi_reference(x)
    es, ec = ulp_error(out[:, 0], ws), ulp_error(out[:, 1], wc)
    print(f"rdc_sincospi_kernel host: worst sin {es.max():.3f} ulp, cos {ec.max():.3f} ulp")
    assert es.max() <= SINCOSPI_ULP and ec.max() <= SINCOSPI_ULP
    # the reduction leaves |x| <= 1/4 unchanged (up to the sign of a zero sine: it returns +0 for -0)
    inside = np.abs(x) <= 0.25
    full = f32(host.run("sincospi", x[inside].view(np.uint32)[:, None]))
    assert np.array_equal(full, out[inside])


# ------------------------------------------------------------------------------------------------------------------
# Ray directions and render.cu's angular culling
# ------------------------------------------------------------------------------------------------------------------
def direction_margin(n):
    """The part of angular_interval's safety (render.cu) that covers the ray directions: half a stratum plus the drift
    of the iterated rotation, 4e-8 n^2 strata. (Its 1e-3 strata_per_rad term covers atan2_bound's error.)"""
    return 0.5 + 4e-8 * float(n) * float(n)


def drift_term(n):
    return 4e-8 * float(n) * float(n)


def stratum_excess(d, n):
    """How far (in strata) the float64 angle of direction i lies outside its stratum [i, i+1]; 0 inside."""
    n = int(n)
    ang = np.arctan2(d[:, 1].astype(np.float64), d[:, 0].astype(np.float64)) * (n / (2.0 * np.pi))
    i = np.arange(len(d), dtype=np.float64)
    off = np.mod(ang - i - 0.5 + n / 2.0, n) - n / 2.0 + 0.5  # angle - i, wrapped around the stratum's middle
    return np.maximum(np.maximum(-off, off - 1.0), 0.0)


def ray_directions(probe, n):
    """Base directions and, per jitter draw u, the jittered directions, for N rays: (restated, probe) pairs."""
    ton = mp.two_over_n(n)
    rs, rc = f32(probe.run("sincospi", [[ton.view(np.uint32)]])[0])
    base = mp.restate_base_dirs(rs, rc, n)
    small = F32(0.0) <= ton <= F32(0.25)
    out = {"base": (base, probe.base_dirs(ton, n))}
    for u in mp.JITTER_U:
        ang = ton * F32(u)
        js, jc = f32(probe.run("sincospi_kernel" if small else "sincospi", [[ang.view(np.uint32)]])[0])
        inp = mp.rows(base[:, 0], base[:, 1], ton, F32(u))
        out[u] = (mp.restate_jitter(base, js, jc), f32(probe.run("jitter", inp)))
    return out


@pytest.mark.parametrize("n", mp.RAY_COUNTS)
def test_ray_directions_stay_in_their_strata(host, n):
    worst = 0.0
    for key, (restated, built) in ray_directions(host, n).items():
        assert np.array_equal(restated.view(np.uint32), built.view(np.uint32)), f"N={n} {key}: probe and restatement differ"
        if key == "base":
            continue
        # |D| = 1 within the iterated rotation's drift, 1e-7 N (rdc_math.h, rdc_inv_dd)
        norm = np.hypot(restated[:, 0].astype(np.float64), restated[:, 1].astype(np.float64))
        assert np.abs(norm - 1.0).max() <= 1e-7 * n
        worst = max(worst, float(stratum_excess(restated, n).max()))
    print(f"N={n}: worst excess outside the stratum {worst:.3g} strata; drift term {drift_term(n):.3g}, margin {direction_margin(n):.3g}")
    assert worst <= direction_margin(n)
    # The drift term alone covers the iterated rotation wherever the render culls (N >= 8).
    if n >= 8:
        assert worst <= drift_term(n)
