"""Texture and sky lookups against a float64 statement of linear filtering (bilinear64, written from the CUDA programming guide's
definition, not from texLookup).  The oracle filters with the same fp32 rule as the product, so an addressing error common to both
(a half-texel offset, the wrap at the seam, the clamp at the poles) would pass every path-for-path test; these tests compare with
an independent statement instead:

- on the CPU, bilinear64 against the oracle's fp32 rule (pins the statement itself);
- on the GPU, call by call (tests/device_probe.cu): texLookup's software filter and the texture unit, fastAtan2 / fastAtan2Inline /
  fastAcos against float64 arctan2 / arccos, and the gamma step fastPow(x, 2.2f);
- end to end through the render kernel with the parity aids (jitter = 0, first_hit = 1): the sky tap at a miss, the material tap
  behind the `tex <= texCount` guard, and texture handles up to 64.

Tolerances name what they absorb; "B200" is the largest value seen on one B200 (1000 W) and the bound keeps headroom over it."""
import numpy as np
import pytest

import pathtracercuda_b200 as pt
from oracle import orc
from tests.device_probe import _rng, probe  # noqa: F401  (probe: the module-scoped fixture that builds device_probe.cu)

PI = np.pi
ULP = 2.0 ** -24            # half an ulp of 1: the relative rounding of one fp32 operation
STEP = 2.0 ** -8            # the texture unit's filter weights: 8 fractional bits (CUDA programming guide, "Linear Filtering")
# The texture unit, measured on the B200 (test_texture_unit_weight_rule): filtering along one axis, each weight is the fractional
# part rounded to the nearest 1/256, a tie rounding up, taken from a coordinate the unit holds to about 2^-21 of the texture's extent -
# so within that distance of a tie the weight may come out one step lower.  RGBA8 taps carry one more rounding, within 2^-17.  The
# rule test uses twice both.
TEX_UNIT_WEIGHTS = "round"
HW_COORD = 2.0 ** -20       # the unit's coordinate error, in u (or v) x max(1, |u|)
HW_LDR = 2.0 ** -16         # the rounding of an RGBA8 tap, relative to the largest texel
SIZES = [(1, 1), (1, 7), (7, 1), (2, 2), (5, 3), (257, 129), (2048, 1024)]  # (W, H)


# ---------------------------------------------------------------------------------------------------------------------------------
# the float64 statement
# ---------------------------------------------------------------------------------------------------------------------------------
def _texels64(texels):
    T = np.asarray(texels).astype(np.float64)
    return T / 255.0 if np.asarray(texels).dtype == np.uint8 else T


def bilinear64(texels, u, v, weight_bits=None, mode="round"):
    """tex2D<float4> of an (H, W, 4) texture (uint8: read as byte / 255; float32 as is) with linear filtering and normalised
    coordinates, in float64 (CUDA programming guide, "Linear Filtering"): x_B = u W - 0.5, i = floor(x_B), alpha = x_B - i (and j,
    beta from v, H); i wraps modulo W, j is clamped to [0, H - 1]; tap = (1 - a)(1 - b) T[j, i] + a (1 - b) T[j, i + 1] + (1 - a) b
    T[j + 1, i] + a b T[j + 1, i + 1].  weight_bits: alpha and beta quantised to that many fractional bits, by rounding to nearest
    with ties up ("round") or by truncation ("trunc").  -> (n, 4)"""
    T = _texels64(texels)
    H, W = T.shape[:2]
    xb = np.asarray(u, np.float64) * W - 0.5  # exact: a float32 u times W < 2^24 fits the float64 significand
    yb = np.asarray(v, np.float64) * H - 0.5
    i, j = np.floor(xb), np.floor(yb)
    a, b = xb - i, yb - j
    if weight_bits is not None:
        s = 2.0 ** weight_bits
        h = 0.5 if mode == "round" else 0.0
        a, b = np.floor(a * s + h) / s, np.floor(b * s + h) / s
    i0, i1 = np.mod(i, W).astype(np.int64), np.mod(i + 1, W).astype(np.int64)
    j0, j1 = np.clip(j, 0, H - 1).astype(np.int64), np.clip(j + 1, 0, H - 1).astype(np.int64)
    a, b = a[:, None], b[:, None]
    return (1 - a) * (1 - b) * T[j0, i0] + a * (1 - b) * T[j0, i1] + (1 - a) * b * T[j1, i0] + a * b * T[j1, i1]


def _cell(T, xb, yb):
    """per lookup: the largest texel difference along x and along y within the cell of (xb, yb), and the largest texel"""
    H, W = T.shape[:2]
    i, j = np.floor(xb), np.floor(yb)
    i0, i1 = np.mod(i, W).astype(np.int64), np.mod(i + 1, W).astype(np.int64)
    j0, j1 = np.clip(j, 0, H - 1).astype(np.int64), np.clip(j + 1, 0, H - 1).astype(np.int64)
    t00, t10, t01, t11 = (T[jj, ii, :3] for jj, ii in ((j0, i0), (j0, i1), (j1, i0), (j1, i1)))
    dx = np.maximum(np.abs(t10 - t00), np.abs(t11 - t01)).max(-1)
    dy = np.maximum(np.abs(t01 - t00), np.abs(t11 - t10)).max(-1)
    m = np.maximum(np.maximum(np.abs(t00), np.abs(t10)), np.maximum(np.abs(t01), np.abs(t11))).max(-1)
    return dx, dy, m


def tap_bound(texels, u, v, eu=0.0, ev=0.0, unit=False, slack=8.0):
    """bound on |tap - bilinear64| per lookup (rgb), for a tap whose coordinates are known to within eu, ev (in u, v) and are then
    scaled and offset in fp32 (u W - 0.5: two roundings, 2^-23 (|u| W + 1) texels).  The tap moves by at most the coordinate
    error times the texel difference along that axis - over every cell the error can reach, since the filter is continuous across
    cell edges.  unit: the texture unit against bilinear64 with TEX_UNIT_WEIGHTS - plus one weight step (2^-8) per axis, and
    HW_LDR for an RGBA8 texture.  Along one axis the step is needed only within the unit's coordinate error of a tie
    (test_texture_unit_weight_rule); filtering in x and y at once, lookups away from any tie are off by up to a step as well (B200:
    up to 1.00 of this bound), so the step is allowed everywhere.  slack: fp32 rounding of the blend, in ulp of the largest of the
    texels involved."""
    T = _texels64(texels)
    H, W = T.shape[:2]
    u, v = np.asarray(u, np.float64), np.asarray(v, np.float64)
    ex = np.asarray(eu, np.float64) * W + 2.0 ** -23 * (np.abs(u) * W + 1)  # in texels
    ey = np.asarray(ev, np.float64) * H + 2.0 ** -23 * (np.abs(v) * H + 1)
    xb, yb = u * W - 0.5, v * H - 0.5
    dx, dy, m = _cell(T, xb, yb)
    for sx in (-1, 1):
        for sy in (-1, 1):
            a, b, c = _cell(T, xb + sx * np.minimum(ex, 1), yb + sy * np.minimum(ey, 1))
            dx, dy, m = np.maximum(dx, a), np.maximum(dy, b), np.maximum(m, c)
    # an error of a texel or more can reach any cell of the row / column
    gx = np.abs(np.diff(np.concatenate([T[..., :3], T[:, :1, :3]], 1), axis=1)).max() if W > 1 else 0.0
    gy = np.abs(np.diff(T[..., :3], axis=0)).max() if H > 1 else 0.0
    dx = np.where(ex >= 1, gx, dx)
    dy = np.where(ey >= 1, gy, dy)
    m = np.where((ex >= 1) | (ey >= 1), np.abs(T[..., :3]).max(), m)
    if not unit:
        return ex * dx + ey * dy + slack * ULP * m
    ldr = HW_LDR if np.asarray(texels).dtype == np.uint8 else 0.0
    return (ex + STEP) * dx + (ey + STEP) * dy + (slack * ULP + ldr) * m


def texture_coords(rng, W, H, n=2048):
    """random (u, v) with |u| <= 8 and v in [-0.5, 1.5], plus texel centres (also shifted by whole periods in u), texel edges, the
    seam (u = 0, 1 and the float32 values next to them) and v at and beyond 0 and 1 -> float32 u, v"""
    f = np.float32
    nx = lambda a, b: float(np.nextafter(f(a), f(b)))  # noqa: E731
    seam = np.array([0.0, 1.0, -1.0, 2.0, -8.0, 8.0, nx(0, 1), nx(0, -1), nx(1, 0), nx(1, 2), nx(-1, 0), 0.5 / W, 1 - 0.5 / W])
    vedge = np.array([0.0, 1.0, -0.3, 1.3, -0.5, 1.5, nx(0, -1), nx(0, 1), nx(1, 0), nx(1, 2), 0.5 / H, 1 - 0.5 / H])
    i, j = rng.integers(0, W, 256), rng.integers(0, H, 256)
    us = [rng.uniform(-8, 8, n), (i + 0.5) / W + rng.integers(-8, 8, 256), i / W, (i + 0.5) / W]
    vs = [rng.uniform(-0.5, 1.5, n), (j + 0.5) / H, j / H, rng.uniform(0, 1, 256)]
    us += [np.repeat(seam, 16), rng.uniform(-8, 8, 16 * len(vedge)), np.repeat(seam, len(vedge))]
    vs += [rng.uniform(-0.5, 1.5, 16 * len(seam)), np.repeat(vedge, 16), np.tile(vedge, len(seam))]
    return np.concatenate(us).astype(f), np.concatenate(vs).astype(f)


def make_texture(rng, W, H, kind):
    """RGBA8 bytes that include 0 and 255, or RGBA32F texels log-uniform over [1e-3, 1e4]"""
    if kind == "ldr":
        img = rng.integers(0, 256, (H, W, 4)).astype(np.uint8)
        flat = img.reshape(-1)
        flat[::5] = 0
        flat[3::7] = 255
        return img
    return np.exp(rng.uniform(np.log(1e-3), np.log(1e4), (H, W, 4))).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. the statement pinned to the oracle's fp32 rule, on the CPU
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["ldr", "hdr"])
def test_bilinear64_matches_the_oracle_rule(kind):
    """orc.Oracle.texture_lookup (the fp32 rule of oracle/pt_oracle.c, which the product's software filter shares) agrees with
    the float64 statement within fp32 rounding of the coordinates and of the blend, on every size and coordinate class"""
    rng = _rng("pin" + kind)
    O = orc.Oracle([pt.make_object("SPHERE")])
    worst = 0.0
    for W, H in SIZES:
        img = make_texture(rng, W, H, kind)
        h = O.add_texture(img)
        u, v = texture_coords(rng, W, H, n=512)
        got = np.array([O.texture_lookup(h, uu, vv) for uu, vv in zip(u, v)], np.float64)
        want = bilinear64(img, u, v)
        err = np.abs(got - want)[:, :3].max(1)
        bound = tap_bound(img, u, v)
        assert (err <= bound).all(), (W, H, np.nonzero(err > bound)[0][:5], u[err > bound][:5], v[err > bound][:5])
        worst = max(worst, float((err / bound).max()))
    print(f"oracle vs bilinear64 ({kind}): largest error / bound {worst:.3f}")


def test_bilinear64_follows_the_definition():
    """the statement on hand-worked taps: texel centres return the texel, the midpoint of two is their mean, u wraps (u = 0 is the
    mean of the last and first column), v clamps (v <= 0.5 / H is the first row), quantised weights round or truncate"""
    img = np.zeros((2, 4, 4), np.float32)
    img[..., 0] = [[1, 2, 3, 4], [10, 20, 30, 40]]
    t = lambda u, v, **k: bilinear64(img, np.float32([u]), np.float32([v]), **k)[0, 0]  # noqa: E731
    assert t(0.125, 0.25) == 1 and t(0.875, 0.75) == 40
    assert t(0.25, 0.25) == 1.5 and t(0.125, 0.5) == 5.5
    assert t(0.0, 0.25) == 2.5 and t(1.0, 0.25) == 2.5 and t(-3.0, 0.25) == 2.5
    assert t(0.125, 0.0) == 1 and t(0.125, -2.0) == 1 and t(0.125, 1.0) == 10 and t(0.125, 7.0) == 10
    # alpha = 0.3 (x_B = 0.3): 77 / 256 rounded, 76 / 256 truncated
    u = np.float32(0.8 / 4)
    a = float(u) * 4 - 0.5
    assert abs(t(u, 0.25, weight_bits=8, mode="round") - (1 + round(a * 256) / 256)) < 1e-12
    assert abs(t(u, 0.25, weight_bits=8, mode="trunc") - (1 + np.floor(a * 256) / 256)) < 1e-12


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. texLookup on the GPU, call by call
# ---------------------------------------------------------------------------------------------------------------------------------
TEX_CASES = pytest.mark.parametrize("kind,W,H", [(k, w, h) for k in ("ldr", "hdr") for w, h in SIZES], ids=lambda x: str(x))


@pytest.mark.gpu
@TEX_CASES
def test_software_filter_matches_bilinear64(probe, kind, W, H):
    """texLookup with texObj = 0 (option tex_unit = 0): exact weights; within fp32 rounding of the coordinates and a few ulp of
    the largest of the four texels"""
    rng = _rng(f"sw{kind}{W}x{H}")
    img = make_texture(rng, W, H, kind)
    u, v = texture_coords(rng, W, H)
    got = probe.tex(img, u, v, 0).astype(np.float64)
    want = bilinear64(img, u, v)[:, :3]
    err = np.abs(got - want).max(1)
    bound = tap_bound(img, u, v, slack=4.0)
    print(f"software filter {kind} {W}x{H}: largest error / bound {(err / bound).max():.3f} over {len(u)} lookups")
    assert (err <= bound).all(), (np.nonzero(err > bound)[0][:5], u[err > bound][:5], v[err > bound][:5])


@pytest.mark.gpu
@TEX_CASES
def test_texture_unit_matches_bilinear64(probe, kind, W, H):
    """texLookup through a texture object with the product's descriptor: bilinear64 with 8-bit weights.  Which quantisation the
    unit applies (the guide does not say) is measured: the model TEX_UNIT_WEIGHTS must do at least as well as the other one.
    Bound: one weight step times the texel difference along each axis, plus fp32 rounding of the coordinates and the blend"""
    rng = _rng(f"hw{kind}{W}x{H}")
    img = make_texture(rng, W, H, kind)
    u, v = texture_coords(rng, W, H)
    got = probe.tex(img, u, v, 1).astype(np.float64)
    errs = {m: np.abs(got - bilinear64(img, u, v, 8, m)[:, :3]).max(1) for m in ("round", "trunc")}
    other = "trunc" if TEX_UNIT_WEIGHTS == "round" else "round"
    err = errs[TEX_UNIT_WEIGHTS]
    bound = tap_bound(img, u, v, unit=True, slack=8.0)
    m = _cell(_texels64(img), u.astype(np.float64) * W - 0.5, v.astype(np.float64) * H - 0.5)[2]
    print(f"texture unit {kind} {W}x{H}: max error / largest texel: round {(errs['round'] / m).max():.3e}, trunc {(errs['trunc'] / m).max():.3e}; "
          f"largest error / bound ({TEX_UNIT_WEIGHTS}) {(err / bound).max():.3f}")
    assert (err <= bound).all(), (np.nonzero(err > bound)[0][:5], u[err > bound][:5], v[err > bound][:5])
    assert err.max() <= errs[other].max()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["ldr", "hdr"])
@pytest.mark.parametrize("axis", ["x", "y"])
def test_texture_unit_weight_rule(probe, kind, axis):
    """the texture unit's weight along one axis, read off a texture of alternating 0 / 1 texels (the tap is the weight): 200 001
    coordinates across 7, 129 and 1024 texels.  Every weight is a multiple of 1/256 (RGBA8: within HW_LDR of one); it is
    floor(256 alpha + 1/2) / 256 of the float64 alpha but within the unit's coordinate error (HW_COORD) of a tie, where it may be
    one step lower; truncating alpha instead gets about every second weight wrong"""
    for N in (7, 129, 1024):
        alt = (np.arange(N) % 2).astype(np.float32)
        img = np.broadcast_to(alt.reshape((1, N, 1) if axis == "x" else (N, 1, 1)), (1, N, 4) if axis == "x" else (N, 1, 4)).copy()
        if kind == "ldr":
            img = (img * 255).astype(np.uint8)
        c = np.linspace(0.0, 1.0, 200001).astype(np.float32)
        half = np.full_like(c, 0.5)
        r = probe.tex(img, c, half, 1) if axis == "x" else probe.tex(img, half, c, 1)
        xb = c.astype(np.float64) * N - 0.5
        i = np.floor(xb)
        inner = (xb > 0.5) & (xb < N - 1.5)  # away from the wrap / clamp at the ends
        w = np.where(i % 2 == 0, r[:, 0], 1 - r[:, 0])[inner] * 256.0
        a = (xb - i)[inner] * 256
        off = np.abs(w - np.rint(w))
        assert off.max() <= (HW_LDR * 256 if kind == "ldr" else 0.0), off.max()  # B200: 1.95e-3 = 2^-17 x 256
        q, model = np.rint(w), np.floor(a + 0.5)
        miss = q != model
        near_tie = np.abs(a - np.floor(a) - 0.5) <= HW_COORD * N * 256  # B200: 0.0146 of a step past the tie at N = 129
        trunc = (q != np.floor(a)).mean()
        print(f"texture unit weights {kind} {axis} N {N}: {miss.sum()} of {len(q)} one step below round-half-up (largest distance "
              f"past the tie {np.max(a[miss] - np.floor(a[miss]) - 0.5, initial=0):.4f} of a step), truncation wrong on {trunc:.3f}; "
              f"RGBA8 rounding {off.max() / 256:.2e}")
        assert (q[miss] == model[miss] - 1).all() and near_tie[miss].all()
        assert trunc > 0.4


# ---------------------------------------------------------------------------------------------------------------------------------
# angles and the gamma step
# ---------------------------------------------------------------------------------------------------------------------------------
def _atan2_inputs(rng):
    f = np.float32
    v = rng.normal(size=(100000, 2))
    t = rng.uniform(1e-3, 10, 2000)
    s = rng.choice([-1.0, 1.0], (2000, 2))
    diag = np.stack([t * s[:, 0], t * s[:, 1]], 1)  # |x| = |y|
    # either side of the reduction threshold tan(pi/8): min / max within +-3 % of it, and within a few ulp
    k = np.concatenate([rng.uniform(-0.03, 0.03, 4000), np.arange(-64, 65) * 2.0 ** -23])
    r = np.tan(PI / 8) * (1 + k)
    mag = np.exp(rng.uniform(np.log(1e-6), np.log(1e6), len(r)))
    swap = rng.random(len(r)) < 0.5
    sg = rng.choice([-1.0, 1.0], (len(r), 2))
    a, b = mag * r, mag
    thr = np.stack([np.where(swap, a, b) * sg[:, 0], np.where(swap, b, a) * sg[:, 1]], 1)
    axes = np.array([[y, x] for y in (0.0, -0.0, 1.0, -1.0, 3e-7, -2.5) for x in (0.0, -0.0, 1.0, -1.0, 2e-7, -4.0)])
    scaled = rng.normal(size=(4000, 2)) * np.exp(rng.uniform(np.log(1e-25), np.log(1e25), (4000, 1)))
    out = np.concatenate([v, diag, thr, axes, scaled]).astype(f)
    return out[:, 0], out[:, 1]


@pytest.mark.gpu
def test_angles_match_float64(probe):
    """fastAtan2 / fastAtan2Inline against float64 arctan2 (axes, +-0, |x| = |y|, either side of the reduction threshold tan(pi/8),
    magnitudes 1e-25 ... 1e25) and fastAcos against float64 arccos over [-1, 1] (with c within a few ulp of +-1, +-0).  The
    direction (+-0, +-0) has no angle: any value in [-pi, pi] is taken.  atan2(-0, x < 0) = -pi may come back as +pi."""
    rng = _rng("angles")
    y, x = _atan2_inputs(rng)
    c = np.concatenate([rng.uniform(-1, 1, 100000), 1 - np.arange(0, 2000) * 2.0 ** -24, -1 + np.arange(0, 2000) * 2.0 ** -24,
                        1 - 2.0 ** -np.arange(1, 25), [0.0, -0.0, 0.5, -0.5]]).astype(np.float32)
    n = max(len(y), len(c))
    yy, xx = np.resize(y, n), np.resize(x, n)
    cc = np.resize(c, n)
    r = probe.angles(yy, xx, cc, np.zeros(n, np.float32)).astype(np.float64)
    ref = np.arctan2(yy.astype(np.float64), xx.astype(np.float64))
    both0 = (yy == 0) & (xx == 0)
    for col, name in ((0, "fastAtan2"), (1, "fastAtan2Inline")):
        e = np.abs(r[:, col] - ref)
        e = np.minimum(e, 2 * PI - e)  # +pi and -pi are the same direction
        assert (np.abs(r[both0, col]) <= np.float32(PI)).all()
        e = e[~both0]
        print(f"{name}: largest error {e.max():.3e} rad")
        assert e.max() < 4e-7  # B200: 2.8e-7
    ea = np.abs(r[:, 2] - np.arccos(cc.astype(np.float64)))
    print(f"fastAcos: largest error {ea.max():.3e} rad (|c| > 0.999: {ea[np.abs(cc) > 0.999].max():.3e})")
    assert ea.max() < 5e-7  # B200: 4.3e-7 (c near -1: pi - r with the float32 pi), 2.1e-7 for |c| > 0.999
    assert r[cc == 1, 2].max() == 0  # acos(1) = 0 exactly: the poles map to v = 0 exactly


@pytest.mark.gpu
def test_gamma_step_matches_float64(probe):
    """fastPow(x, 2.2f) (__powf = ex2.approx(2.2 lg2.approx(x))), the texture's gamma step: relative error against float64
    x ** 2.2f over [0, 1] (every byte value / 255 among them) and the HDR range [1, 1e4]; zero gives exactly 0"""
    rng = _rng("pow")
    ldr = np.concatenate([rng.uniform(0, 1, 100000), np.arange(256) / 255.0, np.exp(rng.uniform(np.log(1e-6), 0, 20000))]).astype(np.float32)
    hdr = np.exp(rng.uniform(0, np.log(1e4), 100000)).astype(np.float32)
    p = np.concatenate([ldr, hdr, [0.0, 1.0]]).astype(np.float32)
    r = probe.angles(np.zeros_like(p), np.ones_like(p), np.zeros_like(p), p)[:, 3].astype(np.float64)
    ref = p.astype(np.float64) ** np.float64(np.float32(2.2))
    nz = p > 0
    e = np.abs(r[nz] - ref[nz]) / ref[nz]
    lo, hi = e[p[nz] <= 1], e[p[nz] > 1]
    print(f"fastPow(x, 2.2f): largest relative error {lo.max():.3e} on (0, 1], {hi.max():.3e} on (1, 1e4]")
    assert r[p == 0][0] == 0.0
    assert lo.max() < 5e-6 and hi.max() < 4e-6  # B200: 4.1e-6, 2.1e-6


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. end to end through the render kernel: with jitter = 0 every sample of a pixel is the pixel-centre ray, and first_hit = 1 reports
# the kernel's own camera-ray hit and t.  Expected rays: the oracle's camera_ray at ((x + 0.5) / W, (y + 0.5) / H); the kernel's
# cameraDir contracts into FMAs and may differ in the last bits, which RAY_ERR (per component) absorbs.
# ---------------------------------------------------------------------------------------------------------------------------------
RAY_ERR = 8 * ULP
ANGLE_ERR = 5e-7  # fastAtan2 / fastAcos (test_angles_match_float64)
# kernel matrix: (variant, spp) x smem_scene x tex_unit; "default": the kernel a user gets at 64 spp, both tex_unit values
FULL = [(var, spp, smem, unit) for var, spp in ((4, 1), (12, 64)) for smem in (1, 0) for unit in (1, 0)]
DEFAULT = [(0, 64, 1, unit) for unit in (1, 0)]
W_IMG, H_IMG = 32, 24


def _camera_rays(cam, W, H):
    O = orc.Oracle([pt.make_object("SPHERE")])
    return np.array([O.camera_ray(cam, np.float32((x + 0.5) / W), np.float32((y + 0.5) / H)) for y in range(H) for x in range(W)], np.float32)


def _render(P, cam, variant, spp, smem, unit, **opts):
    for k, val in dict(jitter=0, first_hit=1, variant=variant, smem_scene=smem, tex_unit=unit, **opts).items():
        P.setOption(k, val)
    P.render(cam, spp, True)
    idx, t = P.firstHit()
    return P.getHDRMean()[..., :3].reshape(-1, 3).astype(np.float64), idx, t


def _look(pos, at, up=(0, 1, 0)):
    return pt.make_camera(pos, at, 70, W_IMG / H_IMG, up=up)


SKY_CAMERAS = {"seam": ((0, 0, 0), (-1, 0.1, 0.05), (0, 1, 0)), "north_pole": ((0, 0, 0), (0, 1, 0), (1, 0, 0)),
               "south_pole": ((0, 0, 0), (0, -1, 0), (0, 0.3, 1)), "oblique": ((0, 0, 0), (0.4, 0.5, -0.7), (0, 1, 0))}
SKIES = {"hdr16x8": (16, 8, "hdr"), "ldr16x8": (16, 8, "ldr"), "hdr1x1": (1, 1, "hdr"), "ldr1x1": (1, 1, "ldr"),
         "ldr1x6": (1, 6, "ldr"), "hdr6x1": (6, 1, "hdr"), "hdr1x5": (1, 5, "hdr"), "ldr9x1": (9, 1, "ldr")}


def _sky_expected(sky, d, unit):
    """the tap at the float64 angles of the float32 ray, and its bound: the ray's last bits and the routines' error, over the
    conditioning of the angles (1 / distance from the pole axis)"""
    d = d.astype(np.float64)
    rho = np.maximum(np.hypot(d[:, 0], d[:, 2]), 1e-30)
    u = np.arctan2(d[:, 2], d[:, 0]) / (2 * PI)
    v = np.arccos(np.clip(d[:, 1], -1, 1)) / PI
    eu = np.minimum((np.sqrt(2) * RAY_ERR / rho + ANGLE_ERR) / (2 * PI) + 2 * ULP, 1.0)
    ev = np.minimum((RAY_ERR / rho + ANGLE_ERR) / PI + 2 * ULP, 1.0)
    want = bilinear64(sky, u, v, 8, TEX_UNIT_WEIGHTS) if unit else bilinear64(sky, u, v)
    return want[:, :3], tap_bound(sky, u, v, eu, ev, unit=bool(unit), slack=16.0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SKIES))
def test_sky_at_a_miss(name):
    """every pixel misses (one small sphere behind the camera): the pixel is the sky's tap at the ray's (u, v) = (atan2(z, x) / 2 pi,
    acos(y) / pi), through the kernel's inlined fastAcos / fastAtan2Inline / texLookup; cameras looking at the seam (-x), at either
    pole and obliquely.  The 16x8 HDR sky runs the whole kernel matrix, the others the default kernel with both tex_unit values."""
    Ws, Hs, kind = SKIES[name]
    rng = _rng("sky" + name)
    sky = make_texture(rng, Ws, Hs, kind)
    worst = {}
    with pt.Pathtracer(W_IMG, H_IMG) as P:
        assert P.loadTextureMem(sky) == 1
        P.setSkyboxTextureHandle(1)
        for cname, (pos, at, up) in SKY_CAMERAS.items():
            cam = _look(pos, at, up)
            d = _camera_rays(cam, W_IMG, H_IMG)[:, 3:]
            view = np.float32(at) / np.linalg.norm(at)
            P.setScene([pt.make_object("SPHERE", position=tuple(-3 * view), scale=(0.1, 0.1, 0.1))])
            for unit in (1, 0):
                want, bound = _sky_expected(sky, d, unit)
                for var, spp, smem, u_ in (FULL if name == "hdr16x8" else DEFAULT):
                    if u_ != unit:
                        continue
                    img, idx, _ = _render(P, cam, var, spp, smem, unit)
                    assert (idx == -1).all()
                    err = np.abs(img - want).max(1)
                    worst[unit] = max(worst.get(unit, 0.0), float((err / bound).max()))
                    bad = err > bound
                    assert not bad.any(), (cname, var, spp, smem, unit, np.nonzero(bad)[0][:5], img[bad][:3], want[bad][:3])
    print(f"sky {name}: largest error / bound: texture unit {worst[1]:.3f}, software filter {worst[0]:.3f}")


@pytest.mark.gpu
def test_sky_handle_out_of_range_is_black():
    """a skybox handle of 0, or above the number of textures loaded, lights nothing: exact zeros (pt_capi.cu sceneDev's guard)"""
    rng = _rng("skyoff")
    with pt.Pathtracer(W_IMG, H_IMG) as P:
        for k in range(3):
            assert P.loadTextureMem(make_texture(rng, 4, 2, "hdr")) == k + 1
        cam = _look((0, 0, 0), (0.4, 0.5, -0.7))
        P.setScene([pt.make_object("SPHERE", position=(0, 0, 5), scale=(0.1, 0.1, 0.1))])
        for handle, lit in ((0, False), (3, True), (4, False), (64, False)):
            P.setSkyboxTextureHandle(handle)
            for var, spp, smem, unit in DEFAULT:
                img, idx, _ = _render(P, cam, var, spp, smem, unit)
                assert (idx == -1).all()
                assert (img > 0).all() if lit else not img.any(), (handle, unit)


# ---------------------------------------------------------------------------------------------------------------------------------
# material taps: one textured LAMBERT shape with a white base under a 1x1 sky of 1.0, max_bounces = 2.  A camera ray that hits the
# outer side of a convex or flat shape scatters once (weight = base, the Lambert f cos / pdf) and reaches the sky, so the pixel is
# tap(u, v)^2.2.  A scattered ray that hits the shape again ends dark: such a pixel holds tap^2.2 x k / spp, k = its samples that
# reached the sky.
# ---------------------------------------------------------------------------------------------------------------------------------
def _uv64(shape, rows, o, d, t):
    """surfaceAt's (u, v) in float64 at o + t d in the object's local frame (rows: world -> local, orc.Oracle.object_info), with the
    bound of each from the local point's fp32 rounding (and, for the angles, its conditioning and the routines' error)"""
    R = rows.reshape(3, 4).astype(np.float64)
    o, d, t = o.astype(np.float64), d.astype(np.float64), t.astype(np.float64)
    lo, ld = o @ R[:, :3].T + R[:, 3], d @ R[:, :3].T
    lp = lo + t[:, None] * ld
    elp = 16 * ULP * (np.abs(lo).max(1) + t * np.abs(ld).max(1) + np.abs(R[:, 3]).max())
    zero = np.zeros(len(t))
    if shape == "SPHERE":
        n = lp / np.linalg.norm(lp, axis=1, keepdims=True)
        rho = np.maximum(np.hypot(n[:, 0], n[:, 2]), 1e-30)
        u = 1 - np.arctan2(n[:, 2], n[:, 0]) / (2 * PI)
        v = np.arccos(np.clip(n[:, 1], -1, 1)) / PI
        en = elp / np.linalg.norm(lp, axis=1) + 4 * ULP  # rsqrt.approx normalisation
        return u, v, (np.sqrt(2) * en / rho + ANGLE_ERR) / (2 * PI) + 2 * ULP, (en / rho + ANGLE_ERR) / PI + 2 * ULP
    if shape == "CYLINDER":
        rho = np.maximum(np.hypot(lp[:, 0], lp[:, 2]), 1e-30)
        u = 1 - np.arctan2(lp[:, 2], lp[:, 0]) / (2 * PI)
        return u, 1 - (lp[:, 1] * 0.5 + 0.5), (np.sqrt(2) * elp / rho + ANGLE_ERR) / (2 * PI) + 2 * ULP, elp / 2 + 2 * ULP
    if shape in ("DISK", "QUAD"):
        return lp[:, 0] * 0.5 + 0.5, 1 - (lp[:, 2] * 0.5 + 0.5), elp / 2 + 2 * ULP, elp / 2 + 2 * ULP
    return zero, zero, zero, zero  # cone, paraboloid, cube: (u, v) defined as 0 (Q3)


def _band(idx, W, H):
    """pixels with a neighbour (8-neighbourhood) that hit something else: the one-pixel silhouette band"""
    a = np.pad(idx.reshape(H, W), 1, mode="edge")
    same = np.ones((H, W), bool)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            same &= a[1 + dy:1 + dy + H, 1 + dx:1 + dx + W] == a[1:1 + H, 1:1 + W]
    return ~same.ravel()


def _check_taps(img, idx, t, rays, spp, unit, expect_of, max_redark, W=W_IMG, H=H_IMG):
    """hit pixels outside the silhouette band: tap^2.2 x k / spp for an integer k (k = spp but for a share of at most max_redark);
    miss pixels: the sky's 1.0 within an ulp.  expect_of(obj, o, d, t, unit) -> (tap^2.2 (n, 3), relative bound (n, 3)).
    -> (largest error / bound, share of pixels with k < spp)"""
    inner = ~_band(idx, W, H)
    miss = inner & (idx == -1)
    assert np.abs(img[miss] - 1.0).max(initial=0) <= 2 * ULP * 2, img[miss].min()
    worst, redark, hits = 0.0, 0, 0
    for obj in np.unique(idx[inner & (idx >= 0)]):
        sel = inner & (idx == obj)
        E, rel = expect_of(int(obj), rays[sel, :3], rays[sel, 3:], t[sel], unit)
        g = img[sel]
        c = np.argmax(E, 1)
        r = np.arange(len(c))
        # (through the texture unit a tap may be off by a weight step: the nearest k is then only the best guess, and the pixel is
        # held to the tap's bound at that k)
        k = np.clip(np.rint(g[r, c] / E[r, c] * spp), 0, spp)
        want = E * (k / spp)[:, None]
        # the tap's bound through the power 2.2, plus __powf (5e-6 relative on [0, 1], 4e-6 above), the Lambert weight f cos / pdf
        # of the scattered direction, which is base only up to MUFU rounding (pixels of one constant tap spread by 3e-5), and the
        # sum of spp samples (spp x 2^-24)
        bound = (rel * 2.2 + 1e-4 + spp * ULP) * E * (k / spp)[:, None] + 1e-30
        err = np.abs(g - want)
        worst = max(worst, float((err / bound).max()))
        assert (err <= bound).all(), (obj, np.nonzero((err > bound).any(1))[0][:5], g[(err > bound).any(1)][:3], want[(err > bound).any(1)][:3])
        redark += int((k < spp).sum())
        hits += len(k)
    share = redark / max(hits, 1)
    assert hits > 0 and share <= max_redark, (hits, share)
    return worst, share


def _one_sky(P):
    h = P.loadTextureMem(np.ones((1, 1, 4), np.float32))
    P.setSkyboxTextureHandle(h)
    return h


def _shape_expect(objs, textures, shapes):
    O = orc.Oracle(objs)
    rows = [O.object_info(i)[0] for i in range(len(objs))]

    def expect_of(obj, o, d, t, unit):
        tex = textures[objs[obj].material.texture - 1]
        u, v, eu, ev = _uv64(shapes[obj], rows[obj], o, d, t)
        tap = (bilinear64(tex, u, v, 8, TEX_UNIT_WEIGHTS) if unit else bilinear64(tex, u, v))[:, :3]
        tb = tap_bound(tex, u, v, eu, ev, unit=bool(unit), slack=16.0)[:, None]
        return tap ** np.float64(np.float32(2.2)), tb / np.maximum(tap, 1e-30)
    return expect_of


# (view from, object rotation in degrees, largest share of pixels with k < spp): the sphere's pole and seam in view, the cylinder
# from the side, disk and quad from above, the cone across both nappes (most rays scattered off one nappe hit the other: every
# pixel is still tap^2.2 x k / spp), the paraboloid from below its rim, the cube on a corner
SHAPE_VIEWS = {"SPHERE": ((-2.2, 2.0, 0.9), (20, 0, 15), 0.01), "CYLINDER": ((-3.0, 0.3, 1.2), (0, 10, 0), 0.01),
               "DISK": ((0.6, 2.5, 1.6), (0, 30, 0), 0.01), "QUAD": ((-0.7, 2.2, -1.8), (0, -20, 0), 0.01),
               "CONE": ((3.0, 0.8, 2.2), (0, 0, 0), 1.0), "PARABOLOID": ((2.5, -1.5, 2.0), (0, 0, 0), 0.5),
               "CUBE": ((2.5, 2.0, 3.0), (0, 25, 0), 0.01)}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPE_VIEWS))
@pytest.mark.parametrize("kind", ["ldr", "hdr"])
def test_material_tap(shape, kind):
    """the material tap behind `tex != 0 && tex <= texCount`, through surfaceAt's (u, v), texLookup and fastPow(tap, 2.2f), against
    (u, v) in float64 at the kernel's own first-hit t, bilinear64 and the power 2.2; the sphere runs the whole kernel matrix, the
    others the default kernel with both tex_unit values"""
    pos, rot, max_redark = SHAPE_VIEWS[shape]
    rng = _rng("mat" + shape + kind)
    tex = make_texture(rng, 8, 4, kind)
    if kind == "ldr":
        tex[..., :3] = np.maximum(tex[..., :3], 160)  # a tap bright enough in every channel to read k off the pixel
    else:
        tex[..., :3] = np.exp(rng.uniform(np.log(0.8), np.log(2.0), (4, 8, 3)))
    objs = [pt.make_object(shape, rotation_deg=rot, material="LAMBERT", base_color=(1, 1, 1), texture=1)]
    cam = _look(pos, (0, 0, 0))
    rays = _camera_rays(cam, W_IMG, H_IMG)
    expect_of = _shape_expect(objs, [tex], [shape])
    worst, shares = {}, []
    with pt.Pathtracer(W_IMG, H_IMG) as P:
        assert P.loadTextureMem(tex) == 1
        _one_sky(P)
        P.setScene(objs)
        for var, spp, smem, unit in (FULL if shape == "SPHERE" else DEFAULT):
            img, idx, t = _render(P, cam, var, spp, smem, unit, max_bounces=2)
            w, share = _check_taps(img, idx, t, rays, spp, unit, expect_of, max_redark)
            worst[unit] = max(worst.get(unit, 0.0), w)
            shares.append(share)
    print(f"material tap {shape} {kind}: largest error / bound: texture unit {worst[1]:.3f}, software filter {worst[0]:.3f}; "
          f"pixels with k < spp: largest share {max(shares):.4f}")


@pytest.mark.gpu
def test_texture_handles():
    """64 textures of mixed kinds and sizes: quads with handles 1, 2, 17, 32, 63 and 64 each show their own texture, handle 0 and 65
    the base colour; in a context with 5 textures, handle 5 is textured and handle 6 shows the base colour (the reference's guard
    `texture <= count`, Material.inl:25-35).  Quads face the camera from below it, in two rows of four."""
    rng = _rng("handles")
    sizes = [(1, 1), (1, 7), (7, 1), (2, 2), (5, 3), (8, 4), (3, 6)]
    textures = []
    for k in range(64):
        W, H = sizes[k % len(sizes)]
        tex = make_texture(rng, W, H, "ldr" if k % 2 else "hdr")
        if k % 2:
            tex[..., :3] = np.maximum(tex[..., :3], 160)
        else:
            tex[..., :3] = np.exp(rng.uniform(np.log(0.8), np.log(2.0), (H, W, 3)))
        textures.append(tex)
    base = (0.3, 0.5, 0.7)
    slots = [(x, z) for z in (-1.5, 1.5) for x in (-4.5, -1.5, 1.5, 4.5)]
    cam = pt.make_camera((0, 10, 0), (0, 0, 0), 50, W_IMG * 2 / (H_IMG * 2), up=(0, 0, -1))
    Wi, Hi = 2 * W_IMG, 2 * H_IMG

    def run(handles, ntex, sky):
        objs = [pt.make_object("QUAD", position=(x, 0, z), material="LAMBERT", base_color=base, texture=h) for (x, z), h in zip(slots, handles)]
        O = orc.Oracle(objs)
        rows = [O.object_info(i)[0] for i in range(len(objs))]
        rays = np.array([O.camera_ray(cam, np.float32((x + 0.5) / Wi), np.float32((y + 0.5) / Hi)) for y in range(Hi) for x in range(Wi)], np.float32)

        def expect_of(obj, o, d, t, unit):
            h = handles[obj]
            if h == 0 or h > ntex:
                return np.tile(np.float64(base), (len(t), 1)), np.zeros((len(t), 3))
            tex = textures[h - 1]
            u, v, eu, ev = _uv64("QUAD", rows[obj], o, d, t)
            tap = (bilinear64(tex, u, v, 8, TEX_UNIT_WEIGHTS) if unit else bilinear64(tex, u, v))[:, :3]
            tb = tap_bound(tex, u, v, eu, ev, unit=bool(unit), slack=16.0)[:, None]
            return tap ** np.float64(np.float32(2.2)), tb / np.maximum(tap, 1e-30)

        with pt.Pathtracer(Wi, Hi) as P:
            for k in range(ntex):
                assert P.loadTextureMem(textures[k]) == k + 1
            P.setSkyboxTextureHandle(sky)
            P.setScene(objs)
            seen = set()
            for var, spp, smem, unit in FULL:
                img, idx, t = _render(P, cam, var, spp, smem, unit, max_bounces=2)
                _check_taps(img, idx, t, rays, spp, unit, expect_of, 0.01, Wi, Hi)
                seen |= set(np.unique(idx[idx >= 0]).tolist())
            assert seen == set(range(len(objs)))

    # the sky, a 1x1 texture of 1.0, is one of the loaded textures that no quad uses: handle 50, and 3 of the first five
    textures[49] = textures[2] = np.ones((1, 1, 4), np.float32)
    run([1, 2, 17, 32, 63, 64, 0, 65], 64, 50)
    run([5, 6, 1, 0, 4, 6, 5, 2], 5, 3)
