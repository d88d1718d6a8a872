"""The trace kernels' per-call device routines on the GPU, one call at a time (tests/device_probe.cu includes trace_device.cuh and
runs each routine once per thread): sampleMaterial / evalMaterial / makeFrame / sampleVNDF against the reference's stored
Material::sample outputs and a float64 statement of brdf.h; testPrimInline + surfaceAt against the reference's stored Hittable::hit
outputs; sampleLight / lightPdfHit / unitLocalNormal against float64 geometry and their own densities; sampleEnv / envPdf against the
table and a float64 statement.  Whole-image tests cannot see a routine that is slightly wrong, or wrong in a branch few paths take;
these look at every call.  Last, the "env_is" / "light_is" kernel twins that the other tests do not reach (scene or stack outside
shared memory) path for path against the restatements.

Tolerances name what they absorb; "B200" is the largest value seen on one B200 (1000 W) and the bound keeps headroom over it."""
import re

import numpy as np
import pytest
from scipy import stats

import pathtracercuda_b200 as pt
from oracle import imgio, orc
from tests.device_probe import ProbeScene, _rng, probe  # noqa: F401  (probe: the module-scoped fixture that builds device_probe.cu)
from tests.helpers import SHAPES7, _local_ok, _mapped_area, bits, golden_objects, load_golden, seven_shape_scene

LAMBERT, GGX, LAMBERT_GGX = 0, 1, 2
PI = np.pi


# ---------------------------------------------------------------------------------------------------------------------------------
# the probe
# ---------------------------------------------------------------------------------------------------------------------------------
def test_probe_compiles_for_sm100a_without_spills(probe):
    kernels = re.findall(r"Compiling entry function '(\w+)' for 'sm_100a'", probe.log)
    assert len(kernels) == 10, probe.log  # material, four hit forms, light, two sky, texture, angles
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", probe.log)
    assert len(spills) == len(kernels) and all(a == "0" and b == "0" for a, b in spills), probe.log


# ---------------------------------------------------------------------------------------------------------------------------------
# materials: float64 statement of evalMaterial (brdf.h D_GGX, V_SmithGGXCorrelated, F_Schlick; MonteCarlo.h's VNDF pdf; the 50/50
# mixture of LAMBERT_GGX), frame-free: N, V (towards the viewer) and L (scattered) in any common frame
# ---------------------------------------------------------------------------------------------------------------------------------
def eval_material64(mtype, base, rough, metal, N, V, L):
    """-> (ok, att[..., 3], pdf) in float64; ok is False where the reference's path ends (attenuation 0 or pdf 0)"""
    mtype, rough, metal = (np.asarray(x, np.float64) for x in (mtype, rough, metal))
    base, N, V, L = (np.asarray(x, np.float64) for x in (base, N, V, L))
    Vz, Lz = (V * N).sum(-1), (L * N).sum(-1)
    a = rough * rough
    a2 = a * a
    NdotV = np.abs(Vz) + 1e-5
    H = V + L
    H = H / np.linalg.norm(H, axis=-1, keepdims=True)
    Hz = (H * N).sum(-1)
    VdotH, NdotH, NdotL = np.clip((V * H).sum(-1), 0, 1), np.clip(Hz, 0, 1), np.clip(Lz, 0, 1)
    with np.errstate(divide="ignore", invalid="ignore"):
        # importanceSampleGGXVNDFPdf (MonteCarlo.h:104-114): D_v(H) / (4 V.H) with D_v = G1(V) V.H D(H) / V.z, D of the unclamped H.z
        dd = (Hz * a2 - Hz) * Hz + 1
        G1 = 2 * Vz / (Vz + np.sqrt(a2 + (1 - a2) * Vz * Vz))
        ggx_pdf = G1 * VdotH * (a2 / (PI * dd * dd)) / Vz / (4 * VdotH)
        # Specular_GGX (brdf.h:56-62): D_GGX * V_SmithGGXCorrelated * F_Schlick
        dn = (NdotH * a2 - NdotH) * NdotH + 1
        D = a2 / (PI * dn * dn)
        Vis = 0.5 / (NdotL * np.sqrt((-NdotV * a2 + NdotV) * NdotV + a2) + NdotV * np.sqrt((-NdotL * a2 + NdotL) * NdotL + a2) + 1e-5)
    F0 = 0.04 * (1 - metal)[..., None] + base * metal[..., None]
    p5 = (1 - VdotH) ** 5
    kS = (D * Vis)[..., None] * (p5[..., None] + F0 * (1 - p5[..., None]))
    lam = (mtype == LAMBERT)[..., None]
    att = np.where(lam, base / PI, np.where((mtype == GGX)[..., None], kS, base * ((1 - metal) / PI)[..., None] + kS))
    pdf = np.where(mtype == LAMBERT, Lz / PI, np.where(mtype == GGX, ggx_pdf, 0.5 * (ggx_pdf + Lz / PI)))
    below = (mtype != LAMBERT) & (Lz < 0)  # Material.inl:82-86, :118-122: attenuation 0 below the horizon
    att = np.where(below[..., None], 0.0, att)
    pdf = np.where(below, 0.0, pdf)
    ok = ~((att == 0).all(-1) | (pdf == 0))
    return ok, att, pdf


def _golden_materials():
    d = load_golden("material_samples")
    m, out = d["mats"], d["out"]
    rough = np.maximum(m[:, 4], np.float32(0.04))  # the reference's Material ctor (Material.inl:12), as scene_compile.cpp stores it
    return m[:, 0].astype(np.int64), m[:, 1:4], rough, m[:, 5], d["N"], d["in_dir"], out


def _ggx_denominator(mtype, rough, N, V, L):
    """dn = alpha^2 + (1 - alpha^2)(1 - H.z^2) of D_GGX, in float64 (1 for LAMBERT).  A float32 evaluation of the GGX terms carries an
    absolute error of a few ulp of 1 in 1 - H.z^2, so its relative error grows as 1 / dn: at roughness 0.04 (alpha^2 = 2.6e-6) near the
    lobe's peak a float32 D is good to a few per cent, however it is computed.  Relative errors of the GGX terms are judged x dn."""
    V, L, N = (np.asarray(x, np.float64) for x in (V, L, N))
    H = V + L
    H = H / np.linalg.norm(H, axis=-1, keepdims=True)
    Hz = (H * N).sum(-1)
    a2 = np.asarray(rough, np.float64) ** 4
    return np.where(np.asarray(mtype) == LAMBERT, 1.0, (Hz * a2 - Hz) * Hz + 1)


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    e = np.abs(a - b) / (np.abs(b) + 1e-30)
    return e.max(-1) if e.ndim > 1 else e


def test_eval_material64_reproduces_the_golden():
    """the float64 statement at the reference's own (V, scattered) pairs gives the reference's attenuation and pdf: it states the
    same function.  The golden is float32 arithmetic on a direction rounded to float32: relative error x dn (_ggx_denominator)
    within 1e-5 (largest on this data: pdf 6.7e-7, attenuation 4.8e-6)"""
    mt, base, rough, metal, N, ind, out = _golden_materials()
    V = -ind.astype(np.float64)
    ok, att, pdf = eval_material64(mt, base, rough, metal, N, V, out[:, 6:9])
    g_ok = ~(((out[:, 2:5] == 0).all(1)) | (out[:, 5] == 0))
    assert np.isfinite(out).all()  # the golden has no NaN rows: nothing to excuse on the device either
    assert np.array_equal(ok, g_ok)
    dn = _ggx_denominator(mt, rough, N, V, out[:, 6:9])[ok]
    e_pdf, e_att = _rel(pdf[ok], out[ok, 5]) * dn, _rel(att[ok], out[ok, 2:5]) * dn
    print(f"float64 statement vs golden: pdf {e_pdf.max():.2e}, att {e_att.max():.2e} (x dn)")
    assert e_pdf.max() < 1e-5 and e_att.max() < 1e-5
    assert np.median(_rel(pdf[ok], out[ok, 5])) < 1e-6


def _mat_input(mt, base, rough, metal, N, ind, r0, r1, sdir=None):
    n = len(mt)
    a = np.zeros((n, 20), np.float32)
    a[:, 0] = mt
    a[:, 1:4] = base
    a[:, 4] = rough
    a[:, 5] = metal
    a[:, 6:9] = N
    a[:, 9:12] = ind
    a[:, 12] = r0
    a[:, 13] = r1
    a[:, 14:17] = (0, 0, 1) if sdir is None else sdir
    return a


@pytest.mark.gpu
def test_sample_material_matches_the_golden(probe):
    mt, base, rough, metal, N, ind, out = _golden_materials()
    r = probe.material(_mat_input(mt, base, rough, metal, N, ind, out[:, 0], out[:, 1]))
    g_ok = ~(((out[:, 2:5] == 0).all(1)) | (out[:, 5] == 0))
    assert np.isfinite(r).all()
    # the path ends exactly where the reference's does
    assert np.array_equal(r[:, 0] == 1, g_ok)
    # the two overloads are the same computation
    assert np.array_equal(bits(r[:, 0:7]), bits(r[:, 8:15]))
    ok = g_ok
    dn = _ggx_denominator(mt, rough, N, -ind, out[:, 6:9])[ok]
    # direction: MUFU sin/cos/sqrt/rsqrt in the lobe samplers and the frame (~1e-6 each) against the reference's IEEE ones
    e_dir = np.abs(r[ok, 1:4] - out[ok, 6:9]).max(1)
    # pdf and weight = att |cos| / pdf (float64 from the golden): MUFU rcp / sqrt in evalMaterial (~2 ulp each, ~10 in a chain) and
    # the direction's own rounding, x dn (_ggx_denominator) for the GGX terms
    e_pdf = _rel(r[ok, 7], out[ok, 5]) * dn
    w64 = out[ok, 2:5].astype(np.float64) * np.abs((out[ok, 6:9] * N[ok]).sum(1, dtype=np.float64))[:, None] / out[ok, 5:6]
    e_w = _rel(r[ok, 4:7], w64) * dn
    print(f"sampleMaterial vs golden ({ok.sum()} rows): direction {e_dir.max():.2e} (99.9 % {np.quantile(e_dir, 0.999):.2e}), "
          f"pdf {e_pdf.max():.2e}, weight {e_w.max():.2e} (x dn); median pdf {np.median(_rel(r[ok, 7], out[ok, 5])):.2e}")
    # (B200: direction 8.5e-6, pdf 1.8e-5, weight 1.3e-4 - the weight carries |cos| of a direction that may graze the surface)
    assert e_dir.max() < 5e-5
    assert e_pdf.max() < 1e-4 and e_w.max() < 5e-4
    # pdfOut is evalMaterial's pdf at the returned direction: bit for bit where the frame round trip is exact (N = +-z: the frame is
    # a signed permutation), to the round trip's rounding elsewhere
    axis = (np.abs(N[:, 2]) == 1) & ok
    assert axis.sum() >= 50 and np.array_equal(r[axis, 20], r[axis, 0])
    assert np.array_equal(bits(r[axis, 24]), bits(r[axis, 7]))
    e_rt = _rel(r[ok, 24], r[ok, 7]) * dn
    print(f"pdfOut vs evalMaterial at toTangent(wi): {e_rt.max():.2e} (x dn)")
    assert e_rt.max() < 1e-5  # B200: 1.7e-6


def _frame_cases(rng, n):
    """normals within 0.001 of +-z (makeFrame's other branch below |N.z| = 0.999 ... above it) and in (0.9, 0.999)"""
    ang = np.concatenate([rng.uniform(0, 0.0447, n // 2), rng.uniform(0.0448, 0.45, n - n // 2)])  # cos(0.0447) = 0.999001
    ang[: n // 8] = rng.uniform(0, 0.001, n // 8)
    phi = rng.uniform(0, 2 * PI, n)
    s = np.where(rng.random(n) < 0.5, 1.0, -1.0)
    N = np.stack([np.sin(ang) * np.cos(phi), np.sin(ang) * np.sin(phi), s * np.cos(ang)], 1)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d = np.where(((d * N).sum(1) > 0)[:, None], -d, d)
    return N.astype(np.float32), d.astype(np.float32)


@pytest.mark.gpu
def test_sample_material_frame_branches_match_the_oracle(probe):
    """near +-z makeFrame switches its helper axis at |N.z| = 0.999 (MonteCarlo.h:5-22); the sampled direction depends on the frame,
    so both sides of the switch are compared with the oracle, which reproduces the reference's Material::sample bit for bit
    (test_material_samples_bit_exact)"""
    rng = _rng("frame")
    n = 3000
    N, ind = _frame_cases(rng, n)
    mt = rng.integers(0, 3, n)
    base = rng.random((n, 3)).astype(np.float32)
    rough = rng.uniform(0.04, 1, n).astype(np.float32)
    metal = rng.random(n).astype(np.float32)
    r0, r1 = rng.random(n).astype(np.float32), rng.random(n).astype(np.float32)
    r = probe.material(_mat_input(mt, base, rough, metal, N, ind, r0, r1))
    O = orc.Oracle([pt.make_object("SPHERE")])
    ref = np.array([O.material_sample(pt.make_object("SPHERE", material=int(mt[k]), base_color=base[k], roughness=float(rough[k]), metalness=float(metal[k])).material,
                                      N[k], ind[k], float(r0[k]), float(r1[k])) for k in range(n)])
    ok = ~(((ref[:, 0:3] == 0).all(1)) | (ref[:, 3] == 0))
    assert np.array_equal(r[:, 0] == 1, ok)
    e_dir = np.abs(r[ok, 1:4] - ref[ok, 4:7]).max(1)
    print(f"frame branches: direction vs oracle {e_dir.max():.2e}")
    assert e_dir.max() < 5e-5  # as in test_sample_material_matches_the_golden (B200: 2.9e-6)


@pytest.mark.gpu
def test_eval_material_matches_float64_on_a_grid(probe):
    """3 types x roughness x metalness x view cosines down to 1e-3 x light directions through the horizon and below it"""
    rows = []
    for mt in (LAMBERT, GGX, LAMBERT_GGX):
        for rough in (0.04, 0.1, 0.3, 0.7, 1.0):
            for metal in (0.0, 0.5, 1.0):
                for cv in (1e-3, 1e-2, 0.1, 0.5, 0.9, 1.0):
                    for cl in (-0.3, -1e-3, 0.0, 1e-3, 1e-2, 0.2, 0.6, 1.0):
                        for pl in np.linspace(0, 2 * PI, 9)[:-1]:
                            rows.append((mt, rough, metal, cv, cl, pl))
    g = np.array(rows)
    n = len(g)
    sv, sl = np.sqrt(1 - g[:, 3] ** 2), np.sqrt(1 - g[:, 4] ** 2)
    V = np.stack([sv * np.cos(0.3), sv * np.sin(0.3), g[:, 3]], 1).astype(np.float32)
    Ld = np.stack([sl * np.cos(g[:, 5]), sl * np.sin(g[:, 5]), g[:, 4]], 1).astype(np.float32)
    base = np.tile(np.float32([0.9, 0.5, 0.1]), (n, 1))
    # N = +z: the probe's tangent frame is then a signed permutation, and V = toTangent(frame, -inDir) comes back exactly
    N = np.tile(np.float32([0, 0, 1]), (n, 1))
    ind = -np.stack([V[:, 1], -V[:, 0], V[:, 2]], 1)
    r = probe.material(_mat_input(g[:, 0], base, g[:, 1], g[:, 2], N, ind, 0.5, 0.5, sdir=Ld))
    assert np.array_equal(r[:, 25:28], V)
    ok, att, pdf = eval_material64(g[:, 0], base, g[:, 1].astype(np.float32), g[:, 2], np.float64([0, 0, 1]), V, Ld)
    assert np.array_equal(r[:, 15] == 1, ok), np.nonzero((r[:, 15] == 1) != ok)[0][:10]
    assert np.isfinite(r[:, 15:20]).all()
    # MUFU rcp / sqrt (~2 ulp each) through ~10 operations, conditioned by the grazing terms: V.z + sqrt(a2 + (1 - a2) V.z^2) and
    # lv + ll + 1e-5 at V.z = 1e-3, and normalize(V + L) where L grazes.  B200: see print
    dn = _ggx_denominator(g[:, 0], g[:, 1].astype(np.float32), np.float64([0, 0, 1]), V, Ld)[ok]
    e_pdf, e_att = _rel(r[ok, 19], pdf[ok]) * dn, _rel(r[ok, 16:19], att[ok]) * dn
    print(f"evalMaterial grid ({ok.sum()} of {n} rows alive): pdf {e_pdf.max():.2e}, att {e_att.max():.2e} (x dn)")
    assert e_pdf.max() < 1e-5 and e_att.max() < 1e-5  # B200: 3.7e-7, 5.1e-7


def _bin_quadrature(f, nc, nphi, sub=48):
    """integral of f(cos theta, phi) over each of nc x nphi bins of the upper hemisphere (d omega = d cos d phi), midpoint rule on
    sub x sub cells per bin"""
    c = (np.arange(nc * sub) + 0.5) / (nc * sub)
    p = (np.arange(nphi * sub) + 0.5) / (nphi * sub) * 2 * PI - PI
    cc, pp = np.meshgrid(c, p, indexing="ij")
    v = f(cc, pp) * (1.0 / (nc * sub)) * (2 * PI / (nphi * sub))
    return v.reshape(nc, sub, nphi, sub).sum((1, 3))


@pytest.mark.gpu
@pytest.mark.parametrize("mt,rough,cv", [(LAMBERT, 0.5, 0.7), (GGX, 0.3, 0.5), (GGX, 0.7, 0.05), (GGX, 1.0, 0.9), (LAMBERT_GGX, 0.3, 0.3), (LAMBERT_GGX, 0.6, 0.02)])
def test_sampler_follows_its_pdf(probe, mt, rough, cv):
    """2^20 draws: chi-square over (cos theta, phi) bins plus the 'path ends' bin (VNDF reflections below the horizon) against the
    float64 pdf integrated per bin, and the mean weight against the float64 integral of f cos over the hemisphere"""
    rng = _rng(f"pdf{mt}{rough}{cv}")
    n = 1 << 20
    base, metal = np.float32([0.8, 0.6, 0.4]), 0.5
    V = np.float64([np.sqrt(1 - cv * cv) * np.cos(0.4), np.sqrt(1 - cv * cv) * np.sin(0.4), cv]).astype(np.float32)
    ind = -np.float32([V[1], -V[0], V[2]])
    r0, r1 = (1.0 - rng.random(n)).astype(np.float32), (1.0 - rng.random(n)).astype(np.float32)  # (0, 1] like uniform01
    r = probe.material(_mat_input(np.full(n, mt), base, rough, metal, np.float32([0, 0, 1]), ind, r0, r1))
    ok = r[:, 0] == 1
    s = r[ok, 28:31].astype(np.float64)
    nc, nphi = 16, 16
    ci = np.minimum((np.clip(s[:, 2], 0, 1) * nc).astype(int), nc - 1)
    pi_ = np.minimum(((np.arctan2(s[:, 1], s[:, 0]) + PI) / (2 * PI) * nphi).astype(int), nphi - 1)
    counts = np.bincount(ci * nphi + pi_, minlength=nc * nphi).astype(np.float64)
    V64 = V.astype(np.float64)

    def dirs(c, p):
        st = np.sqrt(np.maximum(1 - c * c, 0))
        return np.stack([st * np.cos(p), st * np.sin(p), c], -1)

    def pdf_f(c, p):
        return eval_material64(mt, base, np.float32(rough), metal, np.float64([0, 0, 1]), V64, dirs(c, p))[2]

    def fcos_f(c, p):
        _, att, pdf = eval_material64(mt, base, np.float32(rough), metal, np.float64([0, 0, 1]), V64, dirs(c, p))
        return np.where(pdf > 0, att[..., 0] * c, 0.0)

    prob = _bin_quadrature(pdf_f, nc, nphi).ravel()
    obs = np.append(counts, n - ok.sum())
    exp = np.append(prob, max(1.0 - prob.sum(), 0.0)) * n
    keep = exp > 20
    chi2 = ((obs[keep] - exp[keep]) ** 2 / exp[keep]).sum()
    pval = stats.chi2.sf(chi2, keep.sum() - 1)
    # weight: f cos / pdf of each draw, 0 where the path ends; its mean is the float64 integral of f cos
    wsum = np.where(ok, r[:, 4], 0.0).astype(np.float64)
    integral = _bin_quadrature(fcos_f, nc, nphi).sum()
    se = wsum.std() / np.sqrt(n)
    print(f"sampler type {mt} roughness {rough} V.z {cv}: chi2 {chi2:.1f} on {keep.sum() - 1} dof (p {pval:.3g}), ends {n - ok.sum()} vs {exp[-1]:.0f}; "
          f"mean weight {wsum.mean():.6f} vs {integral:.6f} (se {se:.2e})")
    assert abs(exp.sum() - n) < 1e-3 * n and pval > 1e-4
    assert abs(wsum.mean() - integral) < 4 * se + 1e-4 * integral  # (+1e-4: the midpoint quadrature's own error)


# ---------------------------------------------------------------------------------------------------------------------------------
# intersection: testPrimInline<false, EXACT, CLIP> + surfaceAt against the reference's Hittable::hit
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True], ids=["mufu", "exact"])
@pytest.mark.parametrize("clip", [False, True], ids=["noclip", "clip"])
def test_hit_probes_match_the_golden(probe, exact, clip):
    d = load_golden("hit_probes")
    objs, _ = golden_objects(d)
    for o_ in objs:  # the textured flag makes surfaceAt compute the sphere's and cylinder's (u, v) (no texture is read here)
        o_.material.texture = 1
    S = ProbeScene(probe, objs)
    O = orc.Oracle(objs)
    which, o, dd, tmax, res = d["which"], d["o"], d["d"], d["tmax"], d["res"]
    r = S.hit(which, o, dd, tmax, exact, clip)
    g_hit = d["hit"] == 1
    if clip:  # the occlusion form does not take the sphere's far root beyond tMax (Hittable.inl:152-157): that hit is not within tMax
        g_hit = g_hit & (res[:, 0] <= tmax)
    hit = r[:, 0] == 1
    flips = np.nonzero(hit != g_hit)[0]
    for k in flips:
        # a flip is allowed only where the decision lies within float32 rounding: an intersection decision (Oracle.decision_margin,
        # < 100 = within float32 noise of flipping) or t at tMin / tMax
        t = r[k, 1] if hit[k] else res[k, 0]
        near_t = np.isfinite(t) and (abs(t - tmax[k]) <= 1e-5 * abs(t) or abs(t - 0.001) <= 1e-5)
        assert near_t or O.decision_margin(int(which[k]), o[k], dd[k]) < 100, (k, hit[k], g_hit[k], res[k], r[k])
    both = hit & g_hit
    t, tg = r[both, 1], res[both, 0]
    e_t = np.abs(t - tg) / np.abs(tg)
    # t: EXACT form = the reference's IEEE division and square root; what is left is FMA contraction of the local ray and of the
    # quadric's coefficients (nvcc contracts them, the reference's host build does not) times the quadratic's conditioning.  MUFU form:
    # rcp / sqrt (1-2 ulp) on top, which on these probes stays below the contraction's share: B200, both forms, max 2.2e-5 (a grazing
    # probe), 99 % 1.4e-6, no flipped hit decision
    typ = np.array([o_.type for o_ in objs])[which[both]]
    print(f"hit probes exact={exact} clip={clip}: {len(flips)} flips (each within rounding), t max rel {e_t.max():.2e} (99 % {np.quantile(e_t, 0.99):.2e}, 99.9 % {np.quantile(e_t, 0.999):.2e})")
    assert e_t.max() < 1e-4
    assert np.quantile(e_t, 0.99) < 5e-6
    # point, normal (unit, facing the ray), (u, v) except cone / paraboloid / cube, whose u, v the reference never writes (Q3)
    e_p = np.abs(r[both, 2:5] - res[both, 1:4]).max(1) / (1 + np.abs(res[both, 1:4]).max(1))
    e_n = np.abs(r[both, 5:8] - res[both, 4:7]).max(1)
    uvk = ~np.isin(typ, [pt.SHAPES["CONE"], pt.SHAPES["PARABOLOID"], pt.SHAPES["CUBE"]])
    du = np.abs(r[both, 8] - res[both, 7])
    e_uv = np.maximum(np.minimum(du, np.abs(du - 1)), np.abs(r[both, 9] - res[both, 8]))[uvk]  # u wraps at the seam phi = +-pi
    print(f"  p {e_p.max():.2e}, n {e_n.max():.2e}, uv {e_uv.max():.2e}")
    # normal: rsqrt (MUFU) normalisation and the local point's rounding; (u, v): the polynomial acos / atan2 (< 2e-7 rad) and the point
    # (B200: p 4.6e-6, n 3.4e-5, (u, v) 3.6e-6)
    assert e_p.max() < 5e-5 and e_n.max() < 2e-4 and e_uv.max() < 5e-5


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True], ids=["mufu", "exact"])
def test_hit_quirks(probe, exact):
    """a cube entered from inside reports t = tMin (Q2); the sphere's far root beyond tMax is accepted by the closest-hit form (the
    reference, Hittable.inl:152-157) and rejected by the occlusion form (CLIP): the light seen from inside a sphere"""
    rng = _rng("quirks")
    objs = [pt.make_object("CUBE", (0.3, -0.2, 0.1), (20, 30, 40), (1.5, 0.8, 1.1)), pt.make_object("SPHERE", (0, 0, 0), (10, 0, 0), (2.0, 1.0, 1.5))]
    S = ProbeScene(probe, objs)
    n = 512
    o = rng.uniform(-0.3, 0.3, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    big = np.full(n, 3.4028234663852886e38, np.float32)
    for clip in (False, True):
        c = S.hit(np.zeros(n, int), o + np.float32([0.3, -0.2, 0.1]), d, big, exact, clip, tmin=0.001)
        assert (c[:, 0] == 1).all() and (c[:, 1] == np.float32(0.001)).all()
    # sphere: from inside, tMax short of the surface (far root at t >= 1 for every direction here)
    short = np.full(n, 0.5, np.float32)
    a = S.hit(np.ones(n, int), o, d, short, exact, False)
    b = S.hit(np.ones(n, int), o, d, short, exact, True)
    assert (a[:, 0] == 1).all() and (a[:, 1] > 0.5).all()
    assert (b[:, 0] == 0).all()
    full = S.hit(np.ones(n, int), o, d, big, exact, True)
    assert (full[:, 0] == 1).all() and np.array_equal(full[:, 1], a[:, 1])


# ---------------------------------------------------------------------------------------------------------------------------------
# emitters: sampleLight<false> / lightPdfHit<false> / unitLocalNormal
# ---------------------------------------------------------------------------------------------------------------------------------
A_LOCAL = {"SPHERE": 4 * PI, "CYLINDER": 4 * PI, "DISK": PI, "CONE": 2 * np.sqrt(2) * PI, "PARABOLOID": PI * (5 * np.sqrt(5) - 1) / 6, "QUAD": 4.0, "CUBE": 24.0}


def _unit_local_normal64(shape, lp):
    x, y, z = lp[:, 0], lp[:, 1], lp[:, 2]
    if shape == "SPHERE":
        n = lp.copy()
    elif shape == "CYLINDER":
        n = np.stack([x, 0 * y, z], 1)
    elif shape == "CONE":
        n = np.stack([x, -y, z], 1)
    elif shape == "PARABOLOID":
        n = np.stack([2 * x, -np.ones_like(y), 2 * z], 1)
    elif shape == "CUBE":
        n = np.zeros_like(lp)
        ax = np.abs(lp).argmax(1)
        n[np.arange(len(lp)), ax] = 1.0
    else:
        n = np.stack([0 * x, np.ones_like(y), 0 * z], 1)
    return n / np.linalg.norm(n, axis=1, keepdims=True)


def _emitter(shape, rng):
    rot = rng.uniform(-180, 180, 3)
    sc = rng.uniform(0.1, 2.0, 3)
    sc[rng.integers(3)] = 0.1
    sc[(np.argmin(sc) + 1) % 3] = 2.0  # non-uniform up to 1:20
    return pt.make_object(shape, rng.uniform(-1, 1, 3), rot, sc, emissive=(1.0, 2.0, 3.0))


def _origins(rng, n, centre, r=5.0):
    v = rng.normal(size=(n, 3))
    return (centre + r * v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES7)
def test_sample_light_geometry_pdf_and_density(probe, shape):
    rng = _rng("light" + shape)
    o = _emitter(shape, rng)
    S = ProbeScene(probe, [o])
    assert S.emitters == 1
    Wt = orc.Oracle([o]).object_info(0)[0].reshape(3, 4).astype(np.float64)  # the product's world->local rows (bit-identical to the reference's, test_transforms_boxes_bvh_camera)
    n = 1 << 16
    q = rng.integers(0, 2 ** 32, (n, 4), dtype=np.uint64).astype(np.uint32)
    P = _origins(rng, n, np.array(o.position, np.float64))
    r = S.light(q, P)
    assert not np.isnan(r).any()
    ok = r[:, 0] == 1
    assert ok.mean() > 0.999 and (r[ok, 6] == S.prim_of[0]).all()
    w = r[ok, 1:4].astype(np.float64)
    dist = r[ok, 4].astype(np.float64)
    X = P[ok] + dist[:, None] * w
    lp = X @ Wt[:, :3].T + Wt[:, 3]
    # the point lies on the mapped surface: float32 X (|X| ~ 5, ulp ~5e-7) through W (scales up to 10)
    assert _local_ok(shape, lp, 5e-5 * max(1.0, np.abs(lp).max())).all()
    # the pdf: P_sel d^2 / (A_l |det M| |(W^T n_l) . w|) in double, n_l the unit local normal at the point
    nl = _unit_local_normal64(shape, lp)
    wn = nl @ Wt[:, :3]
    detM = 1.0 / abs(np.linalg.det(Wt[:, :3]))
    cosw = np.abs((wn * w).sum(1))
    pdf64 = dist ** 2 / (A_LOCAL[shape] * detM * cosw)
    # cos of the emitter's normal against w: how grazing the direction is (the pdf's conditioning is 1 / that)
    graze = cosw / np.linalg.norm(wn, axis=1)
    e_pdf = np.abs(r[ok, 5] - pdf64) / pdf64
    e_hit = np.abs(r[ok, 7] - r[ok, 5]) / r[ok, 5]
    # Conditioning: the pdf is 1 / cos of the emitter's normal against w (graze), and the float64 normal here is taken at a point
    # rebuilt from float32 (P, w, dist): ~1e-6 of |X| ~ 5, times W (scales down to 0.1).  The cone's normal turns by that over the
    # distance h to the apex.  MUFU rsqrt / rcp / sincos in the device's own point, normal and direction are ~1e-6 relative.
    cond = graze * (np.minimum(np.abs(lp[:, 1]), 1.0) if shape == "CONE" else 1.0)
    print(f"sampleLight {shape}: pdf vs float64 {np.max(e_pdf * cond):.2e} x cond (median {np.median(e_pdf):.2e}); "
          f"lightPdfHit vs pdf {np.max(e_hit * cond):.2e} x cond")
    # B200: largest x cond 1.8e-4 (sphere at scale 1:20), median a few 1e-7
    assert np.max(e_pdf * cond) < 1e-3 and np.median(e_pdf) < 1e-5
    assert np.max(e_hit * cond) < 1e-3 and np.median(e_hit) < 1e-5
    # the points follow the area density: mean of 1 / p_A = world area; p_A = pdf |cos| / d^2 with the float64 cos
    inv_pA = dist ** 2 / (r[ok, 5].astype(np.float64) * graze)
    M = np.concatenate([np.linalg.inv(Wt[:, :3]), (-np.linalg.inv(Wt[:, :3]) @ Wt[:, 3])[:, None]], 1)
    area = _mapped_area(shape, M)
    se = inv_pA.std() / np.sqrt(len(inv_pA))
    assert abs(inv_pA.mean() - area) < 4 * se + 1e-3 * area, (inv_pA.mean(), area, se)
    # ... and uniform by local area: KS of one local coordinate against its analytic CDF
    x, y, z = lp[:, 0], lp[:, 1], lp[:, 2]
    rr = np.sqrt(x * x + z * z)
    if shape in ("SPHERE", "CYLINDER"):
        sample, cdf = y, lambda t: (np.clip(t, -1, 1) + 1) / 2
    elif shape == "DISK":
        sample, cdf = rr, lambda t: np.clip(t, 0, 1) ** 2
    elif shape == "CONE":
        sample, cdf = np.abs(y), lambda t: np.clip(t, 0, 1) ** 2
    elif shape == "PARABOLOID":
        sample, cdf = rr, lambda t: ((1 + 4 * np.clip(t, 0, 1) ** 2) ** 1.5 - 1) / (5 * np.sqrt(5) - 1)
    elif shape == "QUAD":
        sample, cdf = x, lambda t: (np.clip(t, -1, 1) + 1) / 2
    else:  # CUBE: the first in-face coordinate
        ax = np.abs(lp).argmax(1)
        sample, cdf = lp[np.arange(len(lp)), (ax + 1) % 3], lambda t: (np.clip(t, -1, 1) + 1) / 2
    ks = stats.kstest(sample, cdf)
    assert ks.pvalue > 1e-4, (shape, ks)
    # cube faces and cone nappes: chosen in proportion to their (local) area
    if shape == "CUBE":
        face = np.abs(lp).argmax(1) * 2 + (lp[np.arange(len(lp)), np.abs(lp).argmax(1)] > 0)
        assert stats.chisquare(np.bincount(face, minlength=6)).pvalue > 1e-4
    if shape == "CONE":
        assert stats.chisquare(np.bincount((y > 0).astype(int), minlength=2)).pvalue > 1e-4


@pytest.mark.gpu
def test_sample_light_alias_selection(probe):
    """on a scene with 8 emitters of different weights plus one of weight 0 (mean emission <= 0): the selection frequencies are the
    table's probabilities, the weight-0 emitter is never chosen"""
    objs, _ = seven_shape_scene()
    objs.append(pt.make_object("SPHERE", (2, 2, 2), (0, 0, 0), (0.2, 0.2, 0.2), emissive=(1.0, -2.0, 0.0)))
    idx, prob, _, _ = pt.light_distribution(objs)
    assert len(idx) == 9 and prob[-1] == 0 and idx[-1] == len(objs) - 1
    S = ProbeScene(probe, objs)
    rng = _rng("alias")
    n = 1 << 20
    q = rng.integers(0, 2 ** 32, (n, 4), dtype=np.uint64).astype(np.uint32)
    r = S.light(q, np.zeros((n, 3), np.float32) + np.float32([0, 1.5, 2.5]))
    scene = S.object_of[r[:, 6].astype(int)]
    counts = np.array([(scene == i).sum() for i in idx])
    assert counts.sum() == n and counts[-1] == 0
    assert stats.chisquare(counts[:-1], prob[:-1].astype(np.float64) / prob[:-1].sum() * n).pvalue > 1e-4


@pytest.mark.gpu
def test_sample_light_grazing_never_nan(probe):
    """origins in the plane of a quad or disk emitter see it exactly edge-on: false or a finite pdf, never a NaN"""
    rng = _rng("graze")
    for shape in ("QUAD", "DISK"):
        o = pt.make_object(shape, (0.5, 1.0, -0.5), (30, 40, 50), (1.0, 1.0, 0.3), emissive=(1, 1, 1))
        S = ProbeScene(probe, [o])
        Wt = orc.Oracle([o]).object_info(0)[0].reshape(3, 4).astype(np.float64)
        M = np.linalg.inv(Wt[:, :3])
        n = 4096
        loc = np.stack([rng.uniform(-4, 4, n), np.zeros(n), rng.uniform(-4, 4, n)], 1)
        loc[:, 0] += np.sign(loc[:, 0]) * 1.5  # outside the shape
        P = (loc @ M.T - M @ Wt[:, 3]).astype(np.float32)
        q = rng.integers(0, 2 ** 32, (n, 4), dtype=np.uint64).astype(np.uint32)
        r = S.light(q, P)
        assert not np.isnan(r).any()
        ok = r[:, 0] == 1
        assert np.isfinite(r[ok, 5]).all() and (r[ok, 5] > 0).all()
        print(f"{shape} edge-on: {ok.sum()} of {n} samples kept (float32 rounding leaves the origin a hair off the plane)")


# ---------------------------------------------------------------------------------------------------------------------------------
# sky: sampleEnv / envPdf
# ---------------------------------------------------------------------------------------------------------------------------------
_SKY = None


def _sky():
    global _SKY
    if _SKY is None:
        _SKY = imgio.read_hdr(pt.ASSETS + "/skybox.hdr")
    return _SKY


def _env_density64(img):
    """float64 statement of the cell density (env_sampling.h): cell weight = sum over its texels of luminance x sin(theta) plus a
    floor of 1e-4 x the mean, P(cell) = weight / total; density = P(cell) cells / (2 pi^2)"""
    H, W = img.shape[:2]
    bw, bh = (W + 511) // 512, (H + 255) // 256
    cols, rows = (W + bw - 1) // bw, (H + bh - 1) // bh
    lum = img[..., :3].astype(np.float64) @ np.float64([0.2126, 0.7152, 0.0722])
    lum = np.where((lum > 0) & (lum < 1e30), lum, 0.0)
    lum = lum * np.sin(PI * (np.arange(H) + 0.5) / H)[:, None]
    w = np.zeros((rows, cols))
    np.add.at(w, (np.arange(H)[:, None] // bh, np.arange(W)[None, :] // bw), lum)
    w = w.ravel() + 1e-4 * w.sum() / w.size
    return cols, rows, w / w.sum() * w.size / (2 * PI * PI)


@pytest.mark.gpu
def test_sample_env_pdf_table_and_float64(probe):
    img = _sky()
    cols, rows, q, alias, dens = pt.env_distribution(img)
    c64, r64, dens64 = _env_density64(img)
    assert (c64, r64) == (cols, rows) and np.allclose(dens, dens64, rtol=1e-6)
    rng = _rng("env")
    n = 1 << 20
    qq = rng.integers(0, 2 ** 32, (n, 4), dtype=np.uint64).astype(np.uint32)
    r = probe.env(img, qq)
    assert np.isfinite(r).all()
    d, u, v, pdf, pdf_at = r[:, 0:3], r[:, 3], r[:, 4], r[:, 5], r[:, 6]
    # the returned pdf is envPdf at the returned direction: the same cell's density over sin(theta), sin from __sincosf in one and
    # rsqrt(1 - y^2) of the direction in the other (~1e-6 absolute each: relative 1e-6 / sin theta); a draw whose u or v rounds onto
    # the next cell's edge (the uniform is in (0, 1]) is looked up in that cell
    st = np.sin(PI * v.astype(np.float64))
    edge = (np.abs(u * cols - np.round(u * cols)) < 1e-3) | (np.abs(v * rows - np.round(v * rows)) < 1e-3)
    # (near the poles 1 - y^2 of a float32 y cancels: ~1e-7 / sin^2 theta relative)
    e = np.abs(pdf_at - pdf) / pdf * st * st
    print(f"sampleEnv pdf vs envPdf: {e[~edge].max():.2e} x sin^2(theta); {edge.sum()} draws at a cell edge")
    assert e[~edge].max() < 3e-6  # B200: 3.4e-7
    # density / sin(theta) against the float64 statement, cell by cell
    cell = np.minimum((v * rows).astype(int), rows - 1) * cols + np.minimum((u * cols).astype(int), cols - 1)
    # (__sincosf: ~4e-7 absolute in sin theta, relative 4e-7 / sin theta; B200: 1.1e-4 at the smallest sin theta drawn)
    e64 = np.abs(pdf * st - dens64[cell]) / dens64[cell]
    print(f"sampleEnv pdf x sin(theta) vs float64 density: {e64[~edge].max():.2e}")
    assert e64[~edge].max() < 1e-5 / st[~edge].min() + 1e-5
    # the direction is the one of (u, v) (trace.cu:123-127 convention)
    d64 = np.stack([st * np.cos(2 * PI * u), np.cos(PI * v.astype(np.float64)), st * np.sin(2 * PI * u)], 1)
    assert np.abs(d - d64).max() < 1e-5
    # cell frequencies follow the table (chi-square over the cells with enough expected draws, the rest pooled)
    P = dens.astype(np.float64) * 2 * PI * PI / (cols * rows)
    counts = np.bincount(cell, minlength=cols * rows).astype(np.float64)
    exp = P / P.sum() * n
    big = exp > 20
    obs_b, exp_b = np.append(counts[big], counts[~big].sum()), np.append(exp[big], exp[~big].sum())
    chi2 = ((obs_b - exp_b) ** 2 / exp_b).sum()
    pval = stats.chi2.sf(chi2, len(obs_b) - 1)
    print(f"sky cells: chi2 {chi2:.0f} on {len(obs_b) - 1} dof, p {pval:.3g}")
    assert pval > 1e-4


@pytest.mark.gpu
def test_env_pdf_wraps_u_and_clamps_v(probe):
    img = _sky()
    cols, rows, _, _, dens = pt.env_distribution(img)
    rng = _rng("wrap")
    n = 4096
    c, rw = rng.integers(0, cols, n), rng.integers(0, rows, n)
    u = ((c + 0.5) / cols).astype(np.float32)
    v = ((rw + 0.5) / rows).astype(np.float32)
    y = np.cos(PI * v.astype(np.float64)).astype(np.float32)
    base = probe.env(img, np.stack([u, v, y], 1), mode=1)
    # (MUFU rsqrt: ~2 ulp)
    assert np.allclose(base, dens[rw * cols + c] / np.sqrt(np.maximum(1 - y.astype(np.float64) ** 2, 1e-12)), rtol=1e-5)
    for shift in (-1.0, 1.0, -3.0, 2.0):
        got = probe.env(img, np.stack([u + np.float32(shift), v, y], 1), mode=1)
        assert np.array_equal(got, base), shift
    # v at or beyond the poles: the first / last row
    for vv, row in ((-0.25, 0), (0.0, 0), (1.0, rows - 1), (1.5, rows - 1)):
        got = probe.env(img, np.stack([u, np.full(n, vv, np.float32), np.full(n, 0.5, np.float32)], 1), mode=1)
        want = dens[row * cols + c] / np.sqrt(0.75)
        assert np.allclose(got, want, rtol=1e-5), vv


# ---------------------------------------------------------------------------------------------------------------------------------
# the "light_is" / "env_is" kernel twins end to end: variant 4 (32 spp) and 12 (256 spp) x scene in shared / global memory x traversal
# stack in shared / local memory, path for path against the restatements with test_render_matches_oracle_path_for_path's criteria
# ---------------------------------------------------------------------------------------------------------------------------------
_REFS = {}
# Ray counts on seven_shape_scene: the CUDA path traces 0.1 - 0.35 % more rays than the restatement (B200: +0.31 % at 32 spp, +0.34 % at
# 256, +0.13 % at max_bounces 2); with the hoisted panel dark the two agree to 0.003 %.  A shading point ON the emissive panel that
# samples the panel itself sees it exactly edge-on: whether the sample lies above the tangent plane (sl.z > 0: a shadow ray is traced,
# worth ~1e-7 / p_light ~ 0) is decided by the last bits of the hit point, which the CUDA path (MUFU reciprocal, FMA) and the
# restatement (IEEE division, no FMA) round differently.  The image is the same either way; the bound with the panel lit absorbs it.
LIGHT_IS_RAY_TOL = 5e-3


def _path_for_path(a, ra, b, st, spp, ray_tol=1e-3):
    print(f"  rays {st.rays} vs {ra} ({st.rays / ra - 1:+.5f})")
    assert abs(int(st.rays) - int(ra)) <= ray_tol * ra, (st.rays, ra)
    rel = np.abs(a - b)[..., :3] / (np.abs(a[..., :3]) + 1e-3 * spp)
    share = (rel.max(-1) > 1e-3 * max(1.0, spp / 64)).mean()
    print(f"  rays {st.rays} vs {ra}, pixels beyond the per-pixel bound {share:.4f}, mean ratio {a[..., :3].mean() / b[..., :3].mean():.6f}")
    assert share < 0.04
    assert abs(a[..., :3].mean() / b[..., :3].mean() - 1) < 2e-3
    assert imgio.rmse(a / spp, b / spp)[0] < 0.02


def _render(P, cam, spp, **opts):
    for k, v in opts.items():
        P.setOption(k, v)
    P.render(cam, spp, True)
    return P.getHDRMean() * spp, P.stats()


TWINS = pytest.mark.parametrize("spp,variant", [(32, 4), (256, 12)], ids=["v4", "v12"])
PLACEMENT = pytest.mark.parametrize("smem_scene,smem_stack", [(1, 1), (1, 0), (0, 1), (0, 0)], ids=["scene_smem-stack_smem", "scene_smem-stack_local", "scene_global-stack_smem", "scene_global-stack_local"])


@pytest.mark.gpu
@TWINS
@PLACEMENT
@pytest.mark.parametrize("panel", ["lit", "dark"])
def test_light_is_twins_match_the_restatement(spp, variant, smem_scene, smem_stack, panel):
    """seven_shape_scene: 8 emitters (an alias table of 8 entries, every point sampler, lightPdfHit on curved shapes), a hoisted
    panel, GGX and LAMBERT_GGX; with the panel dark, 7 emitters and the ray counts held to the default bound"""
    W, H = 48, 36
    objs, cam = seven_shape_scene(W, H)
    if panel == "dark":
        objs[2].material.emissive = (0.0, 0.0, 0.0)
    if ("light", spp, panel) not in _REFS:
        O = orc.Oracle(objs)
        O.set_light_is(1)
        _REFS["light", spp, panel] = O.render(cam, W, H, spp)
    a, ra = _REFS["light", spp, panel]
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        b, st = _render(P, cam, spp, light_is=1, variant=variant, smem_scene=smem_scene, smem_stack=smem_stack)
    assert st.scene_in_smem == smem_scene
    _path_for_path(a, ra, b, st, spp, ray_tol=LIGHT_IS_RAY_TOL if panel == "lit" else 1e-3)


@pytest.mark.gpu
@TWINS
@PLACEMENT
def test_env_is_twins_match_the_restatement(spp, variant, smem_scene, smem_stack):
    W, H = (96, 54) if spp == 32 else (80, 45)
    objs, _, _, cam = pt.parse_scene_py(f"{pt.ASSETS}/scenes/generated_scene.json", W, H)
    if ("env", spp) not in _REFS:
        O = orc.Oracle(objs)
        O.add_texture(imgio.read_png(pt.ASSETS + "/earth.png"))
        O.set_skybox(O.add_texture(_sky()))
        O.set_env_is(1)
        _REFS["env", spp] = O.render(cam, W, H, spp)
    a, ra = _REFS["env", spp]
    with pt.Pathtracer(W, H) as P:
        cam2 = P.loadSceneFile(f"{pt.ASSETS}/scenes/generated_scene.json", cwd=pt.ASSETS)
        b, st = _render(P, cam2, spp, env_is=1, variant=variant, smem_scene=smem_scene, smem_stack=smem_stack)
    assert st.scene_in_smem == smem_scene
    _path_for_path(a, ra, b, st, spp)


@pytest.mark.gpu
@pytest.mark.parametrize("max_bounces", [1, 2, 3])
def test_light_is_max_bounces_match_the_restatement(max_bounces):
    """paths of at most 1, 2, 3 segments; at 1 no vertex scatters, so no light is sampled: the plain render's image, bit for bit"""
    W, H, spp = 48, 36, 32
    objs, cam = seven_shape_scene(W, H)
    O = orc.Oracle(objs)
    O.set_light_is(1)
    a, ra = O.render(cam, W, H, spp, max_bounces=max_bounces)
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        b, st = _render(P, cam, spp, light_is=1, max_bounces=max_bounces)
        c, st0 = _render(P, cam, spp, light_is=0)
    _path_for_path(a, ra, b, st, spp, ray_tol=LIGHT_IS_RAY_TOL)
    if max_bounces == 1:
        assert np.array_equal(bits(b), bits(c)) and st.rays == st0.rays
    else:
        assert st.rays > st0.rays


@pytest.mark.gpu
@pytest.mark.parametrize("spp", [32, 256])
def test_plain_kernel_stack_in_local_memory(spp):
    """the plain kernels with the traversal stack in local memory (option smem_stack = 0) against the default (shared memory)"""
    W, H = 80, 45
    out = {}
    for s in (-1, 0):
        with pt.Pathtracer(W, H) as P:
            cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/generated_scene.json", cwd=pt.ASSETS)
            out[s], _ = _render(P, cam, spp, smem_stack=s)
    same = np.array_equal(bits(out[-1]), bits(out[0]))
    print(f"smem_stack 0 vs default at {spp} spp: bit-identical {same}, max rel {np.max(np.abs(out[0] - out[-1]) / (np.abs(out[-1]) + 1e-3 * spp)):.2e}")
    assert same
