"""The denoiser: guide buffers (pt_render_aov) and the edge-avoiding a-trous filter (pt_denoise).

The guides of pixel-centre rays are checked against the first-hit queries that are already gated (pt_primary_pass, pt_trace_rays, the
oracle's texture lookup); the filter against a float64 statement of its definition (`atrous64`, written from include/pt_b200.h and
DESIGN.md), fed the GPU's own sums and guides; and the whole against 4096-spp renders.  Nothing of the renderer may move: the trace
kernels' sums, ray counts and first hits are the same bits with and without the new calls in between."""
import os
import re
import subprocess

import numpy as np
import pytest

import pathtracercuda_b200 as pt
from pathtracercuda_b200 import api
from oracle import imgio, orc
from tests.helpers import ROOT, bits, seven_shape_scene

CLI = os.path.join(ROOT, "pathtracercuda_b200", "bin", "pathtracer_b200")
H3 = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
OTHER = dict(sigma_color=0.3, sigma_normal=0.8, sigma_position=0.2)  # a second sigma set for the float64 comparison


def atrous64(sums, albedo, normal, position, n, K, sigma_color, sigma_normal, sigma_position):
    """float64 statement of the filter: K iterations of 5 x 5 B3 taps 2^i apart (taps outside the image skipped, weights renormalised),
    weight h exp(-|c_p - c_q|^2 / (sigma_c n 2^-i)^2 - |n_p - n_q|^2 / sigma_n^2 - |x_p - x_q|^2 / (sigma_x t_p)^2) on the sums c divided
    by max(albedo, 0.01), multiplied back at the end; pixels without a hit pass through, taps count only between pixels that agree on
    that.  Returns the filtered sums."""
    s = sums.astype(np.float64)
    if K == 0:
        return s
    H, W = s.shape[:2]
    hit = albedo[..., 3] > 0
    div = np.maximum(albedo[..., :3].astype(np.float64), 0.01)
    c = s[..., :3] / div
    nrm, pos, t = normal[..., :3].astype(np.float64), position[..., :3].astype(np.float64), position[..., 3].astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv_x = np.where(hit, 1.0 / (sigma_position * t) ** 2, 0.0)
    for i in range(K):
        step = 2 ** i
        pad = 2 * step
        P = lambda a: np.pad(a, [(pad, pad), (pad, pad)] + [(0, 0)] * (a.ndim - 2))
        cP, nP, xP, hP = P(c), P(nrm), P(pos), P(hit)
        acc = np.zeros_like(c)
        wsum = np.zeros((H, W))
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                sl = (slice(pad + dy * step, pad + dy * step + H), slice(pad + dx * step, pad + dx * step + W))
                cq, nq, xq, hq = cP[sl], nP[sl], xP[sl], hP[sl]
                e = (((c - cq) ** 2).sum(-1) / (sigma_color * n / step) ** 2 + ((nrm - nq) ** 2).sum(-1) / sigma_normal ** 2
                     + ((pos - xq) ** 2).sum(-1) * inv_x)
                w = H3[dy + 2] * H3[dx + 2] * np.exp(-e) * hq  # (hq is 0 outside the image: the padding)
                acc += w[..., None] * cq
                wsum += w
        c = np.where(hit[..., None], acc / np.where(hit, wsum, 1.0)[..., None], c)
    out = s.copy()
    out[..., :3] = np.where(hit[..., None], c * div, s[..., :3])
    return out


# ---------------------------------------------------------------------------------------------------------------
# CPU: the statement itself, the header defaults
# ---------------------------------------------------------------------------------------------------------------
def _random_guides(rng, H=12, W=16):
    sums = rng.uniform(0, 20, (H, W, 4))
    albedo = rng.uniform(0, 1, (H, W, 4))
    albedo[..., 3] = (rng.uniform(0, 1, (H, W)) > 0.2) * rng.uniform(0.1, 1, (H, W))
    normal = rng.normal(size=(H, W, 4))
    position = rng.uniform(-1, 1, (H, W, 4))
    position[..., 3] = rng.uniform(1, 3, (H, W))
    return sums, albedo, normal, position


def test_atrous64_zero_iterations_is_identity():
    sums, albedo, normal, position = _random_guides(np.random.default_rng(1))
    assert np.array_equal(atrous64(sums, albedo, normal, position, 16, 0, 1.0, 0.5, 0.05), sums)


def test_atrous64_keeps_a_constant_image():
    """a constant colour over a constant albedo stays what it was, at every iteration count, whatever the other guides do; pixels
    without a hit keep their own value"""
    rng = np.random.default_rng(2)
    _, albedo, normal, position = _random_guides(rng)
    albedo[..., :3] = (0.3, 0.6, 0.9)
    sums = np.ones_like(albedo) * np.array([0.3, 0.6, 0.9, 1.0]) * 16
    miss = albedo[..., 3] == 0
    sums[miss] = (5.0, 6.0, 7.0, 1.0)
    for K in (1, 3, 5):
        out = atrous64(sums, albedo, normal, position, 16, K, 0.5, 0.5, 0.05)
        assert np.allclose(out, sums, rtol=1e-12, atol=0), K


def test_header_defaults_match_python():
    hdr = open(os.path.join(ROOT, "include", "pt_b200.h")).read()
    got = {k.lower(): float(v.rstrip("f")) for k, v in re.findall(r"#define PT_DENOISE_DEFAULT_([A-Z_]+)\s+([0-9.f]+)", hdr)}
    assert got == {k: float(v) for k, v in api.DENOISE_DEFAULTS.items()}


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _load(P, name):
    if name == "seven_shapes":
        objs, cam = seven_shape_scene(P.width, P.height)
        P.setScene(objs)
        return cam, objs
    cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/{name}.json", cwd=pt.ASSETS)
    objs, _, _, _ = pt.parse_scene_py(f"{pt.ASSETS}/scenes/{name}.json", P.width, P.height)
    return cam, objs


def _oracle(name, objs):
    O = orc.Oracle(objs)
    if name == "cornell_box":
        O.add_texture(imgio.read_png(pt.ASSETS + "/earth.png"))
    return O


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "seven_shapes"])
def test_centre_ray_guides_match_first_hit_queries(name):
    """jitter = 0, one ray per pixel: the guides are the first hits of pt_primary_pass's rays.  Hit fraction = idx >= 0, position =
    o + t d with the primary pass's t (1e-6 relative to |o| or t), normals = pt_trace_rays' for the oracle's camera rays (1e-5), albedo = the
    material's base colour exactly; the walk differs (closestHitWW against closestHit), so a pixel may differ only where the oracle
    puts the ray on a rounding boundary of an intersection decision"""
    W, H = 96, 72
    with pt.Pathtracer(W, H) as P:
        cam, objs = _load(P, name)
        P.setOption("jitter", 0)
        P.renderAOV(cam, 1)
        alb, nrm, pos = (P.aov(k).reshape(-1, 4) for k in ("albedo", "normal", "position"))
        idx, t = P.primaryPass(cam)
        O = _oracle(name, objs)
        rays = np.array([O.camera_ray(cam, np.float32((p % W + 0.5) / W), np.float32((p // W + 0.5) / H)) for p in range(W * H)])
        tidx, tt, tn = P.traceRays(rays[:, :3], rays[:, 3:])
    hit = idx >= 0
    expect = rays[:, :3].astype(np.float64) + t[:, None].astype(np.float64) * rays[:, 3:]
    # (relative to the size of the terms of o + t d: the larger of |o| and t)
    pos_ok = np.linalg.norm(pos[:, :3] - expect, axis=1) <= 1e-6 * np.maximum(np.linalg.norm(rays[:, :3], axis=1), t)
    good = (alb[:, 3] == hit) & np.where(hit, pos_ok & (np.abs(pos[:, 3] - t) <= 1e-6 * t), (nrm[:, :3] == 0).all(1) & (alb[:, :3] == 1).all(1))
    boundary = 0
    for p in np.nonzero(~good)[0]:
        m = min(O.decision_margin(k, rays[p, :3], rays[p, 3:]) for k in range(len(objs)))
        assert m < 1.0, f"pixel {p}: guides {alb[p]}, {pos[p]} vs primary pass ({idx[p]}, {t[p]}) off a decision boundary (margin {m:.3g})"
        boundary += 1
    # normals: pt_trace_rays for the oracle's camera rays, the reference's host arithmetic.  Where that query finds the guide's hit (same
    # object, same t bits) the two normals come from the same surfaceAt: 1e-5.  Elsewhere a direction differs from the device's in its last
    # bits (FMA contraction of the image-plane point), which can move the object hit (a silhouette, counted) or, next to the apex of a cone
    # where the normal turns fast, the normal by more (counted, 1e-3)
    same = good & hit & (tidx == idx)
    exact = same & (tt == t)
    assert np.abs(nrm[exact, :3] - tn[exact]).max() <= 1e-5
    moved = same & ~exact
    worst = float(np.abs(nrm[moved, :3] - tn[moved]).max()) if moved.any() else 0.0
    assert worst <= 1e-3
    other = int((good & (tidx != idx)).sum())
    print(f"{name}: {boundary} of {W * H} pixels on a decision boundary of the primitive test, excluded; {other} where pt_trace_rays names "
          f"another object; {int(exact.sum())} normals within 1e-5, {int(moved.sum())} where its t differs (largest normal difference {worst:.3g})")
    assert boundary <= 2e-3 * W * H + 4 and other <= 2e-3 * W * H + 4
    assert hit.mean() > 0.3
    # albedo: the base colour, exactly, on untextured hits; the texture tap on the textured sphere
    mats = np.array([list(o.material.base_color) for o in objs], np.float32)
    tex = np.array([o.material.texture for o in objs])
    plain = good & hit & (tex[np.maximum(idx, 0)] == 0)
    assert plain.sum() > 0.3 * W * H
    assert np.array_equal(alb[plain, :3], mats[idx[plain]])
    textured = good & hit & (tex[np.maximum(idx, 0)] != 0)
    if name == "cornell_box":
        assert textured.sum() > 20
        worst = 0.0
        for p in np.nonzero(textured)[0]:
            rows, _ = O.object_info(int(idx[p]))
            M = rows.reshape(3, 4).astype(np.float64)
            lp = M[:, :3] @ expect[p] + M[:, 3]  # float64 local hit point on the unit sphere
            n = lp / np.linalg.norm(lp)
            u, v = 1.0 - np.arctan2(n[2], n[0]) / (2 * np.pi), np.arccos(n[1]) / np.pi
            ref = O.texture_lookup(int(tex[idx[p]]), np.float32(u), np.float32(v))[:3].astype(np.float64) ** 2.2
            worst = max(worst, float(np.abs(alb[p, :3] - ref).max()))
        # texture unit: one weight step (2^-8) per axis of the unit texel range (DESIGN.md, texture taps), times the slope of x^2.2
        bound = 2.2 * 2 * 2.0 ** -8
        print(f"textured sphere: {textured.sum()} pixels, largest albedo error {worst:.3g} (bound {bound:.3g})")
        assert worst <= bound


@pytest.mark.gpu
def test_jittered_guides():
    """two calls give the same bits; silhouette pixels are partly hit; another seed moves the rays"""
    W, H = 96, 72
    with pt.Pathtracer(W, H) as P:
        cam, _ = _load(P, "seven_shapes")
        P.renderAOV(cam, 16)
        a = [P.aov(k) for k in ("albedo", "normal", "position")]
        P.renderAOV(cam, 16)
        b = [P.aov(k) for k in ("albedo", "normal", "position")]
        P.setOption("jitter", 0)
        P.renderAOV(cam, 1)
        centre_hit = P.aov("albedo")[..., 3] > 0
        P.setOption("jitter", 1)
        P.setOption("seed", 77)
        P.renderAOV(cam, 16)
        c = P.aov("position")
    for x, y in zip(a, b):
        assert np.array_equal(bits(x), bits(y))
    hf = a[0][..., 3]
    # silhouette: a centre ray that hits next to one that misses
    edge = np.zeros_like(centre_hit)
    edge[:, 1:] |= centre_hit[:, 1:] != centre_hit[:, :-1]
    edge[:, :-1] |= centre_hit[:, 1:] != centre_hit[:, :-1]
    edge[1:] |= centre_hit[1:] != centre_hit[:-1]
    edge[:-1] |= centre_hit[1:] != centre_hit[:-1]
    partial = (hf > 0) & (hf < 1)
    assert partial.sum() > 20 and (partial & edge).sum() > 0.5 * partial.sum(), (partial.sum(), (partial & edge).sum())
    assert set(np.unique(hf * 16)) <= set(range(17))
    assert not np.array_equal(bits(c), bits(a[2]))


def _render_state(P, cam, spp, first_hit):
    st = P.stats()
    out = [bits(P.getHDRSum()), int(st.rays), int(st.samples)]
    if first_hit:
        i, t = P.firstHit()
        out += [i, bits(t)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("mode,scene", [("plain", "cornell_box"), ("first_hit", "cornell_box"), ("env_is", "generated_scene"), ("light_is", "cornell_box")])
@pytest.mark.parametrize("spp", [16, 128])
def test_renders_do_not_move(mode, scene, spp):
    """on one context, the render's sums, ray counts and first hits are the same bits with and without pt_render_aov and pt_denoise
    between two progressive renders"""
    W, H = 64, 48
    with pt.Pathtracer(W, H) as P:
        cam, _ = _load(P, scene)
        first_hit = mode == "first_hit"
        if first_hit:  # (pixel-centre rays: every sample of a pixel records the same first hit)
            P.setOption("jitter", 0)
            P.setOption("first_hit", 1)
        elif mode != "plain":
            P.setOption(mode, 1)
        P.render(cam, spp, True)
        P.render(cam, spp, False)
        a = _render_state(P, cam, spp, first_hit)
        P.render(cam, spp, True)
        P.renderAOV(cam, 8)
        P.denoise()
        P.render(cam, spp, False)
        b = _render_state(P, cam, spp, first_hit)
        P.denoise(iterations=3)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("frames_per_spp", [0, 8])
def test_zero_iterations_is_identity(frames_per_spp):
    W, H = 80, 60
    with pt.Pathtracer(W, H) as P:
        cam, _ = _load(P, "cornell_box")
        P.setOption("frames_per_spp", frames_per_spp)
        P.render(cam, 24, True)
        P.render(cam, 16, False)
        P.renderAOV(cam, 4)
        P.denoise(iterations=0)
        pairs = [(P.getHDRImageData(), P.getDenoisedHDR()), (P.getHDRMean(), P.getDenoisedHDRMean()), (P.getImageData(), P.getDenoisedImage())]
    for a, b in pairs:
        assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _gpu_case(name, W=96, H=72, spp=16):
    P = pt.Pathtracer(W, H)
    cam, _ = _load(P, name)
    P.render(cam, spp, True)
    P.renderAOV(cam, 16)
    return P, cam


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "generated_scene"])
def test_filter_matches_float64_statement(name):
    """the GPU's filter against atrous64 on the GPU's own sums and guides, K = 1, 3, 5, at the defaults and another sigma set"""
    P, cam = _gpu_case(name)
    spp = 16
    with P:
        sums = P.getHDRSum()
        g = [P.aov(k).astype(np.float64) for k in ("albedo", "normal", "position")]
        worst = {}
        for K in (1, 3, 5):
            for label, sig in (("defaults", {k: v for k, v in api.DENOISE_DEFAULTS.items() if k != "iterations"}), ("other", OTHER)):
                P.denoise(iterations=K, **sig)
                got = P.getDenoisedHDRMean().astype(np.float64) * spp
                ref = atrous64(sums, *g, spp, K, **sig)
                scale = np.abs(ref[..., :3]).mean()
                err = np.abs(got[..., :3] - ref[..., :3]) / np.maximum(np.abs(ref[..., :3]), 1e-3 * scale)
                worst[(K, label)] = float(err.max())
                assert np.array_equal(got[..., 3], sums[..., 3].astype(np.float64))
    bound = 5e-5  # (measured on the B200: 4.9e-6 at most)
    print(f"{name}: largest relative difference to float64 per (K, sigmas): " + ", ".join(f"{k}: {v:.3g}" for k, v in worst.items()) + f" (bound {bound:g})")
    assert max(worst.values()) <= bound


def _two_quads(kind, W, H):
    """two abutting quads under a constant sky: of different albedo side by side, or a floor and a wall at right angles"""
    if kind == "albedo":
        objs = [pt.make_object("QUAD", (-1, 0, 0), (0, 0, 0), (1, 1, 2), base_color=(0.8, 0.3, 0.1)),
                pt.make_object("QUAD", (1, 0, 0), (0, 0, 0), (1, 1, 2), base_color=(0.1, 0.3, 0.8))]
        cam = pt.make_camera((0, 3.0, 1.5), (0, 0, 0), 50.0, W / H)
    else:
        objs = [pt.make_object("QUAD", (0, 0, 0), (0, 0, 0), (2, 1, 2), base_color=(0.7, 0.7, 0.7)),
                pt.make_object("QUAD", (0, 2, -2), (90, 0, 0), (2, 1, 2), base_color=(0.7, 0.7, 0.7))]
        cam = pt.make_camera((0, 1.0, 2.5), (0, 0.6, -1), 60.0, W / H)
    return objs, cam


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["albedo", "orientation"])
def test_edges_are_kept(kind):
    """16 spp, default filter: pixels two or more from the edge stay within 15 % (relative, per channel) of the 4096-spp value of their
    own side.  Measured on the B200: 3.1 % beside the albedo edge (a jump of 8x in red and blue), 10.3 % beside the crease, where the
    filter also smooths the occlusion gradient of each side (raw 16 spp there: 26 %)"""
    W, H = 96, 72
    objs, cam = _two_quads(kind, W, H)
    sky = np.ones((1, 1, 4), np.float32)
    out = {}
    for spp in (16, 4096):
        with pt.Pathtracer(W, H) as P:
            P.setScene(objs)
            P.setSkyboxTextureHandle(P.loadTextureMem(sky))
            P.setOption("seed", 1984 if spp == 16 else 7)
            P.render(cam, spp, True)
            if spp == 16:
                P.renderAOV(cam, 16)
                P.denoise()
                out["raw"], out["den"] = P.getHDRMean()[..., :3], P.getDenoisedHDRMean()[..., :3]
                idx, _ = P.primaryPass(cam)
            else:
                out["ref"] = P.getHDRMean()[..., :3]
    idx = idx.reshape(H, W)
    assert (idx == 0).sum() > 0.2 * W * H and (idx == 1).sum() > 0.2 * W * H
    near = np.zeros((H, W), bool)  # within two pixels of the other object, or of a miss
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            sh = np.full((H + 4, W + 4), -2)
            sh[2:-2, 2:-2] = idx
            near |= sh[2 + dy:2 + dy + H, 2 + dx:2 + dx + W] != idx
    keep = ~near & (idx >= 0)
    rel = np.abs(out["den"] - out["ref"]) / out["ref"]
    raw = np.abs(out["raw"] - out["ref"]) / out["ref"]
    tol = 0.15
    print(f"{kind}: {keep.sum()} pixels two or more from the edge: largest relative error denoised {rel[keep].max():.3g} (tolerance {tol}), raw 16 spp {raw[keep].max():.3g}")
    assert rel[keep].max() <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cornell_box", "generated_scene"])
def test_denoised_rmse_below_raw(name):
    """480x270, 16 spp: RMSE of the per-sample mean against a 4096-spp render of another seed, denoised (defaults) against raw"""
    W, H = 480, 270
    with pt.Pathtracer(W, H) as R:
        cam = R.loadSceneFile(f"{pt.ASSETS}/scenes/{name}.json", cwd=pt.ASSETS)
        R.setOption("seed", 7)
        R.render(cam, 4096, True)
        ref = R.getHDRMean()[..., :3].astype(np.float64)
    P, cam = _gpu_case(name, W, H, 16)
    with P:
        P.denoise()
        raw = np.sqrt(np.mean((P.getHDRMean()[..., :3] - ref) ** 2))
        den = np.sqrt(np.mean((P.getDenoisedHDRMean()[..., :3] - ref) ** 2))
    need = 3.0  # (measured on the B200: 5.6 on cornell_box, 3.5 on generated_scene)
    print(f"{name}: RMSE raw {raw:.5f}, denoised {den:.5f}: factor {raw / den:.3f} (asserted > {need})")
    assert raw / den > need


@pytest.mark.gpu
def test_errors_and_lifecycle():
    W, H = 64, 48
    with pt.Pathtracer(W, H) as P:
        cam, _ = _load(P, "cornell_box")
        P.render(cam, 16, True)
        with pytest.raises(pt.PtError, match="no guide buffers"):
            P.denoise()
        with pytest.raises(pt.PtError, match="no pt_render_aov"):
            P.aov("albedo")
        with pytest.raises(pt.PtError, match="no pt_denoise"):
            P.getDenoisedHDR()
        with pytest.raises(pt.PtError, match="spp must be at least 1"):
            P.renderAOV(cam, 0)
        P.renderAOV(cam, 4)
        for bad in (dict(sigma_color=-1.0), dict(sigma_normal=float("nan")), dict(sigma_position=float("inf"))):
            with pytest.raises(pt.PtError, match="finite and not negative"):
                P.denoise(**bad)
        with pytest.raises(pt.PtError, match="at most 12"):
            P.denoise(iterations=13)
        P.denoise(iterations=12)
        P.denoise(sigma_color=0.0, sigma_normal=0.0, sigma_position=0.0)
        assert np.isfinite(P.getDenoisedHDR()).all()
        # the defaults through NULL and through the Python mirror of the header's values
        P.denoise()
        a = P.getDenoisedHDRMean()
        P.denoise(**api.DENOISE_DEFAULTS)
        assert np.array_equal(bits(a), bits(P.getDenoisedHDRMean()))
        # a new scene makes the guides stale
        objs, cam2 = seven_shape_scene(W, H)
        P.setScene(objs)
        with pytest.raises(pt.PtError, match="stale"):
            P.denoise()
        P.render(cam2, 16, True)
        P.renderAOV(cam2, 4)
        P.denoise()
        reused = [P.getDenoisedHDR(), P.getDenoisedImage(), P.aov("position")]
    with pt.Pathtracer(W, H) as F:
        F.setScene(objs)
        F.render(cam2, 16, True)
        F.renderAOV(cam2, 4)
        F.denoise()
        fresh = [F.getDenoisedHDR(), F.getDenoisedImage(), F.aov("position")]
    for a, b in zip(reused, fresh):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_two_gpus_pixel_partition_same_bits():
    W, H = 96, 72
    res = []
    for mask in (0, 3):
        with pt.Pathtracer(W, H, device_mask=mask) as P:
            cam, _ = _load(P, "cornell_box")
            P.render(cam, 64, True)
            P.renderAOV(cam, 16)
            P.denoise()
            res.append([P.getDenoisedHDR(), P.getDenoisedHDRMean(), P.getDenoisedImage()])
    for a, b in zip(*res):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


@pytest.mark.gpu
def test_cli_denoise(tmp_path):
    """--denoise 0 writes the bytes of a run without it (PNG, HDR, HDR with --true-mean); --denoise 5 writes another image"""
    scene = f"{pt.ASSETS}/scenes/cornell_box.json"
    out = {}
    for tag, extra in (("plain", []), ("k0", ["--denoise", "0"]), ("k5", ["--denoise", "5", "--aov-spp", "8"])):
        for fmt, flags in (("png", []), ("hdr", ["-ohdr"]), ("mean.hdr", ["-ohdr", "--true-mean"])):
            path = str(tmp_path / f"{tag}.{fmt}")
            subprocess.run([CLI, "-w", "96", "-h", "72", "-spp", "16", *flags, *extra, "-o", path, scene], cwd=pt.ASSETS, check=True, capture_output=True)
            out[tag, fmt] = open(path, "rb").read()
    for fmt in ("png", "hdr", "mean.hdr"):
        assert out["plain", fmt] == out["k0", fmt], fmt
        assert out["plain", fmt] != out["k5", fmt], fmt
