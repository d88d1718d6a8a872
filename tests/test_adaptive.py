"""Option "adaptive": a pixel stops at the first checkpoint (m, 2m, ... up to spp) where the standard error of its mean luminance is small.

CPU: the restatement of the rule (tests/adaptive_oracle.c orc_render_adaptive, on top of the oracle) against numpy statements built from
per-sample oracle renders.
GPU: bit identity with the uniform render when no checkpoint falls below spp, path for path against the oracle, the semantics of the
accumulation buffer and the counts, convergence, the refusals, two GPUs and the CLI."""
import ctypes as C
import functools
import os
import subprocess
import tempfile

import numpy as np
import pytest

import pathtracercuda_b200 as pt
from pathtracercuda_b200.api import PtError
from oracle import imgio, orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "pathtracercuda_b200", "bin", "pathtracer_b200")
FLOOR = 1.0 / 256.0  # PT_ADAPTIVE_FLOOR
LUM = np.array([0.2126, 0.7152, 0.0722])


def checkpoints(spp, m):
    """c0 = min(m, spp), c_{j+1} = min(2 c_j, spp), ending at spp"""
    c = [min(m, spp)]
    while c[-1] < spp:
        c.append(min(2 * c[-1], spp))
    return c


@functools.lru_cache(maxsize=None)
def _adaptive_oracle_so():
    """tests/adaptive_oracle.c (the oracle plus orc_render_adaptive), built once per process into a temporary directory with the oracle's
    flags (oracle/Makefile)"""
    out = os.path.join(tempfile.mkdtemp(prefix="pt_adaptive_oracle_"), "libadaptive_oracle.so")
    subprocess.check_call(["gcc", "-std=c11", "-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-o", out,
                           os.path.join(ROOT, "tests", "adaptive_oracle.c"), "-lm"])
    return out


class AdaptiveOracle(orc.Oracle):
    """orc.Oracle over the library built from tests/adaptive_oracle.c: every method of the oracle, plus render_adaptive"""

    def __init__(self, objects):
        saved = orc.ORACLE_SO
        orc.ORACLE_SO = _adaptive_oracle_so()  # (Oracle.__init__ loads the library named there)
        try:
            super().__init__(objects)
        finally:
            orc.ORACLE_SO = saved

    def render_adaptive(self, cam, w, h, spp, min_spp, tau, seed=1984, max_bounces=5, stratify=None):
        """option "adaptive" -> (accum, counts, margin, rays); margin = the pixel's smallest |lhs / rhs - 1| over the checkpoints it
        evaluated (inf: none); stratify as render()"""
        L = self.L
        L.orc_render_adaptive.restype = C.c_uint64
        L.orc_render_adaptive.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, C.c_uint64,
                                          C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_set_stratify(int(spp >= 128 if stratify is None else stratify))
        accum = np.zeros((h, w, 4), np.float32)
        counts = np.zeros((h, w), np.uint32)
        margin = np.zeros((h, w), np.float64)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        rays = L.orc_render_adaptive(self.s, C.byref(cam), w, h, spp, min_spp, tau, seed, max_bounces, ptr(accum), ptr(counts), ptr(margin))
        return accum, counts, margin, rays


def _oracle(scene, W, H, light_is=False):
    objs, _, _, cam = pt.parse_scene_py(f"{pt.ASSETS}/scenes/{scene}.json", W, H)
    O = AdaptiveOracle(objs)
    O.add_texture(imgio.read_png(pt.ASSETS + "/earth.png"))
    if scene == "generated_scene":
        O.set_skybox(O.add_texture(imgio.read_hdr(pt.ASSETS + "/skybox.hdr")))
    if light_is:
        O.set_light_is(1)
    return O, cam


def _statement(samples, spp, m, tau):
    """numpy statement of the rule on per-sample values (spp, H, W, 3) float32 -> (sums scaled to spp, counts)"""
    y = (samples.astype(np.float64) * LUM).sum(-1)
    s1, s2 = np.cumsum(y, 0), np.cumsum(y * y, 0)
    H, W = samples.shape[1:3]
    counts = np.full((H, W), spp, np.uint32)
    done = np.zeros((H, W), bool)
    for c in checkpoints(spp, m)[:-1]:
        a, b = s1[c - 1], s2[c - 1]
        lhs = np.sqrt(np.maximum(b - a * a / c, 0.0) / (c * (c - 1.0)))
        stop = ~done & (lhs <= tau * np.maximum(a / c, FLOOR))
        counts[stop] = c
        done |= stop
    sums = np.zeros((H, W, 3), np.float64)
    for n in np.unique(counts):
        sel = counts == n
        sums[sel] = samples[:n, sel].astype(np.float64).sum(0) * (np.float32(spp) / np.float32(n))
    return sums, counts


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("scene", ["cornell_box", "generated_scene"])
@pytest.mark.parametrize("tau", [0.05, 0.2])
def test_oracle_adaptive_matches_numpy_statement(scene, tau):
    W, H, spp, m = 32, 24, 256, 32
    O, cam = _oracle(scene, W, H)
    samples = np.stack([O.render(cam, W, H, 1, sample_offset=i, stratify=0)[0][..., :3] for i in range(spp)])
    want, wcounts = _statement(samples, spp, m, tau)
    got, counts, margin, _ = O.render_adaptive(cam, W, H, spp, m, tau, stratify=0)
    assert np.array_equal(counts, wcounts)
    assert np.allclose(got[..., :3], want, rtol=1e-5, atol=1e-5)
    assert (counts < spp).any() and (counts > m).any(), np.unique(counts)  # both kinds of pixel occur at these taus
    assert np.isinf(margin[counts == spp]).sum() == 0 or spp == m


@pytest.mark.parametrize("spp,m", [(256, 32), (200, 32), (3, 32), (96, 128), (256, 256)])
def test_oracle_schedule_and_per_interval_strata(spp, m):
    """every pixel's count is a checkpoint; with a tau no lit pixel passes, the sum is that of the intervals rendered on their own
    (orc_render of L samples from sample_offset c_j stratifies its L samples by the same cell rule: the interval's own grid)"""
    W, H = 24, 18
    O, cam = _oracle("cornell_box", W, H)
    got, counts, _, _ = O.render_adaptive(cam, W, H, spp, m, 1e-9, stratify=1)
    cps = checkpoints(spp, m)
    assert set(np.unique(counts)) <= set(cps)
    starts = [0] + cps[:-1]
    parts = [O.render(cam, W, H, e - s, sample_offset=s, stratify=1)[0][..., :3].astype(np.float64) for s, e in zip(starts, cps)]
    # (pixels that see nothing, or only an emitter, have no variance and stop at c0 whatever tau)
    full, first = counts == spp, counts == cps[0]
    assert (full | first).all() and full.any()
    assert np.allclose(got[..., :3][full], sum(parts)[full], rtol=1e-5, atol=1e-5)
    assert np.allclose(got[..., :3][first], parts[0][first] * (np.float32(spp) / np.float32(cps[0])), rtol=1e-5, atol=1e-5)
    if spp <= m:  # one interval: today's stratification, the same sums as a uniform render
        a, _ = O.render(cam, W, H, spp, stratify=1)
        assert np.array_equal(got.view(np.uint32), a.view(np.uint32))


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------------

def _ctx(scene, W, H, **opts):
    P = pt.Pathtracer(W, H)
    cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/{scene}.json", cwd=pt.ASSETS)
    for k, v in opts.items():
        P.setOption(k, v)
    return P, cam


def _render(P, cam, spp, ignore=True):
    P.render(cam, spp, ignore)
    return P.getHDRSum(), P.stats()


ESTIMATORS = {"plain": ("generated_scene", {}), "env_is": ("generated_scene", {"env_is": 1}), "light_is": ("cornell_box", {"light_is": 1})}


@pytest.mark.gpu
@pytest.mark.parametrize("est", list(ESTIMATORS))
@pytest.mark.parametrize("smem_scene", [0, 1])
@pytest.mark.parametrize("smem_stack", [0, 1])
@pytest.mark.parametrize("spp", [32, 96, 256])
def test_one_interval_is_bit_identical_to_uniform(est, smem_scene, smem_stack, spp):
    scene, opts = ESTIMATORS[est]
    W, H = 64, 48
    extra = {"variant": 12} if spp < 64 else {}  # (below 64 spp the default kernel is one pixel per lane)
    P, cam = _ctx(scene, W, H, smem_scene=smem_scene, smem_stack=smem_stack, **opts, **extra)
    with P:
        a, sa = _render(P, cam, spp)
        P.setOption("adaptive", 0.01)
        P.setOption("adaptive_min_spp", max(spp, 32))
        b, sb = _render(P, cam, spp)
        counts = P.sampleCounts()
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert sa.rays == sb.rays and sa.samples == sb.samples == W * H * spp
    assert (counts == spp).all()


@pytest.mark.gpu
@pytest.mark.parametrize("scene,light_is", [("cornell_box", 0), ("cornell_box", 1), ("generated_scene", 0)])
@pytest.mark.parametrize("tau", [0.02, 0.1])
def test_path_for_path_against_oracle(scene, light_is, tau):
    W, H, spp, m = 48, 36, 512, 64
    O, cam = _oracle(scene, W, H, light_is=bool(light_is))
    a, oc, margin, ra = O.render_adaptive(cam, W, H, spp, m, tau)
    P, cam2 = _ctx(scene, W, H, light_is=light_is, adaptive=tau, adaptive_min_spp=m)
    with P:
        b, st = _render(P, cam2, spp)
        gc = P.sampleCounts()
    differ = gc != oc
    near = margin < 1e-3
    print(f"{scene} light_is={light_is} tau={tau}: counts {np.unique(gc)}, {int(differ.sum())} of {W * H} differ, "
          f"{int((differ & near).sum())} of them within margin 1e-3 of the boundary ({int(near.sum())} such pixels)")
    # a path that parts ways at a silhouette (a last-bit difference) moves a pixel's sums as in the uniform test: a few decisions follow
    assert (differ & ~near).mean() < 0.02
    same = ~differ
    rel = np.abs(a - b)[..., :3] / (np.abs(a[..., :3]) + 1e-3 * spp)
    assert (rel.max(-1)[same] > 1e-3 * spp / 64).mean() < 0.04
    assert abs(a[..., :3][same].mean() / b[..., :3][same].mean() - 1) < 2e-3
    assert st.samples == int(gc.sum())


@pytest.mark.gpu
def test_semantics():
    W, H, spp, m = 64, 48, 512, 64
    P, cam = _ctx("generated_scene", W, H, adaptive=0.05, adaptive_min_spp=m)
    with P:
        with pytest.raises(PtError):
            P.sampleCounts()  # before any adaptive render
        s1, st = _render(P, cam, spp)
        c1 = P.sampleCounts()
        s1b, _ = _render(P, cam, spp)
        assert np.array_equal(s1.view(np.uint32), s1b.view(np.uint32)) and np.array_equal(c1, P.sampleCounts())
        assert set(np.unique(c1)) <= set(checkpoints(spp, m)) and (c1 < spp).any()
        assert st.samples == int(c1.sum())
        assert np.allclose(P.getHDRMean(), P.getHDRSum() / spp, rtol=1e-6, atol=0)
        # a progressive call adds the second call's scaled sums (samples spp .. 2 spp - 1)
        P.render(cam, spp, False)
        both = P.getHDRSum()
        P.renderAOV(cam, 16)
        P.denoise()
        assert np.isfinite(P.getDenoisedHDR()).all()
    Q, cam = _ctx("generated_scene", W, H, adaptive=0.05, adaptive_min_spp=m, sample_offset=spp)
    with Q:
        second, _ = _render(Q, cam, spp)
    assert np.array_equal((s1[..., :3] + second[..., :3]).view(np.uint32), both[..., :3].view(np.uint32))
    # a context that had the option on, then 0, renders a fresh context's bits
    P, cam = _ctx("generated_scene", W, H, adaptive=0.05)
    with P:
        _render(P, cam, spp)
        P.setOption("adaptive", 0)
        reused, _ = _render(P, cam, spp)
        with pytest.raises(PtError):
            P.sampleCounts()
    P, cam = _ctx("generated_scene", W, H)
    with P:
        fresh, _ = _render(P, cam, spp)
    assert np.array_equal(reused.view(np.uint32), fresh.view(np.uint32))


@pytest.mark.gpu
def test_pixel_that_sees_nothing_stops_at_m():
    """no sky: a pixel whose camera rays all miss has y = 0 in every sample and stops at the first checkpoint"""
    W, H, spp, m = 48, 36, 1024, 64
    objs = [pt.make_object("SPHERE", (0, 0, -3), scale=(0.6, 0.6, 0.6), emissive=(2, 2, 2)),
            pt.make_object("SPHERE", (0.9, 0, -3), scale=(0.4, 0.4, 0.4), base_color=(0.7, 0.5, 0.3))]
    cam = pt.make_camera((0, 0, 0), (0, 0, -1), 50.0, W / H)
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        P.setOption("adaptive", 0.01)
        P.setOption("adaptive_min_spp", m)
        P.render(cam, spp, True)
        s, c = P.getHDRSum(), P.sampleCounts()
    black = (s[..., :3] == 0).all(-1)
    assert black.mean() > 0.3 and (c[black] == m).all()
    assert (c[~black] > m).any()


def _rmse(a, b):
    return float(np.sqrt(np.mean((a[..., :3].astype(np.float64) - b[..., :3]) ** 2)))


@pytest.mark.gpu
def test_convergence():
    W, H, spp = 96, 72, 4096

    def mean(seed, n, **opts):
        # (light_is: with the plain estimator a pixel whose first m samples all found no light stops on y = 0, a bias DESIGN.md measures)
        P, cam = _ctx("cornell_box", W, H, seed=seed, light_is=1, **opts)
        with P:
            P.render(cam, n, True)
            out = P.getHDRMean()
            return out, (P.sampleCounts() if opts.get("adaptive") else None)

    ref, _ = mean(7, spp)
    uni, _ = mean(1984, spp)
    floor = _rmse(uni, ref)
    small, c = mean(1984, spp, adaptive=0.002)
    print(f"tau 0.002: median count {np.median(c)}, mean ratio {small[..., :3].mean() / ref[..., :3].mean():.5f}, RMSE {_rmse(small, ref):.5f} "
          f"vs noise floor {floor:.5f}")
    assert np.median(c) >= 1024
    assert abs(small[..., :3].mean() / ref[..., :3].mean() - 1) < 0.01
    assert _rmse(small, ref) < 1.25 * floor
    mod, c = mean(1984, spp, adaptive=0.05)
    eq = max(1, int(round(c.sum() / (W * H))))
    same, _ = mean(1984, eq)
    ratio = _rmse(mod, ref) / _rmse(same, ref)
    print(f"tau 0.05: {c.sum()} samples = {eq} spp uniform; RMSE adaptive / uniform at equal samples {ratio:.3f}")
    # (a guard against a broken rule, not a claim that adaptive sampling pays: on one B200 this ratio measured 1.67 - at equal samples the
    # pixels that stop early on a noisy estimate cost more error than the samples saved buy elsewhere; DESIGN.md has the sweep)
    assert ratio <= 2.0


@pytest.mark.gpu
def test_refusals():
    W, H = 32, 24
    P, cam = _ctx("cornell_box", W, H)
    with P:
        for k, v in [("adaptive", -0.1), ("adaptive", float("nan")), ("adaptive", float("inf")), ("adaptive_min_spp", 31)]:
            with pytest.raises(PtError):
                P.setOption(k, v)
        P.setOption("adaptive", 0.05)
        for k, v in [("jitter", 0), ("first_hit", 1), ("variant", 4)]:
            P.setOption(k, v)
            with pytest.raises(PtError, match="adaptive"):
                P.render(cam, 128, True)
            P.setOption(k, {"jitter": 1, "first_hit": 0, "variant": 0}[k])
        P.render(cam, 128, True)


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_two_gpus():
    W, H, spp = 64, 48, 512
    one, cam = _ctx("generated_scene", W, H, adaptive=0.05, adaptive_min_spp=64)
    with one:
        want, _ = _render(one, cam, spp)
        wc = one.sampleCounts()
    for exchange in (1, 0):
        with pt.Pathtracer(W, H, device_mask=3) as P:
            cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/generated_scene.json", cwd=pt.ASSETS)
            for k, v in [("exchange", exchange), ("adaptive", 0.05), ("adaptive_min_spp", 64)]:
                P.setOption(k, v)
            got, st = _render(P, cam, spp)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)) and np.array_equal(P.sampleCounts(), wc)
            assert st.samples == int(wc.sum())
            P.setOption("partition", 1)
            with pytest.raises(PtError, match="sample partition"):
                P.render(cam, spp, True)


@pytest.mark.gpu
def test_cli(tmp_path):
    scene = f"{pt.ASSETS}/scenes/cornell_box.json"
    out = tmp_path / "a.png"
    r = subprocess.run([CLI, "-w", "64", "-h", "48", "-spp", "512", "--adaptive", "0.05", "--adaptive-min", "64", "--stats", "-o", str(out), scene],
                       cwd=pt.ASSETS, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert out.exists() and out.stat().st_size > 0
    import json
    stats = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert 0 < stats["samples_last_launch"] < 64 * 48 * 512
    r = subprocess.run([CLI, "-w", "64", "-h", "48", "-spp", "512", "--adaptive", "0.05", "--slice", "64", "-o", str(tmp_path / "b.png"), scene],
                       cwd=pt.ASSETS, capture_output=True, text=True)
    assert r.returncode != 0
