"""Option "light_is": next-event estimation of the emissive objects with multiple importance sampling (not in the reference; SURVEY.md
Q10).  What has to hold is that it integrates the SAME measure as the reference's estimator (the image converges to the same
picture) with less variance.  The estimator is restated in the oracle (oracle/pt_oracle.c, marked there as not the reference; switched
on with Oracle.set_light_is).  CPU: the emitter table (product == the restatement == an independent numpy statement), the point
sampler against its pdf for every shape under random affine maps, the estimator in the restatement (same mean, lower error), the
command-line flag.  GPU: the CUDA path against the restatement path for path, the noise-floor gate against the
unmodified reference program's stored renders, the Jacobian on a scene with emitters of all seven shapes, and the option's edges."""
import os
import subprocess

import numpy as np
import pytest

import pathtracercuda_b200 as pt
from oracle import imgio, orc
from tests.helpers import ROOT, SHAPES7, _local_ok, _mapped_area, bits, load_golden, seven_shape_scene


def _cornell(W, H):
    objs, tex, sky, cam = pt.parse_scene_py(f"{pt.ASSETS}/scenes/cornell_box.json", W, H)
    return objs, cam


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _numpy_probabilities(O, objs):
    """independent statement: weight = mean emissive x world area (exact for flat shapes and cubes by Nanson's formula, |det M|^(2/3) A_l
    for the curved ones), over the objects with a non-zero emissive channel, in scene order"""
    area_l = {"SPHERE": 4 * np.pi, "CYLINDER": 4 * np.pi, "DISK": np.pi, "CONE": 2 * np.sqrt(2) * np.pi, "PARABOLOID": np.pi * (5 * np.sqrt(5) - 1) / 6,
              "QUAD": 4.0, "CUBE": 24.0}
    names = {v: k for k, v in pt.SHAPES.items()}
    idx, w = [], []
    for i, o in enumerate(objs):
        e = np.array(o.material.emissive[:], np.float64)
        if not e.any():
            continue
        W = O.object_info(i)[0].reshape(3, 4).astype(np.float64)[:, :3]
        dM = abs(1.0 / np.linalg.det(W))
        name = names[o.type]
        rl = np.linalg.norm(W, axis=1)
        if name in ("QUAD", "DISK"):
            a = area_l[name] * dM * rl[1]
        elif name == "CUBE":
            a = 8 * dM * rl.sum()
        else:
            a = area_l[name] * dM ** (2 / 3)
        idx.append(i)
        w.append(max(e.mean(), 0) * a)
    w = np.array(w)
    return np.array(idx), w / w.sum()


@pytest.mark.parametrize("which", ["cornell_box", "seven_shapes"])
def test_light_table_product_oracle_numpy(which):
    objs = _cornell(32, 32)[0] if which == "cornell_box" else seven_shape_scene()[0]
    idx, prob, q, alias = pt.light_distribution(objs)
    O = orc.Oracle(objs)
    O.set_light_is(1)
    i2, p2, q2, a2 = O.light_table()
    assert np.array_equal(idx, i2) and np.array_equal(bits(prob), bits(p2)) and np.array_equal(bits(q), bits(q2)) and np.array_equal(alias, a2)
    ni, npb = _numpy_probabilities(O, objs)
    assert np.array_equal(idx, ni) and np.allclose(prob, npb, rtol=1e-6)
    # the alias table realises these probabilities
    n = len(prob)
    back = q.astype(np.float64).copy()
    np.add.at(back, alias, 1.0 - q.astype(np.float64))
    assert np.allclose(back / n, npb, rtol=2e-5, atol=1e-12)
    if which == "cornell_box":
        assert len(idx) == 1 and prob[0] == 1.0
    else:
        assert len(idx) == 8
    # nothing emits: no table
    assert len(pt.light_distribution([pt.make_object("SPHERE")])[0]) == 0


@pytest.mark.parametrize("shape", SHAPES7)
def test_sampler_on_surface_and_jacobian(shape):
    rng = np.random.default_rng(abs(hash(shape)) % 1000)
    for trial in range(2):
        rot = rng.uniform(-180, 180, 3)
        sc = rng.uniform(0.3, 2.5, 3)
        o = pt.make_object(shape, rng.uniform(-3, 3, 3), rot, sc, emissive=(1, 2, 3))
        O = orc.Oracle([o])
        O.set_light_is(1)
        n = 40000
        s = O.light_sample_points(rng.integers(0, 2 ** 32, (n, 4), dtype=np.uint64).astype(np.uint32))
        x, pA = s[:, :3].astype(np.float64), s[:, 3].astype(np.float64)
        Wt = O.object_info(0)[0].reshape(3, 4).astype(np.float64)
        lp = x @ Wt[:, :3].T + Wt[:, 3]
        assert _local_ok(shape, lp, 1e-4 * max(1.0, np.abs(lp).max())).all()
        Winv = np.linalg.inv(Wt[:, :3])
        M = np.concatenate([Winv, (-Winv @ Wt[:, 3])[:, None]], 1)
        area = _mapped_area(shape, M)
        est = 1.0 / pA
        se = est.std() / np.sqrt(n)
        assert abs(est.mean() - area) < 3 * se + 1e-3 * area, (shape, est.mean(), area, se)


@pytest.mark.parametrize("which", ["cornell_box", "seven_shapes"])
def test_estimator_same_measure_less_variance(which):
    if which == "cornell_box":
        W, H, spp = 32, 32, 64
        objs, cam = _cornell(W, H)
    else:
        W, H, spp = 32, 24, 64
        objs, cam = seven_shape_scene(W, H)
    P = orc.Oracle(objs)  # (no textures loaded in either oracle: the sphere's texture handle resolves to none in both)
    plain, rp = P.render(cam, W, H, spp, stratify=0)
    ref, _ = P.render(cam, W, H, 2048, seed=4242, stratify=0)
    plain2, _ = P.render(cam, W, H, spp, seed=77, stratify=0)
    O = orc.Oracle(objs)
    O.set_light_is(1)
    mis, rm = O.render(cam, W, H, spp, stratify=0)
    mis2, _ = O.render(cam, W, H, spp, seed=99, stratify=0)
    plain, plain2, mis, mis2, ref = (a[..., :3] / s for a, s in ((plain, spp), (plain2, spp), (mis, spp), (mis2, spp), (ref, 2048)))
    assert rm > rp
    e_plain, e_mis = np.sqrt(((plain - ref) ** 2).mean()), np.sqrt(((mis - ref) ** 2).mean())
    print(f"light_is oracle {which}: RMSE at {spp} spp against plain 2048 spp: light_is {e_mis:.5f}, plain {e_plain:.5f}")
    assert e_mis < 0.8 * e_plain, (e_mis, e_plain)
    # means: the difference against the spread of two independent renders of each estimator
    spread = abs(mis.mean() - mis2.mean()) + abs(plain.mean() - plain2.mean())
    assert abs(0.5 * (mis.mean() + mis2.mean()) - 0.5 * (plain.mean() + plain2.mean())) < 4 * spread + 3e-3 * ref.mean()
    assert abs(0.5 * (mis.mean() + mis2.mean()) / ref.mean() - 1) < 0.02


def test_cli_light_is_flag():
    cli = os.path.join(ROOT, "pathtracercuda_b200", "bin", "pathtracer_b200")
    r = subprocess.run([cli, "--light-is", "--seed", "7", "-w", "8", "-h", "8", "x.json"], capture_output=True, text=True)
    assert "Can't parse argument" not in r.stdout and "Width: 8" in r.stdout
    src = open(os.path.join(ROOT, "pathtracercuda_b200", "csrc", "main_cli.cpp")).read()
    assert 'pt_set_option(ctx, "light_is", 1.0)' in src


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("spp", [32, 256])
def test_light_is_matches_oracle_path_for_path(spp):
    """the CUDA path against the restatement: same Philox counters -> same paths, same light samples, same shadow rays; both kernels
    that carry it (one pixel per lane below 64 spp, one pixel per warp above); against the plain render: same mean, other bits"""
    W, H = 64, 48
    objs, cam = _cornell(W, H)
    O = orc.Oracle(objs)
    O.set_light_is(1)
    a, ra = O.render(cam, W, H, spp)
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        P.setOption("light_is", 1)
        P.render(cam, spp, True)
        b = P.getHDRMean() * spp
        st = P.stats()
        P.render(cam, spp, True)
        b2 = P.getHDRMean() * spp
        P.setOption("light_is", 0)
        P.render(cam, spp, True)
        c = P.getHDRMean() * spp
        st0 = P.stats()
    assert np.array_equal(bits(b), bits(b2))
    assert abs(int(st.rays) - int(ra)) <= 1e-3 * ra and st.rays > st0.rays
    assert not np.array_equal(bits(b), bits(c))
    assert abs(a[..., :3].mean() / b[..., :3].mean() - 1) < 5e-3
    assert abs(b[..., :3].mean() / c[..., :3].mean() - 1) < 0.03


def _file_image(P, spp, path):
    pt.write_hdr(path, P.getHDRImageData())
    return imgio.read_hdr(path)[::-1, :, :3] / np.float32(spp / ((spp + 7) // 8))


@pytest.mark.gpu
def test_light_is_noise_floor_gate(tmp_path):
    """cornell_box: the 4096-spp image passes the same noise-floor gate against the unmodified reference program's stored renders as
    the plain estimator (same measure), and at 256 spp its error against the reference's 8192-spp picture is lower"""
    g = load_golden("refpt_cornell_box")
    W, H, spp = int(g["W"]), int(g["H"]), int(g["spp"])
    A, B = g["A"].astype(np.float32), g["B"].astype(np.float32)
    imgs, ms = {}, {}
    with pt.Pathtracer(W, H) as P:
        cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/cornell_box.json", cwd=pt.ASSETS)
        P.setOption("frames_per_spp", 8)
        for tag, on, n in (("mis4096", 1, spp), ("mis256", 1, 256), ("plain256", 0, 256)):
            P.setOption("light_is", on)
            P.render(cam, n, True)
            ms[tag] = P.getTiming()
            imgs[tag] = _file_image(P, n, str(tmp_path / f"{tag}.hdr"))
    floor, nf = imgio.rmse(A, B)
    ra, nfa = imgio.rmse(imgs["mis4096"], A)
    rb, nfb = imgio.rmse(imgs["mis4096"], B)
    ref = 0.5 * (A + B)
    e_mis, _ = imgio.rmse(imgs["mis256"], ref)
    e_plain, _ = imgio.rmse(imgs["plain256"], ref)
    print(f"light_is cornell_box {W}x{H}: 4096 spp RMSE(A, B) = {floor:.6f}, RMSE(light_is, A) = {ra:.6f}, RMSE(light_is, B) = {rb:.6f}; "
          f"256 spp against the reference's 8192: light_is {e_mis:.6f} ({ms['mis256']:.1f} ms), plain {e_plain:.6f} ({ms['plain256']:.1f} ms), "
          f"ratio {e_mis / e_plain:.3f}")
    assert nfa <= nf + 8 and nfb <= nf + 8
    assert ra <= 1.1 * floor and rb <= 1.1 * floor, (ra, rb, floor)
    fin = np.isfinite(A).all(-1) & np.isfinite(imgs["mis4096"]).all(-1)
    assert abs(imgs["mis4096"][fin].mean() / A[fin].mean() - 1) < 3e-3
    assert e_mis < 0.85 * e_plain, (e_mis, e_plain)


@pytest.mark.gpu
def test_light_is_seven_shapes_same_mean():
    """the Jacobian on the device: emitters of every shape under random rotations and non-uniform scales; light_is against plain at
    high spp, means within the noise"""
    W, H, spp = 96, 72, 2048
    objs, cam = seven_shape_scene(W, H)
    out = {}
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        for on in (0, 1):
            P.setOption("light_is", on)
            for seed in (1, 2):
                P.setOption("seed", seed)
                P.render(cam, spp, True)
                out[on, seed] = P.getHDRMean()[..., :3].astype(np.float64)
    m = {k: v.mean() for k, v in out.items()}
    spread = abs(m[0, 1] - m[0, 2]) + abs(m[1, 1] - m[1, 2])
    diff = abs(0.5 * (m[1, 1] + m[1, 2]) - 0.5 * (m[0, 1] + m[0, 2]))
    e_plain = np.sqrt(((out[0, 1] - out[0, 2]) ** 2).mean())
    e_mis = np.sqrt(((out[1, 1] - out[1, 2]) ** 2).mean())
    print(f"light_is seven shapes: mean plain {0.5 * (m[0, 1] + m[0, 2]):.6f}, light_is {0.5 * (m[1, 1] + m[1, 2]):.6f}; seed-to-seed RMSE plain {e_plain:.5f}, light_is {e_mis:.5f}")
    assert diff < 4 * spread + 2e-3 * m[0, 1], (diff, spread)
    assert e_mis < e_plain


@pytest.mark.gpu
def test_light_is_without_emitters_is_plain():
    W, H, spp = 64, 36, 64
    with pt.Pathtracer(W, H) as P:
        cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/generated_scene.json", cwd=pt.ASSETS)
        P.render(cam, spp, True)
        a = P.getHDRMean()
        P.setOption("light_is", 1)
        P.render(cam, spp, True)
        b = P.getHDRMean()
    assert len(pt.light_distribution(pt.parse_scene_py(f"{pt.ASSETS}/scenes/generated_scene.json", W, H)[0])[0]) == 0
    assert np.array_equal(bits(a), bits(b))


@pytest.mark.gpu
@pytest.mark.parametrize("other", [("env_is", 1), ("jitter", 0), ("first_hit", 1)])
def test_light_is_rejected_combinations(other):
    W, H = 32, 32
    objs, cam = _cornell(W, H)
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        P.setOption("light_is", 1)
        P.setOption(*other)
        with pytest.raises(pt.PtError, match="light_is"):
            P.render(cam, 8, True)


@pytest.mark.gpu
def test_light_is_two_gpus_pixel_partition_bit_identical():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    W, H, spp = 64, 48, 128
    objs, cam = _cornell(W, H)
    out = []
    for mask in (0, 3):
        with pt.Pathtracer(W, H, device_mask=mask) as P:
            P.setScene(objs)
            P.setOption("light_is", 1)
            P.render(cam, spp, True)
            out.append(P.getHDRMean())
    assert np.array_equal(bits(out[0]), bits(out[1]))
