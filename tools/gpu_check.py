#!/usr/bin/env python3
"""Development probe run on the GPU box: parity of the CUDA path vs the oracle + quick throughput numbers, and the
reference binary timed beside it.  Not a test and not the bench (see tests/ and bench.py); writes gpurun_out/gpu_check.json."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pathtracercuda_b200 as pt
from oracle import imgio, orc

out = {}
sky = imgio.read_hdr(pt.ASSETS + "/skybox.hdr")
earth = imgio.read_png(pt.ASSETS + "/earth.png")


def primary_parity(scene, W, H):
    path = f"{pt.ASSETS}/scenes/{scene}.json"
    objs, tex, skyi, cam = pt.parse_scene_py(path, W, H)
    O = orc.Oracle(objs)
    i1, t1, _ = O.primary_pass(cam, W, H)
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        i2, t2 = P.primaryPass(cam)
    mism = np.nonzero(i1 != i2)[0]
    hit = (i1 >= 0) & (i2 >= 0)
    rel = np.abs(t1 - t2)[hit] / t1[hit]
    return {"scene": scene, "W": W, "H": H, "idx_mismatch": int(len(mism)), "max_rel_t": float(rel.max()),
            "mism_examples": [(int(i), int(i1[i]), int(i2[i]), float(t1[i]), float(t2[i])) for i in mism[:8]]}


def primary_3way(scene, W, H):
    import tempfile
    path = f"{pt.ASSETS}/scenes/{scene}.json"
    objs, tex, skyi, cam = pt.parse_scene_py(path, W, H)
    O = orc.Oracle(objs)
    ih, th, _ = O.primary_pass(cam, W, H)
    with tempfile.TemporaryDirectory() as td:
        ig, tg = orc.ref_gpu_primary(objs, cam, W, H, td)
    with pt.Pathtracer(W, H) as P:
        P.setScene(objs)
        io, to = P.primaryPass(cam)
    def cmp(a, ta, b, tb):
        m = np.nonzero(a != b)[0]
        hit = (a >= 0) & (b >= 0) & (a == b)
        rel = np.abs(ta - tb)[hit] / ta[hit]
        near_tie = int(np.sum(np.abs(ta[m] - tb[m]) <= 1e-5 * np.maximum(np.abs(ta[m]), np.abs(tb[m]))))
        return {"idx_mismatch": int(len(m)), "of_which_t_within_1e-5": near_tie, "max_rel_t_same_idx": float(rel.max()),
                "examples": [(int(i), int(a[i]), int(b[i]), float(ta[i]), float(tb[i])) for i in m[:6]]}
    np.save(f"gpurun_out/primary_{scene}_refgpu_idx.npy", ig)
    np.save(f"gpurun_out/primary_{scene}_ours_idx.npy", io)
    np.save(f"gpurun_out/primary_{scene}_refgpu_t.npy", tg)
    np.save(f"gpurun_out/primary_{scene}_ours_t.npy", to)
    return {"scene": scene, "W": W, "H": H, "ours_vs_refgpu": cmp(io, to, ig, tg), "ours_vs_oracle": cmp(io, to, ih, th), "refgpu_vs_oracle": cmp(ig, tg, ih, th)}


def render_parity(scene, W, H, spp):
    path = f"{pt.ASSETS}/scenes/{scene}.json"
    objs, tex, skyi, cam = pt.parse_scene_py(path, W, H)
    O = orc.Oracle(objs)
    O.add_texture(earth)
    if scene == "generated_scene":
        O.set_skybox(O.add_texture(sky))
    a, ra = O.render(cam, W, H, spp)
    with pt.Pathtracer(W, H) as P:
        cam2 = P.loadSceneFile(path, cwd=pt.ASSETS)
        P.render(cam2, spp, True)
        b = P.getHDRMean() * spp
        st = P.stats()
    d = np.abs(a - b)[..., :3]
    rel = d / (np.abs(a[..., :3]) + 1e-3)
    return {"scene": scene, "rays_oracle": int(ra), "rays_gpu": int(st.rays), "max_abs": float(d.max()),
            "frac_rel_gt_1e-3": float((rel.max(-1) > 1e-3).mean()), "mean_oracle": float(a[..., :3].mean() / spp), "mean_gpu": float(b[..., :3].mean() / spp),
            "rmse": imgio.rmse(a / spp, b / spp)[0], "in_smem": int(st.scene_in_smem)}


def perf(scene, W, H, spp, reps=3, **opts):
    path = f"{pt.ASSETS}/scenes/{scene}.json"
    with pt.Pathtracer(W, H) as P:
        cam = P.loadSceneFile(path, cwd=pt.ASSETS)
        for k, v in opts.items():
            P.setOption(k, v)
        if "max_leaf" in opts:
            cam = P.loadSceneFile(path, cwd=pt.ASSETS)
        P.render(cam, 8, True)
        best = None
        for _ in range(reps):
            P.render(cam, spp, True)
            st = P.stats()
            ms = P.getTiming()
            r = {"ms": ms, "Mrays_s": st.rays / ms / 1e3, "Msamples_s": st.samples / ms / 1e3, "rays_per_sample": st.rays / st.samples,
                 "node_visits_per_ray": st.node_visits / max(st.rays, 1), "prim_tests_per_ray": st.prim_tests / max(st.rays, 1), "in_smem": int(st.scene_in_smem)}
            if best is None or r["ms"] < best["ms"]:
                best = r
    best.update({"scene": scene, "W": W, "H": H, "spp": spp, "opts": opts})
    return best


def ref_pt(scene, W, H, spp):
    exe = orc.REF_PT
    if not os.path.exists(exe):
        return {"unavailable": True}
    t0 = time.time()
    p = subprocess.run([exe, "-w", str(W), "-h", str(H), "-spp", str(spp), f"scenes/{scene}.json"], cwd=pt.ASSETS, capture_output=True, text=True)
    wall = time.time() - t0
    ms = None
    for line in p.stdout.splitlines():
        if line.startswith("Finished accumulating"):
            ms = float(line.split(" in ")[1].split(" ms")[0])
    return {"scene": scene, "W": W, "H": H, "spp": spp, "gpu_ms": ms, "wall_s": wall, "rc": p.returncode, "Msamples_s": (W * H * spp / ms / 1e3) if ms else None,
            "stderr": p.stderr[-300:]}


which = sys.argv[1:] or ["parity", "perf", "ref"]
if "parity" in which:
    out["primary"] = [primary_3way("cornell_box", 256, 256), primary_3way("generated_scene", 1920, 1080)]
    print(json.dumps(out["primary"]), flush=True)
    out["render"] = [render_parity("cornell_box", 64, 64, 64), render_parity("generated_scene", 96, 54, 64)]
    print(json.dumps(out["render"]), flush=True)
if "perf" in which:
    out["perf"] = []
    for kw in [dict(variant=0), dict(variant=0, smem_scene=0), dict(variant=0, count_work=1)]:
        r = perf("generated_scene", 1920, 1080, 256, **kw)
        out["perf"].append(r)
        print(json.dumps(r), flush=True)
    r = perf("cornell_box", 1920, 1080, 256, variant=0)
    out["perf"].append(r)
    print(json.dumps(r), flush=True)
if "ref" in which:
    out["ref"] = [ref_pt("generated_scene", 1920, 1080, 512), ref_pt("cornell_box", 1920, 1080, 512)]
    print(json.dumps(out["ref"]), flush=True)
os.makedirs("gpurun_out", exist_ok=True)
with open("gpurun_out/gpu_check.json", "w") as f:
    json.dump(out, f, indent=1)
