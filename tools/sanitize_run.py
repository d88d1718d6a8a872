#!/usr/bin/env python3
"""Small renders of every default code path for compute-sanitizer (memcheck / racecheck / synccheck / initcheck):
  compute-sanitizer --tool racecheck python tools/sanitize_run.py"""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import pathtracercuda_b200 as pt
for scene, W, H in (("generated_scene", 96, 54), ("cornell_box", 48, 48)):
    with pt.Pathtracer(W, H) as P:
        cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/{scene}.json", cwd=pt.ASSETS)
        for variant, spp, opts in ((4, 8, {}), (12, 160, {}), (12, 160, {"beam": 0}), (12, 160, {"smem_scene": 0}), (12, 40, {"tex_unit": 0})):
            P.setOption("variant", variant)
            for k, v in {"beam": -1, "smem_scene": 1, "tex_unit": 1, **opts}.items():
                P.setOption(k, v)
            P.render(cam, spp, True)
            img = P.getHDRMean()
            print(scene, variant, spp, opts, float(img[..., :3].mean()), bool(np.isfinite(img).all()), flush=True)
        # the twin instantiations: sky importance sampling, parity aids
        P.setOption("variant", 0)
        for k, v in {"beam": -1, "smem_scene": 1, "tex_unit": 1}.items():
            P.setOption(k, v)
        for spp in (8, 160):
            P.setOption("env_is", 1)
            P.render(cam, spp, True)
            print(scene, "env_is", spp, float(P.getHDRMean()[..., :3].mean()), flush=True)
            P.setOption("env_is", 0)
            P.setOption("jitter", 0)
            P.setOption("first_hit", 1)
            P.render(cam, spp, True)
            idx, t = P.firstHit()
            print(scene, "aids", spp, int((idx >= 0).sum()), flush=True)
            P.setOption("jitter", 1)
            P.setOption("first_hit", 0)
        P.primaryPass(cam)
        P.getImageData()
