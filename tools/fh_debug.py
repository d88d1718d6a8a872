#!/usr/bin/env python3
"""first-hit debugging: the render kernel's own first hits (options jitter=0, first_hit=1) against the IEEE primary pass, for
combinations of the kernel options.  usage: tools/fh_debug.py scene [spp]"""
import itertools, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import pathtracercuda_b200 as pt
from pathtracercuda_b200 import scenegen
name = sys.argv[1]
spp = int(sys.argv[2]) if len(sys.argv) > 2 else 128
W, H = 1920, 1080
if name.startswith("synthetic_"):
    objs, cam = scenegen.synthetic_scene(int(name.split("_")[1]), W, H)
else:
    objs, tex, sky, cam = pt.parse_scene_py(f"{pt.ASSETS}/scenes/{name}.json", W, H)
with pt.Pathtracer(W, H) as P:
    P.setScene(objs)
    ei, et = P.primaryPass(cam)
    P.setOption("jitter", 0)
    P.setOption("first_hit", 1)
    for variant, beam, sstack, strat, smem in [(0, 1, 1, 1, 1), (0, 0, 1, 1, 1), (0, 1, 0, 1, 1), (0, 1, 1, 0, 1), (0, 1, 1, 1, 0), (0, 0, 0, 0, 0), (4, 0, 0, 0, 1), (4, 0, 1, 0, 1)]:
        for k, v in (("variant", variant), ("beam", beam), ("smem_stack", sstack), ("stratify", strat), ("smem_scene", smem)):
            P.setOption(k, v)
        P.render(cam, spp, True)
        i1, t1 = P.firstHit()
        P.render(cam, spp, True)
        i2, t2 = P.firstHit()
        mm = np.nonzero(i1 != ei)[0]
        same = (i1 == ei) & (ei >= 0)
        rel = (np.abs(t1 - et)[same] / et[same]).max() if same.any() else 0
        print(f"{name} spp={spp} variant={variant} beam={beam} smem_stack={sstack} stratify={strat} smem_scene={smem}: {len(mm)} mismatches vs primary pass, "
              f"run-to-run differing {int((i1 != i2).sum())}, max rel t {rel:.2e}, first {[(int(p), int(i1[p]), int(ei[p])) for p in mm[:4]]}", flush=True)
