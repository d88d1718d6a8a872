#!/usr/bin/env python3
"""first-hit debugging on a large synthetic scene: consistency of (index, t) and the options that matter"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import pathtracercuda_b200 as pt
from pathtracercuda_b200 import scenegen
n = int(sys.argv[1]); W, H = 1920, 1080
objs, cam = scenegen.synthetic_scene(n, W, H)
with pt.Pathtracer(W, H) as P:
    P.setScene(objs)
    ei, et = P.primaryPass(cam)
    P.setOption("jitter", 0); P.setOption("first_hit", 1)
    for variant, beam, sstack in [(0, 1, 1), (0, 0, 1), (0, 1, 0), (4, 0, 0)]:
        P.setOption("variant", variant); P.setOption("beam", beam); P.setOption("smem_stack", sstack)
        for spp in (128, 192):
            P.render(cam, spp, True)
            i1, t1 = P.firstHit()
            bad = np.nonzero((i1 >= 0) & (t1 == 0))[0]
            mm = np.nonzero(i1 != ei)[0]
            print(f"n={n} variant={variant} beam={beam} sstack={sstack} spp={spp}: mismatches {len(mm)} {[(int(p), int(i1[p]), float(t1[p]), int(ei[p]), float(et[p])) for p in mm[:6]]}; idx>=0 with t==0: {len(bad)}", flush=True)
