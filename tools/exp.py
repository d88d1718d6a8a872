#!/usr/bin/env python3
"""Timing experiments: tools/exp.py scene variant spp [key=value ...]  (keys: any pt_set_option key, plus nosky=1, w=, h=)"""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pathtracercuda_b200 as pt
scene, variant, spp = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
kv = dict(a.split("=") for a in sys.argv[4:])
W, H = int(kv.pop("w", 1920)), int(kv.pop("h", 1080))
nosky = int(kv.pop("nosky", 0))
with pt.Pathtracer(W, H) as P:
    for k in ("max_global", "max_leaf"):
        if k in kv:
            P.setOption(k, float(kv.pop(k)))
    cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/{scene}.json", cwd=pt.ASSETS)
    P.setOption("variant", variant)
    for k, v in kv.items():
        P.setOption(k, float(v))
    if nosky:
        P.setSkyboxTextureHandle(0)
    P.render(cam, 8, True)
    best = min((P.render(cam, spp, True), P.getTiming())[1] for _ in range(3))
    st = P.stats()
    import zlib
    crc = zlib.crc32(P.getHDRMean().tobytes())
    print(json.dumps({"crc": crc, "scene": scene, "variant": variant, "spp": spp, "opts": sys.argv[4:], "ms": round(best, 3), "Mrays_s": round(st.rays / best / 1e3, 1),
                      "rays_per_sample": round(st.rays / st.samples, 3), "nodes_per_ray": round(st.node_visits / st.rays, 2), "prims_per_ray": round(st.prim_tests / st.rays, 2),
                      "bvh_nodes": st.bvh_nodes, "smem": st.scene_in_smem}), flush=True)
    import ctypes as C
    raw = (C.c_ulonglong * 24)()
    if variant in (0, 12) and hasattr(P.L, "pt_debug_counters") and P.L.pt_debug_counters(P.h, raw, 24) == 24 and raw[8]:
        cp, cl, cc, sp_, sl, sc, tot = [raw[8 + k] for k in range(7)]
        print(json.dumps({"camera_passes_per_ksample": round(1e3 * cp / st.samples, 2), "lanes_per_camera_pass": round(cl / max(cp, 1), 2), "clocks_per_camera_pass": round(cc / max(cp, 1), 1),
                          "scattered_passes_per_ksample": round(1e3 * sp_ / st.samples, 2), "lanes_per_scattered_pass": round(sl / max(sp_, 1), 2), "clocks_per_scattered_pass": round(sc / max(sp_, 1), 1),
                          "share_camera": round(cc / tot, 3), "share_scattered": round(sc / tot, 3), "share_other": round(1 - (cc + sc) / tot, 3),
                          "traversal_share_of_camera_pass": round(raw[15] / max(cc, 1), 3), "traversal_share_of_scattered_pass": round(raw[16] / max(sc, 1), 3)}))
