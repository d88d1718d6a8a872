"""Times the denoiser's two passes and runs the sweep that chose its defaults (DESIGN.md, "Denoiser").

On generated_scene at 1920x1080: the guide pass (pt_render_aov) at 16 rays per pixel and pt_denoise at the default parameters, each call
timed with a host clock (both calls end in a device synchronise), after warm-up calls.  Then the sweep: every (K, sigma_color,
sigma_normal, sigma_position) of the grid below denoises the same 16-spp renders of generated_scene 1920x1080 and cornell_box 480x270,
scored by RMSE of the per-sample mean (linear RGB) against a 4096-spp render with another seed; the score of a setting is the mean of
its two ratios denoised / raw.  Prints the card and its power limit first: the times are worth nothing without them.

    python tools/denoise_measure.py [--out result.json] [--quick]
"""
import argparse
import itertools
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pathtracercuda_b200 as pt  # noqa: E402
from pathtracercuda_b200 import api  # noqa: E402

GRID = dict(iterations=[3, 4, 5, 6], sigma_color=[1.0, 2.0, 4.0, 8.0, 16.0, 32.0, 64.0], sigma_normal=[0.25, 0.5, 1.0],
            sigma_position=[0.01, 0.02, 0.05])


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def rmse(a, b):
    return float(np.sqrt(np.mean((a[..., :3].astype(np.float64) - b[..., :3]) ** 2)))


class Case:
    """one scene at one size: a 16-spp context with its guide buffers, and the 4096-spp reference of another seed"""

    def __init__(self, scene, W, H, spp=16, ref_spp=4096):
        path = f"{pt.ASSETS}/scenes/{scene}.json"
        with pt.Pathtracer(W, H) as R:
            cam = R.loadSceneFile(path, cwd=pt.ASSETS)
            R.setOption("seed", 7)
            R.render(cam, ref_spp, True)
            self.ref = R.getHDRMean()
        self.P = pt.Pathtracer(W, H)
        self.cam = self.P.loadSceneFile(path, cwd=pt.ASSETS)
        self.P.render(self.cam, spp, True)
        self.frame_ms = self.P.getTiming()
        self.P.renderAOV(self.cam, 16)
        self.raw = rmse(self.P.getHDRMean(), self.ref)
        self.name = f"{scene} {W}x{H}"

    def ratio(self, **q):
        self.P.denoise(**q)
        return rmse(self.P.getDenoisedHDRMean(copy=False), self.ref) / self.raw


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    ap.add_argument("--quick", action="store_true", help="a small grid (rehearsal)")
    a = ap.parse_args()
    res = {"card": card()}
    print("card, power limit:", res["card"], flush=True)
    big = Case("generated_scene", 1920, 1080)
    small = Case("cornell_box", 480, 270)
    P, cam = big.P, big.cam
    for _ in range(3):
        P.renderAOV(cam, 16)
        P.denoise()
    aov_ms = timed(lambda: P.renderAOV(cam, 16), 20)
    den_ms = timed(lambda: P.denoise(), 20)
    res["generated_scene_1080p"] = {"render_16spp_ms": big.frame_ms, "aov_16spp_ms": aov_ms, "denoise_default_ms": den_ms,
                                    "defaults": api.DENOISE_DEFAULTS}
    print(f"generated_scene 1920x1080: pt_render_aov 16 spp median {np.median(aov_ms):.3f} ms (min {min(aov_ms):.3f}), "
          f"pt_denoise {api.DENOISE_DEFAULTS} median {np.median(den_ms):.3f} ms (min {min(den_ms):.3f}); 16-spp render {big.frame_ms:.3f} ms", flush=True)
    for k in (1, 3, 5, 8, 12):
        ms = timed(lambda: P.denoise(iterations=k), 10)
        res["generated_scene_1080p"][f"denoise_K{k}_ms"] = ms
        print(f"  K = {k}: median {np.median(ms):.3f} ms", flush=True)
    grid = {k: v[:2] for k, v in GRID.items()} if a.quick else GRID
    rows = []
    for vals in itertools.product(*grid.values()):
        q = dict(zip(grid.keys(), vals))
        rb, rs = big.ratio(**q), small.ratio(**q)
        rows.append({**q, "ratio_generated_scene": rb, "ratio_cornell_box": rs, "score": 0.5 * (rb + rs)})
    rows.sort(key=lambda r: r["score"])
    res["raw_rmse"] = {big.name: big.raw, small.name: small.raw}
    res["sweep"] = rows
    print(f"raw RMSE: {big.name} {big.raw:.5f}, {small.name} {small.raw:.5f}; best 15 of {len(rows)} settings (RMSE denoised / raw):")
    for r in rows[:15]:
        print("  " + json.dumps(r))
    print("  defaults:", [r for r in rows if all(r[k] == v for k, v in api.DENOISE_DEFAULTS.items())])
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    big.P.close()
    small.P.close()


if __name__ == "__main__":
    main()
