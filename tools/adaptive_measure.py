"""Measures option "adaptive" on the GPU (DESIGN.md "Adaptive sampling"): the cost of the checkpoints, and error against time.

    python tools/adaptive_measure.py [--out adaptive.jsonl] [--quick]

1. Checkpoint overhead: generated_scene 1920x1080, 4096 spp, uniform against adaptive with a tau so small that no lit pixel stops (only
   the drains at m, 2m, ... are added).
2. Error against time: cornell_box (plain and light_is) and generated_scene at 480x270, against a 16384-spp reference of another seed:
   uniform spp 64 ... 4096 and adaptive over a ladder of tau at spp_max 4096 and m in {64, 128, 256}.  Per run: ms, total samples, RMSE of
   the linear mean and of the tone-mapped image (Reinhard, gamma 1/2.2).
Prints the card's name and power limit first; one JSON line per run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pathtracercuda_b200 as pt  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def tonemap(x):
    x = np.maximum(x[..., :3], 0.0)
    return (x / (x + 1.0)) ** (1.0 / 2.2)


def render(scene, W, H, spp, seed, reps=1, **opts):
    with pt.Pathtracer(W, H) as P:
        cam = P.loadSceneFile(f"{pt.ASSETS}/scenes/{scene}.json", cwd=pt.ASSETS)
        P.setOption("seed", seed)
        for k, v in opts.items():
            P.setOption(k, v)
        P.render(cam, min(spp, 64), True)  # warm-up: module load, scene staging
        ms = []
        for _ in range(reps):
            P.render(cam, spp, True)
            ms.append(P.getTiming())
        return P.getHDRMean().astype(np.float64), float(np.median(ms)), int(P.stats().samples)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="fewer points (one m, a shorter ladder)")
    a = ap.parse_args()
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    emit({"card": card()})
    # 1. checkpoint overhead
    W, H = 1920, 1080
    _, t_uni, n_uni = render("generated_scene", W, H, 4096, 1984, reps=3)
    _, t_ad, n_ad = render("generated_scene", W, H, 4096, 1984, reps=3, adaptive=1e-7)
    emit({"what": "overhead", "scene": "generated_scene", "size": [W, H], "spp": 4096, "uniform_ms": t_uni, "adaptive_ms": t_ad,
          "uniform_samples": n_uni, "adaptive_samples": n_ad})
    # 2. error against time
    W, H = 480, 270
    taus = [0.005, 0.01, 0.02, 0.05, 0.1] if not a.quick else [0.01, 0.02, 0.05]
    mins = [64, 128, 256] if not a.quick else [128]
    for scene, opts in [("cornell_box", {}), ("cornell_box", {"light_is": 1}), ("generated_scene", {})]:
        ref, _, _ = render(scene, W, H, 16384, 7, **opts)
        tref = tonemap(ref)

        def err(img):
            return float(np.sqrt(np.mean((img[..., :3] - ref[..., :3]) ** 2))), float(np.sqrt(np.mean((tonemap(img) - tref) ** 2)))

        for spp in [64, 128, 256, 512, 1024, 2048, 4096]:
            img, ms, n = render(scene, W, H, spp, 1984, **opts)
            emit({"what": "uniform", "scene": scene, **opts, "spp": spp, "ms": ms, "samples": n, "rmse": err(img)[0], "rmse_tm": err(img)[1]})
        for m in mins:
            for tau in taus:
                img, ms, n = render(scene, W, H, 4096, 1984, adaptive=tau, adaptive_min_spp=m, **opts)
                emit({"what": "adaptive", "scene": scene, **opts, "tau": tau, "m": m, "spp_max": 4096, "ms": ms, "samples": n,
                      "rmse": err(img)[0], "rmse_tm": err(img)[1]})


if __name__ == "__main__":
    main()
