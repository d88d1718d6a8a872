"""Option "light_is" on one GPU: time per frame of cornell_box at 1920x1080 / 1024 spp (BASELINE.json config 2) with and without the
option, alternated, and the error against the reference program's stored 4096-spp renders (tests/golden/refpt_cornell_box.npz,
256x256) for a ladder of sample counts, both estimators - the error at equal time can be read off.  Prints one JSON object with the
card's name and power limit; also writes it to the file named by the first argument, if any."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pathtracercuda_b200 as pt  # noqa: E402
from oracle import imgio  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q.splitlines()[0] if q else "unknown"


def main(out):
    res = {"card": card(), "timing": [], "ladder": []}
    scene = f"{pt.ASSETS}/scenes/cornell_box.json"
    W, H, spp = 1920, 1080, 1024
    with pt.Pathtracer(W, H) as P:
        cam = P.loadSceneFile(scene, cwd=pt.ASSETS)
        for on in (0, 1):  # warm-up
            P.setOption("light_is", on)
            P.render(cam, 64, True)
        for rep in range(3):
            for on in (0, 1):
                P.setOption("light_is", on)
                P.render(cam, spp, True)
                ms, rays = P.getTiming(), P.stats().rays
                res["timing"].append({"light_is": on, "ms": ms, "grays_per_s": rays / ms / 1e6, "rays": int(rays)})
    g = np.load(os.path.join(ROOT, "tests", "golden", "refpt_cornell_box.npz"))
    Wr, Hr = int(g["W"]), int(g["H"])
    ref = 0.5 * (g["A"].astype(np.float32) + g["B"].astype(np.float32))
    with pt.Pathtracer(Wr, Hr) as P:
        cam = P.loadSceneFile(scene, cwd=pt.ASSETS)
        for n in (16, 64, 256, 1024):
            for on in (0, 1):
                P.setOption("light_is", on)
                P.render(cam, n, True)
                img = P.getHDRMean()[:, :, :3]
                e, _ = imgio.rmse(img.astype(np.float32), ref)
                res["ladder"].append({"spp": n, "light_is": on, "rmse": float(e), "ms": P.getTiming()})
    print(json.dumps(res))
    if out:
        with open(out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
