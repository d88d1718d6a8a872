#!/usr/bin/env python3
"""bench.py — the headline measurement: path tracing throughput on generated_scene.json at 1920x1080, 4096 spp
(BASELINE.json config 3) in Mrays/s, on N B200s of one node.  --scene / --spp / --width / --height select the other configs
(cornell_box: config 2; synthetic_<N> at 256 spp: config 4; 3840x2160 at 16384 spp: config 5).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--spp S] [--impl ours|reference] [--dump-outputs DIR]
  (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

A "step" = one complete render of the configuration: every pixel, `spp` samples, up to 5 path segments per sample
(ray = one closest-hit query, sample = one path; SURVEY.md §8d).  With N GPUs (one process per GPU) the PIXELS are split
(rank r: pixels r, r+N, ... with all their samples - this replaces north_star's sample split, DESIGN.md §6; --partition samples
selects that one) and the float4 accumulation buffers are summed with ONE NCCL reduce inside the timed region: strong scaling.

  value     rays of the whole job / device time of the step (CUDA events on the library's stream around the trace kernel + CUDA
            events around the reduce), max over ranks; scene and accumulation buffer resident in HBM
  e2e       the same metric through the drop-in surface a user of the reference touches - the command line: a FRESH
            `pathtracer_b200 -w W -h H -spp S -ohdr -o out.hdr scene.json` process per step (with --gpus N on N GPUs: the C ABI's
            pt_create_multi), wall clock of the whole process: CUDA context, scene file parse, BVH build, texture decode and
            upload, render, device->host read-back, Radiance file written.  The reference arm times `ref_pt` with the same
            arguments the same way, so the two e2e figures are like for like.  (`e2e.in_process`: pt_set_scene + pt_render +
            pt_get_hdr in the warm process, the round-1 figure.)
  --impl reference   the reference's OWN trace.cu / Pathtracer.cpp / main.cpp rebuilt unmodified for sm_100 (oracle/_ref/ref_pt)
            on the same GPU, same scene / resolution / spp; time = its own "ms GPU time"; rays = its own count
            (oracle/_ref/ref_gpu).  The reference has no CPU renderer; its __host__ __device__ math built with g++
            (oracle/_ref/libref_host.so) is timed on the box's cores as `cpu_baseline` in both arms.
  --dump-outputs DIR   after the timed steps, write what the last one computed as DIR/*.npy (see dump_outputs): the same
            arguments give the same inputs, so two builds can be compared output for output.
"""
import os

# torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU baseline below is an OpenMP program and has to see the box's cores
# (it sets its thread count explicitly as well - this only keeps libgomp from capping it at 1 when it initialises)
if os.environ.get("OMP_NUM_THREADS") == "1":
    os.environ.pop("OMP_NUM_THREADS")

import argparse  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import tempfile  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCENE = "generated_scene"   # --scene: cornell_box | generated_scene | synthetic_<N> (BASELINE.json configs 2-4)
W, H = 1920, 1080
SCENE_DIR = None            # directory holding <SCENE>.json and the assets it names (set by resolve_scene)
CLI = os.path.join(ROOT, "pathtracercuda_b200", "bin", "pathtracer_b200")


def resolve_scene(args):
    """bundled scenes live under assets/scenes; synthetic_<N> is generated into a temporary directory (seed 1984)"""
    global SCENE, W, H, SCENE_DIR
    import pathtracercuda_b200 as pt
    SCENE, W, H = args.scene, args.width, args.height
    if SCENE.startswith("synthetic_"):
        from pathtracercuda_b200 import scenegen
        SCENE_DIR = tempfile.mkdtemp(prefix="ptb_scene_")
        os.symlink(pt.ASSETS + "/skybox.hdr", SCENE_DIR + "/skybox.hdr")
        scenegen.write_synthetic_scene(f"{SCENE_DIR}/{SCENE}.json", int(SCENE.split("_")[1]))
        return f"{SCENE_DIR}/{SCENE}.json", SCENE_DIR
    SCENE_DIR = pt.ASSETS + "/scenes"
    return f"{SCENE_DIR}/{SCENE}.json", pt.ASSETS


def workload_label(spp):
    cfg = {"generated_scene": "BASELINE.json config 3", "cornell_box": "BASELINE.json config 2"}.get(SCENE, "BASELINE.json config 4")
    if SCENE == "generated_scene" and (W, H) == (3840, 2160):
        cfg = "BASELINE.json config 5"
    return f"{SCENE}.json {W}x{H} {spp} spp ({cfg}), stand-in earth.png/skybox.hdr (reference assets not in its checkout)"


def config_dict(args):
    """the SAME dictionary in both arms (the driver compares them): what is rendered, not how"""
    return {"workload": workload_label(args.spp), "scene": SCENE, "width": W, "height": H, "spp": args.spp, "max_path_segments": 5, "gpus": args.gpus}


# algorithmic FP32 operations / bytes per unit of work, counted from the reference source (SURVEY.md §8d table)
OPS_NODE_BOX = 24.0          # one ray/box slab test (AABB.inl:22-44); a two-box node visit = 2 of these
OPS_PRIM_COMMON = 33.0       # world->local ray (Hittable.inl:92-98)
OPS_PRIM_SHAPE_AVG = 33.0    # mean of the per-shape parts over generated_scene's shape mix
OPS_HIT = 40.0               # accepted hit: normal -> world, normalize, point, face-forward
OPS_SHADE = 300.0            # GGX / LAMBERT_GGX sample (483 of 484 materials); Lambert is 140
OPS_MISS = 10.0
OPS_CAMERA = 25.0
BYTES_NODE = 64.0            # our two-box node record (the reference: 2 x 32 B single-box nodes)
BYTES_PRIM = 64.0            # our primitive record (the reference: 96 B Hittable)
BYTES_MAT = 48.0             # material record, once per shade
BYTES_PIXEL = 16.0           # float4 accumulate, once per pixel per render

DUMP_BYTES = 64 << 20        # --dump-outputs budget
DUMP_SAMPLE = 1 << 21        # pixels kept of an image over that budget


def dump_outputs(out_dir, hdr_mean, rays):
    """--dump-outputs: the last timed render as its caller receives it - the per-sample mean radiance, float32 (H, W, 3), as
    hdr_mean.npy - and the rays it traced (whole job) as rays.npy, float64.  An image over DUMP_BYTES is written as a fixed sample
    of DUMP_SAMPLE pixels (seed 0, the same from run to run): hdr_mean.npy (N, 3) with their row-major indices in
    pixel_index.npy (float64 holding exact integers)."""
    os.makedirs(out_dir, exist_ok=True)
    if hdr_mean.nbytes > DUMP_BYTES:
        h, w, c = hdr_mean.shape
        pix = np.sort(np.random.default_rng(0).choice(h * w, DUMP_SAMPLE, replace=False))
        hdr_mean = hdr_mean.reshape(h * w, c)[pix]
        np.save(os.path.join(out_dir, "pixel_index.npy"), pix.astype(np.float64))
    np.save(os.path.join(out_dir, "hdr_mean.npy"), np.ascontiguousarray(hdr_mean, np.float32))
    np.save(os.path.join(out_dir, "rays.npy"), np.array([rays], np.float64))


def clock_sampler(stop, out, index):
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}
        out["sm_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        while not stop.is_set():
            out["samples"].append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
            r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for bit, n in names.items():
                if r & bit:
                    out["reasons"].add(n)
            time.sleep(0.1)
    except Exception as e:  # noqa
        out["error"] = repr(e)


def cpu_baseline(seconds=12.0):
    """the reference's host math (libref_host.so: its own Hittable::hit / AABB::hit / Material::sample with XORWOW, full
    5-segment paths) on this box's cores; falls back to our oracle port when the reference build is absent.  `cores` is
    the number of OpenMP threads the run actually used."""
    import pathtracercuda_b200 as pt
    from oracle import imgio, orc
    want = os.cpu_count() or 1
    w, h = 480, 270
    objs, tex, sky, cam = pt.parse_scene_py(f"{SCENE_DIR}/{SCENE}.json", w, h)
    skyimg = imgio.read_hdr(pt.ASSETS + "/skybox.hdr")
    has_sky = bool(sky) and tex[sky - 1] == "skybox.hdr"  # cornell_box names a file that does not exist: black environment
    if orc.have_ref_host():
        R = orc.RefHost()
        cores = R.threads(want)
        for o in objs:
            o.material.texture = 0
        R.set_scene(objs)
        R.set_camera(cam)
        if has_sky:
            R.set_sky(skyimg)
        run = lambda spp: R.render(w, h, spp)[1]
        kind = "reference"
    else:
        O = orc.Oracle(objs)
        cores = O.threads(want)
        O.add_texture(imgio.read_png(pt.ASSETS + "/earth.png"))
        if has_sky:
            O.set_skybox(O.add_texture(skyimg))
        run = lambda spp: O.render(cam, w, h, spp, stratify=0)[1]
        kind = "port"
    t0 = time.perf_counter()
    rays = run(2)
    rate = rays / (time.perf_counter() - t0)
    spp = int(max(2, min(4096, seconds * rate / (rays / 2))))
    t0 = time.perf_counter()
    rays = run(spp)
    dt = time.perf_counter() - t0
    return {"value": rays / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": kind,
            "sample": f"{SCENE} {w}x{h}, {spp} spp, full 5-segment paths ({rays} rays in {dt:.1f} s), OpenMP over scanlines, {cores} threads"
                      + (", reference host build (base-colour texture taps compiled out by the reference itself)" if kind == "reference" else "")}


def time_cli(exe, scene_path, scene_cwd, spp, steps, extra=()):
    """fresh process per step, same arguments for both arms: -w -h -spp -ohdr -o <file> <scene>.  Returns (mean wall s, mean of
    the program's own 'ms GPU time', last stdout) or raises."""
    walls, gpu_ms, out = [], [], ""
    with tempfile.TemporaryDirectory() as td:
        for _ in range(steps):
            t0 = time.perf_counter()
            p = subprocess.run([exe, "-w", str(W), "-h", str(H), "-spp", str(spp), "-ohdr", "-o", os.path.join(td, "out.hdr"), *extra, os.path.relpath(scene_path, scene_cwd)],
                               cwd=scene_cwd, capture_output=True, text=True)
            walls.append(time.perf_counter() - t0)
            ms = [float(l.split(" in ")[1].split(" ms")[0]) for l in p.stdout.splitlines() if l.startswith("Finished accumulating")]
            if p.returncode != 0 or not ms or not os.path.exists(os.path.join(td, "out.hdr")):
                raise RuntimeError(f"{os.path.basename(exe)} failed: " + (p.stderr or p.stdout)[-300:].replace("\n", " "))
            gpu_ms.append(ms[0])
            out = p.stdout
            os.remove(os.path.join(td, "out.hdr"))
    return float(np.mean(walls)), float(np.mean(gpu_ms)), out


def run_reference(args):
    """--impl reference: the unmodified reference program on this box's GPU 0"""
    import pathtracercuda_b200 as pt
    from oracle import orc
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    scene_path, scene_cwd = resolve_scene(args)
    line = {"impl": "reference", "metric": "Mrays/s", "unit": "Mrays/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args),
            "notes": {"l2": "not flushed: the reference re-launches its kernel every 8 spp, working set 56 KB scene + 133 MB state",
                      "gpus": "the reference is fixed to device 0 (Pathtracer.cpp:40): one GPU whatever --gpus says"}}
    cb = cpu_baseline()
    if not os.path.exists(orc.REF_PT):
        # no GPU build of the reference available: the CPU host build is the reference arm
        line.update({"value": cb["value"], "ms_per_step": None, "cpu_baseline": cb, "reference_device": f"host CPU x{cb['cores']}",
                     "e2e": {"value": cb["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(line))
        return 0
    objs, tex, sky, cam = pt.parse_scene_py(scene_path, W, H)
    with tempfile.TemporaryDirectory() as td:
        cnt = orc.ref_gpu_count(objs, cam, W, H, 32, td)  # the reference's own rays per sample (its seeds, its slicing)
    rps = cnt["rays_per_sample"]
    try:
        if args.warmup:
            time_cli(orc.REF_PT, scene_path, scene_cwd, args.spp, args.warmup)
        wall, ms, _ = time_cli(orc.REF_PT, scene_path, scene_cwd, args.spp, args.steps)
    except RuntimeError as e:
        print(json.dumps({"impl": "reference", "unavailable": str(e)}))
        return 0
    rays = W * H * args.spp * rps
    line.update({"value": rays / ms / 1e3, "ms_per_step": ms, "samples_per_s": W * H * args.spp / ms * 1e3, "rays_per_sample": rps,
                 "reference_device": "B200: the reference's trace.cu / Pathtracer.cpp / main.cpp rebuilt unmodified for sm_100 (oracle/_ref/ref_pt); "
                                     "time = its own 'ms GPU time', rays from oracle/_ref/ref_gpu count",
                 "gpu_launches": (args.spp + 7) // 8 * args.steps, "cpu_baseline": cb,
                 "e2e": {"value": rays / wall / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "wall_s_per_step": wall,
                         "note": "fresh ref_pt process per step, -ohdr -o out.hdr: CUDA init, scene load, BVH build, (spp + 7) / 8 launches, read-back, Radiance file written; "
                                 "wall clock of the whole process (the copies are the program's own, not counted here)"}})
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--spp", type=int, default=4096)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--scene", default="generated_scene")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-cli", action="store_true", help="skip the fresh-process e2e (in-process figure only)")
    ap.add_argument("--partition", default="pixels", choices=["pixels", "samples"],
                    help="N > 1: what is split over the GPUs (pathtracercuda_b200/distributed.py); the single reduce is the same")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's image and ray count to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.spp < 1:
        ap.error("--steps and --spp must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the timed path of --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import pathtracercuda_b200 as pt
    from pathtracercuda_b200.distributed import attach_torch_accumulator, configure_partition, reduce_accumulation

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the trace path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE {world}"

    path, scene_cwd = resolve_scene(args)
    P = pt.Pathtracer(W, H, device=local)
    cam = P.loadSceneFile(path, cwd=scene_cwd)
    P.setOption("variant", args.variant)
    accum = attach_torch_accumulator(P, torch.device("cuda", local))
    count = configure_partition(P, args.spp, rank, world, args.partition)  # spp argument of pt_render on this rank
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def host_wait(tag):
        """ranks > 0 wait on the HOST (no NCCL kernel spinning on their GPUs) until rank 0 has passed this point"""
        flag = os.path.join(tempfile.gettempdir(), f"ptb_bench_{os.environ.get('MASTER_PORT', '0')}_{os.environ.get('TORCHELASTIC_RUN_ID', 'x')}_{tag}")
        if rank == 0:
            open(flag, "w").close()
        else:
            while not os.path.exists(flag):
                time.sleep(0.05)

    def step():
        """one render of the whole configuration: this rank's share + the reduce.  returns (device ms, rays, reduce ms)"""
        flush.zero_()  # evict L2 between steps (outside the timed events)
        torch.cuda.synchronize()
        P.render(cam, count, True)  # blocking; timed by CUDA events on the library's own stream
        ms = P.getTiming()
        rays = P.stats().rays
        red = 0.0
        if dist:
            ev0.record()
            reduce_accumulation(accum, dst=0)
            ev1.record()
            torch.cuda.synchronize()
            red = ev0.elapsed_time(ev1)
        return ms + red, rays, red

    for _ in range(args.warmup):
        step()
    clk = {"samples": [], "reasons": set()}
    stop = threading.Event()
    th = threading.Thread(target=clock_sampler, args=(stop, clk, local), daemon=True)
    th.start()
    barrier()
    t0 = time.perf_counter()
    ms_steps, rays_steps, red_steps = [], [], []
    for _ in range(args.steps):
        ms, rays, red = step()
        ms_steps.append(ms)
        rays_steps.append(rays)
        red_steps.append(red)
    barrier()
    wall = time.perf_counter() - t0
    stop.set()
    th.join(timeout=2)
    # the last timed step's image (rank 0 holds the whole job's sum after the reduce), before the e2e runs below render into the
    # same buffer; pixels outside a rank's share are zero on the other ranks, so only rank 0's copy is the caller's image
    last_hdr = (accum[..., :3].cpu().numpy() / np.float32(args.spp)) if args.dump_outputs and rank == 0 else None

    ms_t = torch.tensor(ms_steps, dtype=torch.float64, device=f"cuda:{local}")
    rays_t = torch.tensor(rays_steps, dtype=torch.float64, device=f"cuda:{local}")
    if dist:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(rays_t, op=dist.ReduceOp.SUM)
    ms_step = float(ms_t.mean())
    rays_step = float(rays_t.mean())
    value = rays_step / ms_step / 1e3  # Mrays/s, whole job

    # ---- e2e, in process: host object array in, host image out, through the C ABI, wall clock (the round-1 figure) ----
    objs, tex, sky, cam_py = pt.parse_scene_py(path, W, H)
    st0 = P.stats()
    h2d_scene = int(st0.scene_bytes)
    barrier()
    t0 = time.perf_counter()
    e2e_rays = 0
    checksum = None
    for _ in range(args.steps):
        P.setScene(objs)              # host object array -> BVH build -> H2D of nodes/primitives/materials
        P.render(cam, count, True)
        e2e_rays += P.stats().rays
        if dist:
            reduce_accumulation(accum, dst=0)
            torch.cuda.synchronize()
        if rank == 0:
            img = P.getHDRImageData(copy=False)  # normalise on device + D2H of W*H*16 bytes into pinned host memory
            checksum = float(img[::97, ::89, :3].sum())
    barrier()
    e2e_wall = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_rays], dtype=torch.float64, device=f"cuda:{local}")
    if dist:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.SUM)
    e2e_in_process = float(e2e_t[0]) / e2e_wall / 1e6

    # ---- e2e, like for like with the reference arm: a fresh process of the drop-in command line per step ----
    cli = None
    if rank == 0 and not args.no_e2e_cli and os.path.exists(CLI):
        try:
            extra = ["--gpus", str(world)] if world > 1 else []
            if world > 1 and args.partition == "samples":
                extra += ["--partition", "samples"]
            time_cli(CLI, path, scene_cwd, args.spp, 1, extra)  # warm the file cache like the reference arm's warm-up does
            cwall, cms, cout = time_cli(CLI, path, scene_cwd, args.spp, args.steps, extra + ["--stats"])
            cli = {"wall_s": cwall, "gpu_ms": cms, "stats": json.loads([l for l in cout.splitlines() if l.startswith("{")][-1])}
        except Exception as e:  # noqa
            cli = {"error": str(e)[:300]}
    torch.cuda.synchronize()
    host_wait("cli_done")
    barrier()
    if rank == 0:
        for f in os.listdir(tempfile.gettempdir()):
            if f.startswith(f"ptb_bench_{os.environ.get('MASTER_PORT', '0')}_"):
                try:
                    os.remove(os.path.join(tempfile.gettempdir(), f))
                except OSError:
                    pass

    if rank == 0:
        # ---- roofline.  Unit counts from ONE untimed counting launch of the SAME configuration as the timed steps (same spp:
        # same kernel instantiation, pixel beams, stratification); a second one with the beams off gives the plain walk's count ----
        P.setOption("count_work", 1)
        P.render(cam, count, True)
        s = P.stats()
        P.setOption("beam", 0)
        P.render(cam, count, True)
        s_plain = P.stats()
        P.setOption("beam", -1)
        P.setOption("count_work", 0)

        def units(st):
            return {"node_visits": st.node_visits / st.rays, "prim_tests": st.prim_tests / st.rays, "shades": st.shades / st.rays, "misses": st.misses / st.rays,
                    "camera_rays": st.samples / st.rays}

        def ops(u):
            return (u["node_visits"] * 2 * OPS_NODE_BOX + u["prim_tests"] * (OPS_PRIM_COMMON + OPS_PRIM_SHAPE_AVG) + u["shades"] * (OPS_HIT + OPS_SHADE)
                    + u["misses"] * OPS_MISS + u["camera_rays"] * OPS_CAMERA)
        per_ray, per_ray_plain = units(s), units(s_plain)
        ops_per_ray, ops_per_ray_plain = ops(per_ray), ops(per_ray_plain)
        bytes_per_ray = per_ray["node_visits"] * BYTES_NODE + per_ray["prim_tests"] * BYTES_PRIM + per_ray["shades"] * BYTES_MAT + BYTES_PIXEL * W * H / max(s.rays, 1)
        sm_mhz = float(np.median(clk["samples"])) if clk["samples"] else None
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        f_mhz = sm_mhz or peaks.get("sm_max_mhz", 1965.0)
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        peak_tops = sms * 128 * f_mhz * 1e6 / 1e12          # FP32 lane-instruction slots per second (an FMA counts once)
        kernel_ms = float(np.mean(ms_steps)) - float(np.mean(red_steps))  # this rank's trace kernel per launch
        achieved = rays_steps[0] * ops_per_ray / (kernel_ms * 1e-3) / 1e12
        achieved_plain = rays_steps[0] * ops_per_ray_plain / (kernel_ms * 1e-3) / 1e12
        in_smem = bool(st0.scene_in_smem)
        hbm_peak = float(peaks.get("hbm_gbs", 6548.8))
        gbs = rays_steps[0] * bytes_per_ray / (kernel_ms * 1e-3) / 1e9
        if in_smem:
            roofline = {"bound": "fp32_issue", "achieved": achieved, "peak": peak_tops, "unit": "T FP32 lane-op/s", "frac": achieved / peak_tops, "traffic": None,
                        "note": "no dense contraction and a 64 KB scene staged in shared memory: neither tensor nor HBM bound. achieved = algorithmic FP32 ops "
                                "(SURVEY.md §8d per-unit counts x the unit counts the TIMED configuration executes, from a counting launch of the same spp with pixel beams "
                                f"and stratification on) / trace-kernel time; peak = {sms} SMs x 128 lanes x {f_mhz:.0f} MHz observed under load. `frac_plain_walk` counts the "
                                "node visits of a walk from the root for every ray instead (work the beams skip). `traffic` (DRAM bytes per launch) is only measured "
                                "under ncu: see profiles/r02_trace_kernel_summary.json"}
        else:
            roofline = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": None,
                        "note": "scene in global memory (L1 / L2 / HBM): achieved = algorithmic bytes (64 B per two-box node visit + 64 B per primitive test + 48 B material per "
                                "shade + 16 B per pixel; unit counts of the timed configuration from a counting launch) / trace-kernel time, against the measured HBM copy "
                                "bandwidth (MEASURED_PEAKS.json). Most of these bytes are served by L1 / L2 (126 MB L2; ncu: profiles/r02_*), so the fraction of the HBM peak "
                                "says how far the kernel is from being bandwidth bound; the instruction-issue figures are given as well"}
        roofline.update({"ops_per_ray": ops_per_ray, "units_per_ray": per_ray, "bytes_per_ray": bytes_per_ray, "algorithmic_gbs": gbs,
                         "fp32_issue_frac": achieved / peak_tops, "frac_plain_walk": achieved_plain / peak_tops, "ops_per_ray_plain_walk": ops_per_ray_plain,
                         "units_per_ray_plain_walk": per_ray_plain})
        e2e = {"unit": "Mrays/s", "d2h_bytes_per_step": W * H * 16, "in_process": e2e_in_process,
               "in_process_note": "per step: pt_set_scene (host BVH build + upload) + pt_render + pt_get_hdr (D2H to pinned memory) in the warm process, wall clock", "checksum": checksum}
        if cli and "wall_s" in cli:
            tex_bytes = 2 * (2048 * 1024 * 4) + 2 * (2048 * 1024 * 16) if SCENE != "cornell_box" else 2 * (2048 * 1024 * 4)
            e2e.update({"value": rays_step / cli["wall_s"] / 1e6, "wall_s_per_step": cli["wall_s"], "cli_gpu_ms": cli["gpu_ms"], "cli_stats": cli["stats"],
                        "h2d_bytes_per_step": h2d_scene * world + tex_bytes * world,
                        "note": "fresh pathtracer_b200 process per step (-w -h -spp -ohdr -o out.hdr" + (f" --gpus {world}" if world > 1 else "") + "): CUDA context, scene file parse, BVH build, "
                                "texture decode + upload (linear copy + CUDA array each), render, D2H, Radiance file written; wall clock of the whole process - the same "
                                "scope as the reference arm's e2e"})
        else:
            e2e.update({"value": e2e_in_process, "h2d_bytes_per_step": h2d_scene, "note": "in-process figure (the command-line e2e was skipped or failed)", "cli": cli})
        line = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args),
            "notes": {"spp_per_gpu": count, "kernel_variant": args.variant,
                      "parallelism": ((f"pixel-partitioned x{world} (rank r: pixels r, r+{world}, ... with all {args.spp} samples; the other pixels of its buffer zero)" if args.partition == "pixels"
                                       else f"sample-partitioned x{world} (rank r: samples r, r+{world}, ... of every pixel)") + " + 1 NCCL sum-reduce of the float4 accumulation buffers") if world > 1 else "single GPU",
                      "l2": f"flushed between steps (256 MiB memset); scene ({st0.scene_bytes / 1e3:.0f} KB) " + ("is staged in shared memory" if in_smem else "is read through L1/L2") + f", output {W * H * 16 / 1e6:.0f} MB accumulation buffer",
                      "reduce_ms_per_step": float(np.mean(red_steps))},
            "samples_per_s": W * H * args.spp / ms_step * 1e3, "samples_per_s_per_gpu": W * H * args.spp / ms_step * 1e3 / world, "rays_per_sample": rays_step / (W * H * args.spp),
            "wall_ms_per_step": wall / args.steps * 1e3,
            "e2e": e2e,
            "gpu_launches": args.steps * world,
            "clocks": {"sm_mhz": sm_mhz, "sm_max_mhz": clk.get("sm_max_mhz"), "reasons": sorted(clk["reasons"]), "n_samples": len(clk["samples"])},
            "roofline": roofline,
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline()
        if last_hdr is not None:
            dump_outputs(args.dump_outputs, last_hdr, float(rays_t[-1]))
        print(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    P.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
