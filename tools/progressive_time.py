"""What progressive rendering costs on config 4: the trianglegrid variant on the 1,048,576-triangle soup
(scenes/gen_mesh.soup(1 << 20)), 1920x1080, 256 spp, kernel and dead_rays "auto", arith "fma" — the frame of bench.py's
headline line — rendered in one launch and as progressions of ranges of 64, 16 and 4 samples (pt_launch_pathtracer_range).

Each form runs on a fresh context (the big-grid tile order records CTA times in the first launch of a geometry, so a
progression's first range and a one-launch frame run in raster order) and on a warmed one (sorted order throughout); the
forms alternate within every repetition.  Every frame's image, accumulation buffer and RNG states must hash (SHA-256) to
the one-launch frame's.  One JSON line per form and context: device ms of the whole frame (sum of its launches' CUDA-event
times) per repetition, the per-range device ms of the median repetition, host wall ms (enqueue to synchronised result),
plus the device name and power limit read in the same run.

    python tools/progressive_time.py [--reps 3] [--ranges 256,64,16,4]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scenes"))

import numpy as np  # noqa: E402

import gen_mesh  # noqa: E402
import opencl_montecarlo_path_tracing_b200 as pt  # noqa: E402
import write_scenes  # noqa: E402

W, H, SPP = 1920, 1080, 256
SEEDS = (1, 2, 3, 4)


def config4_scene():
    with tempfile.TemporaryDirectory() as d:
        write_scenes.write_variant("grid", d)
        s = pt.load_scene_dir(d, "grid")
    tris = gen_mesh.soup(1 << 20)
    lo, hi = gen_mesh.bbox_like_reference(tris)
    return pt.Scene(s.spheres, s.squares, tris, s.lights, lo, hi)


def new_renderer(scene):
    r = pt.Renderer(device=0)
    r.set_scene(scene)
    r.build_grid(pt.grid_dims(scene))
    return r


def gpu_info():
    """name and power limit of the cards (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout
    except (OSError, subprocess.SubprocessError) as e:
        return ["nvidia-smi unavailable: %s" % e]
    return [line.strip() for line in out.splitlines() if line.strip()]


def frame(r, step):
    """one frame in ranges of `step` samples (step == SPP: pt_launch_pathtracer); -> (per-launch device ms, wall ms, digest)"""
    kw = dict(spp=SPP, arith="fma")
    ms = []
    r.synchronize()
    t0 = time.perf_counter()
    for b in range(0, SPP, step):
        last = b + step == SPP
        out = r.render("grid", W, H, SEEDS, samples=None if step == SPP else (b, b + step), read_image=last,
                       want_accum=last, want_rng=last, **kw)
        ms.append(out.ms)
    wall = (time.perf_counter() - t0) * 1e3
    h = hashlib.sha256(out.image.tobytes() + out.accum.tobytes() + out.rng_state.tobytes()).hexdigest()
    return ms, wall, h


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ranges", default="256,64,16,4", help="range lengths to time (%d = one launch)" % SPP)
    args = ap.parse_args()
    steps = [int(s) for s in args.ranges.split(",")]
    if any(SPP % s for s in steps):
        ap.error("every range length must divide %d" % SPP)
    gpus = gpu_info()
    scene = config4_scene()
    warm = new_renderer(scene)
    ref = None
    for s in steps:                                    # warm-up: modules, tile order of the geometry, the one-launch digest
        _, _, h = frame(warm, s)
        if s == SPP:
            ref = h
    if ref is None:
        ref = frame(warm, SPP)[2]
    results = {(s, ctx): [] for s in steps for ctx in ("fresh", "warm")}
    for _ in range(args.reps):
        for s in steps:
            fresh = new_renderer(scene)
            try:
                results[(s, "fresh")].append(frame(fresh, s))
            finally:
                fresh.close()
            results[(s, "warm")].append(frame(warm, s))
    warm.close()
    ok = True
    for (s, ctx), runs in results.items():
        totals = [sum(ms) for ms, _, _ in runs]
        med = int(np.argsort(totals)[len(totals) // 2])
        same = all(h == ref for _, _, h in runs)
        ok &= same
        print(json.dumps({"form": "one launch" if s == SPP else "ranges of %d" % s, "context": ctx, "launches": SPP // s,
                          "device_ms_total": [round(t, 3) for t in totals], "device_ms_median": round(totals[med], 3),
                          "range_ms": [round(m, 3) for m in runs[med][0]], "wall_ms": [round(w, 3) for _, w, _ in runs],
                          "same_sha256_as_one_launch": same, "workload": "config 4: soup 1M, %dx%d, %d spp" % (W, H, SPP),
                          "gpu": gpus}), flush=True)
    if not ok:
        sys.exit("a progression did not end in the one-launch frame")


if __name__ == "__main__":
    main()
