"""What diffuse bounces cost (include/ptcuda.h pt_set_bounces, DESIGN.md 5b): configs 1, 3 and 4 of BASELINE.json at
B = 0, 1, 2 and 4 bounces per path.

  config 1: base, default scene (96 triangles, brute force), 512x512, 64 spp
  config 3: base with triangles.txt, 1920x1080, 1024 spp
  config 4: trianglegrid, 1,048,576-triangle soup (scenes/gen_mesh.soup(1 << 20)), 1920x1080, 256 spp

B = 0 runs the reference kernels (kernel "auto"); B > 0 the path kernel k_bounce_pixel.  Per (config, B): warm-up launches
first, then --steps timed launches, each timed with CUDA events (pt_runtime_ms) with the L2 overwritten (a 256 MiB write)
before it.  One JSON line each: median device ms per frame, traced rays/s and samples/s from the work counters, the share of
bounce rays (rays - samples - shadow rays) among the traced rays, device ns per traced ray, and the card's name and power
limit read in the same run.

    python tools/bounce_time.py [--configs 1,3,4] [--bounces 0,1,2,4] [--steps 3] [--warmup 1]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scenes"))

import torch  # noqa: E402

import gen_mesh  # noqa: E402
import opencl_montecarlo_path_tracing_b200 as pt  # noqa: E402
import write_scenes  # noqa: E402

SEEDS = (1, 2, 3, 4)
CONFIGS = {
    1: dict(variant="base", W=512, H=512, spp=64, soup=0),
    3: dict(variant="base", W=1920, H=1080, spp=1024, soup=0),
    4: dict(variant="grid", W=1920, H=1080, spp=256, soup=1 << 20),
}


def gpu_info():
    """name and power limit of the cards (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout
    except (OSError, subprocess.SubprocessError) as e:
        return ["nvidia-smi unavailable: %s" % e]
    return [line.strip() for line in out.splitlines() if line.strip()]


def scene_of(c):
    with tempfile.TemporaryDirectory() as d:
        write_scenes.write_variant(c["variant"], d)
        s = pt.load_scene_dir(d, c["variant"])
    if c["soup"]:
        tris = gen_mesh.soup(c["soup"])
        lo, hi = gen_mesh.bbox_like_reference(tris)
        s = pt.Scene(s.spheres, s.squares, tris, s.lights, lo, hi)
    return s


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--configs", default="1,3,4")
    ap.add_argument("--bounces", default="0,1,2,4")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    gpus = gpu_info()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")        # > the 126 MB L2
    for cfg in [int(x) for x in args.configs.split(",")]:
        c = CONFIGS[cfg]
        scene = scene_of(c)
        with pt.Renderer(device=0) as r:
            r.set_scene(scene)
            if c["variant"] == "grid":
                r.build_grid(pt.grid_dims(scene))
            for b in [int(x) for x in args.bounces.split(",")]:
                kw = dict(spp=c["spp"], arith="fma", bounces=b, read_image=False)
                for _ in range(args.warmup):
                    r.render(c["variant"], c["W"], c["H"], SEEDS, **kw)
                ms, cnt = [], None
                for k in range(args.steps):
                    flush.fill_(k & 0xFF)
                    torch.cuda.synchronize()
                    out = r.render(c["variant"], c["W"], c["H"], SEEDS, **kw)
                    ms.append(out.ms)
                    cnt = out.counters
                med = statistics.median(ms)
                bounce_rays = cnt["rays"] - cnt["samples"] - cnt["shadow_rays"]
                print(json.dumps({
                    "config": cfg, "variant": c["variant"], "size": "%dx%dx%d" % (c["W"], c["H"], c["spp"]),
                    "triangles": scene.ntriangles, "bounces": b, "kernel": r.last_kernel(),
                    "ms": [round(x, 3) for x in ms], "ms_median": round(med, 3),
                    "rays": cnt["rays"], "shadow_rays": cnt["shadow_rays"], "bounce_rays": bounce_rays,
                    "grays_per_s": round(cnt["rays"] / med / 1e6, 3), "msamples_per_s": round(cnt["samples"] / med / 1e3, 1),
                    "bounce_ray_share": round(bounce_rays / cnt["rays"], 4), "ns_per_ray": round(med * 1e6 / cnt["rays"], 4),
                    "dead_rays": "auto (elide)", "l2": "overwritten before every timed launch", "gpu": gpus}), flush=True)


if __name__ == "__main__":
    main()
