#!/usr/bin/env python3
"""Benchmark of the CLSuperPathTracer hot path (BASELINE.json metric: Mrays/s and samples/s per image).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path over one image: render the workload's frame (all samples of all pixels)
into device memory.  BASELINE.json quotes its metric on no single config, so the defaults are

  N = 1 : BASELINE config 4 — CLSuperPathTracer_trianglegrid, synthetic 1,048,576-triangle mesh, 1920x1080, 256 spp
          (the largest single-GPU config).  The same run also measures configs 1, 2, 3 (both meshes) and the config-5
          scene at 64 of its 4096 spp, each with value / e2e / roofline / cpu_baseline / parity_check, under "configs".
  N > 1 : BASELINE config 5 STRONG-scaled — the 1 M-triangle scene at a FIXED 3840x2160, 64 of the 4096 spp (work is
          exactly linear in spp; stated in config.spp_note), 8-row stripes dealt round-robin to the ranks, one NCCL
          reduce of the float accumulation buffer onto rank 0, rank 0 tone-maps.  `--weak` grows the frame instead.

  value   : Mrays/s, device time (CUDA events on the launching stream, one event pair per step, L2 flushed between
            steps), scene already resident in HBM / constant memory.  1 ray = 1 TraceRay evaluation (primary + shadow),
            counted on the device and cross-checked against the oracle in tests/.
  e2e     : the same metric through the reference-facing C ABI with HOST buffers, wall clock per step:
            N = 1: pt_render_host() = scene upload (H2D) + grid build + launch + blocking read of the RGBA8 image (D2H);
            N > 1: every rank uploads the scene and builds its grid, renders its stripes, the NCCL reduce, rank 0
            tone-maps and ONLY rank 0 reads the frame back.
  parity_check : after timing, row bands of the TIMED output are compared byte for byte with the CPU oracle, and for
            N > 1 the SHA-256 of the reduced frame with a 1-GPU render of the whole frame.  A mismatch exits non-zero.
  roofline: the kernels are FP32-pipe / issue-slot bound (scene in constant or shared memory or L2-resident, 4 B of
            output per pixel; HBM idles).  `achieved` = EXECUTED flop/s (analytic tests of every ray + triangle tests
            after the conservative culls + grid cells + VPL evaluations, from the device counters), `peak` = FP32
            TFLOP/s of a pure FFMA kernel measured live on this GPU (pt_measure_peaks); `frac` = achieved / peak.
            Beside it: the algorithmic figure of SURVEY.md 8d (F_ray = 3 + 12 n_sq + 21 n_sph + 58 n_tri per ray; the
            culls skip work the reference does, so it can exceed the peak) and `issue_frac` = warp instructions per
            launch (ncu, profiles/ncu_reference_numbers.json) / kernel time (live) / measured issue rate (live).
  cpu_baseline: the reference's own CPU run of the same frame (oracle/_ref = unmodified reference compiled through
            oracle/refrt) where it can hold the workload (<= 512 triangles, 64 spp), else the C oracle port on rows
            sampled over the frame, all host cores, thread count verified.
  --impl reference : that CPU measurement alone, once per warm-up and timed step; each step costs about --cpu-budget
            seconds of CPU work (whole light frames: their full reference run), so the run grows with --steps.
  step_ms : the time of every timed step; `steps` is their count.
  --dump-outputs DIR : after the timed steps of the headline workload, what its last step left for the caller is written as
            DIR/<name>.npy in float32: image.npy = the (H, W, 4) RGBA8 frame, and at N > 1 accum.npy = the reduced float
            accumulation buffer.  Inputs are fixed (seeds, scene, synthetic mesh seed), so two builds can be compared file for
            file.  Above 64 MB in all, every array keeps the same seeded sample of rows, listed in rows.npy (float64).
"""
import argparse
import hashlib
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scenes"))

SEEDS = (1, 2, 3, 4)

WORKLOADS = {
    # name: variant, scene dir variant, mesh override, W, H, spp, BASELINE.json config number
    "nodof_512x512x64": dict(variant="nodof", scene="nodof", mesh=None, W=512, H=512, spp=64, config=2,
                             desc="CLSuperPathTracer_lmem_NoDoF scene (5 spheres, 3 squares, 2 lights), 512x512, 64 spp"),
    "base_512x512x64": dict(variant="base", scene="base", mesh=None, W=512, H=512, spp=64, config=1,
                            desc="CLSuperPathTracer default scene (96 triangles brute force), 512x512, 64 spp"),
    "lmem_512x512x64": dict(variant="lmem", scene="lmem", mesh=None, W=512, H=512, spp=64, config=None,
                            desc="CLSuperPathTracer_lmem scene, 512x512, 64 spp"),
    "grid_512x512x64": dict(variant="grid", scene="grid", mesh=None, W=512, H=512, spp=64, config=None,
                            desc="CLSuperPathTracer_trianglegrid default scene (96 triangles, 8x5x6 grid), 512x512, 64 spp"),
    "bidir_512x512x64": dict(variant="bidir", scene="bidir", mesh=None, W=512, H=512, spp=64, config=None,
                             desc="CLSuperBidirectionalPathTracer default scene (512 VPLs per light, 2 lights, 96 triangles), 512x512, "
                                  "64 spp; a step = light-tracing pass + path-tracing pass"),
    "bidir_1920x1080x64": dict(variant="bidir", scene="bidir", mesh=None, W=1920, H=1080, spp=64, config=None,
                               desc="CLSuperBidirectionalPathTracer default scene, 1920x1080, 64 spp; a step = light + path pass"),
    "torus_1920x1080x1024": dict(variant="base", scene="base", mesh="torus", W=1920, H=1080, spp=1024, config=3,
                                 desc="CLSuperPathTracer with torus.txt (32 triangles), DoF, 1920x1080, 1024 spp"),
    "base_1920x1080x1024": dict(variant="base", scene="base", mesh=None, W=1920, H=1080, spp=1024, config=3,
                                desc="CLSuperPathTracer with triangles.txt (96 triangles), DoF, 1920x1080, 1024 spp"),
    "gridsoup1m_1920x1080x256": dict(variant="grid", scene="grid", mesh=None, soup=1 << 20, W=1920, H=1080, spp=256, config=4,
                                     desc="CLSuperPathTracer_trianglegrid, synthetic 1,048,576-triangle soup (scenes/gen_mesh.py seed "
                                          "20261018, 60^3 box, 128^3 grid, 32-bit cell ids), 1920x1080, 256 spp"),
    "gridsoup1m_3840x2160x4096": dict(variant="grid", scene="grid", mesh=None, soup=1 << 20, W=3840, H=2160, spp=4096, config=5,
                                      desc="BASELINE config 5 in full: 1M-triangle soup, 3840x2160, 4096 spp (34 G samples per frame); "
                                           "use with --steps 1"),
    "gridsoup1m_3840x2160x64": dict(variant="grid", scene="grid", mesh=None, soup=1 << 20, W=3840, H=2160, spp=64, config=5,
                                    spp_note="64 of BASELINE config 5's 4096 spp (work is exactly linear in spp: same pixels, same "
                                             "scene, 1/64 of the samples of every pixel)",
                                    desc="config-5 scene (1M-triangle soup) at 3840x2160 with 64 of the 4096 spp"),
}
DEFAULT_N1 = "gridsoup1m_1920x1080x256"
DEFAULT_MULTI = "gridsoup1m_3840x2160x64"
EXTRA_N1 = ["base_512x512x64", "nodof_512x512x64", "base_1920x1080x1024", "torus_1920x1080x1024", "gridsoup1m_3840x2160x64"]


def flops_per_ray(scene):
    nsq = sum(bin(int(v) & 0x7FFFF).count("1") for v in scene.squares)
    nsp = sum(bin(int(v) & 0x7FFFF).count("1") for v in scene.spheres)
    return 3 + 12 * nsq + 21 * nsp + 58 * scene.ntriangles


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append((time.time(), [x.strip() for x in line.split(",")]))
        except Exception:
            pass

    def finish(self, t0, t1):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, f in self.samples:
            if ts < t0 - 0.05 or ts > t1 + 0.15 or len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            for ts, f in self.samples[-3:]:
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


def scene_dir_for(w, tmp):
    import write_scenes
    d = os.path.join(tmp, w["scene"] + ("_" + w["mesh"] if w["mesh"] else ""))
    if not os.path.isdir(d):
        write_scenes.write_variant(w["scene"], d, mesh=w["mesh"])
        if w["variant"] == "nodof":          # the reference NoDoF host reads planes.txt
            import shutil
            shutil.copy(os.path.join(d, "squares.txt"), os.path.join(d, "planes.txt"))
    return d


_SOUP = {}


def soup_triangles(n):
    if n not in _SOUP:
        import gen_mesh
        tris = gen_mesh.soup(n)
        lo, hi = gen_mesh.bbox_like_reference(tris)
        _SOUP[n] = (tris, lo, hi)
    return _SOUP[n]


def load_workload_scene(w, d):
    """pt.Scene of the workload: parsed from the scene directory, triangles replaced by the synthetic soup
    for the config-4/5 workloads (bit-identical to what the parsers would read from its text file)."""
    import opencl_montecarlo_path_tracing_b200 as pt
    scene = pt.load_scene_dir(d, w["variant"])
    if w.get("soup"):
        tris, lo, hi = soup_triangles(w["soup"])
        scene = pt.Scene(scene.spheres, scene.squares, tris, scene.lights, lo, hi)
    return scene


# ------------------------------------------------------------------------------------------ CPU side: oracle / reference
_PORT_CACHE = {}


def port_scene(w, d, contract):
    """(OracleLib, scene dict, grid dict or None) of the workload for the C oracle port; prepared once per contract."""
    from oracle.pyoracle import OracleLib
    key = (w["variant"], w.get("soup"), w.get("mesh"), contract)
    if key not in _PORT_CACHE:
        o = OracleLib(contract)
        sc = o.load_scene_dir(d, w["variant"])
        if w.get("soup"):
            tris, lo, hi = soup_triangles(w["soup"])
            sc.update(triangles=tris, box_min=lo, box_max=hi)
        grid = None
        if w["variant"] == "grid":
            res, cell = o.grid_dims(sc["box_min"], sc["box_max"], sc["triangles"].shape[0], 3.0)
            grid = {"box_min": sc["box_min"], "box_max": sc["box_max"], "res": res, "cell_size": cell}
            grid["csr"] = o.build_grid(sc["triangles"], sc["box_min"], res, cell)
        _PORT_CACHE[key] = (o, sc, grid)
    return _PORT_CACHE[key]


def spread_rows(H):
    """Rows of the frame in bit-reversal (van der Corput) order: any prefix is spread evenly over the image."""
    bits = max(1, (H - 1).bit_length())
    out = []
    for k in range(1 << bits):
        r = int(format(k, "0%db" % bits)[::-1], 2)
        if r < H:
            out.append(r)
    return out


def run_port_sample(w, d, W, H, spp, budget_s=8.0, max_rows=256):
    """Oracle port (all host cores) on single rows spread over the frame until `budget_s` of CPU work is reached.
    -> dict(ms, rays, samples, rows, threads)"""
    o, sc, grid = port_scene(w, d, 0)
    cores = host_cores()
    tot_ms, rays, samples, rows, threads = 0.0, 0, 0, [], cores
    order = spread_rows(H)
    half = order[1:] if len(order) > 1 else order      # row 0 is sky in every workload: start in the middle of the frame
    for r in half[:max_rows]:
        t0 = time.perf_counter()
        out = o.render(w["variant"], W, H, SEEDS, sc, spp=spp, rows=(r, r + 1), grid=grid, want_accum=False, want_rng=False,
                       nthreads=cores)
        tot_ms += (time.perf_counter() - t0) * 1e3
        rays += out["counters"]["rays"]; samples += out["counters"]["samples"]
        rows.append(r)
        threads = min(threads, out["threads"])
        if tot_ms >= budget_s * 1e3:
            break
    return dict(ms=tot_ms, rays=rays, samples=samples, rows=rows, threads=threads)


def ref_exe_name(w):
    return "CLSuperBidirectionalPathTracer" if w["variant"] == "bidir" else "CLSuperPathTracer"


def oracle_cli_stats(w, d, W, H, threads):
    """Whole frame through oracle/_build/oracle_cli -> its ORACLE_STATS dict (time + work counters)."""
    from oracle import pyoracle
    pyoracle.build()
    env = dict(os.environ, PT_SEEDS=",".join(str(s) for s in SEEDS), PT_SPP=str(w["spp"]), PT_THREADS=str(threads),
               OMP_NUM_THREADS=str(threads), PT_OUT=os.path.join(d, "oracle_result.ppm"))
    out = subprocess.run([os.path.join(pyoracle.BUILD, "oracle_cli"), w["variant"], str(W), str(H)], cwd=d, env=env,
                         capture_output=True, text=True, check=True).stdout
    return json.loads(out[out.index("ORACLE_STATS") + len("ORACLE_STATS"):])


def run_reference_binary(w, d, W, H):
    """The unmodified reference (oracle/_ref, built by `make -C oracle ref`) on the whole frame with every host core.
    torchrun exports OMP_NUM_THREADS=1 to its children: the thread count is therefore FORCED here, and read back from
    the device line the reference host prints (refrt names its device "host CPU, <n> OpenMP threads").
    -> (kernel ms, threads) or None when the binary is not there."""
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "bin", w["variant"], ref_exe_name(w))
    if not os.path.exists(ref_bin):
        return None
    cores = host_cores()
    env = dict(os.environ, PT_SEEDS=",".join(str(s) for s in SEEDS), OMP_NUM_THREADS=str(cores), OMP_DYNAMIC="false")
    env.pop("OMP_THREAD_LIMIT", None)
    out = subprocess.run([ref_bin, str(W), str(H)], cwd=d, env=env, capture_output=True, text=True, check=True).stdout
    ms = 0.0
    for pat in (r"rendering : .* in ([0-9.eE+-]+)ms", r"reduce img samples : .* in ([0-9.eE+-]+)ms",
                r"virtual light sampling : .* in ([0-9.eE+-]+)ms"):
        m = re.search(pat, out)
        if m:
            ms += float(m.group(1))
    m = re.search(r"(\d+) OpenMP threads", out)
    threads = int(m.group(1)) if m else None
    return ms, threads


def is_heavy(w):
    return bool(w.get("soup")) or w["spp"] != 64 or w["W"] * w["H"] > 512 * 512


def cpu_reference_measure(w, d, W, H, spp, budget_s=8.0):
    """One bounded CPU measurement of the workload -> dict(mrays, msamples, ms, kind, cores, sample, rays, samples).
    Light workloads (<= 512 triangles, 64 spp, <= 512x512): the unmodified reference binary on the full frame.
    Heavy ones (1 M triangles exceed the reference's MAX_TRIANGLES / 16-bit ids; spp != 64 is an extension): the oracle
    port on single rows spread over the image until ~budget_s of CPU work; throughput = rays of those rows / their time."""
    cores = host_cores()
    if not is_heavy(w) and H == w["H"]:
        got = run_reference_binary(w, d, W, H)
        if got is not None:
            ms, threads = got
            if threads is not None and threads != cores:
                raise RuntimeError("reference ran on %d threads, expected %d" % (threads, cores))
            stats = oracle_cli_stats(w, d, W, H, cores)        # ray / sample count of the same frame (same seeds)
            return dict(mrays=stats["rays"] / 1e3 / ms, msamples=stats["samples"] / 1e3 / ms, ms=ms, kind="reference", cores=cores,
                        rays=stats["rays"], samples=stats["samples"],
                        sample="the full %dx%dx%d frame, unmodified reference host + kernels through oracle/refrt, %s OpenMP threads "
                               "(kernel time printed by the reference host)" % (W, H, spp, threads if threads is not None else cores))
    s = run_port_sample(w, d, W, H, spp, budget_s)
    if s["threads"] != cores:
        raise RuntimeError("oracle port ran on %d threads, expected %d" % (s["threads"], cores))
    return dict(mrays=s["rays"] / 1e3 / s["ms"], msamples=s["samples"] / 1e3 / s["ms"], ms=s["ms"], kind="port", cores=cores,
                rays=s["rays"], samples=s["samples"],
                sample="oracle port, %d single rows spread over the %dx%d frame (bit-reversal order, first %s ...) at the full %d spp, "
                       "%d OpenMP threads verified; throughput = rays of those rows / their time (work is additive over pixels)"
                       % (len(s["rows"]), W, H, s["rows"][:6], spp, s["threads"]))


def reference_opencl_on_gpu(w, d, W, H, rays):
    """The unmodified reference run by NVIDIA's OpenCL runtime on this GPU (oracle/_ref/ocl, if built and the
    ICD is usable): the "same kernel, same box" baseline.  Returns a dict or None."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ocl", w["variant"], ref_exe_name(w))
    if not os.path.exists(exe) or is_heavy(w):
        return None
    env = dict(os.environ, OCL_ICD_FILENAMES="libnvidia-opencl.so.1", PT_SEEDS=",".join(str(s) for s in SEEDS))
    best = None
    try:
        for _ in range(3):
            p = subprocess.run([exe, str(W), str(H)], cwd=d, env=env, capture_output=True, text=True, timeout=300)
            if p.returncode != 0:
                return None
            ms = sum(float(x) for x in re.findall(r"(?:rendering|reduce img samples|virtual light sampling) : .*? in ([0-9.eE+-]+)ms", p.stdout))
            best = ms if best is None else min(best, ms)
    except Exception:
        return None
    if not best:
        return None
    return {"value": rays / 1e3 / best, "unit": "Mrays/s", "kernel_ms": best,
            "what": "unmodified reference .c + .ocl, NVIDIA OpenCL ICD on the same B200, OpenCL event time, best of 3"}


def simple_cpu_tracer_baseline():
    """SimpleCPUTracer (the reference's single-threaded CPU tracer; its own hard-wired scene and rand(), so a reported
    baseline only, never an oracle), built from the reference source into oracle/_ref by `make -C oracle ref`.
    Run at BASELINE.md's two sizes."""
    exe = os.path.join(ROOT, "oracle", "_ref", "bin", "simplecpu", "simpleCPUtracer")
    if not os.path.exists(exe):
        return None
    runs = []
    for n in (256, 512):
        try:
            with tempfile.TemporaryDirectory() as t:
                out = subprocess.run([exe, str(n), str(n)], cwd=t, capture_output=True, text=True, timeout=300, check=True).stdout
            ms = float(re.search(r"rendering \(host\) : .* in ([0-9.eE+-]+)ms", out).group(1))
        except Exception:
            continue
        samples = n * n * 64
        runs.append({"value": samples / 1e3 / ms, "unit": "Msamples/s", "cores": 1, "ms": ms, "kind": "reference",
                     "sample": "SimpleCPUTracer, its built-in scene, %dx%dx64 (serial rand(): one thread by construction)" % (n, n)})
    return runs or None


def bench_reference(args, w, wname):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, args.gpus)
    strong = not args.weak
    W, H, spp = w["W"], (w["H"] if strong or world == 1 else w["H"] * world), w["spp"]
    with tempfile.TemporaryDirectory() as tmp:
        d = scene_dir_for(w, tmp)
        runs = []
        for i in range(args.warmup + args.steps):
            m = cpu_reference_measure(w, d, W, H, spp, budget_s=args.cpu_budget)
            if i >= args.warmup:
                runs.append(m)
    ms = sum(m["ms"] for m in runs) / len(runs)
    mrays = sum(m["mrays"] for m in runs) / len(runs)
    msamples = sum(m["msamples"] for m in runs) / len(runs)
    kind, cores, sample = runs[0]["kind"], runs[0]["cores"], runs[0]["sample"]
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": mrays, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": len(runs),
        "warmup": args.warmup, "ms_per_step": ms, "step_ms": [round(m["ms"], 3) for m in runs], "higher_is_better": True,
        "scaling": "strong" if (strong and world > 1) else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(w, wname, W, H, spp),
        "msamples_per_s": msamples, "rays_per_step": runs[0]["rays"], "samples_per_step": runs[0]["samples"],
        "cpu_baseline": {"value": mrays, "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(w, wname, W, H, spp):
    cfg = {"workload": wname, "baseline_config": w.get("config"), "description": w["desc"], "width": W, "height": H, "spp": spp,
           "seeds": list(SEEDS)}
    if w.get("spp_note"):
        cfg["spp_note"] = w["spp_note"]
    return cfg


# -------------------------------------------------------------------------------------------------- parity of timed output
def parity_bands(W, H, spp):
    nb = max(1, min(4, int(2_000_000 // (W * spp))))
    return [(int(H * f), min(H, int(H * f) + nb)) for f in (0.15, 0.39, 0.66)]


def check_against_oracle(w, d, W, H, spp, image, rerender=None, extra=None):
    """Compare row bands of `image` (H, W, 4 uint8: the output of the timed steps) with the CPU oracle, byte for byte.
    The timed arithmetic policy is FMA (oracle built with -DPT_CONTRACT=1); on a host CPU without FMA the bands are
    re-rendered with the separate-rounding policy (`rerender(rows)`) and compared with the uncontracted oracle."""
    import numpy as np
    from oracle.pyoracle import cpu_has_fma
    fma = cpu_has_fma()
    o, sc, grid = port_scene(w, d, 1 if fma else 0)
    bands = parity_bands(W, H, spp)
    ok, bad = True, 0
    t0 = time.perf_counter()
    for rows in bands:
        kw = dict(extra or {})
        ref = o.render(w["variant"], W, H, SEEDS, sc, spp=spp, rows=rows, grid=grid, want_accum=False, want_rng=False, **kw)
        got = image[rows[0]:rows[1]] if fma else rerender(rows)[rows[0]:rows[1]]
        diff = (got != ref["image"][rows[0]:rows[1]]).any(axis=2)
        bad += int(diff.sum())
        ok = ok and not diff.any()
    return {"rows": [list(b) for b in bands], "bit_exact": bool(ok), "mismatching_pixels": bad,
            "against": "CPU oracle (oracle/oracle.c, %s), RGBA8 bytes of the timed output" % ("-DPT_CONTRACT=1" if fma else
                       "uncontracted; bands re-rendered with PT_ARITH_SEPARATE because the host CPU has no FMA"),
            "oracle_s": round(time.perf_counter() - t0, 2)}


DUMP_LIMIT_BYTES = 64_000_000
DUMP_ROW_SEED = 20261018


def dump_outputs(out_dir, arrays):
    """Writes every (H, ...) array of `arrays` as out_dir/<name>.npy in float32 (RGBA8 values are exact in it).  When they
    exceed DUMP_LIMIT_BYTES in all, each keeps the same fixed, seeded sample of rows, written as rows.npy (float64)."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v, np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        H = next(iter(arrays.values())).shape[0]
        keep = max(1, H * (DUMP_LIMIT_BYTES - (1 << 20)) // total)      # 1 MiB left for the row list and the .npy headers
        rows = np.sort(np.random.default_rng(DUMP_ROW_SEED).choice(H, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ---------------------------------------------------------------------------------------------------- our arm
class Ours:
    def __init__(self, args):
        import torch
        import opencl_montecarlo_path_tracing_b200 as pt
        self.torch, self.pt, self.args = torch, pt, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != max(1, args.gpus) and self.world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d" % (args.gpus, args.gpus))
        torch.cuda.set_device(self.local_rank)
        self.dist = None
        self.saved_stdout = None
        self.outputs = None                          # rank 0, headline workload: what the last timed step computed
        if self.world > 1:
            # NCCL (NCCL_DEBUG=INFO/VERSION) prints on stdout; the contract is ONE JSON line there -> park stdout on stderr
            # for the duration of the run (NCCL_DEBUG itself is left exactly as the caller set it)
            sys.stdout.flush()
            self.saved_stdout = os.dup(1)
            os.dup2(2, 1)
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist
        self.stream = torch.cuda.Stream()            # a real stream (the legacy default stream cannot be graph-captured)
        torch.cuda.set_stream(self.stream)
        self.r = pt.Renderer(device=self.local_rank, stream=self.stream.cuda_stream)
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2
        self.tmp = tempfile.TemporaryDirectory()
        self.props = self.r.device_props()
        self.peaks_file = measured_peaks()
        self.live = self.r.measure_peaks()           # FP32 TFLOP/s and warp-instruction issue rate of THIS GPU, now
        try:
            self.ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_reference_numbers.json")))
        except Exception:
            self.ncu = {}

    def close(self):
        self.r.close()
        self.tmp.cleanup()
        if self.dist:
            self.dist.destroy_process_group()

    def emit(self, line):
        sys.stdout.flush()
        if self.saved_stdout is not None:
            os.dup2(self.saved_stdout, 1)
        print(json.dumps(line), flush=True)
        if self.saved_stdout is not None:
            os.dup2(2, 1)

    # -- one workload: device-timed steps, e2e, parity, roofline, cpu baseline ------------------------------------
    def measure(self, wname, steps, warmup, headline, cpu_baseline=True):
        torch, pt, args, r, dist = self.torch, self.pt, self.args, self.r, self.dist
        import numpy as np
        w = WORKLOADS[wname]
        rank, world = self.rank, self.world
        by_samples = args.shard == "samples" and world > 1
        if by_samples and w["variant"] == "nodof":
            raise SystemExit("--shard samples is for the per-pixel-stream variants (NoDoF shards by tiles)")
        strong = not args.weak
        W, H, spp = w["W"], (w["H"] if strong or by_samples or world == 1 else w["H"] * world), w["spp"]
        if by_samples and not strong:
            spp *= world                             # weak scaling in the sample dimension
        d = scene_dir_for(w, self.tmp.name)
        scene = load_workload_scene(w, d)
        r.set_scene(scene)
        grid = pt.grid_dims(scene) if w["variant"] == "grid" else None
        if grid is not None:
            r.build_grid(grid)
        kw = dict(spp=spp, kernel=args.kernel, arith="fma", dead_rays=args.dead_rays)
        if args.scene_mem:
            kw["scene_mem"] = args.scene_mem
        kw1 = dict(kw)                               # the same launch on one GPU (for the N>1 identity check)
        if by_samples:
            kw.update(sample_block=rank, sample_blocks=world)
        elif world > 1:
            kw.update(interleave=8, rank=rank, nranks=world)
        variant = w["variant"]
        bidir = variant == "bidir"
        rgba = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        accum = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda") if world > 1 else None
        kev = []                                     # (start, stop) events around this rank's render kernel, per step

        def step(record=False):
            if bidir:                                # the light pass is part of the path (every rank traces the same VPLs)
                r.light_tracer(SEEDS, 512, wait=False)
            if world > 1:
                accum.zero_()
                if record:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(self.stream)
                r.render_device(variant, W, H, SEEDS, rgba.data_ptr(), accum.data_ptr(), **kw)
                if record:
                    e1.record(self.stream)
                    kev.append((e0, e1))
                dist.reduce(accum, dst=0)            # the ONLY collective: sum of the per-rank accumulation buffers
                if rank == 0:
                    r.tonemap_device(accum.data_ptr(), rgba.data_ptr(), W, H)
            else:
                r.render_device(variant, W, H, SEEDS, rgba.data_ptr(), None, **kw)

        warm = max(3, warmup)
        for _ in range(warm):
            step()
        torch.cuda.synchronize()
        counters = r.counters()                      # this rank's share of the frame: the work the timed launch really does
        resolved_kernel = r.last_kernel()
        # The metric counts the REFERENCE's rays (1 ray = 1 TraceRay call of the reference for this frame, BASELINE.md 3): with
        # dead shadow rays elided (the default, include/ptcuda.h pt_render_params.dead_rays) the timed launch traces fewer, so
        # one untimed launch in TRACE mode supplies the reference's own counts (they equal the oracle's: tests/).
        counters_ref = counters
        if args.dead_rays != "trace" and variant != "nodof":
            kw_t = dict(kw, dead_rays="trace")
            if world > 1:
                r.render_device(variant, W, H, SEEDS, rgba.data_ptr(), accum.data_ptr(), **kw_t)
            else:
                r.render_device(variant, W, H, SEEDS, rgba.data_ptr(), None, **kw_t)
            torch.cuda.synchronize()
            counters_ref = r.counters()
            step()                                   # leave the buffers as a timed step leaves them
            torch.cuda.synchronize()
        launches_per_render = {"spec": 2}.get(resolved_kernel, 1)     # PT_KERNEL_SPEC = light pass + heavy pass
        if world > 1:
            dist.barrier()
        sampler = None
        if headline:
            sampler = ClockSampler(self.local_rank)
            sampler.start()
            time.sleep(0.25)
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        torch.cuda.synchronize()
        t0 = time.time()
        for k in range(steps):
            self.flush.fill_(k & 0xFF)               # L2 flush between timed iterations (not timed)
            starts[k].record(self.stream)
            step(record=True)
            stops[k].record(self.stream)
        torch.cuda.synchronize()
        t1 = time.time()
        if world > 1:
            dist.barrier()
        clocks = sampler.finish(t0, t1) if sampler else None
        if headline and args.dump_outputs and rank == 0:
            self.outputs = {"image": rgba.cpu().numpy().view(np.uint8).reshape(H, W, 4)}
            if accum is not None:                    # rank 0 holds the reduced sum
                self.outputs["accum"] = accum.cpu().numpy()
        step_ms = [s.elapsed_time(e) for s, e in zip(starts, stops)]
        total_ms = sum(step_ms)
        rays, samples, rays_traced = float(counters_ref["rays"]), float(counters_ref["samples"]), float(counters["rays"])
        per_rank = None
        if world > 1:
            my_kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / max(1, len(kev))
            tot = torch.tensor([total_ms, rays, samples, my_kernel_ms, rays_traced], dtype=torch.float64, device="cuda")
            gathered = [torch.zeros_like(tot) for _ in range(world)]
            dist.all_gather(gathered, tot)
            g = torch.stack(gathered).cpu().numpy()
            total_ms = float(g[:, 0].max())          # max over ranks
            rays, samples, rays_traced = float(g[:, 1].sum()), float(g[:, 2].sum()), float(g[:, 4].sum())
            km = g[:, 3]
            per_rank = {"render_kernel_ms": {"min": float(km.min()), "mean": float(km.mean()), "max": float(km.max()),
                                             "per_rank": [round(float(x), 4) for x in km]},
                        "rays_per_rank": [float(x) for x in g[:, 1]],
                        "step_ms_per_rank": [round(float(x) / steps, 4) for x in g[:, 0]]}
        ms_per_step = total_ms / steps

        # ---- parity of the TIMED output (rank 0 holds the frame)
        parity = None
        if rank == 0 and not args.no_parity:
            timed_img = rgba.cpu().numpy().view(np.uint8).reshape(H, W, 4)

            def rerender(rows):
                res = r.render(variant, W, H, SEEDS, rows=rows, spp=spp, arith="separate", kernel=args.kernel)
                return res.image
            if by_samples:
                parity = {"bit_exact": None, "skipped": "sample-range sharding re-seeds the per-block streams: statistically equivalent, "
                                                         "not bit-identical to one stream per pixel (tests/test_sample_sharding_gpu.py)"}
            else:
                parity = check_against_oracle(w, d, W, H, spp, timed_img, rerender)
            if world > 1 and not by_samples:
                sha_n = hashlib.sha256(timed_img.tobytes()).hexdigest()
                rgba1 = torch.zeros((H, W), dtype=torch.int32, device="cuda")
                if bidir:
                    r.light_tracer(SEEDS, 512, wait=False)
                r.render_device(variant, W, H, SEEDS, rgba1.data_ptr(), None, **kw1)
                torch.cuda.synchronize()
                sha_1 = hashlib.sha256(rgba1.cpu().numpy().tobytes()).hexdigest()
                parity["multi_gpu"] = {"sha256_reduced_frame": sha_n, "sha256_one_gpu_render": sha_1, "identical": sha_n == sha_1}
                parity["bit_exact"] = bool(parity["bit_exact"] and sha_n == sha_1)
                del rgba1
        if world > 1:
            dist.barrier()

        # ---- e2e through the reference-facing API with HOST buffers
        import ctypes as C
        from opencl_montecarlo_path_tracing_b200 import _lib
        lib = _lib.cuda_lib()
        h2d_rank = 2 * (2848 + 48 * min(scene.ntriangles, 512)) + scene.ntriangles * 48   # two policy scene-block prefixes + raw triangles
        heavy_step = ms_per_step > 500.0             # multi-second frames: one warm + one timed end-to-end call is enough
        e2e_warm = 1 if heavy_step else 2
        e2e_steps = 1 if heavy_step else max(3, min(steps, 10))
        if world == 1:
            r2 = pt.Renderer(device=self.local_rank)
            cs = scene.to_c()
            p = pt.make_params(variant, W, H, SEEDS, **kw)
            host_img = np.zeros((H, W, 4), np.uint8)
            for i in range(e2e_warm + e2e_steps):
                if i == e2e_warm:
                    r2.synchronize()
                    te0 = time.perf_counter()
                rc = lib.pt_render_host(r2.ctx, C.byref(cs), C.byref(grid) if grid is not None else None, C.byref(r2.cam), C.byref(p),
                                        host_img.ctypes.data_as(C.POINTER(C.c_uint8)))
                assert rc == 0, lib.pt_last_error()
            e2e_ms = (time.perf_counter() - te0) * 1e3 / e2e_steps
            r2.close()
            e2e_api = "pt_render_host (scene upload + grid build + launch + blocking RGBA8 read)"
            h2d, d2h = h2d_rank, W * H * 4
        else:
            host_img = torch.empty((H, W), dtype=torch.int32, pin_memory=True) if rank == 0 else None
            for i in range(e2e_warm + e2e_steps):
                if i == e2e_warm:
                    torch.cuda.synchronize()
                    dist.barrier()
                    te0 = time.perf_counter()
                r.set_scene(scene)                   # host scene -> device (every rank)
                if grid is not None:
                    r.build_grid(grid)
                step()
                if rank == 0:
                    host_img.copy_(rgba)             # only rank 0 reads the frame back
                torch.cuda.synchronize()
            dist.barrier()
            e2e_ms = (time.perf_counter() - te0) * 1e3 / e2e_steps
            t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t[0])
            e2e_api = ("per rank: pt_set_scene + pt_build_grid (H2D) + pt_render_device of its stripes; NCCL reduce of the accumulation "
                       "buffer; rank 0: pt_tonemap_device + read of the RGBA8 frame into pinned host memory (D2H); wall clock, max over ranks")
            h2d, d2h = h2d_rank * world, W * H * 4

        if rank != 0:
            return None

        # ---- roofline (rank 0's own kernel: at N > 1 its share of the frame and its own kernel time)
        F = flops_per_ray(scene)
        kernel_ms = ms_per_step if world == 1 else per_rank["render_kernel_ms"]["per_rank"][0]
        F_analytic = F - 58 * scene.ntriangles
        flops_exec = F_analytic * counters["rays"] + 58.0 * counters["tri_tests_executed"] + 30.0 * counters["cells_visited"]
        vpl_info = None
        if bidir:
            vp = r.read_vpls()
            nact = int((vp[:, 3] != 0).sum())                  # entries the gather visits (NaN counts, as in the reference)
            hit_samples = counters["shadow_rays"] // max(1, scene.lights.shape[0])
            flops_exec += 22.0 * hit_samples * nact            # ~22 flop per (hit sample, non-zero VPL)
            vpl_info = {"buffer": int(vp.shape[0]), "non_zero": nact, "reference_loop_iterations": counters["vpl_evals"],
                        "executed_evaluations": hit_samples * nact}
        executed = flops_exec / (kernel_ms * 1e-3) / 1e12
        if variant == "grid":                                  # per-ray grid work is data dependent: taken from the TRACE-mode counters
            flops_alg = F_analytic * counters_ref["rays"] + 58.0 * counters_ref["tri_tests_executed"] + 30.0 * counters_ref["cells_visited"]
        else:
            flops_alg = F * float(counters_ref["rays"]) + (22.0 * vpl_info["executed_evaluations"] if vpl_info else 0.0)
        algorithmic = flops_alg / (kernel_ms * 1e-3) / 1e12
        fp32_peak = self.live["fp32_tflops"]
        issue_peak = self.live["mixed_gwarp_inst_per_s"]
        grid_bytes = 8.0 * counters["cells_visited"] + 48.0 * counters["tri_tests_executed"] if variant == "grid" else 0.0
        hbm_peak = (self.peaks_file or {}).get("hbm_gbs", 6650.0)
        out_bytes = W * H * 4 / world
        roof = {"bound": "fp32", "achieved": executed, "peak": fp32_peak, "unit": "TFLOP/s", "frac": executed / fp32_peak, "traffic": None,
                "flops_per_ray": F, "algorithmic_tflops": algorithmic, "algorithmic_frac": algorithmic / fp32_peak,
                "issue_frac": None, "issue_peak_gwarp_inst_per_s": issue_peak,
                "note": "achieved = EXECUTED flop/s from the device counters (analytic tests of every ray + 58 per triangle test that ran "
                        "after the conservative culls + 30 per visited grid cell + 22 per non-zero VPL evaluation) / live kernel time; "
                        "algorithmic_* = SURVEY 8d's F_ray x rays (work the reference does, culled or not).  The kernels are issue-slot "
                        "bound, not flop bound: issue_frac = warp instructions per launch (ncu) / live kernel time / measured issue rate",
                "peak_source": "pt_measure_peaks on this GPU in this run: pure-FFMA kernel %.1f TFLOP/s (148 SM x 128 lanes x 2 x %.0f MHz "
                               "= %.1f derived); issue rate %.0f G warp-inst/s from a mixed FFMA+integer kernel"
                               % (fp32_peak, (self.peaks_file or {}).get("sm_max_mhz", 1965.0),
                                  self.props["sm_count"] * 128 * 2 * (self.peaks_file or {}).get("sm_max_mhz", 1965.0) * 1e6 / 1e12, issue_peak),
                "grid_gather_gbs": grid_bytes / (kernel_ms * 1e-3) / 1e9,
                "hbm_achieved_gbs": out_bytes / (kernel_ms * 1e-3) / 1e9, "hbm_peak_gbs": hbm_peak,
                "hbm_peak_source": "MEASURED_PEAKS.json (measured)" if self.peaks_file else "fallback 6650 GB/s"}
        ncu = self.ncu.get(wname)
        if ncu and world == 1:
            roof["traffic"] = ncu.get("dram_bytes_read", 0) + ncu.get("dram_bytes_write", 0)
            roof["ncu"] = ncu
            if ncu.get("warp_instructions"):
                roof["issue_frac"] = ncu["warp_instructions"] / (kernel_ms * 1e-3) / 1e9 / issue_peak
        line = {
            "metric": "Mrays/s", "value": rays / 1e3 / ms_per_step, "unit": "Mrays/s", "n_gpus": world, "steps": len(step_ms),
            "warmup": warm, "ms_per_step": ms_per_step, "step_ms": [round(x, 4) for x in step_ms], "higher_is_better": True,
            "scaling": ("strong" if strong else "weak") if world > 1 else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(w, wname, W, H, spp), kernel=args.kernel, kernel_resolved=resolved_kernel, scene_mem=args.scene_mem or "auto",
                           arith="fma (bit-exact vs oracle -DPT_CONTRACT=1)", l2="flushed between timed steps (256 MiB write)",
                           sharding=(("sample blocks (spp/N samples of every pixel per rank, re-seeded streams) + one NCCL reduce" if by_samples
                                      else "8-row stripes round-robin over ranks + one NCCL reduce of the float accumulation buffer")
                                     if world > 1 else "single GPU")),
            "msamples_per_s": samples / 1e3 / ms_per_step, "rays_per_step": rays, "samples_per_step": samples,
            "rays_traced_per_step": rays_traced,
            "ray_count": ("rays_per_step = TraceRay calls of the REFERENCE for this frame (device counters of a TRACE-mode launch; equal to "
                          "the oracle's count) — the unit of `value`, `e2e` and of the reference arm; rays_traced_per_step = rays the timed "
                          "launch really traced: dead_rays=%s %s" % (args.dead_rays, "(shadow rays of triangle-material samples, whose result "
                          "the reference never uses, are not traced; same image / accumulation / RNG bits)" if args.dead_rays != "trace" else "")),
            "e2e": {"value": rays / 1e3 / e2e_ms, "unit": "Mrays/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "api": e2e_api},
            "gpu_launches": steps * ((launches_per_render + (2 if bidir else 0)) * world + (1 if world > 1 else 0)),
            "parity_check": parity,
            "roofline": roof,
        }
        if clocks is not None:
            line["clocks"] = clocks
        if per_rank:
            line["per_rank"] = per_rank
        if vpl_info:
            line["vpl"] = vpl_info
        if world == 1 and cpu_baseline and not args.no_cpu_baseline:
            try:
                m = cpu_reference_measure(w, d, W, H, spp, budget_s=args.cpu_budget)
                line["cpu_baseline"] = {"value": m["mrays"], "unit": "Mrays/s", "cores": m["cores"], "kind": m["kind"],
                                        "ms": m["ms"], "sample": m["sample"]}
                ocl = reference_opencl_on_gpu(w, d, W, H, rays)
                if ocl:
                    line["reference_opencl_same_gpu"] = ocl
            except Exception as exc:  # pragma: no cover - reporting only
                line["cpu_baseline"] = {"error": str(exc)}
        return line


def bench_ours(args, wname, default_workload):
    b = Ours(args)
    line = b.measure(wname, args.steps, args.warmup, headline=True)
    if b.outputs is not None:
        dump_outputs(args.dump_outputs, b.outputs)
    ok = True
    if b.rank == 0:
        if b.world == 1 and default_workload and not args.no_extras:
            extras = {}
            for name in EXTRA_N1:
                heavy = WORKLOADS[name]["W"] * WORKLOADS[name]["H"] * WORKLOADS[name]["spp"] > 1 << 26
                sub = b.measure(name, min(args.steps, 5 if heavy else 50), 3, headline=False)
                keep = ("value", "unit", "ms_per_step", "steps", "msamples_per_s", "rays_per_step", "rays_traced_per_step", "samples_per_step", "e2e", "parity_check",
                        "roofline", "cpu_baseline", "reference_opencl_same_gpu", "gpu_launches")
                extras[name] = dict({"baseline_config": WORKLOADS[name]["config"], "description": WORKLOADS[name]["desc"]},
                                    **{k: sub[k] for k in keep if k in sub})
                if sub.get("parity_check") and sub["parity_check"].get("bit_exact") is False:
                    ok = False
            line["configs"] = extras
            if DEFAULT_MULTI in extras:
                # the N > 1 default strong-scales ANOTHER workload (BASELINE config 5) than this line's headline (config 4):
                # its one-GPU point, for whoever computes a scaling efficiency from the per-N lines
                e = extras[DEFAULT_MULTI]
                line["strong_scaling_n1"] = {"workload": DEFAULT_MULTI, "value": e["value"], "unit": e["unit"], "ms_per_step": e["ms_per_step"],
                                             "e2e": e.get("e2e"), "note": "bench.py --gpus N (N > 1) measures this workload; divide its "
                                             "value by N x this one for the strong-scaling efficiency"}
            sct = simple_cpu_tracer_baseline()
            if sct:
                line["simple_cpu_tracer"] = sct
        line["peaks_measured_live"] = b.live
        if line.get("parity_check") and line["parity_check"].get("bit_exact") is False:
            ok = False
        b.emit(line)
    b.close()
    if not ok:
        sys.stderr.write("bench.py: PARITY CHECK FAILED (timed output differs from the oracle / the 1-GPU render)\n")
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps; with --impl reference each step is about --cpu-budget seconds of CPU work")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: %s at N=1 (BASELINE config 4), %s strong-scaled at N>1 (config 5 at 64 of 4096 spp)" % (DEFAULT_N1, DEFAULT_MULTI))
    ap.add_argument("--kernel", default="auto", choices=["auto", "mega", "persistent", "wavefront"])
    ap.add_argument("--scene-mem", default=None, choices=["auto", "const", "smem"])
    ap.add_argument("--dead-rays", default="auto", choices=["auto", "elide", "trace"],
                    help="auto/elide: library default, shadow rays whose result the reference never uses are not traced (same bits); "
                         "trace: every ray of the reference is traced")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N=1 default run: skip the other BASELINE configs")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=8.0, help="seconds of CPU work per sampled CPU measurement")
    ap.add_argument("--shard", default="tiles", choices=["tiles", "samples"],
                    help="N>1: tiles = 8-row stripes (bit-identical to 1 GPU); samples = every rank renders a block of each pixel's "
                         "samples (throughput mode, statistically equivalent)")
    ap.add_argument("--strong", action="store_true", help="(default at N>1) keep the image fixed as N grows")
    ap.add_argument("--weak", action="store_true", help="N>1: grow the image with N (512 x 512N style) instead of strong scaling")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm times CPU rows, not a frame")
    world = max(1, args.gpus, int(os.environ.get("WORLD_SIZE", "1")))
    default_workload = args.workload is None
    wname = args.workload or (DEFAULT_N1 if world == 1 else DEFAULT_MULTI)
    if args.impl == "reference":
        # the CPU arm must use every host core whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1)
        os.environ["OMP_NUM_THREADS"] = str(host_cores())
        args.warmup = min(args.warmup, 1)
        bench_reference(args, WORKLOADS[wname], wname)
    else:
        bench_ours(args, wname, default_workload)


if __name__ == "__main__":
    main()
