/*
 * pthost_cli.c — the drop-in command-line programs.  One driver, parameterised by variant, reproduces
 * the argv, the scene files read from the current directory, the stdout lines (in order) and the
 * result.ppm of the reference mains:
 *   CLSuperPathTracer/CLSuperPathTracer.c:186-339            (PT_VARIANT_BASE)
 *   CLSuperPathTracer_lmem/CLSuperPathTracer.c:195-354       (PT_VARIANT_LMEM)
 *   CLSuperPathTracer_lmem_NoDoF/CLSuperPathTracer.c:219-394 (PT_VARIANT_NODOF)
 *   CLSuperPathTracer_trianglegrid/CLSuperPathTracer.c:383-583 (PT_VARIANT_GRID)
 *   CLSuperBidirectionalPathTracer/CLSuperBidirectionalPathTracer.c:245-422 (PT_VARIANT_BIDIR; argv[3] = N_VLP per light)
 * Where the reference talks to OpenCL through ocl_boiler.h, this talks to libptcuda.so (ptcuda.h).
 *
 * Extensions are env-only so the command line stays a drop-in:
 *   PT_SEEDS=a,b,c,d   fixed seeds (default: wall-clock recipe of the reference)
 *   PT_SPP=n           samples per pixel (default 64)
 *   PT_KERNEL=auto|mega|persistent|wavefront|grid_tma|grid_stream|grid_pool|spec|grid_queue|grid_async
 *   PT_SCENE_MEM=auto|const|smem     PT_ARITH=fma|separate
 *   PT_DEAD_RAYS=trace|elide   (read by libptcuda) trace the shadow rays whose result the reference never uses / skip them (default)
 *   PT_NO_CULL=1       run the full brute-force triangle loop for every ray (default: rays whose line misses
 *                      the mesh's bounding sphere skip it; identical results)
 *   PT_MAX_TRIANGLES=n lift the 512 / 65536 MAX_TRIANGLES cap of the reference hosts
 *   PT_DEVICE / OCL_DEVICE   device index
 *   PT_GPUS=n          render on GPUs 0..n-1 of this box (row stripes + one NCCL reduce of the accumulation buffer)
 *   PT_SHARD=samples   with PT_GPUS=n: shard the SAMPLES of every pixel over the GPUs instead of row stripes (throughput
 *                      mode: other RNG streams per block, statistically equivalent image, not bit-identical)
 *   PT_BOUNCES=n       base, lmem and trianglegrid: n (0..15) diffuse bounces per path with Russian roulette (include/ptcuda.h
 *                      pt_set_bounces, DESIGN.md 5b; also with PT_GPUS=n).  Default 0: the reference's image
 *   PT_NO_WARMUP=1     skip the untimed one-row warm-up launch
 *   PT_EXTRA_OUTPUT=png,ppm   additionally write result.png (RGBA PNG) and/or result_p6.ppm (binary P6) next to result.ppm
 *   PT_STATS=1         append Mrays/s, samples/s and work counters after the reference's own lines
 */
#define _GNU_SOURCE
#include <dlfcn.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "pthost.h"

/* PT_TIMING=1: wall-clock of the host-side phases on stderr (stdout stays the reference's) */
static double g_t0, g_tlast;
static double wall_ms(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec / 1e6;
}
static void tick(const char *what) {
    if (!getenv("PT_TIMING")) return;
    const double now = wall_ms();
    fprintf(stderr, "PT_TIMING %-28s %9.1f ms  (at %9.1f ms)\n", what, now - g_tlast, now - g_t0);
    g_tlast = now;
}

/* CUDA initialisation (1.3 s per device, 8 devices + the NCCL communicators several seconds) does not depend on the scene:
 * it runs on a helper thread while the main thread prints and parses triangles.txt. */
/* The devices this process could see, WITHOUT initialising CUDA: the entries of CUDA_VISIBLE_DEVICES, or (unset) the NVML
 * device count.  cuInit() on an 8-GPU NVSwitch box takes 5.5 s with all eight visible and 1.1 s with one (measured), so the
 * drop-in narrows CUDA_VISIBLE_DEVICES to the devices it is going to use before the first CUDA call.  -1: unknown. */
static int visible_devices(char entries[16][80]) {
    const char *v = getenv("CUDA_VISIBLE_DEVICES");
    int n = 0;
    if (v && v[0]) {
        while (*v && n < 16) {
            size_t len = strcspn(v, ",");
            if (len == 0 || len >= 80) return -1;
            memcpy(entries[n], v, len);
            entries[n][len] = 0;
            ++n;
            v += len;
            if (*v == ',') ++v;
        }
        return *v ? -1 : n;
    }
    void *nvml = dlopen("libnvidia-ml.so.1", RTLD_NOW);
    if (!nvml) return -1;
    int (*init)(void) = (int (*)(void))dlsym(nvml, "nvmlInit_v2");
    int (*count)(unsigned *) = (int (*)(unsigned *))dlsym(nvml, "nvmlDeviceGetCount_v2");
    int (*shutdown)(void) = (int (*)(void))dlsym(nvml, "nvmlShutdown");
    unsigned c = 0;
    if (init && count && init() == 0) {
        if (count(&c) != 0) c = 0;
        if (shutdown) shutdown();
    }
    dlclose(nvml);
    if (c == 0 || c > 16) return -1;
    for (unsigned i = 0; i < c; ++i) snprintf(entries[i], 80, "%u", i);
    return (int)c;
}

struct create_job {
    int ngpus;
    int total_devices, public_dev;   /* what the reference's lines report: all visible devices, the index the user selected */
    int dev_count, dev, query_rc;
    char dev_name[256];
    int info_ready;
    pthread_mutex_t lock;
    pthread_cond_t cond;
    pt_multi multi;
    pt_ctx ctx;
};
static void *create_worker(void *arg) {
    struct create_job *j = (struct create_job *)arg;
    int count = 0, dev = 0;
    int rc = pt_query_device(&count, &dev, j->dev_name, sizeof(j->dev_name));
    if (j->total_devices > 0) {          /* CUDA_VISIBLE_DEVICES was narrowed: report the devices as the user sees them */
        if (!rc && count < 1) rc = 1;
        count = j->total_devices;
        dev = j->public_dev;
    }
    pthread_mutex_lock(&j->lock);
    j->dev_count = count; j->dev = dev; j->query_rc = rc; j->info_ready = 1;
    pthread_cond_signal(&j->cond);
    pthread_mutex_unlock(&j->lock);
    if (rc || dev < 0 || dev >= count) return NULL;            /* the main thread reports it, as select_device does */
    if (j->ngpus > 1) j->multi = pt_multi_create(j->ngpus);
    else j->ctx = pt_create(j->total_devices > 0 ? 0 : dev);
    return NULL;
}

static int env_choice(const char *name, const char *const *opts, int nopts, int dflt) {
    const char *v = getenv(name);
    if (!v || !v[0]) return dflt;
    for (int i = 0; i < nopts; ++i)
        if (!strcmp(v, opts[i])) return i;
    fprintf(stderr, "%s=%s not understood\n", name, v);
    exit(1);
}

int pth_cli_main(int variant, int argc, char **argv) {
    g_t0 = g_tlast = wall_ms();
    int img_width = 512, img_height = 512;
    float cell_size_modifier = 3.0f;
    const int grid = variant == PT_VARIANT_GRID, nodof = variant == PT_VARIANT_NODOF, bidir = variant == PT_VARIANT_BIDIR;
    const int samples_per_pixel_nodof = 64;
    int n_vlp = 512;

    if (grid)
        printf("Usage: %s [img_width] [img_height] [CELL_SIZE_MODIFIER]\nLoads data from triangles.txt, lights.txt, spheres.txt and squares.txt\n", argv[0]);
    else if (nodof)
        printf("Usage: %s [img_width] [img_height]\nLoads data from triangles.txt, lights.txt, spheres.txt and planes.txt", argv[0]);
    else if (bidir)
        printf("Usage: %s [img_width] [img_height] [N_VLP_per_light]\nLoads data from triangles.txt, lights.txt, spheres.txt and squares.txt\n", argv[0]);
    else
        printf("Usage: %s [img_width] [img_height]\nLoads data from triangles.txt, lights.txt, spheres.txt and squares.txt\n", argv[0]);
    if (argc > 1) img_width = atoi(argv[1]);
    if (argc > 2) img_height = atoi(argv[2]);
    if (grid && argc > 3) cell_size_modifier = (float)atof(argv[3]);
    if (bidir && argc > 3) n_vlp = atoi(argv[3]);

    /* select_platform / select_device / create_* of ocl_boiler.h: on a helper thread, started before anything else */
    const int ngpus = getenv("PT_GPUS") ? atoi(getenv("PT_GPUS")) : 1;
    struct create_job job;
    memset(&job, 0, sizeof(job));
    job.ngpus = ngpus;
    {
        char entries[16][80];
        const int total = visible_devices(entries);
        const char *denv = getenv("PT_DEVICE");
        if (!denv || !denv[0]) denv = getenv("OCL_DEVICE");
        const int want = (denv && denv[0]) ? atoi(denv) : 0;
        char narrowed[16 * 81] = "";
        if (total > 1 && ngpus > 1 && ngpus < total) {
            for (int i = 0; i < ngpus; ++i) { if (i) strcat(narrowed, ","); strcat(narrowed, entries[i]); }
            job.total_devices = total; job.public_dev = want;
        } else if (total > 1 && ngpus <= 1 && want >= 0 && want < total) {
            strcpy(narrowed, entries[want]);
            job.total_devices = total; job.public_dev = want;
        }
        if (narrowed[0]) {
            setenv("CUDA_VISIBLE_DEVICES", narrowed, 1);
            setenv("PT_DEVICE", "0", 1);                 /* inside the narrowed set */
        }
    }
    pthread_mutex_init(&job.lock, NULL);
    pthread_cond_init(&job.cond, NULL);
    pthread_t creator;
    const int threaded = pthread_create(&creator, NULL, create_worker, &job) == 0;
    if (!threaded) create_worker(&job);

    /* ... while this thread already reads triangles.txt (a million triangles are 13.6 M text lines); what the reference
     * prints about them comes later, in its order */
    int max_triangles = grid ? 65536 : 512;     /* MAX_TRIANGLES of the respective host */
    if (getenv("PT_MAX_TRIANGLES")) max_triangles = atoi(getenv("PT_MAX_TRIANGLES"));
    float *tris = NULL;
    float box_min[4], box_max[4];
    const int ntriangles_parsed = pth_parse_triangles("triangles.txt", max_triangles, &tris, box_min, box_max);
    tick("parse triangles.txt");

    pthread_mutex_lock(&job.lock);
    while (!job.info_ready) pthread_cond_wait(&job.cond, &job.lock);
    pthread_mutex_unlock(&job.lock);
    printf("number of platforms: %u\n", 1u);
    printf("selected platform %d: %s\n", 0, "NVIDIA CUDA (libptcuda, sm_100a)");
    if (job.query_rc) pt_check(job.query_rc, "counting devices");
    printf("number of devices: %u\n", (unsigned)job.dev_count);
    if (job.dev < 0 || job.dev >= job.dev_count) {
        fprintf(stderr, "no device number %u", (unsigned)job.dev);
        exit(1);
    }
    printf("selected device %d: %s\n", job.dev, job.dev_name);
    tick("device query");
    time_t now = time(NULL);
    printf("compiling:\n// %s#include \"%s\"\n", ctime(&now), bidir ? "bidirectionalpathtracer.ocl" : "pathtracer.ocl");
    printf("=== BUILD LOG ===\n%s\n=========\n", "kernels are precompiled CUDA for sm_100a (libptcuda.so); nothing to build\n");

    uint32_t seeds[4];
    pth_seeds(seeds);
    printf("Seeds: %d, %d, %d, %d\n", (int)seeds[0], (int)seeds[1], (int)seeds[2], (int)seeds[3]);

    long data_size = (long)img_width * img_height * 4;
    printf("Processing image %dx%d with data size %ld bytes\n", img_width, img_height, data_size);

    pt_camera cam;
    pth_camera(&cam);
    printf(grid ? "Cam values:\nCam_forward %f %f %f\nCam_up %f %f %f\nCam_right %f %f %f\neye_offset %f %f %f\n"
                : "Cam values:\nCam_forward %f %f %f\nCam_up %f %f %f\nCam_right %f %f %f\n eye_offset %f %f %f\n",
           cam.cam_forward[0], cam.cam_forward[1], cam.cam_forward[2], cam.cam_up[0], cam.cam_up[1], cam.cam_up[2],
           cam.cam_right[0], cam.cam_right[1], cam.cam_right[2], cam.eye_offset[0], cam.eye_offset[1], cam.eye_offset[2]);

    pt_scene scene;
    memset(&scene, 0, sizeof(scene));
    if (pth_parse_bitmap("spheres.txt", scene.spheres) < 0) pt_check(1, "open spheres.txt");
    const char *squares_file = "squares.txt";
    if (nodof) {
        /* the NoDoF host opens planes.txt, which its directory does not ship; accept either name */
        FILE *probe = fopen("planes.txt", "r");
        if (probe) { fclose(probe); squares_file = "planes.txt"; }
    }
    if (pth_parse_bitmap(squares_file, scene.squares) < 0) pt_check(1, "open %s", squares_file);

    pt_grid gdesc;
    memset(&gdesc, 0, sizeof(gdesc));
    scene.ntriangles = ntriangles_parsed;
    if (scene.ntriangles < 0) pt_check(1, "open triangles.txt");
    scene.triangles = tris;
    if (grid) {
        printf("Triangles bounding box values:\nvmax: %f %f %f, vmin: %f %f %f\n", box_max[0], box_max[1], box_max[2],
               box_min[0], box_min[1], box_min[2]);
        pth_grid_dims(box_min, box_max, scene.ntriangles, cell_size_modifier, &gdesc);
        printf("Triangles grid size: %d x %d x %d\n", gdesc.res[0], gdesc.res[1], gdesc.res[2]);
    }
    scene.nlights = pth_parse_lights("lights.txt", scene.lights, variant != PT_VARIANT_BASE && !bidir);   /* base and bidir do not echo the lights */
    if (scene.nlights < 0) pt_check(1, "open lights.txt");
    printf("Number of triangles: %d\n", scene.ntriangles);
    printf("Number of lights: %d\n", scene.nlights);

    if (threaded) pthread_join(creator, NULL);
    pt_multi multi = job.multi;
    pt_ctx ctx = job.ctx;
    if (ngpus > 1 ? !multi : !ctx) pt_check(1, "create the CUDA context(s)");
    tick("wait for the context(s)");
    if (multi) pt_multi_set_scene(multi, &scene); else pt_set_scene(ctx, &scene);
    tick("upload scene");
    pt_event grid_evt = NULL;
    if (grid) grid_evt = multi ? pt_multi_build_grid(multi, &gdesc) : pt_build_grid(ctx, &gdesc);
    tick("build grid (enqueue)");

    static const char *const kernels[] = {"mega", "persistent", "wavefront", "auto", "grid_tma", "grid_stream", "grid_pool", "spec", "grid_queue", "grid_async"};
    static const char *const mems[] = {"const", "smem", "auto"};
    static const char *const ariths[] = {"separate", "fma"};
    pt_render_params rp;
    memset(&rp, 0, sizeof(rp));
    rp.variant = variant;
    rp.width = img_width;
    rp.height = img_height;
    rp.spp = getenv("PT_SPP") ? atoi(getenv("PT_SPP")) : 64;
    memcpy(rp.seeds, seeds, sizeof(seeds));
    rp.kernel = env_choice("PT_KERNEL", kernels, 10, PT_KERNEL_AUTO);
    rp.scene_mem = env_choice("PT_SCENE_MEM", mems, 3, PT_SCENE_AUTO);
    rp.arith = env_choice("PT_ARITH", ariths, 2, PT_ARITH_FMA);
    rp.no_cull = getenv("PT_NO_CULL") ? atoi(getenv("PT_NO_CULL")) : 0;
    if (!nodof && !bidir && getenv("PT_BOUNCES")) {       /* diffuse bounces per path (0..15, DESIGN.md 5b) */
        const int nb = atoi(getenv("PT_BOUNCES"));
        pt_check(multi ? pt_multi_set_bounces(multi, nb) : pt_set_bounces(ctx, nb), "PT_BOUNCES=%s", getenv("PT_BOUNCES"));
    }
    if (multi && getenv("PT_SHARD") && !strcmp(getenv("PT_SHARD"), "samples")) rp.sample_blocks = ngpus;

    pt_event light_evt = NULL;
    if (bidir && !getenv("PT_NO_WARMUP")) {     /* untimed first light pass (lazy module load), also feeds the warm-up render */
        pt_event w = multi ? pt_multi_launch_lighttracer(multi, n_vlp, seeds, rp.arith) : pt_launch_lighttracer(ctx, n_vlp, seeds, rp.arith);
        pt_wait(w);
        pt_release_event(w);
    } else if (bidir)
        light_evt = multi ? pt_multi_launch_lighttracer(multi, n_vlp, seeds, rp.arith) : pt_launch_lighttracer(ctx, n_vlp, seeds, rp.arith);
    if (!getenv("PT_NO_WARMUP")) {
        /* One untimed single-row launch first: CUDA loads kernel code lazily (and NCCL sets up its rings) on first
         * use, which the reference's OpenCL event times never include (its JIT runs in clBuildProgram). */
        pt_render_params warm = rp;
        warm.row_begin = 0;
        warm.row_end = 1;
        pt_event w = multi ? pt_multi_launch_pathtracer(multi, &cam, &warm) : pt_launch_pathtracer(ctx, &cam, &warm);
        pt_wait(w);
        pt_release_event(w);
    }
    tick("warm-up launch");
    if (bidir && !light_evt)
        light_evt = multi ? pt_multi_launch_lighttracer(multi, n_vlp, seeds, rp.arith) : pt_launch_lighttracer(ctx, n_vlp, seeds, rp.arith);
    pt_event render_evt = multi ? pt_multi_launch_pathtracer(multi, &cam, &rp) : pt_launch_pathtracer(ctx, &cam, &rp);
    pt_event read_evt = NULL;
    void *pixels = multi ? pt_multi_map_render(multi, &read_evt) : pt_map_render(ctx, &read_evt);
    tick("render + read back");

    const char *image_name = "result.ppm";
    if (pth_save_pam(image_name, img_width, img_height, pixels) != 0) {
        fprintf(stderr, "error writing %s\n", image_name);
        exit(1);
    } else
        printf("\nSuccessfully created render image %s in the current directory\n\n", image_name);
    const char *extra = getenv("PT_EXTRA_OUTPUT");
    if (extra && strstr(extra, "png") && pth_save_png("result.png", img_width, img_height, pixels)) pt_check(1, "write result.png");
    if (extra && strstr(extra, "ppm") && pth_save_ppm("result_p6.ppm", img_width, img_height, pixels)) pt_check(1, "write result_p6.ppm");

    tick("write image");
    double render_ms = pt_runtime_ms(render_evt), read_ms = pt_runtime_ms(read_evt), light_ms = 0.0;
    if (bidir) {
        light_ms = pt_runtime_ms(light_evt);
        printf("virtual light sampling : %d virtual lights in %gms: %g GB/s\n", n_vlp * scene.nlights, light_ms,
               n_vlp * scene.nlights * 16 / 1.0e6 / light_ms);
    }
    if (grid) {
        double grid_ms = pt_runtime_ms(grid_evt);
        size_t grid_bytes = (size_t)128 * gdesc.res[0] * gdesc.res[1] * gdesc.res[2];
        printf("init triangles grid : %d cells in %gms: %g GB/s\n", gdesc.res[0] * gdesc.res[1] * gdesc.res[2], grid_ms,
               grid_bytes / 1.0e6 / grid_ms);
    }
    if (nodof) {
        /* the reduction is fused into the render kernel: its separate time is 0 */
        printf("rendering : %d pixels (with %d samples) in %gms: %g GB/s\n", img_width * img_height, samples_per_pixel_nodof,
               render_ms, data_size * samples_per_pixel_nodof * sizeof(float) / 1.0e6 / render_ms);
        printf("reduce img samples : %d pixels (with %d samples) in %gms: %g GB/s\n", img_width * img_height,
               samples_per_pixel_nodof, 0.0, data_size / 1.0e6 / render_ms);
    } else
        printf("rendering : %d pixels in %gms: %g GB/s\n", img_width * img_height, render_ms, data_size / 1.0e6 / render_ms);
    printf("read render data : %ld uchar in %gms: %g GB/s\n", data_size, read_ms, data_size / 1.0e6 / read_ms);
    printf("\nTotal time: %g ms.\n", light_ms + render_ms + read_ms);

    if (getenv("PT_STATS")) {
        pt_counters c;
        if (multi) pt_multi_get_counters(multi, &c); else pt_get_counters(ctx, &c);
        printf("PT_STATS {\"variant\": %d, \"width\": %d, \"height\": %d, \"spp\": %d, \"kernel\": \"%s\", \"scene_mem\": \"%s\", "
               "\"arith\": \"%s\", \"gpus\": %d, \"render_ms\": %.6f, \"samples\": %llu, \"rays\": %llu, \"shadow_rays\": %llu, "
               "\"tri_tests\": %llu, \"cells_visited\": %llu, \"prim_tests\": %llu, \"mrays_per_s\": %.3f, \"msamples_per_s\": %.3f}\n",
               variant, img_width, img_height, rp.spp, kernels[rp.kernel], mems[rp.scene_mem], ariths[rp.arith], ngpus, render_ms,
               (unsigned long long)c.samples, (unsigned long long)c.rays, (unsigned long long)c.shadow_rays,
               (unsigned long long)c.tri_tests, (unsigned long long)c.cells_visited, (unsigned long long)c.prim_tests,
               c.rays / 1.0e3 / render_ms, c.samples / 1.0e3 / render_ms);
    }

    pt_release_event(render_evt);
    pt_release_event(read_evt);
    pt_release_event(grid_evt);
    pt_release_event(light_evt);
    free(tris);
    if (!getenv("PT_CLEAN_EXIT")) {
        /* everything is written: leave without tearing the CUDA contexts and NCCL communicators down one by one (1.2 s of
         * pt_multi_destroy plus ~2 s of driver teardown at 8 GPUs); the driver reclaims them with the process */
        tick("done");
        fflush(NULL);
        _exit(0);
    }
    if (multi) pt_multi_destroy(multi); else pt_destroy(ctx);
    tick("destroy");
    return 0;
}
