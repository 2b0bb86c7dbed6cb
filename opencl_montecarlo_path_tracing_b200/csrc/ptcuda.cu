// ptcuda.cu — implementation of the C ABI declared in include/ptcuda.h (libptcuda.so).
//
// One translation unit on purpose: the kernels share one __constant__ scene block.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 (see csrc/Makefile).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <dlfcn.h>

#include <atomic>
#include <mutex>
#include <thread>
#include <vector>
#include <new>
#include <string>

#include "pt_host.h"
#include "pt_mega.cuh"
#include "pt_persistent.cuh"
#include "pt_wavefront.cuh"
#include "pt_gridbuild.cuh"
#include "pt_gridtma.cuh"
#include "pt_bidir.cuh"
#include "pt_gridstream.cuh"
#include "pt_gridpool.cuh"
#include "pt_spec.cuh"
#include "pt_gridqueue.cuh"
#include "pt_gridasync.cuh"
#include "pt_metropolis.cuh"
#include "pt_bounce.cuh"

// ------------------------------------------------------------------------------------ errors
static std::atomic<int> g_error_mode{PT_ERRORS_EXIT};
static thread_local char g_last_error[1024] = "";

extern "C" void pt_set_error_mode(int mode) { g_error_mode = mode; }
extern "C" const char *pt_last_error(void) { return g_last_error; }

int pt_fail(int err, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    char msg[900];
    vsnprintf(msg, sizeof(msg), fmt, ap);
    va_end(ap);
    snprintf(g_last_error, sizeof(g_last_error), "%s - error %d", msg, err);
    if (g_error_mode == PT_ERRORS_EXIT) {
        fprintf(stderr, "%s\n", g_last_error);
        exit(1);
    }
    return err ? err : 1;
}

int pt_cuda_fail(cudaError_t e, const char *what) {
    return pt_fail((int)e, "%s: %s", what, cudaGetErrorString(e));
}

extern "C" void pt_check(int err, const char *fmt, ...) {
    if (err == 0) return;
    va_list ap;
    va_start(ap, fmt);
    char msg[900];
    vsnprintf(msg, sizeof(msg), fmt, ap);
    va_end(ap);
    fprintf(stderr, "%s - error %d\n", msg, err);
    exit(1);
}

// --------------------------------------------------------------------------- device / context
extern "C" int pt_abi_version(void) { return PTCUDA_ABI_VERSION; }

extern "C" int pt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

// select_device of ocl_boiler.h without the printing: number of devices, the index PT_DEVICE / OCL_DEVICE selects (not
// range-checked) and that device's name.  Lets a host start CUDA on a helper thread and print when it is ready.
extern "C" int pt_query_device(int *count, int *selected, char *name, size_t name_len) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return pt_cuda_fail(e, "counting devices");
    const char *env = getenv("PT_DEVICE");
    if (!env || !env[0]) env = getenv("OCL_DEVICE");
    const int d = (env && env[0]) ? atoi(env) : 0;
    if (count) *count = n;
    if (selected) *selected = d;
    if (name && name_len) {
        name[0] = 0;
        if (d >= 0 && d < n) {
            cudaDeviceProp prop;
            e = cudaGetDeviceProperties(&prop, d);
            if (e != cudaSuccess) return pt_cuda_fail(e, "device name");
            snprintf(name, name_len, "%s", prop.name);
        }
    }
    return 0;
}

extern "C" int pt_select_device(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return -pt_cuda_fail(e, "counting devices");
    printf("number of devices: %u\n", (unsigned)n);
    const char *env = getenv("PT_DEVICE");
    if (!env || !env[0]) env = getenv("OCL_DEVICE");
    int d = (env && env[0]) ? atoi(env) : 0;
    if (d < 0 || d >= n) {
        fprintf(stderr, "no device number %u", (unsigned)d);
        exit(1);
    }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, d);
    if (e != cudaSuccess) return -pt_cuda_fail(e, "device name");
    printf("selected device %d: %s\n", d, prop.name);
    return d;
}

static pt_ctx ctx_new(int device, cudaStream_t stream, bool own) {
    pt_ctx c = (pt_ctx)calloc(1, sizeof(pt_ctx_s));
    c->device = device;
    c->stream = stream;
    c->own_stream = own;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
        c->sm_count = prop.multiProcessorCount;
        c->clock_khz = prop.clockRate;
        snprintf(c->name, sizeof(c->name), "%s", prop.name);
    }
    return c;
}

extern "C" pt_ctx pt_create(int device) {
    PT_CUDA_NULL(cudaSetDevice(device), "select device");
    cudaStream_t s;
    PT_CUDA_NULL(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking), "create stream");
    pt_ctx c = ctx_new(device, s, true);
    PT_CUDA_NULL(cudaMalloc(&c->d_counters, 8 * sizeof(unsigned long long)), "alloc counters");
    return c;
}

extern "C" pt_ctx pt_create_on_stream(int device, void *cuda_stream) {
    PT_CUDA_NULL(cudaSetDevice(device), "select device");
    pt_ctx c = ctx_new(device, (cudaStream_t)cuda_stream, false);
    PT_CUDA_NULL(cudaMalloc(&c->d_counters, 8 * sizeof(unsigned long long)), "alloc counters");
    return c;
}

struct ConstOwner { pt_ctx owner; uint64_t version; int arith; };
static ConstOwner g_const_owner[64];
// The __constant__ scene block is ONE per device, shared by every context on it.  Rebinding it and the launch that reads it
// must not interleave with another host thread doing the same for a different context on that device: both happen under
// this per-device lock (dispatch(), pt_probe_trace, pt_launch_lighttracer), and a change of owner first drains the device.
static std::recursive_mutex g_dev_lock[64];
struct DevLock {
    std::unique_lock<std::recursive_mutex> lk;
    explicit DevLock(int device) { if (device >= 0 && device < 64) lk = std::unique_lock<std::recursive_mutex>(g_dev_lock[device]); }
};
static std::atomic<uint64_t> g_scene_version{1};

extern "C" void pt_destroy(pt_ctx c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    {
        DevLock lock(c->device);
        if (c->device < 64 && g_const_owner[c->device].owner == c) g_const_owner[c->device].owner = nullptr;
    }
    for (int a = 0; a < 2; ++a) {
        if (c->h_scene[a]) cudaFreeHost(c->h_scene[a]);
        cudaFree(c->d_scene[a]);
    }
    cudaFree(c->d_tris_raw);
    cudaFree(c->d_cells); cudaFree(c->d_cells_pad); cudaFree(c->d_recs); cudaFree(c->d_refs); cudaFree(c->d_cell_start); cudaFree(c->d_sph); cudaFree(c->gb_kmax);
    cudaFree(c->gb_count); cudaFree(c->gb_raw_start); cudaFree(c->gb_cursor); cudaFree(c->gb_bsums); cudaFree(c->gb_raw_refs);
    cudaFree(c->d_rgba); cudaFree(c->d_accum); cudaFree(c->d_rng); cudaFree(c->d_counters); cudaFree(c->d_scratch);
    cudaFree(c->d_tile_order); cudaFree(c->d_cta_times);
    if (c->h_tile_order) cudaFreeHost(c->h_tile_order);
    if (c->h_cta_times) cudaFreeHost(c->h_cta_times);
    cudaFree(c->d_vpls); cudaFree(c->d_vpl_active); cudaFree(c->d_vpl_count); cudaFree(c->d_metro_seed); cudaFree(c->d_metro_mutated);
    cudaFree(c->d_vlp_keys); cudaFree(c->d_vlp_cell_start); cudaFree(c->d_vlp_refs);
    if (c->wf_exec) cudaGraphExecDestroy(c->wf_exec);
    free(c->wf_key_args);
    if (c->h_rgba) cudaFreeHost(c->h_rgba);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    free(c);
}

extern "C" int pt_device_name(pt_ctx c, char *buf, size_t len) {
    snprintf(buf, len, "%s", c->name);
    return 0;
}

extern "C" int pt_device_props(pt_ctx c, int *sm_count, int *clock_khz) {
    if (sm_count) *sm_count = c->sm_count;
    if (clock_khz) *clock_khz = c->clock_khz;
    return 0;
}

int pt_ensure_scratch(pt_ctx c, size_t bytes) {
    if (c->scratch_cap >= bytes) return 0;
    cudaFree(c->d_scratch);
    c->d_scratch = nullptr;
    c->scratch_cap = 0;
    PT_CUDA(cudaMalloc(&c->d_scratch, bytes), "alloc scratch");
    c->scratch_cap = bytes;
    return 0;
}

// -------------------------------------------------------------------------------------- scene
// Host-side float helpers for the per-triangle normal.  They mirror pt::Ar<FMA> operation for
// operation (fmaf / sqrtf / division are correctly rounded on the host as on the device), so the
// stored normal is bit-identical to Normalize(cross(edge0, edge2)) evaluated per hit (base:131).
#pragma STDC FP_CONTRACT OFF
namespace {
struct H3 { float x, y, z; };
inline float h_msub(bool fma, float a, float b, float c, float d) {
    volatile float cd = c * d;
    if (fma) return fmaf(a, b, -cd);
    volatile float ab = a * b;
    return ab - cd;
}
inline float h_madd(bool fma, float a, float b, float c) {
    if (fma) return fmaf(a, b, c);
    volatile float ab = a * b;
    return ab + c;
}
inline H3 h_cross(bool fma, H3 a, H3 b) {
    H3 r = {h_msub(fma, a.y, b.z, a.z, b.y), h_msub(fma, a.z, b.x, a.x, b.z), h_msub(fma, a.x, b.y, a.y, b.x)};
    return r;
}
inline float h_dot(bool fma, H3 a, H3 b) {
    volatile float xx = a.x * b.x;
    return h_madd(fma, a.z, b.z, h_madd(fma, a.y, b.y, xx));
}
inline H3 h_normalize(bool fma, H3 a) {
    volatile float s = 1.0f / sqrtf(h_dot(fma, a, a));
    volatile float x = a.x * s, y = a.y * s, z = a.z * s;
    H3 r = {x, y, z};
    return r;
}
}  // namespace

static void decode_bitmap(const int32_t bm[9], bool sphere, float2 *out, int *n) {
    int c = 0;
    for (int k = 19; k--;)        // reference scan order: k = 18..0, j = 8..0 (base:73-74)
        for (int j = 9; j--;)
            if (bm[j] & (1 << k)) {
                out[c].x = sphere ? (float)(-k) : (float)k;
                out[c].y = sphere ? (float)(-j - 4) : (float)(4 + j);
                ++c;
            }
    *n = c;
}

// Bounding sphere of triangles src[0..n) of `tris` (src == nullptr: triangles 0..n-1) for the conservative line/sphere
// culls (pt_device.cuh, AnalyticParams::mesh_*): the centre of the vertices' box, rounded to float, and the largest distance
// (double) from that FLOAT centre to a vertex, inflated by 1 % + 0.01 and rounded up to a float.  Measuring the radius from
// the stored centre keeps every vertex inside however far the mesh lies from the origin (there half an ulp of the centre
// outgrows the 0.01); the inflation covers the float rounding of the device's line/sphere test.  Non-finite radius: +inf.
static float4 tri_bounding_sphere(const float *tris, const int *src, int n) {
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int k = 0; k < n; ++k)
        for (int v = 0; v < 3; ++v)
            for (int a = 0; a < 3; ++a) {
                const double x = tris[12 * (size_t)(src ? src[k] : k) + 4 * v + a];
                if (x < lo[a]) lo[a] = x;
                if (x > hi[a]) hi[a] = x;
            }
    float ctr[3] = {0.f, 0.f, 0.f};
    if (n > 0) for (int a = 0; a < 3; ++a) ctr[a] = (float)(0.5 * (lo[a] + hi[a]));
    double r2 = 0;
    for (int k = 0; k < n; ++k)
        for (int v = 0; v < 3; ++v) {
            const float *q = tris + 12 * (size_t)(src ? src[k] : k) + 4 * v;
            const double dx = (double)q[0] - ctr[0], dy = (double)q[1] - ctr[1], dz = (double)q[2] - ctr[2];
            const double d2 = dx * dx + dy * dy + dz * dz;
            if (d2 > r2) r2 = d2;
        }
    const double r = sqrt(r2) * 1.01 + 0.01;
    float rf = isfinite(r) ? (float)r : INFINITY;
    if ((double)rf < r) rf = nextafterf(rf, INFINITY);
    return make_float4(ctr[0], ctr[1], ctr[2], rf);
}

extern "C" int pt_set_scene(pt_ctx c, const pt_scene *sc) {
    using namespace pt;
    if (!c || !sc) return pt_fail(1, "pt_set_scene: null argument");
    if (sc->nlights < 0 || sc->nlights > 5) return pt_fail(1, "pt_set_scene: nlights %d out of range [0,5]", sc->nlights);
    if (sc->ntriangles < 0) return pt_fail(1, "pt_set_scene: negative triangle count");
    PT_CUDA(cudaSetDevice(c->device), "select device");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync before scene update");
    for (int a = 0; a < 2; ++a) {
        if (!c->h_scene[a]) PT_CUDA(cudaMallocHost(&c->h_scene[a], sizeof(SceneBlock)), "alloc pinned scene");
        if (!c->d_scene[a]) PT_CUDA(cudaMalloc(&c->d_scene[a], sizeof(SceneBlock)), "alloc device scene");
    }
    const int nbrute = sc->ntriangles < PT_MAX_CONST_TRIS ? sc->ntriangles : PT_MAX_CONST_TRIS;
    int kept = 0;
    int kept_src[PT_MAX_CONST_TRIS];            // source triangle of each kept record
    for (int a = 0; a < 2; ++a) {
        const bool fma = a == PT_ARITH_FMA;
        SceneBlock *S = c->h_scene[a];
        memset(S, 0, sizeof(SceneBlock));
        decode_bitmap(sc->squares, false, S->sq, &S->nsq);
        decode_bitmap(sc->spheres, true, S->sp, &S->nsp);
        S->nlights = sc->nlights;
        for (int l = 0; l < sc->nlights; ++l)
            S->lights[l] = make_float4(sc->lights[l][0], sc->lights[l][1], sc->lights[l][2], sc->lights[l][3]);
        S->ntri_counted = nbrute;
        kept = 0;
        for (int i = 0; i < nbrute; ++i) {
            const float *t = sc->triangles + 12 * (size_t)i;
            volatile float e0x = t[4] - t[0], e0y = t[5] - t[1], e0z = t[6] - t[2];
            volatile float e2x = t[8] - t[0], e2y = t[9] - t[1], e2z = t[10] - t[2];
            // |det| = |e0 . (d x e2)| <= |e0||e2||d| with |d| = 1: a triangle whose edge-length product is
            // below half the 0.01 cull threshold (base:118) can never pass it, for any ray — skip it.
            double l0 = sqrt((double)e0x * e0x + (double)e0y * e0y + (double)e0z * e0z);
            double l2 = sqrt((double)e2x * e2x + (double)e2y * e2y + (double)e2z * e2z);
            if (l0 * l2 < 0.005) continue;
            H3 e0 = {e0x, e0y, e0z}, e2 = {e2x, e2y, e2z};
            H3 n = h_normalize(fma, h_cross(fma, e0, e2));
            S->tri[3 * kept + 0] = make_float4(e2.x, e2.y, e2.z, e0.x);
            S->tri[3 * kept + 1] = make_float4(e0.y, e0.z, t[0], t[1]);
            S->tri[3 * kept + 2] = make_float4(t[2], n.x, n.y, n.z);
            kept_src[kept] = i;
            ++kept;
        }
        S->ntri = kept;
        // bounding sphere of every cluster of PT_CLUSTER consecutive records, built like the whole-mesh sphere below
        S->ncl = (kept + PT_CLUSTER - 1) / PT_CLUSTER;
        for (int cl = 0; cl < S->ncl; ++cl) {
            const int k0 = cl * PT_CLUSTER, k1 = k0 + PT_CLUSTER < kept ? k0 + PT_CLUSTER : kept;
            S->csph[cl] = tri_bounding_sphere(sc->triangles, kept_src + k0, k1 - k0);
        }
    }
    c->scene_bytes = (int)(offsetof(SceneBlock, tri) + (size_t)kept * 48);
    {
        // bounding sphere of the brute-force triangles' vertices
        const float4 sph = tri_bounding_sphere(sc->triangles, nullptr, nbrute);
        double kmax = 0;     // max |e0||e2| over the brute-force triangles
        for (int i = 0; i < nbrute; ++i) {
            const float *t = sc->triangles + 12 * (size_t)i;
            double e0 = sqrt(pow((double)t[4] - t[0], 2) + pow((double)t[5] - t[1], 2) + pow((double)t[6] - t[2], 2));
            double e2 = sqrt(pow((double)t[8] - t[0], 2) + pow((double)t[9] - t[1], 2) + pow((double)t[10] - t[2], 2));
            if (e0 * e2 > kmax) kmax = e0 * e2;
        }
        c->mesh_c[0] = sph.x; c->mesh_c[1] = sph.y; c->mesh_c[2] = sph.z;
        c->mesh_r = sph.w;
        c->mesh_k = (float)(2e-4 * kmax + 1e-6);
        if (!isfinite(c->mesh_r) || !isfinite(c->mesh_k)) c->mesh_r = INFINITY;
    }
    for (int a = 0; a < 2; ++a)      // only the used prefix of the block travels (header + primitives + kept triangles)
        PT_CUDA(cudaMemcpyAsync(c->d_scene[a], c->h_scene[a], (size_t)c->scene_bytes, cudaMemcpyHostToDevice, c->stream),
                "upload scene");
    c->ntri_total = sc->ntriangles;
    if ((size_t)sc->ntriangles > c->tris_cap) {       // the raw triangle buffer is reused across scene updates
        cudaFree(c->d_tris_raw);
        c->d_tris_raw = nullptr;
        c->tris_cap = 0;
        PT_CUDA(cudaMalloc(&c->d_tris_raw, (size_t)sc->ntriangles * 48), "alloc triangles");
        c->tris_cap = (size_t)sc->ntriangles;
    }
    if (sc->ntriangles > 0)
        PT_CUDA(cudaMemcpyAsync(c->d_tris_raw, sc->triangles, (size_t)sc->ntriangles * 48, cudaMemcpyHostToDevice, c->stream),
                "upload triangles");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync scene upload");
    c->scene_set = true;
    c->grid_set = false;
    c->scene_version = g_scene_version.fetch_add(1);
    return 0;
}

int pt_bind_const_scene(pt_ctx c, int arith) {
    if (c->device >= 64) return pt_fail(1, "device index too large");
    DevLock lock(c->device);
    ConstOwner &o = g_const_owner[c->device];
    if (o.owner == c && o.version == c->scene_version && o.arith == arith) return 0;
    if (o.owner && o.owner != c) PT_CUDA(cudaDeviceSynchronize(), "sync before rebinding constant scene");
    PT_CUDA(cudaMemcpyToSymbolAsync(pt::c_scene, c->h_scene[arith], (size_t)c->scene_bytes, 0, cudaMemcpyHostToDevice, c->stream),
            "upload constant scene");
    o.owner = c;
    o.version = c->scene_version;
    o.arith = arith;
    return 0;
}

// --------------------------------------------------------------------------------------- events
static pt_event event_new(pt_ctx c) {
    pt_event e = (pt_event)calloc(1, sizeof(pt_event_s));
    e->device = c->device;
    if (cudaEventCreate(&e->start) != cudaSuccess || cudaEventCreate(&e->stop) != cudaSuccess) {
        pt_fail(1, "create events");
        free(e);
        return nullptr;
    }
    return e;
}

extern "C" int pt_wait(pt_event e) {
    if (!e) return 1;
    PT_CUDA(cudaEventSynchronize(e->stop), "wait event");
    return 0;
}

extern "C" double pt_runtime_ms(pt_event e) {
    if (!e) return 0.0;
    float ms = 0.f;
    if (cudaEventSynchronize(e->stop) != cudaSuccess) return -1.0;
    if (cudaEventElapsedTime(&ms, e->start, e->stop) != cudaSuccess) return -1.0;
    return (double)ms;
}

extern "C" void pt_release_event(pt_event e) {
    if (!e) return;
    cudaEventDestroy(e->start);
    cudaEventDestroy(e->stop);
    free(e);
}

extern "C" int pt_synchronize(pt_ctx c) {
    PT_CUDA(cudaStreamSynchronize(c->stream), "synchronize");
    return 0;
}

// ----------------------------------------------------------------------------------------- grid
extern "C" pt_event pt_build_grid(pt_ctx c, const pt_grid *g) {
    if (!c || !g) { pt_fail(1, "pt_build_grid: null argument"); return nullptr; }
    if (!c->scene_set) { pt_fail(1, "pt_build_grid: call pt_set_scene first"); return nullptr; }
    for (int a = 0; a < 3; ++a)
        if (g->res[a] < 1 || g->res[a] > 1024) { pt_fail(1, "pt_build_grid: grid_res[%d] = %d out of range", a, g->res[a]); return nullptr; }
    PT_CUDA_NULL(cudaSetDevice(c->device), "select device");
    pt_event e = event_new(c);
    if (!e) return nullptr;
    c->grid_version++;
    cudaEventRecord(e->start, c->stream);
    if (pt_grid_build_device(c, g)) { pt_release_event(e); return nullptr; }
    cudaEventRecord(e->stop, c->stream);
    return e;
}

extern "C" int pt_read_grid_csr(pt_ctx c, uint32_t *cell_start, uint32_t *refs, uint64_t *total_refs) {
    if (!c || !c->grid_set) return pt_fail(1, "pt_read_grid_csr: no grid built");
    if (total_refs) *total_refs = c->total_refs;
    // The build leaves its last kernels unsynchronised on the context's (non-blocking) stream: read on THAT stream and
    // wait for it, like pt_read_accum / pt_read_vpls (the legacy default stream would not wait for it).
    PT_CUDA(cudaSetDevice(c->device), "select device");
    if (cell_start) PT_CUDA(cudaMemcpyAsync(cell_start, c->d_cell_start, (c->ncells + 1) * 4, cudaMemcpyDeviceToHost, c->stream), "read cell_start");
    if (refs && c->total_refs) PT_CUDA(cudaMemcpyAsync(refs, c->d_refs, c->total_refs * 4, cudaMemcpyDeviceToHost, c->stream), "read refs");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync grid read");
    return 0;
}

extern "C" int pt_read_grid_cells(pt_ctx c, void *cells, size_t ncells) {
    if (!c->grid_set) return pt_fail(1, "pt_read_grid_cells: no grid built");
    if (ncells != c->ncells) return pt_fail(1, "pt_read_grid_cells: expected %zu cells", c->ncells);
    if (c->ntri_total > 65536) return pt_fail(1, "pt_read_grid_cells: 16-bit cell format needs <= 65536 triangles");
    uint32_t *start = (uint32_t *)malloc((ncells + 1) * 4);
    uint32_t *refs = (uint32_t *)malloc((c->total_refs ? c->total_refs : 1) * 4);
    int rc = pt_read_grid_csr(c, start, refs, nullptr);
    if (!rc) {
        unsigned char *out = (unsigned char *)cells;
        memset(out, 0, ncells * 128);
        for (size_t i = 0; i < ncells; ++i) {
            uint32_t n = start[i + 1] - start[i];
            if (n > 62) n = 62;
            memcpy(out + 128 * i, &n, 4);
            for (uint32_t k = 0; k < n; ++k) {
                uint16_t id = (uint16_t)refs[start[i] + k];
                memcpy(out + 128 * i + 4 + 2 * k, &id, 2);
            }
        }
    }
    free(start);
    free(refs);
    return rc;
}

// ---------------------------------------------------------------- VLP bounding box / VLP grid (CLSuperMetropolisPathTracer_vlpgrid)
extern "C" int pt_vlp_bounds(pt_ctx c, float vmin[4], float vmax[4]) {
    if (!c || !vmin || !vmax) return pt_fail(1, "pt_vlp_bounds: null argument");
    if (!c->vpls_set) return pt_fail(1, "pt_vlp_bounds: no VLP buffer (pt_launch_lighttracer or pt_set_vpls first)");
    PT_CUDA(cudaSetDevice(c->device), "select device");
    return pt_vlp_bounds_device(c, vmin, vmax);
}

extern "C" pt_event pt_build_vlp_grid(pt_ctx c, const pt_grid *g) {
    if (!c || !g) { pt_fail(1, "pt_build_vlp_grid: null argument"); return nullptr; }
    if (!c->vpls_set) { pt_fail(1, "pt_build_vlp_grid: no VLP buffer (pt_launch_lighttracer or pt_set_vpls first)"); return nullptr; }
    if (g->res[0] < 1 || g->res[1] < 1 || g->res[2] < 1 || (long long)g->res[0] * g->res[1] * g->res[2] > (1ll << 28)) {
        pt_fail(1, "pt_build_vlp_grid: bad resolution %d x %d x %d", g->res[0], g->res[1], g->res[2]);
        return nullptr;
    }
    PT_CUDA_NULL(cudaSetDevice(c->device), "select device");
    pt_event e = event_new(c);
    if (!e) return nullptr;
    c->vlp_grid_version++;
    cudaEventRecord(e->start, c->stream);
    if (pt_vlp_grid_build_device(c, g)) { pt_release_event(e); return nullptr; }
    cudaEventRecord(e->stop, c->stream);
    return e;
}

extern "C" int pt_read_vlp_grid_csr(pt_ctx c, uint32_t *cell_start, uint32_t *refs, uint64_t *total_refs) {
    if (!c || !c->vlp_grid_set) return pt_fail(1, "pt_read_vlp_grid_csr: no VLP grid built");
    if (total_refs) *total_refs = c->vlp_total_refs;
    PT_CUDA(cudaSetDevice(c->device), "select device");
    if (cell_start) PT_CUDA(cudaMemcpyAsync(cell_start, c->d_vlp_cell_start, (c->vlp_ncells + 1) * 4, cudaMemcpyDeviceToHost, c->stream), "read VLP cell_start");
    if (refs && c->vlp_total_refs) PT_CUDA(cudaMemcpyAsync(refs, c->d_vlp_refs, c->vlp_total_refs * 4, cudaMemcpyDeviceToHost, c->stream), "read VLP refs");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync VLP grid read");
    return 0;
}

// the reference's 128-byte Cell {uint nels; ushort elem_index[62]} (metropolispathtracer.ocl Cell, host .c:39-42)
extern "C" int pt_read_vlp_grid_cells(pt_ctx c, void *cells, size_t ncells) {
    if (!c || !c->vlp_grid_set) return pt_fail(1, "pt_read_vlp_grid_cells: no VLP grid built");
    if (ncells != c->vlp_ncells) return pt_fail(1, "pt_read_vlp_grid_cells: expected %zu cells", c->vlp_ncells);
    if (c->nvpl > 65536) return pt_fail(1, "pt_read_vlp_grid_cells: 16-bit cell format needs <= 65536 VLPs");
    uint32_t *start = (uint32_t *)malloc((ncells + 1) * 4);
    uint32_t *refs = (uint32_t *)malloc((c->vlp_total_refs ? c->vlp_total_refs : 1) * 4);
    int rc = pt_read_vlp_grid_csr(c, start, refs, nullptr);
    if (!rc) {
        unsigned char *out = (unsigned char *)cells;
        memset(out, 0, ncells * 128);
        for (size_t i = 0; i < ncells; ++i) {
            uint32_t n = start[i + 1] - start[i];
            if (n > 62) n = 62;
            memcpy(out + 128 * i, &n, 4);
            for (uint32_t k = 0; k < n; ++k) {
                uint16_t id = (uint16_t)refs[start[i] + k];
                memcpy(out + 128 * i + 4 + 2 * k, &id, 2);
            }
        }
    }
    free(start);
    free(refs);
    return rc;
}

// --------------------------------------------------------------------------------------- render
static int ensure_dev(void **p, size_t *cap, size_t bytes) {
    if (*cap >= bytes && *p) return 0;
    cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    PT_CUDA(cudaMalloc(p, bytes), "alloc render buffer");
    *cap = bytes;
    return 0;
}

static int validate_params(pt_ctx c, const pt_render_params *p) {
    if (!c->scene_set) return pt_fail(1, "render: call pt_set_scene first");
    if (p->variant < 0 || p->variant > PT_VARIANT_VLPGRID) return pt_fail(1, "render: unknown variant %d", p->variant);
    if ((p->variant == PT_VARIANT_BIDIR || p->variant == PT_VARIANT_VLPGRID) && !c->vpls_set)
        return pt_fail(1, "render: the bidirectional variants need pt_launch_lighttracer (or pt_set_vpls) first");
    if (p->variant == PT_VARIANT_VLPGRID && !c->vlp_grid_set)
        return pt_fail(1, "render: the vlpgrid variant needs pt_build_vlp_grid first");
    if (p->variant == PT_VARIANT_VLPGRID && p->sample_blocks > 1) return pt_fail(1, "render: sample sharding is not defined for the vlpgrid variant");
    if (p->width <= 0 || p->height <= 0) return pt_fail(1, "render: bad image size %dx%d", p->width, p->height);
    if (p->spp <= 0) return pt_fail(1, "render: spp must be positive");
    if (p->variant == PT_VARIANT_NODOF && p->spp != 64) return pt_fail(1, "render: the NoDoF variant is defined for 64 samples (8x8 work-items) per pixel");
    if (p->variant == PT_VARIANT_GRID && !c->grid_set) return pt_fail(1, "render: grid variant needs pt_build_grid first");
    if (p->sample_blocks > 1) {
        if (p->variant == PT_VARIANT_NODOF) return pt_fail(1, "render: sample sharding is for the per-pixel-stream variants (NoDoF shards by tiles)");
        if (p->sample_block < 0 || p->sample_block >= p->sample_blocks) return pt_fail(1, "render: sample_block %d outside [0, %d)", p->sample_block, p->sample_blocks);
        if (p->spp % p->sample_blocks) return pt_fail(1, "render: spp %d is not a multiple of sample_blocks %d", p->spp, p->sample_blocks);
    }
    if ((long long)p->width * p->height * (p->variant == PT_VARIANT_NODOF ? 64 : 1) > 0x7fffffffLL)
        return pt_fail(1, "render: work-item ids exceed 31 bits (the reference computes them in int)");
    if (c->max_bounces > 0) {
        if (p->variant != PT_VARIANT_BASE && p->variant != PT_VARIANT_LMEM && p->variant != PT_VARIANT_GRID)
            return pt_fail(1, "render: diffuse bounces (pt_set_bounces %d) are defined for the base, lmem and trianglegrid variants only", c->max_bounces);
        if (p->kernel != PT_KERNEL_MEGA && p->kernel != PT_KERNEL_AUTO)
            return pt_fail(1, "render: diffuse bounces (pt_set_bounces %d) run in the per-pixel kernel only (PT_KERNEL_MEGA / AUTO), not flavour %d",
                           c->max_bounces, p->kernel);
    }
    return 0;
}

// pathtracer.ocl:26-34 on the host (seed derivation of the sample blocks)
static uint32_t host_randomize_id(uint32_t id) {
    id = (id ^ 61u) ^ (id >> 16);
    id *= 9u;
    id = id ^ (id >> 4);
    id *= 0x27d4eb2du;
    id = id ^ (id >> 15);
    return id;
}

static int fill_args(pt_ctx c, const pt_camera *cam, const pt_render_params *p, uint32_t *d_rgba, float4 *d_accum, uint4 *d_rng,
                     pt::LaunchArgs *A) {
    memset(A, 0, sizeof(*A));
    for (int k = 0; k < 3; ++k) { A->cam.up[k] = cam->cam_up[k]; A->cam.right[k] = cam->cam_right[k]; A->cam.eye[k] = cam->eye_offset[k]; }
    A->seeds = make_uint4(p->seeds[0], p->seeds[1], p->seeds[2], p->seeds[3]);
    A->W = p->width; A->H = p->height; A->spp = p->spp;
    A->scale = 224.0f / (float)p->spp;
    A->c0 = 13.0f; A->alpha = 255.0f;
    if (p->sample_blocks > 1) {
        // sample-range sharding ("throughput mode", SURVEY 8e): block b renders spp/blocks samples per pixel; block 0
        // continues the reference's own stream, block b > 0 draws from seeds ^ randomizeId(b); only block 0 carries
        // the bias 13 and alpha 255, so the SUM of the blocks' float buffers is the frame
        A->spp = p->spp / p->sample_blocks;
        if (p->sample_block > 0) {
            const uint32_t h = host_randomize_id((uint32_t)p->sample_block);
            A->seeds = make_uint4(p->seeds[0] ^ h, p->seeds[1] ^ h, p->seeds[2] ^ h, p->seeds[3] ^ h);
            A->c0 = 0.0f; A->alpha = 0.0f;
        }
    }
    int rb = p->row_begin, re = p->row_end;
    if (re <= 0 || re > p->height) re = p->height;
    if (rb < 0) rb = 0;
    if (rb > re) rb = re;
    A->row_begin = rb; A->row_end = re;
    if (p->row_interleave > 0 && p->nranks > 1) {
        int R = re - rb, hs = p->row_interleave;
        int nstripes = (R + hs - 1) / hs;
        int mine = (nstripes - p->rank + p->nranks - 1) / p->nranks;
        if (mine < 0) mine = 0;
        A->stripe_h = hs; A->rank = p->rank; A->nranks = p->nranks;
        A->nrows = mine * hs;
    } else {
        A->stripe_h = 0; A->rank = 0; A->nranks = 1;
        A->nrows = re - rb;
    }
    A->rgba = d_rgba; A->accum = d_accum; A->rng_out = d_rng;
    A->counters = c->d_counters;
    A->grid = c->grid;
    if (p->no_cull) A->grid.sph_k = INFINITY;       // sphere prefilter of the grid traversal off: every record is tested
    const int arith = p->arith != PT_ARITH_SEPARATE ? PT_ARITH_FMA : PT_ARITH_SEPARATE;
    A->gscene = c->d_scene[arith];
    A->scene_bytes = p->variant == PT_VARIANT_GRID ? (int)offsetof(pt::SceneBlock, tri) : c->scene_bytes;  // grid: no brute-force records
    const pt::SceneBlock *hs = c->h_scene[arith];
    A->ap.nsq = hs->nsq; A->ap.nsp = hs->nsp; A->ap.nlights = hs->nlights;
    for (int i = 0; i < PT_FAST_PRIMS; ++i) { A->ap.sq[i] = hs->sq[i]; A->ap.sp[i] = hs->sp[i]; }
    for (int i = 0; i < 5; ++i) A->ap.lights[i] = hs->lights[i];
    A->ap.mesh_cx = c->mesh_c[0]; A->ap.mesh_cy = c->mesh_c[1]; A->ap.mesh_cz = c->mesh_c[2];
    A->ap.mesh_r = p->no_cull ? INFINITY : c->mesh_r;
    A->ap.mesh_k = c->mesh_k;
    {
        // Per-cluster culling removes 60-70 % of the triangle tests of a ray that passes the mesh sphere, but adds a
        // serial chain of sphere tests to it.  Large frames are throughput-bound and gain (1080p x 1024 spp: torus
        // 79.9 -> 70.8 ms, 96-triangle mesh 90.6 -> 84.2 ms); small frames are bound by the serial sample chain of
        // their heaviest pixels and lose 8-11 % (512x512: 1.85 -> 2.01 ms).  Same threshold as the kernel choice.
        const long long pixels = (long long)p->width * (long long)A->nrows;     // THIS launch's share of the frame (rows / stripes)
        static int force = -2;
        if (force == -2) { const char *e = getenv("PT_CLUSTER_CULL"); force = e ? atoi(e) : -1; }
        bool on = force >= 0 ? force != 0 : pixels > 400000;
        if (p->cluster_cull == PT_CLUSTER_CULL_ON) on = true;
        if (p->cluster_cull == PT_CLUSTER_CULL_OFF) on = false;
        A->ap.ncl = (p->no_cull || !on) ? 0 : hs->ncl;
    }
    {
        // bounding box of all squares (x in [k-1,k+1], |y| <= 1, z = 4+j) and unit spheres (centre (k,0,j+4))
        float lo[3] = {1e30f, 1e30f, 1e30f}, hi[3] = {-1e30f, -1e30f, -1e30f};
        for (int i = 0; i < hs->nsq; ++i) {
            const float k = hs->sq[i].x, z = hs->sq[i].y;
            lo[0] = fminf(lo[0], k - 1.f); hi[0] = fmaxf(hi[0], k + 1.f);
            lo[1] = fminf(lo[1], -1.f);    hi[1] = fmaxf(hi[1], 1.f);
            lo[2] = fminf(lo[2], z);       hi[2] = fmaxf(hi[2], z);
        }
        for (int i = 0; i < hs->nsp; ++i) {
            const float k = -hs->sp[i].x, z = -hs->sp[i].y;
            lo[0] = fminf(lo[0], k - 1.f); hi[0] = fmaxf(hi[0], k + 1.f);
            lo[1] = fminf(lo[1], -1.f);    hi[1] = fmaxf(hi[1], 1.f);
            lo[2] = fminf(lo[2], z - 1.f); hi[2] = fmaxf(hi[2], z + 1.f);
        }
        for (int a = 0; a < 3; ++a) {
            A->ap.box_lo[a] = p->no_cull ? -INFINITY : lo[a];      // the per-ray margin is added on the device
            A->ap.box_hi[a] = p->no_cull ? INFINITY : hi[a];
        }
    }
    {
        static int env = -2;                      // PT_DEAD_RAYS=trace|elide overrides AUTO
        if (env == -2) { const char *e = getenv("PT_DEAD_RAYS"); env = !e ? -1 : (e[0] == 't' || e[0] == 'T' || e[0] == '1') ? 1 : 0; }
        bool trace = p->dead_rays == PT_DEAD_RAYS_TRACE || p->no_cull;
        if (p->dead_rays == PT_DEAD_RAYS_AUTO && env >= 0) trace = env == 1 || p->no_cull;
        A->ap.elide_dead = trace ? 0 : 1;
    }
    A->ap.ntri_hint = p->variant == PT_VARIANT_GRID ? 0 : hs->ntri;
    A->ap.tri_coop = 0;    // set by the launchers that stage the records in shared memory
    A->vpl = c->d_vpl_active; A->nvpl_active = c->d_vpl_count;
    if (p->variant == PT_VARIANT_VLPGRID) {
        A->vpl_raw = c->d_vpls; A->vg_start = c->d_vlp_cell_start; A->vg_refs = c->d_vlp_refs;
        for (int a = 0; a < 3; ++a) { A->vg_bmin[a] = c->vlp_grid_desc.box_min[a]; A->vg_cell[a] = c->vlp_grid_desc.cell_size[a]; A->vg_res[a] = c->vlp_grid_desc.res[a]; }
    }
    return 0;
}

// PT_KERNEL_AUTO / PT_SCENE_AUTO: measured best per variant on B200 (DESIGN.md section 4)
// Estimated number of pixels of this launch that have to scan the brute-force mesh at all — what PT_KERNEL_SPEC's first
// pass would queue: through a 48 x 48 grid of pixel centres (lens centre, no jitter; camera as base:233-236) the camera
// ray, and the shadow lines from its floor hit to every light, against the mesh's bounding sphere (inflated by ~1 % of
// the distance for lens blur and pixel footprint).  Only steers the kernel choice.
static double estimate_mesh_pixels(pt_ctx c, const pt::LaunchArgs &A) {
    if (c->h_scene[0]->ntri == 0) return 0.0;
    if (!(A.ap.mesh_r < 1e30f)) return (double)A.W * (double)A.nrows;      // no mesh cull (no_cull, or no finite sphere): every ray scans
    struct Key { int W, nrows, row_begin, row_end, stripe_h, rank, nranks; unsigned long long scene_version; pt::Camera cam; } key;
    memset(&key, 0, sizeof(key));
    key.W = A.W; key.nrows = A.nrows; key.row_begin = A.row_begin; key.row_end = A.row_end; key.stripe_h = A.stripe_h; key.rank = A.rank;
    key.nranks = A.nranks; key.scene_version = c->scene_version; key.cam = A.cam;
    static_assert(sizeof(Key) <= sizeof(c->mesh_est_key), "estimate key buffer too small");
    if (c->mesh_est_valid && memcmp(&key, c->mesh_est_key, sizeof(key)) == 0) return c->mesh_est;
    const int G = 48;
    const double C[3] = {c->mesh_c[0], c->mesh_c[1], c->mesh_c[2]};
    auto line_near = [&](const double o[3], const double d[3]) {           // d need not be normalised
        double dd = 0.0, b = 0.0, oc2 = 0.0;
        for (int a = 0; a < 3; ++a) { const double oc = C[a] - o[a]; dd += d[a] * d[a]; b += oc * d[a]; oc2 += oc * oc; }
        if (dd == 0.0) return false;
        const double dist2 = oc2 - b * b / dd, r = (double)c->mesh_r + 0.01 * sqrt(oc2);
        return dist2 <= r * r;
    };
    int heavy = 0;
    const pt::SceneBlock *hs = c->h_scene[0];
    for (int gy = 0; gy < G; ++gy)
        for (int gx = 0; gx < G; ++gx) {
            const int vr = (int)((gy + 0.5) / G * A.nrows);
            const double row = (double)pt::map_row(A, vr < A.nrows ? vr : A.nrows - 1) + 0.5, col = (gx + 0.5) / G * A.W;
            double d[3];
            for (int a = 0; a < 3; ++a) d[a] = (double)A.cam.right[a] * row + (double)A.cam.up[a] * col + (double)A.cam.eye[a];
            const double o[3] = {17.0, 16.0, 8.0};
            bool h = line_near(o, d);
            if (!h && d[2] < 0.0) {                                        // floor hit: do its shadow lines pass the mesh?
                const double t = -o[2] / d[2];
                const double X[3] = {o[0] + t * d[0], o[1] + t * d[1], 0.0};
                for (int l = 0; l < hs->nlights && !h; ++l) {
                    const double ld[3] = {hs->lights[l].x + 0.5 - X[0], hs->lights[l].y + 0.5 - X[1], hs->lights[l].z - X[2]};
                    h = line_near(X, ld);
                }
            }
            heavy += h;
        }
    c->mesh_est = (double)heavy / (G * G) * (double)A.W * (double)A.nrows;
    memcpy(c->mesh_est_key, &key, sizeof(key));
    c->mesh_est_valid = true;
    return c->mesh_est;
}

static pt_render_params resolve_auto(pt_ctx c, const pt_render_params *in, const pt::LaunchArgs &A) {
    const int nrows = A.nrows;
    pt_render_params p = *in;
    if (p.kernel == PT_KERNEL_AUTO) {
        if (c->max_bounces > 0) p.kernel = PT_KERNEL_MEGA;             // k_bounce_pixel: the one flavour that traces paths
        else if (p.variant == PT_VARIANT_BIDIR || p.variant == PT_VARIANT_VLPGRID) p.kernel = PT_KERNEL_MEGA;
        else if (p.variant == PT_VARIANT_NODOF) p.kernel = PT_KERNEL_MEGA;   // single-copy Sample(): 0.433 ms vs 0.479 ms persistent (512x512)
        else if (p.variant == PT_VARIANT_GRID) p.kernel = PT_KERNEL_MEGA;
        else {
            // brute-force triangle scenes: a pixel that sees the mesh is a ~1.7 ms serial chain at 64 spp.  While the mesh
            // covers few pixels the frame is bounded by those chains -> PT_KERNEL_SPEC traces 32 samples of such a pixel at
            // once (512x512 default scene 0.89 ms vs 1.76 persistent, 2.20 mega).  With enough heavy pixels to fill the GPU
            // (torus at 512x512: half the frame; any 1080p frame) the thread-per-pixel megakernel's dense lane-serial scan
            // is the cheaper form (1.17 vs 2.02 ms; 20.6 vs 31.1 ms per 256 spp at 1080p).
            static double thresh = -1.0;
            if (thresh < 0.0) { const char *e = getenv("PT_SPEC_MAX_MESH_PIXELS"); thresh = e ? atof(e) : 50000.0; }
            const double mesh_pixels = estimate_mesh_pixels(c, A);
            if (getenv("PT_DEBUG_AUTO")) fprintf(stderr, "ptcuda: AUTO %dx%d rows: estimated mesh pixels %.0f (threshold %.0f)\n", p.width, nrows, mesh_pixels, thresh);
            p.kernel = mesh_pixels <= thresh ? PT_KERNEL_SPEC : PT_KERNEL_MEGA;
        }
    }
    if (p.scene_mem == PT_SCENE_AUTO)
        p.scene_mem = (p.variant == PT_VARIANT_NODOF || p.variant == PT_VARIANT_GRID) ? PT_SCENE_CONST : PT_SCENE_SMEM;
    return p;
}

// p: the params as resolve_auto left them
static int dispatch(pt_ctx c, const pt_render_params *p, const pt::LaunchArgs &A) {
    c->last_kernel = p->kernel;
    DevLock lock(c->device);     // constant-scene bind + launch are one critical section per device
    PT_CUDA(cudaMemsetAsync(c->d_counters, 0, 8 * sizeof(unsigned long long), c->stream), "clear counters");
    if (A.nrows <= 0) return 0;
    if (p->variant == PT_VARIANT_BIDIR || p->variant == PT_VARIANT_VLPGRID) {
        if (p->kernel != PT_KERNEL_MEGA) return pt_fail(1, "render: the bidirectional variants have the megakernel flavour only (PT_KERNEL_MEGA / AUTO)");
        return pt_launch_bidir(c, p, A);
    }
    if (c->max_bounces > 0) return pt_launch_bounce(c, p, A, c->max_bounces);     // validate_params: MEGA, base / lmem / grid
    switch (p->kernel) {
        case PT_KERNEL_MEGA: return pt_launch_mega(c, p, A);
        case PT_KERNEL_PERSISTENT: return pt_launch_persistent(c, p, A);
        case PT_KERNEL_GRID_STREAM:
            if (p->variant != PT_VARIANT_GRID) return pt_fail(1, "PT_KERNEL_GRID_STREAM applies to the trianglegrid variant only");
            return pt_launch_stream_grid(c, p, A);
        case PT_KERNEL_SPEC: return pt_launch_spec(c, p, A);
        case PT_KERNEL_GRID_POOL:
            if (p->variant != PT_VARIANT_GRID) return pt_fail(1, "PT_KERNEL_GRID_POOL applies to the trianglegrid variant only");
            return pt_launch_grid_pool(c, p, A);
        case PT_KERNEL_GRID_QUEUE:
            if (p->variant != PT_VARIANT_GRID) return pt_fail(1, "PT_KERNEL_GRID_QUEUE applies to the trianglegrid variant only");
            return pt_launch_grid_queue(c, p, A);
        case PT_KERNEL_GRID_ASYNC:
            if (p->variant != PT_VARIANT_GRID) return pt_fail(1, "PT_KERNEL_GRID_ASYNC applies to the trianglegrid variant only");
            return pt_launch_grid_async(c, p, A);
        case PT_KERNEL_WAVEFRONT: return pt_launch_wavefront(c, p, A);
        case PT_KERNEL_GRID_TMA: return pt_launch_grid_tma(c, p, A);
    }
    return pt_fail(1, "render: unknown kernel kind %d", p->kernel);
}

// ---- progressive rendering: checks shared by range launches and pt_set_render_state, and the progression key
static int progression_params(pt_ctx c, const pt_camera *cam, const pt_render_params *p, const char *who, pt_progression_key *key) {
    if (p->variant == PT_VARIANT_NODOF)
        return pt_fail(1, "%s: the NoDoF variant has no per-pixel sample chain to continue (64 streams per pixel, fixed 8x8 reduction)", who);
    if (p->sample_blocks > 1) return pt_fail(1, "%s: sample_blocks > 1 (sample sharding) cannot be rendered in ranges", who);
    memset(key, 0, sizeof(*key));
    key->variant = p->variant; key->width = p->width; key->height = p->height; key->spp = p->spp;
    key->arith = p->arith != PT_ARITH_SEPARATE ? PT_ARITH_FMA : PT_ARITH_SEPARATE;
    key->row_begin = p->row_begin; key->row_end = p->row_end;
    key->row_interleave = p->row_interleave; key->rank = p->rank; key->nranks = p->nranks;
    memcpy(key->seeds, p->seeds, sizeof(key->seeds));
    key->cam = *cam;
    key->scene_version = c->scene_version;
    if (p->variant == PT_VARIANT_GRID) key->grid_version = c->grid_version;
    if (p->variant == PT_VARIANT_BIDIR || p->variant == PT_VARIANT_VLPGRID) key->vpl_version = c->vpl_version;
    if (p->variant == PT_VARIANT_VLPGRID) key->vlp_grid_version = c->vlp_grid_version;
    key->max_bounces = c->max_bounces;
    return 0;
}

// The one-launch render (range == false: samples [0, spp), state kept only as want_accum / want_rng ask) and a range
// [b, e) of a progression (state always kept in d_accum / d_rng) share validation, fill_args and dispatch.
static pt_event launch_render(pt_ctx c, const pt_camera *cam, const pt_render_params *p, bool range, int b, int e) {
    const char *who = range ? "pt_launch_pathtracer_range" : "pt_launch_pathtracer";
    if (!c || !cam || !p) { pt_fail(1, "%s: null argument", who); return nullptr; }
    if (validate_params(c, p)) return nullptr;
    pt_progression_key key;
    if (range) {
        if (progression_params(c, cam, p, who, &key)) return nullptr;
        if (b < 0 || e <= b || e > p->spp) { pt_fail(1, "%s: samples [%d, %d) are not a range of [0, %d)", who, b, e, p->spp); return nullptr; }
        if (b > 0) {
            if (!c->prog_active) { pt_fail(1, "%s: sample %d continues no progression (start at 0 or pt_set_render_state)", who, b); return nullptr; }
            if (memcmp(&key, &c->prog_key, sizeof(key)) != 0) {
                pt_fail(1, "%s: params, camera, scene, grid or VPLs differ from the progression's", who);
                return nullptr;
            }
            if (b != c->prog_next) { pt_fail(1, "%s: the progression continues at sample %d, not %d", who, c->prog_next, b); return nullptr; }
        }
    }
    PT_CUDA_NULL(cudaSetDevice(c->device), "select device");
    const size_t npix = (size_t)p->width * p->height;
    const size_t nitems = p->variant == PT_VARIANT_NODOF ? npix * 64 : npix;
    const bool keep_accum = range || p->want_accum, keep_rng = range || p->want_rng;
    // (a continuation has the key of the range before it, so the same size: these never grow, never lose the state)
    if (ensure_dev((void **)&c->d_rgba, &c->rgba_cap, npix * 4)) return nullptr;
    if (keep_accum && ensure_dev((void **)&c->d_accum, &c->accum_cap, npix * 16)) return nullptr;
    if (keep_rng && ensure_dev((void **)&c->d_rng, &c->rng_cap, nitems * 16)) return nullptr;
    pt::LaunchArgs A;
    fill_args(c, cam, p, c->d_rgba, keep_accum ? c->d_accum : nullptr, keep_rng ? c->d_rng : nullptr, &A);
    if (range) {
        A.spp = e - b;                                         // loop count; A.scale stays 224 / spp of the frame
        if (b > 0) { A.accum_in = c->d_accum; A.rng_in = c->d_rng; }
        if (e < p->spp) A.preview = (float)p->spp / (float)e;
    }
    const pt_render_params resolved = resolve_auto(c, p, A);
    if (range && resolved.kernel != PT_KERNEL_MEGA && resolved.kernel != PT_KERNEL_SPEC) {
        pt_fail(1, "%s: kernel flavour %d cannot render sample ranges; MEGA, SPEC and AUTO can", who, resolved.kernel);
        return nullptr;
    }
    c->prog_active = false;                 // from here on the state buffers may be overwritten
    const bool partial = A.nrows != p->height || A.stripe_h > 0;
    if (partial) {
        cudaMemsetAsync(c->d_rgba, 0, npix * 4, c->stream);
        if (keep_accum && b == 0) cudaMemsetAsync(c->d_accum, 0, npix * 16, c->stream);
        if (keep_rng && b == 0) cudaMemsetAsync(c->d_rng, 0, nitems * 16, c->stream);
    }
    pt_event ev = event_new(c);
    if (!ev) return nullptr;
    cudaEventRecord(ev->start, c->stream);
    if (dispatch(c, &resolved, A)) { pt_release_event(ev); return nullptr; }
    cudaEventRecord(ev->stop, c->stream);
    c->last_w = p->width; c->last_h = p->height; c->last_variant = p->variant;
    // what pt_read_accum / pt_read_rng_state may copy: only what THIS launch wrote
    c->accum_valid_w = keep_accum ? p->width : 0; c->accum_valid_h = keep_accum ? p->height : 0;
    c->rng_valid_items = keep_rng ? nitems : 0;
    if (range) { c->prog_active = true; c->prog_key = key; c->prog_next = e; }
    return ev;
}

extern "C" pt_event pt_launch_pathtracer(pt_ctx c, const pt_camera *cam, const pt_render_params *p) {
    return launch_render(c, cam, p, false, 0, p ? p->spp : 0);
}

extern "C" pt_event pt_launch_pathtracer_range(pt_ctx c, const pt_camera *cam, const pt_render_params *p, int sample_begin,
                                               int sample_end) {
    return launch_render(c, cam, p, true, sample_begin, sample_end);
}

extern "C" int pt_set_render_state(pt_ctx c, const pt_camera *cam, const pt_render_params *p, int samples_done, const float *accum,
                                   const uint32_t *rng_state) {
    const char *who = "pt_set_render_state";
    if (!c || !cam || !p || !accum || !rng_state) return pt_fail(1, "%s: null argument", who);
    int rc = validate_params(c, p);
    if (rc) return rc;
    pt_progression_key key;
    rc = progression_params(c, cam, p, who, &key);
    if (rc) return rc;
    if (samples_done <= 0 || samples_done >= p->spp) return pt_fail(1, "%s: samples_done %d outside (0, %d)", who, samples_done, p->spp);
    PT_CUDA(cudaSetDevice(c->device), "select device");
    const size_t npix = (size_t)p->width * p->height;
    c->prog_active = false;
    if (ensure_dev((void **)&c->d_accum, &c->accum_cap, npix * 16) || ensure_dev((void **)&c->d_rng, &c->rng_cap, npix * 16)) return 1;
    PT_CUDA(cudaMemcpyAsync(c->d_accum, accum, npix * 16, cudaMemcpyHostToDevice, c->stream), "upload accumulation buffer");
    PT_CUDA(cudaMemcpyAsync(c->d_rng, rng_state, npix * 16, cudaMemcpyHostToDevice, c->stream), "upload RNG states");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync state upload");     // the host buffers may be pageable
    c->accum_valid_w = p->width; c->accum_valid_h = p->height; c->rng_valid_items = npix;
    c->prog_active = true; c->prog_key = key; c->prog_next = samples_done;
    return 0;
}

// ------------------------------------------------------------------------------- bidirectional: VPLs
static int ensure_vpls(pt_ctx c, int n) {
    if (!c->d_vpl_count) PT_CUDA(cudaMalloc(&c->d_vpl_count, 2 * sizeof(int)), "alloc VPL count");
    const size_t need = n > 0 ? (size_t)n : 1;
    if (c->vpls_cap >= need) return 0;
    cudaFree(c->d_vpls); cudaFree(c->d_vpl_active);
    c->d_vpls = c->d_vpl_active = nullptr;
    c->vpls_cap = 0;
    PT_CUDA(cudaMalloc(&c->d_vpls, need * sizeof(float4)), "alloc VPL buffer");
    PT_CUDA(cudaMalloc(&c->d_vpl_active, need * sizeof(float4)), "alloc VPL list");
    c->vpls_cap = need;
    return 0;
}

extern "C" pt_event pt_launch_lighttracer(pt_ctx c, int n_vlp_per_light, const uint32_t seeds[4], int arith) {
    if (!c || !seeds) { pt_fail(1, "pt_launch_lighttracer: null argument"); return nullptr; }
    if (!c->scene_set) { pt_fail(1, "pt_launch_lighttracer: call pt_set_scene first"); return nullptr; }
    if (n_vlp_per_light <= 0 || (long long)n_vlp_per_light * 5 > 0x7fffffffLL) { pt_fail(1, "pt_launch_lighttracer: bad N_VLP %d", n_vlp_per_light); return nullptr; }
    PT_CUDA_NULL(cudaSetDevice(c->device), "select device");
    const int ar = arith != PT_ARITH_SEPARATE ? PT_ARITH_FMA : PT_ARITH_SEPARATE;
    const int nl = c->h_scene[ar]->nlights;
    if (ensure_vpls(c, n_vlp_per_light * nl)) return nullptr;
    pt_camera cam0;
    memset(&cam0, 0, sizeof(cam0));
    pt_render_params rp0;
    memset(&rp0, 0, sizeof(rp0));
    rp0.variant = PT_VARIANT_LMEM; rp0.width = 1; rp0.height = 1; rp0.spp = 64; rp0.arith = ar;
    memcpy(rp0.seeds, seeds, sizeof(rp0.seeds));
    pt::LaunchArgs LA;
    fill_args(c, &cam0, &rp0, nullptr, nullptr, nullptr, &LA);
    pt_event e = event_new(c);
    if (!e) return nullptr;
    c->vpl_version++;
    cudaEventRecord(e->start, c->stream);
    DevLock lock(c->device);
    if (pt_launch_light_tracer_kernels(c, ar, LA, n_vlp_per_light, c->d_vpls, nullptr, c->d_vpl_active, c->d_vpl_count)) {
        pt_release_event(e);
        return nullptr;
    }
    cudaEventRecord(e->stop, c->stream);
    c->nvpl = n_vlp_per_light * nl;
    c->vlp_grid_set = false;          // a VLP grid built on the previous buffer is stale
    c->vpls_set = true;
    return e;
}

// CLSuperMetropolisPathTracer(_vlpgrid): kernels lightTracer (seed paths) + MetropolisLightTracer, FIX mode (pt_metropolis.cuh)
extern "C" pt_event pt_launch_metropolis_lighttracer(pt_ctx c, int n_paths_per_light, const uint32_t seeds[4], int mutation_rounds, int arith) {
    if (!c || !seeds) { pt_fail(1, "pt_launch_metropolis_lighttracer: null argument"); return nullptr; }
    if (!c->scene_set) { pt_fail(1, "pt_launch_metropolis_lighttracer: call pt_set_scene first"); return nullptr; }
    if (n_paths_per_light <= 0 || (long long)n_paths_per_light * 20 > 0x7fffffffLL || mutation_rounds < 0) {
        pt_fail(1, "pt_launch_metropolis_lighttracer: bad arguments (%d paths, %d rounds)", n_paths_per_light, mutation_rounds);
        return nullptr;
    }
    PT_CUDA_NULL(cudaSetDevice(c->device), "select device");
    const int ar = arith != PT_ARITH_SEPARATE ? PT_ARITH_FMA : PT_ARITH_SEPARATE;
    const int nl = c->h_scene[ar]->nlights;
    const int npaths = n_paths_per_light * nl;
    if (ensure_vpls(c, 4 * npaths)) return nullptr;
    const size_t need = (size_t)(npaths > 0 ? npaths : 1) * 80;
    if (c->metro_cap < need) {
        cudaFree(c->d_metro_seed); cudaFree(c->d_metro_mutated);
        c->d_metro_seed = c->d_metro_mutated = nullptr;
        c->metro_cap = 0;
        PT_CUDA_NULL(cudaMalloc(&c->d_metro_seed, need), "alloc seed paths");
        PT_CUDA_NULL(cudaMalloc(&c->d_metro_mutated, need), "alloc mutated paths");
        c->metro_cap = need;
    }
    pt_camera cam0;
    memset(&cam0, 0, sizeof(cam0));
    pt_render_params rp0;
    memset(&rp0, 0, sizeof(rp0));
    rp0.variant = PT_VARIANT_LMEM; rp0.width = 1; rp0.height = 1; rp0.spp = 64; rp0.arith = ar;
    memcpy(rp0.seeds, seeds, sizeof(rp0.seeds));
    pt::LaunchArgs LA;
    fill_args(c, &cam0, &rp0, nullptr, nullptr, nullptr, &LA);
    pt_event e = event_new(c);
    if (!e) return nullptr;
    c->vpl_version++;
    cudaEventRecord(e->start, c->stream);
    DevLock lock(c->device);
    if (pt_launch_metropolis_kernels(c, ar, LA, n_paths_per_light, mutation_rounds, c->d_vpls, c->d_metro_seed, c->d_metro_mutated,
                                     c->d_vpl_active, c->d_vpl_count)) {
        pt_release_event(e);
        return nullptr;
    }
    cudaEventRecord(e->stop, c->stream);
    c->nvpl = 4 * npaths;
    c->n_metro_paths = npaths;
    c->vlp_grid_set = false;          // a VLP grid built on the previous buffer is stale
    c->vpls_set = true;
    return e;
}

extern "C" int pt_read_metropolis_paths(pt_ctx c, uint32_t *paths, int capacity_paths, int mutated) {
    if (!c) { pt_fail(1, "pt_read_metropolis_paths: null context"); return -1; }
    if (!paths) return c->n_metro_paths;
    if (capacity_paths < c->n_metro_paths) { pt_fail(1, "pt_read_metropolis_paths: buffer too small (%d < %d)", capacity_paths, c->n_metro_paths); return -1; }
    if (cudaSetDevice(c->device) != cudaSuccess) { pt_fail(1, "select device"); return -1; }
    if (c->n_metro_paths > 0 &&
        (cudaMemcpyAsync(paths, mutated ? c->d_metro_mutated : c->d_metro_seed, (size_t)c->n_metro_paths * 80, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
         cudaStreamSynchronize(c->stream) != cudaSuccess)) {
        pt_fail(1, "pt_read_metropolis_paths: copy failed");
        return -1;
    }
    return c->n_metro_paths;
}

extern "C" int pt_set_vpls(pt_ctx c, const float *vpls, int n) {
    if (!c || n < 0 || (n > 0 && !vpls)) return pt_fail(1, "pt_set_vpls: bad argument");
    PT_CUDA(cudaSetDevice(c->device), "select device");
    c->vpl_version++;
    int rc = ensure_vpls(c, n);
    if (rc) return rc;
    if (n > 0) PT_CUDA(cudaMemcpyAsync(c->d_vpls, vpls, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, c->stream), "upload VPLs");
    pt::k_compact_vpls<<<1, 256, 0, c->stream>>>(c->d_vpls, n, c->d_vpl_active, c->d_vpl_count);
    PT_CUDA(cudaGetLastError(), "launch k_compact_vpls");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync VPL upload");     // the host buffer may be pageable
    c->nvpl = n;
    c->vlp_grid_set = false;          // a VLP grid built on the previous buffer is stale
    c->vpls_set = true;
    return 0;
}

extern "C" int pt_read_vpls(pt_ctx c, float *vpls, int capacity) {
    if (!c || !c->vpls_set) { pt_fail(1, "pt_read_vpls: no VPL buffer (pt_launch_lighttracer / pt_set_vpls first)"); return -1; }
    if (!vpls) return c->nvpl;
    if (capacity < c->nvpl) { pt_fail(1, "pt_read_vpls: buffer too small (%d < %d)", capacity, c->nvpl); return -1; }
    if (cudaSetDevice(c->device) != cudaSuccess) { pt_fail(1, "select device"); return -1; }
    if (c->nvpl > 0 && cudaMemcpyAsync(vpls, c->d_vpls, (size_t)c->nvpl * sizeof(float4), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) {
        pt_fail(1, "read VPLs");
        return -1;
    }
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) { pt_fail(1, "sync"); return -1; }
    return c->nvpl;
}

extern "C" int pt_render_device(pt_ctx c, const pt_camera *cam, const pt_render_params *p, void *d_rgba8, void *d_accum_f32) {
    if (!c || !cam || !p || !d_rgba8) return pt_fail(1, "pt_render_device: null argument");
    int rc = validate_params(c, p);
    if (rc) return rc;
    PT_CUDA(cudaSetDevice(c->device), "select device");
    pt::LaunchArgs A;
    fill_args(c, cam, p, (uint32_t *)d_rgba8, (float4 *)d_accum_f32, nullptr, &A);
    c->last_variant = p->variant;
    c->prog_active = false;
    const pt_render_params resolved = resolve_auto(c, p, A);
    return dispatch(c, &resolved, A);
}

extern "C" void *pt_map_render(pt_ctx c, pt_event *evt) {
    if (!c || !c->d_rgba || c->last_w <= 0) { pt_fail(1, "pt_map_render: nothing rendered"); return nullptr; }
    PT_CUDA_NULL(cudaSetDevice(c->device), "select device");
    const size_t bytes = (size_t)c->last_w * c->last_h * 4;
    if (c->h_rgba_cap < bytes) {
        if (c->h_rgba) cudaFreeHost(c->h_rgba);
        c->h_rgba = nullptr;
        PT_CUDA_NULL(cudaMallocHost(&c->h_rgba, bytes), "alloc pinned render buffer");
        c->h_rgba_cap = bytes;
    }
    pt_event e = evt ? event_new(c) : nullptr;
    if (e) cudaEventRecord(e->start, c->stream);
    PT_CUDA_NULL(cudaMemcpyAsync(c->h_rgba, c->d_rgba, bytes, cudaMemcpyDeviceToHost, c->stream), "read render data");
    if (e) cudaEventRecord(e->stop, c->stream);
    PT_CUDA_NULL(cudaStreamSynchronize(c->stream), "map render buffer");
    if (evt) *evt = e;
    return c->h_rgba;
}

extern "C" int pt_read_accum(pt_ctx c, float *dst, size_t nfloats) {
    if (!c || !c->d_accum || c->accum_valid_w <= 0) return pt_fail(1, "pt_read_accum: last launch did not set want_accum");
    PT_CUDA(cudaSetDevice(c->device), "select device");
    size_t have = (size_t)c->accum_valid_w * c->accum_valid_h * 4;
    if (nfloats < have) return pt_fail(1, "pt_read_accum: buffer too small");
    PT_CUDA(cudaMemcpyAsync(dst, c->d_accum, have * 4, cudaMemcpyDeviceToHost, c->stream), "read accum");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync");
    return 0;
}

extern "C" int pt_read_rng_state(pt_ctx c, uint32_t *dst, size_t nwords) {
    if (!c || !c->d_rng || c->rng_valid_items == 0) return pt_fail(1, "pt_read_rng_state: last launch did not set want_rng");
    PT_CUDA(cudaSetDevice(c->device), "select device");
    size_t have = c->rng_valid_items * 4;
    if (nwords < have) return pt_fail(1, "pt_read_rng_state: buffer too small");
    PT_CUDA(cudaMemcpyAsync(dst, c->d_rng, have * 4, cudaMemcpyDeviceToHost, c->stream), "read rng");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync");
    return 0;
}

extern "C" int pt_get_counters(pt_ctx c, pt_counters *out) {
    unsigned long long h[8];
    PT_CUDA(cudaMemcpyAsync(h, c->d_counters, sizeof(h), cudaMemcpyDeviceToHost, c->stream), "read counters");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync");
    out->samples = h[0]; out->rays = h[1]; out->shadow_rays = h[2]; out->tri_tests = h[3];
    out->cells_visited = h[4]; out->prim_tests = h[5]; out->tri_tests_executed = h[6];
    out->vpl_evals = 0;
    if (c->last_variant == PT_VARIANT_BIDIR && c->scene_set && c->h_scene[1]->nlights > 0)   // nlights shadow rays per hit sample
        out->vpl_evals = h[2] / (uint64_t)c->h_scene[1]->nlights * (uint64_t)c->nvpl;
    return 0;
}

namespace pt {
__global__ void k_tonemap(const float4 *__restrict__ accum, uint32_t *__restrict__ rgba, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        float4 v = accum[i];
        rgba[i] = pack_rgba8_rz(v.x, v.y, v.z, v.w);
    }
}

template <bool FMA>
__global__ void k_probe_trace(int variant, int n, const float *o, const float *d, float *t, int *m, float *nrm, uint32_t *cells,
                              uint32_t *tests, const __grid_constant__ LaunchArgs P) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    V3 oo = mk3(o[3 * i], o[3 * i + 1], o[3 * i + 2]), dd = mk3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
    float tt = t[i];
    Counters cnt = {0, 0, 0, 0, 0, 0};
    int hit;
    V3 nn = mk3(0.f, 0.f, 0.f);
    if (variant == PT_VARIANT_BASE) {
        hit = trace_ray<FMA, false, false>(P.ap, &c_scene, P.grid, oo, dd, tt, cnt);
        if (hit) nn = hit_normal<FMA, false>(P.ap, &c_scene, P.grid, hit, oo, dd, tt);
    } else if (variant == PT_VARIANT_GRID) {
        hit = trace_ray<FMA, true, true>(P.ap, &c_scene, P.grid, oo, dd, tt, cnt);
        if (hit) nn = hit_normal<FMA, true>(P.ap, &c_scene, P.grid, hit, oo, dd, tt);
    } else {
        hit = trace_ray<FMA, true, false>(P.ap, &c_scene, P.grid, oo, dd, tt, cnt);
        if (hit) nn = hit_normal<FMA, false>(P.ap, &c_scene, P.grid, hit, oo, dd, tt);
    }
    t[i] = tt; m[i] = hit_material(hit);
    nrm[3 * i] = nn.x; nrm[3 * i + 1] = nn.y; nrm[3 * i + 2] = nn.z;
    cells[i] = cnt.cells;
    tests[i] = variant == PT_VARIANT_GRID ? cnt.gtri : cnt.btests;
}

__global__ void k_probe_rng(uint4 seeds, uint32_t gid, int nsteps, float *out_f, uint32_t *out_state) {
    Rng r = rng_seed(seeds, gid);
    for (int k = 0; k < nsteps; ++k) rng_next(r, out_f[2 * k], out_f[2 * k + 1]);
    out_state[0] = r.x0; out_state[1] = r.x1; out_state[2] = r.c0; out_state[3] = r.c1;
}
}  // namespace pt

extern "C" int pt_tonemap_device(pt_ctx c, const void *d_accum, void *d_rgba8, int width, int height) {
    size_t n = (size_t)width * height;
    pt::k_tonemap<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>((const float4 *)d_accum, (uint32_t *)d_rgba8, n);
    PT_CUDA(cudaGetLastError(), "tonemap");
    return 0;
}

extern "C" int pt_probe_trace_counts(pt_ctx c, int variant, int arith, int n, const float *o, const float *d, float *t_inout,
                                     int32_t *m_out, float *n_out, uint32_t *cells_out, uint32_t *tests_out) {
    if (!c->scene_set) return pt_fail(1, "pt_probe_trace: no scene");
    if (variant == PT_VARIANT_GRID && !c->grid_set) return pt_fail(1, "pt_probe_trace: no grid");
    if (n < 0) return pt_fail(1, "pt_probe_trace: n < 0");
    if (n == 0) return 0;
    PT_CUDA(cudaSetDevice(c->device), "select device");
    const int ar = arith != PT_ARITH_SEPARATE ? PT_ARITH_FMA : PT_ARITH_SEPARATE;
    DevLock lock(c->device);
    int rc = pt_bind_const_scene(c, ar);
    if (rc) return rc;
    const size_t nn = (size_t)n;
    float *d_o, *d_d, *d_t, *d_n;
    int *d_m;
    uint32_t *d_cells, *d_tests;
    PT_CUDA(cudaMalloc(&d_o, nn * 12), "alloc"); PT_CUDA(cudaMalloc(&d_d, nn * 12), "alloc");
    PT_CUDA(cudaMalloc(&d_t, nn * 4), "alloc"); PT_CUDA(cudaMalloc(&d_n, nn * 12), "alloc");
    PT_CUDA(cudaMalloc(&d_m, nn * 4), "alloc");
    PT_CUDA(cudaMalloc(&d_cells, nn * 4), "alloc"); PT_CUDA(cudaMalloc(&d_tests, nn * 4), "alloc");
    cudaMemcpyAsync(d_o, o, nn * 12, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(d_d, d, nn * 12, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(d_t, t_inout, nn * 4, cudaMemcpyHostToDevice, c->stream);
    pt_camera cam0;
    memset(&cam0, 0, sizeof(cam0));
    pt_render_params rp0;
    memset(&rp0, 0, sizeof(rp0));
    rp0.variant = variant; rp0.width = 1; rp0.height = 1; rp0.spp = 64; rp0.arith = ar;
    pt::LaunchArgs LA;
    fill_args(c, &cam0, &rp0, nullptr, nullptr, nullptr, &LA);
    if (ar == PT_ARITH_FMA)
        pt::k_probe_trace<true><<<(n + 127) / 128, 128, 0, c->stream>>>(variant, n, d_o, d_d, d_t, d_m, d_n, d_cells, d_tests, LA);
    else
        pt::k_probe_trace<false><<<(n + 127) / 128, 128, 0, c->stream>>>(variant, n, d_o, d_d, d_t, d_m, d_n, d_cells, d_tests, LA);
    PT_CUDA(cudaGetLastError(), "probe trace");
    cudaMemcpyAsync(t_inout, d_t, nn * 4, cudaMemcpyDeviceToHost, c->stream);
    if (m_out) cudaMemcpyAsync(m_out, d_m, nn * 4, cudaMemcpyDeviceToHost, c->stream);
    if (n_out) cudaMemcpyAsync(n_out, d_n, nn * 12, cudaMemcpyDeviceToHost, c->stream);
    if (cells_out) cudaMemcpyAsync(cells_out, d_cells, nn * 4, cudaMemcpyDeviceToHost, c->stream);
    if (tests_out) cudaMemcpyAsync(tests_out, d_tests, nn * 4, cudaMemcpyDeviceToHost, c->stream);
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync probe");
    cudaFree(d_o); cudaFree(d_d); cudaFree(d_t); cudaFree(d_n); cudaFree(d_m); cudaFree(d_cells); cudaFree(d_tests);
    return 0;
}

extern "C" int pt_probe_trace(pt_ctx c, int variant, int arith, int n, const float *o, const float *d, float *t_inout,
                              int32_t *m_out, float *n_out) {
    return pt_probe_trace_counts(c, variant, arith, n, o, d, t_inout, m_out, n_out, nullptr, nullptr);
}

extern "C" int pt_selftest_fastmath(pt_ctx c, uint64_t npairs, uint32_t seed, uint64_t out[3]) {
    PT_CUDA(cudaSetDevice(c->device), "select device");
    unsigned long long *d;
    PT_CUDA(cudaMalloc(&d, 3 * sizeof(unsigned long long)), "alloc");
    cudaMemsetAsync(d, 0, 3 * sizeof(unsigned long long), c->stream);
    pt::k_selftest_fastmath<<<c->sm_count * 8, 256, 0, c->stream>>>((unsigned long long)npairs, seed, d);
    PT_CUDA(cudaGetLastError(), "selftest");
    unsigned long long h[3];
    cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, c->stream);
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync selftest");
    cudaFree(d);
    out[0] = h[0]; out[1] = h[1]; out[2] = h[2];
    return 0;
}

extern "C" int pt_probe_rng(pt_ctx c, const uint32_t seeds[4], uint32_t gid, int nsteps, float *out_f, uint32_t out_state[4]) {
    PT_CUDA(cudaSetDevice(c->device), "select device");
    float *d_f;
    uint32_t *d_s;
    PT_CUDA(cudaMalloc(&d_f, (size_t)nsteps * 8 + 8), "alloc"); PT_CUDA(cudaMalloc(&d_s, 16), "alloc");
    pt::k_probe_rng<<<1, 1, 0, c->stream>>>(make_uint4(seeds[0], seeds[1], seeds[2], seeds[3]), gid, nsteps, d_f, d_s);
    PT_CUDA(cudaGetLastError(), "probe rng");
    cudaMemcpyAsync(out_f, d_f, (size_t)nsteps * 8, cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpyAsync(out_state, d_s, 16, cudaMemcpyDeviceToHost, c->stream);
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync probe");
    cudaFree(d_f); cudaFree(d_s);
    return 0;
}

// ---- measured peaks of THIS device for the roofline the benchmark reports (FP32 pipe and issue slots) ----
namespace pt {
// 8 independent FFMA chains per thread, 512 FFMAs per loop trip: the loop overhead is < 1 % of the instructions
__global__ void __launch_bounds__(256) k_peak_ffma(float *out, int trips, float a, float b) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
    for (int t = 0; t < trips; ++t) {
#pragma unroll
        for (int k = 0; k < 64; ++k) {
            x0 = __fmaf_rn(x0, a, b); x1 = __fmaf_rn(x1, a, b); x2 = __fmaf_rn(x2, a, b); x3 = __fmaf_rn(x3, a, b);
            x4 = __fmaf_rn(x4, a, b); x5 = __fmaf_rn(x5, a, b); x6 = __fmaf_rn(x6, a, b); x7 = __fmaf_rn(x7, a, b);
        }
    }
    const float r = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (r == 123.456f) out[0] = r;                 // never true: keeps the chains alive
}
// the instruction mix of the tracers' inner loops in miniature: FP32 (FMA pipe), integer add / logic (ALU pipe) and
// 32-bit integer multiply-add (the RNG), all independent — measures how many warp instructions per second the
// schedulers really issue when no pipe is the limit by itself
__global__ void __launch_bounds__(256) k_peak_issue(unsigned *out, int trips, float a, float b, unsigned m) {
    float f0 = threadIdx.x * 1e-3f, f1 = f0 + 1.f, f2 = f0 + 2.f, f3 = f0 + 3.f;
    unsigned i0 = threadIdx.x, i1 = i0 + 1u, i2 = i0 + 2u, i3 = i0 + 3u;
    for (int t = 0; t < trips; ++t) {
#pragma unroll
        for (int k = 0; k < 64; ++k) {
            f0 = __fmaf_rn(f0, a, b); i0 = (i0 ^ m) + i1;
            f1 = __fmaf_rn(f1, a, b); i1 = (i1 + m) ^ i2;
            f2 = __fmaf_rn(f2, a, b); i2 = (i2 ^ m) + i3;
            f3 = __fmaf_rn(f3, a, b); i3 = (i3 + m) ^ i0;
        }
    }
    const float r = (f0 + f1) + (f2 + f3);
    const unsigned q = (i0 ^ i1) + (i2 ^ i3);
    if (r == 123.456f && q == 77u) out[0] = q;
}
}  // namespace pt

// out[0] = measured FP32 TFLOP/s (FFMA = 2 flop), out[1] = FFMA warp instructions per second (G),
// out[2] = warp instructions per second of the mixed FP32 + integer kernel (G), out[3] = its duration in ms
extern "C" int pt_last_kernel(pt_ctx c) { return c ? c->last_kernel : -1; }

extern "C" int pt_set_bounces(pt_ctx c, int max_bounces) {
    if (!c) return pt_fail(1, "pt_set_bounces: null context");
    if (max_bounces < 0 || max_bounces > PT_MAX_BOUNCES) return pt_fail(1, "pt_set_bounces: %d outside [0, %d]", max_bounces, PT_MAX_BOUNCES);
    c->max_bounces = max_bounces;
    return 0;
}

// diagnostics: copy `bytes` of the context's scratch buffer (offset 256: per-CTA timing table of PT_CTA_TIMES=1) to the host
extern "C" int pt_debug_read_scratch(pt_ctx c, void *dst, size_t offset, size_t bytes) {
    if (!c || !dst || offset + bytes > c->scratch_cap) return pt_fail(1, "pt_debug_read_scratch: out of range");
    PT_CUDA(cudaSetDevice(c->device), "select device");
    PT_CUDA(cudaMemcpyAsync(dst, (char *)c->d_scratch + offset, bytes, cudaMemcpyDeviceToHost, c->stream), "read scratch");
    PT_CUDA(cudaStreamSynchronize(c->stream), "sync");
    return 0;
}

extern "C" int pt_measure_peaks(pt_ctx c, double out[4]) {
    if (!c || !out) return pt_fail(1, "pt_measure_peaks: null argument");
    PT_CUDA(cudaSetDevice(c->device), "select device");
    float *d = nullptr;
    PT_CUDA(cudaMalloc(&d, 64), "alloc");
    cudaEvent_t e0, e1;
    PT_CUDA(cudaEventCreate(&e0), "event"); PT_CUDA(cudaEventCreate(&e1), "event");
    const int blocks = c->sm_count * 8, threads = 256, trips = 256;
    float best_f = 1e30f, best_i = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {              // rep 0 warms the clocks up
        cudaEventRecord(e0, c->stream);
        pt::k_peak_ffma<<<blocks, threads, 0, c->stream>>>(d, trips, 1.0000001f, 1e-7f);
        cudaEventRecord(e1, c->stream);
        PT_CUDA(cudaEventSynchronize(e1), "peak kernel");
        float ms = 0.f; cudaEventElapsedTime(&ms, e0, e1);
        if (rep && ms < best_f) best_f = ms;
        cudaEventRecord(e0, c->stream);
        pt::k_peak_issue<<<blocks, threads, 0, c->stream>>>((unsigned *)d, trips, 1.0000001f, 1e-7f, 0x9E3779B9u);
        cudaEventRecord(e1, c->stream);
        PT_CUDA(cudaEventSynchronize(e1), "peak kernel");
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep && ms < best_i) best_i = ms;
    }
    PT_CUDA(cudaGetLastError(), "peak kernels");
    const double threads_total = (double)blocks * threads, warps = threads_total / 32.0;
    const double ffma_per_thread = (double)trips * 64 * 8;
    out[0] = threads_total * ffma_per_thread * 2.0 / (best_f * 1e-3) / 1e12;
    out[1] = warps * ffma_per_thread / (best_f * 1e-3) / 1e9;
    out[2] = warps * ((double)trips * 64 * 12) / (best_i * 1e-3) / 1e9;     // 4 FFMA + 4 x (LOP3 + IADD) per inner step
    out[3] = best_i;
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    return 0;
}

extern "C" int pt_render_host(pt_ctx c, const pt_scene *scene, const pt_grid *grid, const pt_camera *cam,
                              const pt_render_params *p, uint8_t *rgba8_out) {
    int rc = pt_set_scene(c, scene);
    if (rc) return rc;
    if (p->variant == PT_VARIANT_GRID) {
        if (!grid) return pt_fail(1, "pt_render_host: grid variant needs a pt_grid");
        pt_event g = pt_build_grid(c, grid);
        if (!g) return 1;
        pt_release_event(g);
    }
    if (p->variant == PT_VARIANT_VLPGRID)
        return pt_fail(1, "pt_render_host: the vlpgrid variant needs its VPL buffer and VLP grid set up explicitly (pt_set_vpls / pt_launch_lighttracer, pt_vlp_bounds, pt_build_vlp_grid, then pt_launch_pathtracer)");
    if (p->variant == PT_VARIANT_BIDIR) {
        pt_event l = pt_launch_lighttracer(c, p->n_vlp > 0 ? p->n_vlp : 512, p->seeds, p->arith);
        if (!l) return 1;
        pt_release_event(l);
    }
    pt_event e = pt_launch_pathtracer(c, cam, p);
    if (!e) return 1;
    void *h = pt_map_render(c, nullptr);
    pt_release_event(e);
    if (!h) return 1;
    memcpy(rgba8_out, h, (size_t)p->width * p->height * 4);
    return 0;
}


// ------------------------------------------------------------------------- single-process multi-GPU
// NCCL is reached through dlopen so that libptcuda.so carries no link-time dependency on it (a process
// that already loaded torch's bundled libnccl.so.2 keeps using that one).  Minimal local declarations of the
// few entry points used (public NCCL API: ncclCommInitAll, ncclReduce, group calls).
typedef struct ncclComm *pt_ncclComm_t;
enum { PT_NCCL_FLOAT32 = 7, PT_NCCL_SUM = 0 };
struct pt_nccl_api {
    void *lib;
    int (*CommInitAll)(pt_ncclComm_t *, int, const int *);
    int (*CommDestroy)(pt_ncclComm_t);
    int (*GroupStart)(void);
    int (*GroupEnd)(void);
    int (*Reduce)(const void *, void *, size_t, int, int, int, pt_ncclComm_t, cudaStream_t);
    const char *(*GetErrorString)(int);
};

struct pt_multi_s {
    int n;
    pt_ctx ctx[16];
    float4 *accum[16];
    uint32_t *rgba_scratch[16];
    size_t cap_pixels;
    pt_nccl_api nccl;
    pt_ncclComm_t comms[16];
    int last_w, last_h;
};

static int nccl_load(pt_nccl_api *a) {
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    a->lib = nullptr;
    for (const char *nm : names) {
        a->lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (a->lib) break;
    }
    if (!a->lib) return pt_fail(1, "pt_multi_create: cannot load libnccl.so.2 (%s)", dlerror());
    *(void **)&a->CommInitAll = dlsym(a->lib, "ncclCommInitAll");
    *(void **)&a->CommDestroy = dlsym(a->lib, "ncclCommDestroy");
    *(void **)&a->GroupStart = dlsym(a->lib, "ncclGroupStart");
    *(void **)&a->GroupEnd = dlsym(a->lib, "ncclGroupEnd");
    *(void **)&a->Reduce = dlsym(a->lib, "ncclReduce");
    *(void **)&a->GetErrorString = dlsym(a->lib, "ncclGetErrorString");
    if (!a->CommInitAll || !a->CommDestroy || !a->GroupStart || !a->GroupEnd || !a->Reduce)
        return pt_fail(1, "pt_multi_create: libnccl lacks a required symbol");
    return 0;
}

extern "C" void pt_multi_destroy(pt_multi m);

// run f(i) for i = 0..n-1 on n host threads (one per device: CUDA context creation, scene uploads and grid builds of the
// devices are independent and each takes a noticeable fraction of a second); returns the first non-zero result
template <class F>
static int for_each_device(int n, F f) {
    std::vector<int> rc((size_t)n, 0);
    std::vector<std::string> msg((size_t)n);
    std::vector<std::thread> th;
    for (int i = 1; i < n; ++i)
        th.emplace_back([&, i] {
            rc[(size_t)i] = f(i);
            if (rc[(size_t)i]) msg[(size_t)i] = g_last_error;      // the message lives in the worker's thread-local buffer
        });
    rc[0] = f(0);
    for (auto &t : th) t.join();
    for (int i = 0; i < n; ++i)
        if (rc[(size_t)i]) {
            if (i > 0) snprintf(g_last_error, sizeof(g_last_error), "%s", msg[(size_t)i].c_str());
            return rc[(size_t)i];
        }
    return 0;
}

extern "C" pt_multi pt_multi_create(int ngpus) {
    if (ngpus < 1 || ngpus > 16 || ngpus > pt_device_count()) { pt_fail(1, "pt_multi_create: %d GPUs requested, %d visible", ngpus, pt_device_count()); return nullptr; }
    pt_multi m = (pt_multi)calloc(1, sizeof(pt_multi_s));
    m->n = ngpus;
    // the contexts (CUDA initialisation of every device) in parallel, the NCCL library load beside them
    int nccl_rc = 0;
    std::thread loader;
    if (ngpus > 1) loader = std::thread([&] { nccl_rc = nccl_load(&m->nccl); });
    const int crc = for_each_device(ngpus, [&](int i) { m->ctx[i] = pt_create(i); return m->ctx[i] ? 0 : 1; });
    if (loader.joinable()) loader.join();
    if (crc) { pt_multi_destroy(m); return nullptr; }           // releases the contexts created so far
    if (ngpus > 1) {
        if (nccl_rc) { pt_multi_destroy(m); return nullptr; }
        int devs[16];
        for (int i = 0; i < ngpus; ++i) devs[i] = i;
        int rc = m->nccl.CommInitAll(m->comms, ngpus, devs);
        if (rc) {
            for (int i = 0; i < ngpus; ++i) m->comms[i] = nullptr;
            pt_fail(rc, "ncclCommInitAll: %s", m->nccl.GetErrorString ? m->nccl.GetErrorString(rc) : "?");
            pt_multi_destroy(m);
            return nullptr;
        }
    }
    return m;
}

extern "C" void pt_multi_destroy(pt_multi m) {
    if (!m) return;
    for (int i = 0; i < m->n; ++i) {
        cudaSetDevice(i);
        if (m->n > 1 && m->comms[i] && m->nccl.CommDestroy) m->nccl.CommDestroy(m->comms[i]);
        cudaFree(m->accum[i]);
        cudaFree(m->rgba_scratch[i]);
        pt_destroy(m->ctx[i]);          // NULL-safe
    }
    free(m);
}

extern "C" int pt_multi_set_scene(pt_multi m, const pt_scene *scene) {
    // the scene is replicated on every device; the uploads (pageable host memory -> staged copies) run side by side
    return for_each_device(m->n, [&](int i) { return pt_set_scene(m->ctx[i], scene); });
}

extern "C" pt_event pt_multi_build_grid(pt_multi m, const pt_grid *grid) {
    pt_event ev[16] = {nullptr};
    const int rc = for_each_device(m->n, [&](int i) { ev[i] = pt_build_grid(m->ctx[i], grid); return ev[i] ? 0 : 1; });
    for (int i = 1; i < m->n; ++i) pt_release_event(ev[i]);
    if (rc) { pt_release_event(ev[0]); return nullptr; }
    return ev[0];
}

// every device traces the (tiny) light pass itself: identical seeds -> identical VPL buffers, no exchange needed
extern "C" pt_event pt_multi_launch_lighttracer(pt_multi m, int n_vlp_per_light, const uint32_t seeds[4], int arith) {
    pt_event first = nullptr;
    for (int i = 0; i < m->n; ++i) {
        pt_event e = pt_launch_lighttracer(m->ctx[i], n_vlp_per_light, seeds, arith);
        if (!e) return nullptr;
        if (i == 0) first = e; else pt_release_event(e);
    }
    return first;
}

extern "C" pt_event pt_multi_launch_pathtracer(pt_multi m, const pt_camera *cam, const pt_render_params *params) {
    if (!m || !cam || !params) { pt_fail(1, "pt_multi_launch_pathtracer: null argument"); return nullptr; }
    if (m->n == 1) {
        pt_render_params p1 = *params;
        p1.sample_blocks = 0;
        return pt_launch_pathtracer(m->ctx[0], cam, &p1);
    }
    // ---- everything that can be rejected is rejected BEFORE any event or NCCL group exists
    // sample_blocks > 1 asks for sample-range sharding instead of tiles: device i renders sample block i of the WHOLE image
    const bool by_samples = params->sample_blocks > 1;
    if (by_samples && params->sample_blocks != m->n) { pt_fail(1, "pt_multi: sample_blocks (%d) must equal the number of GPUs (%d)", params->sample_blocks, m->n); return nullptr; }
    pt_render_params dev_params[16];
    for (int i = 0; i < m->n; ++i) {
        pt_render_params &p = dev_params[i];
        p = *params;
        if (by_samples) { p.sample_block = i; p.row_interleave = 0; p.rank = 0; p.nranks = 1; }
        else { p.row_interleave = 8; p.rank = i; p.nranks = m->n; p.sample_block = 0; p.sample_blocks = 0; }
        if (validate_params(m->ctx[i], &p)) return nullptr;
    }
    const size_t npix = (size_t)params->width * params->height;
    for (int i = 0; i < m->n; ++i) {
        PT_CUDA_NULL(cudaSetDevice(i), "select device");
        if (m->cap_pixels < npix) {
            cudaFree(m->accum[i]); cudaFree(m->rgba_scratch[i]);
            m->accum[i] = nullptr; m->rgba_scratch[i] = nullptr;
            m->cap_pixels = 0;                 // a failure below must not leave a stale capacity behind
            PT_CUDA_NULL(cudaMalloc(&m->accum[i], npix * 16), "alloc accumulation buffer");
            PT_CUDA_NULL(cudaMalloc(&m->rgba_scratch[i], npix * 4), "alloc scratch image");
        }
    }
    // (cap_pixels is per multi-context: all devices were (re)allocated together above)
    if (m->cap_pixels < npix) m->cap_pixels = npix;
    pt_ctx c0 = m->ctx[0];
    PT_CUDA_NULL(cudaSetDevice(0), "select device");
    if (ensure_dev((void **)&c0->d_rgba, &c0->rgba_cap, npix * 4)) return nullptr;
    pt_event e = event_new(c0);
    if (!e) return nullptr;
    bool group_open = false;
    int rc = 0;
    cudaEventRecord(e->start, c0->stream);
    for (int i = 0; i < m->n && !rc; ++i) {
        if (cudaSetDevice(i) != cudaSuccess) { rc = pt_fail(1, "select device"); break; }
        if (cudaMemsetAsync(m->accum[i], 0, npix * 16, m->ctx[i]->stream) != cudaSuccess) { rc = pt_fail(1, "clear accumulation buffer"); break; }
        rc = pt_render_device(m->ctx[i], cam, &dev_params[i], m->rgba_scratch[i], m->accum[i]);
    }
    if (!rc) {
        // the only collective: sum the accumulation buffers onto device 0 (rows a device does not own are zero)
        m->nccl.GroupStart();
        group_open = true;
        for (int i = 0; i < m->n && !rc; ++i) {
            int nrc = m->nccl.Reduce(m->accum[i], m->accum[i], npix * 4, PT_NCCL_FLOAT32, PT_NCCL_SUM, 0, m->comms[i], m->ctx[i]->stream);
            if (nrc) rc = pt_fail(nrc, "ncclReduce failed: %s", m->nccl.GetErrorString ? m->nccl.GetErrorString(nrc) : "?");
        }
    }
    if (group_open) {                              // never leave the NCCL group open, whatever happened inside it
        int nrc = m->nccl.GroupEnd();
        if (nrc && !rc) rc = pt_fail(nrc, "ncclGroupEnd failed: %s", m->nccl.GetErrorString ? m->nccl.GetErrorString(nrc) : "?");
    }
    if (!rc && cudaSetDevice(0) != cudaSuccess) rc = pt_fail(1, "select device");
    if (!rc) rc = pt_tonemap_device(c0, m->accum[0], c0->d_rgba, params->width, params->height);
    if (rc) { pt_release_event(e); return nullptr; }
    cudaEventRecord(e->stop, c0->stream);
    c0->last_w = params->width; c0->last_h = params->height; c0->last_variant = params->variant;
    c0->accum_valid_w = c0->accum_valid_h = 0; c0->rng_valid_items = 0;
    m->last_w = params->width; m->last_h = params->height;
    return e;
}

extern "C" int pt_multi_set_bounces(pt_multi m, int max_bounces) {
    if (!m) return pt_fail(1, "pt_multi_set_bounces: null argument");
    if (max_bounces < 0 || max_bounces > PT_MAX_BOUNCES) return pt_fail(1, "pt_multi_set_bounces: %d outside [0, %d]", max_bounces, PT_MAX_BOUNCES);
    for (int i = 0; i < m->n; ++i) {
        const int rc = pt_set_bounces(m->ctx[i], max_bounces);
        if (rc) return rc;
    }
    return 0;
}

extern "C" void *pt_multi_map_render(pt_multi m, pt_event *evt) {
    for (int i = 1; i < m->n; ++i) { cudaSetDevice(i); cudaStreamSynchronize(m->ctx[i]->stream); }
    cudaSetDevice(0);
    return pt_map_render(m->ctx[0], evt);
}

extern "C" int pt_multi_get_counters(pt_multi m, pt_counters *out) {
    memset(out, 0, sizeof(*out));
    for (int i = 0; i < m->n; ++i) {
        pt_counters c;
        cudaSetDevice(i);
        int rc = pt_get_counters(m->ctx[i], &c);
        if (rc) return rc;
        out->samples += c.samples; out->rays += c.rays; out->shadow_rays += c.shadow_rays; out->tri_tests += c.tri_tests;
        out->cells_visited += c.cells_visited; out->prim_tests += c.prim_tests; out->tri_tests_executed += c.tri_tests_executed;
        out->vpl_evals += c.vpl_evals;
    }
    return 0;
}
