// pt_host.h — host-side state shared by the translation units of libptcuda.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ptcuda.h"
#include "pt_device.cuh"

namespace pt {

struct LaunchArgs {
    Camera cam;
    uint4 seeds;
    int W, H, spp;          // spp: samples per pixel THIS launch runs (a range of a progression: its length)
    float scale;            // 224/spp (3.5 at 64 spp) of the whole frame
    float c0, alpha;        // accumulation start value and alpha written to the float buffer: 13 / 255, or 0 / 0 for the
                            //   sample blocks b > 0 of a sample-sharded frame (pt_render_params.sample_blocks)
    int row_begin, row_end; // image rows [row_begin, row_end) are eligible
    int nrows;              // number of (virtual) rows this launch walks (see map_row)
    int stripe_h, rank, nranks;  // row interleave (stripe_h == 0: contiguous rows)
    uint32_t *rgba;
    float4 *accum;          // optional
    uint4 *rng_out;         // optional
    unsigned long long *counters;  // 6 x u64: samples rays shadow tri_tests cells prim_tests
    GridDev grid;
    AnalyticParams ap;             // floor/squares/spheres/lights in kernel-parameter space
    const SceneBlock *gscene;      // global-memory copy of the scene block (shared-memory staging source)
    int scene_bytes;               // bytes of the block actually used (header + prims + ntri records)
    uint32_t scatter_mul;          // persistent kernel: work item w -> (w * scatter_mul) % nitems (0 = identity)
    const uint32_t *tile_order;    // big-grid megakernel: CTA b renders tile tile_order[b] (heavy tiles first); NULL = identity
    uint32_t tiles_x;              //   tiles per row of that launch
    unsigned long long *cta_times; // diagnostics (PT_CTA_TIMES=1, big-grid megakernel): per CTA {start ns, end ns} of globaltimer
    const float4 *vpl;             // bidirectional variant: non-zero VPLs, dense, in buffer order
    const int *nvpl_active;        //   their number (device memory: written by k_compact_vpls)
    // PT_VARIANT_VLPGRID: the raw VPL buffer and the VLP grid (CSR, lists in ascending light order, <= 62 per cell); NULL otherwise
    const float4 *vpl_raw;
    const uint32_t *vg_start, *vg_refs;
    float vg_bmin[3], vg_cell[3];
    int vg_res[3];
    // progressive rendering (pt_launch_pathtracer_range): a range that does not start at sample 0 continues every pixel from
    // the colour sum and RNG state the previous range left (NULL: seed from `seeds`, start at c0); a range that does not end
    // the frame writes the preview ((c - 13) * preview) + 13 into rgba, preview = spp / end (0: the colour itself)
    const float4 *accum_in;
    const uint4 *rng_in;
    float preview;
};

// virtual row -> image row (identity, or the rank's interleaved stripes)
__host__ __device__ inline int map_row(const LaunchArgs &P, int vr) {
    if (P.stripe_h <= 0) return P.row_begin + vr;
    int s = vr / P.stripe_h, o = vr - s * P.stripe_h;
    return P.row_begin + (s * P.nranks + P.rank) * P.stripe_h + o;
}

}  // namespace pt

struct pt_event_s {
    cudaEvent_t start, stop;
    int device;
};

// What has to stay the same over the ranges of one progression (memcmp'ed: built from a zeroed object)
struct pt_progression_key {
    int variant, width, height, spp, arith, row_begin, row_end, row_interleave, rank, nranks;
    uint32_t seeds[4];
    pt_camera cam;
    uint64_t scene_version, grid_version, vpl_version, vlp_grid_version;   // the inputs the variant reads (0: not read)
    int max_bounces;                                                        // pt_set_bounces
};

struct pt_ctx_s {
    int device;
    cudaStream_t stream;
    bool own_stream;
    int sm_count, clock_khz;
    char name[256];

    // scene
    bool scene_set;
    uint64_t scene_version;
    pt::SceneBlock *h_scene[2];   // [PT_ARITH_SEPARATE], [PT_ARITH_FMA] (normals differ)
    pt::SceneBlock *d_scene[2];
    int scene_bytes;
    float mesh_c[3], mesh_r, mesh_k;  // bounding sphere of the brute-force mesh + distance-proportional margin (conservative cull)
    float *d_tris_raw;            // ntri_total x 12 floats (grid build input)
    size_t tris_cap;              // capacity of d_tris_raw in triangles
    int ntri_total;

    // grid
    bool grid_set;
    pt_grid grid_desc;
    pt::GridDev grid;
    uint2 *d_cells;
    uint2 *d_cells_pad;           // the same words inside a one-cell sentinel border (GridDev::cells_pad)
    float4 *d_recs;
    float4 *d_sph;                // per record: bounding sphere of its triangle (sphere prefilter of the traversal)
    uint32_t *gb_kmax;            // bit pattern of max |e0||e2| over the mesh (grid build)
    uint32_t *d_refs;             // capped refs (triangle ids), CSR order
    uint32_t *d_cell_start;       // ncells + 1
    uint64_t total_refs;
    size_t ncells;
    uint32_t *gb_count, *gb_raw_start, *gb_cursor, *gb_bsums, *gb_raw_refs;   // build scratch, kept between builds
    size_t gb_cap[12];            // capacities (bytes) of the five scratch buffers, cell_start, cells, refs, recs

    // VLP grid of CLSuperMetropolisPathTracer_vlpgrid on the context's VLP buffer (pt_build_vlp_grid)
    bool vlp_grid_set;
    pt_grid vlp_grid_desc;
    unsigned *d_vlp_keys;
    uint32_t *d_vlp_cell_start, *d_vlp_refs;
    size_t vlp_keys_cap, vlp_start_cap, vlp_refs_cap, vlp_ncells;
    uint64_t vlp_total_refs;

    // render targets owned by the context
    uint32_t *d_rgba;
    float4 *d_accum;
    uint4 *d_rng;
    size_t rgba_cap, accum_cap, rng_cap;
    uint8_t *h_rgba;              // pinned
    size_t h_rgba_cap;
    unsigned long long *d_counters;
    int last_w, last_h, last_variant;
    int last_kernel;              // PT_KERNEL_* the most recent render resolved to (after PT_KERNEL_AUTO)
    int accum_valid_w, accum_valid_h;   // extent of d_accum the most recent launch wrote (0: it did not request it)
    size_t rng_valid_items;             // work-items of d_rng the most recent launch wrote

    // diffuse bounces per path (pt_set_bounces, DESIGN.md 5b); 0 = the reference's single-vertex sample
    int max_bounces;

    // progressive rendering: d_accum / d_rng hold the state of this progression after its first `prog_next` samples
    bool prog_active;
    int prog_next;
    pt_progression_key prog_key;
    uint64_t grid_version, vpl_version, vlp_grid_version;   // bumped by every grid build, VPL buffer change, VLP grid build

    // bidirectional variant: VPL buffer as the reference defines it + its compacted non-zero entries
    bool vpls_set;
    int nvpl;                     // entries of d_vpls (n_vlp_per_light * nlights)
    float4 *d_vpls, *d_vpl_active;
    uint32_t *d_metro_seed, *d_metro_mutated;   // Metropolis FIX mode: seed paths / mutated paths, n_metro_paths x 20 words each
    size_t metro_cap; int n_metro_paths;
    int *d_vpl_count;
    size_t vpls_cap;              // entries allocated

    // launch order of the big-grid megakernel's tiles (heavy first), cached while the launch geometry stays the same
    uint32_t *d_tile_order, *h_tile_order;
    unsigned long long *d_cta_times, *h_cta_times;   // per CTA {start, end} of globaltimer (ns)
    size_t tile_order_cap;
    unsigned char tile_order_key[192];
    int tile_order_state;         // 0 none, 1 the first launch of the geometry is recording (raster order), 2 sorted from its durations

    // AUTO kernel choice of the brute-force variants: cached estimate of the pixels that scan the mesh
    double mesh_est;
    unsigned char mesh_est_key[96];
    bool mesh_est_valid;

    // wavefront / persistent scratch
    void *d_scratch;
    size_t scratch_cap;
    // wavefront: the ~500 launches of a frame captured once as a CUDA graph and replayed while nothing changes
    cudaGraphExec_t wf_exec;
    pt::LaunchArgs *wf_key_args;   // launch arguments the captured graph was built for (+ variant/arith/scratch below)
    int wf_key_variant, wf_key_fma;
    void *wf_key_scratch;
};

// internal helpers (ptcuda.cu)
int pt_fail(int err, const char *fmt, ...);
int pt_cuda_fail(cudaError_t e, const char *what);
#define PT_CUDA(call, what)                                       \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) return pt_cuda_fail(e__, what);   \
    } while (0)
#define PT_CUDA_NULL(call, what)                                  \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) { pt_cuda_fail(e__, what); return NULL; } \
    } while (0)

int pt_ensure_scratch(pt_ctx ctx, size_t bytes);
// makes the scene block for `arith` current in this device's __constant__ memory (no-op if it already is)
int pt_bind_const_scene(pt_ctx ctx, int arith);

// launchers implemented in the kernel translation units
int pt_launch_mega(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_launch_persistent(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_launch_wavefront(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_launch_grid_tma(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_grid_build_device(pt_ctx ctx, const pt_grid *g);
int pt_vlp_bounds_device(pt_ctx ctx, float vmin[4], float vmax[4]);
int pt_vlp_grid_build_device(pt_ctx ctx, const pt_grid *g);
int pt_launch_stream_grid(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_launch_spec(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_launch_grid_pool(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_launch_bidir(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args);
int pt_launch_bounce(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args, int max_bounces);
int pt_launch_light_tracer_kernels(pt_ctx ctx, int arith, const pt::LaunchArgs &args, int n, float4 *vpl, uint4 *rng_out,
                                   float4 *active, int *count);
