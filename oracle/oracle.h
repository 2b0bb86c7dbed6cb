/*
 * oracle.h — CPU restatement of the reference's CLSuperPathTracer hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may build, load or call this.  The product
 * library (opencl_montecarlo_path_tracing_b200/csrc) never links or calls it.
 *
 * PARITY PIN: this restatement is pinned against the reference ITSELF — the
 * unmodified reference host .c and kernel .ocl compiled from /root/reference
 * through oracle/refrt (see oracle/Makefile `ref`).  tests/test_oracle_vs_ref.py
 * checks result.ppm byte-equality for all five variants in this container, and
 * tests/golden/ holds vectors generated from that reference build (script
 * committed) so the pin travels to machines without /root/reference.
 *
 * Variants (reference directories):
 *   0 base   CLSuperPathTracer/            t reset in TraceRay, zero-intensity light skip
 *   1 lmem   CLSuperPathTracer_lmem/       running t bound, floor test `r < t`
 *   2 nodof  CLSuperPathTracer_lmem_NoDoF/ lmem semantics, 1 work-item per sample + 8x8 tree reduce
 *   3 grid   CLSuperPathTracer_trianglegrid/ lmem semantics, triangles through the uniform grid (DDA)
 *   4 bidir  CLSuperBidirectionalPathTracer/ lmem TraceRay; lightTracer kernel deposits virtual point lights
 *            (VPLs), Sample gathers all of them unshadowed, then SUBTRACTS 1/nlights per occluded real light
 *   5 vlpgrid  kernel pathTracer of CLSuperMetropolisPathTracer_vlpgrid/metropolispathtracer.ocl:649-684 with its Sample
 *            (:296-386): the bidir Sample, except that the gather visits only the VPLs listed in the VLP-grid cell that
 *            contains the hit point (no zero-intensity skip, linear cell index without per-axis range checks).  The VPL
 *            buffer (vpls/nvpl) and the VLP grid (box_min, grid_res, cell_size, cell_start/cell_refs in CSR form, lists in
 *            ascending light order, <= 62 per cell) are inputs.
 *
 * Arithmetic policy (compile-time PT_CONTRACT):
 *   0  every float operation individually rounded (what g++ makes of the reference .ocl; image bytes
 *      identical to oracle/_ref; pow(x,4) is the correctly rounded x^4 where glibc's powf, which _ref
 *      uses, may be 1 ulp off for ~1e-5 of the sky samples);
 *   1  fused multiply-adds exactly where the CUDA kernels place __fmaf_rn (DESIGN.md "contraction
 *      contract"), pow(x,4) as (x*x)*(x*x): bit-exact target for the CUDA path.  Both are legal
 *      OpenCL C behaviours (FP_CONTRACT is ON by default; pow has a 16-ulp budget).
 */
#ifndef PT_ORACLE_H
#define PT_ORACLE_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { ORACLE_BASE = 0, ORACLE_LMEM = 1, ORACLE_NODOF = 2, ORACLE_GRID = 3, ORACLE_BIDIR = 4, ORACLE_VLPGRID = 5 };

typedef struct {
    uint64_t samples;        /* Sample() calls                         */
    uint64_t rays;           /* TraceRay() calls (primary + shadow)    */
    uint64_t shadow_rays;    /* of which shadow rays                   */
    uint64_t tri_tests;      /* Moller-Trumbore evaluations started    */
    uint64_t cells_visited;  /* grid cells loaded by the DDA           */
    uint64_t prim_tests;     /* square + sphere tests (set bits)       */
} oracle_counters;

typedef struct {
    int32_t variant;
    int32_t width, height;
    int32_t spp;             /* 64 = reference; other values: documented extension (scale 224/spp) */
    int32_t row_begin, row_end; /* rows [row_begin,row_end) are rendered; others left untouched */
    uint32_t seeds[4];
    int32_t spheres[9];
    int32_t squares[9];
    const float *triangles;  /* ntriangles x 12 floats: v0.xyzw v1.xyzw v2.xyzw (w = 0) */
    int32_t ntriangles;
    float lights[5][4];      /* x y z intensity */
    int32_t nlights;
    float cam_up[4], cam_right[4], eye_offset[4];
    /* grid variant only */
    float box_min[4], box_max[4];
    int32_t grid_res[4];
    float cell_size[4];
    const uint32_t *cell_start; /* ncells+1 offsets into cell_refs */
    const uint32_t *cell_refs;  /* triangle ids, per cell in triangle-id order, <= 62 per cell */
    int32_t nthreads;           /* 0 = OpenMP default */
    /* bidir variant only: the buffer lightTracer filled, nvpl x (x y z intensity), in buffer order */
    const float *vpls;
    int32_t nvpl;
    /* sample-range sharding (ptcuda.h pt_render_params.sample_block/sample_blocks): block b of R renders spp/R
     * samples, scale 224/spp, seeds ^ randomizeId(b) and start value 0 / alpha 0 for b > 0.  0 or 1 = off. */
    int32_t sample_block, sample_blocks;
} oracle_job;

/* Outputs may be NULL.  rgba8: W*H*4 bytes.  accum: W*H*4 floats (the value handed to
 * convert_uchar4, w = 255).  rng_state: final {x.x,x.y,c.x,c.y} per work-item (W*H for variants
 * 0,1,3; 64*W*H in the 8W x 8H work-item order for nodof).  Returns 0, or -1 on bad arguments. */
int oracle_render(const oracle_job *job, uint8_t *rgba8, float *accum, uint32_t *rng_state,
                  oracle_counters *counters);
/* OpenMP team size the most recent oracle_render really ran with (1 without OpenMP) */
int oracle_threads_used(void);

/* Kernel lightTracer of CLSuperBidirectionalPathTracer/bidirectionalpathtracer.ocl:280-326 for a 1-D range of
 * n_vlp_per_light work-items (scene, lights and seeds from `job`; its variant/size fields are ignored).
 * vpl_out: n_vlp_per_light*nlights x 4 floats, entry [gi + l*n_vlp_per_light] as in the reference (:324).
 * rng_state (optional): final RNG state per work-item.  Returns 0, -1 on bad arguments. */
int oracle_light_tracer(const oracle_job *job, int n_vlp_per_light, float *vpl_out, uint32_t *rng_state,
                        oracle_counters *counters);

/* Kernels lightTracer + MetropolisLightTracer of CLSuperMetropolisPathTracer(_vlpgrid)/metropolispathtracer.ocl in FIX mode
 * (VerifyIntersection's uninitialised hit bound = 1e9, seed paths in their own buffer; see oracle.c).  paths_out (optional):
 * n_paths*nlights x 20 words in the reference's Path layout; vpl_out: 4*n_paths*nlights x 4 floats.  0, or -1 on bad arguments. */
int oracle_metropolis_light_tracer(const oracle_job *job, int n_paths, int mutation_rounds, uint32_t *paths_out, float *vpl_out);

int oracle_metropolis_mutate(const oracle_job *job, uint32_t gid, const float origin[3], uint32_t path[20], int rounds);

/* policy this library was built with (0 / 1) */
int oracle_contract_mode(void);

/* RNG known-answer helper: seeds for work-item gid, then nsteps draws (2 floats each). */
void oracle_rng_kat(const uint32_t seeds[4], uint32_t gid, int nsteps, float *out_f, uint32_t *out_u32,
                    uint32_t out_state[4]);
uint32_t oracle_randomize_id(uint32_t id);

/* Single-ray probe of TraceRay for brute-force variants (carry = 0: base semantics, 1: lmem). */
int oracle_trace_ray(int carry, const float o[3], const float d[3], float *t_inout, float n_out[3],
                     const int32_t spheres[9], const int32_t squares[9], const float *tris12, int ntris);
/* TraceRay on n rays (o, d: n x 3 floats) with the scene of `job`: job->variant ORACLE_BASE (t reset per call), ORACLE_GRID
 * (triangles through job's uniform grid, set up as for oracle_render) or any other (lmem semantics, brute force).  t_inout is
 * each ray's carried hit bound and receives its final t.  Optional outputs per ray: material m_out, normal n_out (n x 3, zero
 * on a miss), grid cells the walk visited (cells_out) and Moller-Trumbore tests started (tests_out).  0, or -1 on bad arguments. */
int oracle_trace_rays(const oracle_job *job, int n, const float *o, const float *d, float *t_inout, int32_t *m_out,
                      float *n_out, uint32_t *cells_out, uint32_t *tests_out);

/* ---- host-side restatements (oracle_host.c) ---- */
/* CLSuperPathTracer.c:236-243 */
void oracle_camera(float cam_forward[4], float cam_up[4], float cam_right[4], float eye_offset[4]);
/* CLSuperPathTracer.c:62-74.  Returns number of lines consumed (<= 9), -1 if the file cannot be opened. */
int oracle_parse_array(const char *path, int32_t arr[9]);
/* CLSuperPathTracer.c:77-118 (+ bbox of ..._trianglegrid/CLSuperPathTracer.c:136-209 when box != NULL).
 * tris12 must hold max_triangles*12 floats. */
int oracle_parse_triangles(const char *path, float *tris12, int max_triangles, float box_min[4], float box_max[4]);
/* CLSuperPathTracer.c:121-139 */
int oracle_parse_lights(const char *path, float lights[5][4]);
/* ..._trianglegrid/CLSuperPathTracer.c:476-484 */
void oracle_grid_dims(const float box_min[4], const float box_max[4], int ntriangles, float cell_size_modifier,
                      int32_t grid_res[4], float cell_size[4]);
/* Deterministic grid binning: the cell set of the device kernel (pathtracer.ocl:311-330), entries in
 * triangle-id order as in initTrianglesGrid_host (..._trianglegrid/CLSuperPathTracer.c:233-265),
 * at most `cap` (62) per cell.  Pass cell_refs = NULL to only count: cell_start then receives the
 * ncells+1 offsets.  Returns total refs stored. */
uint64_t oracle_build_grid(const float *tris12, int ntris, const float box_min[4], const int32_t grid_res[4],
                           const float cell_size[4], int cap, uint32_t *cell_start, uint32_t *cell_refs);
/* CLSuperMetropolisPathTracer_vlpgrid: VLP bounding box (kernels reduceMinAndMax_lmem + _nwg, metropolispathtracer.ocl:538-619)
 * and VLP grid (kernel initVLPsGrid, :621-647; ascending light indices per cell, at most `cap`).  The grid's resolution is
 * oracle_grid_dims(vmin, vmax, n_vlp, modifier) (CLSuperMetropolisPathTracer.c:628-636). */
void oracle_vlp_bounds(const float *vpl4, int n, float vmin[4], float vmax[4]);
uint64_t oracle_build_vlp_grid(const float *vpl4, int n, const float box_min[4], const int32_t grid_res[4], const float cell_size[4],
                               int cap, uint32_t *cell_start, uint32_t *cell_refs);
/* pamalign.h:212-238 */
int oracle_save_pam(const char *path, int width, int height, const uint8_t *rgba8);

#ifdef __cplusplus
}
#endif
#endif
