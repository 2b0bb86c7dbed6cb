/*
 * oracle_paths.h — CPU restatement of the opt-in diffuse bounces (include/ptcuda.h, DESIGN.md 5b).
 *
 * TEST INFRASTRUCTURE ONLY, like oracle/: only tests/ and tools/ may build, load or call this; the product library never
 * links it.  oracle_paths.c compiles oracle/oracle.c into the same translation unit and builds the path on the oracle's own
 * TraceRay, Sample pieces and RNG, so a path of zero bounces IS the oracle's sample.  Same two arithmetic policies
 * (PT_CONTRACT 0 / 1, liboracle_paths.so / liboracle_paths_fma.so), with the fused multiply-adds of the bounce arithmetic
 * where the CUDA kernel places them (DESIGN.md "contraction contract").
 */
#ifndef PT_ORACLE_PATHS_H
#define PT_ORACLE_PATHS_H

#include "../oracle/oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
    uint64_t bounce_rays;        /* bounce rays traced                                                          */
    uint64_t rr_terminations;    /* paths ended by Russian roulette                                             */
    uint64_t tmin_rejections;    /* square / triangle hits a bounce ray refused for r <= 0.01 (the reference's  */
                                 /*   bounds would have taken them)                                             */
    uint64_t disk_exhausted;     /* paths ended because 32 disk draws all missed                                */
} oracle_path_counters;

/* oracle_render for variants base, lmem and grid with max_bounces (0..15) bounces per path; the same job fields (rows,
 * sample blocks, threads) and outputs.  max_bounces = 0 runs the same code and gives oracle_render's results.
 * path_counters may be NULL.  0, or -1 on bad arguments. */
int oracle_render_bounces(const oracle_job *job, int max_bounces, uint8_t *rgba8, float *accum, uint32_t *rng_state,
                          oracle_counters *counters, oracle_path_counters *path_counters);

/* One path from origin o along d (vertex 0 = the reference's Sample for that ray), with job's scene and variant (base, lmem,
 * grid).  rng_state: 4 words {x.x, x.y, c.x, c.y}, advanced in place.  rr_enabled = 0 switches Russian roulette off (paths
 * run to max_bounces; a test switch for checking that roulette is unbiased, never used by the product).  out_rgb: L.
 * counters / path_counters (may be NULL) are ADDED to.  0, or -1 on bad arguments. */
int oracle_path_sample(const oracle_job *job, const float o[3], const float d[3], uint32_t rng_state[4], int max_bounces,
                       int rr_enabled, float out_rgb[3], oracle_counters *counters, oracle_path_counters *path_counters);

/* oracle_path_sample for n paths with the same origin and direction, from n RNG states (n x 4 words, advanced in place);
 * out_rgb: n x 3.  Runs on OpenMP threads.  0, or -1 on bad arguments. */
int oracle_path_samples(const oracle_job *job, int n, const float o[3], const float d[3], uint32_t *rng_states, int max_bounces,
                        int rr_enabled, float *out_rgb, oracle_path_counters *path_counters);

#ifdef __cplusplus
}
#endif
#endif
