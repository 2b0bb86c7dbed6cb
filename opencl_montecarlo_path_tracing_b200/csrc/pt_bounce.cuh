// pt_bounce.cuh — opt-in diffuse bounces with Russian roulette (DESIGN.md 5b) for the base, lmem and trianglegrid variants.
//
//  k_bounce_pixel : k_mega_pixel's layout (one thread per pixel, its whole sample sequence; a warp covers an 8x4 pixel tile,
//                   a CTA 16x8 pixels) with sample_bounces() in place of sample().  Launched in raster order: the
//                   longest-tile-first table of the big-grid megakernel is neither read nor recorded, so the reference
//                   mode's launch order is not disturbed by frames with bounces.  max_bounces = 0 never reaches it.
#pragma once

#include "pt_host.h"

// Registers: the path adds a throughput, a colour sum, the vertex's incoming direction and its depth to sample()'s state.
// 128 threads and at least 6 CTAs per SM (80 registers, no spills); big grids 8 CTAs (64 registers, 132 / 112-116 bytes of
// spill stores / loads), as k_mega_pixel.  Measured on a B200 (tools/bounce_time.py, B = 1, DESIGN.md 5b): 1 M-triangle soup
// 387 ms with 6 CTAs, 342 ms with 8; default brute-force scene at 512x512 1.26-1.34 ms with 6, 1.30 ms with 8.

namespace pt {

// BIG: brute-force variants — per-cluster triangle culling compiled in (tri_loop<.., CL>), as in k_mega_pixel; trianglegrid —
// a grid above 16 k triangles (the same instantiation split as k_mega_pixel).
template <int VARIANT, bool FMA, int MEM, bool BIG>
__global__ void __launch_bounds__(128, (BIG && VARIANT == PT_VARIANT_GRID) ? 8 : 6) k_bounce_pixel(const __grid_constant__ LaunchArgs P,
                                                                                                   int max_bounces) {
    constexpr bool CARRY = VARIANT != PT_VARIANT_BASE;
    constexpr bool GRID = VARIANT == PT_VARIANT_GRID;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SceneBlock *S = (MEM == PT_SCENE_SMEM) ? stage_scene_smem(P, smem_raw) : &c_scene;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // 16x8 pixel tile: 2x2 warps of 8x4 pixels
    const int i = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
    const int vr = blockIdx.y * 8 + (warp >> 1) * 4 + (lane >> 3);
    Counters cnt = {0, 0, 0, 0, 0, 0};
    const int j = map_row(P, vr);
    if (i < P.W && vr < P.nrows && j < P.row_end) {
        Rng rng;
        float cx, cy, cz;
        pixel_state_in(P, (uint32_t)(j * P.W + i), rng, cx, cy, cz);
        for (int s = 0; s < P.spp; ++s) {
            V3 o, d;
            camera_ray<FMA>(P.cam, rng, i, j, o, d);
            const V3 c = sample_bounces<FMA, CARRY, GRID, BIG && !GRID>(P.ap, S, P.grid, o, d, rng, cnt, max_bounces);
            cx = Ar<FMA>::madd(c.x, P.scale, cx);
            cy = Ar<FMA>::madd(c.y, P.scale, cy);
            cz = Ar<FMA>::madd(c.z, P.scale, cz);
        }
        pixel_state_out(P, (size_t)j * P.W + i, rng, cx, cy, cz);
    }
    if (GRID) cnt.btests = cnt.gtri;        // trace_grid tests every record of the cells it visits
    flush_counters(P, cnt, GRID ? 0 : S->ntri_counted, P.ap.nsq + P.ap.nsp);
}

template <int VARIANT, bool FMA, int MEM, bool BIG>
static int launch_bounce_b(pt_ctx ctx, const LaunchArgs &args_in, int max_bounces) {
    LaunchArgs args = args_in;
    args.ap.tri_coop = MEM == PT_SCENE_SMEM;
    const dim3 grid((args.W + 15) / 16, (args.nrows + 7) / 8), block(128);
    const size_t smem = MEM == PT_SCENE_SMEM ? (size_t)args.scene_bytes : 0;
    if (smem > 48 * 1024)
        PT_CUDA(cudaFuncSetAttribute(k_bounce_pixel<VARIANT, FMA, MEM, BIG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                "opt-in shared memory");
    k_bounce_pixel<VARIANT, FMA, MEM, BIG><<<grid, block, smem, ctx->stream>>>(args, max_bounces);
    PT_CUDA(cudaGetLastError(), "launch k_bounce_pixel");
    return 0;
}

template <int VARIANT, bool FMA, int MEM>
static int launch_bounce_v(pt_ctx ctx, const LaunchArgs &args, int max_bounces) {
    if (VARIANT == PT_VARIANT_GRID ? ctx->ntri_total > 16384 : args.ap.ncl > 0) return launch_bounce_b<VARIANT, FMA, MEM, true>(ctx, args, max_bounces);
    return launch_bounce_b<VARIANT, FMA, MEM, false>(ctx, args, max_bounces);
}

template <bool FMA, int MEM>
static int launch_bounce_am(pt_ctx ctx, int variant, const LaunchArgs &args, int max_bounces) {
    switch (variant) {
        case PT_VARIANT_BASE: return launch_bounce_v<PT_VARIANT_BASE, FMA, MEM>(ctx, args, max_bounces);
        case PT_VARIANT_LMEM: return launch_bounce_v<PT_VARIANT_LMEM, FMA, MEM>(ctx, args, max_bounces);
        case PT_VARIANT_GRID: return launch_bounce_v<PT_VARIANT_GRID, FMA, MEM>(ctx, args, max_bounces);
    }
    return pt_fail(1, "render: diffuse bounces are defined for the base, lmem and trianglegrid variants only");
}

}  // namespace pt

int pt_launch_bounce(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args, int max_bounces) {
    using namespace pt;
    const bool fma = p->arith != PT_ARITH_SEPARATE;
    if (p->scene_mem == PT_SCENE_SMEM)
        return fma ? launch_bounce_am<true, PT_SCENE_SMEM>(ctx, p->variant, args, max_bounces)
                   : launch_bounce_am<false, PT_SCENE_SMEM>(ctx, p->variant, args, max_bounces);
    int rc = pt_bind_const_scene(ctx, fma ? PT_ARITH_FMA : PT_ARITH_SEPARATE);
    if (rc) return rc;
    return fma ? launch_bounce_am<true, PT_SCENE_CONST>(ctx, p->variant, args, max_bounces)
               : launch_bounce_am<false, PT_SCENE_CONST>(ctx, p->variant, args, max_bounces);
}
