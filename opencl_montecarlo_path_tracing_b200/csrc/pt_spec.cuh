// pt_spec.cuh — PT_KERNEL_SPEC for the brute-force variants (base / lmem): break the per-pixel serial sample chain.
//
// Why.  A pixel draws all its samples from ONE RNG stream (base:220-241), so its 64 samples are a serial chain; a pixel
// that sees the triangle mesh scans 96 triangles for up to three rays per sample — a 1.7 ms chain — and the 512x512 frame
// takes as long as its heaviest pixels: 1.85 ms with 15 of 32 lanes busy (profiles/r1_18), however the pixels are dealt
// out.  But the chain is only an OFFSET into the stream: a sample draws 2 pairs for the camera ray plus, if and only if
// its camera ray hits something, one pair per light (base:168, drawn before any skip).  Where sample k starts is known
// as soon as hit-or-sky of the samples before it is known — and that is the same answer for sample after sample on
// almost every pixel.  So:
//   pass 1, k_spec_light : thread per pixel (8x4 tile per warp) exactly as the megakernel, except that a pixel whose
//       CAMERA ray has to scan the triangles (it passes the mesh's bounding sphere), or whose shadow rays have had to
//       more than a few times, does not: the lane rewinds to the start of that sample and QUEUES the pixel — index,
//       samples done, RNG state, colour sum.  Everything else (floor, sky, spheres, squares, the odd grazing shadow
//       ray: most of the frame) finishes here, cheaply.
//   pass 2, k_spec_heavy : warp per queued pixel.  Lane l takes sample k0 + l and walks the stream to where that sample
//       starts IF the samples before it behave like the last one whose outcome is known (all hit / all sky); all 32
//       samples are traced at once — same pixel, coherent rays, every lane scans the mesh — then one ballot compares
//       predicted and actual outcomes: the samples up to and including the first surprise are valid, their colours are
//       added in order (color = Sample * scale + color is replayed serially with shuffles), the stream continues from
//       the last valid sample's own final state, and the rest of the batch is redone with the corrected prediction.
// Bit-exact by construction: every accepted sample ran from exactly the state the serial order gives it, the colour
// sums are formed in the serial order, counters count accepted samples only.  Interior pixels validate whole batches.
#pragma once
#include "pt_mega.cuh"

namespace pt {

struct SpecEntry {            // 48 bytes
    uint32_t pix, sdone;      // linear pixel index, samples of THIS launch already accumulated (P.spp = the launch's samples)
    float cx, cy;
    float cz, pad0, pad1, pad2;
    uint4 rng;                // state at the start of sample `sdone`
};

// 72 registers / 7 CTAs per SM: at 64 the pass spills inside the sample loop (base 512x512 light pass 0.57 ms, issue slots 58 %,
// long-scoreboard stalls on local memory), at 80 it loses more occupancy than it gains: whole frame 1.05 / 0.87 / 0.92 ms.
template <int VARIANT, bool FMA>
__global__ void __launch_bounds__(128, 7) k_spec_light(const __grid_constant__ LaunchArgs P, SpecEntry *queue, uint32_t *queue_len, int scan_budget) {
    constexpr bool CARRY = VARIANT != PT_VARIANT_BASE;
    const SceneBlock *S = &c_scene;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
    const int vr = blockIdx.y * 8 + (warp >> 1) * 4 + (lane >> 3);
    Counters cnt = {0, 0, 0, 0, 0, 0};
    const int j = map_row(P, vr);
    bool queued = false;
    Rng rng = {0u, 0u, 0u, 0u};
    float cx = P.c0, cy = P.c0, cz = P.c0;
    int s = 0;
    const bool mine = i < P.W && vr < P.nrows && j < P.row_end;
    if (mine) pixel_state_in(P, (uint32_t)(j * P.W + i), rng, cx, cy, cz);
    // Every lane of the warp walks this loop together and re-converges once per sample.  (Written as a per-lane loop with a
    // `break` for the lanes that leave, the base variant's warps never re-converged after their first divergent sample: one
    // 8x4 tile on a sphere's terminator ran its 32 lanes one after the other — 6.9 M cycles, 3.7 ms for the whole pass.)
    bool live = mine;
    int budget = scan_budget;          // triangle scans (shadow rays only) this pixel may run here before it counts as heavy
    for (int it = 0; it < P.spp; ++it) {
        if (live) {
            const Rng rng0 = rng;
            const Counters cnt0 = cnt;
            V3 o, d;
            camera_ray<FMA>(P.cam, rng, i, j, o, d);
            int b = budget;
            V3 c = sample<FMA, CARRY, false, false, true>(P.ap, S, P.grid, o, d, rng, cnt, &b);
            if (b < 0) {                                       // this sample belongs to pass 2: rewind to its start
                rng = rng0; cnt = cnt0; queued = true; live = false;
            } else {
                budget = b;
                cx = Ar<FMA>::madd(c.x, P.scale, cx);
                cy = Ar<FMA>::madd(c.y, P.scale, cy);
                cz = Ar<FMA>::madd(c.z, P.scale, cz);
                ++s;
            }
        }
        __syncwarp();
        if (!__any_sync(0xffffffffu, live)) break;
    }
    if (mine && !queued) pixel_state_out(P, (size_t)j * P.W + i, rng, cx, cy, cz);
    // one warp-aggregated atomicAdd reserves the queue slots of the warp's heavy pixels
    const unsigned qm = __ballot_sync(0xffffffffu, queued);
    if (qm) {
        const int leader = __ffs(qm) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(queue_len, (uint32_t)__popc(qm));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (queued) {
            SpecEntry e;
            e.pix = (uint32_t)(j * P.W + i); e.sdone = (uint32_t)s;
            e.cx = cx; e.cy = cy; e.cz = cz; e.pad0 = e.pad1 = e.pad2 = 0.f;
            e.rng = make_uint4(rng.x0, rng.x1, rng.c0, rng.c1);
            queue[base + __popc(qm & ((1u << lane) - 1u))] = e;
        }
    }
    flush_counters(P, cnt, S->ntri_counted, P.ap.nsq + P.ap.nsp);
}

// Sample() for the 32 samples of one pixel that a warp traces together, in ROUNDS every lane of `lanes` walks: round 0
// the camera rays, round l + 1 the shadow rays towards light l (lanes without one idle).  Per lane the operations and
// the order of its RNG draws are those of sample(); what the rounds add is that the whole group ARRIVES TOGETHER at the
// triangle scan, so tri_loop sees all the lanes that need it — same pixel, coherent rays: usually all of them or none.
// (With sample()'s per-lane ray loop the group reached the scan in pieces of ~11 lanes and scanned once per piece.)
// `keep(hit)` is called by every lane of `lanes` after the camera-ray round and tells the lane whether its sample is part
// of the pixel's chain at all (window mode discards the candidates the chain steps over before they cost shadow rays).
template <bool FMA, bool CARRY, bool CL, class Keep>
PT_DEV V3 sample_rounds(const AnalyticParams &AP, const SceneBlock *S, const GridDev &G, unsigned lanes, bool active, V3 o, V3 d, Rng &rng,
                        Counters &cnt, bool &primary_hit, Keep keep) {
    typedef Ar<FMA> A;
    if (active) cnt.samples++;
    float t = 1e9f, illum = 0.0f, lam = 0.0f;
    V3 ro = o, rd = d, X = o, n = o, out = mk3(0.f, 0.f, 0.f);
    int m = 0;
    bool alive = active;                     // the sample still runs (false after a sky hit)
    bool has_ray = active;                   // this lane traces a ray in the current round
    for (int l = -1; l < AP.nlights; ++l) {
        if (l >= 0) {                        // round l + 1: does this lane send a shadow ray to light l?
            has_ray = false;
            if (alive) {
                float r0, r1;
                rng_next(rng, r0, r1);                                  // drawn before any skip (base:168)
                const float4 L = AP.lights[l];
                if (!(!CARRY && L.w == 0.0f) && !(AP.elide_dead && m == 4)) {   // base:171 only; dead shadow rays: AnalyticParams::elide_dead
                    light_dir<FMA>(L, r0, r1, X, n, rd, lam);
                    if (!(lam < 0.0f)) { ro = X; cnt.shadow++; has_ray = true; }
                }
            }
        }
        // ---- TraceRay for the lanes with a ray; everybody meets at the scan
        int hit = HIT_NONE;
        bool need = false;
        if (has_ray) {
            cnt.rays++;
            if (!CARRY) t = 1e9f;
            trace_analytic<FMA, CARRY>(AP, S, ro, rd, t, hit);
            if (AP.ntri_hint != 0) {
                const float ox = AP.mesh_cx - ro.x, oy = AP.mesh_cy - ro.y, oz = AP.mesh_cz - ro.z;
                const float b = fmaf(oz, rd.z, fmaf(oy, rd.y, ox * rd.x));
                const float oc2 = fmaf(oz, oz, fmaf(oy, oy, ox * ox));
                const float dist2 = oc2 - b * b;
                const float rm = fmaf(AP.mesh_k, fabsf(ox) + fabsf(oy) + fabsf(oz), AP.mesh_r);
                need = !(dist2 > fmaf(rm, rm, 1e-6f * oc2)) && S->ntri > 0;
            }
        }
        __syncwarp(lanes);
        if (AP.ntri_hint != 0) tri_loop<FMA, CL, false>(AP, S, AP.tri_coop != 0, need, ro, rd, t, hit, cnt, lanes);
        __syncwarp(lanes);
        if (l < 0) {
            primary_hit = active && hit != HIT_NONE;
            const bool kept = keep(primary_hit);               // converged: may vote
            if (active) {
                if (hit == HIT_NONE) { out = shade_sky<FMA>(d); alive = false; }
                else {
                    m = hit_material(hit);
                    n = hit_normal<FMA, false>(AP, S, G, hit, o, d, t);
                    X = A::vmadd(d, t, o);
                }
                if (!kept) alive = false;
            }
        } else if (has_ray && hit == HIT_NONE) {
            illum = light_add<FMA>(AP.lights[l], X, lam, illum);
        }
    }
    if (alive) out = shade_material<FMA>(m, illum, X, n, d);
    return out;
}

template <int VARIANT, bool FMA, int MEM, bool CL>
__global__ void __launch_bounds__(128, 6) k_spec_heavy(const __grid_constant__ LaunchArgs P, const SpecEntry *queue, const uint32_t *queue_len,
                                                       uint32_t *next_entry) {
    constexpr bool CARRY = VARIANT != PT_VARIANT_BASE;
    typedef Ar<FMA> A;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SceneBlock *S = (MEM == PT_SCENE_SMEM) ? stage_scene_smem(P, smem_raw) : &c_scene;
    const unsigned lane = threadIdx.x & 31;
    Counters cnt = {0, 0, 0, 0, 0, 0};
    const uint32_t n = *queue_len;
    for (;;) {
        uint32_t e = 0;
        if (lane == 0) e = atomicAdd(next_entry, 1u);              // dynamic: heavy pixels differ a lot in what is left to do
        e = __shfl_sync(0xffffffffu, e, 0);
        if (e >= n) break;
        const SpecEntry E = queue[e];
        const int j = (int)(E.pix / (uint32_t)P.W), i = (int)(E.pix - (uint32_t)j * (uint32_t)P.W);
        Rng base;
        base.x0 = E.rng.x; base.x1 = E.rng.y; base.c0 = E.rng.z; base.c1 = E.rng.w;
        float cx = E.cx, cy = E.cy, cz = E.cz;
        int k0 = (int)E.sdone;
        // Two ways to place 32 lanes on the stream (a sample draws 2 pairs, plus nlights more if its camera ray hits):
        //  RUN    : lane l = sample k0 + l, assuming the samples before it all end like the last known one (`pred`): a whole
        //           batch of 32 samples per pass while that holds; the first surprise invalidates the lanes behind it.
        //  WINDOW : after a surprise (silhouette pixels, blurred by the lens, alternate between hit and sky): lane l = the
        //           CANDIDATE sample that would start g * l pairs into the stream, g = gcd of the two step sizes — every
        //           place a sample can start.  All candidates trace their camera ray; the outcomes then say which candidates
        //           the chain really visits (0, then +2/g or +(2+nlights)/g lanes ...), and only those go on to their shadow
        //           rays.  No prediction, 16-32 samples per pass; a window whose samples all end alike returns to RUN.
        bool pred = true;                                          // the sample that queued the pixel passes the mesh: expect hits
        bool window = false;
        const int nl = P.ap.nlights;
        const int g = (nl & 1) ? 1 : 2, step_miss = 2 / g, step_hit = (2 + nl) / g;
        while (k0 < P.spp) {
            const int left = P.spp - k0;
            Rng r = base;
            Counters lc = {0, 0, 0, 0, 0, 0};
            bool hit = false;
            V3 o = mk3(0.f, 0.f, 0.f), d = o, c;
            unsigned valid;                                        // lanes whose samples are part of the chain, in lane order
            if (!window) {
                const int nb = min(32, left);
                const bool active = (int)lane < nb;
                const int stride = 2 + (pred ? nl : 0);
                for (int q = (int)lane * stride; q > 0; --q) rng_skip(r);
                if (active) camera_ray<FMA>(P.cam, r, i, j, o, d);
                __syncwarp();
                c = sample_rounds<FMA, CARRY, CL>(P.ap, S, P.grid, 0xffffffffu, active, o, d, r, lc, hit, [](bool) { return true; });
                const unsigned act = nb == 32 ? 0xffffffffu : ((1u << nb) - 1u);
                const unsigned hits = __ballot_sync(0xffffffffu, hit);
                const unsigned wrong = (hits ^ (pred ? act : 0u)) & act;
                const int nvalid = wrong ? __ffs(wrong) : nb;      // up to and including the first surprise
                valid = nvalid == 32 ? 0xffffffffu : ((1u << nvalid) - 1u);
                pred = (hits >> (nvalid - 1)) & 1u;
                window = wrong != 0u;
            } else {
                for (int q = (int)lane * g; q > 0; --q) rng_skip(r);
                camera_ray<FMA>(P.cam, r, i, j, o, d);
                __syncwarp();
                unsigned visited = 0u, vhits = 0u;
                c = sample_rounds<FMA, CARRY, CL>(P.ap, S, P.grid, 0xffffffffu, true, o, d, r, lc, hit, [&](bool h) {
                    const unsigned hits = __ballot_sync(0xffffffffu, h);
                    int pos = 0, count = 0;
                    while (pos < 32 && count < left) {             // warp-uniform: follow the chain through the window
                        visited |= 1u << pos;
                        ++count;
                        pos += ((hits >> pos) & 1u) ? step_hit : step_miss;
                    }
                    vhits = hits & visited;
                    return ((visited >> lane) & 1u) != 0u;
                });
                valid = visited;
                const int last = 31 - __clz((int)visited);
                pred = (vhits >> last) & 1u;
                window = !(vhits == 0u || vhits == visited);       // all alike: predictable again
            }
            if ((valid >> lane) & 1u) { cnt.rays += lc.rays; cnt.shadow += lc.shadow; cnt.samples += lc.samples; }
            cnt.btests += lc.btests;                               // executed work, discarded samples included
            // color = Sample * scale + color, in sample order (base:238)
            for (unsigned m = valid; m; m &= m - 1u) {
                const int q = __ffs((int)m) - 1;
                const float qx = __shfl_sync(0xffffffffu, c.x, q), qy = __shfl_sync(0xffffffffu, c.y, q), qz = __shfl_sync(0xffffffffu, c.z, q);
                cx = A::madd(qx, P.scale, cx);
                cy = A::madd(qy, P.scale, cy);
                cz = A::madd(qz, P.scale, cz);
            }
            const int lastv = 31 - __clz((int)valid);
            base.x0 = __shfl_sync(0xffffffffu, r.x0, lastv); base.x1 = __shfl_sync(0xffffffffu, r.x1, lastv);
            base.c0 = __shfl_sync(0xffffffffu, r.c0, lastv); base.c1 = __shfl_sync(0xffffffffu, r.c1, lastv);
            k0 += __popc(valid);
        }
        if (lane == 0) pixel_state_out(P, E.pix, base, cx, cy, cz);
    }
    flush_counters(P, cnt, S->ntri_counted, P.ap.nsq + P.ap.nsp);
}

template <int VARIANT, bool FMA, int MEM>
static int launch_spec(pt_ctx ctx, const LaunchArgs &args_in) {
    LaunchArgs args = args_in;
    args.ap.tri_coop = MEM == PT_SCENE_SMEM;                       // few lanes need the scan -> cooperative; (nearly) all -> lane-serial (tri_loop decides)
    const size_t npix = (size_t)args.W * args.nrows;
    const size_t qbytes = 256 + npix * sizeof(SpecEntry);
    if (pt_ensure_scratch(ctx, qbytes)) return 1;
    uint32_t *counters = (uint32_t *)ctx->d_scratch;               // [0] queue length, [1] next entry
    SpecEntry *queue = (SpecEntry *)((char *)ctx->d_scratch + 256);
    PT_CUDA(cudaMemsetAsync(counters, 0, 8, ctx->stream), "clear queue counters");
    dim3 grid((args.W + 15) / 16, (args.nrows + 7) / 8), block(128);
    static int budget = -1;
    if (budget < 0) { const char *e = getenv("PT_SPEC_BUDGET"); budget = e ? atoi(e) : 0; }
    k_spec_light<VARIANT, FMA><<<grid, block, 0, ctx->stream>>>(args, queue, counters, budget);
    PT_CUDA(cudaGetLastError(), "launch k_spec_light");
    const size_t smem = MEM == PT_SCENE_SMEM ? (size_t)args.scene_bytes : 0;
    const bool cl = args.ap.ncl > 0;
    auto kern = cl ? k_spec_heavy<VARIANT, FMA, MEM, true> : k_spec_heavy<VARIANT, FMA, MEM, false>;
    if (smem > 48 * 1024) PT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "opt-in shared memory");
    int per_sm = 0;
    PT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 128, smem), "occupancy query");
    if (per_sm < 1) per_sm = 1;
    uint32_t blocks = (uint32_t)(ctx->sm_count * per_sm);
    const uint32_t need_blocks = (uint32_t)((npix + 3) / 4);
    if (blocks > need_blocks) blocks = need_blocks;
    kern<<<blocks, 128, smem, ctx->stream>>>(args, queue, counters, counters + 1);
    PT_CUDA(cudaGetLastError(), "launch k_spec_heavy");
    return 0;
}

}  // namespace pt

int pt_launch_spec(pt_ctx ctx, const pt_render_params *p, const pt::LaunchArgs &args) {
    using namespace pt;
    if (p->variant != PT_VARIANT_BASE && p->variant != PT_VARIANT_LMEM)
        return pt_fail(1, "PT_KERNEL_SPEC applies to the brute-force variants (base, lmem) only");
    const bool fma = p->arith != PT_ARITH_SEPARATE;
    int rc = pt_bind_const_scene(ctx, fma ? PT_ARITH_FMA : PT_ARITH_SEPARATE);     // pass 1 (and CONST pass 2) read the __constant__ scene
    if (rc) return rc;
    const bool smem = p->scene_mem == PT_SCENE_SMEM;
    if (p->variant == PT_VARIANT_BASE) {
        if (fma) return smem ? launch_spec<PT_VARIANT_BASE, true, PT_SCENE_SMEM>(ctx, args) : launch_spec<PT_VARIANT_BASE, true, PT_SCENE_CONST>(ctx, args);
        return smem ? launch_spec<PT_VARIANT_BASE, false, PT_SCENE_SMEM>(ctx, args) : launch_spec<PT_VARIANT_BASE, false, PT_SCENE_CONST>(ctx, args);
    }
    if (fma) return smem ? launch_spec<PT_VARIANT_LMEM, true, PT_SCENE_SMEM>(ctx, args) : launch_spec<PT_VARIANT_LMEM, true, PT_SCENE_CONST>(ctx, args);
    return smem ? launch_spec<PT_VARIANT_LMEM, false, PT_SCENE_SMEM>(ctx, args) : launch_spec<PT_VARIANT_LMEM, false, PT_SCENE_CONST>(ctx, args);
}
