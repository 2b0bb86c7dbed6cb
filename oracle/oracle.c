/*
 * oracle.c — scalar-float C restatement of the CLSuperPathTracer device code.
 * TEST INFRASTRUCTURE ONLY — see oracle.h for who may use it and how it is pinned.
 *
 * Every function cites the reference lines it follows (paths relative to /root/reference).
 * "base"  = CLSuperPathTracer/pathtracer.ocl
 * "lmem"  = CLSuperPathTracer_lmem/pathtracer.ocl
 * "nodof" = CLSuperPathTracer_lmem_NoDoF/pathtracer.ocl
 * "grid"  = CLSuperPathTracer_trianglegrid/pathtracer.ocl
 * "bidir" = CLSuperBidirectionalPathTracer/bidirectionalpathtracer.ocl
 */
#include "oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#ifndef PT_CONTRACT
#define PT_CONTRACT 0
#endif

/* ------------------------------------------------------------ arithmetic policy */
#if PT_CONTRACT
static inline float MADD(float a, float b, float c) { return fmaf(a, b, c); } /* a*b + c, one rounding */
static inline float MSUB(float a, float b, float c, float d) { return fmaf(a, b, -(c * d)); } /* a*b - c*d */
static inline float POW4(float x) { float x2 = x * x; return x2 * x2; }
#else
static inline float MADD(float a, float b, float c) { return a * b + c; }
static inline float MSUB(float a, float b, float c, float d) { return a * b - c * d; }
/* pow(1-d.z, 4): the product is formed in double and rounded ONCE to float, i.e. the correctly rounded
 * x^4.  glibc's powf (what g++ gives the reference .ocl) is within 0.82 ulp of that and equal to it for all
 * but ~1e-5 of the arguments; OpenCL allows pow 16 ulp, so this is one legal reference behaviour. */
static inline float POW4(float x) { double xd = (double)x; return (float)(xd * xd * xd * xd); }
#endif

int oracle_contract_mode(void) { return PT_CONTRACT; }

typedef struct { float x, y, z; } V3;

static inline V3 v3(float x, float y, float z) { V3 r = {x, y, z}; return r; }
static inline V3 vsub(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline V3 vscale(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
/* a*s + b per component */
static inline V3 vmadd(V3 a, float s, V3 b) { return v3(MADD(a.x, s, b.x), MADD(a.y, s, b.y), MADD(a.z, s, b.z)); }
/* dot(): x,y,z summed left to right (w lanes are 0 in the reference) */
static inline float dot3(V3 a, V3 b) { return MADD(a.z, b.z, MADD(a.y, b.y, a.x * b.x)); }
static inline V3 cross3(V3 a, V3 b) {
    return v3(MSUB(a.y, b.z, a.z, b.y), MSUB(a.z, b.x, a.x, b.z), MSUB(a.x, b.y, a.y, b.x));
}
/* base:44-46  Normalize(x) = (1/sqrt(dot(x,x))) * x */
static inline V3 normalize3(V3 a) { float s = 1.0f / sqrtf(dot3(a, a)); return vscale(a, s); }

/* OpenCL fmin/fmax: NaN-ignoring */
static inline float cl_fmin(float x, float y) { if (x != x) return y; if (y != y) return x; return y < x ? y : x; }
static inline float cl_fmax(float x, float y) { if (x != x) return y; if (y != y) return x; return x < y ? y : x; }
/* convert_int / (int) cast: truncation; out-of-range saturates, NaN -> 0 (GPU behaviour) */
static inline int f2i_rz_sat(float f) {
    if (f != f) return 0;
    if (f >= 2147483648.0f) return 2147483647;
    if (f <= -2147483648.0f) return (-2147483647 - 1);
    return (int)f;
}
static inline uint8_t f2u8_rz_sat(float f) {
    if (f != f) return 0;
    if (f >= 255.0f) return 255;
    if (f <= 0.0f) return 0;
    return (uint8_t)(int)f;
}

/* ------------------------------------------------------------------------- RNG */
typedef struct { uint32_t x0, x1, c0, c1; } Rng;

/* base:26-34 */
uint32_t oracle_randomize_id(uint32_t id) {
    id = (id ^ 61u) ^ (id >> 16);
    id *= 9u;
    id = id ^ (id >> 4);
    id *= 0x27d4eb2du;
    id = id ^ (id >> 15);
    return id;
}

/* base:37-41 — the same hash is XOR-ed into all four words */
static inline Rng rng_seed(const uint32_t seeds[4], uint32_t gid) {
    uint32_t h = oracle_randomize_id(gid);
    Rng r = {seeds[0] ^ h, seeds[1] ^ h, seeds[2] ^ h, seeds[3] ^ h};
    return r;
}

/* base:12-23.  Per lane: res = x^c; hi = mul_hi(x,A); x = x*A + c; c = hi + (x < c ? 0xFFFFFFFF : 0)
 * — vector compare yields -1, convert_uint2 wraps, so the "carry" ADDS 0xFFFFFFFF (not 1).
 * Returned value: 0.0f + float(res) * ((1.0f - 0.0f) / 4294967295) where the integer literal is a
 * 64-bit long that converts to 2^32 as float, i.e. float(res) * 2^-32 (round-to-nearest-even cvt). */
static inline void rng_next(Rng *s, float *u0, float *u1, uint32_t *raw0, uint32_t *raw1) {
    const uint32_t A = 4294883355u;
    uint32_t r0 = s->x0 ^ s->c0, r1 = s->x1 ^ s->c1;
    uint32_t hi0 = (uint32_t)(((uint64_t)s->x0 * A) >> 32), hi1 = (uint32_t)(((uint64_t)s->x1 * A) >> 32);
    uint32_t nx0 = s->x0 * A + s->c0, nx1 = s->x1 * A + s->c1;
    uint32_t nc0 = hi0 + (nx0 < s->c0 ? 0xFFFFFFFFu : 0u), nc1 = hi1 + (nx1 < s->c1 ? 0xFFFFFFFFu : 0u);
    s->x0 = nx0; s->x1 = nx1; s->c0 = nc0; s->c1 = nc1;
    const float scale = (1.0f - 0.0f) / 4294967296.0f;
    *u0 = 0.0f + (float)r0 * scale;
    *u1 = 0.0f + (float)r1 * scale;
    if (raw0) *raw0 = r0;
    if (raw1) *raw1 = r1;
}

/* bidir:12-23 with the limits (-1, 1) of bidir:320: (1 - -1)/4294967295 -> 2^-31; the product is exact, the
 * addition of -1 rounds once (so a contracted fma gives the same value). */
static inline void rng_next_pm1(Rng *s, float *u0, float *u1) {
    float a, b; uint32_t r0, r1;
    rng_next(s, &a, &b, &r0, &r1);
    const float scale = (1.0f - -1.0f) / 4294967296.0f;
    *u0 = -1.0f + (float)r0 * scale;
    *u1 = -1.0f + (float)r1 * scale;
}

void oracle_rng_kat(const uint32_t seeds[4], uint32_t gid, int nsteps, float *out_f, uint32_t *out_u32,
                    uint32_t out_state[4]) {
    Rng s = rng_seed(seeds, gid);
    for (int k = 0; k < nsteps; ++k) {
        float a, b; uint32_t ra, rb;
        rng_next(&s, &a, &b, &ra, &rb);
        if (out_f) { out_f[2 * k] = a; out_f[2 * k + 1] = b; }
        if (out_u32) { out_u32[2 * k] = ra; out_u32[2 * k + 1] = rb; }
    }
    out_state[0] = s.x0; out_state[1] = s.x1; out_state[2] = s.c0; out_state[3] = s.c1;
}

/* ----------------------------------------------------------------------- scene */
typedef struct {
    int carry;               /* 0: base (t reset per TraceRay, no r<t on the floor), 1: lmem family */
    int skip_zero_light;     /* base:171 */
    int use_grid;
    const int32_t *spheres, *squares;
    const float *tris; int ntris;
    const float (*lights)[4]; int nlights;
    V3 box_min, box_max; int res[3]; V3 cell;
    const uint32_t *cell_start, *cell_refs;
    int bidir; const float *vpls; int nvpl;
    int vlpgrid;             /* bidir Sample with the VLP-grid gather (vlpgrid:323-348); the grid is in box_min/res/cell/cell_start/cell_refs */
} Scene;

/* base:111-134 / grid:61-85 — Moller-Trumbore on one triangle; returns 1 if *t improved */
static inline int triangle_intersect(const float *tri, V3 o, V3 d, float *t, V3 *n, oracle_counters *cnt) {
    cnt->tri_tests++;
    V3 v0 = v3(tri[0], tri[1], tri[2]), v1 = v3(tri[4], tri[5], tri[6]), v2 = v3(tri[8], tri[9], tri[10]);
    V3 e0 = vsub(v1, v0), e2 = vsub(v2, v0);
    V3 pvec = cross3(d, e2);
    float det = dot3(e0, pvec);
    if (fabsf(det) < 0.01f) return 0;
    float inv = 1.0f / det;
    V3 tvec = vsub(o, v0);
    float u = dot3(tvec, pvec) * inv;
    if (u < 0.0f || u > 1.0f) return 0;
    V3 qvec = cross3(tvec, e0);
    float v = dot3(d, qvec) * inv;
    if (v < 0.0f || u + v > 1.0f) return 0;
    float r = dot3(e2, qvec) * inv;
    if (r < *t) {                      /* no lower bound on r (base:129) */
        *t = r;
        *n = normalize3(cross3(e0, e2));
        return 1;
    }
    return 0;
}

/* floor, squares, spheres: base:64-108 / lmem:63-106 / grid:112-156 */
static inline int trace_analytic(const Scene *S, V3 o, V3 d, float *t, V3 *n, oracle_counters *cnt) {
    int m = 0;
    float r = -o.z / d.z;
    if (S->carry ? (0.01f < r && r < *t) : (0.01f < r)) { *t = r; *n = v3(0, 0, 1); m = 1; }
    for (int k = 19; k--;)
        for (int j = 9; j--;)
            if (S->squares[j] & (1 << k)) {
                cnt->prim_tests++;
                r = ((float)(4 + j) - o.z) / d.z;
                V3 P = vmadd(d, r, o);
                if (r < *t && fabsf((float)k - P.x) < 1.0f && fabsf(P.y) < 1.0f) { *t = r; *n = v3(0, 0, 1); m = 3; }
            }
    for (int k = 19; k--;)
        for (int j = 9; j--;)
            if (S->spheres[j] & (1 << k)) {
                cnt->prim_tests++;
                V3 p = v3(o.x + (float)(-k), o.y + 0.0f, o.z + (float)(-j - 4));
                float b = dot3(p, d);
                float c = dot3(p, p) - 1.0f;
                float q = MADD(b, b, -c);
                if (q > 0.0f) {
                    r = -b - sqrtf(q);
                    if (r < *t && r > 0.01f) { *t = r; *n = normalize3(vmadd(d, *t, p)); m = 3; }
                }
            }
    return m;
}

static inline float comp(V3 v, int a) { return a == 0 ? v.x : (a == 1 ? v.y : v.z); }

/* grid:157-198 */
static inline int trace_grid(const Scene *S, V3 o, V3 d, float *t, V3 *n, int m, oracle_counters *cnt) {
    float tE[3], tX[3], dl[3], next[3];
    int idx[3], step[3], stop[3];
    for (int a = 0; a < 3; ++a) {
        float inv = 1.0f / comp(d, a);
        float l1 = (comp(S->box_min, a) - comp(o, a)) * inv;
        float l2 = (comp(S->box_max, a) - comp(o, a)) * inv;
        tE[a] = cl_fmin(l1, l2);
        tX[a] = cl_fmax(l1, l2);
    }
    float t0 = cl_fmax(cl_fmax(tE[0], tE[1]), cl_fmax(tE[0], tE[2]));
    float t1 = cl_fmin(cl_fmin(tX[0], tX[1]), cl_fmin(tX[0], tX[2]));
    if (t0 > t1) return m;
    int inside = o.x >= S->box_min.x && o.x <= S->box_max.x && o.y >= S->box_min.y && o.y <= S->box_max.y &&
                 o.z >= S->box_min.z && o.z <= S->box_max.z;
    V3 p = inside ? o : vmadd(d, t0, o);
    for (int a = 0; a < 3; ++a) {
        int hi = S->res[a] - 1;
        int v = f2i_rz_sat((comp(p, a) - comp(S->box_min, a)) / comp(S->cell, a));
        idx[a] = v < 0 ? 0 : (v > hi ? hi : v);   /* clamp(x,lo,hi) = min(max(x,lo),hi) */
        dl[a] = (tX[a] - tE[a]) / (float)S->res[a];
        int pos = comp(d, a) > 0.0f;
        next[a] = pos ? MADD((float)(idx[a] + 1), dl[a], tE[a]) : MADD((float)(S->res[a] - idx[a]), dl[a], tE[a]);
        step[a] = pos ? 1 : -1;
        stop[a] = pos ? S->res[a] : -1;
    }
    static const unsigned char map[8] = {2, 1, 2, 1, 2, 2, 0, 0};
    for (;;) {
        size_t ci = (size_t)idx[2] * S->res[0] * S->res[1] + (size_t)idx[1] * S->res[0] + idx[0];
        cnt->cells_visited++;
        uint32_t b = S->cell_start[ci], e = S->cell_start[ci + 1];
        int found = 0;
        for (uint32_t k = b; k < e; ++k)
            if (triangle_intersect(S->tris + 12 * (size_t)S->cell_refs[k], o, d, t, n, cnt)) found = 1;
        if (found) m = 4;
        int kk = ((next[0] < next[1]) << 2) + ((next[0] < next[2]) << 1) + (next[1] < next[2]);
        int axis = map[kk];
        next[axis] += dl[axis];
        if (*t < next[axis]) break;      /* compared AFTER the increment (grid:194-195) */
        idx[axis] += step[axis];
        if (idx[axis] == stop[axis]) break;
    }
    return m;
}

static inline int trace_ray(const Scene *S, V3 o, V3 d, float *t, V3 *n, oracle_counters *cnt) {
    cnt->rays++;
    if (!S->carry) *t = 1e9f;            /* base:52 */
    int m = trace_analytic(S, o, d, t, n, cnt);
    if (S->use_grid) return trace_grid(S, o, d, t, n, m, cnt);
    for (int i = 0; i < S->ntris; ++i)
        if (triangle_intersect(S->tris + 12 * (size_t)i, o, d, t, n, cnt)) m = 4;
    return m;
}

/* base:139-218 / lmem:138-216 / grid:203-283.  The 5-iteration loop always returns in iteration 1
 * because TraceRay only yields materials 0,1,3,4. */
static inline V3 sample(const Scene *S, V3 o, V3 d, Rng *rng, oracle_counters *cnt) {
    cnt->samples++;
    float t = 1e9f;                       /* lmem:155 (base resets inside TraceRay anyway) */
    V3 n = v3(0, 0, 0), dummy;
    int m = trace_ray(S, o, d, &t, &n, cnt);
    if (!m) {
        float p = POW4(1.0f - d.z);
        return v3(0.7f * p, 0.6f * p, 1.0f * p);
    }
    V3 X = vmadd(d, t, o);
    float illum = 0.0f;
    if (S->bidir) {
      if (S->vlpgrid) {
        /* vlpgrid:323-348 — the VPLs of the cell that contains the hit point.  convert_int4 truncates (and saturates); the
         * linear index is formed WITHOUT per-axis range checks (:325-326), so a point outside the box can alias into a cell */
        const int ix = f2i_rz_sat((X.x - S->box_min.x) / S->cell.x), iy = f2i_rz_sat((X.y - S->box_min.y) / S->cell.y),
                  iz = f2i_rz_sat((X.z - S->box_min.z) / S->cell.z);
        const uint32_t rx = (uint32_t)S->res[0], ry = (uint32_t)S->res[1], rz = (uint32_t)S->res[2];
        const int32_t index = (int32_t)((uint32_t)iz * rx * ry + (uint32_t)iy * rx + (uint32_t)ix);
        if (index >= 0 && index < (int32_t)(rx * ry * rz)) {
            for (uint32_t k = S->cell_start[index]; k < S->cell_start[index + 1]; ++k) {
                const float *P = S->vpls + 4 * (size_t)S->cell_refs[k];
                float I = P[3];
                V3 dv = vsub(v3(P[0], P[1], P[2]), X);
                float dist = sqrtf(dot3(dv, dv));
                V3 ld = v3(dv.x / dist, dv.y / dist, dv.z / dist);
                float lam = dot3(ld, n);
                if (lam < 0.0f) continue;
                float f = I / (dist * dist);
                f = 1.0f < f ? 1.0f : f;
                illum = MADD(lam, f, illum);
            }
        }
      } else {
        /* bidir:165-187 — every VPL, unshadowed */
        for (int i = 0; i < S->nvpl; ++i) {
            const float *P = S->vpls + 4 * (size_t)i;
            float I = P[3];
            if (I == 0.0f) continue;
            V3 dv = vsub(v3(P[0], P[1], P[2]), X);
            float dist = sqrtf(dot3(dv, dv));           /* distance(light_pos, intersection) */
            V3 ld = v3(dv.x / dist, dv.y / dist, dv.z / dist);
            float lam = dot3(ld, n);
            if (lam < 0.0f) continue;
            float f = I / (dist * dist);
            f = 1.0f < f ? 1.0f : f;
            illum = MADD(lam, f, illum);
        }
      }
        if (illum > 1.0f) illum = 1.0f;
        /* bidir:190-201 — soft shadows: each occluded real light SUBTRACTS 1/nlights; the shadow ray is bounded by
         * the un-jittered distance to the light (t = distanceFromLight, TraceRay keeps the running bound) */
        for (int i = 0; i < S->nlights; ++i) {
            float r0, r1;
            rng_next(rng, &r0, &r1, NULL, NULL);
            V3 L = v3(S->lights[i][0], S->lights[i][1], S->lights[i][2]);
            V3 dv = vsub(L, X);
            float dist = sqrtf(dot3(dv, dv));
            V3 ld = v3((L.x + r0) + X.x * -1.0f, (L.y + r1) + X.y * -1.0f, (L.z + 0.0f) + X.z * -1.0f);
            ld = normalize3(ld);
            t = dist;
            cnt->shadow_rays++;
            if (trace_ray(S, X, ld, &t, &dummy, cnt)) illum -= 1.0f / (float)S->nlights;
        }
    } else
    for (int i = 0; i < S->nlights; ++i) {
        float r0, r1;
        rng_next(rng, &r0, &r1, NULL, NULL);          /* drawn before any skip (base:168) */
        float I = S->lights[i][3];
        if (S->skip_zero_light && I == 0.0f) continue; /* base:171 only */
        V3 L = v3(S->lights[i][0], S->lights[i][1], S->lights[i][2]);
        /* light_pos + (r0,r1,0,0) + intersection*(-1) */
        V3 ld = v3((L.x + r0) + X.x * -1.0f, (L.y + r1) + X.y * -1.0f, (L.z + 0.0f) + X.z * -1.0f);
        ld = normalize3(ld);
        float lam = dot3(ld, n);
        if (lam < 0.0f) continue;
        cnt->shadow_rays++;
        if (trace_ray(S, X, ld, &t, &dummy, cnt)) continue;
        V3 dv = vsub(L, X);
        float dist = sqrtf(dot3(dv, dv));
        float f = I / (dist * dist);
        f = 1.0f < f ? 1.0f : f;                      /* min(x, 1.0f) = 1.0f < x ? 1.0f : x */
        illum = MADD(lam, f, illum);
    }
    if (!S->bidir && illum > 1.0f) illum = 1.0f;  /* bidir clamps BEFORE the shadow subtraction (bidir:188) */
    illum /= 4.0f;
    if (m == 1) {
        V3 Y = vscale(X, 0.2f);
        int odd = f2i_rz_sat(ceilf(Y.x) + ceilf(Y.y)) & 1;
        return odd ? v3(3.0f * illum, 1.0f * illum, 1.0f * illum) : v3(3.0f * illum, 3.0f * illum, 3.0f * illum);
    }
    if (m == 3) return v3(2.0f * illum, 3.0f * illum, 2.0f * illum);
    /* m == 4: facing ratio, lighting ignored (base:203-205) */
    float fr = dot3(n, v3(-d.x, -d.y, -d.z));
    fr = 0.0f < fr ? fr : 0.0f;                       /* max(0.0f, x) = 0.0f < x ? x : 0.0f */
    return v3(fr, fr, fr);
}

/* base:233-236 — thin-lens camera ray for pixel column i, row j */
static inline void camera_ray(const oracle_job *J, Rng *rng, int i, int j, V3 *o, V3 *d) {
    float u0, u1, u2, u3;
    rng_next(rng, &u0, &u1, NULL, NULL);
    rng_next(rng, &u2, &u3, NULL, NULL);
    V3 up = v3(J->cam_up[0], J->cam_up[1], J->cam_up[2]), right = v3(J->cam_right[0], J->cam_right[1], J->cam_right[2]);
    V3 eye = v3(J->eye_offset[0], J->eye_offset[1], J->eye_offset[2]);
    float a = (u0 - 0.5f) * 99.0f, b = (u1 - 0.5f) * 99.0f;
    V3 delta = vmadd(right, b, vscale(up, a));
    *o = v3(17.0f + delta.x, 16.0f + delta.y, 8.0f + delta.z);
    float su = u2 + (float)i, sr = (float)j + u3;
    V3 A = vmadd(right, sr, vscale(up, su));
    A = v3(A.x + eye.x, A.y + eye.y, A.z + eye.z);
    V3 nd = v3(delta.x * -1.0f, delta.y * -1.0f, delta.z * -1.0f);
    *d = normalize3(vmadd(A, 16.0f, nd));
}

/* the grid of a trianglegrid job is given (the CSR arrays; refs may be absent only without triangles) */
static int grid_job_ok(const oracle_job *J) { return J->cell_start && (J->cell_refs || J->ntriangles <= 0); }

static void scene_from_job(const oracle_job *J, Scene *S) {
    memset(S, 0, sizeof(*S));
    S->carry = J->variant != ORACLE_BASE;
    S->skip_zero_light = J->variant == ORACLE_BASE;
    S->use_grid = J->variant == ORACLE_GRID;
    S->spheres = J->spheres; S->squares = J->squares;
    S->tris = J->triangles; S->ntris = J->ntriangles;
    S->lights = J->lights; S->nlights = J->nlights;
    S->box_min = v3(J->box_min[0], J->box_min[1], J->box_min[2]);
    S->box_max = v3(J->box_max[0], J->box_max[1], J->box_max[2]);
    S->res[0] = J->grid_res[0]; S->res[1] = J->grid_res[1]; S->res[2] = J->grid_res[2];
    S->cell = v3(J->cell_size[0], J->cell_size[1], J->cell_size[2]);
    S->cell_start = J->cell_start; S->cell_refs = J->cell_refs;
    S->bidir = J->variant == ORACLE_BIDIR || J->variant == ORACLE_VLPGRID;
    S->vlpgrid = J->variant == ORACLE_VLPGRID;
    S->vpls = J->vpls; S->nvpl = J->nvpl;
}

/* bidir:230-278 SampleFromLightSource — one ray from a light; the hit point becomes a VPL whose intensity is the
 * light's Lambert term at the hit.  NB the reference dots the INCOMING direction with the outward normal, so
 * only surfaces hit from behind (squares seen from below) ever get a non-zero VPL; triangles (material 4)
 * and misses give the all-zero "dummy" light. */
static inline void sample_from_light(const Scene *S, V3 o, V3 d, float I, int total_vlp, float out[4], oracle_counters *cnt) {
    float t = 1e9f;
    V3 n = v3(0, 0, 0);
    out[0] = out[1] = out[2] = out[3] = 0.0f;
    int m = trace_ray(S, o, d, &t, &n, cnt);
    if (!m) return;
    V3 X = vmadd(d, t, o);
    float lam = dot3(d, n);
    if (lam < 0.0f) lam = 0.0f;
    else {
        V3 dv = vsub(o, X);
        float dist = sqrtf(dot3(dv, dv));
        float f = I / (dist * dist);
        f = 1.0f < f ? 1.0f : f;
        lam = lam * f;
    }
    if (lam > 1.0f) lam = 1.0f;
    float k = m == 1 ? 70.0f : (m == 2 ? 5.0f : (m == 3 ? 40.0f : 0.0f));
    if (k == 0.0f) return;                              /* material 4: (float4)(0) */
    out[0] = X.x; out[1] = X.y; out[2] = X.z;
    out[3] = (k * lam) / (float)(total_vlp / 512);      /* integer division first (bidir:267) */
}

int oracle_light_tracer(const oracle_job *J, int n, float *vpl_out, uint32_t *rng_state, oracle_counters *counters) {
    if (!J || n <= 0 || !vpl_out || J->nlights < 0 || J->nlights > 5) return -1;
    oracle_job Jl = *J;
    Jl.variant = ORACLE_LMEM;                            /* lmem TraceRay semantics, brute-force triangles */
    Scene S;
    scene_from_job(&Jl, &S);
    oracle_counters cnt;
    memset(&cnt, 0, sizeof(cnt));
    const int total = n * J->nlights;
    for (int gi = 0; gi < n; ++gi) {
        Rng rng = rng_seed(J->seeds, (uint32_t)gi);
        float r0 = 0.0f, r1 = 0.0f, sum = 2.0f;          /* randSum is NOT reset between lights (bidir:292,319): */
        for (int l = 0; l < J->nlights; ++l) {           /* lights after the first reuse the same direction     */
            while (sum >= 1.0f) {
                rng_next_pm1(&rng, &r0, &r1);
                sum = MADD(r1, r1, r0 * r0);
            }
            float sq = sqrtf(1.0f - sum);
            V3 d = v3((2.0f * r0) * sq, (2.0f * r1) * sq, 1.0f - 2.0f * sum);
            V3 o = v3(J->lights[l][0], J->lights[l][1], J->lights[l][2]);
            sample_from_light(&S, o, d, J->lights[l][3], total, vpl_out + 4 * ((size_t)gi + (size_t)l * n), &cnt);
        }
        if (rng_state) {
            uint32_t *q = rng_state + 4 * (size_t)gi;
            q[0] = rng.x0; q[1] = rng.x1; q[2] = rng.c0; q[3] = rng.c1;
        }
    }
    if (counters) *counters = cnt;
    return 0;
}


/* ------------------------------------------------------------------------------------------------------------------
 * CLSuperMetropolisPathTracer(_vlpgrid)/metropolispathtracer.ocl in FIX mode: kernels lightTracer (seed paths, :430-468 of
 * the plain program / vlpgrid:502-536) and MetropolisLightTracer (:470-531 / vlpgrid:538-...), with VerifyIntersection's
 * uninitialised hit bound replaced by the default distance 1e9 (the one-line patch oracle/Makefile applies to the reference
 * for libref_vlpgrid_fix.so) and the seed paths in their own buffer (the reference host hands lightTracer the VPL buffer).
 * Everything else is restated as written — including that every helper takes the RNG state BY VALUE (:146,159,172,184,241),
 * so a work-item's "random" directions repeat: GetRandomPath shoots its four segments along one direction, every mutation
 * round draws the same numbers. */
typedef struct { V3 v[4]; uint32_t length; } MPath;

/* :146-156 — rng by value: the caller's state is untouched */
static inline V3 metro_random_direction(Rng rng) {
    float r0 = 0.0f, r1 = 0.0f, sum = 2.0f;
    while (sum >= 1.0f) {
        rng_next_pm1(&rng, &r0, &r1);
        sum = MADD(r1, r1, r0 * r0);
    }
    float sq = sqrtf(1.0f - sum);
    return v3((2.0f * r0) * sq, (2.0f * r1) * sq, 1.0f - 2.0f * sum);
}

/* :158-170 */
static inline int metro_add_vertex(const Scene *S, V3 origin, V3 *vertex, MPath *path, Rng rng, oracle_counters *cnt) {
    const V3 d = metro_random_direction(rng);
    V3 n = v3(0, 0, 0);
    float t = 1e9f;
    if (trace_ray(S, origin, d, &t, &n, cnt)) {
        *vertex = vmadd(d, t, origin);
        path->length += 1;
        return 1;
    }
    return 0;
}

/* :172-182 */
static inline MPath metro_random_path(const Scene *S, V3 origin, Rng rng, oracle_counters *cnt) {
    MPath p;
    memset(&p, 0, sizeof(p));
    V3 cur = origin;
    for (int i = 0; i < 4; ++i) {
        if (!metro_add_vertex(S, cur, &p.v[i], &p, rng, cnt)) break;
        cur = p.v[i];
    }
    return p;
}

static inline float metro_perturb1(float vertex, float r, float dx) {
    if (r < 0.5f) return vertex < 1.0f ? vertex + dx : vertex + dx - 1.0f;
    return vertex < 0.0f ? vertex - dx + 1.0f : vertex - dx;
}

/* :184-221 — two RNG pairs (x, y from the first, z from the second), rng by value */
static inline V3 metro_perturbation(V3 vertex, Rng rng) {
    float a0, a1, b0, b1;
    rng_next(&rng, &a0, &a1, NULL, NULL);
    rng_next(&rng, &b0, &b1, NULL, NULL);
    const float s1 = 1.0f / 512.0f, s2 = 1.0f / 16.0f;
    const float q = s1 / s2, tail = s1 / (q + 1.0f);
    const float dx = s1 / (q + fabsf(2.0f * a0 - 1.0f)) - tail;
    const float dy = s1 / (q + fabsf(2.0f * a1 - 1.0f)) - tail;
    const float dz = s1 / (q + fabsf(2.0f * b0 - 1.0f)) - tail;
    return v3(metro_perturb1(vertex.x, a0, dx), metro_perturb1(vertex.y, a1, dy), metro_perturb1(vertex.z, b0, dz));
}

/* :223-236 with the FIX: t = 1e9 */
static inline int metro_verify(const Scene *S, V3 origin, V3 dest, oracle_counters *cnt) {
    float t = 1e9f;
    V3 n = v3(0, 0, 0);
    const V3 d = normalize3(vsub(dest, origin));
    if (!trace_ray(S, origin, d, &t, &n, cnt)) return 0;
    const V3 X = vmadd(d, t, origin);
    return dest.x == X.x && dest.y == X.y && dest.z == X.z;
}

/* :238-294 */
static inline void metro_mutate(const Scene *S, MPath *seed, V3 origin, Rng rng, oracle_counters *cnt) {
    if (seed->length == 0) {
        *seed = metro_random_path(S, origin, rng, cnt);
        if (seed->length == 0) return;
    }
    float y0, y1;
    rng_next(&rng, &y0, &y1, NULL, NULL);
    const float prob = 1.0f / ((float)seed->length + 0.2f);
    if (prob < y0) return;
    MPath tmp;
    memset(&tmp, 0, sizeof(tmp));
    V3 cur = origin;
    for (uint32_t i = 0; i < seed->length; ++i) {
        tmp.v[i] = metro_perturbation(seed->v[i], rng);
        if (metro_verify(S, cur, tmp.v[i], cnt)) { tmp.length++; cur = tmp.v[i]; }
        else break;
    }
    if (tmp.length == seed->length) *seed = tmp;
    if (seed->length == 1) {
        if (y1 > 0.3f) { if (!metro_add_vertex(S, seed->v[0], &seed->v[1], seed, rng, cnt)) return; }
        if (y1 > 0.7f) { if (!metro_add_vertex(S, seed->v[1], &seed->v[2], seed, rng, cnt)) return; }
        if (y1 > 0.9f) metro_add_vertex(S, seed->v[2], &seed->v[3], seed, rng, cnt);
    } else if (seed->length == 2) {
        if (y1 < 0.3f) { if (!metro_add_vertex(S, seed->v[1], &seed->v[2], seed, rng, cnt)) return; }
        if (y1 < 0.2f) metro_add_vertex(S, seed->v[2], &seed->v[3], seed, rng, cnt);
    } else if (seed->length == 3) {
        if (y1 < 0.2f) metro_add_vertex(S, seed->v[2], &seed->v[3], seed, rng, cnt);
    }
}

/* :380-428 SampleFromLightSource of the Metropolis programs (constants 400 / 10 / 40, total_paths / 256) */
static inline void metro_sample_from_light(const Scene *S, V3 o, V3 d, float I, int total_paths, float out[4], oracle_counters *cnt) {
    float t = 1e9f;
    V3 n = v3(0, 0, 0);
    out[0] = out[1] = out[2] = out[3] = 0.0f;
    int m = trace_ray(S, o, d, &t, &n, cnt);
    if (!m) return;
    V3 X = vmadd(d, t, o);
    float lam = dot3(d, n);
    if (lam < 0.0f) lam = 0.0f;
    else {
        V3 dv = vsub(o, X);
        float dist = sqrtf(dot3(dv, dv));
        float f = I / (dist * dist);
        f = 1.0f < f ? 1.0f : f;
        lam = lam * f;
    }
    if (lam > 1.0f) lam = 1.0f;
    float k = m == 1 ? 400.0f : (m == 2 ? 10.0f : (m == 3 ? 40.0f : 0.0f));
    if (k == 0.0f) return;
    out[0] = X.x; out[1] = X.y; out[2] = X.z;
    out[3] = (k * lam) / (float)(total_paths / 256);
}

/* paths_out (optional): n_paths*nlights x 20 words, the reference's Path layout {float4 v[4]; uint length; pad[3]} — only
 * v[0..length) and length are defined.  vpl_out: 4*n_paths*nlights x 4 floats, entry 4*(gi + l*n_paths) + i. */
int oracle_metropolis_light_tracer(const oracle_job *J, int n_paths, int mutation_rounds, uint32_t *paths_out, float *vpl_out) {
    if (!J || n_paths <= 0 || mutation_rounds < 0 || !vpl_out || J->nlights < 0 || J->nlights > 5) return -1;
    oracle_job Jl = *J;
    Jl.variant = ORACLE_LMEM;
    Scene S;
    scene_from_job(&Jl, &S);
    oracle_counters cnt;
    memset(&cnt, 0, sizeof(cnt));
    const int total_paths = n_paths * J->nlights;
    for (int gi = 0; gi < n_paths; ++gi) {
        const Rng rng = rng_seed(J->seeds, (uint32_t)gi);
        for (int l = 0; l < J->nlights; ++l) {
            V3 origin = v3(J->lights[l][0], J->lights[l][1], J->lights[l][2]);
            const float I = J->lights[l][3];
            MPath seed = metro_random_path(&S, origin, rng, &cnt);            /* kernel lightTracer */
            if (paths_out) {
                uint32_t *q = paths_out + 20 * ((size_t)gi + (size_t)l * n_paths);
                memset(q, 0, 80);
                for (uint32_t i = 0; i < seed.length; ++i) { memcpy(q + 4 * i, &seed.v[i], 12); }
                q[16] = seed.length;
            }
            for (int m = 0; m < mutation_rounds; ++m) metro_mutate(&S, &seed, origin, rng, &cnt);   /* kernel MetropolisLightTracer */
            float *out = vpl_out + 16 * ((size_t)gi + (size_t)l * n_paths);
            memset(out, 0, 64);
            for (uint32_t i = 0; i < seed.length; ++i) {
                const V3 d = normalize3(vsub(seed.v[i], origin));
                metro_sample_from_light(&S, origin, d, I / (float)(1 << i), total_paths, out + 4 * i, &cnt);
                if (out[4 * i + 3] == 0.0f) break;
                origin = seed.v[i];
            }
        }
    }
    return 0;
}

/* Mutate applied `rounds` times to one path (reference Path layout, 20 words), seeded as work-item gid: the counterpart of
 * refrt's ref_probe_mutate — the kernel keeps the mutated path private, the probes make it comparable. */
int oracle_metropolis_mutate(const oracle_job *J, uint32_t gid, const float origin[3], uint32_t path[20], int rounds) {
    if (!J || !path || rounds < 0) return -1;
    oracle_job Jl = *J;
    Jl.variant = ORACLE_LMEM;
    Scene S;
    scene_from_job(&Jl, &S);
    oracle_counters cnt;
    memset(&cnt, 0, sizeof(cnt));
    const Rng rng = rng_seed(J->seeds, gid);
    MPath p;
    memset(&p, 0, sizeof(p));
    p.length = path[16];
    if (p.length > 4) return -1;
    for (uint32_t i = 0; i < 4; ++i) memcpy(&p.v[i], path + 4 * i, 12);
    for (int m = 0; m < rounds; ++m) metro_mutate(&S, &p, v3(origin[0], origin[1], origin[2]), rng, &cnt);
    for (uint32_t i = 0; i < 4; ++i) { memcpy(path + 4 * i, &p.v[i], 12); path[4 * i + 3] = 0; }
    path[16] = p.length;
    return 0;
}

static inline void cnt_add(oracle_counters *a, const oracle_counters *b) {
    a->samples += b->samples; a->rays += b->rays; a->shadow_rays += b->shadow_rays;
    a->tri_tests += b->tri_tests; a->cells_visited += b->cells_visited; a->prim_tests += b->prim_tests;
}

static int g_threads_used = 0;
/* OpenMP team size of the most recent oracle_render (bench.py asserts the CPU baseline really ran on the cores it states) */
int oracle_threads_used(void) { return g_threads_used; }

int oracle_render(const oracle_job *J, uint8_t *rgba8, float *accum, uint32_t *rng_state, oracle_counters *counters) {
    if (!J || J->width <= 0 || J->height <= 0 || J->spp <= 0 || J->variant < 0 || J->variant > 5) return -1;
    if ((J->variant == ORACLE_BIDIR || J->variant == ORACLE_VLPGRID) && (J->nvpl < 0 || (J->nvpl > 0 && !J->vpls))) return -1;
    if (J->variant == ORACLE_VLPGRID && (!J->cell_start || !J->cell_refs)) return -1;
    if (J->variant == ORACLE_NODOF && J->spp != 64) return -1;
    if (J->variant == ORACLE_GRID && !grid_job_ok(J)) return -1;
    Scene S;
    scene_from_job(J, &S);
    const int W = J->width, H = J->height;
    int r0 = J->row_begin, r1 = J->row_end;
    if (r1 <= 0 || r1 > H) r1 = H;
    if (r0 < 0) r0 = 0;
    oracle_counters total;
    memset(&total, 0, sizeof(total));
    const float scale = 224.0f / (float)J->spp;      /* = 3.5f at the reference's 64 spp */
    /* sample blocks (extension, oracle.h): fewer samples from a re-seeded stream, bias only in block 0 */
    const int R = J->sample_blocks > 1 ? J->sample_blocks : 1, blk = R > 1 ? J->sample_block : 0;
    if (R > 1 && (J->variant == ORACLE_NODOF || blk < 0 || blk >= R || J->spp % R)) return -1;
    const int spp_local = J->spp / R;
    const float c0 = blk == 0 ? 13.0f : 0.0f, alpha = blk == 0 ? 255.0f : 0.0f;
    uint32_t seeds[4] = {J->seeds[0], J->seeds[1], J->seeds[2], J->seeds[3]};
    if (blk > 0) { const uint32_t h = oracle_randomize_id((uint32_t)blk); for (int k = 0; k < 4; ++k) seeds[k] ^= h; }
#ifdef _OPENMP
    int nthreads = J->nthreads > 0 ? J->nthreads : omp_get_max_threads();
#pragma omp parallel num_threads(nthreads)
#endif
    {
        oracle_counters cnt;
        memset(&cnt, 0, sizeof(cnt));
#ifdef _OPENMP
        if (omp_get_thread_num() == 0) g_threads_used = omp_get_num_threads();
#pragma omp for schedule(dynamic, 64)
#else
        g_threads_used = 1;
#endif
        for (long lin = (long)r0 * W; lin < (long)r1 * W; ++lin) {
            {
                const int j = (int)(lin / W), i = (int)(lin - (long)j * W);
                float col[4];
                size_t pix = (size_t)j * W + i;
                if (J->variant != ORACLE_NODOF) {
                    /* base:224-240 */
                    Rng rng = rng_seed(seeds, (uint32_t)(j * W + i));
                    V3 c = v3(c0, c0, c0);
                    for (int r = spp_local; r--;) {
                        V3 o, d;
                        camera_ray(J, &rng, i, j, &o, &d);
                        V3 s = sample(&S, o, d, &rng, &cnt);
                        c = v3(MADD(s.x, scale, c.x), MADD(s.y, scale, c.y), MADD(s.z, scale, c.z));
                    }
                    col[0] = c.x; col[1] = c.y; col[2] = c.z;
                    if (rng_state) {
                        uint32_t *q = rng_state + 4 * pix;
                        q[0] = rng.x0; q[1] = rng.x1; q[2] = rng.c0; q[3] = rng.c1;
                    }
                } else {
                    /* nodof:217-250 then 253-274: 8x8 work-items per pixel, each its own stream */
                    V3 acc[64];
                    for (int ly = 0; ly < 8; ++ly)
                        for (int lx = 0; lx < 8; ++lx) {
                            int gi = 8 * i + lx, gj = 8 * j + ly;
                            uint32_t gid = (uint32_t)(gj * (8 * W) + gi);
                            Rng rng = rng_seed(J->seeds, gid);
                            V3 o, d;
                            camera_ray(J, &rng, i, j, &o, &d);
                            V3 s = sample(&S, o, d, &rng, &cnt);
                            acc[ly * 8 + lx] = vscale(s, 3.5f);
                            if (rng_state) {
                                uint32_t *q = rng_state + 4 * (size_t)gid;
                                q[0] = rng.x0; q[1] = rng.x1; q[2] = rng.c0; q[3] = rng.c1;
                            }
                        }
                    for (int working = 32; working > 0; working >>= 1)
                        for (int li = 0; li < working; ++li) {
                            acc[li].x += acc[li + working].x;
                            acc[li].y += acc[li + working].y;
                            acc[li].z += acc[li + working].z;
                        }
                    col[0] = acc[0].x + 13.0f; col[1] = acc[0].y + 13.0f; col[2] = acc[0].z + 13.0f;
                }
                col[3] = J->variant == ORACLE_NODOF ? 255.0f : alpha;
                if (accum) memcpy(accum + 4 * pix, col, sizeof(col));
                if (rgba8)
                    for (int k = 0; k < 4; ++k) rgba8[4 * pix + k] = f2u8_rz_sat(col[k]);
            }
        }
#ifdef _OPENMP
#pragma omp critical
#endif
        cnt_add(&total, &cnt);
    }
    if (counters) *counters = total;
    return 0;
}

int oracle_trace_rays(const oracle_job *J, int n, const float *o, const float *d, float *t_inout, int32_t *m_out,
                      float *n_out, uint32_t *cells_out, uint32_t *tests_out) {
    if (!J || n < 0 || (n > 0 && (!o || !d || !t_inout)) || J->variant < 0 || J->variant > 5) return -1;
    if (J->variant == ORACLE_GRID && !grid_job_ok(J)) return -1;
    oracle_job Jr = *J;
    if (Jr.variant != ORACLE_BASE && Jr.variant != ORACLE_GRID) Jr.variant = ORACLE_LMEM;   /* lmem TraceRay semantics */
    Scene S;
    scene_from_job(&Jr, &S);
    for (int k = 0; k < n; ++k) {
        oracle_counters cnt;
        memset(&cnt, 0, sizeof(cnt));
        V3 nn = v3(0, 0, 0);
        const int m = trace_ray(&S, v3(o[3 * k], o[3 * k + 1], o[3 * k + 2]), v3(d[3 * k], d[3 * k + 1], d[3 * k + 2]),
                                t_inout + k, &nn, &cnt);
        if (m_out) m_out[k] = m;
        if (n_out) { n_out[3 * k] = nn.x; n_out[3 * k + 1] = nn.y; n_out[3 * k + 2] = nn.z; }
        if (cells_out) cells_out[k] = (uint32_t)cnt.cells_visited;
        if (tests_out) tests_out[k] = (uint32_t)cnt.tri_tests;
    }
    return 0;
}

int oracle_trace_ray(int carry, const float o[3], const float d[3], float *t_inout, float n_out[3],
                     const int32_t spheres[9], const int32_t squares[9], const float *tris12, int ntris) {
    Scene S;
    memset(&S, 0, sizeof(S));
    S.carry = carry; S.spheres = spheres; S.squares = squares; S.tris = tris12; S.ntris = ntris;
    oracle_counters cnt;
    memset(&cnt, 0, sizeof(cnt));
    V3 n = v3(0, 0, 0);
    int m = trace_ray(&S, v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), t_inout, &n, &cnt);
    n_out[0] = n.x; n_out[1] = n.y; n_out[2] = n.z;
    return m;
}
