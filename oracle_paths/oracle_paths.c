/*
 * oracle_paths.c — diffuse bounces with Russian roulette (DESIGN.md 5b) on top of the C oracle.  TEST INFRASTRUCTURE ONLY
 * (see oracle_paths.h).
 *
 * oracle/oracle.c is compiled into this translation unit unchanged: camera and shadow rays go through its trace_ray, the
 * light loop and shading are its sample()'s, the RNG is its rng_next.  What is new here is stated once:
 *   - bounce rays: the oracle's TraceRay with the lower bound r > 0.01 on squares and triangles (trace_bounce);
 *   - the path: throughput, Russian roulette, the cosine-weighted direction and the accumulation (path_sample).
 * Fused multiply-adds (PT_CONTRACT = 1) of the new arithmetic, the same sites as the CUDA kernel (pt_device.cuh
 * bounce_direction / sample_bounces): s = a*a + b*b; T.x = (sign n.x n.x) e + 1; U.y = (n.y n.y) e + sign; the two
 * multiply-adds of a T + b U + z n_f; L += beta * c.
 */
#include "../oracle/oracle.c"

#include "oracle_paths.h"

#define PATH_TMIN 0.01f

/* triangle_intersect for bounce rays: a hit counts only at r > PATH_TMIN */
static inline int tri_bounce(const float *tri, V3 o, V3 d, float *t, V3 *n, oracle_counters *cnt, oracle_path_counters *pc) {
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
    if (r < *t) {
        if (!(r > PATH_TMIN)) { pc->tmin_rejections++; return 0; }
        *t = r;
        *n = normalize3(cross3(e0, e2));
        return 1;
    }
    return 0;
}

/* trace_analytic for bounce rays: squares count only at r > PATH_TMIN (floor and spheres already have r > 0.01) */
static inline int analytic_bounce(const Scene *S, V3 o, V3 d, float *t, V3 *n, oracle_counters *cnt, oracle_path_counters *pc) {
    int m = 0;
    float r = -o.z / d.z;
    if (S->carry ? (0.01f < r && r < *t) : (0.01f < r)) { *t = r; *n = v3(0, 0, 1); m = 1; }
    for (int k = 19; k--;)
        for (int j = 9; j--;)
            if (S->squares[j] & (1 << k)) {
                cnt->prim_tests++;
                r = ((float)(4 + j) - o.z) / d.z;
                V3 P = vmadd(d, r, o);
                if (r < *t && fabsf((float)k - P.x) < 1.0f && fabsf(P.y) < 1.0f) {
                    if (r > PATH_TMIN) { *t = r; *n = v3(0, 0, 1); m = 3; }
                    else pc->tmin_rejections++;
                }
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

/* trace_grid for bounce rays (grid:157-198 with tri_bounce) */
static inline int grid_bounce(const Scene *S, V3 o, V3 d, float *t, V3 *n, int m, oracle_counters *cnt, oracle_path_counters *pc) {
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
        idx[a] = v < 0 ? 0 : (v > hi ? hi : v);
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
            if (tri_bounce(S->tris + 12 * (size_t)S->cell_refs[k], o, d, t, n, cnt, pc)) found = 1;
        if (found) m = 4;
        int kk = ((next[0] < next[1]) << 2) + ((next[0] < next[2]) << 1) + (next[1] < next[2]);
        int axis = map[kk];
        next[axis] += dl[axis];
        if (*t < next[axis]) break;
        idx[axis] += step[axis];
        if (idx[axis] == stop[axis]) break;
    }
    return m;
}

/* TraceRay of a bounce ray (t = 1e9 from the caller) */
static inline int trace_bounce(const Scene *S, V3 o, V3 d, float *t, V3 *n, oracle_counters *cnt, oracle_path_counters *pc) {
    cnt->rays++;
    pc->bounce_rays++;
    if (!S->carry) *t = 1e9f;
    int m = analytic_bounce(S, o, d, t, n, cnt, pc);
    if (S->use_grid) return grid_bounce(S, o, d, t, n, m, cnt, pc);
    for (int i = 0; i < S->ntris; ++i)
        if (tri_bounce(S->tris + 12 * (size_t)i, o, d, t, n, cnt, pc)) m = 4;
    return m;
}

/* One path vertex: the oracle's sample() (non-bidirectional branch) for the ray (o, d) that reaches it, without its samples
 * count; also hands out the material, hit point and normal the bounce needs. */
static inline V3 path_vertex(const Scene *S, V3 o, V3 d, int bounce, Rng *rng, oracle_counters *cnt, oracle_path_counters *pc,
                             int *m_out, V3 *X_out, V3 *n_out) {
    float t = 1e9f;
    V3 n = v3(0, 0, 0), dummy;
    int m = bounce ? trace_bounce(S, o, d, &t, &n, cnt, pc) : trace_ray(S, o, d, &t, &n, cnt);
    *m_out = m;
    if (!m) {
        float p = POW4(1.0f - d.z);
        return v3(0.7f * p, 0.6f * p, 1.0f * p);
    }
    V3 X = vmadd(d, t, o);
    *X_out = X;
    *n_out = n;
    float illum = 0.0f;
    for (int i = 0; i < S->nlights; ++i) {
        float r0, r1;
        rng_next(rng, &r0, &r1, NULL, NULL);
        float I = S->lights[i][3];
        if (S->skip_zero_light && I == 0.0f) continue;
        V3 L = v3(S->lights[i][0], S->lights[i][1], S->lights[i][2]);
        V3 ld = v3((L.x + r0) + X.x * -1.0f, (L.y + r1) + X.y * -1.0f, (L.z + 0.0f) + X.z * -1.0f);
        ld = normalize3(ld);
        float lam = dot3(ld, n);
        if (lam < 0.0f) continue;
        cnt->shadow_rays++;
        if (trace_ray(S, X, ld, &t, &dummy, cnt)) continue;
        V3 dv = vsub(L, X);
        float dist = sqrtf(dot3(dv, dv));
        float f = I / (dist * dist);
        f = 1.0f < f ? 1.0f : f;
        illum = MADD(lam, f, illum);
    }
    if (illum > 1.0f) illum = 1.0f;
    illum /= 4.0f;
    if (m == 1) {
        V3 Y = vscale(X, 0.2f);
        int odd = f2i_rz_sat(ceilf(Y.x) + ceilf(Y.y)) & 1;
        return odd ? v3(3.0f * illum, 1.0f * illum, 1.0f * illum) : v3(3.0f * illum, 3.0f * illum, 3.0f * illum);
    }
    if (m == 3) return v3(2.0f * illum, 3.0f * illum, 2.0f * illum);
    float fr = dot3(n, v3(-d.x, -d.y, -d.z));
    fr = 0.0f < fr ? fr : 0.0f;
    return v3(fr, fr, fr);
}

/* Cosine-weighted direction about the face-forward normal: disk by rejection (<= 32 pairs), Malley lift, basis of Duff et al.
 * 2017.  0 when all pairs miss the disk. */
static inline int bounce_direction(V3 n, V3 d, Rng *rng, V3 *w, oracle_path_counters *pc) {
    const V3 nf = dot3(n, d) < 0.0f ? n : v3(-n.x, -n.y, -n.z);
    float a = 0.0f, b = 0.0f, s = 1.0f;
    int k = 0;
    for (; k < 32; ++k) {
        float u0, u1;
        rng_next(rng, &u0, &u1, NULL, NULL);
        a = 2.0f * u0 - 1.0f;
        b = 2.0f * u1 - 1.0f;
        s = MADD(b, b, a * a);
        if (s < 1.0f) break;
    }
    if (k == 32) { pc->disk_exhausted++; return 0; }
    const float z = sqrtf(1.0f - s);
    const float sign = copysignf(1.0f, nf.z);
    const float e = -1.0f / (sign + nf.z);
    const float f = (nf.x * nf.y) * e;
    const float sx = sign * nf.x;
    const V3 T = v3(MADD(sx * nf.x, e, 1.0f), sign * f, -sx);
    const V3 U = v3(f, MADD(nf.y * nf.y, e, sign), -nf.y);
    *w = normalize3(vmadd(nf, z, vmadd(U, b, vscale(T, a))));
    return 1;
}

/* A path: vertex 0 for (o, d), then up to B bounces.  rr = 0 disables Russian roulette (test switch). */
static V3 path_sample(const Scene *S, V3 o, V3 d, Rng *rng, int B, int rr, oracle_counters *cnt, oracle_path_counters *pc) {
    cnt->samples++;
    V3 beta = v3(1.0f, 1.0f, 1.0f), L = v3(0.0f, 0.0f, 0.0f);
    for (int k = 0;; ++k) {
        int m;
        V3 X = v3(0, 0, 0), n = v3(0, 0, 0);
        const V3 c = path_vertex(S, o, d, k > 0, rng, cnt, pc, &m, &X, &n);
        L = k == 0 ? c : v3(MADD(beta.x, c.x, L.x), MADD(beta.y, c.y, L.y), MADD(beta.z, c.z, L.z));
        if ((m != 1 && m != 3) || k >= B) break;
        V3 rho;
        if (m == 1) {
            V3 Y = vscale(X, 0.2f);
            int odd = f2i_rz_sat(ceilf(Y.x) + ceilf(Y.y)) & 1;
            rho = odd ? v3(0.75f, 0.25f, 0.25f) : v3(0.75f, 0.75f, 0.75f);
        } else {
            rho = v3(0.5f, 0.75f, 0.5f);
        }
        beta = v3(beta.x * rho.x, beta.y * rho.y, beta.z * rho.z);
        if (k >= 1 && rr) {                       /* bounce k+1 >= 2 */
            float xi, unused;
            rng_next(rng, &xi, &unused, NULL, NULL);
            const float q = fminf(0.95f, fmaxf(beta.x, fmaxf(beta.y, beta.z)));
            if (xi >= q) { pc->rr_terminations++; break; }
            beta = v3(beta.x / q, beta.y / q, beta.z / q);
        }
        V3 w;
        if (!bounce_direction(n, d, rng, &w, pc)) break;
        o = X;
        d = w;
    }
    return L;
}

static inline void path_cnt_add(oracle_path_counters *a, const oracle_path_counters *b) {
    a->bounce_rays += b->bounce_rays; a->rr_terminations += b->rr_terminations;
    a->tmin_rejections += b->tmin_rejections; a->disk_exhausted += b->disk_exhausted;
}

static int path_job_ok(const oracle_job *J, int max_bounces) {
    if (!J || max_bounces < 0 || max_bounces > 15) return 0;
    if (J->variant != ORACLE_BASE && J->variant != ORACLE_LMEM && J->variant != ORACLE_GRID) return 0;
    if (J->variant == ORACLE_GRID && !grid_job_ok(J)) return 0;
    return J->nlights >= 0 && J->nlights <= 5;
}

int oracle_render_bounces(const oracle_job *J, int max_bounces, uint8_t *rgba8, float *accum, uint32_t *rng_state,
                          oracle_counters *counters, oracle_path_counters *path_counters) {
    if (!path_job_ok(J, max_bounces) || J->width <= 0 || J->height <= 0 || J->spp <= 0) return -1;
    Scene S;
    scene_from_job(J, &S);
    const int W = J->width, H = J->height;
    int r0 = J->row_begin, r1 = J->row_end;
    if (r1 <= 0 || r1 > H) r1 = H;
    if (r0 < 0) r0 = 0;
    oracle_counters total;
    oracle_path_counters ptotal;
    memset(&total, 0, sizeof(total));
    memset(&ptotal, 0, sizeof(ptotal));
    const float scale = 224.0f / (float)J->spp;
    const int R = J->sample_blocks > 1 ? J->sample_blocks : 1, blk = R > 1 ? J->sample_block : 0;
    if (R > 1 && (blk < 0 || blk >= R || J->spp % R)) return -1;
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
        oracle_path_counters pc;
        memset(&cnt, 0, sizeof(cnt));
        memset(&pc, 0, sizeof(pc));
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 64)
#endif
        for (long lin = (long)r0 * W; lin < (long)r1 * W; ++lin) {
            const int j = (int)(lin / W), i = (int)(lin - (long)j * W);
            const size_t pix = (size_t)j * W + i;
            Rng rng = rng_seed(seeds, (uint32_t)(j * W + i));
            V3 c = v3(c0, c0, c0);
            for (int r = spp_local; r--;) {
                V3 o, d;
                camera_ray(J, &rng, i, j, &o, &d);
                V3 s = path_sample(&S, o, d, &rng, max_bounces, 1, &cnt, &pc);
                c = v3(MADD(s.x, scale, c.x), MADD(s.y, scale, c.y), MADD(s.z, scale, c.z));
            }
            const float col[4] = {c.x, c.y, c.z, alpha};
            if (rng_state) {
                uint32_t *q = rng_state + 4 * pix;
                q[0] = rng.x0; q[1] = rng.x1; q[2] = rng.c0; q[3] = rng.c1;
            }
            if (accum) memcpy(accum + 4 * pix, col, sizeof(col));
            if (rgba8)
                for (int k = 0; k < 4; ++k) rgba8[4 * pix + k] = f2u8_rz_sat(col[k]);
        }
#ifdef _OPENMP
#pragma omp critical
#endif
        {
            cnt_add(&total, &cnt);
            path_cnt_add(&ptotal, &pc);
        }
    }
    if (counters) *counters = total;
    if (path_counters) *path_counters = ptotal;
    return 0;
}

int oracle_path_sample(const oracle_job *J, const float o[3], const float d[3], uint32_t rng_state[4], int max_bounces,
                       int rr_enabled, float out_rgb[3], oracle_counters *counters, oracle_path_counters *path_counters) {
    if (!path_job_ok(J, max_bounces) || !o || !d || !rng_state || !out_rgb) return -1;
    Scene S;
    scene_from_job(J, &S);
    oracle_counters cnt;
    oracle_path_counters pc;
    memset(&cnt, 0, sizeof(cnt));
    memset(&pc, 0, sizeof(pc));
    Rng rng = {rng_state[0], rng_state[1], rng_state[2], rng_state[3]};
    const V3 L = path_sample(&S, v3(o[0], o[1], o[2]), v3(d[0], d[1], d[2]), &rng, max_bounces, rr_enabled != 0, &cnt, &pc);
    rng_state[0] = rng.x0; rng_state[1] = rng.x1; rng_state[2] = rng.c0; rng_state[3] = rng.c1;
    out_rgb[0] = L.x; out_rgb[1] = L.y; out_rgb[2] = L.z;
    if (counters) cnt_add(counters, &cnt);
    if (path_counters) path_cnt_add(path_counters, &pc);
    return 0;
}

int oracle_path_samples(const oracle_job *J, int n, const float o[3], const float d[3], uint32_t *rng_states, int max_bounces,
                        int rr_enabled, float *out_rgb, oracle_path_counters *path_counters) {
    if (!path_job_ok(J, max_bounces) || n < 0 || !o || !d || (n > 0 && (!rng_states || !out_rgb))) return -1;
    oracle_path_counters total;
    memset(&total, 0, sizeof(total));
#ifdef _OPENMP
    int nthreads = J->nthreads > 0 ? J->nthreads : omp_get_max_threads();
#pragma omp parallel num_threads(nthreads)
#endif
    {
        oracle_path_counters pc;
        memset(&pc, 0, sizeof(pc));
#ifdef _OPENMP
#pragma omp for schedule(static)
#endif
        for (int k = 0; k < n; ++k)
            oracle_path_sample(J, o, d, rng_states + 4 * (size_t)k, max_bounces, rr_enabled, out_rgb + 3 * (size_t)k, NULL, &pc);
#ifdef _OPENMP
#pragma omp critical
#endif
        path_cnt_add(&total, &pc);
    }
    if (path_counters) path_cnt_add(path_counters, &total);
    return 0;
}
