/*
 * scanerf_oracle.c -- CPU restatement of the reference's native hot-path ops.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity oracle and the CPU
 * baseline for bench.py.  Nothing in the product package may link, import or
 * call it; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs use it.
 *
 * Every function cites the reference file:line it restates (paths relative to
 * the reference checkout).  Arithmetic follows the reference's fp32 operation
 * order.  Where nvcc (default -fmad=true) is expected to contract a*b+c into
 * one FMA in the reference build, fmaf() is written explicitly; this file is
 * compiled with -ffp-contract=off so nothing else is fused.
 *
 * Pinning status: the reference ships no tests or golden vectors (SURVEY.md
 * section 4).  The oracle is pinned against outputs of the reference CUDA
 * extensions rebuilt unmodified for sm_100a (oracle/build_ref.py ->
 * oracle/_ref/ *.so) and run on the B200 box; the vectors that run produced are
 * committed under tests/golden/ (tests/golden/make_ref_golden.py).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <unistd.h>

#define ORACLE_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------- */
/* tiny pthread parallel-for (the image's gcc has no libgomp)                  */
/* ------------------------------------------------------------------------- */
typedef void (*range_fn)(int begin, int end, void *ctx);
typedef struct { range_fn fn; void *ctx; int begin, end; } pf_job_t;
static void *pf_tramp(void *a) { pf_job_t *j = (pf_job_t *)a; j->fn(j->begin, j->end, j->ctx); return NULL; }

ORACLE_API int oracle_num_threads(void)
{
    const char *e = getenv("ORACLE_THREADS");
    int n = e ? atoi(e) : (int)sysconf(_SC_NPROCESSORS_ONLN);
    return n < 1 ? 1 : (n > 256 ? 256 : n);
}

static void parallel_for(int n, range_fn fn, void *ctx)
{
    int nt = oracle_num_threads();
    if (nt > n) nt = n;
    if (nt <= 1) { fn(0, n, ctx); return; }
    pthread_t th[256]; pf_job_t jobs[256];
    for (int t = 0; t < nt; ++t) {
        jobs[t].fn = fn; jobs[t].ctx = ctx;
        jobs[t].begin = (int)((long long)n * t / nt);
        jobs[t].end = (int)((long long)n * (t + 1) / nt);
        pthread_create(&th[t], NULL, pf_tramp, &jobs[t]);
    }
    for (int t = 0; t < nt; ++t) pthread_join(th[t], NULL);
}

/* ------------------------------------------------------------------------- */
/* helpers restating cutil_math.h                                             */
/* ------------------------------------------------------------------------- */

/* cuda/include/cutil_math.h:913-916  signf(0) = +1 */
static inline int signf_i(float a) { return a >= 0.0f ? 1 : -1; }
/* cuda/include/cutil_math.h:924-926 */
static inline float safe_divide(float a, float b) { return b != 0.0f ? a / b : 100000000.0f; }
static inline int imin(int a, int b) { return a < b ? a : b; }
static inline int imax(int a, int b) { return a > b ? a : b; }
static inline int iclamp(int v, int lo, int hi) { return imax(lo, imin(v, hi)); }

/* ------------------------------------------------------------------------- */
/* 1. multi-resolution hash-grid encode                                       */
/* ------------------------------------------------------------------------- */

/* hashgrid/src/hashgrid_bg_kernel.cu:14-24 (same in hashgrid_kernel.cu): only
 * three primes are used, uint32 wrap-around, mask with T-1. */
static inline uint32_t hash3(int x, int y, int z, uint32_t mask)
{
    uint32_t r = 0;
    r ^= (uint32_t)x * 1u;
    r ^= (uint32_t)y * 2654435761u;
    r ^= (uint32_t)z * 805459861u;
    return r & mask;
}

/* hashgrid_bg_kernel.cu:79-90: corner order c = 4*dx + 2*dy + dz */
static inline void corner_indices(uint32_t idx[8], int ix, int iy, int iz, uint32_t mask)
{
    for (int c = 0; c < 8; ++c)
        idx[c] = hash3(ix + ((c >> 2) & 1), iy + ((c >> 1) & 1), iz + (c & 1), mask);
}

/* hashgrid_bg_kernel.cu:26-38: products evaluated left to right */
static inline void linear_weight(float w[8], float ox, float oy, float oz)
{
    w[0] = (1 - ox) * (1 - oy) * (1 - oz);
    w[1] = (1 - ox) * (1 - oy) * oz;
    w[2] = (1 - ox) * oy * (1 - oz);
    w[3] = (1 - ox) * oy * oz;
    w[4] = ox * (1 - oy) * (1 - oz);
    w[5] = ox * (1 - oy) * oz;
    w[6] = ox * oy * (1 - oz);
    w[7] = ox * oy * oz;
}

/* hashgrid_bg_kernel.cu:40-77 */
static inline void dweights(float dx[8], float dy[8], float dz[8], float ox, float oy, float oz)
{
    dx[0] = (-1.0f) * (1 - oy) * (1 - oz); dx[1] = (-1.0f) * (1 - oy) * oz;
    dx[2] = (-1.0f) * oy * (1 - oz);       dx[3] = (-1.0f) * oy * oz;
    dx[4] = (1 - oy) * (1 - oz);           dx[5] = (1 - oy) * oz;
    dx[6] = oy * (1 - oz);                 dx[7] = oy * oz;
    dy[0] = (1 - ox) * (-1.0f) * (1 - oz); dy[1] = (1 - ox) * (-1.0f) * oz;
    dy[2] = (1 - ox) * (1 - oz);           dy[3] = (1 - ox) * oz;
    dy[4] = ox * (-1.0f) * (1 - oz);       dy[5] = ox * (-1.0f) * oz;
    dy[6] = ox * (1 - oz);                 dy[7] = ox * oz;
    dz[0] = (1 - ox) * (1 - oy) * (-1.0f); dz[1] = (1 - ox) * (1 - oy);
    dz[2] = (1 - ox) * oy * (-1.0f);       dz[3] = (1 - ox) * oy;
    dz[4] = ox * (1 - oy) * (-1.0f);       dz[5] = ox * (1 - oy);
    dz[6] = ox * oy * (-1.0f);             dz[7] = ox * oy;
}

typedef struct { int ix, iy, iz; float ox, oy, oz; float sx, sy, sz; } cellpos_t;

/* BG variant prologue, hashgrid_bg_kernel.cu:123-130 and :177-184.
 * (p + 2.0f) / 4.0f is add then multiply by 1.0f/4.0f (cutil_math.h:411-415). */
static inline cellpos_t locate_bg(const float *p, const int *res)
{
    cellpos_t c;
    const float inv4 = 1.0f / 4.0f;
    float ux = (p[0] + 2.0f) * inv4, uy = (p[1] + 2.0f) * inv4, uz = (p[2] + 2.0f) * inv4;
    float vx = ux * (float)(res[0] - 1), vy = uy * (float)(res[1] - 1), vz = uz * (float)(res[2] - 1);
    c.ix = (int)vx; c.iy = (int)vy; c.iz = (int)vz;
    c.ox = vx - (float)c.ix; c.oy = vy - (float)c.iy; c.oz = vz - (float)c.iz;
    /* doffset_dpts = (res-1)/4.0f  (:186) */
    c.sx = (float)(res[0] - 1) * inv4; c.sy = (float)(res[1] - 1) * inv4; c.sz = (float)(res[2] - 1) * inv4;
    return c;
}

static inline float clampf(float v, float lo, float hi) { return fmaxf(lo, fminf(v, hi)); }

/* bbox variant prologue, hashgrid/src/hashgrid_kernel.cu:126-141; the product
 * float(i)*g + corner is one FMA under nvcc's default contraction. */
static inline cellpos_t locate_bbox(const float *p, const int *res, const float *corner, const float *size)
{
    cellpos_t c;
    float q[3], g[3], o[3]; int i[3];
    for (int a = 0; a < 3; ++a) {
        q[a] = clampf(p[a], corner[a], corner[a] + size[a]);
        g[a] = size[a] / (float)(res[a] - 1);
        i[a] = (int)((q[a] - corner[a]) / g[a]);
        float vmin = fmaf((float)i[a], g[a], corner[a]);
        o[a] = (q[a] - vmin) / g[a];
    }
    c.ix = i[0]; c.iy = i[1]; c.iz = i[2];
    c.ox = o[0]; c.oy = o[1]; c.oz = o[2];
    /* backward scale 1.0f / grid_size (hashgrid_kernel.cu:237-239) */
    c.sx = 1.0f / g[0]; c.sy = 1.0f / g[1]; c.sz = 1.0f / g[2];
    return c;
}

/* Forward.  hashgrid_bg_kernel.cu:106-150 (bbox==NULL) / hashgrid_kernel.cu:105-158.
 * points[B,3], table[L,T,2], res[L,3] -> out[B,L,2]; optional idx_out[B,L,8]
 * returns the hashed corner indices so tests can assert them bit-exactly. */
typedef struct {
    const float *points, *grad_in, *table; const int *res; const float *corner, *size;
    float *out; uint32_t *idx_out; float *grad_points, *grad_table, *gp_lvl; int B, L, T;
} enc_ctx_t;

static void enc_fwd_range(int b0, int b1, void *vctx)
{
    enc_ctx_t *x = (enc_ctx_t *)vctx;
    const float *points = x->points, *table = x->table, *corner = x->corner, *size = x->size;
    const int *res = x->res; float *out = x->out; uint32_t *idx_out = x->idx_out;
    const int L = x->L, T = x->T;
    const uint32_t mask = (uint32_t)T - 1u;
    for (int b = b0; b < b1; ++b) {
        for (int l = 0; l < L; ++l) {
            const float *lev = table + (size_t)l * T * 2;
            cellpos_t c = corner ? locate_bbox(points + 3 * b, res + 3 * l, corner, size)
                                 : locate_bg(points + 3 * b, res + 3 * l);
            uint32_t idx[8]; float w[8];
            corner_indices(idx, c.ix, c.iy, c.iz, mask);
            linear_weight(w, c.ox, c.oy, c.oz);
            float ax = 0.0f, ay = 0.0f;
            for (int k = 0; k < 8; ++k) { /* acc = acc + w*F contracts to FMA */
                ax = fmaf(w[k], lev[2 * (size_t)idx[k]], ax);
                ay = fmaf(w[k], lev[2 * (size_t)idx[k] + 1], ay);
            }
            out[((size_t)b * L + l) * 2] = ax;
            out[((size_t)b * L + l) * 2 + 1] = ay;
            if (idx_out) memcpy(idx_out + ((size_t)b * L + l) * 8, idx, sizeof(idx));
        }
    }
}

ORACLE_API void oracle_hash_encode_fwd(const float *points, const float *table, const int *res,
                                       const float *corner, const float *size,
                                       float *out, uint32_t *idx_out, int B, int L, int T)
{
    enc_ctx_t x; memset(&x, 0, sizeof(x));
    x.points = points; x.table = table; x.res = res; x.corner = corner; x.size = size;
    x.out = out; x.idx_out = idx_out; x.B = B; x.L = L; x.T = T;
    parallel_for(B, enc_fwd_range, &x);
}

/* Backward.  hashgrid_bg_kernel.cu:152-226 / hashgrid_kernel.cu:160-243.
 * grad_table and grad_points are ACCUMULATED into (the reference atomically adds
 * into caller-zeroed buffers).  Levels are independent in grad_table, so the
 * parallel loop is over levels and the summation order is deterministic
 * (point-ascending) -- the reference's own order is not. */
static void enc_bwd_range(int l0, int l1, void *vctx)
{
    enc_ctx_t *x = (enc_ctx_t *)vctx;
    const float *points = x->points, *grad_in = x->grad_in, *table = x->table, *corner = x->corner, *size = x->size;
    const int *res = x->res; float *grad_table = x->grad_table, *gp_lvl = x->gp_lvl;
    const int B = x->B, L = x->L, T = x->T;
    const uint32_t mask = (uint32_t)T - 1u;
    for (int l = l0; l < l1; ++l) {
        const float *lev = table + (size_t)l * T * 2;
        float *glev = grad_table + (size_t)l * T * 2;
        for (int b = 0; b < B; ++b) {
            cellpos_t c = corner ? locate_bbox(points + 3 * b, res + 3 * l, corner, size)
                                 : locate_bg(points + 3 * b, res + 3 * l);
            float gx = grad_in[((size_t)b * L + l) * 2], gy = grad_in[((size_t)b * L + l) * 2 + 1];
            uint32_t idx[8]; float w[8], dx[8], dy[8], dz[8];
            corner_indices(idx, c.ix, c.iy, c.iz, mask);
            linear_weight(w, c.ox, c.oy, c.oz);
            dweights(dx, dy, dz, c.ox, c.oy, c.oz);
            float ddx[2] = {0, 0}, ddy[2] = {0, 0}, ddz[2] = {0, 0};
            for (int k = 0; k < 8; ++k) {
                float fx = lev[2 * (size_t)idx[k]], fy = lev[2 * (size_t)idx[k] + 1];
                glev[2 * (size_t)idx[k]] += w[k] * gx;
                glev[2 * (size_t)idx[k] + 1] += w[k] * gy;
                ddx[0] = fmaf(fx, dx[k], ddx[0]); ddx[1] = fmaf(fy, dx[k], ddx[1]);
                ddy[0] = fmaf(fx, dy[k], ddy[0]); ddy[1] = fmaf(fy, dy[k], ddy[1]);
                ddz[0] = fmaf(fx, dz[k], ddz[0]); ddz[1] = fmaf(fy, dz[k], ddz[1]);
            }
            float *gp = gp_lvl + ((size_t)l * B + b) * 3;
            gp[0] = c.sx * fmaf(gx, ddx[0], gy * ddx[1]);
            gp[1] = c.sy * fmaf(gx, ddy[0], gy * ddy[1]);
            gp[2] = c.sz * fmaf(gx, ddz[0], gy * ddz[1]);
        }
    }
}

static void enc_gp_range(int b0, int b1, void *vctx)
{
    enc_ctx_t *x = (enc_ctx_t *)vctx;
    for (int b = b0; b < b1; ++b)
        for (int l = 0; l < x->L; ++l)
            for (int a = 0; a < 3; ++a)
                x->grad_points[(size_t)b * 3 + a] += x->gp_lvl[((size_t)l * x->B + b) * 3 + a];
}

ORACLE_API void oracle_hash_encode_bwd(const float *points, const float *grad_in, const float *table,
                                       const int *res, const float *corner, const float *size,
                                       float *grad_points, float *grad_table, int B, int L, int T)
{
    enc_ctx_t x; memset(&x, 0, sizeof(x));
    x.points = points; x.grad_in = grad_in; x.table = table; x.res = res; x.corner = corner; x.size = size;
    x.grad_points = grad_points; x.grad_table = grad_table; x.B = B; x.L = L; x.T = T;
    x.gp_lvl = (float *)calloc((size_t)L * B * 3, sizeof(float));
    parallel_for(L, enc_bwd_range, &x);
    parallel_for(B, enc_gp_range, &x);
    free(x.gp_lvl);
}

/* ------------------------------------------------------------------------- */
/* 2. ray generation, ray/box test, occupancy-grid sampler                    */
/* ------------------------------------------------------------------------- */

/* cuda/include/cuda_utils.h:143-155 (get_rays, +0.5 pixel centre) via
 * cuda/compute_ray_kernel.cu:17-43.  locs[B,3] = (view, px, py). */
ORACLE_API void oracle_compute_ray_fwd(float *rays_o, float *rays_d, const float *Ks, const float *C2Ws,
                                       const int *locs, int B)
{
    for (int i = 0; i < B; ++i) {
        const int v = locs[3 * i], px = locs[3 * i + 1], py = locs[3 * i + 2];
        const float *K = Ks + 9 * v, *M = C2Ws + 12 * v;
        const float x = (1.0f * px + 0.5f - K[2]) / K[0];
        const float y = (1.0f * py + 0.5f - K[5]) / K[4];
        rays_d[3 * i + 0] = fmaf(M[1], y, M[0] * x) + M[2];
        rays_d[3 * i + 1] = fmaf(M[5], y, M[4] * x) + M[6];
        rays_d[3 * i + 2] = fmaf(M[9], y, M[8] * x) + M[10];
        rays_o[3 * i + 0] = M[3]; rays_o[3 * i + 1] = M[7]; rays_o[3 * i + 2] = M[11];
    }
}

/* cuda/compute_ray_kernel.cu:45-92.  ref_index_bug != 0 reproduces the reference's
 * read of grad_rays_*[view_idx] (:71-72); 0 reads grad_rays_*[ray] (the correct
 * gradient of the forward above).  Accumulates into grad_C2Ws[N,12]. */
ORACLE_API void oracle_compute_ray_bwd(const float *g_o, const float *g_d, const float *Ks, float *grad_C2Ws,
                                       const int *locs, int B, int ref_index_bug)
{
    for (int i = 0; i < B; ++i) {
        const int v = locs[3 * i], px = locs[3 * i + 1], py = locs[3 * i + 2];
        const float *K = Ks + 9 * v;
        const float x = (1.0f * px + 0.5f - K[2]) / K[0];
        const float y = (1.0f * py + 0.5f - K[5]) / K[4];
        const int gi = ref_index_bug ? v : i;
        const float *go = g_o + 3 * gi, *gd = g_d + 3 * gi;
        float *g = grad_C2Ws + 12 * v;
        g[3] += go[0]; g[7] += go[1]; g[11] += go[2];
        g[0] += gd[0] * x; g[1] += gd[0] * y; g[2] += gd[0];
        g[4] += gd[1] * x; g[5] += gd[1] * y; g[6] += gd[1];
        g[8] += gd[2] * x; g[9] += gd[2] * y; g[10] += gd[2];
    }
}

/* cuda/include/cuda_utils.h:564-613 (float3 half-size overload) */
static void ray_aabb1(const float *o, const float *d, const float *c, const float *h, float *lo_out, float *hi_out)
{
    float f_low = 0.0f, f_high = 100000.0f;
    for (int a = 0; a < 3; ++a) {
        float inv = safe_divide(1.0f, d[a]);
        float lo = (c[a] - h[a] - o[a]) * inv;
        float hi = (c[a] + h[a] - o[a]) * inv;
        if (hi < lo) { float t = lo; lo = hi; hi = t; }
        if (hi < f_low || lo > f_high) { *lo_out = -1.0f; *hi_out = -1.0f; return; }
        f_low = lo > f_low ? lo : f_low;
        f_high = hi < f_high ? hi : f_high;
        if (f_low > f_high) { *lo_out = -1.0f; *hi_out = -1.0f; return; }
    }
    *lo_out = f_low; *hi_out = f_high;
}

/* cuda/helper_kernel.cu:107-197: boxes given as center[K,3], size[K,3]; bounds[B,K,2] */
ORACLE_API void oracle_ray_aabb(const float *rays_o, const float *rays_d, const float *centers, const float *sizes,
                                float *bounds, int B, int K)
{
    for (int i = 0; i < B; ++i)
        for (int k = 0; k < K; ++k) {
            float h[3] = {sizes[3 * k] * 0.5f, sizes[3 * k + 1] * 0.5f, sizes[3 * k + 2] * 0.5f};
            ray_aabb1(rays_o + 3 * i, rays_d + 3 * i, centers + 3 * k, h,
                      bounds + ((size_t)i * K + k) * 2, bounds + ((size_t)i * K + k) * 2 + 1);
        }
}

/* cuda/include/dda.h:206-268 (DDASatateScene_v2) */
typedef struct {
    int c[3], s[3], m[3], n[3];
    float tmax[3], tdelta[3], t0, t1;
} walk_t;

static void walk_init(walk_t *w, const float *o_in, const float *d, float t_near, float t_far, const int *n, const float *cell)
{
    float o[3];
    for (int a = 0; a < 3; ++a) {
        w->n[a] = n[a];
        o[a] = fmaf(t_near, d[a], o_in[a]);                 /* origin + t*dir contracts */
        w->c[a] = iclamp((int)(o[a] / cell[a]), 0, n[a] - 1);
        w->s[a] = signf_i(d[a]);
        float nb = (float)(w->c[a] + w->s[a]) * cell[a];
        if (w->s[a] < 0) nb += cell[a];
        w->tmax[a] = fmaxf(safe_divide(nb - o[a], d[a]), 0.0f) + t_near;
        w->tdelta[a] = fabsf(safe_divide(cell[a], d[a]));
    }
    w->t0 = t_near; w->t1 = t_far;
}
static void walk_next(walk_t *w)
{
    w->m[0] = (w->tmax[0] < w->tmax[1]) & (w->tmax[0] <= w->tmax[2]);
    w->m[1] = (w->tmax[1] < w->tmax[2]) & (w->tmax[1] <= w->tmax[0]);
    w->m[2] = !(w->m[0] | w->m[1]);
    w->t1 = w->m[0] ? w->tmax[0] : (w->m[1] ? w->tmax[1] : w->tmax[2]);
}
static void walk_step(walk_t *w)
{
    w->t0 = w->t1;
    for (int a = 0; a < 3; ++a) {
        w->tmax[a] = fmaf((float)w->m[a], w->tdelta[a], w->tmax[a]);
        w->c[a] += w->m[a] * w->s[a];
    }
}
static int walk_done(const walk_t *w)
{
    for (int a = 0; a < 3; ++a) if (w->c[a] < 0 || w->c[a] >= w->n[a]) return 1;
    return w->tmax[0] <= 0 && w->tmax[1] <= 0 && w->tmax[2] <= 0;
}

/* cuda/helper_kernel.cu:539-671 (sample_points_sparse_single_ray + launcher).
 * z_vals/dists[B,S] keep the caller's fill for rays that miss or see nothing.
 * counts[B] (optional) = number of occupied segments with positive length. */
ORACLE_API void oracle_sample_points_grid(const float *rays_o, const float *rays_d, float *z_vals, float *dists,
                                          const float *corner, const float *size, const unsigned char *occ,
                                          const int *log2dim, int *counts, int B, int S)
{
    const int n[3] = {1 << log2dim[0], 1 << log2dim[1], 1 << log2dim[2]};
    const int ly = log2dim[1], lz = log2dim[2];
    float cell[3], half[3], center[3];
    for (int a = 0; a < 3; ++a) {
        cell[a] = size[a] / (float)n[a];
        half[a] = size[a] * 0.5f;
        center[a] = corner[a] + half[a];
    }
    for (int i = 0; i < B; ++i) {
        const float *o = rays_o + 3 * i, *d = rays_d + 3 * i;
        float tn, tf;
        if (counts) counts[i] = 0;
        ray_aabb1(o, d, center, half, &tn, &tf);
        if (tn == -1.0f) continue;
        float ol[3] = {o[0] - corner[0], o[1] - corner[1], o[2] - corner[2]};
        walk_t w;
        walk_init(&w, ol, d, tn, tf, n, cell);
        float total = 0.0f; int count = 0;
        while (!walk_done(&w)) {
            walk_next(&w);
            uint32_t idx = ((uint32_t)w.c[0] << (ly + lz)) | ((uint32_t)w.c[1] << lz) | (uint32_t)w.c[2];
            if (occ[idx]) { float len = w.t1 - w.t0; if (len > 0) { total += len; ++count; } }
            walk_step(&w);
        }
        if (counts) counts[i] = count;
        if (count == 0) continue;
        walk_init(&w, ol, d, tn, tf, n, cell);
        int left = S, seen = 0;
        while (!walk_done(&w)) {
            walk_next(&w);
            uint32_t idx = ((uint32_t)w.c[0] << (ly + lz)) | ((uint32_t)w.c[1] << lz) | (uint32_t)w.c[2];
            if (occ[idx]) {
                float len = w.t1 - w.t0;
                if (len > 0) {
                    int num = imin(imax((int)((float)S * len / total), 1), left);
                    if (seen == count - 1) num = left;
                    /* uniform_sample_bound_v3, cuda_utils.h:101-113 */
                    float interval = (w.t1 - w.t0) / (float)num;
                    for (int k = 0; k < num; ++k) {
                        z_vals[(size_t)i * S + (S - left) + k] = fmaf((float)k, interval, w.t0);
                        dists[(size_t)i * S + (S - left) + k] = interval;
                    }
                    left -= num; ++seen;
                }
            }
            walk_step(&w);
        }
    }
}

/* ------------------------------------------------------------------------- */
/* 3. multi-tile render tracing (hashgrid/src/rendering_kernel.cu)            */
/* ------------------------------------------------------------------------- */

#define RENDER_MISS 10000000.0f

/* The scene of the multi-tile renderer: nb tiles (corner, size), their occupancy grids
 * concatenated at starts[b] with (2^lx, 2^ly, 2^lz) cells; isect[B, nb, 2] = (near, far), 1e7 on a
 * miss; order[B, nb] = the tiles of each ray near to far. */
typedef struct {
    const float *rays_o, *rays_d, *corners, *sizes, *isect;
    const unsigned char *occ; const long long *starts; const int *log2dim, *order;
    int *tracing_idx; float *z_start, *z_vals, *dists; short *hit, *ids; float *w;
    unsigned char *tgt; int nb, S, bidx, skip;
} trace_ctx_t;

typedef struct { float corner[3], cell[3]; int n[3], ly, lz; const unsigned char *occ; } tile_grid_t;

static void tile_grid(const trace_ctx_t *x, int b, tile_grid_t *g)
{
    for (int a = 0; a < 3; ++a) {
        g->n[a] = 1 << x->log2dim[3 * b + a];
        g->corner[a] = x->corners[3 * b + a];
        g->cell[a] = x->sizes[3 * b + a] / (float)g->n[a];
    }
    g->ly = x->log2dim[3 * b + 1]; g->lz = x->log2dim[3 * b + 2];
    g->occ = x->occ + x->starts[b];
}
static void tile_walk(const tile_grid_t *g, walk_t *w, const float *o, const float *d, float t_near, float t_far)
{
    float ol[3] = {o[0] - g->corner[0], o[1] - g->corner[1], o[2] - g->corner[2]};
    walk_init(w, ol, d, t_near, t_far, g->n, g->cell);
}
static int tile_on(const tile_grid_t *g, const walk_t *w)
{
    return g->occ[((uint32_t)w->c[0] << (g->ly + g->lz)) | ((uint32_t)w->c[1] << g->lz) | (uint32_t)w->c[2]] != 0;
}

/* rendering_kernel.cu:178-382 (sample_points): one call advances every ray to the next tile of its order
 * that has occupied segments beyond z_start and places S samples there, n = (int)(len / total * S) per
 * segment, the last segment taking the rest.  The walk starts at the tile's near on a ray's first tile
 * and at z_start (the previous tile's far) after it.  z_vals / dists keep the caller's fill elsewhere. */
static void render_sample_range(int i0, int i1, void *vctx)
{
    const trace_ctx_t *x = (const trace_ctx_t *)vctx;
    const int nb = x->nb, S = x->S;
    for (int i = i0; i < i1; ++i) {
        const float *o = x->rays_o + 3 * (size_t)i, *d = x->rays_d + 3 * (size_t)i;
        const int *order = x->order + (size_t)i * nb;
        const float *isect = x->isect + (size_t)i * nb * 2;
        float *zr = x->z_vals + (size_t)i * S, *dr = x->dists + (size_t)i * S;
        int step = x->tracing_idx[i];
        float t = x->z_start[i];
        while (step < nb) {
            const int b = order[step];
            const float near = isect[2 * b], far = isect[2 * b + 1];
            if (near == RENDER_MISS) break;
            if (t >= far) { ++step; continue; }
            if (step == 0) t = near;
            tile_grid_t g; walk_t w;
            tile_grid(x, b, &g);
            tile_walk(&g, &w, o, d, t, 0.0f);
            int num_seg = 0; float total = 0.0f;
            while (!walk_done(&w)) {
                walk_next(&w);
                if (tile_on(&g, &w)) { float len = w.t1 - w.t0; if (len > 0) { total += len; ++num_seg; } }
                walk_step(&w);
            }
            if (num_seg == 0) { t = far; ++step; continue; }
            tile_walk(&g, &w, o, d, t, 0.0f);
            int num = 0, count = 0;
            while (!walk_done(&w)) {
                walk_next(&w);
                if (tile_on(&g, &w)) {
                    float len = w.t1 - w.t0;
                    if (len > 0) {
                        int n = imin(imax((int)(len / total * (float)S), 1), S - num);
                        if (count == num_seg - 1) n = S - num;
                        if (n > 0) {
                            float interval = (w.t1 - w.t0) / (float)n;        /* uniform_sample_bound_v3 */
                            for (int k = 0; k < n; ++k) { zr[num + k] = fmaf((float)k, interval, w.t0); dr[num + k] = interval; }
                        }
                        num += n; ++count;
                    }
                }
                walk_step(&w);
            }
            t = far; ++step;
            break;
        }
        x->tracing_idx[i] = step;
        x->z_start[i] = t;
    }
}

ORACLE_API void oracle_render_sample(const float *rays_o, const float *rays_d, const float *corners, const float *sizes,
                                     const unsigned char *occ, const long long *starts, const int *log2dim,
                                     const int *order, const float *isect, int *tracing_idx, float *z_start,
                                     float *z_vals, float *dists, int B, int nb, int S)
{
    trace_ctx_t x; memset(&x, 0, sizeof(x));
    x.rays_o = rays_o; x.rays_d = rays_d; x.corners = corners; x.sizes = sizes; x.occ = occ; x.starts = starts;
    x.log2dim = log2dim; x.order = order; x.isect = isect; x.tracing_idx = tracing_idx; x.z_start = z_start;
    x.z_vals = z_vals; x.dists = dists; x.nb = nb; x.S = S;
    parallel_for(B, render_sample_range, &x);
}

/* rendering_kernel.cu:704-812 (ray_firsthit_block): the tile with the nearest far among the tiles whose
 * walk from near meets an occupied cell; else, where hit[i] is still -1, the last tile the ray enters. */
static void firsthit_range(int i0, int i1, void *vctx)
{
    const trace_ctx_t *x = (const trace_ctx_t *)vctx;
    const int nb = x->nb;
    for (int i = i0; i < i1; ++i) {
        const float *o = x->rays_o + 3 * (size_t)i, *d = x->rays_d + 3 * (size_t)i;
        const int *order = x->order + (size_t)i * nb;
        const float *isect = x->isect + (size_t)i * nb * 2;
        float dis = RENDER_MISS;
        int last = -1;
        for (int s = 0; s < nb; ++s) {
            const int b = order[s];
            const float near = isect[2 * b], far = isect[2 * b + 1];
            if (near == RENDER_MISS) break;
            tile_grid_t g; walk_t w;
            tile_grid(x, b, &g);
            tile_walk(&g, &w, o, d, near, far);
            int any = 0;
            while (!walk_done(&w)) {
                walk_next(&w);
                if (tile_on(&g, &w)) { any = 1; break; }
                walk_step(&w);
            }
            if (any && dis > far) { x->hit[i] = (short)b; dis = far; }
            last = b;
        }
        if (last != -1 && x->hit[i] == -1) x->hit[i] = (short)last;
    }
}

ORACLE_API void oracle_firsthit_block(const float *rays_o, const float *rays_d, const float *corners, const float *sizes,
                                      const unsigned char *occ, const long long *starts, const int *log2dim,
                                      const int *order, const float *isect, short *hit, int B, int nb)
{
    trace_ctx_t x; memset(&x, 0, sizeof(x));
    x.rays_o = rays_o; x.rays_d = rays_d; x.corners = corners; x.sizes = sizes; x.occ = occ; x.starts = starts;
    x.log2dim = log2dim; x.order = order; x.isect = isect; x.hit = hit; x.nb = nb;
    parallel_for(B, firsthit_range, &x);
}

/* rendering_kernel.cu:1478-1565 (process_occupied_grid): each occupied cell of tile bidx (cell index t in
 * [0, total_grid), decomposed with bidx's own grid) marks, in every other tile b, the cell of b's grid that
 * holds each of its eight corners, if that corner lies in [0, 1)^3 of b.  The cell origin float(i) * cell +
 * corner is one FMA under nvcc's contraction.  Runs over the target tiles so that no two threads write
 * the same grid. */
static void occupied_range(int b0, int b1, void *vctx)
{
    const trace_ctx_t *x = (const trace_ctx_t *)vctx;
    const int bidx = x->bidx;
    tile_grid_t src;
    tile_grid(x, bidx, &src);
    const int ry = src.n[1], rz = src.n[2], total = x->S;
    for (int b = b0; b < b1; ++b) {
        if (b == bidx) continue;
        const float *c = x->corners + 3 * b, *sz = x->sizes + 3 * b;
        const int *l = x->log2dim + 3 * b;
        unsigned char *tg = x->tgt + x->starts[b];
        for (int t = 0; t < total; ++t) {
            if (!src.occ[t]) continue;
            const int ix0 = t / (ry * rz), rem = t - ix0 * (ry * rz), iy0 = rem / rz, iz0 = rem % rz;
            const float p0[3] = {fmaf((float)ix0, src.cell[0], src.corner[0]), fmaf((float)iy0, src.cell[1], src.corner[1]),
                                 fmaf((float)iz0, src.cell[2], src.corner[2])};
            for (int j = 0; j < 8; ++j) {
                const int v[3] = {(j >> 2) & 1, (j >> 1) & 1, j & 1};
                float q[3]; int inside = 1, id[3];
                for (int a = 0; a < 3; ++a) {
                    q[a] = (fmaf((float)v[a], src.cell[a], p0[a]) - c[a]) / sz[a];
                    inside &= q[a] >= 0 && q[a] < 1;
                }
                if (!inside) continue;
                for (int a = 0; a < 3; ++a) id[a] = (int)(q[a] * (float)(1 << l[a]));
                tg[(id[0] << (l[1] + l[2])) | (id[1] << l[2]) | id[2]] = 1;
            }
        }
    }
}

ORACLE_API void oracle_process_occupied(int bidx, int total_grid, const float *corners, const float *sizes,
                                        const unsigned char *occ, const long long *starts, const int *log2dim,
                                        unsigned char *tgt, int nb)
{
    trace_ctx_t x; memset(&x, 0, sizeof(x));
    x.corners = corners; x.sizes = sizes; x.occ = occ; x.starts = starts; x.log2dim = log2dim; x.tgt = tgt;
    x.bidx = bidx; x.S = total_grid; x.nb = nb;
    parallel_for(nb, occupied_range, &x);
}

/* rendering_kernel.cu:1262-1401 (update_outgoing_bidx): the tiles sharing the largest far among those the
 * ray enters (without skip: up to the first tile that starts beyond the current far), at most 4; one tile
 * gets weight 1, several get the x / z face distances of the exit point o + far d (one FMA) in each. */
static void outgoing_range(int i0, int i1, void *vctx)
{
    const trace_ctx_t *x = (const trace_ctx_t *)vctx;
    const int nb = x->nb;
    for (int i = i0; i < i1; ++i) {
        const int *order = x->order + (size_t)i * nb;
        const float *isect = x->isect + (size_t)i * nb * 2;
        float far = -1.0f;
        int index = 0, cur[4] = {-1, -1, -1, -1};
        for (int s = 0; s < nb; ++s) {
            const int b = order[s];
            const float n = isect[2 * b], f = isect[2 * b + 1];
            if (n == RENDER_MISS) break;
            if (!x->skip && (n > far && far != -1.0f)) break;
            if (f > far) { far = f; cur[0] = b; cur[1] = cur[2] = cur[3] = -1; index = 1; }
            else if (f == far && index < 4) cur[index++] = b;
        }
        if (far == -1.0f) continue;
        short *ob = x->ids + (size_t)i * 4;
        float *ow = x->w + (size_t)i * 4;
        if (index == 1) { ow[0] = 1.0f; ob[0] = (short)cur[0]; continue; }
        const float *o = x->rays_o + 3 * (size_t)i, *d = x->rays_d + 3 * (size_t)i;
        const float p[3] = {fmaf(far, d[0], o[0]), fmaf(far, d[1], o[1]), fmaf(far, d[2], o[2])};
        for (int k = 0; k < 4 && cur[k] != -1; ++k) {
            const int b = cur[k];
            float dis[3];
            for (int a = 0; a < 3; ++a) {
                const float sz = x->sizes[3 * b + a];
                const float q = clampf((p[a] - x->corners[3 * b + a]) / sz, 0.0f, 1.0f);
                dis[a] = (0.5f - fabsf(q - 0.5f)) * sz;
            }
            ow[k] = dis[0] != 0 && dis[2] != 0 ? dis[0] * dis[2] : (dis[0] != 0 ? dis[0] : (dis[2] != 0 ? dis[2] : 0.0f));
            ob[k] = (short)b;
        }
    }
}

ORACLE_API void oracle_outgoing_bidx(const float *rays_o, const float *rays_d, const float *corners, const float *sizes,
                                     const int *order, const float *isect, short *ids, float *w, int skip, int B, int nb)
{
    trace_ctx_t x; memset(&x, 0, sizeof(x));
    x.rays_o = rays_o; x.rays_d = rays_d; x.corners = corners; x.sizes = sizes; x.order = order; x.isect = isect;
    x.ids = ids; x.w = w; x.skip = skip; x.nb = nb;
    parallel_for(B, outgoing_range, &x);
}

/* cuda/sample_kernel.cu:17-44 + uniform_sample_bound (cuda_utils.h:77-87) */
ORACLE_API void oracle_background_sampling(const float *starts, const float *bg_depth, float *z_vals,
                                           int B, int S, float range)
{
    for (int i = 0; i < B; ++i) {
        float near = fmaxf(starts[i] + 0.00001f, fmaf(-range, 0.5f, bg_depth[i]));
        float far = near + range;
        float interval = (far - near) / (float)(S - 1);
        for (int k = 0; k < S; ++k) z_vals[(size_t)i * S + k] = fmaf((float)k, interval, near);
    }
}

/* cuda/sample_kernel.cu:70-100 + inverse_z_sample_bound (cuda_utils.h:61-75).
 * Returns the number of rays that miss the box (the reference device-asserts). */
ORACLE_API int oracle_sample_insideout(const float *rays_o, const float *rays_d, int S, int Sbg, const float *center,
                                       const float *size, float far, float *z_vals, float *z_bg, int B)
{
    int misses = 0;
    float half[3] = {size[0] * 0.5f, size[1] * 0.5f, size[2] * 0.5f};
    for (int i = 0; i < B; ++i) {
        float tn, tf;
        ray_aabb1(rays_o + 3 * i, rays_d + 3 * i, center, half, &tn, &tf);
        if (tn == -1.0f || tf == -1.0f) { ++misses; continue; }
        float interval = (tf - tn) / (float)(S - 1);
        for (int k = 0; k < S; ++k) z_vals[(size_t)i * S + k] = fmaf((float)k, interval, tn);
        float inv_near = 1.0f / tf, inv_far = 1.0f / far, inv_bound = inv_far - inv_near;
        float step = 1.0f / (float)(Sbg - 1);
        for (int k = 0; k < Sbg; ++k) z_bg[(size_t)i * Sbg + k] = 1.0f / fmaf(step * (float)k, inv_bound, inv_near);
    }
    return misses;
}

/* ------------------------------------------------------------------------- */
/* 6. sparse Adam                                                             */
/* ------------------------------------------------------------------------- */

/* cuda/adam_kernel.cu:23-69 (adam_step_kernel): element (k,d) at k*row_stride+d (the reference
 * hard-codes 8); grad == 0 -> skipped; `step` is the value the kernel sees (host passes step+1).
 * half_state != 0 restates adam_step_fp16_kernel (:97-144) with the moments passed as floats
 * that the caller rounds to half (state arrays here are float; rounding is applied in place). */
static float round_to_half(float x)
{
    /* IEEE binary16 round-to-nearest-even of a float, returned as float */
    _Float16 h = (_Float16)x;
    return (float)h;
}

ORACLE_API void oracle_adam_step(float *params, const float *grads, float *exp_avg, float *exp_avg_sq,
                                 long long rows, int dim, int row_stride, int half_state,
                                 float lr, float beta1, float beta2, float eps, int step)
{
    const float bc1 = 1.0f - powf(beta1, (float)step);
    const float bc2 = 1.0f - powf(beta2, (float)step);
    for (long long k = 0; k < rows; ++k)
        for (int d = 0; d < dim; ++d) {
            const long long i = k * row_stride + d;
            if (!half_state) {
                const float g = grads[i];
                if (g == 0.0f) continue;
                const float m = beta1 * exp_avg[i] + (1.0f - beta1) * g;
                const float v = beta2 * exp_avg_sq[i] + (1.0f - beta2) * g * g;
                const float denom = sqrtf(v / bc2) + eps;
                const float step_size = lr / bc1;
                params[i] = params[i] - step_size * m / denom;
                exp_avg[i] = m; exp_avg_sq[i] = v;
            } else {
                const float g = grads[i] * 128.0f;
                if (g == 0.0f) continue;
                const float m = beta1 * exp_avg[i] + (1.0f - beta1) * g;
                const float v = beta2 * exp_avg_sq[i] + (1.0f - beta2) * g * g;
                const float denom = sqrtf(v / (bc2 * 128.0f * 128.0f)) + eps;
                const float step_size = lr / bc1;
                params[i] = params[i] - step_size * m / (denom * 128.0f);
                exp_avg[i] = round_to_half(m); exp_avg_sq[i] = round_to_half(v);
            }
        }
}
