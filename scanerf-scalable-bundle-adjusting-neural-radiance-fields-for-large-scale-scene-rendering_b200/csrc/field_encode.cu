// Fused training-path field encode: sample position -> space contraction -> 16-level hash encode,
// forward and backward, sm_100a.
//
// Replaces (behaviour, not code) this chain of HashGrid.render_batch_rays (hashgrid/__init__.py:512-545):
//   samples = rays_o + z * rays_d                              (:522)
//   contract_fore / contract_bg                                (:394-411)
//   HashEmbeddingBGAutoGrad.forward / .backward                (hashgrid/PyHashGridBG.py:9-30 ->
//                                                               hashgrid/src/hashgrid_bg_kernel.cu:106-275)
// and the autograd of all of it back to (rays_o, rays_d) and the table.
//
// Data layout in HBM (level-major, so that every access of a warp is one contiguous 256-byte run):
//   out  [L][N]     float2    encoded features            (the reference operator writes [N][L])
//   jac  [L][3][N]  float2    d out / d contracted point  (training only)
//   grad [L][N]     float2    incoming gradient
// The forward stores the 2x3 Jacobian of every (sample, level) -- 24 bytes -- so that the backward
// never re-gathers the table (8 random sectors per level in the reference, :195-222): it is a pure
// gradient scatter.  The scatter walks each level's table slice in `passes` index ranges so that the
// live part of the gradient table (128 MiB per level at T = 2^24) stays L2-resident while it is
// being reduced into; every sector then travels to HBM once per range instead of once per touch.
// d L / d rays is reduced per warp (32 consecutive samples of one ray) before it touches memory.
#include "hash_common.cuh"
#include "adam_core.cuh"
using namespace hashgrid;

namespace {

constexpr int kThreads = 256;
enum Contract { kNone = 0, kRays = 1 };      // kRays: samples on rays; rays [0, ray_split) use the fore map, the rest the background map

struct Pt {
    f3 c;          // contracted point in [-2,2]^3
    f3 jd;         // diagonal of d c / d x  (affine part times f)
    f3 u;          // affine-normalised point (background only)
    float fp;      // f'(n) * a_k   (background only): the rank-one part acts along axis k
    int k;         // arg-max axis of |u|
};

// o + z d with separately rounded multiply and add, as torch evaluates it (hashgrid/__init__.py:522):
// an FMA here could move a sample across a cell boundary relative to the reference path.
__device__ __forceinline__ f3 sample_pos(f3 o, f3 d, float z)
{
    return mk3(__fadd_rn(o.x, __fmul_rn(z, d.x)), __fadd_rn(o.y, __fmul_rn(z, d.y)), __fadd_rn(o.z, __fmul_rn(z, d.z)));
}

// x -> contracted coordinates.  fore: c = (x - min) / size * 4 - 2 (hashgrid/__init__.py:394-395);
// back: u = that, n = |u|_inf, c = u (2 - 1/n) / n (:397-411).
__device__ __forceinline__ Pt contract(bool back, f3 x, f3 bmin, f3 bsize)
{
    Pt p;
    const f3 u = mk3((x.x - bmin.x) / bsize.x * 4.0f - 2.0f, (x.y - bmin.y) / bsize.y * 4.0f - 2.0f, (x.z - bmin.z) / bsize.z * 4.0f - 2.0f);
    const f3 a = mk3(4.0f / bsize.x, 4.0f / bsize.y, 4.0f / bsize.z);
    if (!back) {
        p.c = u; p.jd = a; p.u = u; p.fp = 0.0f; p.k = 0;
    } else {
        const float ax = fabsf(u.x), ay = fabsf(u.y), az = fabsf(u.z);
        float n = ax; int k = 0;                       // torch.max returns the first maximal index
        if (ay > n) { n = ay; k = 1; }
        if (az > n) { n = az; k = 2; }
        const float f = (2.0f - 1.0f / n) / n;
        // rounded product: the encode adds 2 next, and an FMA would differ from torch's separately rounded u * f
        p.c = mk3(__fmul_rn(u.x, f), __fmul_rn(u.y, f), __fmul_rn(u.z, f));
        p.jd = a * f;
        p.u = u;
        const float uk = k == 0 ? u.x : (k == 1 ? u.y : u.z);
        const float ak = k == 0 ? a.x : (k == 1 ? a.y : a.z);
        // f(n) = 2/n - 1/n^2, f'(n) = -2/n^2 + 2/n^3; d n / d u_k = sign(u_k)
        p.fp = (-2.0f / (n * n) + 2.0f / (n * n * n)) * (uk >= 0.0f ? 1.0f : -1.0f) * ak;
        p.k = k;
    }
    return p;
}

// g_c (gradient w.r.t. the contracted point) -> gradient w.r.t. the world-space sample
__device__ __forceinline__ f3 contract_bwd(bool back, const Pt& p, f3 gc)
{
    f3 gx = gc * p.jd;
    if (back) {
        const float s = dot3(gc, p.u) * p.fp;          // rank-one term: (g . u) f'(n) dn/du_k a_k on axis k
        if (p.k == 0) gx.x += s; else if (p.k == 1) gx.y += s; else gx.z += s;
    }
    return gx;
}

// L2 eviction policy of the forward's table gathers (snrf_field_set_fwd_l2_policy).  A level slice at T = 2^24 is 128 MiB
// against 126 MB of L2 that the kernel's own output streams also pass through: under the default policy the slice thrashes
// (lts hit rate 27 %, every sector fetched ~3x per launch).  mode 1: every gather evict_last; mode 2: the first `pin_bytes`
// of the level slice evict_last and the rest evict_first (a pinned part that does fit, instead of an LRU cycle over a
// working set that does not); mode 3: the same split as a fraction of the accesses (`pin_bytes` / 2^16).
__device__ __forceinline__ uint64_t fwd_table_policy(int mode, const float2* slice, uint32_t slice_bytes, uint32_t pin_bytes)
{
    uint64_t p = 0;
    if (mode == 1) {
        asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    } else if (mode == 2) {
        asm volatile("createpolicy.range.global.L2::evict_last.L2::evict_first.b64 %0, [%1], %2, %3;" : "=l"(p) : "l"(slice), "r"(pin_bytes), "r"(slice_bytes));
    } else if (mode == 3) {
        const float frac = (float)pin_bytes * (1.0f / 65536.0f);
        asm volatile("createpolicy.fractional.L2::evict_last.L2::evict_first.b64 %0, %1;" : "=l"(p) : "f"(frac));
    }
    return p;
}
__device__ __forceinline__ float2 ldg2_policy(const float2* a, uint64_t pol)
{
    float2 v;
    asm volatile("ld.global.nc.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;" : "=f"(v.x), "=f"(v.y) : "l"(a), "l"(pol));
    return v;
}

// x-pair gathers (snrf_field_set_fwd_pair_loads).  The hash is linear in x, so the two corners of an x-edge sit in one
// aligned 16-byte slot when the cell's x is even, and in one 32-byte sector three times out of four.  Issued as two 8-byte
// loads they arrive at the L2 as two sector requests (the L1 does not merge them: ncu counts exactly 8 sector requests per
// sample and level on the fine levels).  mode 1: one 16-byte load for an aligned pair; mode 2: one 32-byte load of the
// sector of the first corner, the second corner picked from it when it lies in the same sector, fetched by itself otherwise.
__device__ __forceinline__ float2 pick2(const float v[8], uint32_t s)
{
    const float ax = (s & 1u) ? v[2] : v[0], ay = (s & 1u) ? v[3] : v[1];
    const float bx = (s & 1u) ? v[6] : v[4], by = (s & 1u) ? v[7] : v[5];
    return make_float2((s & 2u) ? bx : ax, (s & 2u) ? by : ay);
}
__device__ __forceinline__ void ld_sector(const float2* a, uint64_t pol, bool hint, float v[8])
{
    if (hint)
        asm volatile("ld.global.nc.L2::cache_hint.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(a), "l"(pol));
    else
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(a));
}
__device__ __forceinline__ float4 ld_pair16(const float2* a, uint64_t pol, bool hint)
{
    float4 v;
    if (hint) asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(a), "l"(pol));
    else v = __ldg(reinterpret_cast<const float4*>(a));
    return v;
}

template <int MODE, bool JAC, bool POLICY, int PAIR>
__global__ void __launch_bounds__(kThreads, (PAIR == 0 ? 5 : 4))      // 5 CTAs per SM: 4 (58 registers) 1.74 ms, 5 (46) 1.68 ms, 6 (40) 1.78 ms at C2
field_fwd_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ z_vals,
                 const float* __restrict__ points, const float* __restrict__ bmin_p, const float* __restrict__ bsize_p,
                 const float2* __restrict__ table, const int* __restrict__ res, float2* __restrict__ out, float2* __restrict__ jac,
                 const unsigned char* __restrict__ ray_valid, int ray_split, int N, int S, int L, uint32_t T, int lpb, int l_base,
                 int l2_mode, uint32_t pin_bytes, int pair_level)
{
    const uint32_t mask = T - 1u;
    f3 bmin = mk3(0, 0, 0), bsize = mk3(1, 1, 1);
    if (MODE != kNone) { bmin = ld3(bmin_p); bsize = ld3(bsize_p); }
    // lpb < 0: CTA row y walks the level PAIR (y, L - 1 - y): a coarse level (few vertices, L2 hits) next to a fine one (one
    // DRAM sector per corner), so that the two kinds of latency overlap inside a thread instead of running as separate waves
    const bool paired = lpb < 0;
    const int l_begin = paired ? (int)blockIdx.y : l_base + blockIdx.y * lpb, l_end = paired ? l_begin + 2 : min(L, l_begin + lpb);
    uint64_t pol = 0;
    if (POLICY) pol = fwd_table_policy(l2_mode, table + (size_t)l_begin * T, T * 8u, pin_bytes);   // POLICY: one level per CTA row
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
        f3 c;
        if (MODE == kNone) {
            c = ld3(points + 3 * (size_t)n);
        } else {
            const int r = n / S;
            if (ray_valid != nullptr && !ray_valid[r]) continue;        // masked-out ray: its rows are never read
            c = contract(r >= ray_split, sample_pos(ld3(rays_o + 3 * (size_t)r), ld3(rays_d + 3 * (size_t)r), z_vals[n]), bmin, bsize).c;
        }
        for (int li = l_begin; li < l_end; ++li) {
            const int l = (paired && li > l_begin) ? L - 1 - l_begin : li;
            if (paired && li > l_begin && l == l_begin) break;         // odd L: the middle level once
            const Cell cell = locate_bg(c, res + 3 * l);
            uint32_t idx[8];
            corner_idx(idx, cell, mask);
            const float2* tl = table + (size_t)l * T;
            float2 f[8];
            if (PAIR == 2 && l >= pair_level) {
                float v[4][8];
#pragma unroll
                for (int j = 0; j < 4; ++j) ld_sector(tl + (idx[j] & ~3u), pol, POLICY, v[j]);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if ((idx[j] >> 2) != (idx[j + 4] >> 2)) f[j + 4] = POLICY ? ldg2_policy(tl + idx[j + 4], pol) : ldg2(tl + idx[j + 4]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    f[j] = pick2(v[j], idx[j] & 3u);
                    if ((idx[j] >> 2) == (idx[j + 4] >> 2)) f[j + 4] = pick2(v[j], idx[j + 4] & 3u);
                }
            } else if (PAIR == 1 && l >= pair_level) {
                float4 v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const bool paired16 = (idx[j] ^ idx[j + 4]) == 1u;
                    if (paired16) v[j] = ld_pair16(tl + (idx[j] & ~1u), pol, POLICY);
                    else {
                        f[j] = POLICY ? ldg2_policy(tl + idx[j], pol) : ldg2(tl + idx[j]);
                        f[j + 4] = POLICY ? ldg2_policy(tl + idx[j + 4], pol) : ldg2(tl + idx[j + 4]);
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if ((idx[j] ^ idx[j + 4]) == 1u) {
                        const bool odd = (idx[j] & 1u) != 0u;
                        f[j] = odd ? make_float2(v[j].z, v[j].w) : make_float2(v[j].x, v[j].y);
                        f[j + 4] = odd ? make_float2(v[j].x, v[j].y) : make_float2(v[j].z, v[j].w);
                    }
            } else {
#pragma unroll
                for (int k = 0; k < 8; ++k) f[k] = POLICY ? ldg2_policy(tl + idx[k], pol) : ldg2(tl + idx[k]);
            }
            float w[8];
            corner_w(w, cell);
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < 8; ++k) { acc.x += w[k] * f[k].x; acc.y += w[k] * f[k].y; }
            __stcs(out + (size_t)l * N + n, acc);          // streaming: the table, not the outputs, should stay in L2
            if (JAC) {
                const float ax = 1.0f - cell.ox, ay = 1.0f - cell.oy, az = 1.0f - cell.oz;
                const float dxw[8] = {-ay * az, -ay * cell.oz, -cell.oy * az, -cell.oy * cell.oz, ay * az, ay * cell.oz, cell.oy * az, cell.oy * cell.oz};
                const float dyw[8] = {-ax * az, -ax * cell.oz, ax * az, ax * cell.oz, -cell.ox * az, -cell.ox * cell.oz, cell.ox * az, cell.ox * cell.oz};
                const float dzw[8] = {-ax * ay, ax * ay, -ax * cell.oy, ax * cell.oy, -cell.ox * ay, cell.ox * ay, -cell.ox * cell.oy, cell.ox * cell.oy};
                float2 dx = make_float2(0.f, 0.f), dy = dx, dz = dx;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    dx.x += f[k].x * dxw[k]; dx.y += f[k].y * dxw[k];
                    dy.x += f[k].x * dyw[k]; dy.y += f[k].y * dyw[k];
                    dz.x += f[k].x * dzw[k]; dz.y += f[k].y * dzw[k];
                }
                float2* j = jac + (size_t)l * 3 * N + n;
                __stcs(j, make_float2(dx.x * cell.sx, dx.y * cell.sx));
                __stcs(j + (size_t)N, make_float2(dy.x * cell.sy, dy.y * cell.sy));
                __stcs(j + 2 * (size_t)N, make_float2(dz.x * cell.sz, dz.y * cell.sz));
            }
        }
    }
}

// Backward: gradient scatter into the table (index range `pass` of `1 << pass_bits` per level) and,
// on pass 0, d L / d (rays_o, rays_d) or d L / d points from the stored Jacobians.
template <int MODE>
__global__ void __launch_bounds__(kThreads)
field_bwd_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ z_vals,
                 const float* __restrict__ points, const float* __restrict__ bmin_p, const float* __restrict__ bsize_p,
                 const int* __restrict__ res, const float2* __restrict__ grad, const float2* __restrict__ jac,
                 float* __restrict__ grad_o, float* __restrict__ grad_d, float* __restrict__ grad_points, float2* __restrict__ grad_table,
                 const unsigned char* __restrict__ ray_valid, int ray_split, int N, int S, int L, uint32_t T, int pass_bits,
                 int range_shift, int aggregate_levels)
{
    const uint32_t mask = T - 1u;
    const int lane = threadIdx.x & 31;
    const int l = blockIdx.y >> pass_bits;
    const uint32_t pass = blockIdx.y & ((1u << pass_bits) - 1u);
    f3 bmin = mk3(0, 0, 0), bsize = mk3(1, 1, 1);
    if (MODE != kNone) { bmin = ld3(bmin_p); bsize = ld3(bsize_p); }
    const bool want_rays = (pass == 0) && jac != nullptr && (MODE == kNone ? grad_points != nullptr : (grad_o != nullptr || grad_d != nullptr));
    float2* gl = grad_table + (size_t)l * T;

    const int warp_base0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31;
    for (int wb = warp_base0; wb < N; wb += gridDim.x * blockDim.x) {
        const int n = wb + lane;
        const bool live = n < N && (MODE == kNone || ray_valid == nullptr || ray_valid[n / S] != 0);
        Pt p;
        float z = 0.0f;
        int r = -1;
        if (MODE == kNone) {
            p.c = live ? ld3(points + 3 * (size_t)n) : mk3(0, 0, 0);
        } else {
            r = live ? n / S : -1;
            z = live ? z_vals[n] : 0.0f;
            const f3 x = live ? sample_pos(ld3(rays_o + 3 * (size_t)r), ld3(rays_d + 3 * (size_t)r), z) : mk3(0, 0, 0);
            p = contract(r >= ray_split, x, bmin, bsize);
        }
        const float2 g = live ? __ldcs(grad + (size_t)l * N + n) : make_float2(0.f, 0.f);
        const Cell cell = locate_bg(p.c, res + 3 * l);
        uint32_t idx[8]; float w[8];
        corner_idx(idx, cell, mask);
        corner_w(w, cell);

        // ---- table gradient: only the corners whose index falls into this pass's range
        bool done = false;
        if (l < aggregate_levels) {
            const unsigned long long key = live
                ? (((unsigned long long)(uint32_t)cell.ix & 0x1fffffull) << 42) | (((unsigned long long)(uint32_t)cell.iy & 0x1fffffull) << 21) |
                  ((unsigned long long)(uint32_t)cell.iz & 0x1fffffull)
                : ~0ull;
            const unsigned long long prev = __shfl_up_sync(0xffffffffu, key, 1);
            const bool head = (lane == 0) || (prev != key);
            const unsigned heads = __ballot_sync(0xffffffffu, head);
            if (__popc(heads) <= 12) {
                const int seg = __popc(heads & ((2u << lane) - 1u));
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float sx = seg_sum(w[k] * g.x, seg, lane);
                    const float sy = seg_sum(w[k] * g.y, seg, lane);
                    if (head && live && (idx[k] >> range_shift) == pass) atomicAdd(gl + idx[k], make_float2(sx, sy));
                }
                done = true;
            }
        }
        if (!done && live) {
            // The hash is linear in x (h = x ^ ...): the two corners of an x-edge with even x differ in bit 0 only, i.e.
            // they are the two halves of one aligned 16-byte slot -> one red.v4 instead of two red.v2 (the L2 reduction
            // units, not HBM, bound this kernel: profiles/r1c_top_kernels_full.md; measured 1.98 -> 1.85 ms).
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t i0 = idx[j], i1 = idx[j + 4];
                const float2 v0 = make_float2(w[j] * g.x, w[j] * g.y), v1 = make_float2(w[j + 4] * g.x, w[j + 4] * g.y);
                if ((i0 ^ i1) == 1u) {
                    if ((i0 >> range_shift) == pass) {
                        const bool swap = (i0 & 1u) != 0u;
                        atomicAdd(reinterpret_cast<float4*>(gl + (i0 & ~1u)),
                                  swap ? make_float4(v1.x, v1.y, v0.x, v0.y) : make_float4(v0.x, v0.y, v1.x, v1.y));
                    }
                } else {
                    if ((i0 >> range_shift) == pass) atomicAdd(gl + i0, v0);
                    if ((i1 >> range_shift) == pass) atomicAdd(gl + i1, v1);
                }
            }
        }

        // ---- gradient w.r.t. the sample position, from the stored Jacobian
        if (want_rays) {
            f3 gc = mk3(0, 0, 0);
            if (live) {
                const float2* j = jac + (size_t)l * 3 * N + n;
                const float2 jx = __ldcs(j), jy = __ldcs(j + (size_t)N), jz = __ldcs(j + 2 * (size_t)N);
                gc = mk3(g.x * jx.x + g.y * jx.y, g.x * jy.x + g.y * jy.y, g.x * jz.x + g.y * jz.y);
            }
            if (MODE == kNone) {
                if (live) {
                    atomicAdd(grad_points + 3 * (size_t)n + 0, gc.x);
                    atomicAdd(grad_points + 3 * (size_t)n + 1, gc.y);
                    atomicAdd(grad_points + 3 * (size_t)n + 2, gc.z);
                }
            } else {
                f3 gx = live ? contract_bwd(r >= ray_split, p, gc) : mk3(0, 0, 0);
                f3 gz = gx * z;
                // all lanes of the warp usually belong to one ray: reduce first
                const int r0 = __shfl_sync(0xffffffffu, r, 0);
                if (__all_sync(0xffffffffu, r == r0 || r < 0)) {
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) {
                        gx.x += __shfl_xor_sync(0xffffffffu, gx.x, off); gx.y += __shfl_xor_sync(0xffffffffu, gx.y, off);
                        gx.z += __shfl_xor_sync(0xffffffffu, gx.z, off);
                        gz.x += __shfl_xor_sync(0xffffffffu, gz.x, off); gz.y += __shfl_xor_sync(0xffffffffu, gz.y, off);
                        gz.z += __shfl_xor_sync(0xffffffffu, gz.z, off);
                    }
                    if (lane == 0 && r0 >= 0) {
                        if (grad_o) { atomicAdd(grad_o + 3 * (size_t)r0, gx.x); atomicAdd(grad_o + 3 * (size_t)r0 + 1, gx.y); atomicAdd(grad_o + 3 * (size_t)r0 + 2, gx.z); }
                        if (grad_d) { atomicAdd(grad_d + 3 * (size_t)r0, gz.x); atomicAdd(grad_d + 3 * (size_t)r0 + 1, gz.y); atomicAdd(grad_d + 3 * (size_t)r0 + 2, gz.z); }
                    }
                } else if (live) {
                    if (grad_o) { atomicAdd(grad_o + 3 * (size_t)r, gx.x); atomicAdd(grad_o + 3 * (size_t)r + 1, gx.y); atomicAdd(grad_o + 3 * (size_t)r + 2, gx.z); }
                    if (grad_d) { atomicAdd(grad_d + 3 * (size_t)r, gz.x); atomicAdd(grad_d + 3 * (size_t)r + 1, gz.y); atomicAdd(grad_d + 3 * (size_t)r + 2, gz.z); }
                }
            }
        }
    }
}

// Backward, second form: every thread owns R consecutive samples of the level-major arrays (consecutive samples of one
// ray) and merges the samples that fall into the same cell IN REGISTERS before it touches the table: a run of samples in
// one cell costs 16 FMAs per sample and one set of 8 corner reductions per run.  On the coarse and middle levels runs
// are long (the cell is larger than the sample spacing), on the fine levels every sample is its own run and the kernel
// degenerates to the plain scatter.  An alternative to the cross-lane segmented sums of field_bwd_kernel, which spend ~320
// shuffle / select instructions per sample on the aggregated levels (ncu, profiles/r1e_top_kernels_full.md: 60 % of the
// issue slots busy, 613 instructions per sample-level, L2 reduction units at 29 %); see g_run_length for the measurement.
template <int MODE, int R>
__global__ void __launch_bounds__(kThreads)
field_bwd_runs_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ z_vals,
                      const float* __restrict__ points, const float* __restrict__ bmin_p, const float* __restrict__ bsize_p,
                      const int* __restrict__ res, const float2* __restrict__ grad, const float2* __restrict__ jac,
                      float* __restrict__ grad_o, float* __restrict__ grad_d, float* __restrict__ grad_points, float2* __restrict__ grad_table,
                      const unsigned char* __restrict__ ray_valid, int ray_split, int N, int S, int L, uint32_t T, int pass_bits,
                      int range_shift)
{
    const uint32_t mask = T - 1u;
    const int lane = threadIdx.x & 31;
    const int l = blockIdx.y >> pass_bits;
    const uint32_t pass = blockIdx.y & ((1u << pass_bits) - 1u);
    f3 bmin = mk3(0, 0, 0), bsize = mk3(1, 1, 1);
    if (MODE != kNone) { bmin = ld3(bmin_p); bsize = ld3(bsize_p); }
    const bool want_rays = (pass == 0) && jac != nullptr && (MODE == kNone ? grad_points != nullptr : (grad_o != nullptr || grad_d != nullptr));
    float2* gl = grad_table + (size_t)l * T;
    const int* rl = res + 3 * l;

    uint32_t ridx[8];
    float ax[8], ay[8];
    int cx = 0, cy = 0, cz = 0;
    bool have = false;
    auto flush = [&]() {
        // x-adjacent corners that share an aligned 16-byte slot go out as one red.v4 (see field_bwd_kernel)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t i0 = ridx[j], i1 = ridx[j + 4];
            if ((i0 ^ i1) == 1u) {
                if ((i0 >> range_shift) == pass) {
                    const bool swap = (i0 & 1u) != 0u;
                    atomicAdd(reinterpret_cast<float4*>(gl + (i0 & ~1u)),
                              swap ? make_float4(ax[j + 4], ay[j + 4], ax[j], ay[j]) : make_float4(ax[j], ay[j], ax[j + 4], ay[j + 4]));
                }
            } else {
                if ((i0 >> range_shift) == pass) atomicAdd(gl + i0, make_float2(ax[j], ay[j]));
                if ((i1 >> range_shift) == pass) atomicAdd(gl + i1, make_float2(ax[j + 4], ay[j + 4]));
            }
        }
    };

    const long long warp0 = (long long)(blockIdx.x * blockDim.x + threadIdx.x) & ~31ll;
    for (long long wb = warp0; wb * R < N; wb += (long long)gridDim.x * blockDim.x) {
        const long long n0 = (wb + lane) * R;
        int r0 = -1, rem0 = 0;
        if (MODE != kNone && n0 < N) { r0 = (int)(n0 / S); rem0 = (int)(n0 - (long long)r0 * S); }
        f3 sum_x = mk3(0, 0, 0), sum_z = mk3(0, 0, 0);         // d L / d rays_o, d L / d rays_d of ray r0 from this thread's samples
        have = false;
#pragma unroll
        for (int i = 0; i < R; ++i) {
            const long long n = n0 + i;
            if (n >= N) break;
            int r = r0;
            if (MODE != kNone) {
                int rem = rem0 + i;
                while (rem >= S) { rem -= S; ++r; }
                if (ray_valid != nullptr && !ray_valid[r]) continue;
            }
            Pt p;
            float z = 0.0f;
            if (MODE == kNone) {
                p.c = ld3(points + 3 * (size_t)n);
            } else {
                z = z_vals[n];
                p = contract(r >= ray_split, sample_pos(ld3(rays_o + 3 * (size_t)r), ld3(rays_d + 3 * (size_t)r), z), bmin, bsize);
            }
            const float2 g = __ldcs(grad + (size_t)l * N + n);
            const Cell cell = locate_bg(p.c, rl);
            float w[8];
            corner_w(w, cell);
            if (have && cell.ix == cx && cell.iy == cy && cell.iz == cz) {
#pragma unroll
                for (int k = 0; k < 8; ++k) { ax[k] += w[k] * g.x; ay[k] += w[k] * g.y; }
            } else {
                if (have) flush();
                corner_idx(ridx, cell, mask);
#pragma unroll
                for (int k = 0; k < 8; ++k) { ax[k] = w[k] * g.x; ay[k] = w[k] * g.y; }
                cx = cell.ix; cy = cell.iy; cz = cell.iz;
                have = true;
            }
            if (want_rays) {
                const float2* j = jac + (size_t)l * 3 * N + n;
                const float2 jx = __ldcs(j), jy = __ldcs(j + (size_t)N), jz = __ldcs(j + 2 * (size_t)N);
                const f3 gc = mk3(g.x * jx.x + g.y * jx.y, g.x * jy.x + g.y * jy.y, g.x * jz.x + g.y * jz.y);
                if (MODE == kNone) {
                    atomicAdd(grad_points + 3 * (size_t)n + 0, gc.x);
                    atomicAdd(grad_points + 3 * (size_t)n + 1, gc.y);
                    atomicAdd(grad_points + 3 * (size_t)n + 2, gc.z);
                } else {
                    const f3 gx = contract_bwd(r >= ray_split, p, gc);
                    if (r == r0) { sum_x = sum_x + gx; sum_z = sum_z + gx * z; }
                    else {                                      // the thread's samples straddle two rays (S not a multiple of R)
                        if (grad_o) { atomicAdd(grad_o + 3 * (size_t)r, gx.x); atomicAdd(grad_o + 3 * (size_t)r + 1, gx.y); atomicAdd(grad_o + 3 * (size_t)r + 2, gx.z); }
                        if (grad_d) { atomicAdd(grad_d + 3 * (size_t)r, gx.x * z); atomicAdd(grad_d + 3 * (size_t)r + 1, gx.y * z); atomicAdd(grad_d + 3 * (size_t)r + 2, gx.z * z); }
                    }
                }
            }
        }
        if (have) flush();
        if (want_rays && MODE != kNone) {
            // the 32 R samples of a warp usually belong to one ray: reduce across the warp first
            const int rl0 = __shfl_sync(0xffffffffu, r0, 0);
            if (__all_sync(0xffffffffu, r0 == rl0 || r0 < 0)) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    sum_x.x += __shfl_xor_sync(0xffffffffu, sum_x.x, off); sum_x.y += __shfl_xor_sync(0xffffffffu, sum_x.y, off);
                    sum_x.z += __shfl_xor_sync(0xffffffffu, sum_x.z, off);
                    sum_z.x += __shfl_xor_sync(0xffffffffu, sum_z.x, off); sum_z.y += __shfl_xor_sync(0xffffffffu, sum_z.y, off);
                    sum_z.z += __shfl_xor_sync(0xffffffffu, sum_z.z, off);
                }
                if (lane == 0 && rl0 >= 0) {
                    if (grad_o) { atomicAdd(grad_o + 3 * (size_t)rl0, sum_x.x); atomicAdd(grad_o + 3 * (size_t)rl0 + 1, sum_x.y); atomicAdd(grad_o + 3 * (size_t)rl0 + 2, sum_x.z); }
                    if (grad_d) { atomicAdd(grad_d + 3 * (size_t)rl0, sum_z.x); atomicAdd(grad_d + 3 * (size_t)rl0 + 1, sum_z.y); atomicAdd(grad_d + 3 * (size_t)rl0 + 2, sum_z.z); }
                }
            } else if (r0 >= 0) {
                if (grad_o) { atomicAdd(grad_o + 3 * (size_t)r0, sum_x.x); atomicAdd(grad_o + 3 * (size_t)r0 + 1, sum_x.y); atomicAdd(grad_o + 3 * (size_t)r0 + 2, sum_x.z); }
                if (grad_d) { atomicAdd(grad_d + 3 * (size_t)r0, sum_z.x); atomicAdd(grad_d + 3 * (size_t)r0 + 1, sum_z.y); atomicAdd(grad_d + 3 * (size_t)r0 + 2, sum_z.z); }
            }
        }
    }
}

// =====================================================================================================================
// Backward, third form: the scatter fused with the sparse Adam update of the table ("scatter + update").
//
// The table gradient never exists as a [L][T] array in HBM.  The backward runs as a short sequence of launches:
//   (1) geometry + ray gradient, once per sample: contracted point c -> cpts [3][N] (SoA, NaN = masked-out sample),
//       g_c = sum_l g_l . J_l over all levels, the contraction's backward, one warp reduction and one set of atomics per
//       32 samples (field_bwd_kernel redoes the contraction -- ~10 IEEE divisions -- and the warp reduction for every
//       (level, index range); that prologue was 60 % of its issue slots, profiles/r1f_top_kernels_full.md);
//   (2) for every index-range slice of the table that fits the L2-resident scratch (2^23 entries = 64 MiB: half a level at
//       T = 2^24, several whole levels at small T):  scatter the slice's gradient into the scratch (reductions hit L2 --
//       the scratch is reused by every slice and stays resident, so no sector is fetched from / evicted to HBM), then
//   (3) apply Adam to the slice: read the scratch (L2), update p / m / v where the gradient is non-zero (the only HBM
//       traffic: 24 B per touched float), clear the scratch behind it.
// Semantics = snrf_field_encode_bwd into a zeroed gradient table followed by snrf_adam_step(zero_grad = 1).
// =====================================================================================================================

// L2 residency hints for the scratch of the scatter + update fusion: reductions into it and the Adam pass's read / clear of
// it carry an evict_last cache policy, the streams that pass by once (gradients, p / m / v) an evict-first one, so that the
// 64 MiB slice being reduced into is what the L2 keeps (without hints a fine-level slice wrote 95 MB to and re-read 68 MB
// from DRAM per scatter, and the Adam pass fetched its 67 MB again: profiles/r2d_fused_bwd_full.md).
// Programmatic dependent launch (snrf_field_set_pdl): the scatter / Adam slices of the fused backward are 56 short dependent
// launches; launched with the programmatic-stream-serialization attribute a kernel's CTAs are scheduled while the previous
// kernel drains its last wave and wait here until it has completed and flushed.  A no-op for a plain launch.
// (launch_dependents right behind the wait: once every CTA of this grid has STARTED, the next grid's CTAs may take the slots
// its last wave frees -- they then sit in their own wait until this grid has completed.)
__device__ __forceinline__ void grid_dependency_wait()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void red_add2(float2* a, float x, float y, uint64_t pol, bool hint)
{
    if (hint) asm volatile("red.global.add.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(a), "f"(x), "f"(y), "l"(pol) : "memory");
    else atomicAdd(a, make_float2(x, y));
}
__device__ __forceinline__ void red_add4(float4* a, float x, float y, float z, float w, uint64_t pol, bool hint)
{
    if (hint) asm volatile("red.global.add.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(a), "f"(x), "f"(y), "f"(z), "f"(w), "l"(pol) : "memory");
    else atomicAdd(a, make_float4(x, y, z, w));
}
__device__ __forceinline__ float4 ld4_hint(const float4* a, uint64_t pol, bool hint)
{
    float4 v;
    if (hint) asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(a), "l"(pol));
    else v = __ldcg(a);
    return v;
}
__device__ __forceinline__ void st4_hint(float4* a, float4 v, uint64_t pol, bool hint)
{
    if (hint) asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
    else *a = v;
}

template <int MODE>
__global__ void __launch_bounds__(kThreads)
field_geom_raygrad_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, const float* __restrict__ z_vals,
                          const float* __restrict__ points, const float* __restrict__ bmin_p, const float* __restrict__ bsize_p,
                          const float2* __restrict__ grad, const float2* __restrict__ jac,
                          float* __restrict__ grad_o, float* __restrict__ grad_d, float* __restrict__ grad_points,
                          float* __restrict__ cpts, const unsigned char* __restrict__ ray_valid, int ray_split, int N, int S, int L,
                          const unsigned char* __restrict__ sample_live)
{
    const int lane = threadIdx.x & 31;
    f3 bmin = mk3(0, 0, 0), bsize = mk3(1, 1, 1);
    if (MODE != kNone) { bmin = ld3(bmin_p); bsize = ld3(bsize_p); }
    const bool want_rays = jac != nullptr && (MODE == kNone ? grad_points != nullptr : (grad_o != nullptr || grad_d != nullptr));
    const float qnan = __int_as_float(0x7fc00000);
    const int warp_base0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31;
    for (int wb = warp_base0; wb < N; wb += gridDim.x * blockDim.x) {
        const int n = wb + lane;
        // (sample_live: early-ray-termination flags -- a dead sample has no gradient row and is marked like a masked-out one)
        const bool live = n < N && (MODE == kNone || ray_valid == nullptr || ray_valid[n / S] != 0) && (sample_live == nullptr || sample_live[n] != 0);
        Pt p;
        float z = 0.0f;
        int r = -1;
        if (MODE == kNone) {
            p.c = live ? ld3(points + 3 * (size_t)n) : mk3(0, 0, 0);
        } else {
            r = live ? n / S : -1;
            z = live ? z_vals[n] : 0.0f;
            const f3 x = live ? sample_pos(ld3(rays_o + 3 * (size_t)r), ld3(rays_d + 3 * (size_t)r), z) : mk3(0, 0, 0);
            p = contract(r >= ray_split, x, bmin, bsize);
        }
        if (n < N) {
            __stcg(cpts + n, live ? p.c.x : qnan);
            __stcg(cpts + (size_t)N + n, live ? p.c.y : qnan);
            __stcg(cpts + 2 * (size_t)N + n, live ? p.c.z : qnan);
        }
        if (!want_rays) continue;
        f3 gc = mk3(0, 0, 0);
        if (live) {
#pragma unroll 4
            for (int l = 0; l < L; ++l) {
                const float2 g = __ldcs(grad + (size_t)l * N + n);
                const float2* j = jac + (size_t)l * 3 * N + n;
                const float2 jx = __ldcs(j), jy = __ldcs(j + (size_t)N), jz = __ldcs(j + 2 * (size_t)N);
                gc.x += g.x * jx.x + g.y * jx.y;
                gc.y += g.x * jy.x + g.y * jy.y;
                gc.z += g.x * jz.x + g.y * jz.y;
            }
        }
        if (MODE == kNone) {
            if (live) {       // ACCUMULATES, as snrf_field_encode_bwd does
                atomicAdd(grad_points + 3 * (size_t)n + 0, gc.x);
                atomicAdd(grad_points + 3 * (size_t)n + 1, gc.y);
                atomicAdd(grad_points + 3 * (size_t)n + 2, gc.z);
            }
        } else {
            f3 gx = live ? contract_bwd(r >= ray_split, p, gc) : mk3(0, 0, 0);
            f3 gz = gx * z;
            const int r0 = __shfl_sync(0xffffffffu, r, 0);
            if (__all_sync(0xffffffffu, r == r0 || r < 0)) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    gx.x += __shfl_xor_sync(0xffffffffu, gx.x, off); gx.y += __shfl_xor_sync(0xffffffffu, gx.y, off);
                    gx.z += __shfl_xor_sync(0xffffffffu, gx.z, off);
                    gz.x += __shfl_xor_sync(0xffffffffu, gz.x, off); gz.y += __shfl_xor_sync(0xffffffffu, gz.y, off);
                    gz.z += __shfl_xor_sync(0xffffffffu, gz.z, off);
                }
                if (lane == 0 && r0 >= 0) {
                    if (grad_o) { atomicAdd(grad_o + 3 * (size_t)r0, gx.x); atomicAdd(grad_o + 3 * (size_t)r0 + 1, gx.y); atomicAdd(grad_o + 3 * (size_t)r0 + 2, gx.z); }
                    if (grad_d) { atomicAdd(grad_d + 3 * (size_t)r0, gz.x); atomicAdd(grad_d + 3 * (size_t)r0 + 1, gz.y); atomicAdd(grad_d + 3 * (size_t)r0 + 2, gz.z); }
                }
            } else if (live) {
                if (grad_o) { atomicAdd(grad_o + 3 * (size_t)r, gx.x); atomicAdd(grad_o + 3 * (size_t)r + 1, gx.y); atomicAdd(grad_o + 3 * (size_t)r + 2, gx.z); }
                if (grad_d) { atomicAdd(grad_d + 3 * (size_t)r, gz.x); atomicAdd(grad_d + 3 * (size_t)r + 1, gz.y); atomicAdd(grad_d + 3 * (size_t)r + 2, gz.z); }
            }
        }
    }
}

// Scatter of levels [l0, l0 + gridDim.y), index range `pass` (of 1 << pass_bits per level), into the scratch:
// entry idx of level l lands at scratch[(l - l0) * slice + (idx & (slice - 1))], slice = T >> pass_bits.
// Reads only cpts (12 B) and the incoming gradient (8 B) per sample and level.
template <bool HINT>
__global__ void __launch_bounds__(kThreads)
field_scatter_slice_kernel(const float* __restrict__ cpts, const int* __restrict__ res, const float2* __restrict__ grad,
                           float2* __restrict__ scratch, int N, int l0, uint32_t T, uint32_t pass, int range_shift, int aggregate_levels)
{
    const uint32_t mask = T - 1u;
    constexpr bool hint = HINT;
    const uint64_t pol = l2_policy_evict_last();
    const uint32_t slice_mask = (1u << range_shift) - 1u;
    grid_dependency_wait();             // (programmatic dependent launch: everything above overlapped the previous kernel's tail)
    const int lane = threadIdx.x & 31;
    const int l = l0 + blockIdx.y;
    float2* gl = scratch + ((size_t)blockIdx.y << range_shift);
    const float2* gin = grad + (size_t)l * N;
    const int* rl = res + 3 * l;
    const bool aggregate = l < aggregate_levels;
    const int warp_base0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31;
    for (int wb = warp_base0; wb < N; wb += gridDim.x * blockDim.x) {
        const int n = wb + lane;
        f3 c = mk3(0, 0, 0);
        float2 g = make_float2(0.f, 0.f);
        bool live = false;
        if (n < N) {
            c = mk3(__ldcg(cpts + n), __ldcg(cpts + (size_t)N + n), __ldcg(cpts + 2 * (size_t)N + n));
            live = c.x == c.x;                         // NaN marks a sample of a masked-out ray
            if (live) g = __ldcs(gin + n);
        }
        const Cell cell = locate_bg(c, rl);
        uint32_t idx[8]; float w[8];
        corner_idx(idx, cell, mask);
        corner_w(w, cell);
        // per-corner contributions of this lane; on the aggregated levels lanes of one cell are merged first (segmented
        // warp sums over runs of equal cells in consecutive lanes) and only the run's first lane emits
        float vx[8], vy[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { vx[k] = w[k] * g.x; vy[k] = w[k] * g.y; }
        bool emit = live;
        if (aggregate) {
            const unsigned long long key = live
                ? (((unsigned long long)(uint32_t)cell.ix & 0x1fffffull) << 42) | (((unsigned long long)(uint32_t)cell.iy & 0x1fffffull) << 21) |
                  ((unsigned long long)(uint32_t)cell.iz & 0x1fffffull)
                : ~0ull;
            const unsigned long long prev = __shfl_up_sync(0xffffffffu, key, 1);
            const bool head = (lane == 0) || (prev != key);
            const unsigned heads = __ballot_sync(0xffffffffu, head);
            if (__popc(heads) <= 16) {
                // The lane's run ends right before the next head above it: lane + off is inside the run iff it is below that
                // bound -- one comparison per step instead of a second shuffle of the run id; as many doubling steps as the
                // longest run of the warp needs (warp-uniform): the mid levels have runs of 1-4 samples.
                const unsigned above = heads & ~((2u << lane) - 1u);            // heads in lanes > lane
                const int run_end = above ? __ffs(above) - 1 : 32;               // first lane past my run
                const int longest = __reduce_max_sync(0xffffffffu, run_end - lane);
                for (int off = 1; off < longest; off <<= 1) {
                    const bool take = lane + off < run_end;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float ox = __shfl_down_sync(0xffffffffu, vx[k], off);
                        const float oy = __shfl_down_sync(0xffffffffu, vy[k], off);
                        if (take) { vx[k] += ox; vy[k] += oy; }
                    }
                }
                emit = head && live;
            }
        }
        if (emit) {
            // x-adjacent corners that share an aligned 16-byte slot go out as one red.v4 (see field_bwd_kernel)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t i0 = idx[j], i1 = idx[j + 4];
                if ((i0 ^ i1) == 1u) {
                    if ((i0 >> range_shift) == pass) {
                        const bool swap = (i0 & 1u) != 0u;
                        float4* dst = reinterpret_cast<float4*>(gl + ((i0 & slice_mask) & ~1u));
                        if (swap) red_add4(dst, vx[j + 4], vy[j + 4], vx[j], vy[j], pol, hint);
                        else red_add4(dst, vx[j], vy[j], vx[j + 4], vy[j + 4], pol, hint);
                    }
                } else {
                    if ((i0 >> range_shift) == pass) red_add2(gl + (i0 & slice_mask), vx[j], vy[j], pol, hint);
                    if ((i1 >> range_shift) == pass) red_add2(gl + (i1 & slice_mask), vx[j + 4], vy[j + 4], pol, hint);
                }
            }
        }
    }
}

// Adam over one contiguous slice of the table: n4 float4 groups (two entries each) of p / m / v starting at the slice
// base, gradient from the scratch (cleared behind the read).  Elements whose gradient is exactly zero are skipped
// (cuda/adam_kernel.cu:43-51).
template <bool HINT>
__global__ void __launch_bounds__(kThreads)
adam_slice_kernel(float4* __restrict__ p4, float4* __restrict__ m4, float4* __restrict__ v4, float4* __restrict__ g4, long long n4,
                  adamcore::Hyper h)
{
    constexpr bool hint = HINT;
    const uint64_t pol = l2_policy_evict_last();
    __shared__ float s_bc[2];
    if (threadIdx.x == 0) {
        s_bc[0] = 1.0f - powf(h.b1, (float)h.step);
        s_bc[1] = 1.0f - powf(h.b2, (float)h.step);
    }
    grid_dependency_wait();             // (programmatic dependent launch: the scatter of this slice has to be complete from here on)
    __syncthreads();
    const float bc1 = s_bc[0], bc2 = s_bc[1];
    constexpr int kUnroll = 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x * kUnroll + threadIdx.x; base < n4; base += stride * kUnroll) {
        float4 gg[kUnroll], pp[kUnroll], mm[kUnroll], vv[kUnroll];
        bool act[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const long long i = base + (long long)u * blockDim.x;
            gg[u] = i < n4 ? ld4_hint(g4 + i, pol, hint) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const long long i = base + (long long)u * blockDim.x;
            act[u] = !(gg[u].x == 0.0f && gg[u].y == 0.0f && gg[u].z == 0.0f && gg[u].w == 0.0f);
            // (plain loads: evict-first hints on p / m / v were measured slower, 1.69 -> 2.2 ms per step)
            if (act[u]) { pp[u] = p4[i]; mm[u] = m4[i]; vv[u] = v4[i]; }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            if (!act[u]) continue;
            const long long i = base + (long long)u * blockDim.x;
            if (gg[u].x != 0.0f) adamcore::adam_elem(pp[u].x, gg[u].x, mm[u].x, vv[u].x, h, bc1, bc2);
            if (gg[u].y != 0.0f) adamcore::adam_elem(pp[u].y, gg[u].y, mm[u].y, vv[u].y, h, bc1, bc2);
            if (gg[u].z != 0.0f) adamcore::adam_elem(pp[u].z, gg[u].z, mm[u].z, vv[u].z, h, bc1, bc2);
            if (gg[u].w != 0.0f) adamcore::adam_elem(pp[u].w, gg[u].w, mm[u].w, vv[u].w, h, bc1, bc2);
            __stcs(p4 + i, pp[u]);          // streaming: p / m / v are not read again this step; the scratch should stay in L2
            __stcs(m4 + i, mm[u]);
            __stcs(v4 + i, vv[u]);
            st4_hint(g4 + i, make_float4(0.f, 0.f, 0.f, 0.f), pol, hint);
        }
    }
}

int g_occ_smem = 0;            // snrf_field_set_occupancy_smem: dynamic shared memory (unused) per CTA of the scatter / Adam slices
int g_pdl = 1;                 // snrf_field_set_pdl: scatter / Adam slices of the fused backward as programmatic dependent launches
// snrf_field_set_persist_mib (experiment, default 0 = off): the gradient scratch of the scatter + update fusion as a PERSISTING
// access-policy window of the slice launches (hardware L2 set-aside, cudaLimitPersistingL2CacheSize) on top of / instead of
// the per-instruction evict_last hints.
// Measured on B200 at C2 and REJECTED (profiles/r5g_persist_sweep.json): the set-aside shrinks the L2 everything else lives in --
// 48 / 64 / 72 MiB: step 8.87 -> 9.32 / 9.92 / 11.07 ms (encode forward 1.68 -> 1.80 / 2.08 / 2.55 ms, fused backward 4.15 -> 4.51 /
// 4.76 / 5.42 ms) -- and the window itself buys nothing over the hints (same times with the limit set and the window off).
int g_persist_mib = 0;
int g_persist_reserved_mib[64] = {};
size_t g_persist_max_window[64] = {}, g_persist_set_aside[64] = {};
thread_local cudaAccessPolicyWindow t_window = {};
thread_local bool t_window_on = false;
template <typename... KArgs, typename... Args>
inline void launch_dep(void (*kernel)(KArgs...), dim3 grid, cudaStream_t s, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = (size_t)g_occ_smem;      // (> 0 only in occupancy experiments: caps the resident CTAs per SM)
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (g_pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (t_window_on) {
        attr[n].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[n].val.accessPolicyWindow = t_window;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Reserves the L2 set-aside once per device and describes `bytes` at `base` as the persisting window of the following launches.
inline void persist_window_begin(void* base, size_t bytes)
{
    t_window_on = false;
    if (g_persist_mib <= 0) return;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return;
    int* reserved_mib = g_persist_reserved_mib;
    size_t *max_window = g_persist_max_window, *set_aside = g_persist_set_aside;
    if (reserved_mib[dev] != g_persist_mib) {
        int max_persist = 0, max_win = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
        cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, dev);
        size_t want = (size_t)g_persist_mib << 20;
        if (want > (size_t)max_persist) want = (size_t)max_persist;
        if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) != cudaSuccess) { cudaGetLastError(); return; }
        reserved_mib[dev] = g_persist_mib;
        set_aside[dev] = want;
        max_window[dev] = (size_t)max_win;
    }
    if (set_aside[dev] == 0 || max_window[dev] == 0) return;
    if (bytes > max_window[dev]) bytes = max_window[dev];
    t_window.base_ptr = base;
    t_window.num_bytes = bytes;
    t_window.hitRatio = bytes <= set_aside[dev] ? 1.0f : (float)((double)set_aside[dev] / (double)bytes);
    t_window.hitProp = cudaAccessPropertyPersisting;
    t_window.missProp = cudaAccessPropertyStreaming;
    t_window_on = true;
}
inline void persist_window_end() { t_window_on = false; }

inline int grid_x(int N)
{
    const int sms = snrf_sm_count();
    const int want = snrf_div_up(N, kThreads);
    const int wave = sms * 8;
    if (want <= wave) return want > 0 ? want : 1;
    const int waves = (want + wave - 1) / wave;
    return wave * (waves > 4 ? 4 : waves);
}

thread_local const unsigned char* t_sample_live = nullptr;     // set by the *_ert entry points around their call of the plain ones
int g_pass_bits_override = -1;
int g_aggregate_override = -1;
// Samples per thread of field_bwd_runs_kernel; 0 = the cross-lane kernel (default).  Measured on B200 at C2 (4.19 M samples,
// tools/sweep_field.py): cross-lane 3.69 ms, run-merging 4.15 / 4.35 / 4.39 ms at R = 2 / 4 / 8 -- merging R samples
// leaves 32 / R times more same-address reductions on the coarse levels than the cross-lane sums do, and that costs
// more than the shuffles it saves.  Kept selectable (and parity-tested) for tables / sample densities where runs are longer.
int g_fwd_pairing = 0;         // snrf_field_encode_fwd: CTA rows walk level pairs (y, L-1-y) (experiment)
int g_fwd_l2_mode = 0;         // snrf_field_set_fwd_l2_policy (no policy beats the default: profiles/r3a_fwd_per_level.md, r3e_fwd_sweep.json)
int g_fwd_pin_mib = 0;
int g_fwd_split_levels = 0;    // one forward launch per level (measurement hook)
int g_fwd_pair_mode = 0;       // snrf_field_set_fwd_pair_loads
int g_fwd_pair_level = 0;
int g_run_length = 0;
int g_bwd_impl = 1;            // snrf_field_encode_bwd: 1 = geometry / ray-gradient kernel + slim scatter per level and range (round 2), 0 = field_bwd_kernel (round 1)
int g_levels_per_group = 0;
long long g_slice_cap = 1ll << 23;      // entries of one fine slice (64 MiB of gradient: what stays L2-resident while it is reduced into)
int g_l2_hints = 1;                    // evict_last policy on the scratch accesses of the scatter + update fusion (see l2_policy_evict_last)
int g_coarse_concurrent = 1;           // the single-pass coarse levels run on a side stream next to the fine chain
int g_last_launches = 0;       // kernels launched by the last snrf_field_encode_bwd_adam call
int g_profile = 0;             // snrf_field_encode_bwd_adam: time the three kernel classes with CUDA events (synchronises!)
float g_profile_ms[4] = {0.f, 0.f, 0.f, 0.f};
// snrf_field_encode_bwd_adam: scatter of slice k+1 overlaps the Adam of slice k (two streams, split scratch).  Measured on
// B200 at C2 (profiles/r2c_fused_sweep.json): serial with a 64 MiB scratch 4.94 ms for the scatter + Adam phase; overlapped
// with two 64 MiB halves 4.73 ms, with two 32 MiB halves (four index ranges per level) 5.70 ms.  The two kernel classes
// both live on the L2 slices (reductions / HBM streaming through L2), so they contend instead of complementing each
// other; the 4 % do not pay for a second 64 MiB of scratch, hence off by default.
int g_overlap = 0;     // geometry + ray gradient, scatter slices, Adam slices of the last profiled call   // snrf_field_encode_bwd_adam: cap on whole levels per scatter / update pair (0 = as many as fit the scratch)
inline int pick_lpb(int L, int T)
{
    const long long level_bytes = (long long)T * 8;
    int lpb = 1;
    while (lpb * 2 <= L && (long long)lpb * 2 * level_bytes <= (16ll << 20)) lpb *= 2;
    return lpb;
}
// Index ranges per level for the scatter: keep the live gradient slice <= 64 MiB (half of the L2).
// Measured on B200 at T = 2^24, 2.1 M points (tools/sweep_field.py): 1 range 2.22 ms, 2 ranges 2.00 ms,
// 4 ranges 2.57 ms, 8 ranges 4.43 ms -- every extra pass re-derives the hash indices (~0.49 ms), which beyond two
// ranges costs more than the better L2 residency of the reductions saves.
inline int pick_pass_bits(int T)
{
    if (g_pass_bits_override >= 0) return g_pass_bits_override;
    int bits = 0;
    while (((long long)T * 8) >> bits > (64ll << 20) && bits < 4) ++bits;
    return bits;
}

}  // namespace

// ------------------------------- C ABI --------------------------------------
SNRF_API void snrf_field_set_passes_log2(int bits) { g_pass_bits_override = bits; }
SNRF_API void snrf_field_set_aggregate_levels(int n) { g_aggregate_override = n; }
// measurement hook (bench.py's roofline): when on, snrf_field_encode_bwd_adam brackets each of its launches with CUDA
// events, SYNCHRONISES the stream at the end and keeps the summed milliseconds per kernel class for
// snrf_field_last_profile(out[4]) = {geometry + ray gradient, scatter, Adam, scatter-and-Adam phase as a whole}.  With the
// two-stream overlap on, the two classes run concurrently and only [0] and [3] are meaningful.  Off by default.
SNRF_API int snrf_field_last_launch_count() { return g_last_launches; }
SNRF_API void snrf_field_set_profile(int on) { g_profile = on ? 1 : 0; }
SNRF_API void snrf_field_last_profile(float* out4) { for (int i = 0; i < 4; ++i) out4[i] = g_profile_ms[i]; }
SNRF_API void snrf_field_set_overlap(int on) { g_overlap = on ? 1 : 0; }
SNRF_API void snrf_field_set_l2_hints(int on) { g_l2_hints = on ? 1 : 0; }
// measurement hook: unused dynamic shared memory per CTA of the scatter / Adam slices, i.e. a cap on their resident CTAs per SM
SNRF_API void snrf_field_set_occupancy_smem(int bytes) { g_occ_smem = bytes > 0 ? (bytes > 48 * 1024 ? 48 * 1024 : bytes) : 0; }
// tuning hook: 1 (default) = the scatter / Adam slices of snrf_field_encode_bwd_adam are programmatic dependent launches
SNRF_API void snrf_field_set_pdl(int on) { g_pdl = on ? 1 : 0; }
// tuning hook (experiment): > 0 = MiB of hardware L2 set-aside; the gradient scratch of snrf_field_encode_bwd_adam becomes a
// persisting access-policy window of its slice launches.  0 (default) = off.
SNRF_API void snrf_field_set_persist_mib(int mib)
{
    g_persist_mib = mib > 0 ? mib : 0;
    int dev = 0;
    if (g_persist_mib == 0 && cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64 && g_persist_reserved_mib[dev] != 0) {
        // give the set-aside back: it costs L2 capacity even while no window is active
        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0);
        cudaCtxResetPersistingL2Cache();
        cudaGetLastError();
        g_persist_reserved_mib[dev] = 0;
        g_persist_set_aside[dev] = 0;
    }
}
SNRF_API void snrf_field_set_coarse_concurrent(int on) { g_coarse_concurrent = on ? 1 : 0; }
SNRF_API void snrf_field_set_slice_log2(int bits) { g_slice_cap = 1ll << (bits < 2 ? 2 : (bits > 30 ? 30 : bits)); }
SNRF_API void snrf_field_set_levels_per_group(int n) { g_levels_per_group = n > 0 ? n : 0; }
SNRF_API void snrf_field_set_fwd_pairing(int on) { g_fwd_pairing = on ? 1 : 0; }
// mode 0: default policy; 1: evict_last on every table gather; 2: the first `pin_mib` MiB of each level slice evict_last,
// the rest evict_first; 3: evict_last on the fraction pin_mib / 128 of the gathers, evict_first on the rest.  Applies when a
// CTA row walks ONE level (large tables); see fwd_table_policy.
SNRF_API void snrf_field_set_fwd_l2_policy(int mode, int pin_mib) { g_fwd_l2_mode = (mode >= 0 && mode <= 3) ? mode : 0; g_fwd_pin_mib = pin_mib > 0 ? pin_mib : 0; }
// x-pair gathers of the forward on levels >= first_level: 0 = eight 8-byte loads, 1 = one 16-byte load per aligned pair,
// 2 = one 32-byte sector load per pair + the second corner by itself when it lies in another sector
SNRF_API void snrf_field_set_fwd_pair_loads(int mode, int first_level) { g_fwd_pair_mode = (mode >= 0 && mode <= 2) ? mode : 0; g_fwd_pair_level = first_level > 0 ? first_level : 0; }
// measurement hook: one launch per level (ncu then reports L2 hit rate / DRAM bytes per level)
SNRF_API void snrf_field_set_fwd_split_levels(int on) { g_fwd_split_levels = on ? 1 : 0; }
SNRF_API void snrf_field_set_bwd_impl(int v) { g_bwd_impl = v ? 1 : 0; }
SNRF_API void snrf_field_set_run_length(int r) { g_run_length = (r == 2 || r == 4 || r == 8) ? r : 0; }

// mode 0: `points` [N,3] are already contracted (rays_o / rays_d / z_vals unused);
// mode 1 / 2: sample n = rays_o[n / S] + z_vals[n] * rays_d[n / S], contracted with the fore / background map of the
// box (box_min, box_size: device float[3], the DOUBLED tile box of HashGrid); mode 3: rays [0, split) fore, the rest
// background -- both render chains of a step in one launch, so that the table is streamed through L2 once.
SNRF_API int snrf_field_encode_fwd(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                                   const float* box_min, const float* box_size, int mode, const float* table, const int* res,
                                   float* out_lm, float* jac_lm, const unsigned char* ray_valid, int split_ray, int N, int S, int L, int T,
                                   void* stream)
{
    SNRF_CHECK_ARG(N >= 0 && L > 0 && T > 0 && (T & (T - 1)) == 0, "snrf_field_encode_fwd: T must be a power of two (N=%d L=%d T=%d)", N, L, T);
    SNRF_CHECK_ARG(mode >= 0 && mode <= 3 && (mode == 0 ? points != nullptr : (rays_o && rays_d && z_vals && box_min && box_size && S > 0)),
                   "snrf_field_encode_fwd: inconsistent arguments for mode %d", mode);
    if (N == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const bool pair_levels = g_fwd_pairing && pick_lpb(L, T) == 1 && L >= 2;
    const int lpb = pair_levels ? -1 : pick_lpb(L, T);
    const float2* tb = (const float2*)table;
    float2 *o = (float2*)out_lm, *j = (float2*)jac_lm;
    // the eviction policy needs one level per CTA row and a slice the 32-bit range operands can describe
    const bool policy = g_fwd_l2_mode != 0 && lpb == 1 && (long long)T * 8 < (1ll << 32);
    uint32_t pin = 0;
    if (policy && g_fwd_l2_mode == 2) { const long long b = (long long)g_fwd_pin_mib << 20; pin = (uint32_t)(b < (long long)T * 8 ? b : (long long)T * 8); }
    if (policy && g_fwd_l2_mode == 3) pin = (uint32_t)(g_fwd_pin_mib >= 128 ? 65536 : g_fwd_pin_mib * 512);
    const bool split = g_fwd_split_levels && lpb == 1;
    const int ray_split = mode == 1 ? 0x7fffffff : (mode == 2 ? 0 : split_ray);
    const int pair = (lpb >= 1 && T >= 4) ? g_fwd_pair_mode : 0;
#define SNRF_FWD_K(MODE, JAC, POL, PAIR, GRID, LBASE) field_fwd_kernel<MODE, JAC, POL, PAIR><<<GRID, kThreads, 0, s>>>(rays_o, rays_d, z_vals, points, box_min, box_size, tb, res, o, j, ray_valid, ray_split, N, S, L, (uint32_t)T, lpb, LBASE, g_fwd_l2_mode, pin, g_fwd_pair_level)
#define SNRF_FWD_P(MODE, JAC, POL, GRID, LBASE)                                              \
    do {                                                                                     \
        if (pair == 2) SNRF_FWD_K(MODE, JAC, POL, 2, GRID, LBASE);                            \
        else if (pair == 1) SNRF_FWD_K(MODE, JAC, POL, 1, GRID, LBASE);                       \
        else SNRF_FWD_K(MODE, JAC, POL, 0, GRID, LBASE);                                      \
    } while (0)
#define SNRF_FWD(MODE, GRID, LBASE)                                                          \
    do {                                                                                     \
        if (j) { if (policy) SNRF_FWD_P(MODE, true, true, GRID, LBASE); else SNRF_FWD_P(MODE, true, false, GRID, LBASE); }   \
        else   { if (policy) SNRF_FWD_P(MODE, false, true, GRID, LBASE); else SNRF_FWD_P(MODE, false, false, GRID, LBASE); } \
    } while (0)
    if (split) {
        for (int l = 0; l < L; ++l) {
            const dim3 grid(grid_x(N), 1);
            if (mode == 0) SNRF_FWD(kNone, grid, l); else SNRF_FWD(kRays, grid, l);
        }
    } else {
        const dim3 grid(grid_x(N), pair_levels ? (L + 1) / 2 : snrf_div_up(L, lpb));
        if (mode == 0) SNRF_FWD(kNone, grid, 0); else SNRF_FWD(kRays, grid, 0);
    }
#undef SNRF_FWD
#undef SNRF_FWD_P
#undef SNRF_FWD_K
    SNRF_RETURN_LAUNCH("snrf_field_encode_fwd");
}

// grad_lm [L,N,2]; jac_lm from the forward (NULL: no position gradient).  ACCUMULATES grad_table [L,T,2] and
// grad_rays_o / grad_rays_d [R,3] (mode 1, 2; either may be NULL) or grad_points [N,3] (mode 0).
SNRF_API int snrf_field_encode_bwd(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                                   const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                                   const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points, float* grad_table,
                                   const unsigned char* ray_valid, int split, int N, int S, int L, int T, void* stream)
{
    SNRF_CHECK_ARG(N >= 0 && L > 0 && T > 0 && (T & (T - 1)) == 0, "snrf_field_encode_bwd: T must be a power of two (N=%d L=%d T=%d)", N, L, T);
    SNRF_CHECK_ARG(mode >= 0 && mode <= 3 && (mode == 0 ? points != nullptr : (rays_o && rays_d && z_vals && box_min && box_size && S > 0)),
                   "snrf_field_encode_bwd: inconsistent arguments for mode %d", mode);
    SNRF_CHECK_ARG(grad_table != nullptr && grad_lm != nullptr, "snrf_field_encode_bwd: grad_lm and grad_table are required");
    if (N == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    int pass_bits = pick_pass_bits(T);
    int log2T = 0;
    while ((1 << log2T) < T) ++log2T;
    if (pass_bits > log2T) pass_bits = log2T;
    const int range_shift = log2T - pass_bits;
    const dim3 grid(grid_x(N), L << pass_bits);
    const float2 *g = (const float2*)grad_lm, *j = (const float2*)jac_lm;
    float2* gt = (float2*)grad_table;
    const int agg = g_aggregate_override >= 0 ? g_aggregate_override : L / 2;
#define SNRF_BWD(MODE) field_bwd_kernel<MODE><<<grid, kThreads, 0, s>>>(rays_o, rays_d, z_vals, points, box_min, box_size, res, g, j, grad_rays_o, grad_rays_d, grad_points, gt, ray_valid, ray_split, N, S, L, (uint32_t)T, pass_bits, range_shift, agg)
    const int ray_split = mode == 1 ? 0x7fffffff : (mode == 2 ? 0 : split);
#define SNRF_RUNS(MODE, R) field_bwd_runs_kernel<MODE, R><<<dim3(grid_x((N + R - 1) / R), L << pass_bits), kThreads, 0, s>>>(rays_o, rays_d, z_vals, points, box_min, box_size, res, g, j, grad_rays_o, grad_rays_d, grad_points, gt, ray_valid, ray_split, N, S, L, (uint32_t)T, pass_bits, range_shift)
    if (g_bwd_impl == 1 && g_run_length == 0) {
        // round-2 kernels (the pair the fused path uses, writing straight into the gradient table): geometry + ray gradient
        // once per sample, then one slim scatter launch per level and index range.  3.65 -> 2.9 ms at C2.
        float* cpts = nullptr;
        cudaError_t e = snrf_scratch_alloc((void**)&cpts, (size_t)N * 3 * sizeof(float), s);
        if (e != cudaSuccess) { snrf_set_error("snrf_field_encode_bwd: scratch allocation: %s", cudaGetErrorString(e)); return (int)e; }
        if (mode == 0)
            field_geom_raygrad_kernel<kNone><<<grid_x(N), kThreads, 0, s>>>(rays_o, rays_d, z_vals, points, box_min, box_size, g, j, grad_rays_o, grad_rays_d, grad_points, cpts, ray_valid, ray_split, N, S, L, t_sample_live);
        else
            field_geom_raygrad_kernel<kRays><<<grid_x(N), kThreads, 0, s>>>(rays_o, rays_d, z_vals, points, box_min, box_size, g, j, grad_rays_o, grad_rays_d, grad_points, cpts, ray_valid, ray_split, N, S, L, t_sample_live);
        const long long slice = 1ll << range_shift;
        if (pass_bits == 0) {                              // whole levels: all of them in one launch
            field_scatter_slice_kernel<false><<<dim3(grid_x(N), L), kThreads, 0, s>>>(cpts, res, g, gt, N, 0, (uint32_t)T, 0u, range_shift, agg);
        } else {
            for (int l = 0; l < L; ++l)
                for (int pass = 0; pass < (1 << pass_bits); ++pass)
                    field_scatter_slice_kernel<false><<<dim3(grid_x(N), 1), kThreads, 0, s>>>(cpts, res, g, gt + (size_t)l * T + (size_t)pass * slice, N, l, (uint32_t)T, (uint32_t)pass, range_shift, agg);
        }
        e = cudaGetLastError();
        cudaFreeAsync(cpts, s);
        if (e != cudaSuccess) { snrf_set_error("snrf_field_encode_bwd: %s", cudaGetErrorString(e)); return (int)e; }
        return 0;
    }
    SNRF_CHECK_ARG(t_sample_live == nullptr, "snrf_field_encode_bwd_ert: the sample flags need the geometry + scatter kernel pair (snrf_field_set_bwd_impl(1), run length 0)");
    if (g_run_length == 2) { if (mode == 0) SNRF_RUNS(kNone, 2); else SNRF_RUNS(kRays, 2); }
    else if (g_run_length == 4) { if (mode == 0) SNRF_RUNS(kNone, 4); else SNRF_RUNS(kRays, 4); }
    else if (g_run_length == 8) { if (mode == 0) SNRF_RUNS(kNone, 8); else SNRF_RUNS(kRays, 8); }
    else if (mode == 0) SNRF_BWD(kNone); else SNRF_BWD(kRays);
#undef SNRF_RUNS
#undef SNRF_BWD
    SNRF_RETURN_LAUNCH("snrf_field_encode_bwd");
}

// Private side stream + dependency events of the scatter / update pipeline, one set per device.
struct FusedSide {
    cudaStream_t stream = nullptr;
    cudaEvent_t scat[2] = {nullptr, nullptr}, adam[2] = {nullptr, nullptr}, fork = nullptr, join = nullptr;
};
static FusedSide g_side[64];
static FusedSide* fused_side()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    FusedSide& f = g_side[dev];
    if (f.stream == nullptr) {
        if (cudaStreamCreateWithFlags(&f.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        for (int i = 0; i < 2; ++i) {
            cudaEventCreateWithFlags(&f.scat[i], cudaEventDisableTiming);
            cudaEventCreateWithFlags(&f.adam[i], cudaEventDisableTiming);
        }
        cudaEventCreateWithFlags(&f.fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&f.join, cudaEventDisableTiming);
    }
    return &f;
}

// Backward of snrf_field_encode_fwd fused with the sparse Adam update of the table (see the kernels above).
// table / exp_avg / exp_avg_sq [L,T,2] are UPDATED in place with the step-`step` Adam rule on every element that received a
// non-zero gradient; grad_rays_o / grad_rays_d / grad_points are ACCUMULATED as by snrf_field_encode_bwd.
// grad_scratch: caller-owned device buffer of scratch_entries float2, ALL ZERO on entry and left all zero on exit;
// cpts_scratch: [3][N] floats, overwritten.
//
// How the table is cut into slices.  What has to stay L2-resident while a slice is being reduced into is the set of
// TOUCHED sectors, not the address range:
//   * levels [0, small_levels) have few grid vertices (the caller counts them: (rx+1)(ry+1)(rz+1) <= 2^22), so their
//     touched set is small whatever T is: they are scattered in ONE pass over the whole level, into the first T entries of
//     the scratch (needs scratch_entries >= T + the fine slice; otherwise they are treated like the others);
//   * the other levels touch (nearly) every entry: their slice is an index range of at most g_slice_cap entries
//     (2^23 = 64 MiB of gradient), 2 ranges per level at T = 2^24, several whole levels per slice at small T.
// The coarse levels are issue-bound (cross-lane segmented sums), the fine ones bound by the L2 reduction rate
// (profiles/r2d_*): with g_coarse_concurrent the coarse chain runs on a private side stream next to the fine chain.
// g_overlap (off by default, see there) additionally overlaps scatter k+1 with Adam k inside the fine chain.
SNRF_API int snrf_field_encode_bwd_adam(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                                        const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                                        const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points,
                                        float* table, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                        int step, float* grad_scratch, long long scratch_entries, int small_levels, float* cpts_scratch,
                                        const unsigned char* ray_valid, int split, int N, int S, int L, int T, void* stream)
{
    SNRF_CHECK_ARG(N >= 0 && L > 0 && T > 1 && (T & (T - 1)) == 0, "snrf_field_encode_bwd_adam: T must be a power of two (N=%d L=%d T=%d)", N, L, T);
    SNRF_CHECK_ARG(mode >= 0 && mode <= 3 && (mode == 0 ? points != nullptr : (rays_o && rays_d && z_vals && box_min && box_size && S > 0)),
                   "snrf_field_encode_bwd_adam: inconsistent arguments for mode %d", mode);
    SNRF_CHECK_ARG(grad_lm && table && exp_avg && exp_avg_sq && grad_scratch && cpts_scratch, "snrf_field_encode_bwd_adam: NULL argument");
    SNRF_CHECK_ARG(scratch_entries >= 4, "snrf_field_encode_bwd_adam: scratch_entries must be at least 4");
    SNRF_CHECK_ARG(step >= 1, "snrf_field_encode_bwd_adam: step counts from 1 (got %d)", step);
    if (N == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const float2 *g = (const float2*)grad_lm, *j = (const float2*)jac_lm;
    const int ray_split = mode == 1 ? 0x7fffffff : (mode == 2 ? 0 : split);
    int log2T = 0;
    while ((1 << log2T) < T) ++log2T;

    // ---- slicing plan
    long long fine_cap = 1;                                  // largest power of two <= min(scratch, g_slice_cap)
    while (fine_cap * 2 <= scratch_entries && fine_cap * 2 <= g_slice_cap) fine_cap *= 2;
    if (small_levels < 0) small_levels = 0;
    if (small_levels > L) small_levels = L;
    // single-pass coarse levels only make a difference when a level does not fit a fine slice, and need their own T entries
    const bool coarse_single = small_levels > 0 && (long long)T > fine_cap && scratch_entries >= (long long)T + fine_cap;
    if (!coarse_single) small_levels = 0;
    float* coarse_buf = grad_scratch;
    float* fine_buf = coarse_single ? grad_scratch + (size_t)T * 2 : grad_scratch;
    FusedSide* side = (g_overlap || (coarse_single && g_coarse_concurrent)) ? fused_side() : nullptr;
    const bool overlap = g_overlap && side != nullptr;
    const bool coarse_on_side = coarse_single && g_coarse_concurrent && side != nullptr && !overlap;
    const long long capacity = overlap ? fine_cap / 2 : fine_cap;                  // entries per in-flight fine slice
    int pass_bits = 0;
    while (((long long)T >> pass_bits) > capacity) ++pass_bits;
    if (g_pass_bits_override > pass_bits && g_pass_bits_override <= log2T - 1) pass_bits = g_pass_bits_override;
    const int range_shift = log2T - pass_bits;
    const long long slice = 1ll << range_shift;
    int lpg = pass_bits > 0 ? 1 : (int)(capacity / slice);            // whole levels per scatter / update pair
    if (lpg > L) lpg = L;
    if (g_levels_per_group > 0 && g_levels_per_group < lpg) lpg = g_levels_per_group;
    const int agg = g_aggregate_override >= 0 ? g_aggregate_override : L / 2;
    const adamcore::Hyper h{lr, beta1, beta2, eps, step};
    const int sms = snrf_sm_count();

    // profiling mode: one event after every launch on the caller's stream (class of launch k in cls[]); when kernel classes
    // run concurrently (overlap / coarse chain on the side stream) only the whole phase can be timed: class 3
    constexpr int kMaxEv = 600;
    static cudaEvent_t ev[kMaxEv];
    static int n_ev_created = 0;
    int cls[kMaxEv], n_ev = 0;
    const bool prof = g_profile != 0;
    const bool concurrent = overlap || coarse_on_side;
    auto mark = [&](int c, bool force = false) {
        if (!prof || n_ev >= kMaxEv) return;
        if (concurrent && c > 0 && !force) return;
        if (n_ev >= n_ev_created) { cudaEventCreate(&ev[n_ev]); n_ev_created = n_ev + 1; }
        cudaEventRecord(ev[n_ev], s);
        cls[n_ev++] = c;
    };
    auto adam_launch = [&](cudaStream_t st, float* buf, int l0, int nl, long long base_entry, long long entries) {
        const size_t base = ((size_t)l0 * T + (size_t)base_entry) * 2;                  // floats
        const long long n4 = (long long)nl * entries / 2;                                // float4 groups (two entries each)
        long long gx = (n4 + kThreads * 2 - 1) / (kThreads * 2);
        if (gx > (long long)sms * 16) gx = (long long)sms * 16;
        if (g_l2_hints) launch_dep(adam_slice_kernel<true>, dim3((unsigned)gx), st, (float4*)(table + base), (float4*)(exp_avg + base), (float4*)(exp_avg_sq + base), (float4*)buf, n4, h);
        else launch_dep(adam_slice_kernel<false>, dim3((unsigned)gx), st, (float4*)(table + base), (float4*)(exp_avg + base), (float4*)(exp_avg_sq + base), (float4*)buf, n4, h);
    };

    persist_window_begin(fine_buf, (size_t)fine_cap * 2 * sizeof(float));
    mark(-1);
    if (mode == 0)
        field_geom_raygrad_kernel<kNone><<<grid_x(N), kThreads, 0, s>>>(rays_o, rays_d, z_vals, points, box_min, box_size, g, j, grad_rays_o, grad_rays_d, grad_points, cpts_scratch, ray_valid, ray_split, N, S, L, t_sample_live);
    else
        field_geom_raygrad_kernel<kRays><<<grid_x(N), kThreads, 0, s>>>(rays_o, rays_d, z_vals, points, box_min, box_size, g, j, grad_rays_o, grad_rays_d, grad_points, cpts_scratch, ray_valid, ray_split, N, S, L, t_sample_live);
    mark(0);
    int launches = 1;

    // ---- coarse chain: one pass per level over the whole level slice
    if (coarse_single) {
        cudaStream_t sc = s;
        if (coarse_on_side) {
            cudaEventRecord(side->fork, s);
            cudaStreamWaitEvent(side->stream, side->fork, 0);
            sc = side->stream;
        }
        for (int l = 0; l < small_levels; ++l) {
            if (g_l2_hints) launch_dep(field_scatter_slice_kernel<true>, dim3(grid_x(N), 1), sc, (const float*)cpts_scratch, res, g, (float2*)coarse_buf, N, l, (uint32_t)T, 0u, log2T, agg);
            else launch_dep(field_scatter_slice_kernel<false>, dim3(grid_x(N), 1), sc, (const float*)cpts_scratch, res, g, (float2*)coarse_buf, N, l, (uint32_t)T, 0u, log2T, agg);
            if (!coarse_on_side) mark(1);
            adam_launch(sc, coarse_buf, l, 1, 0, T);
            if (!coarse_on_side) mark(2);
            launches += 2;
        }
        if (coarse_on_side) cudaEventRecord(side->join, sc);
    }

    // ---- fine chain
    int k = 0;                                            // slice counter
    for (int l0 = small_levels; l0 < L; l0 += lpg) {
        const int nl = l0 + lpg <= L ? lpg : L - l0;
        for (int pass = 0; pass < (1 << pass_bits); ++pass, ++k) {
            const int b = overlap ? (k & 1) : 0;
            float* buf = fine_buf + (size_t)b * capacity * 2;
            if (overlap && k >= 2) cudaStreamWaitEvent(s, side->adam[b], 0);         // the half is free again
            if (g_l2_hints) launch_dep(field_scatter_slice_kernel<true>, dim3(grid_x(N), nl), s, (const float*)cpts_scratch, res, g, (float2*)buf, N, l0, (uint32_t)T, (uint32_t)pass, range_shift, agg);
            else launch_dep(field_scatter_slice_kernel<false>, dim3(grid_x(N), nl), s, (const float*)cpts_scratch, res, g, (float2*)buf, N, l0, (uint32_t)T, (uint32_t)pass, range_shift, agg);
            mark(1);
            cudaStream_t sa = s;
            if (overlap) {
                cudaEventRecord(side->scat[b], s);
                cudaStreamWaitEvent(side->stream, side->scat[b], 0);
                sa = side->stream;
            }
            adam_launch(sa, buf, l0, nl, (long long)pass * slice, slice);
            if (overlap) cudaEventRecord(side->adam[b], sa);
            mark(2);
            launches += 2;
        }
    }
    if (overlap) {
        if (k >= 1) cudaStreamWaitEvent(s, side->adam[0], 0);
        if (k >= 2) cudaStreamWaitEvent(s, side->adam[1], 0);
    }
    if (coarse_on_side) cudaStreamWaitEvent(s, side->join, 0);
    persist_window_end();
    g_last_launches = launches;
    if (prof) {
        if (concurrent) mark(3, true);                     // closing event on the caller's stream (after the joins)
        cudaStreamSynchronize(s);
        for (int i = 0; i < 4; ++i) g_profile_ms[i] = 0.f;
        for (int i = 1; i < n_ev; ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
            g_profile_ms[cls[i]] += ms;
        }
        if (!concurrent) g_profile_ms[3] = g_profile_ms[1] + g_profile_ms[2];
    }
    SNRF_RETURN_LAUNCH("snrf_field_encode_bwd_adam");
}

// The two backward entry points with the per-sample early-ray-termination flags of snrf_composite_fwd_ert (sample_live [N], may
// be NULL): a dead sample contributes no table gradient and no ray gradient (its gradient row is never read).
SNRF_API int snrf_field_encode_bwd_ert(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                                       const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                                       const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points, float* grad_table,
                                       const unsigned char* ray_valid, int split, int N, int S, int L, int T,
                                       const unsigned char* sample_live, void* stream)
{
    t_sample_live = sample_live;
    const int rc = snrf_field_encode_bwd(rays_o, rays_d, z_vals, points, box_min, box_size, mode, res, grad_lm, jac_lm, grad_rays_o, grad_rays_d,
                                         grad_points, grad_table, ray_valid, split, N, S, L, T, stream);
    t_sample_live = nullptr;
    return rc;
}
SNRF_API int snrf_field_encode_bwd_adam_ert(const float* rays_o, const float* rays_d, const float* z_vals, const float* points,
                                            const float* box_min, const float* box_size, int mode, const int* res, const float* grad_lm,
                                            const float* jac_lm, float* grad_rays_o, float* grad_rays_d, float* grad_points,
                                            float* table, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                            int step, float* grad_scratch, long long scratch_entries, int small_levels, float* cpts_scratch,
                                            const unsigned char* ray_valid, int split, int N, int S, int L, int T,
                                            const unsigned char* sample_live, void* stream)
{
    t_sample_live = sample_live;
    const int rc = snrf_field_encode_bwd_adam(rays_o, rays_d, z_vals, points, box_min, box_size, mode, res, grad_lm, jac_lm, grad_rays_o,
                                              grad_rays_d, grad_points, table, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, step, grad_scratch,
                                              scratch_entries, small_levels, cpts_scratch, ray_valid, split, N, S, L, T, stream);
    t_sample_live = nullptr;
    return rc;
}

// ---------------------------------------------------------------------------------------------------------------------------
// Surface normals of the density field, forward only: the out_normal branch of HashGrid.render_batch_rays
// (hashgrid/__init__.py:547-556), which the reference obtains from torch.autograd.grad of sigma w.r.t. the samples.
// sigma = softplus(W_s H[:32] + b_s), H = W2 a1 + b2, a1 = exp(-50 z1^2), z1 = W1 (f m) + b1.  Layer 2 is linear, so its
// sigma rows fold into u = W2[:32,:]^T w_s and c = w_s . b2[:32] + b_s once per CTA: sigma_pre = u . a1 + c and
//   d sigma / d f = softplus'(sigma_pre) m (W1^T (-100 z1 a1 u)).
// One pass over the 64 rows of W1 forms z1_j, sigma_pre and the W1^T accumulation together (softplus' is a common factor
// applied at the end), so a thread holds 32 masked features and 32 gradient accumulators, nothing of width 64.  The gradient
// w.r.t. the contracted point comes from the encode's Jacobians jac_lm, the one w.r.t. the sample from contract_bwd.
// fp32 on the CUDA cores: ~4 k FMAs and 512 bytes of reads per sample, W1 broadcast from shared memory.
// ---------------------------------------------------------------------------------------------------------------------------
namespace {

constexpr int kNormalThreads = 256;
constexpr int kNormalCtasPerSm = 2;            // grid-stride: at most this many CTAs per SM (the register budget allows 2)

__global__ void __launch_bounds__(kNormalThreads, kNormalCtasPerSm)
field_normal_kernel(const float2* __restrict__ feats, const float2* __restrict__ jac, const float* __restrict__ mask32,
                    const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
                    const float* __restrict__ ws, const float* __restrict__ bs, const float* __restrict__ rays_o,
                    const float* __restrict__ rays_d, const float* __restrict__ z_vals, const float* __restrict__ bmin_p,
                    const float* __restrict__ bsize_p, const unsigned char* __restrict__ ray_valid, int back,
                    float* __restrict__ normal, float* __restrict__ grad_x, int N, int S)
{
    __shared__ __align__(16) float s_w1[64 * 32];
    __shared__ float s_b1[64], s_u[64], s_m[32];
    __shared__ float s_c;
    for (int i = threadIdx.x; i < 64 * 32; i += blockDim.x) s_w1[i] = W1[i];
    if (threadIdx.x < 64) {
        const int j = threadIdx.x;
        float u = 0.0f;
        for (int i = 0; i < 32; ++i) u = fmaf(W2[i * 64 + j], ws[i], u);
        s_u[j] = u;
        s_b1[j] = b1[j];
    }
    if (threadIdx.x < 32) s_m[threadIdx.x] = mask32 != nullptr ? mask32[threadIdx.x] : 1.0f;
    if (threadIdx.x == 0) {
        float c = bs[0];
        for (int i = 0; i < 32; ++i) c = fmaf(ws[i], b2[i], c);
        s_c = c;
    }
    __syncthreads();
    const f3 bmin = ld3(bmin_p), bsize = ld3(bsize_p);
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
        const int r = n / S;
        if (ray_valid != nullptr && !ray_valid[r]) continue;          // masked-out ray: its rows are left untouched
        float fm[32], g[32];
#pragma unroll
        for (int l = 0; l < 16; ++l) {
            const float2 f = ldg2(feats + (size_t)l * N + n);
            fm[2 * l] = f.x * s_m[2 * l];
            fm[2 * l + 1] = f.y * s_m[2 * l + 1];
            g[2 * l] = 0.0f;
            g[2 * l + 1] = 0.0f;
        }
        float sp = s_c;
        // rows in groups of 8: the eight t_j first, then the W1^T accumulation re-reads the rows from shared memory, so
        // that no row is held in registers between the two uses.  ptxas (-O3, sm_100a): 128 registers (the cap of
        // kNormalCtasPerSm), 8 bytes of stack: one 8-byte value stored and reloaded once per sample after this loop,
        // where the 48 Jacobian loads are issued together; the loop itself has no local-memory traffic
#pragma unroll 1
        for (int j0 = 0; j0 < 64; j0 += 8) {
            float t[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const float4* w = reinterpret_cast<const float4*>(s_w1 + (j0 + jj) * 32);
                float z = s_b1[j0 + jj];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 v = w[q];
                    z = fmaf(v.x, fm[4 * q], z); z = fmaf(v.y, fm[4 * q + 1], z);
                    z = fmaf(v.z, fm[4 * q + 2], z); z = fmaf(v.w, fm[4 * q + 3], z);
                }
                const float a = expf(-50.0f * z * z);
                const float u = s_u[j0 + jj];
                sp = fmaf(u, a, sp);
                t[jj] = -100.0f * z * a * u;
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const float4 v = reinterpret_cast<const float4*>(s_w1 + (j0 + jj) * 32)[q];
                    g[4 * q] = fmaf(v.x, t[jj], g[4 * q]); g[4 * q + 1] = fmaf(v.y, t[jj], g[4 * q + 1]);
                    g[4 * q + 2] = fmaf(v.z, t[jj], g[4 * q + 2]); g[4 * q + 3] = fmaf(v.w, t[jj], g[4 * q + 3]);
                }
            }
        }
        // torch's softplus backward (beta 1, threshold 20): 1 above the threshold, e^x / (e^x + 1) below it
        const float e = sp > 20.0f ? 0.0f : expf(sp);
        const float dsp = sp > 20.0f ? 1.0f : e / (e + 1.0f);
        f3 gc = mk3(0.0f, 0.0f, 0.0f);
#pragma unroll
        for (int l = 0; l < 16; ++l) {
            const float g0 = dsp * s_m[2 * l] * g[2 * l], g1 = dsp * s_m[2 * l + 1] * g[2 * l + 1];
            const float2* jl = jac + (size_t)l * 3 * N + n;
            const float2 jx = __ldcs(jl), jy = __ldcs(jl + (size_t)N), jz = __ldcs(jl + 2 * (size_t)N);    // read once
            gc.x = fmaf(g0, jx.x, fmaf(g1, jx.y, gc.x));
            gc.y = fmaf(g0, jy.x, fmaf(g1, jy.y, gc.y));
            gc.z = fmaf(g0, jz.x, fmaf(g1, jz.y, gc.z));
        }
        const Pt p = contract(back != 0, sample_pos(ld3(rays_o + 3 * (size_t)r), ld3(rays_d + 3 * (size_t)r), z_vals[n]), bmin, bsize);
        const f3 gx = contract_bwd(back != 0, p, gc);
        const float den = sqrtf(dot3(gx, gx)) + 1e-8f;
        st3(normal + 3 * (size_t)n, mk3(-gx.x / den, -gx.y / den, -gx.z / den));
        if (grad_x != nullptr) st3(grad_x + 3 * (size_t)n, gx);
    }
}

}  // namespace

// feats_lm [16][N] float2 and jac_lm [16][3][N] float2 from snrf_field_encode_fwd (mode 1 / 2, same rays and box);
// params as snrf_decoder_fwd (host array of 16 device pointers, only the first six are read).  -> normal [N,3] =
// -g / (|g| + 1e-8), grad_x [N,3] (optional) = g = d sigma / d sample.  Rows of masked-out rays are left untouched.
SNRF_API int snrf_field_normal(const float* feats_lm, const float* jac_lm, const float* mask32, const float* const* params, int mode,
                               const float* box_min, const float* box_size, const float* rays_o, const float* rays_d,
                               const float* z_vals, const unsigned char* ray_valid, float* normal, float* grad_x, int N, int S,
                               void* stream)
{
    SNRF_CHECK_ARG(N >= 0 && S > 0 && (mode == 1 || mode == 2), "snrf_field_normal: need N >= 0, S > 0, mode 1 or 2 (N=%d S=%d mode=%d)", N, S, mode);
    SNRF_CHECK_ARG(feats_lm && jac_lm && params && box_min && box_size && rays_o && rays_d && z_vals && normal,
                   "snrf_field_normal: a required pointer is NULL");
    if (N == 0) return 0;
    for (int i = 0; i < 6; ++i) SNRF_CHECK_ARG(params[i] != nullptr, "snrf_field_normal: decoder parameter %d is NULL", i);
    const int want = snrf_div_up(N, kNormalThreads), cap = snrf_sm_count() * kNormalCtasPerSm;
    field_normal_kernel<<<want < cap ? want : cap, kNormalThreads, 0, (cudaStream_t)stream>>>(
        (const float2*)feats_lm, (const float2*)jac_lm, mask32, params[0], params[1], params[2], params[3], params[4], params[5],
        rays_o, rays_d, z_vals, box_min, box_size, ray_valid, mode == 2 ? 1 : 0, normal, grad_x, N, S);
    SNRF_RETURN_LAUNCH("snrf_field_normal");
}
