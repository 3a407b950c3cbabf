// Render-side field evaluation: fp16 hash-table encode + decoder MLP on the tensor cores + per-sample alpha and
// tile-overlap blending, sm_100a.
//
// Replaces (behaviour, not code) the reference's per-thread-MLP kernels
//   pts_inference        hashgrid/src/rendering_kernel.cu:467-621  (foreground, <= 4 overlapping tiles per sample)
//   bg_pts_inference     :871-1008, 1172-1208                      (background, blend weights per ray)
//   bg_pts_inference_v2  :1011-1171                                (background, one tile slot per call)
// with get_multilevel_features<16> (:79-114) and Decoder::inference (hashgrid/include/decoder.h:169-218).
//
// The reference evaluates the 13 994-parameter MLP per thread out of global memory.  Here the encode is a pass of
// its own that writes level-major features, and the decoder runs on 128-sample tiles as tcgen05 MMAs with the
// accumulators in TMEM and a scene tile's weights staged once per CTA as bf16x3 operand tiles (decoder_core.cuh).
// launch() picks one of two implementations from the input:
//   one scene tile (foreground, or one background slot)  -> launch_two_pass: every sample belongs to that tile;
//   several scene tiles, or blended background          -> launch_work: the (sample, slot) pairs are grouped by tile.
#include "decoder_core.cuh"
#include <cuda_fp16.h>
using namespace dec;

namespace {

constexpr int kMaxPts = 4;
enum Mode { kFore = 0, kBackBlend = 1, kBackSlot = 2 };

__device__ __forceinline__ uint32_t hash3(int x, int y, int z, uint32_t mask)
{
    return (((uint32_t)x) ^ ((uint32_t)y * 2654435761u) ^ ((uint32_t)z * 805459861u)) & mask;
}

struct InferArgs {
    const float *rays_o, *rays_d, *z_vals, *dists;
    const short* slots;          // kFore: block_idxs [B*S,4]; kBack*: per-ray ids [B,4]
    const float* blend;          // kBackBlend: blend weights [B,4]
    const __half2* tables;       // [nb,16,T]
    const float* params;         // [nb,13994]
    const int* resolution;       // [nb,16,3]
    const unsigned char* grid_occ;
    const long long* grid_starts;
    const int* grid_log2dim;
    const float *corners, *sizes;
    float *out_diffuse, *out_specular, *out_alpha;
    int B, S, step;
    uint32_t T;
};

// ------------------------------------------------------------------------------------------------------------------
// Single-tile path: three passes over chunks of samples.
//   pass 0 (infer_geometry_kernel): per-sample table coordinate / weight / alpha scale / state, once.
//   pass 1 (infer_encode_kernel): fp16 gathers, ONE LEVEL PER CTA ROW -> level-major features [16][Nc].
//           The whole GPU walks one 64 MiB level slice at a time, which stays L2-resident: the table streams from HBM
//           once per chunk, whereas gathering every level of a sample at once pulls a 32-byte sector per corner from
//           HBM -- ~4 KB per sample, the floor of a 1080p frame is then ~170 ms per pass.
//   pass 2: decoder layers on the tensor cores (no gathers here, so the L1 is not needed), inference activations,
//           alpha, the reference's weight normalisation.  infer_decode4_kernel (four tiles in flight per CTA) when
//           S >= kMinS4, infer_decode_kernel (two tiles in flight) otherwise.
// Per-sample state byte: 0 = write zeros (foreground sample outside occupied space), 1 = evaluate, 2 = leave the
// caller's rows untouched (background ray without a tile in this slot).
struct Geom {
    f3 u;
    float w;
    bool member, active;
};

template <int MODE>
__device__ __forceinline__ Geom sample_geom(const InferArgs& a, int b, int ray, int slot, f3 p)
{
    Geom g;
    g.u = mk3(0, 0, 0); g.w = 0.0f; g.member = slot >= 0; g.active = false;
    if (!g.member) return g;
    const f3 bc = ld3(a.corners + 3 * b), bs = ld3(a.sizes + 3 * b);
    if (MODE == kFore) {
        const f3 q = mk3((p.x - bc.x) / bs.x, (p.y - bc.y) / bs.y, (p.z - bc.z) / bs.z);          // [0,1]
        const f3 dis = mk3((0.5f - fabsf(q.x - 0.5f)) * bs.x, (0.5f - fabsf(q.y - 0.5f)) * bs.y, (0.5f - fabsf(q.z - 0.5f)) * bs.z);
        if (dis.x != 0 && dis.z != 0) g.w = dis.x * dis.z;
        else if (dis.x != 0) g.w = dis.x;
        else if (dis.z != 0) g.w = dis.z;
        const int lx = a.grid_log2dim[3 * b], ly = a.grid_log2dim[3 * b + 1], lz = a.grid_log2dim[3 * b + 2];
        const int gx = min(max((int)(q.x * (float)(1 << lx)), 0), (1 << lx) - 1);
        const int gy = min(max((int)(q.y * (float)(1 << ly)), 0), (1 << ly) - 1);
        const int gz = min(max((int)(q.z * (float)(1 << lz)), 0), (1 << lz) - 1);
        g.active = a.grid_occ[a.grid_starts[b] + ((gx << (ly + lz)) | (gy << lz) | gz)] != 0;
        g.u = mk3(q.x * 0.5f + 0.25f, q.y * 0.5f + 0.25f, q.z * 0.5f + 0.25f);                     // [0.25, 0.75]
    } else {
        // contraction of the 2x-normalised position (rendering_kernel.cu:1060-1095)
        float q[3] = {2.0f * (p.x - bc.x) / bs.x - 1.0f, 2.0f * (p.y - bc.y) / bs.y - 1.0f, 2.0f * (p.z - bc.z) / bs.z - 1.0f};
        float nrm = fabsf(q[0]);
        if (fabsf(q[1]) > nrm) nrm = fabsf(q[1]);
        if (fabsf(q[2]) > nrm) nrm = fabsf(q[2]);
        const float ratio = (2.0f - 1.0f / nrm) / nrm;
        g.u = mk3((q[0] * ratio + 2.0f) * 0.25f, (q[1] * ratio + 2.0f) * 0.25f, (q[2] * ratio + 2.0f) * 0.25f);
        g.w = MODE == kBackBlend ? a.blend[(size_t)ray * kMaxPts + slot] : 1.0f;
        g.active = true;
    }
    return g;
}

// pass 0 of the single-tile path: the geometry of every sample ONCE (table coordinate, blend weight, alpha scale, state);
// the encode pass below then costs a coalesced 16-byte load per (sample, level) instead of recomputing the ray / box
// arithmetic and the occupancy lookup 16 times (ncu: that kernel ran at 61 % of the issue slots, 314 instructions per
// sample-level)
template <int MODE>
__global__ void __launch_bounds__(256)
infer_geometry_kernel(InferArgs a, long long n0, int Nc, float4* __restrict__ uw, float2* __restrict__ aux, unsigned char* __restrict__ state)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Nc; i += gridDim.x * blockDim.x) {
        const long long n = n0 + i;
        const int ray = (int)(n / a.S), k = (int)(n % a.S);
        const f3 o = ld3(a.rays_o + 3 * (size_t)ray), d = ld3(a.rays_d + 3 * (size_t)ray);
        const float zv = a.z_vals[n];
        int id;
        float step_len;
        if (MODE == kFore) { id = a.slots[(size_t)n * kMaxPts]; step_len = a.dists[n]; }
        else {
            id = a.slots[(size_t)ray * kMaxPts + (MODE == kBackSlot ? a.step : 0)];
            step_len = (k == a.S - 1) ? 10000000.0f : a.z_vals[n + 1] - zv;
        }
        const Geom g = sample_geom<MODE>(a, 0, ray, id == 0 ? 0 : -1, o + zv * d);
        state[i] = g.active ? 1 : ((MODE == kBackSlot && !g.member) ? 2 : 0);
        aux[i] = make_float2(g.w, MODE == kFore ? step_len * sqrtf(dot3(d, d)) : step_len);
        uw[i] = make_float4(g.u.x, g.u.y, g.u.z, g.w);
    }
}

__global__ void __launch_bounds__(256)
infer_encode_kernel(InferArgs a, int Nc, const float4* __restrict__ uw, const unsigned char* __restrict__ state, float2* __restrict__ feats_lm)
{
    const int l = blockIdx.y;
    const uint32_t mask = a.T - 1u;
    const int rx = a.resolution[3 * l] - 1, ry = a.resolution[3 * l + 1] - 1, rz = a.resolution[3 * l + 2] - 1;
    const __half2* tl = a.tables + (size_t)l * a.T;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Nc; i += gridDim.x * blockDim.x) {
        if (state[i] != 1) continue;
        const float4 u = __ldg(uw + i);
        const float vx = u.x * (float)rx, vy = u.y * (float)ry, vz = u.z * (float)rz;
        const int ix = (int)vx, iy = (int)vy, iz = (int)vz;
        const float ox = vx - (float)ix, oy = vy - (float)iy, oz = vz - (float)iz;
        float2 f[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) f[c] = __half22float2(__ldg(tl + hash3(ix + ((c >> 2) & 1), iy + ((c >> 1) & 1), iz + (c & 1), mask)));
        const float ax = 1 - ox, ay = 1 - oy, az = 1 - oz;
        const float w[8] = {ax * ay * az, ax * ay * oz, ax * oy * az, ax * oy * oz, ox * ay * az, ox * ay * oz, ox * oy * az, ox * oy * oz};
        float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
        for (int c = 0; c < 8; ++c) { s0 += w[c] * f[c].x; s1 += w[c] * f[c].y; }
        feats_lm[(size_t)l * Nc + i] = make_float2(s0, s1);
    }
}

// Decoder layers + inference activations for one 128-row tile of precomputed level-major features (row r of this
// thread at f0[level * stride]).  Returns false when no row of the tile is active (nothing evaluated); sigma / dif /
// spe are valid for the active rows of column group 0.
__device__ __forceinline__ bool eval_tile(Ctx<true, 2>& c, const Tiles& Tl, bool active, const float2* __restrict__ f0, size_t stride,
                                          f3 d, float& sigma, f3& dif, f3& spe)
{
    if (!c.any(active)) return false;
    const int cg = c.cg;
    float x[16], sh[16];
    if (active) {
#pragma unroll
        for (int l = 0; l < 8; ++l) {
            const float2 v = __ldg(f0 + (size_t)(8 * cg + l) * stride);
            x[2 * l] = v.x; x[2 * l + 1] = v.y;
        }
        const f3 dn = d * rsqrtf(dot3(d, d));                 // normalize(): decoder.h:201, no epsilon
        sh16(dn.x, dn.y, dn.z, sh);
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) { x[j] = 0.0f; sh[j] = 0.0f; }
    }
    store_input_row<true, 2>(Tl, c.row, cg, x, sh + 8 * cg);
    float head[10], zh[7];
    forward_layers<true, 2>(c, Tl, head, zh);
    if (cg == 0) {
        float zs[16];
        umma::tmem_ld16(c.tmem + cDh + c.lane_addr, zs);
        umma::tc_wait_ld();
        // Decoder::inference activations (decoder.h:134-146): softplus without threshold, expf sigmoids
        sigma = logf(1.0f + expf(zh[0]));
        dif = mk3(1.0f / (1.0f + expf(-zh[1])), 1.0f / (1.0f + expf(-zh[2])), 1.0f / (1.0f + expf(-zh[3])));
        const f3 tint = mk3(1.0f / (1.0f + expf(-zh[4])), 1.0f / (1.0f + expf(-zh[5])), 1.0f / (1.0f + expf(-zh[6])));
        spe = mk3(tint.x / (1.0f + expf(-(zs[0] + c.bias[oB5 + 0]))), tint.y / (1.0f + expf(-(zs[1] + c.bias[oB5 + 1]))),
                  tint.z / (1.0f + expf(-(zs[2] + c.bias[oB5 + 2]))));
    }
    return true;
}

// common prologue of the two decode kernels: TMEM, barriers, operand tile pointers of this thread's group
#define SNRF_DECODE_PROLOGUE(STAGE_PARAMS)                                                                        \
    extern __shared__ __align__(1024) unsigned char smem_raw[];                                                  \
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);                      \
    __shared__ uint64_t bars[2];                                                                                 \
    __shared__ uint32_t tmem_slot;                                                                               \
    const int tid = threadIdx.x, warp = tid >> 5;                                                                \
    if (STAGE_PARAMS) stage_all_weights<true>(smem, flat_params(STAGE_PARAMS), nullptr, tid, kThreadsDec);        \
    if (warp == 0) umma::tmem_alloc<512>(&tmem_slot);                                                            \
    if (tid == 0) { umma::mbar_init(&bars[0], 1); umma::mbar_init(&bars[1], 1); umma::mbar_fence_init(); }       \
    umma::fence_async_smem();                                                                                    \
    umma::tc_fence_before();                                                                                     \
    __syncthreads();                                                                                             \
    umma::tc_fence_after();                                                                                      \
    Ctx<true, 2> c;                                                                                              \
    c.init(smem, bars, tmem_slot);                                                                               \
    const int row = c.row, cg = c.cg;                                                                            \
    unsigned char* T0 = smem + off_tiles<true>() + c.group * fwd_tiles<true>() * kTile;                          \
    unsigned char* T1 = T0 + kTile;                                                                              \
    unsigned char* T2 = T1 + kTile;                                                                              \
    unsigned char* LOa = T2 + kTile;                                                                             \
    unsigned char* LOb = LOa + kTile;                                                                            \
    const Tiles Tl{T0, T1, T2, T1, T2, LOa, LOb};                                                                \
    (void)row; (void)cg;

template <int MODE>
__global__ void __launch_bounds__(kThreadsDec, 1)
infer_decode_kernel(InferArgs a, long long n0, int Nc, const float2* __restrict__ feats_lm, const float2* __restrict__ aux,
                    const unsigned char* __restrict__ state, int num_tiles)
{
    SNRF_DECODE_PROLOGUE(a.params)
    for (int tile = 2 * blockIdx.x + c.group; tile < num_tiles; tile += 2 * gridDim.x) {
        const int i = tile * kRows + row;
        const int st = i < Nc ? state[i] : 2;
        const bool active = st == 1;
        const long long n = n0 + i;
        float sigma = 0.0f;
        f3 dif = mk3(0, 0, 0), spe = mk3(0, 0, 0);
        const f3 d = active ? ld3(a.rays_d + 3 * (size_t)(n / a.S)) : mk3(0, 0, 1);
        const bool done = eval_tile(c, Tl, active, feats_lm + i, (size_t)Nc, d, sigma, dif, spe);
        if (cg != 0) continue;
        if (done && active) {
            const float2 ws = aux[i];
            const float al = 1.0f - expf(-1.0f * sigma * ws.y);
            float wa = ws.x * al;
            dif = dif * wa; spe = spe * wa;
            if (MODE != kBackSlot && ws.x > 0) {               // the reference divides by the weight sum when it is positive
                const float inv = 1.0f / ws.x;
                dif = dif * inv; spe = spe * inv; wa *= inv;
            }
            st3(a.out_diffuse + 3 * (size_t)n, dif);
            st3(a.out_specular + 3 * (size_t)n, spe);
            a.out_alpha[n] = wa;
        } else if (st == 0) {                                  // unoccupied / unassigned foreground sample: zeros
            st3(a.out_diffuse + 3 * (size_t)n, mk3(0, 0, 0));
            st3(a.out_specular + 3 * (size_t)n, mk3(0, 0, 0));
            a.out_alpha[n] = 0.0f;
        }
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 0) umma::tmem_free<512>(tmem_slot);
}


// The same decode pass with FOUR tiles in flight per CTA (decoder_core.cuh: forward_layers4 -- operand tiles in place, the
// SH term of the first directional layer added per ray in fp32, the activation-free layer 2 folded into its consumers):
// one thread per sample row.  Needs a.S >= kMinS4.
template <int MODE>
__global__ void __launch_bounds__(kThreadsDec, 1)
infer_decode4_kernel(InferArgs a, long long n0, int Nc, const float2* __restrict__ feats_lm, const float2* __restrict__ aux,
                     const unsigned char* __restrict__ state, int num_tiles)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t bars[kGroups4];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    const DecoderParams prm = flat_params(a.params);
    stage_all_weights<true>(smem, prm, nullptr, tid, kThreadsDec);
    float* w3sh = reinterpret_cast<float*>(smem + off_w3sh<true>());
    stage_w3sh(w3sh, prm, tid, kThreadsDec);
    stage_fold_weights4<true>(smem, prm, reinterpret_cast<float*>(smem + off_tiles4<true>()), tid, kThreadsDec);
    if (warp == 0) umma::tmem_alloc<512>(&tmem_slot);
    if (tid == 0) {
        for (int g = 0; g < kGroups4; ++g) umma::mbar_init(&bars[g], 1);
        umma::mbar_fence_init();
    }
    umma::fence_async_smem();
    umma::tc_fence_before();
    __syncthreads();
    umma::tc_fence_after();
    Ctx4 c;
    c.init(bars, tmem_slot);
    unsigned char* P = smem + off_tiles4<true>() + c.group * 2 * kTile;
    unsigned char* Q = P + kTile;
    float* rb = reinterpret_cast<float*>(smem + off_raybias4<true>()) + c.group * kMaxRays4 * 64;
    const float* bias = reinterpret_cast<const float*>(smem + off_bias<true>());
    const int row = c.row;

    for (int tile = kGroups4 * blockIdx.x + c.group; tile < num_tiles; tile += kGroups4 * gridDim.x) {
        const int i0 = tile * kRows, i = i0 + row;
        const int st = i < Nc ? state[i] : 2;
        const bool active = st == 1;
        const long long n = n0 + i;
        {   // L2 prefetch of this group's next tile (one 32-byte sector holds four rows of a level)
            const int in = i + kGroups4 * (int)gridDim.x * kRows;
            if (in < Nc && (row & 3) == 0) {
#pragma unroll
                for (int l = 0; l < 16; ++l) prefetch_l2(feats_lm + in + (size_t)l * Nc);
            }
        }
        if (c.any(active)) {
            float x[32];
            if (active) {
#pragma unroll
                for (int l = 0; l < 16; ++l) {
                    const float2 v = __ldg(feats_lm + i + (size_t)l * Nc);
                    x[2 * l] = v.x; x[2 * l + 1] = v.y;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) x[j] = 0.0f;
            }
            const int ray0 = (int)((n0 + i0) / a.S);
            const long long last_n = n0 + (i0 + kRows - 1 < Nc ? i0 + kRows - 1 : Nc - 1);
            const int nrays = (int)(last_n / a.S) - ray0 + 1;
            const int my_ray = active ? (int)(n / a.S) - ray0 : 0;
            float head[10], zh[7];
            forward_layers4<true>(c, smem, P, Q, x, rb + my_ray * 64, head, zh,
                                  [&]() { ray_vectors4<true>(rb, w3sh, a.rays_d, ray0, nrays, c.gtid); });   // under the L1 MMAs
            float zs[16];
            umma::tmem_ld16(c.tmem + c4Dh + c.lane_addr, zs);
            umma::tc_wait_ld();
            if (active) {
                // Decoder::inference activations (decoder.h:134-146): softplus without threshold, expf sigmoids
                const float sigma = logf(1.0f + expf(zh[0]));
                f3 dif = mk3(1.0f / (1.0f + expf(-zh[1])), 1.0f / (1.0f + expf(-zh[2])), 1.0f / (1.0f + expf(-zh[3])));
                const f3 tint = mk3(1.0f / (1.0f + expf(-zh[4])), 1.0f / (1.0f + expf(-zh[5])), 1.0f / (1.0f + expf(-zh[6])));
                f3 spe = mk3(tint.x / (1.0f + expf(-(zs[0] + bias[oB5 + 0]))), tint.y / (1.0f + expf(-(zs[1] + bias[oB5 + 1]))),
                             tint.z / (1.0f + expf(-(zs[2] + bias[oB5 + 2]))));
                const float2 ws = aux[i];
                const float al = 1.0f - expf(-1.0f * sigma * ws.y);
                float wa = ws.x * al;
                dif = dif * wa; spe = spe * wa;
                if (MODE != kBackSlot && ws.x > 0) {               // the reference divides by the weight sum when it is positive
                    const float inv = 1.0f / ws.x;
                    dif = dif * inv; spe = spe * inv; wa *= inv;
                }
                st3(a.out_diffuse + 3 * (size_t)n, dif);
                st3(a.out_specular + 3 * (size_t)n, spe);
                a.out_alpha[n] = wa;
            }
        }
        if (st == 0) {                                         // unoccupied / unassigned foreground sample: zeros
            st3(a.out_diffuse + 3 * (size_t)n, mk3(0, 0, 0));
            st3(a.out_specular + 3 * (size_t)n, mk3(0, 0, 0));
            a.out_alpha[n] = 0.0f;
        }
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 0) umma::tmem_free<512>(tmem_slot);
}

// ------------------------------------------------------------------------------------------------------------------
// Multi-tile path: the (sample, slot) pairs that need the field of a scene tile are grouped by tile id (counting sort,
// each tile's segment padded to whole 256-row blocks), encoded level-major per tile and decoded block by block -- a
// decode CTA takes a contiguous run of blocks, so the decoder weights are restaged only when the run crosses into
// the next scene tile -- and a last pass sums every sample's pairs in slot order (the order of the reference's loop,
// rendering_kernel.cu:520-600) and applies the weight normalisation.  Cost is proportional to the number of active
// pairs, not to the number of tiles.
struct Work {
    int *counts, *cursor, *offsets, *total_rows;   // [nb] x 3, [1]
    int* blk_tile;                                 // [max_rows / 256] scene tile of each 256-row block
    int* row_sample;                               // [max_rows] sample index inside the chunk (-1: padding)
    float4* row_uw;                                // [max_rows] table coordinate u, blend weight w
    float* row_scale;                              // [max_rows] alpha scale (step length x |d|, or the bg step)
    int* pair_row;                                 // [Nc][4] row of the pair in slot s (-1: none)
    float* wsum;                                   // [Nc] sum of the member weights (< 0: leave the caller's rows alone)
    float2* feats;                                 // [16][max_rows]
    float4* rowout;                                // [max_rows][2] w * alpha * (diffuse, specular), w * alpha
    int max_rows;
};
constexpr int kBlockRows = 2 * kRows;

struct Pairs {
    int id[kMaxPts];
    f3 u[kMaxPts];
    float w[kMaxPts];
    float wsum, scale;
};

// the slots of sample n that need a field evaluation (id[s] = -1: none), in slot order
template <int MODE>
__device__ __forceinline__ void sample_pairs(const InferArgs& a, long long n, bool live, Pairs& P)
{
#pragma unroll
    for (int s = 0; s < kMaxPts; ++s) { P.id[s] = -1; P.u[s] = mk3(0, 0, 0); P.w[s] = 0.0f; }
    P.wsum = 0.0f; P.scale = 0.0f;
    if (!live) return;
    const int ray = (int)(n / a.S), k = (int)(n % a.S);
    const f3 o = ld3(a.rays_o + 3 * (size_t)ray), d = ld3(a.rays_d + 3 * (size_t)ray);
    const float zv = a.z_vals[n];
    short ids[kMaxPts] = {-1, -1, -1, -1};
    if (MODE == kFore) {
        const short4 s4 = *reinterpret_cast<const short4*>(a.slots + (size_t)n * kMaxPts);
        ids[0] = s4.x; ids[1] = s4.y; ids[2] = s4.z; ids[3] = s4.w;
        P.scale = a.dists[n] * sqrtf(dot3(d, d));
    } else {
        const short* sl = a.slots + (size_t)ray * kMaxPts;
        if (MODE == kBackSlot) ids[0] = sl[a.step];
        else { ids[0] = sl[0]; ids[1] = sl[1]; ids[2] = sl[2]; ids[3] = sl[3]; }
        P.scale = (k == a.S - 1) ? 10000000.0f : a.z_vals[n + 1] - zv;
    }
    if (MODE == kBackSlot && ids[0] < 0) { P.wsum = -1.0f; return; }
    const f3 p = o + zv * d;
    bool open = true;
#pragma unroll
    for (int s = 0; s < kMaxPts; ++s) {
        open = open && ids[s] >= 0;                           // slots after the first -1 are ignored
        bool first = open;
#pragma unroll
        for (int j = 0; j < s; ++j) first = first && ids[j] != ids[s];
        if (!first) continue;
        const Geom g = sample_geom<MODE>(a, ids[s], ray, s, p);
        P.wsum += g.w;
        if (g.active) { P.id[s] = ids[s]; P.u[s] = g.u; P.w[s] = g.w; }
    }
}

template <int MODE, bool FILL>
__global__ void __launch_bounds__(256)
work_plan_kernel(InferArgs a, long long n0, int Nc, Work w)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
    Pairs P;
    sample_pairs<MODE>(a, n0 + i, i < Nc, P);
    int rows[kMaxPts];
#pragma unroll
    for (int s = 0; s < kMaxPts; ++s) {
        // one atomic per warp and distinct tile: the lanes of a warp that want the same tile take consecutive rows
        const int b = P.id[s];
        const unsigned m = __match_any_sync(0xffffffffu, b);
        const int leader = __ffs(m) - 1;
        int base = 0;
        if (b >= 0 && lane == leader) base = atomicAdd((FILL ? w.cursor : w.counts) + b, __popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        rows[s] = -1;
        if (FILL && b >= 0) {
            const int r = w.offsets[b] + base + __popc(m & ((1u << lane) - 1u));
            rows[s] = r;
            w.row_sample[r] = i;
            w.row_uw[r] = make_float4(P.u[s].x, P.u[s].y, P.u[s].z, P.w[s]);
            w.row_scale[r] = P.scale;
        }
    }
    if (FILL && i < Nc) {
        *reinterpret_cast<int4*>(w.pair_row + (size_t)i * kMaxPts) = make_int4(rows[0], rows[1], rows[2], rows[3]);
        w.wsum[i] = P.wsum;
    }
}

// exclusive scan of the per-tile row counts, padded to whole blocks; one CTA
__global__ void __launch_bounds__(256)
work_scan_kernel(Work w, int nb)
{
    __shared__ int warp_sum[8];
    __shared__ int carry;
    __shared__ int seg_start[256], seg_blocks[256];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nb; b0 += 256) {
        const int b = b0 + tid;
        const int padded = b < nb ? (w.counts[b] + kBlockRows - 1) / kBlockRows * kBlockRows : 0;
        int incl = padded;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += v;
        }
        if (lane == 31) warp_sum[wid] = incl;
        __syncthreads();
        int before = carry;
        for (int j = 0; j < wid; ++j) before += warp_sum[j];
        const int start = before + incl - padded;
        if (b < nb) w.offsets[b] = start;
        seg_start[tid] = start / kBlockRows;
        seg_blocks[tid] = padded / kBlockRows;
        __syncthreads();
        if (tid == 255) carry = start + padded;
        for (int q = 0; q < 256 && b0 + q < nb; ++q)           // the whole CTA labels each segment's blocks
            for (int j = tid; j < seg_blocks[q]; j += 256) w.blk_tile[seg_start[q] + j] = b0 + q;
        __syncthreads();
    }
    if (tid == 0) *w.total_rows = carry;
}

__global__ void __launch_bounds__(256)
work_encode_kernel(InferArgs a, Work w)
{
    const int l = blockIdx.y, total = *w.total_rows;
    const uint32_t mask = a.T - 1u;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < total; r += gridDim.x * blockDim.x) {
        if (w.row_sample[r] < 0) continue;
        const int b = w.blk_tile[r / kBlockRows];
        const int* res = a.resolution + (size_t)b * 48 + 3 * l;
        const __half2* tl = a.tables + ((size_t)b * 16 + l) * a.T;
        const float4 uw = w.row_uw[r];
        const float vx = uw.x * (float)(res[0] - 1), vy = uw.y * (float)(res[1] - 1), vz = uw.z * (float)(res[2] - 1);
        const int ix = (int)vx, iy = (int)vy, iz = (int)vz;
        const float ox = vx - (float)ix, oy = vy - (float)iy, oz = vz - (float)iz;
        float2 f[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = __half22float2(__ldg(tl + hash3(ix + ((k >> 2) & 1), iy + ((k >> 1) & 1), iz + (k & 1), mask)));
        const float ax = 1 - ox, ay = 1 - oy, az = 1 - oz;
        const float wt[8] = {ax * ay * az, ax * ay * oz, ax * oy * az, ax * oy * oz, ox * ay * az, ox * ay * oz, ox * oy * az, ox * oy * oz};
        float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; ++k) { s0 += wt[k] * f[k].x; s1 += wt[k] * f[k].y; }
        w.feats[(size_t)l * w.max_rows + r] = make_float2(s0, s1);
    }
}

__global__ void __launch_bounds__(kThreadsDec, 1)
work_decode_kernel(InferArgs a, long long n0, Work w)
{
    SNRF_DECODE_PROLOGUE((const float*)nullptr)
    const int blocks = *w.total_rows / kBlockRows;
    const int per = (blocks + gridDim.x - 1) / gridDim.x;
    const int blk_end = min(blocks, ((int)blockIdx.x + 1) * per);
    int staged = -1;
    for (int blk = blockIdx.x * per; blk < blk_end; ++blk) {
        const int b = w.blk_tile[blk];
        if (b != staged) {                                     // CTA-uniform: both groups are done with the old weights
            __syncthreads();
            stage_all_weights<true>(smem, flat_params(a.params + (size_t)b * 13994), nullptr, tid, kThreadsDec);
            umma::fence_async_smem();
            __syncthreads();
            staged = b;
        }
        const int r = blk * kBlockRows + c.group * kRows + row;
        const int i = w.row_sample[r];
        const bool active = i >= 0;
        float sigma = 0.0f;
        f3 dif = mk3(0, 0, 0), spe = mk3(0, 0, 0);
        const f3 d = active ? ld3(a.rays_d + 3 * (size_t)((n0 + i) / a.S)) : mk3(0, 0, 1);
        const bool done = eval_tile(c, Tl, active, w.feats + r, (size_t)w.max_rows, d, sigma, dif, spe);
        if (done && active && cg == 0) {
            const float wgt = w.row_uw[r].w;
            const float wa = wgt * (1.0f - expf(-1.0f * sigma * w.row_scale[r]));
            w.rowout[2 * (size_t)r] = make_float4(wa * dif.x, wa * dif.y, wa * dif.z, wa);
            w.rowout[2 * (size_t)r + 1] = make_float4(wa * spe.x, wa * spe.y, wa * spe.z, 0.0f);
        }
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 0) umma::tmem_free<512>(tmem_slot);
}

template <int MODE>
__global__ void __launch_bounds__(256)
work_combine_kernel(InferArgs a, long long n0, int Nc, Work w)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Nc; i += gridDim.x * blockDim.x) {
        const float wsum = w.wsum[i];
        if (wsum < 0.0f) continue;                             // background ray without a tile in this slot
        const int4 rows4 = *reinterpret_cast<const int4*>(w.pair_row + (size_t)i * kMaxPts);
        const int rows[kMaxPts] = {rows4.x, rows4.y, rows4.z, rows4.w};
        f3 acc_d = mk3(0, 0, 0), acc_s = mk3(0, 0, 0);
        float acc_a = 0.0f;
#pragma unroll
        for (int s = 0; s < kMaxPts; ++s) {
            if (rows[s] < 0) continue;
            const float4 p0 = w.rowout[2 * (size_t)rows[s]], p1 = w.rowout[2 * (size_t)rows[s] + 1];
            acc_d = acc_d + mk3(p0.x, p0.y, p0.z);
            acc_s = acc_s + mk3(p1.x, p1.y, p1.z);
            acc_a += p0.w;
        }
        if (MODE != kBackSlot && wsum > 0) {
            const float inv = 1.0f / wsum;                     // float3 /= float: multiply by the reciprocal
            acc_d = acc_d * inv; acc_s = acc_s * inv; acc_a = acc_a * inv;
        }
        const long long n = n0 + i;
        st3(a.out_diffuse + 3 * (size_t)n, acc_d);
        st3(a.out_specular + 3 * (size_t)n, acc_s);
        a.out_alpha[n] = acc_a;
    }
}

int g_chunk_log2 = 24;       // single-tile path: log2 of the samples per chunk (snrf_infer_set_chunk_log2; 22: 221 ms, 24: 218 ms per 1080p frame)

// Scratch for both paths comes from a private stream-ordered pool that keeps its memory across
// synchronisations (the default pool hands it back to the driver at every sync; re-mapping 3 GB per call costs tens of
// milliseconds).  snrf_infer_release_scratch() trims it.
inline cudaError_t scratch_alloc(void** ptr, size_t bytes, cudaStream_t s) { return snrf_scratch_alloc(ptr, bytes, s); }

// single-tile driver: chunks of samples, scratch from the stream-ordered allocator
template <int MODE>
int launch_two_pass(const InferArgs& a, void* stream, const char* name)
{
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(infer_decode_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd_smem<true>());
        if (e == cudaSuccess) e = cudaFuncSetAttribute(infer_decode4_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd4_smem<true>());
        if (e != cudaSuccess) { snrf_set_error("%s: %s", name, cudaGetErrorString(e)); return (int)e; }
        configured = true;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const long long total = (long long)a.B * a.S;
    // samples per chunk: every chunk streams the whole table from HBM once (level slice by level slice through L2), so the table
    // traffic of a frame is (samples / chunk) GiB -- 128 GiB per 1080p frame at 4 Mi samples, ~10 % of its time; the scratch is
    // 153 B per sample of a chunk (snrf_infer_set_chunk_log2)
    const long long chunk = 1ll << g_chunk_log2;
    const long long cap = total < chunk ? total : chunk;
    void* scratch = nullptr;
    const size_t bytes = (size_t)cap * (16 * 8 + 16 + 8 + 1) + 256;
    cudaError_t e = scratch_alloc(&scratch, bytes, s);
    if (e != cudaSuccess) { snrf_set_error("%s: scratch allocation of %zu bytes: %s", name, bytes, cudaGetErrorString(e)); return (int)e; }
    float2* feats = (float2*)scratch;
    float4* uw = (float4*)(feats + (size_t)cap * 16);
    float2* aux = (float2*)(uw + cap);
    unsigned char* state = (unsigned char*)(aux + cap);
    const int sms = snrf_sm_count();
    for (long long n0 = 0; n0 < total; n0 += chunk) {
        const int Nc = (int)(total - n0 < chunk ? total - n0 : chunk);
        int gx = snrf_div_up(Nc, 256);
        if (gx > sms * 32) gx = sms * 32;
        infer_geometry_kernel<MODE><<<gx, 256, 0, s>>>(a, n0, Nc, uw, aux, state);
        infer_encode_kernel<<<dim3(gx, 16), 256, 0, s>>>(a, Nc, uw, state, feats);
        const int num_tiles = snrf_div_up(Nc, kRows);
        int grid = sms;
        if (a.S >= kMinS4) {                                     // four tiles in flight per CTA
            if (grid > (num_tiles + 3) / 4) grid = (num_tiles + 3) / 4;
            infer_decode4_kernel<MODE><<<grid, kThreadsDec, fwd4_smem<true>(), s>>>(a, n0, Nc, feats, aux, state, num_tiles);
            continue;
        }
        if (grid > (num_tiles + 1) / 2) grid = (num_tiles + 1) / 2;
        infer_decode_kernel<MODE><<<grid, kThreadsDec, fwd_smem<true>(), s>>>(a, n0, Nc, feats, aux, state, num_tiles);
    }
    e = cudaGetLastError();
    cudaFreeAsync(scratch, s);
    if (e != cudaSuccess) { snrf_set_error("%s: %s", name, cudaGetErrorString(e)); return (int)e; }
    return 0;
}

// multi-tile driver: chunks of samples; worst case every sample holds kMaxPts pairs
template <int MODE>
int launch_work(const InferArgs& a, int nb, void* stream, const char* name)
{
    static bool configured = false;
    if (!configured) {
        const cudaError_t e = cudaFuncSetAttribute(work_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd_smem<true>());
        if (e != cudaSuccess) { snrf_set_error("%s: %s", name, cudaGetErrorString(e)); return (int)e; }
        configured = true;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const long long total = (long long)a.B * a.S;
    constexpr int slots = MODE == kBackSlot ? 1 : kMaxPts;
    // 4 Mi samples per chunk: every chunk streams the level slices of the tiles it touches from HBM once, so small
    // chunks multiply the table traffic; worst-case scratch (every foreground sample in 4 tiles) = 3.1 GB
    const long long chunk = 4ll << 20;
    const long long cap = total < chunk ? total : chunk;
    // every tile's segment is padded to whole blocks: at most one partial block per tile that has pairs
    const long long tiles_hit = (long long)nb < cap * slots ? nb : cap * slots;
    const long long max_rows = (cap * slots + tiles_hit * (kBlockRows - 1) + kBlockRows - 1) / kBlockRows * kBlockRows;
    if (max_rows > 0x7fffffffll) { snrf_set_error("%s: work list too large", name); return 1; }
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_counts = take((size_t)(3 * nb + 1) * 4), o_blk = take((size_t)(max_rows / kBlockRows) * 4), o_sample = take((size_t)max_rows * 4),
                 o_uw = take((size_t)max_rows * 16), o_scale = take((size_t)max_rows * 4), o_pair = take((size_t)cap * kMaxPts * 4),
                 o_wsum = take((size_t)cap * 4), o_feats = take((size_t)max_rows * 16 * 8), o_out = take((size_t)max_rows * 32);
    unsigned char* base = nullptr;
    cudaError_t e = scratch_alloc((void**)&base, off, s);
    if (e != cudaSuccess) { snrf_set_error("%s: scratch allocation of %zu bytes: %s", name, off, cudaGetErrorString(e)); return (int)e; }
    Work w;
    w.counts = (int*)(base + o_counts); w.cursor = w.counts + nb; w.offsets = w.cursor + nb; w.total_rows = w.offsets + nb;
    w.blk_tile = (int*)(base + o_blk); w.row_sample = (int*)(base + o_sample); w.row_uw = (float4*)(base + o_uw);
    w.row_scale = (float*)(base + o_scale); w.pair_row = (int*)(base + o_pair); w.wsum = (float*)(base + o_wsum);
    w.feats = (float2*)(base + o_feats); w.rowout = (float4*)(base + o_out); w.max_rows = (int)max_rows;
    const int sms = snrf_sm_count();
    for (long long n0 = 0; n0 < total; n0 += chunk) {
        const int Nc = (int)(total - n0 < chunk ? total - n0 : chunk);
        const int gp = snrf_div_up(Nc, 256);
        e = cudaMemsetAsync(w.counts, 0, (size_t)(3 * nb + 1) * 4, s);
        if (e == cudaSuccess) e = cudaMemsetAsync(w.row_sample, 0xff, (size_t)max_rows * 4, s);
        if (e != cudaSuccess) break;
        work_plan_kernel<MODE, false><<<gp, 256, 0, s>>>(a, n0, Nc, w);
        work_scan_kernel<<<1, 256, 0, s>>>(w, nb);
        work_plan_kernel<MODE, true><<<gp, 256, 0, s>>>(a, n0, Nc, w);
        int gx = snrf_div_up((long long)Nc * slots, 256);
        if (gx > sms * 32) gx = sms * 32;
        work_encode_kernel<<<dim3(gx, 16), 256, 0, s>>>(a, w);
        work_decode_kernel<<<sms, kThreadsDec, fwd_smem<true>(), s>>>(a, n0, w);
        work_combine_kernel<MODE><<<gp < sms * 32 ? gp : sms * 32, 256, 0, s>>>(a, n0, Nc, w);
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    cudaFreeAsync(base, s);
    if (e != cudaSuccess) { snrf_set_error("%s: %s", name, cudaGetErrorString(e)); return (int)e; }
    return 0;
}

// nb = number of scene tiles behind `params` / `tables`
template <int MODE>
int launch(const InferArgs& a, int nb, void* stream, const char* name)
{
    return (nb == 1 && MODE != kBackBlend) ? launch_two_pass<MODE>(a, stream, name) : launch_work<MODE>(a, nb, stream, name);
}

}  // namespace

// ------------------------------- C ABI --------------------------------------
// tuning hook: log2 of the samples per chunk of the single-tile path (20 .. 26; scratch = 153 B per sample of a chunk)
SNRF_API void snrf_infer_set_chunk_log2(int bits) { g_chunk_log2 = bits < 20 ? 20 : (bits > 26 ? 26 : bits); }
SNRF_API int snrf_infer_release_scratch(void) { return snrf_scratch_release(); }

SNRF_API int snrf_pts_inference(const float* rays_o, const float* rays_d, const float* z_vals, const float* dists,
                                const short* block_idxs, const void* features_tables, const float* params, const int* resolution,
                                const unsigned char* grid_occupied, const long long* grid_starts, const int* grid_log2dim,
                                const float* corners, const float* sizes, float* diffuse, float* specular, float* alpha, int B,
                                int S, int T, int nb, void* stream)
{
    SNRF_CHECK_ARG(T > 0 && (T & (T - 1)) == 0, "snrf_pts_inference: hashmap size must be a power of two (got %d)", T);
    if (B <= 0 || S <= 0) return 0;
    InferArgs a{rays_o, rays_d, z_vals, dists, block_idxs, nullptr, (const __half2*)features_tables, params, resolution, grid_occupied,
                grid_starts, grid_log2dim, corners, sizes, diffuse, specular, alpha, B, S, 0, (uint32_t)T};
    return launch<kFore>(a, nb, stream, "snrf_pts_inference");
}

SNRF_API int snrf_bg_pts_inference(const float* rays_o, const float* rays_d, const float* z_vals, const short* outgoing_bidxs,
                                   const float* blend_weights, const float* corners, const float* sizes, const int* resolution,
                                   const void* features_tables, const float* params, float* diffuse, float* specular, float* alpha,
                                   int B, int S, int T, int nb, void* stream)
{
    SNRF_CHECK_ARG(T > 0 && (T & (T - 1)) == 0, "snrf_bg_pts_inference: hashmap size must be a power of two (got %d)", T);
    if (B <= 0 || S <= 0) return 0;
    InferArgs a{rays_o, rays_d, z_vals, nullptr, outgoing_bidxs, blend_weights, (const __half2*)features_tables, params, resolution, nullptr,
                nullptr, nullptr, corners, sizes, diffuse, specular, alpha, B, S, 0, (uint32_t)T};
    return launch<kBackBlend>(a, nb, stream, "snrf_bg_pts_inference");
}

SNRF_API int snrf_bg_pts_inference_v2(const float* rays_o, const float* rays_d, const float* z_vals, const short* bg_idxs, int step,
                                      const float* corners, const float* sizes, const int* resolution, const void* features_tables,
                                      const float* params, float* diffuse, float* specular, float* alpha, int B, int S, int T,
                                      int nb, void* stream)
{
    SNRF_CHECK_ARG(T > 0 && (T & (T - 1)) == 0, "snrf_bg_pts_inference_v2: hashmap size must be a power of two (got %d)", T);
    SNRF_CHECK_ARG(step >= 0 && step < kMaxPts, "snrf_bg_pts_inference_v2: step must be in [0,4) (got %d)", step);
    if (B <= 0 || S <= 0) return 0;
    InferArgs a{rays_o, rays_d, z_vals, nullptr, bg_idxs, nullptr, (const __half2*)features_tables, params, resolution, nullptr,
                nullptr, nullptr, corners, sizes, diffuse, specular, alpha, B, S, step, (uint32_t)T};
    return launch<kBackSlot>(a, nb, stream, "snrf_bg_pts_inference_v2");
}
