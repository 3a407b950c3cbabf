// Density / colour decoder MLP on the 5th-generation tensor cores (tcgen05.mma, accumulators
// in TMEM), forward and backward, sm_100a.
//
// Replaces (behaviour, not code) network.ShallowMLP.forward (network.py:151-190) and its
// autograd backward, which the reference runs as 8 cuBLAS SGEMMs + ~25 elementwise torch
// kernels per direction:
//   x   = feat(32) * level_mask(32)
//   h1  = g(W1 x + b1)            32 -> 64      g(v) = exp(-v^2 / 0.02)
//   H   = W2 h1 + b2              64 -> 64      (no activation)
//   sigma   = softplus(ws  . H[0:32] + bs)
//   diffuse = sigmoid (Wd    H[0:32] + bd)      3
//   tint    = sigmoid (Wt    H[0:32] + bt)      3
//   x2  = [H[32:64], SH16(d / (|d| + 1e-8))]    48
//   specular = sigmoid(W5 g(W4 g(W3 x2 + b3) + b4) + b5)    48 -> 64 -> 64 -> 3
//
// Design (B200).  A CTA owns tiles of 128 consecutive samples (M = 128, one TMEM lane and one
// thread per sample).  Every operand -- activations and weights -- is a bf16 tile with 128-byte
// rows, 128B-swizzled (umma.cuh); a layer is a handful of tcgen05.mma (K = 16 each) issued by one
// thread, completion is signalled through an mbarrier (tcgen05.commit), the epilogue pulls the
// fp32 accumulator row out of TMEM (tcgen05.ld), applies bias + activation in registers and
// writes the next layer's operand tile.  Weights are converted to bf16 tiles once per CTA
// (persistent grid).  Nothing but the 40-byte head row per sample is written to HBM in the
// forward; the backward recomputes the forward per tile, keeps every intermediate in shared
// memory, accumulates all weight / bias gradients in TMEM across the CTA's tiles (M = 64
// accumulators) and flushes them once at the end.
//
// Precision.  The Gaussian activation amplifies operand rounding (d a / a = -100 z dz), so plain
// bf16 operands cost ~1 % in the directional branch.  SPLIT mode (the default) therefore feeds the
// tensor cores error-compensated operands in every forward GEMM: v = hi + lo with hi = bf16(v),
// lo = bf16(v - hi), and  A W^T ~= A_hi W_hi^T + A_lo W_hi^T + A_hi W_lo^T  (three MMAs into the
// same fp32 accumulator, ~16 mantissa bits).  In the backward the input-gradient GEMMs (the chain
// that ends in d/d features -> table and pose gradients) are compensated the same way, with
// dz = dz_hi + dz_lo; the weight-gradient GEMMs use the hi parts only (their rounding errors are
// independent per sample and average out over the batch).
#include "decoder_core.cuh"

using namespace dec;

namespace {

// ------------------------------- forward ------------------------------------
// feats [N,32] f32, rays_d [R,3] (sample n belongs to ray n / S), out [N,10] f32 =
// (sigma, tint3, diffuse3, specular3).
template <bool SPLIT>
__global__ void __launch_bounds__(kThreadsDec, 1)
decoder_fwd_kernel(const float* __restrict__ feats, const float* __restrict__ mask32, const float* __restrict__ rays_d,
                   DecoderParams p, float* __restrict__ out, int N, int S, int num_tiles, long long level_stride,
                   const unsigned char* __restrict__ ray_valid)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t bars[2];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;

    stage_all_weights<SPLIT>(smem, p, mask32, tid, kThreadsDec);
    if (warp == 0) umma::tmem_alloc<512>(&tmem_slot);
    if (tid == 0) { umma::mbar_init(&bars[0], 1); umma::mbar_init(&bars[1], 1); umma::mbar_fence_init(); }
    umma::fence_async_smem();
    umma::tc_fence_before();
    __syncthreads();
    umma::tc_fence_after();
    Ctx<SPLIT, 2> c;                                    // two tiles in flight: group = warp >> 3 owns one
    c.init(smem, bars, tmem_slot);
    unsigned char* T0 = smem + off_tiles<SPLIT>() + c.group * fwd_tiles<SPLIT>() * kTile;
    unsigned char* T1 = T0 + kTile;
    unsigned char* T2 = T1 + kTile;
    unsigned char* LOa = SPLIT ? T2 + kTile : T1;      // never written when !SPLIT
    unsigned char* LOb = SPLIT ? LOa + kTile : T2;
    const Tiles T{T0, T1, T2, T1, T2, LOa, LOb};

    for (int tile = 2 * blockIdx.x + c.group; tile < num_tiles; tile += 2 * gridDim.x) {
        const int n = tile * kRows + c.row;
        const bool live = n < N && (ray_valid == nullptr || ray_valid[n / S] != 0);
        if (ray_valid != nullptr && !c.any(live)) continue;     // every sample of the tile belongs to a masked-out ray
        float head[10], zh[7];
        f3 d = mk3(0.f, 0.f, 1.f);
        float dn = 1.0f;
        forward_tile<SPLIT, 2>(c, T, feats, rays_d, n, live, S, head, zh, d, dn, level_stride);
        if (c.cg == 0) {
            float z[16];
            umma::tmem_ld16(c.tmem + cDh + c.lane_addr, z);
            umma::tc_wait_ld();
#pragma unroll
            for (int j = 0; j < 3; ++j) head[7 + j] = sigmoidf(z[j] + c.bias[oB5 + j]);
            if (live) {
                float2* o = reinterpret_cast<float2*>(out + (size_t)n * 10);
#pragma unroll
                for (int j = 0; j < 5; ++j) o[j] = make_float2(head[2 * j], head[2 * j + 1]);
            }
        }
        // every MMA of this tile has completed; the next tile's first sync_operands() orders its
        // operand stores and this tile's TMEM loads before the next accumulator writes
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 0) umma::tmem_free<512>(tmem_slot);
}


// ------------------------------- forward, four tiles in flight ---------------
// (decoder_core.cuh: forward_layers4; same results as decoder_fwd_kernel, S >= kMinS4)
template <bool SPLIT>
__global__ void __launch_bounds__(kThreadsDec, 1)
decoder_fwd4_kernel(const float* __restrict__ feats, const float* __restrict__ mask32, const float* __restrict__ rays_d,
                    DecoderParams p, float* __restrict__ out, int N, int S, int num_tiles, long long level_stride,
                    const unsigned char* __restrict__ ray_valid)
{
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t bars[kGroups4];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;

    stage_all_weights<SPLIT>(smem, p, mask32, tid, kThreadsDec);
    float* w3sh = reinterpret_cast<float*>(smem + off_w3sh<SPLIT>());
    stage_w3sh(w3sh, p, tid, kThreadsDec);
    stage_fold_weights4<SPLIT>(smem, p, reinterpret_cast<float*>(smem + off_tiles4<SPLIT>()), tid, kThreadsDec);
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
    unsigned char* P = smem + off_tiles4<SPLIT>() + c.group * 2 * kTile;
    unsigned char* Q = P + kTile;
    float* rb = reinterpret_cast<float*>(smem + off_raybias4<SPLIT>()) + c.group * kMaxRays4 * 64;
    const float* mask = reinterpret_cast<const float*>(smem + off_mask<SPLIT>());
    const float* bias = reinterpret_cast<const float*>(smem + off_bias<SPLIT>());

    for (int tile = kGroups4 * blockIdx.x + c.group; tile < num_tiles; tile += kGroups4 * gridDim.x) {
        const int n0 = tile * kRows, n = n0 + c.row;
        const bool live = n < N && (ray_valid == nullptr || ray_valid[n / S] != 0);
        if (ray_valid != nullptr && !c.any(live)) continue;     // every sample of the tile belongs to a masked-out ray
        {   // L2 prefetch of this group's next tile (one 32-byte sector holds four rows of a level)
            const long long nn = (long long)(tile + kGroups4 * gridDim.x) * kRows + c.row;
            if (nn < N) {
                if (level_stride == 0) { prefetch_l2(feats + (size_t)nn * 32); prefetch_l2(feats + (size_t)nn * 32 + 16); }
                else if ((c.row & 3) == 0) {
#pragma unroll
                    for (int l = 0; l < 16; ++l) prefetch_l2(reinterpret_cast<const float2*>(feats) + nn + (size_t)l * level_stride);
                }
            }
        }
        float x[32];
        if (live) {
            if (level_stride == 0) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 a = __ldg(reinterpret_cast<const float4*>(feats + (size_t)n * 32 + 4 * q));
                    x[4 * q] = a.x; x[4 * q + 1] = a.y; x[4 * q + 2] = a.z; x[4 * q + 3] = a.w;
                }
            } else {
                const float2* f2 = reinterpret_cast<const float2*>(feats) + n;
#pragma unroll
                for (int l = 0; l < 16; ++l) {
                    const float2 a = __ldg(f2 + (size_t)l * level_stride);
                    x[2 * l] = a.x; x[2 * l + 1] = a.y;
                }
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) x[j] *= mask[j];
        } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) x[j] = 0.0f;
        }
        // the rays of this tile (the previous tile's epilogues are done with rb: every thread passed its last wait_mma,
        // and the first sync_operands of forward_layers4 orders these writes before any read)
        const int ray0 = n0 / S;
        const int last = (n0 + kRows - 1 < N ? n0 + kRows - 1 : N - 1) / S;
        const int my_ray = (live ? n / S : ray0) - ray0;
        float head[10], zh[7];
        // the ray vectors are formed under the L1 MMAs: the first barrier of forward_layers4 has every thread of the group past
        // its last read of rb (the previous tile's z3 epilogue), two more barriers follow before the next read
        forward_layers4<SPLIT>(c, smem, P, Q, x, rb + my_ray * 64, head, zh,
                               [&]() { ray_vectors4<false>(rb, w3sh, rays_d, ray0, last - ray0 + 1, c.gtid); });
        float z[16];
        umma::tmem_ld16(c.tmem + c4Dh + c.lane_addr, z);
        umma::tc_wait_ld();
#pragma unroll
        for (int j = 0; j < 3; ++j) head[7 + j] = sigmoidf(z[j] + bias[oB5 + j]);
        if (live) {
            float2* o = reinterpret_cast<float2*>(out + (size_t)n * 10);
#pragma unroll
            for (int j = 0; j < 5; ++j) o[j] = make_float2(head[2 * j], head[2 * j + 1]);
        }
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 0) umma::tmem_free<512>(tmem_slot);
}

// ------------------------------- backward ------------------------------------------------------------------------------
// Per tile: recompute the forward keeping the intermediates in shared memory, then walk the layers backwards.  Each stage
// commits its input-gradient GEMM (dA = dz W, the weight tile read MN-major) first and issues its weight-gradient GEMMs
// (dW += dz^T A, both operands MN-major, M = 64 accumulators that stay in TMEM for the whole kernel) behind the commit, so
// that they execute under the epilogue; a tile ends with a commit on `bar_tail`, waited for before the next tile overwrites
// the operand tiles.  The weight-gradient GEMMs read the hi parts of both operands: the two roundings are symmetric (2^-12,
// unbiased, independent per sample) and average out over the batch.
//
// Layer 2 of the decoder has NO activation (network.py:160-163: H = W2 h1 + b2 feeds the heads and the directional branch
// linearly), so it composes with its consumers:
//     z3 = H[32:64] W3a^T + SH W3b^T + b3 = a1 (W3a W2b)^T + SH W3b^T + (W3a b2b + b3)         W32 := W3a W2b   [64 x 64]
//     zh = H[0:32]  Wh^T + bh             = a1 (Wh  W2a)^T + (Wh b2a + bh)                     Wh2 := Wh  W2a   [ 7 x 64]
// (W2a / W2b = rows 0..31 / 32..63 of W2, b2a / b2b likewise).  With the forward's head values at hand the backward needs
// neither H nor dH as tensors:
//     dA1 = dz3 W32 + dzh Wh2                                  (one stage; was: dH = [dzh Wh | dz3 W3a], then dA1 = dH W2)
//     G  := dz3^T a1 [64 x 64],  Gh := dzh^T a1 [7 x 64]       (the only weight-gradient GEMMs of layers 2 / 3a / heads)
//     dW3a = G W2b^T + db3 (x) b2b      dWh = Gh W2a^T + dbh (x) b2a      dW2 = [Wh^T Gh ; W3a^T G]      db2 = [Wh^T dbh ; W3a^T db3]
// where the second line is evaluated ONCE per CTA in fp32 after the last tile (0.3 M multiply-adds).  Per tile that leaves
// SIX dependent stages (L1 | z3 | L4 + first backward stage | B2 | B3 | B5) instead of the ten of a layer-by-layer recompute
// and backward, nine operand tiles instead of ten, 33 + 42 issue-side MMAs less, and no epilogue at all for H / dH.  W32 / Wh2 are formed in
// fp32 from the fp32 parameters when the CTA stages its weights and split hi + lo like every other operand.
namespace fold {
constexpr int oW1 = 0, oW32 = 8192, oW32l = 16384, oW3b = 24576, oW4 = 32768, oW4l = 40960, oWh2 = 49152, oWh2l = 51200,
              oW5 = 53248, oW5l = 55296, weights_end = 57344;
constexpr int oB1 = 0, oB32 = 64, oB4 = 128, nB = 192;                 // fp32 biases: b1, b32 = W3a b2b + b3, b4
constexpr int off_bias = weights_end, off_mask = off_bias + nB * 4;
constexpr int off_tiles = ((off_mask + 128 + 1023) / 1024) * 1024;
constexpr int kTiles = 9;
constexpr int smem_bytes = off_tiles + kTiles * kTile + 1024;
// TMEM columns: two working accumulators + d[SH], then the persistent gradient accumulators
constexpr int cDa = 0, cDb = 64, cSH = 128, gW1 = 144, gG = 192, gW3b = 256, gW4 = 272, gGhT = 336, gW5T = 352;   // ends at 368
}  // namespace fold

template <bool SPLIT>
__global__ void __launch_bounds__(kThreadsDec, 1)
decoder_bwd_fold_kernel(const float* __restrict__ feats, const float* __restrict__ mask32, const float* __restrict__ rays_d,
                        DecoderParams p, const float* __restrict__ grad_heads, float* __restrict__ grad_feats,
                        float* __restrict__ grad_rays_d, DecoderGrads gp, int N, int S, int num_tiles, long long level_stride,
                        const unsigned char* __restrict__ ray_valid, const unsigned* __restrict__ gmax_bits,
                        const float* __restrict__ heads_fwd, const unsigned char* __restrict__ sample_live)
{
    using namespace fold;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char* base = smem + off_tiles;
    unsigned char *tA0 = base, *tLOb = base + kTile, *ta1 = base + 2 * kTile, *tg1 = base + 3 * kTile, *ta3 = base + 4 * kTile,
                  *tg3 = base + 5 * kTile, *ta4 = base + 6 * kTile, *tg4 = base + 7 * kTile, *tLOa = base + 8 * kTile;
    unsigned char* Tdz = tLOb;           // [dz_heads | dz_spec | their lo parts] (x_lo is dead after the L1 GEMM)
    __shared__ uint64_t bar;
    __shared__ uint64_t bar_tail;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint32_t tail_phase = 0, phase = 0;
    bool tail_pending = false;
    // Power-of-two scale of the incoming gradient: max |grad_heads| (bits in *gmax_bits, from grad_absmax_kernel) is
    // mapped into [0.5, 1), so that the fp16 dz operands keep 15 binary orders of headroom above it for the growth along
    // the backward chain and 14 (24 with subnormals) below it.  Everything downstream is linear in the gradient:
    // outputs are multiplied by ginv (exact).  A zero / non-finite maximum leaves the scale at 1.
    float gscale = 1.0f, ginv = 1.0f;
    if (kOpBf16 == 0 && gmax_bits != nullptr) {
        const int e = (int)((*gmax_bits >> 23) & 0xffu);            // gmax = m 2^(e - 127), m in [1, 2)
        if (e > 0 && e < 255) {
            int se = 253 - e;                                        // exponent field of 2^(126 - e): gmax * scale in [0.5, 1)
            se = se < 1 ? 1 : (se > 253 ? 253 : se);
            gscale = __uint_as_float((uint32_t)se << 23);
            ginv = __uint_as_float((uint32_t)(254 - se) << 23);
        }
    }

    // ---- weights: composed matrices in fp32 (scratch = the operand-tile area), then every operand tile as hi + lo
    for (int i = tid; i < weights_end / 16; i += kThreadsDec) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
    float* s32 = reinterpret_cast<float*>(base);                       // W32 [64][64]
    float* sh2 = s32 + 64 * 64;                                        // Wh2 [7][64]
    // fp32 copies of the factors, row pitch 65 / 33 (conflict-free whichever index the lanes run over): W2 [64][64], W3a =
    // W3[:, 0:32] [64][32], Wh [7][32], b2 [64] -- the composition below and the flush at the end read them from shared memory
    // (from global memory the 64-term sums cost ~75 us per launch in dependent, strided L1 / L2 loads)
    float* sW2 = sh2 + 8 * 64;
    float* sW3a = sW2 + 64 * 65;
    float* sWh = sW3a + 64 * 33;
    float* sb2 = sWh + 8 * 33;
    auto load_factors = [&]() {
        for (int i = tid; i < 64 * 64; i += kThreadsDec) sW2[(i >> 6) * 65 + (i & 63)] = w_at(p.W2, i >> 6, i & 63, 64, 64, p.flat);
        for (int i = tid; i < 64 * 32; i += kThreadsDec) sW3a[(i >> 5) * 33 + (i & 31)] = w_at(p.W3, i >> 5, i & 31, 64, 48, p.flat);
        for (int i = tid; i < 7 * 32; i += kThreadsDec) sWh[(i >> 5) * 33 + (i & 31)] = wh_at(p, i >> 5, i & 31);
        for (int i = tid; i < 64; i += kThreadsDec) sb2[i] = p.b2[i];
    };
    float* bias = reinterpret_cast<float*>(smem + off_bias);
    float* maskv = reinterpret_cast<float*>(smem + off_mask);
    load_factors();
    __syncthreads();
    for (int i = tid; i < 64 * 64; i += kThreadsDec) {
        const int o = i >> 6, j = i & 63;
        float acc = 0.0f;
#pragma unroll 8
        for (int k = 0; k < 32; ++k) acc += sW3a[o * 33 + k] * sW2[(32 + k) * 65 + j];
        s32[i] = acc;
    }
    for (int i = tid; i < 7 * 64; i += kThreadsDec) {
        const int h = i >> 6, j = i & 63;
        float acc = 0.0f;
#pragma unroll 8
        for (int k = 0; k < 32; ++k) acc += sWh[h * 33 + k] * sW2[k * 65 + j];
        sh2[i] = acc;
    }
    for (int i = tid; i < nB; i += kThreadsDec) {
        float v;
        if (i < 64) v = p.b1[i];
        else if (i < 128) {
            const int o = i - 64;
            v = p.b3[o];
            for (int k = 0; k < 32; ++k) v += sW3a[o * 33 + k] * sb2[32 + k];
        } else v = p.b4[i - 128];
        bias[i] = v;
    }
    for (int i = tid; i < 32; i += kThreadsDec) maskv[i] = mask32 ? mask32[i] : 1.0f;
    __syncthreads();
    stage_weight<SPLIT>(smem + oW1, smem + oW1, 0, p.W1, 64, 32, p.flat, tid, kThreadsDec);
    stage_weight<SPLIT>(smem + oW4, smem + oW4l, 0, p.W4, 64, 64, p.flat, tid, kThreadsDec);
    stage_weight<SPLIT>(smem + oW5, smem + oW5l, 0, p.W5, 3, 64, p.flat, tid, kThreadsDec);
    stage_weight<SPLIT>(smem + oW32, smem + oW32l, 0, s32, 64, 64, 0, tid, kThreadsDec);
    stage_weight<SPLIT>(smem + oWh2, smem + oWh2l, 0, sh2, 7, 64, 0, tid, kThreadsDec);
    for (int t = tid; t < 64 * 2; t += kThreadsDec) {                  // W3b = W3[:, 32:48]: hi in columns 0..15, lo in columns 32..47
        const int r = t >> 1, c = t & 1;
        float hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float w = w_at(p.W3, r, 32 + 8 * c + j, 64, 48, p.flat);
            hi[j] = w;
            lo[j] = w - op_round(w);
        }
        op_tile_store8(smem + oW3b, r, c, hi);
        if (SPLIT) op_tile_store8(smem + oW3b, r, 4 + c, lo);
    }
    if (warp == 0) umma::tmem_alloc<512>(&tmem_slot);
    if (tid == 0) { umma::mbar_init(&bar, 1); umma::mbar_init(&bar_tail, 1); umma::mbar_fence_init(); }
    umma::fence_async_smem();
    umma::tc_fence_before();
    __syncthreads();
    umma::tc_fence_after();

    const int row = 32 * (warp & 3) + lane, cg = warp >> 2;           // thread (row, column group): 16 of the 64 columns of a layer
    const uint32_t tmem = tmem_slot, lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    const uint32_t aA0 = umma::smem_u32(tA0), aa1 = umma::smem_u32(ta1), ag1 = umma::smem_u32(tg1), aa3 = umma::smem_u32(ta3),
                   ag3 = umma::smem_u32(tg3), aa4 = umma::smem_u32(ta4), ag4 = umma::smem_u32(tg4), aLOa = umma::smem_u32(tLOa),
                   aLOb = umma::smem_u32(tLOb), adz = aLOb;
    const uint32_t aW1 = umma::smem_u32(smem + oW1), aW32 = umma::smem_u32(smem + oW32), aW32l = umma::smem_u32(smem + oW32l),
                   aW3b = umma::smem_u32(smem + oW3b), aW4 = umma::smem_u32(smem + oW4), aW4l = umma::smem_u32(smem + oW4l),
                   aWh2 = umma::smem_u32(smem + oWh2), aWh2l = umma::smem_u32(smem + oWh2l), aW5 = umma::smem_u32(smem + oW5),
                   aW5l = umma::smem_u32(smem + oW5l);
    constexpr uint32_t idf64 = umma::idesc_f16(128, 64, 0, 0, kOpBf16, kOpBf16);
    constexpr uint32_t idg64 = umma::idesc_f16(128, 64, 0, 1, kOpBf16, kOpBf16), idg32 = umma::idesc_f16(128, 32, 0, 1, kOpBf16, kOpBf16),
                       idg16 = umma::idesc_f16(128, 16, 0, 1, kOpBf16, kOpBf16);
    constexpr uint32_t idw64 = umma::idesc_f16(64, 64, 1, 1, kOpBf16, kOpBf16), idw48 = umma::idesc_f16(64, 48, 1, 1, kOpBf16, kOpBf16),
                       idw16 = umma::idesc_f16(64, 16, 1, 1, kOpBf16, kOpBf16);
    // dA (+)= dz W over nk k-steps: A = dz rows (K-major, hi + lo), B = the weight tile read MN-major (hi, lo)
    auto dgrad = [&](int col, uint32_t dz_tile, int dz_k, uint32_t dzlo_tile, int dzlo_k, uint32_t w_hi, uint32_t w_lo, int nk,
                     uint32_t idesc, bool acc) {
        for (int k = 0; k < nk; ++k)
            umma::mma_bf16(tmem + col, umma::desc_kmajor(dz_tile, dz_k + k), umma::desc_mnmajor(w_hi, k), idesc, acc || k > 0);
        if (SPLIT) {
            for (int k = 0; k < nk; ++k)
                umma::mma_bf16(tmem + col, umma::desc_kmajor(dz_tile, dz_k + k), umma::desc_mnmajor(w_lo, k), idesc, 1);
            for (int k = 0; k < nk; ++k)
                umma::mma_bf16(tmem + col, umma::desc_kmajor(dzlo_tile, dzlo_k + k), umma::desc_mnmajor(w_hi, k), idesc, 1);
        }
    };
    // dW += A^T B over the 128 rows of the tile (both operands MN-major, hi parts); init: first group ever into that accumulator
    auto wgrad = [&](int col, uint32_t a_tile, uint32_t b_tile_plus_off, uint32_t idesc, bool init) {
        for (int k = 0; k < 8; ++k)
            umma::mma_bf16(tmem + col, umma::desc_mnmajor(a_tile, k), umma::desc_mnmajor(b_tile_plus_off, k), idesc, (!init) || k > 0);
    };
    auto sync_operands = [&]() {
        umma::fence_async_smem();
        umma::tc_fence_before();
        __syncthreads();
        umma::tc_fence_after();
    };
    auto wait_mma = [&]() {
        umma::mbar_wait(&bar, phase);
        phase ^= 1u;
        umma::tc_fence_after();
    };
    float v[16];
    float acc_b4[16], acc_small[10];
#pragma unroll
    for (int j = 0; j < 16; ++j) acc_b4[j] = 0.0f;
#pragma unroll
    for (int j = 0; j < 10; ++j) acc_small[j] = 0.0f;
    // Gaussian layer epilogue on this thread's 16 columns: a = exp(-50 z^2) -> (Ta hi, Tlo lo), g = da/dz -> Tg
    auto gauss_epilogue = [&](int col, int boff, unsigned char* Ta, unsigned char* Tlo, unsigned char* Tg) {
        float g[16];
        umma::tmem_ld16(tmem + col + lane_addr + 16 * cg, v);
        umma::tc_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float z = v[j] + bias[boff + 16 * cg + j];
            const float a = gauss_act(z);
            v[j] = a;
            g[j] = -100.0f * z * a;
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            store8_act<SPLIT>(Ta, 2 * cg + q, Tlo, 2 * cg + q, row, v + 8 * q);
            umma::tile_store8_f16(Tg, row, 2 * cg + q, g + 8 * q);
        }
    };
    // dz = dA * g on this thread's 16 columns: hi in place over the g tile, lo into Tlo
    auto mul_inplace = [&](int col, unsigned char* Tg, unsigned char* Tlo) {
        umma::tmem_ld16(tmem + col + lane_addr + 16 * cg, v);
        umma::tc_wait_ld();
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const uint4 w4 = *reinterpret_cast<const uint4*>(Tg + umma::tile_chunk_off(row, 2 * cg + q));
            const uint32_t w[4] = {w4.x, w4.y, w4.z, w4.w};
            float o[8];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const __half2 h2 = *reinterpret_cast<const __half2*>(&w[e]);
                o[2 * e] = v[8 * q + 2 * e] * __low2float(h2);
                o[2 * e + 1] = v[8 * q + 2 * e + 1] * __high2float(h2);
            }
            store8_act<SPLIT>(Tg, 2 * cg + q, Tlo, 2 * cg + q, row, o);
        }
    };
    const bool lead_warp = umma::warp_uniform() == 4;
    bool first = true;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int n = tile * kRows + row;
        const bool live = n < N && (ray_valid == nullptr || ray_valid[n / S] != 0) && (sample_live == nullptr || sample_live[n] != 0);
        if ((ray_valid != nullptr || sample_live != nullptr) && !__syncthreads_or(live)) continue;     // masked-out / terminated samples only
        if (cg == 0 && live) {
            prefetch_l2(grad_heads + (size_t)n * 10);
            prefetch_l2(grad_heads + (size_t)n * 10 + 8);
            prefetch_l2(heads_fwd + (size_t)n * 10);
            prefetch_l2(heads_fwd + (size_t)n * 10 + 8);
        }
        {
            const long long nn = (long long)(tile + gridDim.x) * kRows + row;
            if (nn < N) {
                if (level_stride == 0) prefetch_l2(feats + (size_t)nn * 32 + 8 * cg);
                else {
#pragma unroll
                    for (int l = 0; l < 4; ++l) if ((row & 3) == 0) prefetch_l2(reinterpret_cast<const float2*>(feats) + nn + (size_t)(4 * cg + l) * level_stride);
                }
            }
        }
        // ---- input rows: 8 features per thread times the level mask (the SH columns follow under the L1 MMAs)
        f3 d = mk3(0.f, 0.f, 1.f);
        float dn = 1.0f;
        {
            float x[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) x[j] = 0.0f;
            if (live) {
                if (level_stride == 0) {
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const float4 a = __ldg(reinterpret_cast<const float4*>(feats + (size_t)n * 32 + 8 * cg + 4 * q));
                        x[4 * q] = a.x; x[4 * q + 1] = a.y; x[4 * q + 2] = a.z; x[4 * q + 3] = a.w;
                    }
                } else {
                    const float2* f2 = reinterpret_cast<const float2*>(feats) + n;
#pragma unroll
                    for (int l = 0; l < 4; ++l) {
                        const float2 a = __ldg(f2 + (size_t)(4 * cg + l) * level_stride);
                        x[2 * l] = a.x; x[2 * l + 1] = a.y;
                    }
                }
                if (cg >= 2) d = ld3(rays_d + 3 * (size_t)(n / S));      // (issued now, consumed under the L1 MMAs)
#pragma unroll
                for (int j = 0; j < 8; ++j) x[j] *= maskv[8 * cg + j];
            }
            // the previous tile's trailing weight-gradient MMAs still read the operand tiles: waited for here, after this
            // tile's global loads have been issued
            if (tail_pending) {
                umma::mbar_wait(&bar_tail, tail_phase);
                umma::tc_fence_after();
                tail_phase ^= 1u;
                tail_pending = false;
            }
            store8_act<SPLIT>(tA0, cg, tLOb, cg, row, x);               // x_hi -> A0 columns 8 cg .., x_lo -> LOb
        }
        sync_operands();
        // ---- L1: Da = x W1^T (K = 32)
        if (lead_warp && umma::elect_one()) {
            fwd_gemm<SPLIT>(tmem + cDa, aA0, 0, aLOb, 0, aW1, 0, aW1, 2, 2, idf64, false);
            umma::mma_commit(&bar);
        }
        // (under the L1 MMAs, which read columns 0..31 of A0 only) SH of d / (|d| + 1e-8) -> A0 columns 32..47 (hi) / 48..63 (lo):
        // column group 2 stores SH 0..7, column group 3 SH 8..15; the z3 stage's sync_operands orders the stores
        if (cg >= 2) {
            float sh[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) sh[j] = 0.0f;
            if (live) {
                dn = sqrtf(d.x * d.x + d.y * d.y + d.z * d.z);
                const float inv = 1.0f / (dn + 1e-8f);
                sh16(d.x * inv, d.y * inv, d.z * inv, sh);
            }
            store8_act<SPLIT>(tA0, 4 + (cg - 2), tA0, 6 + (cg - 2), row, sh + 8 * (cg - 2));
            if (!SPLIT) umma::tile_zero8(tA0, row, 6 + (cg - 2));
        }
        wait_mma();
        gauss_epilogue(cDa, oB1, ta1, tLOa, tg1);
        sync_operands();
        // ---- z3 straight from a1: Db = a1 W32^T (K = 64) + SH W3b^T (K = 16)
        if (lead_warp && umma::elect_one()) {
            fwd_gemm<SPLIT>(tmem + cDb, aa1, 0, aLOa, 0, aW32, 0, aW32l, 0, 4, idf64, false);
            fwd_gemm<SPLIT>(tmem + cDb, aA0, 2, aA0, 3, aW3b, 0, aW3b, 2, 1, idf64, true);
            umma::mma_commit(&bar);
        }
        // (under the MMAs) d(loss)/d(pre-activations) of the 7 heads and the 3 specular outputs, from the forward's head values
        if (cg == 0) {
            float dzh[16], dzs[16], gh[10], hv[10];
            if (live) {
                const float2* gsrc = reinterpret_cast<const float2*>(grad_heads + (size_t)n * 10);
                const float2* hsrc = reinterpret_cast<const float2*>(heads_fwd + (size_t)n * 10);
#pragma unroll
                for (int j = 0; j < 5; ++j) {
                    const float2 t = __ldg(gsrc + j), h = __ldg(hsrc + j);
                    gh[2 * j] = t.x * gscale; gh[2 * j + 1] = t.y * gscale;
                    hv[2 * j] = h.x; hv[2 * j + 1] = h.y;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 10; ++j) { gh[j] = 0.0f; hv[j] = 0.0f; }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) { dzh[j] = 0.0f; dzs[j] = 0.0f; }
            dzh[0] = gh[0] * (hv[0] > 20.0f ? 1.0f : -expm1f(-hv[0]));          // softplus' = sigmoid(z) = 1 - exp(-sigma)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                dzh[1 + j] = gh[4 + j] * hv[4 + j] * (1.0f - hv[4 + j]);        // diffuse
                dzh[4 + j] = gh[1 + j] * hv[1 + j] * (1.0f - hv[1 + j]);        // tint
                dzs[j] = gh[7 + j] * hv[7 + j] * (1.0f - hv[7 + j]);            // specular
            }
            // Tdz = [dz_heads 0..15 | dz_spec 16..31 | dz_heads_lo 32..47 | dz_spec_lo 48..63]  (x_lo: the L1 GEMM has completed)
            store8_act<SPLIT>(Tdz, 0, Tdz, 4, row, dzh);
            store8_act<SPLIT>(Tdz, 1, Tdz, 5, row, dzh + 8);
            store8_act<SPLIT>(Tdz, 2, Tdz, 6, row, dzs);
            store8_act<SPLIT>(Tdz, 3, Tdz, 7, row, dzs + 8);
#pragma unroll
            for (int j = 0; j < 10; ++j) acc_small[j] += j < 7 ? dzh[j] : dzs[j - 7];
        }
        wait_mma();
        gauss_epilogue(cDb, oB32, ta3, tLOa, tg3);
        sync_operands();
        // ---- L4 + first backward stage: Da = a3 W4^T ; Db = dA4 = dz_spec W5 ; GhT += a1^T dz_heads
        if (lead_warp && umma::elect_one()) {
            fwd_gemm<SPLIT>(tmem + cDa, aa3, 0, aLOa, 0, aW4, 0, aW4l, 0, 4, idf64, false);
            dgrad(cDb, adz, 1, adz, 3, aW5, aW5l, 1, idg64, false);
            umma::mma_commit(&bar);
            wgrad(gGhT, aa1, adz, idw16, first);
        }
        wait_mma();
        {   // a4 = g(z4) (hi part only: nothing reads a4_lo), dz5 = dA4 * g'(z4) with g' still in registers
            float z4[16];
            umma::tmem_ld16(tmem + cDa + lane_addr + 16 * cg, z4);
            umma::tmem_ld16(tmem + cDb + lane_addr + 16 * cg, v);
            umma::tc_wait_ld();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float z = z4[j] + bias[oB4 + 16 * cg + j];
                const float a = gauss_act(z);
                z4[j] = a;
                v[j] *= -100.0f * z * a;
                acc_b4[j] += v[j];
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                umma::tile_store8_f16(ta4, row, 2 * cg + q, z4 + 8 * q);
                store8_act<SPLIT>(tg4, 2 * cg + q, tLOa, 2 * cg + q, row, v + 8 * q);
            }
        }
        sync_operands();
        // ---- B2: dA3 = dz5 W4 ; dW4 += dz5^T a3 ; dW5^T += a4^T dz_spec
        if (lead_warp && umma::elect_one()) {
            dgrad(cDa, ag4, 0, aLOa, 0, aW4, aW4l, 4, idg64, false);
            umma::mma_commit(&bar);
            wgrad(gW4, ag4, aa3, idw64, first);
            wgrad(gW5T, aa4, adz + 32, idw16, first);
        }
        wait_mma();
        mul_inplace(cDa, tg3, tLOa);                                 // dz3 (the deferred MMAs read g4 / a3 / a4 / Tdz, not g3 / LOa)
        sync_operands();
        // ---- B3: dA1 = dz3 W32 + dz_heads Wh2 ; d[SH] = dz3 W3b ; G += dz3^T a1 ; dW3b += dz3^T SH (column 0 -> db3)
        if (lead_warp && umma::elect_one()) {
            dgrad(cDb, ag3, 0, aLOa, 0, aW32, aW32l, 4, idg64, false);
            dgrad(cDb, adz, 0, adz, 2, aWh2, aWh2l, 1, idg64, true);
            dgrad(cSH, ag3, 0, aLOa, 0, aW3b, aW3b + 64, 4, idg16, false);    // (N = 16: cheap; reads the dz3 lo tile this epilogue overwrites)
            umma::mma_commit(&bar);
            wgrad(gG, ag3, aa1, idw64, first);
            wgrad(gW3b, ag3, aA0 + 64, idw16, first);
        }
        wait_mma();
        mul_inplace(cDb, tg1, tLOa);                                 // dz1
        sync_operands();
        // ---- B5: dx = dz1 W1 (32 columns) ; dW1 += dz1^T [x | SH] (column 32 -> db1)
        if (lead_warp && umma::elect_one()) {
            dgrad(cDa, ag1, 0, aLOa, 0, aW1, aW1 + 64, 4, idg32, false);
            umma::mma_commit(&bar);
            wgrad(gW1, ag1, aA0, idw48, first);
            umma::mma_commit(&bar_tail);                            // everything this tile issued
        }
        // (under the B5 MMAs) d/d(ray direction) through the SH encoding, one thread per row of column group 3
        if (grad_rays_d != nullptr && cg == 3) {
            float dsh[16];
            umma::tmem_ld16(tmem + cSH + lane_addr, dsh);
            umma::tc_wait_ld();
            float gx = 0.f, gy = 0.f, gz = 0.f;
            if (live) {
                const float inv = 1.0f / (dn + 1e-8f);
                const float x = d.x * inv, y = d.y * inv, z = d.z * inv;
                const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
                const float C1 = 0.4886025119029199f, C2a = 1.0925484305920792f, C2c = 0.31539156525252005f,
                            C2e = 0.5462742152960396f, C3a = 0.5900435899266435f, C3b = 2.890611442640554f,
                            C3c = 0.4570457994644658f, C3d = 0.3731763325901154f, C3e = 1.445305721320277f;
                float vx = 0.f, vy = 0.f, vz = 0.f;
                vy += dsh[1] * C1; vz += dsh[2] * C1; vx += dsh[3] * C1;
                vx += dsh[4] * C2a * y; vy += dsh[4] * C2a * x;
                vy += dsh[5] * -C2a * z; vz += dsh[5] * -C2a * y;
                vx += dsh[6] * C2c * -2.f * x; vy += dsh[6] * C2c * -2.f * y; vz += dsh[6] * C2c * 4.f * z;
                vx += dsh[7] * -C2a * z; vz += dsh[7] * -C2a * x;
                vx += dsh[8] * C2e * 2.f * x; vy += dsh[8] * C2e * -2.f * y;
                vx += dsh[9] * -C3a * 6.f * xy; vy += dsh[9] * -C3a * (3.f * xx - 3.f * yy);
                vx += dsh[10] * C3b * yz; vy += dsh[10] * C3b * xz; vz += dsh[10] * C3b * xy;
                vx += dsh[11] * -C3c * -2.f * xy; vy += dsh[11] * -C3c * (4.f * zz - xx - 3.f * yy); vz += dsh[11] * -C3c * 8.f * yz;
                vx += dsh[12] * C3d * -6.f * xz; vy += dsh[12] * C3d * -6.f * yz; vz += dsh[12] * C3d * (6.f * zz - 3.f * xx - 3.f * yy);
                vx += dsh[13] * -C3c * (4.f * zz - 3.f * xx - yy); vy += dsh[13] * -C3c * -2.f * xy; vz += dsh[13] * -C3c * 8.f * xz;
                vx += dsh[14] * C3e * 2.f * xz; vy += dsh[14] * C3e * -2.f * yz; vz += dsh[14] * C3e * (xx - yy);
                vx += dsh[15] * -C3a * (3.f * xx - 3.f * yy); vy += dsh[15] * -C3a * -6.f * xy;
                const float ddv = d.x * vx + d.y * vy + d.z * vz;
                const float k2 = dn > 0.f ? ddv * inv * inv / dn : 0.f;
                gx = (vx * inv - d.x * k2) * ginv; gy = (vy * inv - d.y * k2) * ginv; gz = (vz * inv - d.z * k2) * ginv;
            }
            const int ray = live ? n / S : -1;
            const int ray0 = __shfl_sync(0xffffffffu, ray, 0);
            if (__all_sync(0xffffffffu, ray == ray0 || ray < 0)) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    gx += __shfl_xor_sync(0xffffffffu, gx, off);
                    gy += __shfl_xor_sync(0xffffffffu, gy, off);
                    gz += __shfl_xor_sync(0xffffffffu, gz, off);
                }
                if (lane == 0 && ray0 >= 0) {
                    atomicAdd(grad_rays_d + 3 * (size_t)ray0 + 0, gx);
                    atomicAdd(grad_rays_d + 3 * (size_t)ray0 + 1, gy);
                    atomicAdd(grad_rays_d + 3 * (size_t)ray0 + 2, gz);
                }
            } else if (live) {
                atomicAdd(grad_rays_d + 3 * (size_t)ray + 0, gx);
                atomicAdd(grad_rays_d + 3 * (size_t)ray + 1, gy);
                atomicAdd(grad_rays_d + 3 * (size_t)ray + 2, gz);
            }
        }
        wait_mma();
        umma::tmem_ld8(tmem + cDa + lane_addr + 8 * cg, v);         // d/d x, columns 8 cg .. 8 cg + 7 = levels 4 cg .. 4 cg + 3
        umma::tc_wait_ld();
        if (live) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] *= maskv[8 * cg + j] * ginv;
            if (level_stride == 0) {
                float4* dst = reinterpret_cast<float4*>(grad_feats + (size_t)n * 32 + 8 * cg);
                dst[0] = make_float4(v[0], v[1], v[2], v[3]);
                dst[1] = make_float4(v[4], v[5], v[6], v[7]);
            } else {
                float2* dst = reinterpret_cast<float2*>(grad_feats) + n;
#pragma unroll
                for (int l = 0; l < 4; ++l) dst[(size_t)(4 * cg + l) * level_stride] = make_float2(v[2 * l], v[2 * l + 1]);
            }
        }
        tail_pending = true;
        first = false;
    }
    if (tail_pending) {
        umma::mbar_wait(&bar_tail, tail_phase);
        umma::tc_fence_after();
    }

    // ================= flush: TMEM accumulators -> global gradients, the folded ones through the composition =================
    umma::tc_fence_after();
    float* sG = reinterpret_cast<float*>(base);            // G [64][64]
    float* sGh = sG + 64 * 64;                             // Gh [8][64] (7 used)
    float* sdb3 = sGh + 8 * 64;                            // [64]
    float* sdbh = sdb3 + 64;                               // [8]  (7 used)
    // the factors again (their copies of the prologue were overwritten by the operand tiles), behind the four arrays above
    sW2 = sdbh + 8;
    sW3a = sW2 + 64 * 65;
    sWh = sW3a + 64 * 33;
    sb2 = sWh + 8 * 33;
    load_factors();
    if (tid < 8) sdbh[tid] = 0.0f;
    __syncthreads();
    if (!first) {
        const int m = 16 * (warp & 3) + lane;              // M = 64 accumulators: row m in TMEM lane 32 (m / 16) + m % 16
        const bool own = lane < 16 && cg == 0;
        float w[32];
        auto flush = [&](int col, int ncols, float* dst, int ld, int col0) {
            for (int c0 = 0; c0 < ncols; c0 += 32) {
                const int nc = ncols - c0 >= 32 ? 32 : ncols - c0;
                if (nc == 32) umma::tmem_ld32(tmem + col + c0 + lane_addr, w);
                else umma::tmem_ld16(tmem + col + c0 + lane_addr, w);
                umma::tc_wait_ld();
                if (own)
                    for (int j = 0; j < nc; ++j) atomicAdd(dst + (size_t)m * ld + col0 + c0 + j, w[j] * ginv);
            }
        };
        flush(gW1, 32, gp.W1, 32, 0);
        flush(gW3b, 16, gp.W3, 48, 32);
        flush(gW4, 64, gp.W4, 64, 0);
        for (int c0 = 0; c0 < 64; c0 += 32) {              // G -> shared memory
            umma::tmem_ld32(tmem + gG + c0 + lane_addr, w);
            umma::tc_wait_ld();
            if (own)
                for (int j = 0; j < 32; ++j) sG[m * 64 + c0 + j] = w[j] * ginv;
        }
        float b8[16];
        umma::tmem_ld16(tmem + gW1 + 32 + lane_addr, b8);  // d/d b1 = column 32 (SH_0) of the [64 x 48] dW1 accumulator / SH_0
        umma::tc_wait_ld();
        if (own) atomicAdd(gp.b1 + m, b8[0] * kInvSH0 * ginv);
        umma::tmem_ld16(tmem + gW3b + lane_addr, b8);      // d/d b3 = column 0 of dW3b / SH_0
        umma::tc_wait_ld();
        if (own) { const float t = b8[0] * kInvSH0 * ginv; atomicAdd(gp.b3 + m, t); sdb3[m] = t; }
        umma::tmem_ld16(tmem + gGhT + lane_addr, b8);      // GhT: row = a1 feature j, column = head h
        umma::tc_wait_ld();
        if (own)
            for (int h = 0; h < 7; ++h) sGh[h * 64 + m] = b8[h] * ginv;
        umma::tmem_ld16(tmem + gW5T + lane_addr, b8);
        umma::tc_wait_ld();
        if (own)
            for (int o = 0; o < 3; ++o) atomicAdd(gp.W5 + o * 64 + m, b8[o] * ginv);
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        float t4 = acc_b4[j];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t4 += __shfl_xor_sync(0xffffffffu, t4, off);
        if (lane == 0 && !first) atomicAdd(gp.b4 + 16 * cg + j, t4 * ginv);
    }
    if (cg == 0) {
#pragma unroll
        for (int j = 0; j < 10; ++j) {
            float t = acc_small[j];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
            if (lane == 0 && !first) {
                float* dst = j == 0 ? gp.bs : (j < 4 ? gp.bd + (j - 1) : (j < 7 ? gp.bt + (j - 4) : gp.b5 + (j - 7)));
                atomicAdd(dst, t * ginv);
                if (j < 7) atomicAdd(sdbh + j, t * ginv);
            }
        }
    }
    __syncthreads();
    if (!first) {
        // dW3a [o][k] = sum_j G[o][j] W2[32 + k][j] + db3[o] b2[32 + k]
        for (int i = tid; i < 64 * 32; i += kThreadsDec) {
            const int o = i >> 5, k = i & 31;
            float acc = sdb3[o] * sb2[32 + k];
#pragma unroll 8
            for (int j = 0; j < 64; ++j) acc += sG[o * 64 + j] * sW2[(32 + k) * 65 + j];
            atomicAdd(gp.W3 + o * 48 + k, acc);
        }
        // dW2 [32 + k][j] = sum_o W3[o][k] G[o][j] ;  dW2 [k][j] = sum_h Wh[h][k] Gh[h][j]
        for (int i = tid; i < 32 * 64; i += kThreadsDec) {
            const int k = i >> 6, j = i & 63;
            float acc = 0.0f, acch = 0.0f;
#pragma unroll 8
            for (int o = 0; o < 64; ++o) acc += sW3a[o * 33 + k] * sG[o * 64 + j];
#pragma unroll
            for (int h = 0; h < 7; ++h) acch += sWh[h * 33 + k] * sGh[h * 64 + j];
            atomicAdd(gp.W2 + (32 + k) * 64 + j, acc);
            atomicAdd(gp.W2 + k * 64 + j, acch);
        }
        // dWh [h][k] = sum_j Gh[h][j] W2[k][j] + dbh[h] b2[k]
        for (int i = tid; i < 7 * 32; i += kThreadsDec) {
            const int h = i >> 5, k = i & 31;
            float acc = sdbh[h] * sb2[k];
#pragma unroll 8
            for (int j = 0; j < 64; ++j) acc += sGh[h * 64 + j] * sW2[k * 65 + j];
            float* dst = h == 0 ? gp.Ws + k : (h < 4 ? gp.Wd + (h - 1) * 32 + k : gp.Wt + (h - 4) * 32 + k);
            atomicAdd(dst, acc);
        }
        // db2 [32 + k] = sum_o W3[o][k] db3[o] ;  db2 [k] = sum_h Wh[h][k] dbh[h]
        for (int k = tid; k < 32; k += kThreadsDec) {
            float acc = 0.0f, acch = 0.0f;
            for (int o = 0; o < 64; ++o) acc += sW3a[o * 33 + k] * sdb3[o];
            for (int h = 0; h < 7; ++h) acch += sWh[h * 33 + k] * sdbh[h];
            atomicAdd(gp.b2 + 32 + k, acc);
            atomicAdd(gp.b2 + k, acch);
        }
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 0) umma::tmem_free<512>(tmem);
}

// max |grad_heads| over the live samples, as float bits (non-negative floats order like unsigned integers; a NaN sorts
// above inf and is treated as "no scale" by the backward)
__global__ void __launch_bounds__(256)
grad_absmax_kernel(const float* __restrict__ g, int N, int S, const unsigned char* __restrict__ ray_valid, unsigned* __restrict__ out)
{
    // one head row (10 floats = 5 float2) per thread and trip: 32-bit index arithmetic, one division per row
    unsigned m = 0u;
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
        if (ray_valid != nullptr && !ray_valid[n / S]) continue;              // rows of masked-out rays are never written
        const float2* row = reinterpret_cast<const float2*>(g + (size_t)n * 10);
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            const float2 t = __ldg(row + j);
            const unsigned a = __float_as_uint(t.x) & 0x7fffffffu, b = __float_as_uint(t.y) & 0x7fffffffu;
            m = a > m ? a : m;
            m = b > m ? b : m;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) { const unsigned o = __shfl_xor_sync(0xffffffffu, m, off); m = o > m ? o : m; }
    if ((threadIdx.x & 31) == 0 && m != 0u) atomicMax(out, m);
}
__device__ unsigned g_gmax_slots[64];      // a ring: concurrent backward launches on different streams use different slots
int g_gmax_next = 0;

int g_split = 1;       // 1 = error-compensated bf16x3 operands in the forward GEMMs (default), 0 = plain bf16

template <typename K>
int set_smem(K kernel, int bytes, const char* name)
{
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) { snrf_set_error("%s: %s", name, cudaGetErrorString(e)); return (int)e; }
    return 0;
}

// snrf_decoder_bwd / snrf_decoder_bwd_ert; sample_live (may be NULL): the early-ray-termination flags of snrf_composite_fwd_ert
int decoder_bwd(const float* feats, const float* mask32, const float* rays_d, const float* const* params, const float* grad_heads,
                float* grad_feats, float* grad_rays_d, float* const* grad_params, int N, int S, int level_major,
                const unsigned char* ray_valid, const float* heads_fwd, const unsigned char* sample_live, void* stream)
{
    SNRF_CHECK_ARG(N >= 0 && S > 0, "snrf_decoder_bwd: need N >= 0, S > 0 (N=%d S=%d)", N, S);
    SNRF_CHECK_ARG(params != nullptr && grad_params != nullptr, "snrf_decoder_bwd: params and grad_params are required");
    SNRF_CHECK_ARG(heads_fwd != nullptr, "snrf_decoder_bwd: heads_fwd (the output of snrf_decoder_fwd) is required");
    if (N == 0) return 0;
    DecoderParams p{params[0], params[1], params[2], params[3], params[4], params[5], params[6], params[7],
                    params[8], params[9], params[10], params[11], params[12], params[13], params[14], params[15]};
    DecoderGrads g{grad_params[0], grad_params[1], grad_params[2], grad_params[3], grad_params[4], grad_params[5],
                   grad_params[6], grad_params[7], grad_params[8], grad_params[9], grad_params[10], grad_params[11],
                   grad_params[12], grad_params[13], grad_params[14], grad_params[15]};
    static bool configured = false;
    if (!configured) {
        int rc = set_smem(decoder_bwd_fold_kernel<true>, fold::smem_bytes, "snrf_decoder_bwd");
        if (rc == 0) rc = set_smem(decoder_bwd_fold_kernel<false>, fold::smem_bytes, "snrf_decoder_bwd");
        if (rc) return rc;
        configured = true;
    }
    const int num_tiles = snrf_div_up(N, kRows);
    int grid = snrf_sm_count();            // one CTA per SM: all 512 TMEM columns, 200-225 KB of shared memory
    if (grid > num_tiles) grid = num_tiles;
    cudaStream_t s = (cudaStream_t)stream;
    // gradient scale for the fp16 operands: max |grad_heads| -> a device slot the backward kernel reads (no host sync)
    unsigned* slots = nullptr;
    cudaError_t e = cudaGetSymbolAddress((void**)&slots, g_gmax_slots);
    if (e != cudaSuccess) { snrf_set_error("snrf_decoder_bwd: %s", cudaGetErrorString(e)); return (int)e; }
    unsigned* slot = slots + (g_gmax_next++ & 63);
    cudaMemsetAsync(slot, 0, sizeof(unsigned), s);
    {
        int gx = snrf_div_up(N, 256 * 4);
        if (gx > snrf_sm_count() * 8) gx = snrf_sm_count() * 8;
        grad_absmax_kernel<<<gx > 0 ? gx : 1, 256, 0, s>>>(grad_heads, N, S, ray_valid, slot);
    }
    if (g_split)
        decoder_bwd_fold_kernel<true><<<grid, kThreadsDec, fold::smem_bytes, s>>>(feats, mask32, rays_d, p, grad_heads, grad_feats, grad_rays_d, g, N, S, num_tiles, level_major ? (long long)N : 0ll, ray_valid, slot, heads_fwd, sample_live);
    else
        decoder_bwd_fold_kernel<false><<<grid, kThreadsDec, fold::smem_bytes, s>>>(feats, mask32, rays_d, p, grad_heads, grad_feats, grad_rays_d, g, N, S, num_tiles, level_major ? (long long)N : 0ll, ray_valid, slot, heads_fwd, sample_live);
    SNRF_RETURN_LAUNCH("snrf_decoder_bwd");
}

}  // namespace

// ------------------------------- C ABI --------------------------------------
// 0 = plain bf16 operands (fastest), 1 = bf16x3 split operands in the forward GEMMs (default)
SNRF_API void snrf_decoder_set_precision(int split) { g_split = split ? 1 : 0; }

// params: HOST array of 16 DEVICE pointers in network.ShallowMLP state_dict order
SNRF_API int snrf_decoder_fwd(const float* feats, const float* mask32, const float* rays_d, const float* const* params,
                              float* heads_out, int N, int S, int level_major, const unsigned char* ray_valid, void* stream)
{
    SNRF_CHECK_ARG(N >= 0 && S > 0, "snrf_decoder_fwd: need N >= 0, S > 0 (N=%d S=%d)", N, S);
    SNRF_CHECK_ARG(params != nullptr, "snrf_decoder_fwd: params is required");
    if (N == 0) return 0;
    DecoderParams p{params[0], params[1], params[2], params[3], params[4], params[5], params[6], params[7],
                    params[8], params[9], params[10], params[11], params[12], params[13], params[14], params[15]};
    static bool configured = false;
    if (!configured) {
        int rc = set_smem(decoder_fwd_kernel<true>, fwd_smem<true>(), "snrf_decoder_fwd");
        if (rc == 0) rc = set_smem(decoder_fwd_kernel<false>, fwd_smem<false>(), "snrf_decoder_fwd");
        if (rc == 0) rc = set_smem(decoder_fwd4_kernel<true>, fwd4_smem<true>(), "snrf_decoder_fwd");
        if (rc == 0) rc = set_smem(decoder_fwd4_kernel<false>, fwd4_smem<false>(), "snrf_decoder_fwd");
        if (rc) return rc;
        configured = true;
    }
    const int num_tiles = snrf_div_up(N, kRows);
    const long long level_stride = level_major ? (long long)N : 0ll;
    cudaStream_t s = (cudaStream_t)stream;
    int grid = snrf_sm_count();                     // one 16-warp CTA per SM
    if (S >= kMinS4) {                              // four tiles in flight each (a tile spans at most kMaxRays4 rays)
        if (grid > (num_tiles + 3) / 4) grid = (num_tiles + 3) / 4;
        if (g_split)
            decoder_fwd4_kernel<true><<<grid, kThreadsDec, fwd4_smem<true>(), s>>>(feats, mask32, rays_d, p, heads_out, N, S, num_tiles, level_stride, ray_valid);
        else
            decoder_fwd4_kernel<false><<<grid, kThreadsDec, fwd4_smem<false>(), s>>>(feats, mask32, rays_d, p, heads_out, N, S, num_tiles, level_stride, ray_valid);
        SNRF_RETURN_LAUNCH("snrf_decoder_fwd");
    }
    if (grid > (num_tiles + 1) / 2) grid = (num_tiles + 1) / 2;   // two tiles in flight each
    if (g_split)
        decoder_fwd_kernel<true><<<grid, kThreadsDec, fwd_smem<true>(), s>>>(feats, mask32, rays_d, p, heads_out, N, S, num_tiles, level_stride, ray_valid);
    else
        decoder_fwd_kernel<false><<<grid, kThreadsDec, fwd_smem<false>(), s>>>(feats, mask32, rays_d, p, heads_out, N, S, num_tiles, level_stride, ray_valid);
    SNRF_RETURN_LAUNCH("snrf_decoder_fwd");
}

// Backward of snrf_decoder_fwd.  heads_fwd: the [N,10] output of the forward (required: the backward takes the head
// activations from it instead of recomputing the last layers).  grad_heads[N,10] (same column order as heads) ->
// grad_feats[N,32] (WRITTEN), grad_rays_d[R,3] (ACCUMULATED; may be NULL: the view direction
// only enters through the SH encoding), grad_params = HOST array of 16 DEVICE pointers,
// same order and shapes as params (ACCUMULATED).
SNRF_API int snrf_decoder_bwd(const float* feats, const float* mask32, const float* rays_d, const float* const* params,
                              const float* grad_heads, float* grad_feats, float* grad_rays_d, float* const* grad_params,
                              int N, int S, int level_major, const unsigned char* ray_valid, const float* heads_fwd, void* stream)
{
    return decoder_bwd(feats, mask32, rays_d, params, grad_heads, grad_feats, grad_rays_d, grad_params, N, S, level_major, ray_valid,
                       heads_fwd, nullptr, stream);
}

// snrf_decoder_bwd with the per-sample early-ray-termination flags of snrf_composite_fwd_ert (sample_live [N], may be NULL):
// dead samples are treated like the samples of masked-out rays -- tiles without a live sample are skipped, grad_feats rows of
// dead samples are left unwritten.
SNRF_API int snrf_decoder_bwd_ert(const float* feats, const float* mask32, const float* rays_d, const float* const* params,
                                  const float* grad_heads, float* grad_feats, float* grad_rays_d, float* const* grad_params,
                                  int N, int S, int level_major, const unsigned char* ray_valid, const float* heads_fwd,
                                  const unsigned char* sample_live, void* stream)
{
    return decoder_bwd(feats, mask32, rays_d, params, grad_heads, grad_feats, grad_rays_d, grad_params, N, S, level_major, ray_valid,
                       heads_fwd, sample_live, stream);
}
