// Shared device code of the tensor-core decoder kernels (decoder.cu: training forward / backward,
// infer.cu: the render-side fused encode + decoder): shared-memory plan, weight staging, the
// per-tile forward pass.  See decoder.cu for the design notes.
#pragma once
#include "common.cuh"
#include "umma.cuh"

namespace dec {

constexpr int kRows = 128;                 // samples per tile
constexpr int kTile = kRows * 128;         // bytes of one operand tile (128 rows x 64 bf16)
constexpr float kGaussLog2 = -50.0f * 1.4426950408889634f;   // exp(-v^2/0.02) = exp2(v^2 * kGaussLog2)
// Operand format.  Everything the tensor core reads is a 16-bit hi part + a 16-bit lo part of the same format.
// Round 1 used bf16 (kOpBf16 = 1): 16 mantissa bits for the compensated products, but the weight-gradient GEMMs can
// only read the hi part of the ACTIVATIONS (their lo tiles are recycled by then), i.e. 8 bits -- that rounding,
// relative to the sum of magnitudes of the per-sample terms, was the measured source of the 0.07 dB end-to-end
// PSNR deficit (DESIGN 6).  fp16 activations against bf16 gradients / weights are not an option: tcgen05.mma
// kind::f16 with a_format != b_format faults on sm_100a (tried in round 1).  So EVERY operand is fp16 now
// (kOpBf16 = 0): hi parts carry 11 bits (8x less rounding where only hi is read), hi + lo 22 bits.  fp16's range is
// handled explicitly: conversions saturate (never inf), and the backward scales the incoming gradient by a power of two
// taken from its largest magnitude (snrf_decoder_bwd: max |grad_heads| -> [0.5, 1)), un-scaling every output exactly.
constexpr int kOpBf16 = 0;
constexpr int kActBf16 = kOpBf16;
constexpr float kInvSH0 = kOpBf16 ? 1.0f / 0.28125f : 1.0f / 0.281982421875f;   // 1 / round(0.28209479): the SH_0 column doubles as the ones column

// parameter tensors in network.ShallowMLP state_dict order (weight, bias per Linear)
struct DecoderParams {
    const float *W1, *b1, *W2, *b2, *Ws, *bs, *Wd, *bd, *Wt, *bt, *W3, *b3, *W4, *b4, *W5, *b5;
    int flat;     // 0: W[out, in] row-major (nn.Linear); 1: W^T flattened input-major (the renderer's flat layout)
};
// The renderer's flat parameter vector (13 994 floats per tile, hashgrid/include/decoder.h:48-67,
// rendering.py:101-113): for each Linear in state_dict order, bias[out] then W^T [in][out].
__host__ __device__ inline DecoderParams flat_params(const float* p)
{
    DecoderParams d;
    d.b1 = p;         d.W1 = p + 64;            // 32 -> 64
    d.b2 = p + 2112;  d.W2 = p + 2112 + 64;     // 64 -> 64
    d.bs = p + 6272;  d.Ws = p + 6272 + 1;      // 32 -> 1
    d.bd = p + 6305;  d.Wd = p + 6305 + 3;      // 32 -> 3
    d.bt = p + 6404;  d.Wt = p + 6404 + 3;      // 32 -> 3
    d.b3 = p + 6503;  d.W3 = p + 6503 + 64;     // 48 -> 64
    d.b4 = p + 9639;  d.W4 = p + 9639 + 64;     // 64 -> 64
    d.b5 = p + 13799; d.W5 = p + 13799 + 3;     // 64 -> 3   (ends at 13994)
    d.flat = 1;
    return d;
}
struct DecoderGrads {
    float *W1, *b1, *W2, *b2, *Ws, *bs, *Wd, *bd, *Wt, *bt, *W3, *b3, *W4, *b4, *W5, *b5;
};

// ---- shared-memory plan (byte offsets from the 1024-aligned base)
// weight tiles: W1 [64 rows: cols 0..31 hi | cols 32..63 lo], W2, W3 (48 cols used: 32 H + 16 SH),
// W4 [64 x 64], Wh [16 rows = sigma, diffuse3, tint3: cols 0..31 hi | 32..63 lo], W5 [16 rows, 3 used];
// in SPLIT mode W2, W3, W4, W5 have a second tile holding their lo parts.
constexpr int oW1 = 0, oW2 = 8192, oW3 = 16384, oW4 = 24576, oWh = 32768, oW5 = 34816;
constexpr int oW2l = 36864, oW3l = 45056, oW4l = 53248, oW5l = 61440;
template <bool SPLIT> constexpr int weights_end() { return SPLIT ? 63488 : 36864; }
// biases (fp32): b1[64] b2[64] bh[16] b3[64] b4[64] b5[16]; then mask[32], small bias grads[16]
constexpr int nB = 64 + 64 + 16 + 64 + 64 + 16;
constexpr int oB1 = 0, oB2 = 64, oBh = 128, oB3 = 144, oB4 = 208, oB5 = 272;
template <bool SPLIT> constexpr int off_bias() { return weights_end<SPLIT>(); }
template <bool SPLIT> constexpr int off_mask() { return off_bias<SPLIT>() + nB * 4; }
template <bool SPLIT> constexpr int off_small() { return off_mask<SPLIT>() + 128; }
template <bool SPLIT> constexpr int off_tiles() { return ((off_small<SPLIT>() + 64 + 1023) / 1024) * 1024; }
template <bool SPLIT> constexpr int fwd_tiles() { return SPLIT ? 5 : 3; }     // operand tiles of one in-flight forward tile
template <bool SPLIT> constexpr int fwd_smem() { return off_tiles<SPLIT>() + 2 * fwd_tiles<SPLIT>() * kTile + 1024; }   // two tiles in flight

// TMEM columns of the working accumulators
constexpr int cDa = 0, cDb = 64, cDh = 128;

__device__ __forceinline__ float gauss_act(float v) { return exp2f(v * v * kGaussLog2); }
__device__ __forceinline__ float sigmoidf(float v) { return 1.0f / (1.0f + __expf(-v)); }
// torch.nn.Softplus(beta=1, threshold=20)
__device__ __forceinline__ float softplusf(float v) { return v > 20.0f ? v : log1pf(__expf(v)); }

// Degree-3 real spherical harmonics of a unit vector in the order of network.py:38-77.
__device__ __forceinline__ void sh16(float x, float y, float z, float* o)
{
    const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
    o[0] = 0.28209479177387814f;
    o[1] = 0.4886025119029199f * y; o[2] = 0.4886025119029199f * z; o[3] = 0.4886025119029199f * x;
    o[4] = 1.0925484305920792f * xy; o[5] = -1.0925484305920792f * yz;
    o[6] = 0.31539156525252005f * (2.0f * zz - xx - yy);
    o[7] = -1.0925484305920792f * xz; o[8] = 0.5462742152960396f * (xx - yy);
    o[9] = -0.5900435899266435f * y * (3.0f * xx - yy); o[10] = 2.890611442640554f * xy * z;
    o[11] = -0.4570457994644658f * y * (4.0f * zz - xx - yy);
    o[12] = 0.3731763325901154f * z * (2.0f * zz - 3.0f * xx - 3.0f * yy);
    o[13] = -0.4570457994644658f * x * (4.0f * zz - xx - yy);
    o[14] = 1.445305721320277f * z * (xx - yy); o[15] = -0.5900435899266435f * x * (xx - 3.0f * yy);
}

__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
// round to the operand format / store 8 values of a tile row in it
__device__ __forceinline__ float op_round(float v) { return kOpBf16 ? bf16_round(v) : __half2float(__float2half_rn(v)); }
__device__ __forceinline__ void op_tile_store8(unsigned char* tile, int row, int chunk, const float* v)
{
    if constexpr (kOpBf16 != 0) umma::tile_store8(tile, row, chunk, v);
    else umma::tile_store8_f16(tile, row, chunk, v);
}

// store 8 values as the hi tile chunk and (SPLIT) their bf16 residuals as the lo tile chunk.
// The packed hi words serve both the store and the residual (hi as float = the 16 bits shifted up): 4 + 4 packing
// conversions per 8 values and no scalar float->bf16 round trips -- those run on the 16-lane XU pipe, which ncu
// showed saturated (profiles/r1c_top_kernels_full.md) when the residuals were formed with one conversion each.
template <bool SPLIT>
__device__ __forceinline__ void store8_hl(unsigned char* Thi, int chi, unsigned char* Tlo, int clo, int row, const float* v)
{
    uint32_t h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = umma::pack_bf16(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(Thi + umma::tile_chunk_off(row, chi)) = make_uint4(h[0], h[1], h[2], h[3]);
    if (SPLIT) {
        uint32_t l[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            l[i] = umma::pack_bf16(v[2 * i] - __uint_as_float(h[i] << 16), v[2 * i + 1] - __uint_as_float(h[i] & 0xffff0000u));
        *reinterpret_cast<uint4*>(Tlo + umma::tile_chunk_off(row, clo)) = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// the same in the operand format (fp16 hi / lo unless kOpBf16)
template <bool SPLIT>
__device__ __forceinline__ void store8_act(unsigned char* Thi, int chi, unsigned char* Tlo, int clo, int row, const float* v)
{
    if constexpr (kActBf16 != 0) {
        store8_hl<SPLIT>(Thi, chi, Tlo, clo, row, v);
    } else {
        uint32_t h[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) h[i] = umma::pack_f16(v[2 * i], v[2 * i + 1]);
        *reinterpret_cast<uint4*>(Thi + umma::tile_chunk_off(row, chi)) = make_uint4(h[0], h[1], h[2], h[3]);
        if (SPLIT) {
            uint32_t l[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h[i]));
                l[i] = umma::pack_f16(v[2 * i] - f.x, v[2 * i + 1] - f.y);
            }
            *reinterpret_cast<uint4*>(Tlo + umma::tile_chunk_off(row, clo)) = make_uint4(l[0], l[1], l[2], l[3]);
        }
    }
}

// W[out, in] (row-major f32, nn.Linear layout) -> rows [row0, row0+out) of an operand tile: hi part in
// columns [0, in), and in SPLIT mode the lo part either in columns [32, 32+in) of the same tile
// (lo_tile == tile, needs in <= 32) or in columns [0, in) of `lo_tile`.
template <bool SPLIT>
__device__ void stage_weight(unsigned char* tile, unsigned char* lo_tile, int row0, const float* __restrict__ W, int out,
                             int in, int flat, int tid, int nthreads)
{
    const int rs = flat ? 1 : in, cs = flat ? out : 1;      // element (r, col) at W[r * rs + col * cs]
    const bool packed = (lo_tile == tile);
    for (int t = tid; t < out * 8; t += nthreads) {
        const int r = t >> 3, c = t & 7;
        float hi[8], lo[8];
        const int src_c = (SPLIT && packed && c >= 4) ? c - 4 : c;     // packed lo chunks mirror chunks 0..3
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int col = src_c * 8 + j;
            const float w = col < in ? W[r * rs + col * cs] : 0.0f;
            hi[j] = w;
            lo[j] = w - op_round(w);
        }
        if (SPLIT && packed) {
            op_tile_store8(tile, row0 + r, c, c >= 4 ? lo : hi);
        } else {
            op_tile_store8(tile, row0 + r, c, hi);
            if (SPLIT) op_tile_store8(lo_tile, row0 + r, c, lo);
        }
    }
}
__device__ inline void zero_tile_rows(unsigned char* tile, int rows, int tid, int nthreads)
{
    for (int t = tid; t < rows * 8; t += nthreads) umma::tile_zero8(tile, t >> 3, t & 7);
}

template <bool SPLIT>
__device__ void stage_all_weights(unsigned char* smem, const DecoderParams& p, const float* __restrict__ mask32, int tid, int nthreads)
{
    zero_tile_rows(smem + oWh, 16, tid, nthreads);
    zero_tile_rows(smem + oW5, 16, tid, nthreads);
    if (SPLIT) zero_tile_rows(smem + oW5l, 16, tid, nthreads);
    __syncthreads();
    stage_weight<SPLIT>(smem + oW1, smem + oW1, 0, p.W1, 64, 32, p.flat, tid, nthreads);
    stage_weight<SPLIT>(smem + oW2, smem + oW2l, 0, p.W2, 64, 64, p.flat, tid, nthreads);
    stage_weight<SPLIT>(smem + oW3, smem + oW3l, 0, p.W3, 64, 48, p.flat, tid, nthreads);
    stage_weight<SPLIT>(smem + oW4, smem + oW4l, 0, p.W4, 64, 64, p.flat, tid, nthreads);
    stage_weight<SPLIT>(smem + oW5, smem + oW5l, 0, p.W5, 3, 64, p.flat, tid, nthreads);
    stage_weight<SPLIT>(smem + oWh, smem + oWh, 0, p.Ws, 1, 32, p.flat, tid, nthreads);
    stage_weight<SPLIT>(smem + oWh, smem + oWh, 1, p.Wd, 3, 32, p.flat, tid, nthreads);
    stage_weight<SPLIT>(smem + oWh, smem + oWh, 4, p.Wt, 3, 32, p.flat, tid, nthreads);
    float* b = reinterpret_cast<float*>(smem + off_bias<SPLIT>());
    for (int i = tid; i < nB; i += nthreads) {
        float v = 0.0f;
        if (i < 64) v = p.b1[i];
        else if (i < 128) v = p.b2[i - 64];
        else if (i < 144) { const int j = i - 128; v = j == 0 ? p.bs[0] : (j < 4 ? p.bd[j - 1] : (j < 7 ? p.bt[j - 4] : 0.0f)); }
        else if (i < 208) v = p.b3[i - 144];
        else if (i < 272) v = p.b4[i - 208];
        else { const int j = i - 272; v = j < 3 ? p.b5[j] : 0.0f; }
        b[i] = v;
    }
    float* m = reinterpret_cast<float*>(smem + off_mask<SPLIT>());
    for (int i = tid; i < 32; i += nthreads) m[i] = mask32 ? mask32[i] : 1.0f;
    float* sg = reinterpret_cast<float*>(smem + off_small<SPLIT>());
    for (int i = tid; i < 16; i += nthreads) sg[i] = 0.0f;
}

// Forward GEMM D (+)= A W^T over `nk` k-steps, issued by one thread.  A = (a_hi tile from k-step
// a_hi_k, a_lo tile from a_lo_k), W likewise; in SPLIT mode three MMAs per k-step.
template <bool SPLIT>
__device__ __forceinline__ void fwd_gemm(uint32_t d, uint32_t a_hi, int a_hi_k, uint32_t a_lo, int a_lo_k, uint32_t w_hi,
                                         int w_hi_k, uint32_t w_lo, int w_lo_k, int nk, uint32_t idesc, bool accumulate)
{
    for (int k = 0; k < nk; ++k)
        umma::mma_bf16(d, umma::desc_kmajor(a_hi, a_hi_k + k), umma::desc_kmajor(w_hi, w_hi_k + k), idesc, accumulate || k > 0);
    if (SPLIT) {
        for (int k = 0; k < nk; ++k)
            umma::mma_bf16(d, umma::desc_kmajor(a_lo, a_lo_k + k), umma::desc_kmajor(w_hi, w_hi_k + k), idesc, 1);
        for (int k = 0; k < nk; ++k)
            umma::mma_bf16(d, umma::desc_kmajor(a_hi, a_hi_k + k), umma::desc_kmajor(w_lo, w_lo_k + k), idesc, 1);
    }
}

// The tiles one forward pass writes (a1 and a3 may share a tile, H and a4 likewise).
struct Tiles {
    unsigned char *A0, *a1, *H, *a3, *a4, *LOa, *LOb;
};

// Thread layout of the two-tile decoder kernels: kThreadsDec = 512 threads = 16 warps per CTA, TWO tiles in flight per CTA
// (NCG = 2).  group = warp >> 3 owns a tile (own operand tiles, TMEM columns, mbarrier and named barrier); thread (row, cg),
// row = 32 (warp & 3) + lane is the sample / TMEM lane (a warp can only read the TMEM lane quadrant warp % 4), the group's
// 8 warps form 2 column groups cg of 32 columns.  While one group waits for its MMAs the other runs its epilogue (and, in
// the inference kernel, its table gathers).  Four warps per scheduler hide the latency a one-thread-per-row layout leaves
// exposed.
constexpr int kThreadsDec = 512;
constexpr int kTmemGroup = 160;           // TMEM columns of one in-flight forward tile (cDa, cDb, cDh = 144, padded)

__device__ __forceinline__ void bar_sync(uint32_t id, uint32_t nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// barrier + OR-reduction of a predicate over the threads of a named barrier (group-scoped __syncthreads_or)
__device__ __forceinline__ bool bar_or(uint32_t id, uint32_t nthreads, bool pred)
{
    uint32_t r;
    asm volatile(
        "{\n.reg .pred p, q;\nsetp.ne.u32 q, %1, 0;\nbar.red.or.pred p, %2, %3, q;\nselp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(r)
        : "r"((uint32_t)pred), "r"(id), "r"(nthreads)
        : "memory");
    return r != 0;
}

// Per-thread context shared by the forward stages
template <bool SPLIT, int NCG>
struct Ctx {
    static constexpr int W = 64 / NCG;          // accumulator columns per thread in a 64-wide layer
    unsigned char* smem;
    uint64_t* bar;
    uint32_t tmem, lane_addr, phase, bar_id, nthr;
    int tid, row, cg, group;
    bool leader_warp;                           // (warp-uniform) this warp holds the thread that issues this group's MMAs
    const float* bias;
    const float* mask;
    // `bars`: one mbarrier per group; `tmem_base`: the CTA's TMEM allocation
    __device__ __forceinline__ void init(unsigned char* smem_, uint64_t* bars, uint32_t tmem_base)
    {
        smem = smem_; phase = 0;
        tid = threadIdx.x;
        const int warp = tid >> 5;
        row = 32 * (warp & 3) + (tid & 31);
        group = warp >> 3; cg = (warp >> 2) & 1; nthr = kThreadsDec / 2;
        bar = bars + group;
        bar_id = 1 + group;
        leader_warp = umma::warp_uniform() == group * (kThreadsDec / 64);
        tmem = tmem_base + group * kTmemGroup;
        lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
        bias = reinterpret_cast<const float*>(smem + off_bias<SPLIT>());
        mask = reinterpret_cast<const float*>(smem + off_mask<SPLIT>());
    }
    __device__ __forceinline__ bool leader() const { return leader_warp && umma::elect_one(); }
    __device__ __forceinline__ void sync() { bar_sync(bar_id, nthr); }
    __device__ __forceinline__ bool any(bool pred) { return bar_or(bar_id, nthr, pred); }
    __device__ __forceinline__ void sync_operands()
    {   // my shared-memory stores and TMEM loads are done -> the next MMAs may run
        umma::fence_async_smem();
        umma::tc_fence_before();
        bar_sync(bar_id, nthr);
        umma::tc_fence_after();
    }
    __device__ __forceinline__ void wait_mma()
    {
        umma::mbar_wait(bar, phase);
        phase ^= 1u;
        umma::tc_fence_after();
    }
    // this thread's W accumulator columns [W cg, W cg + W) of the 64-wide accumulator at `col`
    __device__ __forceinline__ void load_cols(int col, float* v)
    {
        umma::tmem_ld32(tmem + col + lane_addr + 32 * cg, v);
        umma::tc_wait_ld();
    }
};

// Operand row of one sample: A0 = [x_hi (0..31) | SH_hi (32..47) | SH_lo (48..63)], LOb = [x_lo (0..31)].
// Thread (row, cg) stores its 32 / NCG (already masked) features x (chunks (4 / NCG) cg ...) and SH chunk cg
// (sh8 = that chunk's 8 values).
template <bool SPLIT, int NCG>
__device__ __forceinline__ void store_input_row(const Tiles& T, int row, int cg, const float* x, const float* sh8)
{
    constexpr int XC = 4 / NCG;
#pragma unroll
    for (int q = 0; q < XC; ++q) store8_act<SPLIT>(T.A0, XC * cg + q, T.LOb, XC * cg + q, row, x + 8 * q);
    store8_act<SPLIT>(T.A0, 4 + cg, T.A0, 6 + cg, row, sh8);
    if (!SPLIT) umma::tile_zero8(T.A0, row, 6 + cg);
}

// The decoder layers of one tile up to (and including) the L5 GEMM, from operand rows already in
// A0 / LOb.  Writes the operand tiles; the threads with cg == 0 return sigma/diffuse/tint activated in
// head[0..6] (torch semantics) and their pre-activations in zh[0..6]; the specular pre-activations are
// left in TMEM columns cDh..cDh+2.
template <bool SPLIT, int NCG>
__device__ __forceinline__ void forward_layers(Ctx<SPLIT, NCG>& c, const Tiles& T, float* head, float* zh)
{
    constexpr int W = 64 / NCG, CH = W / 8;
    unsigned char* smem = c.smem;
    const int row = c.row, cg = c.cg;
    const uint32_t tmem = c.tmem, lane_addr = c.lane_addr;
    const float* bias = c.bias;
    const uint32_t aA0 = umma::smem_u32(T.A0), aa1 = umma::smem_u32(T.a1), aH = umma::smem_u32(T.H), aa3 = umma::smem_u32(T.a3),
                   aa4 = umma::smem_u32(T.a4), aLOa = umma::smem_u32(T.LOa), aLOb = umma::smem_u32(T.LOb);
    const uint32_t aW1 = umma::smem_u32(smem + oW1), aW2 = umma::smem_u32(smem + oW2), aW3 = umma::smem_u32(smem + oW3),
                   aW4 = umma::smem_u32(smem + oW4), aWh = umma::smem_u32(smem + oWh), aW5 = umma::smem_u32(smem + oW5),
                   aW2l = umma::smem_u32(smem + oW2l), aW3l = umma::smem_u32(smem + oW3l), aW4l = umma::smem_u32(smem + oW4l),
                   aW5l = umma::smem_u32(smem + oW5l);
    // forward GEMMs: A = activations, B = weights, both K-major, both in the operand format
    constexpr uint32_t id64 = umma::idesc_f16(128, 64, 0, 0, kOpBf16, kOpBf16), id16 = umma::idesc_f16(128, 16, 0, 0, kOpBf16, kOpBf16);

    c.sync_operands();
    // ---- L1: Da = x W1^T (K = 32)
    if (c.leader()) {
        fwd_gemm<SPLIT>(tmem + cDa, aA0, 0, aLOb, 0, aW1, 0, aW1, 2, 2, id64, false);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
    float v[W];
    // Gaussian layer epilogue on this thread's W columns: a = exp(-50 z^2) -> (Ta, lo in Tlo)
    auto gauss_epilogue = [&](int col, int boff, unsigned char* Ta, unsigned char* Tlo) {
        c.load_cols(col, v);
#pragma unroll
        for (int j = 0; j < W; ++j) v[j] = gauss_act(v[j] + bias[boff + W * cg + j]);
#pragma unroll
        for (int q = 0; q < CH; ++q) store8_act<SPLIT>(Ta, CH * cg + q, Tlo, CH * cg + q, row, v + 8 * q);
    };
    gauss_epilogue(cDa, oB1, T.a1, T.LOa);
    c.sync_operands();
    // ---- L2: Db = h1 W2^T (K = 64)
    if (c.leader()) {
        fwd_gemm<SPLIT>(tmem + cDb, aa1, 0, aLOa, 0, aW2, 0, aW2l, 0, 4, id64, false);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
    c.load_cols(cDb, v);
#pragma unroll
    for (int j = 0; j < W; ++j) v[j] += bias[oB2 + W * cg + j];
#pragma unroll
    for (int q = 0; q < CH; ++q) store8_act<SPLIT>(T.H, CH * cg + q, T.LOb, CH * cg + q, row, v + 8 * q);
    c.sync_operands();
    // ---- heads: Dh = H[0:32] Wh^T (K = 32, N = 16);   L3: Da = [H[32:64] | SH] W3^T (K = 48)
    if (c.leader()) {
        fwd_gemm<SPLIT>(tmem + cDh, aH, 0, aLOb, 0, aWh, 0, aWh, 2, 2, id16, false);
        fwd_gemm<SPLIT>(tmem + cDa, aH, 2, aLOb, 2, aW3, 0, aW3l, 0, 2, id64, false);
        fwd_gemm<SPLIT>(tmem + cDa, aA0, 2, aA0, 3, aW3, 2, aW3l, 2, 1, id64, true);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
    if (cg == 0) {
        float z[16];
        umma::tmem_ld16(tmem + cDh + lane_addr, z);
        umma::tc_wait_ld();
#pragma unroll
        for (int j = 0; j < 7; ++j) zh[j] = z[j] + bias[oBh + j];
        head[0] = softplusf(zh[0]);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            head[4 + j] = sigmoidf(zh[1 + j]);     // diffuse
            head[1 + j] = sigmoidf(zh[4 + j]);     // tint
        }
    }
    gauss_epilogue(cDa, oB3, T.a3, T.LOa);
    c.sync_operands();
    // ---- L4: Db = a3 W4^T (K = 64)
    if (c.leader()) {
        fwd_gemm<SPLIT>(tmem + cDb, aa3, 0, aLOa, 0, aW4, 0, aW4l, 0, 4, id64, false);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
    gauss_epilogue(cDb, oB4, T.a4, T.LOb);
    c.sync_operands();
    // ---- L5: Dh = a4 W5^T (K = 64, N = 16)
    if (c.leader()) {
        fwd_gemm<SPLIT>(tmem + cDh, aa4, 0, aLOb, 0, aW5, 0, aW5l, 0, 4, id16, false);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
}

// Training-side input: features from HBM times the level mask, SH of d / (|d| + 1e-8) (network.py:172-190).
// feats: [N,32] row-major (level_stride = 0) or level-major [16][N] float2 (level_stride = N).
// d / dn (the ray direction and its norm) are returned to the threads that hold an SH chunk.
template <bool SPLIT, int NCG>
__device__ __forceinline__ void forward_tile(Ctx<SPLIT, NCG>& c, const Tiles& T, const float* __restrict__ feats,
                                             const float* __restrict__ rays_d, int n, bool live, int S, float* head, float* zh,
                                             f3& d, float& dn, long long level_stride)
{
    constexpr int NX = 32 / NCG;                // features per thread
    const float* mask = c.mask;
    const int cg = c.cg;
    float x[NX], sh[16];
#pragma unroll
    for (int j = 0; j < NX; ++j) x[j] = 0.0f;
#pragma unroll
    for (int j = 0; j < 16; ++j) sh[j] = 0.0f;
    if (live) {
        if (level_stride == 0) {
#pragma unroll
            for (int q = 0; q < NX / 4; ++q) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(feats + (size_t)n * 32 + NX * cg + 4 * q));
                x[4 * q] = a.x; x[4 * q + 1] = a.y; x[4 * q + 2] = a.z; x[4 * q + 3] = a.w;
            }
        } else {
            const float2* f2 = reinterpret_cast<const float2*>(feats) + n;
#pragma unroll
            for (int l = 0; l < NX / 2; ++l) {
                const float2 a = __ldg(f2 + (size_t)((NX / 2) * cg + l) * level_stride);
                x[2 * l] = a.x; x[2 * l + 1] = a.y;
            }
        }
#pragma unroll
        for (int j = 0; j < NX; ++j) x[j] *= mask[NX * cg + j];
        d = ld3(rays_d + 3 * (size_t)(n / S));
        dn = sqrtf(d.x * d.x + d.y * d.y + d.z * d.z);
        const float inv = 1.0f / (dn + 1e-8f);
        sh16(d.x * inv, d.y * inv, d.z * inv, sh);
    }
    store_input_row<SPLIT, NCG>(T, c.row, cg, x, sh + 8 * (cg & 1));
    forward_layers<SPLIT, NCG>(c, T, head, zh);
}

// =====================================================================================================================
// Forward with FOUR tiles in flight per CTA (training forward; the render-side single-tile decode pass).
//
// The two-tile forward above is bound by the dependent chain of its five stages (operands -> MMAs -> commit -> TMEM load
// -> epilogue): 36 % of the issue slots busy, 13 % tensor pipe (profiles/r2d_encode_fwd_decoder_full.md), two tiles are
// too few to fill the gaps, and five 16 KB operand tiles per in-flight tile leave no room for more.  Two observations
// shrink an in-flight tile to TWO operand tiles (hi, lo):
//   * every MMA of a stage has completed before its epilogue starts (the commit was waited for), and the epilogue reads its
//     inputs from TMEM, not from shared memory: a layer's output can overwrite the layer's input tiles IN PLACE;
//   * the SH view encoding is a function of the RAY: its contribution W3[:, 32:48] SH(d) to the pre-activation of layer 3
//     is one 64-vector per ray, computed once per ray in fp32 on the CUDA cores and added like a bias in the epilogue --
//     no SH columns in any operand tile, three MMAs less per tile, and that term exact instead of split-compensated.
// One group = 4 consecutive warps = 128 threads = one thread per sample row (all four TMEM lane quadrants), 64
// accumulator columns per thread, handled as two halves of 32.  TMEM: one 64-column accumulator + 16 head columns per
// group.  Shared memory: weights (as above) + 4 KB W3_sh (fp32, transposed) + 4 x (32 KB tiles + 2.5 KB ray vectors).
// Needs S >= kMinS4 (a 128-sample tile then spans at most kMaxRays4 rays); smaller S keeps the two-tile kernel.
constexpr int kGroups4 = 4, kGroupThreads4 = 128, kTmemGroup4 = 128;
constexpr int kMinS4 = 16, kMaxRays4 = 128 / kMinS4 + 1;
constexpr int c4D = 0, c4Dh = 64;
template <bool SPLIT> constexpr int off_w3sh() { return off_small<SPLIT>() + 64; }                       // float [16][64]
template <bool SPLIT> constexpr int off_raybias4() { return off_w3sh<SPLIT>() + 16 * 64 * 4; }           // float [4][kMaxRays4][64]
template <bool SPLIT> constexpr int off_tiles4() { return ((off_raybias4<SPLIT>() + kGroups4 * kMaxRays4 * 64 * 4 + 1023) / 1024) * 1024; }
template <bool SPLIT> constexpr int fwd4_smem() { return off_tiles4<SPLIT>() + kGroups4 * 2 * kTile + 1024; }

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

struct Ctx4 {
    uint64_t* bar;
    uint32_t tmem, lane_addr, phase, bar_id;
    int tid, row, group, gtid;
    bool leader_warp;
    __device__ __forceinline__ void init(uint64_t* bars, uint32_t tmem_base)
    {
        phase = 0;
        tid = threadIdx.x;
        const int warp = tid >> 5;
        group = warp >> 2;
        row = 32 * (warp & 3) + (tid & 31);
        gtid = tid - group * kGroupThreads4;
        bar = bars + group;
        bar_id = 1 + group;
        leader_warp = umma::warp_uniform() == 4 * group;
        tmem = tmem_base + group * kTmemGroup4;
        lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    }
    __device__ __forceinline__ bool leader() const { return leader_warp && umma::elect_one(); }
    __device__ __forceinline__ void sync() { bar_sync(bar_id, kGroupThreads4); }
    __device__ __forceinline__ bool any(bool pred) { return bar_or(bar_id, kGroupThreads4, pred); }
    __device__ __forceinline__ void sync_operands()
    {
        umma::fence_async_smem();
        umma::tc_fence_before();
        bar_sync(bar_id, kGroupThreads4);
        umma::tc_fence_after();
    }
    __device__ __forceinline__ void wait_mma()
    {
        umma::mbar_wait(bar, phase);
        phase ^= 1u;
        umma::tc_fence_after();
    }
};

// W3[:, 32:48] (the SH columns of the first directional layer) as fp32, transposed to [16][64]
__device__ inline void stage_w3sh(float* dst, const DecoderParams& p, int tid, int nthreads)
{
    for (int i = tid; i < 16 * 64; i += nthreads) {
        const int k = i >> 6, o = i & 63;                       // dst[k][o] = W3[o][32 + k]
        dst[i] = p.flat ? p.W3[(32 + k) * 64 + o] : p.W3[o * 48 + 32 + k];
    }
}

// element (r, c) of a Linear weight [out, in] in either parameter layout
__device__ __forceinline__ float w_at(const float* __restrict__ W, int r, int c, int out, int in, int flat)
{
    return flat ? W[c * out + r] : W[r * in + c];
}
// row h of the stacked heads matrix Wh [7 x 32] = (sigma, diffuse3, tint3)
__device__ __forceinline__ float wh_at(const DecoderParams& p, int h, int k)
{
    return h == 0 ? w_at(p.Ws, 0, k, 1, 32, p.flat) : (h < 4 ? w_at(p.Wd, h - 1, k, 3, 32, p.flat) : w_at(p.Wt, h - 4, k, 3, 32, p.flat));
}

// Composed weights of the FOLD forward, written over what stage_all_weights left (call after it; ends with the data in place
// but NOT synchronised: the caller's fence + __syncthreads() follows).  `scratch`: >= 48 KB of shared memory not in use yet
// (the operand-tile area).  W32 = W3[:, 0:32] W2[32:64, :] -> the W2 tiles; Wh2 = Wh W2[0:32, :] -> the Wh tile (hi) and
// rows 0..15 of the W3-lo tile (lo); b32 = W3[:, 0:32] b2[32:64] + b3 -> the b3 slot; bh2 = Wh b2[0:32] + bh -> the head slot.
template <bool SPLIT>
__device__ void stage_fold_weights4(unsigned char* smem, const DecoderParams& p, float* scratch, int tid, int nthreads)
{
    float* s32 = scratch;                 // [64][64]
    float* sh2 = scratch + 64 * 64;       // [7][64]
    // fp32 copies of the factors (row pitch 65 / 33: conflict-free): the 32-term sums below read shared memory, not L1 / L2
    float* sW2 = sh2 + 8 * 64;            // W2 [64][64]
    float* sW3a = sW2 + 64 * 65;          // W3[:, 0:32] [64][32]
    float* sWh = sW3a + 64 * 33;          // Wh [7][32]
    float* sb2 = sWh + 8 * 33;            // b2 [64]
    for (int i = tid; i < 64 * 64; i += nthreads) sW2[(i >> 6) * 65 + (i & 63)] = w_at(p.W2, i >> 6, i & 63, 64, 64, p.flat);
    for (int i = tid; i < 64 * 32; i += nthreads) sW3a[(i >> 5) * 33 + (i & 31)] = w_at(p.W3, i >> 5, i & 31, 64, 48, p.flat);
    for (int i = tid; i < 7 * 32; i += nthreads) sWh[(i >> 5) * 33 + (i & 31)] = wh_at(p, i >> 5, i & 31);
    for (int i = tid; i < 64; i += nthreads) sb2[i] = p.b2[i];
    __syncthreads();                      // (also: stage_all_weights' stores to the tiles overwritten below are complete)
    for (int i = tid; i < 64 * 64; i += nthreads) {
        const int o = i >> 6, j = i & 63;
        float acc = 0.0f;
#pragma unroll 8
        for (int k = 0; k < 32; ++k) acc += sW3a[o * 33 + k] * sW2[(32 + k) * 65 + j];
        s32[i] = acc;
    }
    for (int i = tid; i < 7 * 64; i += nthreads) {
        const int h = i >> 6, j = i & 63;
        float acc = 0.0f;
#pragma unroll 8
        for (int k = 0; k < 32; ++k) acc += sWh[h * 33 + k] * sW2[k * 65 + j];
        sh2[i] = acc;
    }
    float* b = reinterpret_cast<float*>(smem + off_bias<SPLIT>());
    for (int i = tid; i < 64 + 7; i += nthreads) {
        if (i < 64) {
            float v = p.b3[i];
            for (int k = 0; k < 32; ++k) v += sW3a[i * 33 + k] * sb2[32 + k];
            b[oB3 + i] = v;
        } else {
            const int h = i - 64;
            float v = h == 0 ? p.bs[0] : (h < 4 ? p.bd[h - 1] : p.bt[h - 4]);
            for (int k = 0; k < 32; ++k) v += sWh[h * 33 + k] * sb2[k];
            b[oBh + h] = v;
        }
    }
    zero_tile_rows(smem + oWh, 16, tid, nthreads);
    if (SPLIT) zero_tile_rows(smem + oW3l, 16, tid, nthreads);
    __syncthreads();
    stage_weight<SPLIT>(smem + oW2, smem + oW2l, 0, s32, 64, 64, 0, tid, nthreads);
    stage_weight<SPLIT>(smem + oWh, smem + oW3l, 0, sh2, 7, 64, 0, tid, nthreads);
}

// The layers of one tile, operands in place in (P, Q) = (hi, lo).  x (already masked) is this thread's whole input row;
// rb = this row's ray vector W3_sh SH(d) (64 floats in shared memory).  Returns sigma / diffuse / tint activated in
// head[0..6] and leaves the specular pre-activations in TMEM columns c4Dh .. c4Dh + 2 (after the last wait).
// Layer 2 (linear, no activation) is composed into its consumers when the weights are staged (stage_fold_weights4):
// the W2 tiles hold W32 = W3[:, 0:32] W2[32:64, :], the Wh tile / the first rows of the W3-lo tile hold Wh2 = Wh W2[0:32, :]
// (hi / lo), the b3 / head bias slots the composed biases -- z3 and the heads come straight from a1 in ONE stage, H is never
// formed: four dependent stages per tile instead of five, 12 MMAs and one 64-column epilogue less.
struct NoHook4 { __device__ __forceinline__ void operator()() const {} };
// under_l1(): called by every thread of the group right after the L1 MMAs have been issued -- work that is not needed before
// the z3 epilogue (the per-ray SH vectors rb) runs there instead of in front of the tile's first barrier.
template <bool SPLIT, class Hook = NoHook4>
__device__ __forceinline__ void forward_layers4(Ctx4& c, unsigned char* smem, unsigned char* P, unsigned char* Q, const float* x,
                                                const float* rb, float* head, float* zh, Hook under_l1 = Hook())
{
    const int row = c.row;
    const uint32_t tmem = c.tmem, lane_addr = c.lane_addr;
    const float* bias = reinterpret_cast<const float*>(smem + off_bias<SPLIT>());
    const uint32_t aP = umma::smem_u32(P), aQ = umma::smem_u32(Q);
    const uint32_t aW1 = umma::smem_u32(smem + oW1), aW2 = umma::smem_u32(smem + oW2), aW4 = umma::smem_u32(smem + oW4),
                   aWh = umma::smem_u32(smem + oWh), aW5 = umma::smem_u32(smem + oW5), aW2l = umma::smem_u32(smem + oW2l),
                   aW3l = umma::smem_u32(smem + oW3l), aW4l = umma::smem_u32(smem + oW4l), aW5l = umma::smem_u32(smem + oW5l);
    constexpr uint32_t id64 = umma::idesc_f16(128, 64, 0, 0, kOpBf16, kOpBf16), id16 = umma::idesc_f16(128, 16, 0, 0, kOpBf16, kOpBf16);
    // input row, packed: x_hi in columns 0..31 of P, x_lo in columns 32..63 of P
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        store8_act<SPLIT>(P, q, P, 4 + q, row, x + 8 * q);
        if (!SPLIT) umma::tile_zero8(P, row, 4 + q);
    }
    c.sync_operands();
    if (c.leader()) {          // L1: D = x W1^T (K = 32)
        fwd_gemm<SPLIT>(tmem + c4D, aP, 0, aP, 2, aW1, 0, aW1, 2, 2, id64, false);
        umma::mma_commit(c.bar);
    }
    under_l1();
    c.wait_mma();
    float v[32];
    // Gaussian epilogue of a 64-wide layer on this thread's row, 32 columns at a time: v = g(D + bias (+ extra)) -> (P, Q)
    auto epilogue = [&](int boff, const float* extra) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            umma::tmem_ld32(tmem + c4D + lane_addr + 32 * half, v);
            umma::tc_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                float z = v[j] + bias[boff + 32 * half + j];
                if (extra != nullptr) z += extra[32 * half + j];
                v[j] = gauss_act(z);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) store8_act<SPLIT>(P, 4 * half + q, Q, 4 * half + q, row, v + 8 * q);
        }
    };
    epilogue(oB1, nullptr);                                               // a1
    c.sync_operands();
    if (c.leader()) {          // heads: Dh = a1 Wh2^T (K = 64, N = 16);  z3: D = a1 W32^T (K = 64)
        fwd_gemm<SPLIT>(tmem + c4Dh, aP, 0, aQ, 0, aWh, 0, aW3l, 0, 4, id16, false);
        fwd_gemm<SPLIT>(tmem + c4D, aP, 0, aQ, 0, aW2, 0, aW2l, 0, 4, id64, false);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
    {
        float z[16];
        umma::tmem_ld16(tmem + c4Dh + lane_addr, z);
        umma::tc_wait_ld();
#pragma unroll
        for (int j = 0; j < 7; ++j) zh[j] = z[j] + bias[oBh + j];
        head[0] = softplusf(zh[0]);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            head[4 + j] = sigmoidf(zh[1 + j]);      // diffuse
            head[1 + j] = sigmoidf(zh[4 + j]);      // tint
        }
    }
    epilogue(oB3, rb);                                                    // a3 (+ the ray's SH term)
    c.sync_operands();
    if (c.leader()) {          // L4: D = a3 W4^T (K = 64)
        fwd_gemm<SPLIT>(tmem + c4D, aP, 0, aQ, 0, aW4, 0, aW4l, 0, 4, id64, false);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
    epilogue(oB4, nullptr);                                               // a4
    c.sync_operands();
    if (c.leader()) {          // L5: Dh = a4 W5^T (K = 64, N = 16)
        fwd_gemm<SPLIT>(tmem + c4Dh, aP, 0, aQ, 0, aW5, 0, aW5l, 0, 4, id16, false);
        umma::mma_commit(c.bar);
    }
    c.wait_mma();
}

// Ray vectors of one tile: rays [ray0, ray0 + nrays) -> rb[i][0..63] = W3_sh SH(unit(d_i)), by the group's 128 threads.
// unit(d) = d / (|d| + 1e-8) in training (network.py:172-176), d * rsqrt(d.d) in the renderer (decoder.h:201).
template <bool RENDER_NORM>
__device__ __forceinline__ void ray_vectors4(float* rb, const float* __restrict__ w3sh, const float* __restrict__ rays_d, int ray0,
                                             int nrays, int gtid)
{
    for (int i = gtid; i < nrays * 64; i += kGroupThreads4) {
        const int r = i >> 6, o = i & 63;
        const f3 d = ld3(rays_d + 3 * (size_t)(ray0 + r));
        const float inv = RENDER_NORM ? rsqrtf(d.x * d.x + d.y * d.y + d.z * d.z) : 1.0f / (sqrtf(d.x * d.x + d.y * d.y + d.z * d.z) + 1e-8f);
        float sh[16];
        sh16(d.x * inv, d.y * inv, d.z * inv, sh);
        float acc = 0.0f;
#pragma unroll
        for (int k = 0; k < 16; ++k) acc += w3sh[k * 64 + o] * sh[k];
        rb[r * 64 + o] = acc;
    }
}

}  // namespace dec
