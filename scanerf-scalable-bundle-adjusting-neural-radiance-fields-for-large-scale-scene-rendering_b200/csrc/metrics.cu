// Image-quality metrics of rendered views against ground truth: per-image MSE, mean SSIM and the number of
// pixels they are taken over, sm_100a.  No reference kernel: the reference scores its held-out views on the host
// (tile.py:810-864, rendering.py val mode) with tools/ssim.py.
//
// SSIM as the NeRF code of this lineage computes it (pytorch-ssim):
//   window   11 x 11, w[a][b] = g[a] g[b], g[i] = exp(-(i-5)^2 / 4.5) / sum_j exp(-(j-5)^2 / 4.5)  (sigma 1.5)
//   per channel, zero-padded correlation with padding 5 (F.conv2d(img, window, padding=5, groups=3)):
//     mu_x, mu_y, s_xx = E[x^2] - mu_x^2, s_yy = E[y^2] - mu_y^2, s_xy = E[xy] - mu_x mu_y
//   map      ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)),  C1 = 0.01^2, C2 = 0.03^2
// The mask does not change the local statistics: it only selects which map values and squared errors are averaged.
// Both means run over the masked pixels and the 3 channels; an empty mask gives NaN and a count of 0.
//
// One CTA per TILE_H x TILE_W output tile of one image: for each channel it stages the tile plus its 5-pixel halo of
// both images (zero outside the image), runs the window as a horizontal pass over the five moments into shared memory
// and a vertical pass in registers, and evaluates the map.  The moments and the map are accumulated in fp64: in fp32,
// E[x^2] - mu^2 loses ~1e-7 to cancellation, which against C2 = 9e-4 is a 1e-4 error of one map value.  Every CTA
// writes its three fp64 partial sums to the caller's scratch; a second kernel reduces them per image in a fixed order,
// so the same inputs give the same bits.  No allocation, no host synchronisation.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int TILE_W = 32, TILE_H = 16, R = 5, WIN = 2 * R + 1;
constexpr int SW = TILE_W + 2 * R, SH = TILE_H + 2 * R;   // staged region
constexpr int THREADS = 256;
constexpr int ROWS_PER_THREAD = TILE_H * TILE_W / THREADS;  // output pixels per thread, one column
constexpr double C1 = 0.01 * 0.01, C2 = 0.03 * 0.03;

struct Window {
    double g[WIN];
};

__device__ __forceinline__ float load_gt(const void* gt, int gt_is_u8, long long i)
{
    // u8: the value torch's gt.float() / 255 gives (IEEE division, no fast math in this build)
    return gt_is_u8 ? (float)static_cast<const unsigned char*>(gt)[i] / 255.0f : static_cast<const float*>(gt)[i];
}

__device__ __forceinline__ void block_sum3(double v[3], double (*red)[3])
{
    // fixed-order reduction: shuffle tree inside each warp, then warp 0 adds the warps in order
    for (int off = 16; off > 0; off >>= 1)
        for (int k = 0; k < 3; ++k) v[k] += __shfl_down_sync(0xffffffffu, v[k], off);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0)
        for (int k = 0; k < 3; ++k) red[warp][k] = v[k];
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 0; k < 3; ++k) v[k] = red[0][k];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
            for (int k = 0; k < 3; ++k) v[k] += red[w][k];
    }
}

// grid (tiles_x, tiles_y, N); partial[(n * tiles + tile) * 3 + {0,1,2}] = (sum of map values, sum of squared errors,
// masked pixel count) of that tile, all channels.
__global__ void __launch_bounds__(THREADS) ssim_tile_kernel(const float* __restrict__ pred, const void* __restrict__ gt, int gt_is_u8,
                                                            const unsigned char* __restrict__ mask, int H, int W, Window win,
                                                            double* __restrict__ partial)
{
    __shared__ float sx[SH][SW], sy[SH][SW];
    __shared__ double hm[5][SH][TILE_W];
    __shared__ double red[THREADS / 32][3];

    const int n = blockIdx.z, x0 = blockIdx.x * TILE_W, y0 = blockIdx.y * TILE_H;
    const long long img = (long long)n * H * W;
    const int col = threadIdx.x % TILE_W, row0 = threadIdx.x / TILE_W;
    constexpr int ROW_STEP = THREADS / TILE_W;

    bool use[ROWS_PER_THREAD];
    double cnt = 0.0;
#pragma unroll
    for (int r = 0; r < ROWS_PER_THREAD; ++r) {
        const int y = y0 + row0 + r * ROW_STEP, x = x0 + col;
        use[r] = y < H && x < W && (mask == nullptr || mask[img + (long long)y * W + x] != 0);
        cnt += use[r] ? 1.0 : 0.0;
    }
    double ssim_sum = 0.0, se_sum = 0.0;

    for (int c = 0; c < 3; ++c) {
        for (int i = threadIdx.x; i < SH * SW; i += THREADS) {
            const int ly = i / SW, lx = i % SW, y = y0 + ly - R, x = x0 + lx - R;
            float vx = 0.0f, vy = 0.0f;
            if (y >= 0 && y < H && x >= 0 && x < W) {
                const long long e = (img + (long long)y * W + x) * 3 + c;
                vx = pred[e];
                vy = load_gt(gt, gt_is_u8, e);
            }
            sx[ly][lx] = vx;
            sy[ly][lx] = vy;
        }
        __syncthreads();
        // horizontal pass: the five moments of every staged row at every output column
        for (int i = threadIdx.x; i < SH * TILE_W; i += THREADS) {
            const int ly = i / TILE_W, lx = i % TILE_W;
            double m[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int k = 0; k < WIN; ++k) {
                const double a = sx[ly][lx + k], b = sy[ly][lx + k], g = win.g[k];
                m[0] += g * a;
                m[1] += g * b;
                m[2] += g * (a * a);
                m[3] += g * (b * b);
                m[4] += g * (a * b);
            }
#pragma unroll
            for (int q = 0; q < 5; ++q) hm[q][ly][lx] = m[q];
        }
        __syncthreads();
        // vertical pass, map and squared error of this thread's output pixels
#pragma unroll
        for (int r = 0; r < ROWS_PER_THREAD; ++r) {
            const int ly = row0 + r * ROW_STEP;
            double m[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int k = 0; k < WIN; ++k) {
                const double g = win.g[k];
#pragma unroll
                for (int q = 0; q < 5; ++q) m[q] += g * hm[q][ly + k][col];
            }
            if (use[r]) {
                const double mx = m[0], my = m[1];
                const double sxx = m[2] - mx * mx, syy = m[3] - my * my, sxy = m[4] - mx * my;
                ssim_sum += ((2.0 * mx * my + C1) * (2.0 * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2));
                const double d = (double)sx[ly + R][col + R] - (double)sy[ly + R][col + R];
                se_sum += d * d;
            }
        }
        __syncthreads();   // the next channel overwrites sx / sy / hm
    }

    double v[3] = {ssim_sum, se_sum, cnt};
    block_sum3(v, red);
    if (threadIdx.x == 0) {
        const long long tiles = (long long)gridDim.x * gridDim.y;
        double* p = partial + ((long long)n * tiles + (long long)blockIdx.y * gridDim.x + blockIdx.x) * 3;
        p[0] = v[0];
        p[1] = v[1];
        p[2] = v[2];
    }
}

// one CTA per image: fixed-order sum of its tiles' partials -> MSE, mean SSIM, count
__global__ void __launch_bounds__(THREADS) ssim_reduce_kernel(const double* __restrict__ partial, int tiles, float* __restrict__ out_mse,
                                                              float* __restrict__ out_ssim, float* __restrict__ out_count)
{
    __shared__ double red[THREADS / 32][3];
    const int n = blockIdx.x;
    const double* p = partial + (long long)n * tiles * 3;
    double v[3] = {0.0, 0.0, 0.0};
    for (int t = threadIdx.x; t < tiles; t += THREADS)
        for (int k = 0; k < 3; ++k) v[k] += p[(long long)t * 3 + k];
    block_sum3(v, red);
    if (threadIdx.x == 0) {
        const double cnt = v[2];
        out_ssim[n] = cnt > 0.0 ? (float)(v[0] / (3.0 * cnt)) : NAN;
        out_mse[n] = cnt > 0.0 ? (float)(v[1] / (3.0 * cnt)) : NAN;
        out_count[n] = (float)cnt;
    }
}

Window make_window()
{
    Window w;
    double s = 0.0;
    for (int i = 0; i < WIN; ++i) s += (w.g[i] = exp(-(double)((i - R) * (i - R)) / 4.5));
    for (int i = 0; i < WIN; ++i) w.g[i] /= s;
    return w;
}

}  // namespace

SNRF_API int snrf_image_metrics(const float* pred, const void* gt, int gt_is_u8, const unsigned char* mask, int N, int H, int W,
                                float* out_mse, float* out_ssim, float* out_count, void* scratch, size_t scratch_bytes, void* stream)
{
    SNRF_CHECK_ARG(N >= 0 && H >= 0 && W >= 0, "snrf_image_metrics: negative size (N=%d H=%d W=%d)", N, H, W);
    if (N == 0) return 0;
    SNRF_CHECK_ARG(N <= 65535, "snrf_image_metrics: at most 65535 images per call (N=%d)", N);
    const int tx = snrf_div_up(W, TILE_W), ty = snrf_div_up(H, TILE_H);
    SNRF_CHECK_ARG(ty <= 65535 && (long long)tx * ty <= 0x7fffffffLL, "snrf_image_metrics: %d x %d is too large", H, W);
    const size_t need = (size_t)N * tx * ty * 3 * sizeof(double);
    SNRF_CHECK_ARG(scratch != nullptr || need == 0, "snrf_image_metrics: scratch is NULL");
    SNRF_CHECK_ARG(scratch_bytes >= need, "snrf_image_metrics: scratch holds %zu bytes, %zu needed", scratch_bytes, need);
    static const Window win = make_window();
    cudaStream_t s = (cudaStream_t)stream;
    if (tx > 0 && ty > 0)
        ssim_tile_kernel<<<dim3(tx, ty, N), THREADS, 0, s>>>(pred, gt, gt_is_u8, mask, H, W, win, (double*)scratch);
    ssim_reduce_kernel<<<N, THREADS, 0, s>>>((const double*)scratch, tx * ty, out_mse, out_ssim, out_count);
    SNRF_RETURN_LAUNCH("snrf_image_metrics");
}
