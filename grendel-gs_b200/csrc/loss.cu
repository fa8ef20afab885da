// Fused per-strip L1 + SSIM loss, forward and backward.
// Replaces the ~20 torch kernels (5 depthwise 11x11 F.conv2d + elementwise) of
// /root/reference/gaussian_renderer/loss_distribution.py:2536-2585 with utils/loss_utils.py:88-132:
//   Ll1  = sum |x - y|      / (3 H W)          (pixelwise_l1_with_mask, mask == all ones in the live path)
//   ssim = sum ssim_map(x,y) / (3 H W)          (11x11 Gaussian window sigma 1.5, ZERO padding at the strip
//                                               edges -- the live path exchanges no halo)
// with x = rendered strip rows [row0,row1) of the full (3,H,W) image, y = clamp(gt_u8/255, 0, 1).
// The window is applied separably (row pass then column pass) from shared memory, four outputs per thread from a
// 14-value sliding window in registers.
//
// HBM bound: forward reads 15 B and writes 36 B per pixel-channel triple (three derivative maps kept for
// the backward), backward reads 51 B and writes 12 B; no tensor-core shaped work.
//
// The same forward kernel, instantiated in a metrics mode (gs_metrics_batched), evaluates held-out views: per view and
// channel the fp64 sums of |x - y|, (x - y)^2 and ssim_map(x, y) over the counted rows, with x = clamp(image, 0, 1)
// (train_internal.py:471-478) or that image after the 8-bit PNG round trip of render.py:127-138 -> metrics.py:26-36.
// It reads 15 B per pixel-channel triple and writes only the 9 sums per view.
#include "common.cuh"

#define LS_TILE 32
#define LS_HALO 5
#define LS_IN (LS_TILE + 2 * LS_HALO)
#define LS_THREADS 256

__device__ __constant__ float c_gauss[11];
static unsigned long long g_gauss_ready = 0ull;  // bit d: window uploaded to device d's constant memory

static int ensure_gauss() {
    int dev = 0;
    GS_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 64 && ((g_gauss_ready >> dev) & 1ull)) return GS_OK;
    // utils/loss_utils.py:26-34: fp32 exp values normalised in fp32
    float g[11], s = 0.f;
    for (int k = 0; k < 11; k++) { g[k] = (float)exp(-((double)(k - 5) * (k - 5)) / (2.0 * 1.5 * 1.5)); s += g[k]; }
    for (int k = 0; k < 11; k++) g[k] = g[k] / s;
    GS_CUDA_TRY(cudaMemcpyToSymbol(c_gauss, g, sizeof(g)));
    if (dev < 64) g_gauss_ready |= 1ull << dev;
    return GS_OK;
}

extern "C" size_t gs_loss_temp_bytes(int rows, int image_width) {
    return (size_t)9 * (size_t)(rows > 0 ? rows : 0) * (size_t)image_width * sizeof(float) + 256;
}

// The strips of up to GS_MAX_VIEWS cameras handled by one launch (blockIdx.z = view); passed by value.
struct LossViews {
    int row0[GS_MAX_VIEWS], rows[GS_MAX_VIEWS];       // window rows [row0, row0+rows) of the view's image
    int crow0[GS_MAX_VIEWS], crow1[GS_MAX_VIEWS];     // counted rows, relative to row0
    const uint8_t *gt[GS_MAX_VIEWS];                  // (3, rows, W) uint8 ground truth of the window
    unsigned long long map_off[GS_MAX_VIEWS];         // float offset of the view's 9 derivative planes in `maps`
};

// What k_loss_fwd computes from the rendered pixel x and the ground truth y = gt_u8 / 255.
enum LossMode {
    LS_LOSS = 0,            // training loss: x as rendered; sums[2 view + {0,1}] = sum |x-y|, sum ssim_map; derivative maps
    LS_METRICS_REPORT = 1,  // x = clamp(x, 0, 1); sums[9 view + 3 q + c] (q = |x-y|, (x-y)^2, ssim_map; c = channel); no maps
    LS_METRICS_SAVED = 2,   // as REPORT, x quantised to 8 bits the way torchvision.utils.save_image does, then read back
};

// The evaluated pixel value.  SAVED: save_image's mul(255).add_(0.5).clamp_(0, 255).to(uint8) with the multiply and the
// add rounded separately (no FMA contraction), then to_tensor's division by 255.
template <int MODE>
__device__ __forceinline__ float metric_input(float v) {
    v = fminf(1.f, fmaxf(0.f, v));
    if (MODE == LS_METRICS_SAVED) {
        const float q = fminf(255.f, fmaxf(0.f, __fadd_rn(__fmul_rn(v, 255.f), 0.5f)));
        v = (float)(int)q / 255.0f;
    }
    return v;
}

// temp layout: [0,16) two double accumulators per view; then maps (3 maps x 3 channels x rows x W per view)
template <int MODE>
__global__ void __launch_bounds__(LS_THREADS)
k_loss_fwd(int W, int H, const LossViews lv, const float *__restrict__ image, float *__restrict__ maps,
           double *__restrict__ sums) {
    constexpr bool kMetrics = MODE != LS_LOSS;
    __shared__ float s_x[LS_IN][LS_IN + 1], s_y[LS_IN][LS_IN + 1];
    __shared__ float s_h[5][LS_IN][LS_TILE + 1];
    __shared__ float s_red[2][LS_THREADS / 32];
    const int view = blockIdx.z;
    const int row0 = lv.row0[view], rows = lv.rows[view], crow0 = lv.crow0[view], crow1 = lv.crow1[view];
    const int tx0 = blockIdx.x * LS_TILE, ty0 = blockIdx.y * LS_TILE;  // strip-local tile origin
    if (ty0 >= rows) return;  // the grid is sized for the tallest strip of the batch
    const size_t HW = (size_t)H * W, SW = (size_t)rows * W;
    const uint8_t *__restrict__ gt = lv.gt[view];
    image += (size_t)view * 3 * HW;
    if constexpr (kMetrics) {
        sums += 9 * view;
    } else {
        maps += lv.map_off[view];
        sums += 2 * view;
    }
    const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
    float l1 = 0.f, ss = 0.f;
    // metrics: every per-pixel term is added in fp64, so a view's sums do not depend on how its rows are split into
    // windows and tiles beyond the order of fp64 additions
    __shared__ double s_msum[3][3][LS_THREADS / 32];   // [quantity][channel][warp]; allocated only where it is used
    double m_sad = 0.0, m_sse = 0.0, m_ssim = 0.0;
    for (int ch = 0; ch < 3; ch++) {
        for (int k = threadIdx.x; k < LS_IN * LS_IN; k += LS_THREADS) {
            const int r = k / LS_IN, c = k % LS_IN;
            const int y = ty0 + r - LS_HALO, x = tx0 + c - LS_HALO;
            float vx = 0.f, vy = 0.f;
            if (y >= 0 && y < rows && x >= 0 && x < W) {
                vx = image[ch * HW + (size_t)(row0 + y) * W + x];
                if constexpr (kMetrics) vx = metric_input<MODE>(vx);
                vy = fminf(1.f, fmaxf(0.f, (float)gt[ch * SW + (size_t)y * W + x] / 255.0f));
            }
            s_x[r][c] = vx; s_y[r][c] = vy;
        }
        __syncthreads();
        // row pass, 4 consecutive outputs per thread from a 14-value sliding window held in registers
        // (28 shared loads feed 220 FMAs; one output per thread needed 22 loads for 55)
        for (int k = threadIdx.x; k < LS_IN * (LS_TILE / 4); k += LS_THREADS) {
            const int r = k / (LS_TILE / 4), c0 = (k % (LS_TILE / 4)) * 4;
            float wx[14], wy[14];
#pragma unroll
            for (int t = 0; t < 14; t++) { wx[t] = s_x[r][c0 + t]; wy[t] = s_y[r][c0 + t]; }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
#pragma unroll
                for (int t = 0; t < 11; t++) {
                    const float g = c_gauss[t], vx = wx[q + t], vy = wy[q + t];
                    a0 += g * vx; a1 += g * vy; a2 += g * vx * vx; a3 += g * vy * vy; a4 += g * vx * vy;
                }
                s_h[0][r][c0 + q] = a0; s_h[1][r][c0 + q] = a1; s_h[2][r][c0 + q] = a2; s_h[3][r][c0 + q] = a3;
                s_h[4][r][c0 + q] = a4;
            }
        }
        __syncthreads();
        // column pass: each thread owns one column and 4 consecutive output rows (14-row window per plane)
        {
            const int c = threadIdx.x % LS_TILE, r0 = (threadIdx.x / LS_TILE) * 4, x = tx0 + c;
            float m1[4] = {0.f, 0.f, 0.f, 0.f}, m2[4] = {0.f, 0.f, 0.f, 0.f}, e11[4] = {0.f, 0.f, 0.f, 0.f},
                  e22[4] = {0.f, 0.f, 0.f, 0.f}, e12[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < 14; t++) {
                const float v0 = s_h[0][r0 + t][c], v1 = s_h[1][r0 + t][c], v2 = s_h[2][r0 + t][c], v3 = s_h[3][r0 + t][c],
                            v4 = s_h[4][r0 + t][c];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    if (t - q >= 0 && t - q < 11) {
                        const float g = c_gauss[t - q];
                        m1[q] += g * v0; m2[q] += g * v1; e11[q] += g * v2; e22[q] += g * v3; e12[q] += g * v4;
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int r = r0 + q, y = ty0 + r;
                if constexpr (kMetrics) {
                    if (y < rows && x < W && y >= crow0 && y < crow1) {
                        const float s1 = e11[q] - m1[q] * m1[q], s2 = e22[q] - m2[q] * m2[q], s12 = e12[q] - m1[q] * m2[q];
                        const float A = 2.f * m1[q] * m2[q] + C1, B = 2.f * s12 + C2,
                                    Cc = m1[q] * m1[q] + m2[q] * m2[q] + C1, D = s1 + s2 + C2;
                        const float iCD = 1.f / (Cc * D);
                        m_ssim += (double)(A * B * iCD);
                        const float d = s_x[r + LS_HALO][c + LS_HALO] - s_y[r + LS_HALO][c + LS_HALO];
                        m_sad += (double)fabsf(d);
                        m_sse += (double)d * (double)d;
                    }
                } else if (y < rows && x < W) {
                    const size_t o = (size_t)ch * SW + (size_t)y * W + x;
                    if (y < crow0 || y >= crow1) {  // halo row: feeds the neighbours' windows, carries no loss itself
                        maps[o] = 0.f; maps[3 * SW + o] = 0.f; maps[6 * SW + o] = 0.f;
                    } else {
                        const float s1 = e11[q] - m1[q] * m1[q], s2 = e22[q] - m2[q] * m2[q], s12 = e12[q] - m1[q] * m2[q];
                        const float A = 2.f * m1[q] * m2[q] + C1, B = 2.f * s12 + C2,
                                    Cc = m1[q] * m1[q] + m2[q] * m2[q] + C1, D = s1 + s2 + C2;
                        const float iCD = 1.f / (Cc * D);
                        ss += A * B * iCD;
                        const float vx = s_x[r + LS_HALO][c + LS_HALO], vy = s_y[r + LS_HALO][c + LS_HALO];
                        l1 += fabsf(vx - vy);
                        // d map / d(mu1), d(E[x^2]), d(E[xy])
                        maps[o] = 2.f * m2[q] * (B - A) * iCD - 2.f * m1[q] * A * B * (D - Cc) * iCD * iCD;
                        maps[3 * SW + o] = -A * B * iCD / D;
                        maps[6 * SW + o] = 2.f * A * iCD;
                    }
                }
            }
        }
        if constexpr (kMetrics) {   // this channel's three sums: warp tree, then one slot per warp
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                m_sad += __shfl_xor_sync(0xffffffffu, m_sad, o);
                m_sse += __shfl_xor_sync(0xffffffffu, m_sse, o);
                m_ssim += __shfl_xor_sync(0xffffffffu, m_ssim, o);
            }
            if ((threadIdx.x & 31) == 0) {
                s_msum[0][ch][threadIdx.x >> 5] = m_sad; s_msum[1][ch][threadIdx.x >> 5] = m_sse;
                s_msum[2][ch][threadIdx.x >> 5] = m_ssim;
            }
            m_sad = m_sse = m_ssim = 0.0;
        }
        __syncthreads();
    }
    if constexpr (kMetrics) {
        if (threadIdx.x < 9) {
            const int q = threadIdx.x / 3, c = threadIdx.x % 3;
            double a = 0.0;
            for (int w = 0; w < LS_THREADS / 32; w++) a += s_msum[q][c][w];
            atomicAdd(&sums[3 * q + c], a);
        }
    } else {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { l1 += __shfl_xor_sync(0xffffffffu, l1, o); ss += __shfl_xor_sync(0xffffffffu, ss, o); }
        if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x >> 5] = l1; s_red[1][threadIdx.x >> 5] = ss; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0.0, b = 0.0;
            for (int w = 0; w < LS_THREADS / 32; w++) { a += (double)s_red[0][w]; b += (double)s_red[1][w]; }
            atomicAdd(&sums[0], a); atomicAdd(&sums[1], b);
        }
    }
}

__global__ void k_loss_finalize(int n, const double *__restrict__ sums, double inv_norm, float *__restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;  // 2 values (Ll1, ssim) per view
    if (k < 2 * n) out[k] = (float)(sums[k] * inv_norm);
}

__global__ void __launch_bounds__(LS_THREADS)
k_loss_bwd(int W, int H, const LossViews lv, const float *__restrict__ image, const float *__restrict__ maps,
           const float *__restrict__ grad_l1, const float *__restrict__ grad_ssim, float inv_norm,
           float *__restrict__ dimg) {
    __shared__ float s_m[3][LS_IN][LS_IN + 1];
    __shared__ float s_h[3][LS_IN][LS_TILE + 1];
    const int view = blockIdx.z;
    const int row0 = lv.row0[view], rows = lv.rows[view], crow0 = lv.crow0[view], crow1 = lv.crow1[view];
    const int tx0 = blockIdx.x * LS_TILE, ty0 = blockIdx.y * LS_TILE;
    if (ty0 >= rows) return;
    const size_t HW = (size_t)H * W, SW = (size_t)rows * W;
    const uint8_t *__restrict__ gt = lv.gt[view];
    image += (size_t)view * 3 * HW;
    dimg += (size_t)view * 3 * HW;
    maps += lv.map_off[view];
    const float gl1 = grad_l1[view] * inv_norm, gss = grad_ssim[view] * inv_norm;
    for (int ch = 0; ch < 3; ch++) {
        for (int k = threadIdx.x; k < LS_IN * LS_IN; k += LS_THREADS) {
            const int r = k / LS_IN, c = k % LS_IN;
            const int y = ty0 + r - LS_HALO, x = tx0 + c - LS_HALO;
            float v0 = 0.f, v1 = 0.f, v2 = 0.f;
            if (y >= 0 && y < rows && x >= 0 && x < W) {
                const size_t o = (size_t)ch * SW + (size_t)y * W + x;
                v0 = maps[o]; v1 = maps[3 * SW + o]; v2 = maps[6 * SW + o];
            }
            s_m[0][r][c] = v0; s_m[1][r][c] = v1; s_m[2][r][c] = v2;
        }
        __syncthreads();
        for (int k = threadIdx.x; k < LS_IN * (LS_TILE / 4); k += LS_THREADS) {
            const int r = k / (LS_TILE / 4), c0 = (k % (LS_TILE / 4)) * 4;
            float w0[14], w1[14], w2[14];
#pragma unroll
            for (int t = 0; t < 14; t++) { w0[t] = s_m[0][r][c0 + t]; w1[t] = s_m[1][r][c0 + t]; w2[t] = s_m[2][r][c0 + t]; }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
                for (int t = 0; t < 11; t++) {
                    const float g = c_gauss[t];
                    a0 += g * w0[q + t]; a1 += g * w1[q + t]; a2 += g * w2[q + t];
                }
                s_h[0][r][c0 + q] = a0; s_h[1][r][c0 + q] = a1; s_h[2][r][c0 + q] = a2;
            }
        }
        __syncthreads();
        {
            const int c = threadIdx.x % LS_TILE, r0 = (threadIdx.x / LS_TILE) * 4, x = tx0 + c;
            float b0[4] = {0.f, 0.f, 0.f, 0.f}, b1[4] = {0.f, 0.f, 0.f, 0.f}, b2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int t = 0; t < 14; t++) {
                const float v0 = s_h[0][r0 + t][c], v1 = s_h[1][r0 + t][c], v2 = s_h[2][r0 + t][c];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    if (t - q >= 0 && t - q < 11) {
                        const float g = c_gauss[t - q];
                        b0[q] += g * v0; b1[q] += g * v1; b2[q] += g * v2;
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int y = ty0 + r0 + q;
                if (y < rows && x < W) {
                    const size_t oi = ch * HW + (size_t)(row0 + y) * W + x;
                    const float vx = image[oi];
                    const float vy = fminf(1.f, fmaxf(0.f, (float)gt[ch * SW + (size_t)y * W + x] / 255.0f));
                    const float d = vx - vy;
                    const float sgn = (y < crow0 || y >= crow1) ? 0.f : (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
                    dimg[oi] = gl1 * sgn + gss * (b0[q] + 2.f * vx * b1[q] + vy * b2[q]);
                }
            }
        }
        __syncthreads();
    }
}

// bytes in front of the derivative maps: the per-view double accumulators (one view: the original 256-byte header)
#define LS_HEADER_1 ((size_t)256)
#define LS_HEADER_B ((size_t)(2 * sizeof(double) * GS_MAX_VIEWS))

// rows4: (num_views, 4) HOST ints = row0, row1, count_row0, count_row1 per view; row1 == row0 skips the view.
// Fills the kernel-side table; returns the tallest window in *max_rows and the total window rows in *sum_rows.
static int make_loss_views(int num_views, int H, int W, const int32_t *rows4, const void *const *gts, LossViews &lv,
                           int *max_rows, size_t *sum_rows) {
    GS_REQUIRE(num_views >= 1 && num_views <= GS_MAX_VIEWS, "num_views must be in [1, GS_MAX_VIEWS]");
    GS_REQUIRE(H > 0 && W > 0 && rows4 && gts, "sizes");
    size_t off = 0;
    int mx = 0;
    for (int v = 0; v < GS_MAX_VIEWS; v++) {
        lv.row0[v] = lv.rows[v] = lv.crow0[v] = lv.crow1[v] = 0;
        lv.gt[v] = nullptr;
        lv.map_off[v] = 0ull;
        if (v >= num_views) continue;
        const int row0 = rows4[4 * v], row1 = rows4[4 * v + 1], c0 = rows4[4 * v + 2], c1 = rows4[4 * v + 3];
        const int rows = row1 - row0;
        GS_REQUIRE(row0 >= 0 && row1 <= H && rows >= 0, "strip rows");
        if (rows == 0) continue;
        GS_REQUIRE(c0 >= row0 && c1 <= row1 && c1 >= c0, "count rows must lie inside [row0,row1)");
        GS_REQUIRE(gts[v] != nullptr, "null ground-truth pointer");
        lv.row0[v] = row0; lv.rows[v] = rows; lv.crow0[v] = c0 - row0; lv.crow1[v] = c1 - row0;
        lv.gt[v] = (const uint8_t *)gts[v];
        lv.map_off[v] = (unsigned long long)off;
        off += (size_t)9 * rows * W;
        mx = rows > mx ? rows : mx;
    }
    *max_rows = mx;
    *sum_rows = off / ((size_t)9 * W);
    return GS_OK;
}

static int loss_forward_impl(int num_views, int H, int W, const int32_t *rows4, const float *image, const void *const *gts,
                             float *out, void *temp, size_t temp_bytes, size_t header, cudaStream_t stream) {
    GS_REQUIRE(image && out && temp, "null pointer");
    LossViews lv;
    int max_rows = 0;
    size_t sum_rows = 0;
    int rc = make_loss_views(num_views, H, W, rows4, gts, lv, &max_rows, &sum_rows);
    if (rc != GS_OK) return rc;
    if (temp_bytes < header + (size_t)9 * sum_rows * W * sizeof(float)) {
        gs_set_error("gs_loss_forward: temp too small");
        return GS_ENOMEM;
    }
    rc = ensure_gauss();
    if (rc != GS_OK) return rc;
    double *sums = (double *)temp;
    float *maps = (float *)((char *)temp + header);
    GS_CUDA_TRY(cudaMemsetAsync(sums, 0, 2 * sizeof(double) * (size_t)num_views, stream));
    GsStageTimer timer(GS_STAGE_LOSS_FWD, stream);
    if (max_rows > 0) {
        dim3 grid((W + LS_TILE - 1) / LS_TILE, (max_rows + LS_TILE - 1) / LS_TILE, num_views);
        k_loss_fwd<LS_LOSS><<<grid, LS_THREADS, 0, stream>>>(W, H, lv, image, maps, sums);
        GS_LAUNCH_CHECK();
    }
    k_loss_finalize<<<1, 2 * GS_MAX_VIEWS, 0, stream>>>(num_views, sums, 1.0 / (3.0 * (double)H * (double)W), out);
    GS_LAUNCH_CHECK();
    return GS_OK;
}

static int loss_backward_impl(int num_views, int H, int W, const int32_t *rows4, const float *image,
                              const void *const *gts, const void *temp, const float *grad_l1, const float *grad_ssim,
                              float *dimg, size_t header, cudaStream_t stream) {
    GS_REQUIRE(image && temp && grad_l1 && grad_ssim && dimg, "null pointer");
    LossViews lv;
    int max_rows = 0;
    size_t sum_rows = 0;
    int rc = make_loss_views(num_views, H, W, rows4, gts, lv, &max_rows, &sum_rows);
    if (rc != GS_OK) return rc;
    rc = ensure_gauss();
    if (rc != GS_OK) return rc;
    const float *maps = (const float *)((const char *)temp + header);
    const size_t HW = (size_t)H * W;
    // rows outside the windows carry no loss
    if (num_views == 1) {
        const int row0 = lv.row0[0], row1 = lv.row0[0] + lv.rows[0];
        for (int ch = 0; ch < 3; ch++) {
            if (row0 > 0) GS_CUDA_TRY(cudaMemsetAsync(dimg + ch * HW, 0, sizeof(float) * (size_t)row0 * W, stream));
            if (row1 < H)
                GS_CUDA_TRY(cudaMemsetAsync(dimg + ch * HW + (size_t)row1 * W, 0, sizeof(float) * (size_t)(H - row1) * W, stream));
        }
    } else if (sum_rows < (size_t)num_views * H) {
        GS_CUDA_TRY(cudaMemsetAsync(dimg, 0, sizeof(float) * 3 * HW * (size_t)num_views, stream));
    }
    if (max_rows == 0) return GS_OK;
    dim3 grid((W + LS_TILE - 1) / LS_TILE, (max_rows + LS_TILE - 1) / LS_TILE, num_views);
    GsStageTimer timer(GS_STAGE_LOSS_BWD, stream);
    k_loss_bwd<<<grid, LS_THREADS, 0, stream>>>(W, H, lv, image, maps, grad_l1, grad_ssim,
                                                (float)(1.0 / (3.0 * (double)H * (double)W)), dimg);
    GS_LAUNCH_CHECK();
    return GS_OK;
}

extern "C" int gs_loss_forward(int image_height, int image_width, int row0, int row1, int count_row0, int count_row1,
                               const float *image, const uint8_t *gt_u8, float *out_l1_ssim, void *temp,
                               size_t temp_bytes, void *stream_) {
    GS_REQUIRE(row1 > row0, "strip rows");
    GS_REQUIRE(gt_u8, "null pointer");
    const int32_t rows4[4] = {row0, row1, count_row0, count_row1};
    const void *gts[1] = {gt_u8};
    return loss_forward_impl(1, image_height, image_width, rows4, image, gts, out_l1_ssim, temp, temp_bytes, LS_HEADER_1,
                             (cudaStream_t)stream_);
}

extern "C" size_t gs_loss_temp_bytes_batched(int num_views, const int32_t *rows4_host, int image_width) {
    size_t rows = 0;
    for (int v = 0; v < num_views && rows4_host; v++) {
        const int r = rows4_host[4 * v + 1] - rows4_host[4 * v];
        rows += r > 0 ? (size_t)r : 0;
    }
    return LS_HEADER_B + (size_t)9 * rows * (size_t)(image_width > 0 ? image_width : 0) * sizeof(float) + 256;
}

extern "C" int gs_loss_forward_batched(int num_views, int image_height, int image_width, const int32_t *rows4_host,
                                       const float *image, const void *const *gt_u8_ptrs_host, float *out_l1_ssim,
                                       void *temp, size_t temp_bytes, void *stream_) {
    return loss_forward_impl(num_views, image_height, image_width, rows4_host, image, gt_u8_ptrs_host, out_l1_ssim, temp,
                             temp_bytes, LS_HEADER_B, (cudaStream_t)stream_);
}

extern "C" int gs_loss_backward(int image_height, int image_width, int row0, int row1, int count_row0, int count_row1,
                                const float *image, const uint8_t *gt_u8, const void *temp, const float *grad_l1,
                                const float *grad_ssim, float *dL_dimage, void *stream_) {
    GS_REQUIRE(row1 > row0, "strip rows");
    GS_REQUIRE(gt_u8, "null pointer");
    const int32_t rows4[4] = {row0, row1, count_row0, count_row1};
    const void *gts[1] = {gt_u8};
    return loss_backward_impl(1, image_height, image_width, rows4, image, gts, temp, grad_l1, grad_ssim, dL_dimage,
                              LS_HEADER_1, (cudaStream_t)stream_);
}

extern "C" int gs_loss_backward_batched(int num_views, int image_height, int image_width, const int32_t *rows4_host,
                                        const float *image, const void *const *gt_u8_ptrs_host, const void *temp,
                                        const float *grad_l1, const float *grad_ssim, float *dL_dimage, void *stream_) {
    return loss_backward_impl(num_views, image_height, image_width, rows4_host, image, gt_u8_ptrs_host, temp, grad_l1,
                              grad_ssim, dL_dimage, LS_HEADER_B, (cudaStream_t)stream_);
}

extern "C" int gs_metrics_batched(int num_views, int image_height, int image_width, const int32_t *rows4_host,
                                  const float *images, const uint8_t *const *gt_u8_host_array, int saved_mode,
                                  double *out_sums, void *stream_) {
    GS_REQUIRE(images && out_sums, "null pointer");
    GS_REQUIRE(saved_mode == 0 || saved_mode == 1, "saved_mode must be 0 or 1");
    const cudaStream_t stream = (cudaStream_t)stream_;
    LossViews lv;
    int max_rows = 0;
    size_t sum_rows = 0;
    int rc = make_loss_views(num_views, image_height, image_width, rows4_host, (const void *const *)gt_u8_host_array, lv,
                             &max_rows, &sum_rows);
    if (rc != GS_OK) return rc;
    rc = ensure_gauss();
    if (rc != GS_OK) return rc;
    GS_CUDA_TRY(cudaMemsetAsync(out_sums, 0, 9 * sizeof(double) * (size_t)num_views, stream));
    if (max_rows == 0) return GS_OK;
    dim3 grid((image_width + LS_TILE - 1) / LS_TILE, (max_rows + LS_TILE - 1) / LS_TILE, num_views);
    if (saved_mode)
        k_loss_fwd<LS_METRICS_SAVED><<<grid, LS_THREADS, 0, stream>>>(image_width, image_height, lv, images, nullptr,
                                                                       out_sums);
    else
        k_loss_fwd<LS_METRICS_REPORT><<<grid, LS_THREADS, 0, stream>>>(image_width, image_height, lv, images, nullptr,
                                                                        out_sums);
    GS_LAUNCH_CHECK();
    return GS_OK;
}
