// Fused SSIM of two image stacks and its gradient with respect to the first one.
//
// Reference behaviour restated here (3DGS utils/loss_utils.py, used by taekkii/deblurgs and its evaluation):
//   window   = outer product of the 11-tap Gaussian (sigma 1.5, normalised in fp32)          create_window / gaussian
//   mu       = conv2d(img, window, padding=5, groups=C)   (zero padding, NOT renormalised)     _ssim
//   sigma1^2 = conv2d(img1*img1) - mu1^2, sigma2^2 likewise, sigma12 = conv2d(img1*img2) - mu1*mu2
//   map      = ((2 mu1 mu2 + C1)(2 sigma12 + C2)) / ((mu1^2 + mu2^2 + C1)(sigma1^2 + sigma2^2 + C2)), C1 = 0.01^2, C2 = 0.03^2
//   ssim     = mean over N*C*H*W (size_average) or one mean per image
// The torch statement is 5 depthwise 11x11 convolutions plus ~15 elementwise kernels forward and about twice that
// backward.  Here one tile kernel computes the five windowed moments separably from shared memory (horizontal pass
// into shared memory, vertical pass per output pixel), the map value, its per-block sum and, when a gradient is wanted,
// three per-pixel maps; a one-block kernel sums the per-block partials in a fixed order (no atomics: repeated calls and
// graph replays give the same bits).  The backward is the same tile structure over the three maps:
//   dL/dx(q) = g * sum_p w(p - q) [dmu(p) + 2 x(q) ds/dsigma1^2(p) + y(q) ds/dsigma12(p)]
#include "dgs_b200.h"
#include "dgs_internal.cuh"

#include <cmath>

namespace dgs {

constexpr int SSIM_TW = 32, SSIM_TH = 16;                 // output tile; one thread per output pixel
constexpr int SSIM_R = 5, SSIM_K = 2 * SSIM_R + 1;        // window radius / taps
constexpr int SSIM_SW = SSIM_TW + 2 * SSIM_R, SSIM_SH = SSIM_TH + 2 * SSIM_R;
constexpr int SSIM_THREADS = SSIM_TW * SSIM_TH;
constexpr int SSIM_FIN_THREADS = 256;

struct SsimWindow { float w[SSIM_K]; };   // passed by value: a graph node keeps its own copy

// create_window(11, C) of the reference: gaussian() evaluates exp in double and stores fp32, then divides by torch's
// fp32 sum of the 11 stored values.  For these 11 values that sum is their exact sum rounded once to fp32 (a
// left-to-right fp32 sum is 1 ulp lower); tests/test_ssim_algebra.py pins the weights to torch's bit for bit.
static SsimWindow ssim_window()
{
    SsimWindow win;
    double sum = 0.0;
    for (int i = 0; i < SSIM_K; i++) {
        win.w[i] = (float)std::exp(-(double)((i - SSIM_R) * (i - SSIM_R)) / (2.0 * 1.5 * 1.5));
        sum += (double)win.w[i];
    }
    const float fsum = (float)sum;
    for (int i = 0; i < SSIM_K; i++) win.w[i] = win.w[i] / fsum;
    return win;
}

// Zero-padded halo of one (image, channel) plane: tile origin (x0, y0) minus the window radius.
__device__ __forceinline__ float ld_halo(const float* __restrict__ p, int H, int W, int gy, int gx)
{
    return (gy >= 0 && gy < H && gx >= 0 && gx < W) ? p[(size_t)gy * W + gx] : 0.f;
}

__global__ void __launch_bounds__(SSIM_THREADS) k_ssim_fwd(int H, int W, SsimWindow win, const float* __restrict__ x,
                                                           const float* __restrict__ y, double* __restrict__ partial,
                                                           float* __restrict__ maps, size_t map_stride)
{
    __shared__ float sx[SSIM_SH][SSIM_SW], sy[SSIM_SH][SSIM_SW];
    __shared__ float hm[5][SSIM_SH][SSIM_TW];     // horizontal pass of x, y, x^2, y^2, xy
    __shared__ double red[SSIM_THREADS / 32];
    const int x0 = blockIdx.x * SSIM_TW, y0 = blockIdx.y * SSIM_TH;
    const size_t plane = (size_t)blockIdx.z * H * W;
    const float* xp = x + plane;
    const float* yp = y + plane;
    const int tid = threadIdx.y * SSIM_TW + threadIdx.x;

    for (int i = tid; i < SSIM_SH * SSIM_SW; i += SSIM_THREADS) {
        const int r = i / SSIM_SW, c = i - r * SSIM_SW;
        sx[r][c] = ld_halo(xp, H, W, y0 - SSIM_R + r, x0 - SSIM_R + c);
        sy[r][c] = ld_halo(yp, H, W, y0 - SSIM_R + r, x0 - SSIM_R + c);
    }
    __syncthreads();
    for (int i = tid; i < SSIM_SH * SSIM_TW; i += SSIM_THREADS) {
        const int r = i / SSIM_TW, c = i - r * SSIM_TW;
        float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
#pragma unroll
        for (int k = 0; k < SSIM_K; k++) {
            const float a = sx[r][c + k], b = sy[r][c + k], w = win.w[k];
            m0 += w * a;
            m1 += w * b;
            m2 += w * (a * a);
            m3 += w * (b * b);
            m4 += w * (a * b);
        }
        hm[0][r][c] = m0; hm[1][r][c] = m1; hm[2][r][c] = m2; hm[3][r][c] = m3; hm[4][r][c] = m4;
    }
    __syncthreads();

    float mu1 = 0.f, mu2 = 0.f, e11 = 0.f, e22 = 0.f, e12 = 0.f;
#pragma unroll
    for (int k = 0; k < SSIM_K; k++) {
        const int r = threadIdx.y + k;
        const float w = win.w[k];
        mu1 += w * hm[0][r][threadIdx.x];
        mu2 += w * hm[1][r][threadIdx.x];
        e11 += w * hm[2][r][threadIdx.x];
        e22 += w * hm[3][r][threadIdx.x];
        e12 += w * hm[4][r][threadIdx.x];
    }
    const int ox = x0 + threadIdx.x, oy = y0 + threadIdx.y;
    const bool valid = ox < W && oy < H;
    const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
    const float mu1_sq = mu1 * mu1, mu2_sq = mu2 * mu2, mu12 = mu1 * mu2;
    const float s1 = e11 - mu1_sq, s2 = e22 - mu2_sq, s12 = e12 - mu12;
    const float A1 = 2.f * mu12 + C1, A2 = 2.f * s12 + C2;
    const float B1 = mu1_sq + mu2_sq + C1, B2 = s1 + s2 + C2;
    const float s = (A1 * A2) / (B1 * B2);
    if (valid && maps != nullptr) {
        const float inv = 1.f / (B1 * B2);
        const float d_s1 = -s / B2;                  // ds/dsigma1^2
        const float d_s12 = 2.f * A1 * inv;          // ds/dsigma12
        // total derivative in mu1 with E[x^2], E[xy] held (sigma1^2 and sigma12 both depend on mu1)
        const float d_mu = 2.f * mu2 * A2 * inv - 2.f * mu1 * s / B1 - 2.f * mu1 * d_s1 - mu2 * d_s12;
        const size_t o = plane + (size_t)oy * W + ox;
        maps[o] = d_mu;
        maps[map_stride + o] = d_s1;
        maps[2 * map_stride + o] = d_s12;
    }

    double a = valid ? (double)s : 0.0;
    for (int d = 16; d >= 1; d >>= 1) a += __shfl_xor_sync(0xffffffffu, a, d);
    if ((tid & 31) == 0) red[tid >> 5] = a;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int i = 0; i < SSIM_THREADS / 32; i++) t += red[i];
        partial[((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = t;
    }
}

// out[0] = mean over every map value, out[1 + n] = mean over image n.  One block; every sum in a fixed order.
__global__ void __launch_bounds__(SSIM_FIN_THREADS) k_ssim_finalize(int N, size_t per_image, double count_image,
                                                                    const double* __restrict__ partial,
                                                                    float* __restrict__ out)
{
    __shared__ double red[SSIM_FIN_THREADS];
    double total = 0.0;
    for (int n = 0; n < N; n++) {
        double a = 0.0;
        for (size_t i = threadIdx.x; i < per_image; i += SSIM_FIN_THREADS) a += partial[(size_t)n * per_image + i];
        red[threadIdx.x] = a;
        __syncthreads();
        for (int h = SSIM_FIN_THREADS / 2; h >= 1; h >>= 1) {
            if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            out[1 + n] = (float)(red[0] / count_image);
            total += red[0];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = (float)(total / (count_image * N));
}

__global__ void __launch_bounds__(SSIM_THREADS) k_ssim_bwd(int C, int H, int W, SsimWindow win,
                                                           const float* __restrict__ x, const float* __restrict__ y,
                                                           const float* __restrict__ maps, size_t map_stride,
                                                           const float* __restrict__ grad_out, int per_image,
                                                           float inv_count, float* __restrict__ dx)
{
    __shared__ float sm[3][SSIM_SH][SSIM_SW];
    __shared__ float hm[3][SSIM_SH][SSIM_TW];
    const int x0 = blockIdx.x * SSIM_TW, y0 = blockIdx.y * SSIM_TH;
    const size_t plane = (size_t)blockIdx.z * H * W;
    const int tid = threadIdx.y * SSIM_TW + threadIdx.x;

    for (int i = tid; i < SSIM_SH * SSIM_SW; i += SSIM_THREADS) {
        const int r = i / SSIM_SW, c = i - r * SSIM_SW;
#pragma unroll
        for (int m = 0; m < 3; m++)
            sm[m][r][c] = ld_halo(maps + m * map_stride + plane, H, W, y0 - SSIM_R + r, x0 - SSIM_R + c);
    }
    __syncthreads();
    for (int i = tid; i < SSIM_SH * SSIM_TW; i += SSIM_THREADS) {
        const int r = i / SSIM_TW, c = i - r * SSIM_TW;
        float m0 = 0.f, m1 = 0.f, m2 = 0.f;
#pragma unroll
        for (int k = 0; k < SSIM_K; k++) {
            const float w = win.w[k];
            m0 += w * sm[0][r][c + k];
            m1 += w * sm[1][r][c + k];
            m2 += w * sm[2][r][c + k];
        }
        hm[0][r][c] = m0; hm[1][r][c] = m1; hm[2][r][c] = m2;
    }
    __syncthreads();

    const int ox = x0 + threadIdx.x, oy = y0 + threadIdx.y;
    if (ox >= W || oy >= H) return;
    float c0 = 0.f, c1 = 0.f, c2 = 0.f;
#pragma unroll
    for (int k = 0; k < SSIM_K; k++) {
        const int r = threadIdx.y + k;
        const float w = win.w[k];
        c0 += w * hm[0][r][threadIdx.x];
        c1 += w * hm[1][r][threadIdx.x];
        c2 += w * hm[2][r][threadIdx.x];
    }
    const float go = grad_out ? grad_out[per_image ? (int)(blockIdx.z / C) : 0] : 1.0f;
    const size_t o = plane + (size_t)oy * W + ox;
    dx[o] = go * inv_count * (c0 + 2.f * x[o] * c1 + y[o] * c2);
}

static bool ssim_dims_ok(int N, int C, int H, int W)
{
    return N > 0 && C > 0 && H > 0 && W > 0 && (int64_t)N * C <= 65535;   // planes ride on gridDim.z
}

static dim3 ssim_grid(int N, int C, int H, int W)
{
    return dim3((unsigned)((W + SSIM_TW - 1) / SSIM_TW), (unsigned)((H + SSIM_TH - 1) / SSIM_TH), (unsigned)(N * C));
}

}  // namespace dgs

extern "C" {

using dgs::ssim_dims_ok;
using dgs::ssim_grid;

size_t dgs_ssim_scratch_bytes(int N, int C, int H, int W)
{
    if (!ssim_dims_ok(N, C, H, W)) return 0;
    const dim3 g = ssim_grid(N, C, H, W);
    return (size_t)g.x * g.y * g.z * sizeof(double);
}

int dgs_ssim_forward(int N, int C, int H, int W, const float* img1, const float* img2, float* ssim_out,
                     double* scratch, float* maps, void* stream)
{
    if (!ssim_dims_ok(N, C, H, W)) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_ssim_forward: invalid size");
    if (!img1 || !img2 || !ssim_out || !scratch)
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_ssim_forward: invalid argument");
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 g = ssim_grid(N, C, H, W);
    const size_t plane = (size_t)H * W;
    dgs::k_ssim_fwd<<<g, dim3(dgs::SSIM_TW, dgs::SSIM_TH), 0, st>>>(H, W, dgs::ssim_window(), img1, img2, scratch,
                                                                    maps, (size_t)N * C * plane);
    dgs::k_ssim_finalize<<<1, dgs::SSIM_FIN_THREADS, 0, st>>>(N, (size_t)g.x * g.y * C, (double)C * (double)plane,
                                                               scratch, ssim_out);
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_ssim_forward"); }
}

int dgs_ssim_backward(int N, int C, int H, int W, const float* img1, const float* img2, const float* maps,
                      const float* grad_out, int per_image, float* dL_dimg1, void* stream)
{
    if (!ssim_dims_ok(N, C, H, W)) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_ssim_backward: invalid size");
    if (!img1 || !img2 || !maps || !dL_dimg1)
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_ssim_backward: invalid argument");
    const size_t plane = (size_t)H * W;
    const double count = per_image ? (double)C * (double)plane : (double)N * C * (double)plane;
    dgs::k_ssim_bwd<<<ssim_grid(N, C, H, W), dim3(dgs::SSIM_TW, dgs::SSIM_TH), 0, (cudaStream_t)stream>>>(
        C, H, W, dgs::ssim_window(), img1, img2, maps, (size_t)N * C * plane, grad_out, per_image ? 1 : 0,
        (float)(1.0 / count), dL_dimg1);
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_ssim_backward"); }
}

}  // extern "C"
