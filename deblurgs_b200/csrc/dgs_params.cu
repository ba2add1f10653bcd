// The two steps either side of the rasterizer on the Gaussian parameter store (SURVEY.md 8f rank 3):
// the activations `render` reads, and the Adam update that consumes the rasterizer's gradients.
//
// Reference behaviour restated here (taekkii/deblurgs):
//   get_scaling   = exp(_scaling) + scale_lb  (isotropic: column 0 expanded)   scene/gaussian_model.py:114-119,
//                                                                              scene/gaussian_activation.py:43-52
//   get_rotation  = _rotation / max(|_rotation|_2, 1e-12)  (F.normalize)       scene/gaussian_model.py:50,121-123
//   get_opacity   = clamp(_opacity, 0, 1)                                      scene/gaussian_activation.py:29-34
//   get_features  = cat(_features_dc, _features_rest, dim=1)                   scene/gaussian_model.py:129-133
//   optimizer     = torch.optim.Adam(groups, lr=0.0, eps=1e-15)                scene/gaussian_model.py:181-190
// The reference evaluates the four getters once per SUB-FRAME render (~8 elementwise launches and a
// 12*M-byte cat copy each, again in backward) and steps Adam with one multi-kernel foreach pass per
// parameter tensor.  Here: one launch activates the whole store, one launch back-propagates through
// it, one launch steps every parameter tensor of the model.  All three are pure streaming kernels
// (HBM-bound): flat, coalesced indexing; the per-Gaussian maths rides on the first P threads.
#include "dgs_b200.h"
#include "dgs_internal.cuh"

#include <cmath>
#include <cstring>

namespace dgs {

// s'_i = sqrt(s_i^2 + f^2) and r_i = s_i / s'_i, rounded as the torch statement (square, add, sqrt, divide: no FMA)
__device__ __forceinline__ void filter3d_scales(float a0, float a1, float a2, float f, float* out, float& r0,
                                                float& r1, float& r2)
{
    const float f2 = __fmul_rn(f, f);
    const float b0 = sqrtf(__fadd_rn(__fmul_rn(a0, a0), f2)), b1 = sqrtf(__fadd_rn(__fmul_rn(a1, a1), f2)),
                b2 = sqrtf(__fadd_rn(__fmul_rn(a2, a2), f2));
    out[0] = b0; out[1] = b1; out[2] = b2;
    r0 = __fdiv_rn(a0, b0); r1 = __fdiv_rn(a1, b1); r2 = __fdiv_rn(a2, b2);
}

// sh [P, M, 3] = cat(dc [P,1,3], rest [P,M-1,3]);  per Gaussian: scales, rotations, opacities.
// FILTER: Mip-Splatting's 3-D smoothing filter f = filter3d[g] (a constant): s'_i = sqrt(s_i^2 + f^2) and
// opacity' = clamp(o) * r_0 * r_1 * r_2 with r_i = s_i / s'_i -- get_{scaling,opacity}_with_3D_filter, whose
// sqrt(det1 / det2) is written as a product of per-axis ratios because prod(s_i^2) underflows in fp32 for s < ~1e-7.
template <bool FILTER>
__global__ void __launch_bounds__(256) k_activate_fwd(int P, int M, const float* __restrict__ dc,
                                                      const float* __restrict__ rest,
                                                      const float* __restrict__ scaling,
                                                      const float* __restrict__ rotation,
                                                      const float* __restrict__ opacity, float scale_lb,
                                                      int isotropic, float* __restrict__ sh,
                                                      float* __restrict__ scales, float* __restrict__ rot,
                                                      float* __restrict__ opac, const float* __restrict__ filter3d)
{
    const size_t row = (size_t)3 * M, total = (size_t)P * row;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (total < 0xF0000000ull) {   // 32-bit index arithmetic (a 64-bit divide per element would make this ALU-bound); headroom for i += stride
        const uint32_t row32 = (uint32_t)row;
        for (uint32_t i = (uint32_t)t0; i < (uint32_t)total; i += (uint32_t)stride) {
            const uint32_t g = i / row32, r = i - g * row32;
            sh[i] = r < 3 ? dc[g * 3 + r] : rest[(size_t)g * (row32 - 3) + (r - 3)];
        }
    } else {
        for (size_t i = t0; i < total; i += stride) {
            const size_t g = i / row, r = i - g * row;
            sh[i] = r < 3 ? dc[g * 3 + r] : rest[g * (row - 3) + (r - 3)];
        }
    }
    for (size_t g = t0; g < (size_t)P; g += stride) {
        const float s0 = scaling[3 * g], s1 = scaling[3 * g + 1], s2 = scaling[3 * g + 2];
        if constexpr (FILTER) {
            const float a0 = expf(s0) + scale_lb, a1 = expf(isotropic ? s0 : s1) + scale_lb,
                        a2 = expf(isotropic ? s0 : s2) + scale_lb;
            float r0, r1, r2;
            filter3d_scales(a0, a1, a2, filter3d[g], scales + 3 * g, r0, r1, r2);
            const float4 q = reinterpret_cast<const float4*>(rotation)[g];
            const float n = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
            reinterpret_cast<float4*>(rot)[g] = make_float4(q.x / n, q.y / n, q.z / n, q.w / n);
            opac[g] = fminf(fmaxf(opacity[g], 0.0f), 1.0f) * r0 * r1 * r2;
        } else {
            scales[3 * g] = expf(s0) + scale_lb;
            scales[3 * g + 1] = expf(isotropic ? s0 : s1) + scale_lb;
            scales[3 * g + 2] = expf(isotropic ? s0 : s2) + scale_lb;
            const float4 q = reinterpret_cast<const float4*>(rotation)[g];
            const float n = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
            reinterpret_cast<float4*>(rot)[g] = make_float4(q.x / n, q.y / n, q.z / n, q.w / n);
            opac[g] = fminf(fmaxf(opacity[g], 0.0f), 1.0f);
        }
    }
}

// Chain rule of the above.  Any of the incoming gradients may be NULL (treated as zero).  FILTER (f has no gradient):
//   dL/ds_i = g_s'_i r_i + g_o' clamp(o) (prod_{j != i} r_j) f^2 / s'_i^3,   dL/dclamp(o) = g_o' r_0 r_1 r_2,
// then the exp / isotropic chain and the clamp mask as without the filter.
template <bool FILTER>
__global__ void __launch_bounds__(256) k_activate_bwd(int P, int M, const float* __restrict__ scaling,
                                                      const float* __restrict__ rotation,
                                                      const float* __restrict__ opacity, int isotropic,
                                                      const float* __restrict__ dsh,
                                                      const float* __restrict__ dscales,
                                                      const float* __restrict__ drot,
                                                      const float* __restrict__ dopac, float* __restrict__ ddc,
                                                      float* __restrict__ drest, float* __restrict__ dscaling,
                                                      float* __restrict__ drotation, float* __restrict__ dopacity,
                                                      float scale_lb, const float* __restrict__ filter3d)
{
    const size_t row = (size_t)3 * M, total = (size_t)P * row;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (total < 0xF0000000ull) {
        const uint32_t row32 = (uint32_t)row;
        for (uint32_t i = (uint32_t)t0; i < (uint32_t)total; i += (uint32_t)stride) {
            const uint32_t g = i / row32, r = i - g * row32;
            const float v = dsh ? dsh[i] : 0.f;
            if (r < 3) ddc[g * 3 + r] = v; else drest[(size_t)g * (row32 - 3) + (r - 3)] = v;
        }
    } else {
        for (size_t i = t0; i < total; i += stride) {
            const size_t g = i / row, r = i - g * row;
            const float v = dsh ? dsh[i] : 0.f;
            if (r < 3) ddc[g * 3 + r] = v; else drest[g * (row - 3) + (r - 3)] = v;
        }
    }
    for (size_t g = t0; g < (size_t)P; g += stride) {
        // exp: d/dx = exp(x) (torch multiplies by the saved result; the lower bound is an additive constant)
        const float s0 = scaling[3 * g], s1 = scaling[3 * g + 1], s2 = scaling[3 * g + 2];
        float g0 = dscales ? dscales[3 * g] : 0.f, g1 = dscales ? dscales[3 * g + 1] : 0.f,
              g2 = dscales ? dscales[3 * g + 2] : 0.f;
        float opac_scale = 1.f;   // FILTER: r_0 r_1 r_2, the factor between the clamped and the filtered opacity
        if constexpr (FILTER) {
            const float a0 = expf(s0) + scale_lb, a1 = expf(isotropic ? s0 : s1) + scale_lb,
                        a2 = expf(isotropic ? s0 : s2) + scale_lb;
            const float f = filter3d[g];
            float b[3], r0, r1, r2;
            filter3d_scales(a0, a1, a2, f, b, r0, r1, r2);
            const float go = dopac ? dopac[g] : 0.f;
            // f^2 / s'^3 as (f / s')^2 / s': no cube to underflow for tiny scales, and exactly 0 for f = 0
            const float t = go * fminf(fmaxf(opacity[g], 0.0f), 1.0f);
            const float q0 = f / b[0], q1 = f / b[1], q2 = f / b[2];
            g0 = g0 * r0 + t * (r1 * r2) * (q0 * q0) / b[0];
            g1 = g1 * r1 + t * (r0 * r2) * (q1 * q1) / b[1];
            g2 = g2 * r2 + t * (r0 * r1) * (q2 * q2) / b[2];
            opac_scale = r0 * r1 * r2;
        }
        if (isotropic) {
            // the expanded column 0 collects the three gradients; columns 1, 2 are unused parameters
            const float e0 = expf(s0);
            dscaling[3 * g] = g0 * e0 + g1 * e0 + g2 * e0;
            dscaling[3 * g + 1] = 0.f;
            dscaling[3 * g + 2] = 0.f;
        } else {
            dscaling[3 * g] = g0 * expf(s0);
            dscaling[3 * g + 1] = g1 * expf(s1);
            dscaling[3 * g + 2] = g2 * expf(s2);
        }
        // normalize: r = q / n  =>  dq = (g - r (r.g)) / n   (n clamped at 1e-12: then dq = g / 1e-12)
        const float4 q = reinterpret_cast<const float4*>(rotation)[g];
        const float4 gr = drot ? reinterpret_cast<const float4*>(drot)[g] : make_float4(0.f, 0.f, 0.f, 0.f);
        const float nn = sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
        float4 dq;
        if (nn > 1e-12f) {
            const float inv = 1.0f / nn;
            const float rx = q.x * inv, ry = q.y * inv, rz = q.z * inv, rw = q.w * inv;
            const float dot = rx * gr.x + ry * gr.y + rz * gr.z + rw * gr.w;
            dq = make_float4((gr.x - rx * dot) * inv, (gr.y - ry * dot) * inv, (gr.z - rz * dot) * inv,
                             (gr.w - rw * dot) * inv);
        } else {
            dq = make_float4(gr.x * 1e12f, gr.y * 1e12f, gr.z * 1e12f, gr.w * 1e12f);
        }
        reinterpret_cast<float4*>(drotation)[g] = dq;
        // clamp: gradient passes where 0 <= x <= 1
        const float o = opacity[g];
        if constexpr (FILTER)
            dopacity[g] = (o >= 0.0f && o <= 1.0f) ? (dopac ? dopac[g] : 0.f) * opac_scale : 0.f;
        else
            dopacity[g] = (o >= 0.0f && o <= 1.0f) ? (dopac ? dopac[g] : 0.f) : 0.f;
    }
}

// ---- Adam over up to DGS_ADAM_MAX_TENSORS parameter tensors in one launch ---------------------
struct AdamTensor {
    float* p;
    const float* g;
    float* m;
    float* v;
    long long n;
    long long first_block;   // blocks [first_block, first_block + ceil(n / ADAM_CHUNK)) belong to this tensor
    float step_size;         // lr / (1 - beta1^t)
    float bc2_sqrt;          // sqrt(1 - beta2^t)
};
struct AdamBatch {
    AdamTensor t[DGS_ADAM_MAX_TENSORS];
    int count;
    float w1, beta2, w2, eps;   // w1 = 1 - beta1, w2 = 1 - beta2 (rounded from double, like torch's scalars)
    float clip;                 // clip_grad_value_ bound, <= 0: off (train.py:204-205)
};
#define ADAM_PER_THREAD 8
#define ADAM_CHUNK (256 * ADAM_PER_THREAD)   // elements per block

// torch.optim.Adam (single-tensor path, amsgrad / weight_decay / maximize off), same operation order:
//   m <- lerp(m, g, 1 - beta1) = m + (1 - beta1) (g - m)
//   v <- (v * beta2) + ((1 - beta2) * g) * g
//   p <- p + (-step_size) * (m / (sqrt(v) / sqrt(bc2) + eps))
// 28 B of HBM traffic per element and nothing else: every thread first issues all of its loads
// (4 x ADAM_PER_THREAD independent requests in flight), then computes, then stores.
__global__ void __launch_bounds__(256) k_adam(const AdamBatch b)
{
    int ti = 0;
#pragma unroll
    for (int k = 1; k < DGS_ADAM_MAX_TENSORS; k++)
        if (k < b.count && (long long)blockIdx.x >= b.t[k].first_block) ti = k;
    const AdamTensor& t = b.t[ti];
    const long long base = ((long long)blockIdx.x - t.first_block) * ADAM_CHUNK + threadIdx.x;
    float g[ADAM_PER_THREAD], m[ADAM_PER_THREAD], v[ADAM_PER_THREAD], p[ADAM_PER_THREAD];
#pragma unroll
    for (int k = 0; k < ADAM_PER_THREAD; k++) {
        const long long i = base + k * 256;
        if (i < t.n) { g[k] = __ldg(t.g + i); m[k] = t.m[i]; v[k] = t.v[i]; p[k] = t.p[i]; }
    }
#pragma unroll
    for (int k = 0; k < ADAM_PER_THREAD; k++) {
        const long long i = base + k * 256;
        if (i < t.n) {
            float gk = g[k];
            if (b.clip > 0.f) gk = fminf(fmaxf(gk, -b.clip), b.clip);
            const float mk = fmaf(b.w1, gk - m[k], m[k]);
            const float vk = fmaf(b.w2 * gk, gk, __fmul_rn(v[k], b.beta2));
            const float denom = __fdiv_rn(sqrtf(vk), t.bc2_sqrt) + b.eps;
            t.m[i] = mk;
            t.v[i] = vk;
            t.p[i] = fmaf(-t.step_size, __fdiv_rn(mk, denom), p[k]);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Densify / prune on the SoA parameter store (reference: scene/gaussian_model.py:300-454 -- prune_points,
// cat_tensors_to_optimizer / densification_postfix, densify_and_clone, densify_and_split).  Every one of those
// operations is "new row r of EVERY per-Gaussian tensor = old row src[r]" with the Adam moments of appended rows
// zeroed; the reference runs it as ~40 torch index / cat launches over the 6 parameter tensors, their 12 moment
// tensors and the 3 statistics vectors.  Here one launch rebuilds all of them: a thread per output float, rows of
// one tensor contiguous across the block so loads and stores are coalesced along the row.
// ---------------------------------------------------------------------------------------
struct GatherTensor { const float* in; float* out; int width; int zero_new; long long first_block; };
struct GatherBatch { GatherTensor t[DGS_GATHER_MAX_TENSORS]; int count; long long n_out; };

__global__ void __launch_bounds__(256) k_rows_gather(const GatherBatch b, const long long* __restrict__ src,
                                                     const unsigned char* __restrict__ carry)
{
    int ti = 0;
#pragma unroll 1
    for (int k = 1; k < b.count; k++)
        if ((long long)blockIdx.x >= b.t[k].first_block) ti = k;
    const GatherTensor& t = b.t[ti];
    const long long i = ((long long)blockIdx.x - t.first_block) * 256 + threadIdx.x;     // output float index
    if (i >= b.n_out * t.width) return;
    const long long row = i / t.width;
    const int c = (int)(i - row * t.width);
    float v = 0.f;
    if (!(t.zero_new && carry != nullptr && carry[row] == 0)) v = __ldg(t.in + src[row] * t.width + c);
    t.out[i] = v;
}

// ---- Mip-Splatting's 3-D filter: the sampling-rate sweep (compute_3D_filter) ------------------------------------
// d_min(g) = min over the cameras that see Gaussian g of its view-space depth z: seen = z > z_near and the projected
// centre within [-0.15, 1.15] x the image.  One thread per Gaussian loops over the cameras, staged in shared memory
// FILTER3D_CHUNK at a time (the three columns of the row-vector world-to-view transform that give x, y, z); the
// result is min-combined with min_depth[g].  A float min is exact: any order or split of the cameras gives the same
// bits.  A camera whose z is not below the running minimum cannot change it and is skipped before the divisions.
struct Filter3dCamera { float fx, fy, cx, cy, u_lo, u_hi, v_lo, v_hi, z_near; };
#define FILTER3D_CHUNK 128

__global__ void __launch_bounds__(256) k_filter3d_depth(long long P, const float* __restrict__ means, int n_cams,
                                                        const float* __restrict__ views, const Filter3dCamera c,
                                                        float* __restrict__ min_depth)
{
    __shared__ float4 cols[FILTER3D_CHUNK][3];   // cols[k][j] = (V[0][j], V[1][j], V[2][j], V[3][j]) of camera k
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float x = 0.f, y = 0.f, z = 0.f;
    if (g < P) { x = means[3 * g]; y = means[3 * g + 1]; z = means[3 * g + 2]; }
    float d = __int_as_float(0x7f800000);
    for (int c0 = 0; c0 < n_cams; c0 += FILTER3D_CHUNK) {
        const int n = min(FILTER3D_CHUNK, n_cams - c0);
        __syncthreads();
        for (int k = threadIdx.x; k < n * 3; k += blockDim.x) {
            const float* v = views + (size_t)(c0 + k / 3) * 16 + k % 3;
            cols[k / 3][k % 3] = make_float4(v[0], v[4], v[8], v[12]);
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < n; k++) {
            const float4 cz = cols[k][2];
            const float pz = fmaf(x, cz.x, fmaf(y, cz.y, fmaf(z, cz.z, cz.w)));
            if (pz > c.z_near && pz < d) {
                const float4 cx = cols[k][0], cy = cols[k][1];
                const float px = fmaf(x, cx.x, fmaf(y, cx.y, fmaf(z, cx.z, cx.w)));
                const float py = fmaf(x, cy.x, fmaf(y, cy.y, fmaf(z, cy.z, cy.w)));
                const float zc = fmaxf(pz, 0.001f);
                const float u = __fadd_rn(__fmul_rn(__fdiv_rn(px, zc), c.fx), c.cx);
                const float v = __fadd_rn(__fmul_rn(__fdiv_rn(py, zc), c.fy), c.cy);
                if (u >= c.u_lo && u <= c.u_hi && v >= c.v_lo && v <= c.v_hi) d = pz;
            }
        }
    }
    if (g < P) min_depth[g] = fminf(min_depth[g], d);
}

template <bool FILTER>
static void activate_forward_t(int P, int M, const float* dc, const float* rest, const float* scaling,
                              const float* rotation, const float* opacity, float lb, int isotropic, float* shs,
                              float* scales, float* rots, float* opac, const float* filter3d, cudaStream_t st)
{
    const size_t total = (size_t)P * 3 * M;
    const size_t want = (total + 255) / 256;
    const int blocks = (int)(want < (size_t)148 * 16 ? want : (size_t)148 * 16);
    StageTimer timer(ST_ACTIVATE_FWD, st, 1);
    k_activate_fwd<FILTER><<<blocks, 256, 0, st>>>(P, M, dc, rest, scaling, rotation, opacity, lb, isotropic, shs,
                                                   scales, rots, opac, filter3d);
}

// filter3d == NULL: the plain activations (FILTER = false)
static int activate_forward(int P, int sh_coeffs, const float* features_dc, const float* features_rest,
                            const float* scaling, const float* rotation, const float* opacity, float scale_lower_bound,
                            int isotropic, float* shs, float* scales, float* rotations, float* opacities,
                            const float* filter3d, void* stream)
{
    if (P < 0 || sh_coeffs < 1) return fail(DGS_ERR_INVALID_ARGUMENT, "dgs_activate_forward: invalid argument");
    if (P == 0) return DGS_OK;
    if (!features_dc || (sh_coeffs > 1 && !features_rest) || !scaling || !rotation || !opacity || !shs ||
        !scales || !rotations || !opacities)
        return fail(DGS_ERR_INVALID_ARGUMENT, "dgs_activate_forward: invalid argument");
    if (filter3d)
        activate_forward_t<true>(P, sh_coeffs, features_dc, features_rest, scaling, rotation, opacity, scale_lower_bound,
                                 isotropic, shs, scales, rotations, opacities, filter3d, (cudaStream_t)stream);
    else
        activate_forward_t<false>(P, sh_coeffs, features_dc, features_rest, scaling, rotation, opacity,
                                  scale_lower_bound, isotropic, shs, scales, rotations, opacities, nullptr,
                                  (cudaStream_t)stream);
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : fail_cuda(e, "dgs_activate_forward"); }
}

template <bool FILTER>
static void activate_backward_t(int P, int M, const float* scaling, const float* rotation, const float* opacity,
                                int isotropic, const float* dsh, const float* dscales, const float* drot,
                                const float* dopac, float* ddc, float* drest, float* dscaling, float* drotation,
                                float* dopacity, float lb, const float* filter3d, cudaStream_t st)
{
    const size_t total = (size_t)P * 3 * M;
    const size_t want = (total + 255) / 256;
    const int blocks = (int)(want < (size_t)148 * 16 ? want : (size_t)148 * 16);
    StageTimer timer(ST_ACTIVATE_BWD, st, 1);
    k_activate_bwd<FILTER><<<blocks, 256, 0, st>>>(P, M, scaling, rotation, opacity, isotropic, dsh, dscales, drot,
                                                   dopac, ddc, drest, dscaling, drotation, dopacity, lb, filter3d);
}

static int activate_backward(int P, int sh_coeffs, const float* scaling, const float* rotation, const float* opacity,
                             int isotropic, const float* dL_dshs, const float* dL_dscales, const float* dL_drotations,
                             const float* dL_dopacities, float* dL_dfeatures_dc, float* dL_dfeatures_rest,
                             float* dL_dscaling, float* dL_drotation, float* dL_dopacity, float scale_lower_bound,
                             const float* filter3d, void* stream)
{
    if (P < 0 || sh_coeffs < 1) return fail(DGS_ERR_INVALID_ARGUMENT, "dgs_activate_backward: invalid argument");
    if (P == 0) return DGS_OK;
    if (!scaling || !rotation || !opacity || !dL_dfeatures_dc || (sh_coeffs > 1 && !dL_dfeatures_rest) ||
        !dL_dscaling || !dL_drotation || !dL_dopacity)
        return fail(DGS_ERR_INVALID_ARGUMENT, "dgs_activate_backward: invalid argument");
    if (filter3d)
        activate_backward_t<true>(P, sh_coeffs, scaling, rotation, opacity, isotropic, dL_dshs, dL_dscales,
                                  dL_drotations, dL_dopacities, dL_dfeatures_dc, dL_dfeatures_rest, dL_dscaling,
                                  dL_drotation, dL_dopacity, scale_lower_bound, filter3d, (cudaStream_t)stream);
    else
        activate_backward_t<false>(P, sh_coeffs, scaling, rotation, opacity, isotropic, dL_dshs, dL_dscales,
                                   dL_drotations, dL_dopacities, dL_dfeatures_dc, dL_dfeatures_rest, dL_dscaling,
                                   dL_drotation, dL_dopacity, 0.f, nullptr, (cudaStream_t)stream);
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : fail_cuda(e, "dgs_activate_backward"); }
}

}  // namespace dgs

extern "C" {

int dgs_rows_gather(int n_tensors, const float* const* in, float* const* out, const int* width, const int* zero_new,
                    int64_t n_out, const int64_t* src_rows, const uint8_t* carry, void* stream)
{
    if (n_tensors < 0 || n_tensors > DGS_GATHER_MAX_TENSORS || n_out < 0)
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_rows_gather: invalid argument");
    if (n_tensors == 0 || n_out == 0) return DGS_OK;
    if (!in || !out || !width || !zero_new || !src_rows) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_rows_gather: null argument");
    dgs::GatherBatch b;
    memset(&b, 0, sizeof(b));
    b.n_out = n_out;
    long long blocks = 0;
    for (int k = 0; k < n_tensors; k++) {
        if (width[k] <= 0 || !in[k] || !out[k]) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_rows_gather: bad tensor");
        dgs::GatherTensor& t = b.t[b.count++];
        t.in = in[k]; t.out = out[k]; t.width = width[k]; t.zero_new = zero_new[k]; t.first_block = blocks;
        blocks += ((long long)n_out * width[k] + 255) / 256;
    }
    if (blocks > 0x7fffffffLL) return dgs::fail(DGS_ERR_UNSUPPORTED, "dgs_rows_gather: size not supported");
    {
        dgs::StageTimer timer(dgs::ST_DENSIFY, (cudaStream_t)stream, 1);
        dgs::k_rows_gather<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(b, (const long long*)src_rows, carry);
    }
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_rows_gather"); }
}

int dgs_activate_forward_filter3d(int P, int sh_coeffs, const float* features_dc, const float* features_rest,
                                  const float* scaling, const float* rotation, const float* opacity,
                                  float scale_lower_bound, int isotropic, float* shs, float* scales, float* rotations,
                                  float* opacities, const float* filter3d, void* stream)
{
    if (!filter3d) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_activate_forward_filter3d: filter3d is NULL");
    return dgs::activate_forward(P, sh_coeffs, features_dc, features_rest, scaling, rotation, opacity, scale_lower_bound,
                                 isotropic, shs, scales, rotations, opacities, filter3d, stream);
}

int dgs_activate_forward(int P, int sh_coeffs, const float* features_dc, const float* features_rest,
                         const float* scaling, const float* rotation, const float* opacity,
                         float scale_lower_bound, int isotropic,
                         float* shs, float* scales, float* rotations, float* opacities, void* stream)
{
    return dgs::activate_forward(P, sh_coeffs, features_dc, features_rest, scaling, rotation, opacity, scale_lower_bound,
                                 isotropic, shs, scales, rotations, opacities, nullptr, stream);
}

int dgs_activate_backward_filter3d(int P, int sh_coeffs, const float* scaling, const float* rotation,
                                   const float* opacity, int isotropic, const float* dL_dshs, const float* dL_dscales,
                                   const float* dL_drotations, const float* dL_dopacities, float* dL_dfeatures_dc,
                                   float* dL_dfeatures_rest, float* dL_dscaling, float* dL_drotation,
                                   float* dL_dopacity, float scale_lower_bound, const float* filter3d, void* stream)
{
    if (!filter3d) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_activate_backward_filter3d: filter3d is NULL");
    return dgs::activate_backward(P, sh_coeffs, scaling, rotation, opacity, isotropic, dL_dshs, dL_dscales,
                                  dL_drotations, dL_dopacities, dL_dfeatures_dc, dL_dfeatures_rest, dL_dscaling,
                                  dL_drotation, dL_dopacity, scale_lower_bound, filter3d, stream);
}

int dgs_activate_backward(int P, int sh_coeffs, const float* scaling, const float* rotation, const float* opacity,
                          int isotropic, const float* dL_dshs, const float* dL_dscales, const float* dL_drotations,
                          const float* dL_dopacities, float* dL_dfeatures_dc, float* dL_dfeatures_rest,
                          float* dL_dscaling, float* dL_drotation, float* dL_dopacity, void* stream)
{
    return dgs::activate_backward(P, sh_coeffs, scaling, rotation, opacity, isotropic, dL_dshs, dL_dscales,
                                  dL_drotations, dL_dopacities, dL_dfeatures_dc, dL_dfeatures_rest, dL_dscaling,
                                  dL_drotation, dL_dopacity, 0.f, nullptr, stream);
}

int dgs_filter3d_depth(int64_t P, const float* means3D, int n_cams, const float* viewmatrices, float focal_x,
                       float focal_y, int width, int height, float z_near, float* min_depth, void* stream)
{
    if (P < 0 || n_cams < 0 || !(focal_x > 0.f) || !(focal_y > 0.f) || width <= 0 || height <= 0)
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_filter3d_depth: invalid argument");
    if (P == 0 || n_cams == 0) return DGS_OK;
    if (!means3D || !viewmatrices || !min_depth)
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_filter3d_depth: null argument");
    const long long blocks = (P + 255) / 256;
    if (blocks > 0x7fffffffLL) return dgs::fail(DGS_ERR_UNSUPPORTED, "dgs_filter3d_depth: size not supported");
    // the screen bounds as a float32 torch comparison rounds them: formed in double, rounded once
    const dgs::Filter3dCamera cam = {focal_x, focal_y, (float)(width / 2.0), (float)(height / 2.0),
                                     (float)(-0.15 * width), (float)(1.15 * width), (float)(-0.15 * height),
                                     (float)(1.15 * height), z_near};
    {
        dgs::StageTimer timer(dgs::ST_DENSIFY, (cudaStream_t)stream, 1);   // store maintenance: counted with densify
        dgs::k_filter3d_depth<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(P, means3D, n_cams, viewmatrices,
                                                                                   cam, min_depth);
    }
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_filter3d_depth"); }
}

int dgs_adam_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                  float* const* exp_avg_sq, const int64_t* numel, const double* lr, const int64_t* step,
                  double beta1, double beta2, double eps, double clip_grad_value, void* stream)
{
    if (n_tensors < 0 || n_tensors > DGS_ADAM_MAX_TENSORS) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_adam_step: invalid argument");
    if (n_tensors == 0) return DGS_OK;
    if (!params || !grads || !exp_avg || !exp_avg_sq || !numel || !lr || !step) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_adam_step: invalid argument");
    dgs::AdamBatch b;
    memset(&b, 0, sizeof(b));
    // scalars are formed in double and rounded once, as torch does with its Python floats
    b.w1 = (float)(1.0 - beta1); b.beta2 = (float)beta2; b.w2 = (float)(1.0 - beta2); b.eps = (float)eps;
    b.clip = (float)clip_grad_value;
    long long blocks = 0;
    for (int k = 0; k < n_tensors; k++) {
        if (numel[k] < 0 || step[k] < 1) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_adam_step: invalid argument");
        if (numel[k] == 0) continue;
        if (!params[k] || !grads[k] || !exp_avg[k] || !exp_avg_sq[k]) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_adam_step: invalid argument");
        dgs::AdamTensor& t = b.t[b.count++];
        t.p = params[k]; t.g = grads[k]; t.m = exp_avg[k]; t.v = exp_avg_sq[k];
        t.n = numel[k];
        t.first_block = blocks;
        const double bc1 = 1.0 - pow(beta1, (double)step[k]);
        const double bc2 = 1.0 - pow(beta2, (double)step[k]);
        t.step_size = (float)(lr[k] / bc1);
        t.bc2_sqrt = (float)sqrt(bc2);
        blocks += (numel[k] + ADAM_CHUNK - 1) / ADAM_CHUNK;
    }
    if (blocks == 0) return DGS_OK;
    if (blocks > 0x7fffffffLL) return dgs::fail(DGS_ERR_UNSUPPORTED, "dgs_adam_step: size not supported");
    {
        dgs::StageTimer timer(dgs::ST_ADAM, (cudaStream_t)stream, 1);
        dgs::k_adam<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(b);
    }
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_adam_step"); }
}

}  // extern "C"
