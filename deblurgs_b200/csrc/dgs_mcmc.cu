// 3DGS-MCMC densification (Kheradmand et al., NeurIPS 2024; gsplat `MCMCStrategy`) on the SoA parameter store.
//
//   k_mcmc_relocation  per relocation entry r: the source's new opacity and scaling after it is split N[r] ways,
//                      o' = 1 - (1 - o)^(1/N) and s' = o / D(o', N) * s (the paper's relocation formula), into a
//                      scratch record.  D is evaluated in fp64 in closed form (below), not as the original's fp32
//                      double loop.
//   k_rows_relocate    in-place multi-tensor row scatter, the in-place counterpart of k_rows_gather: dst[r] <- src[r]
//                      for copied tensors, the scratch values at dst[r] and src[r] for opacity / scaling, zeros at
//                      dst[r] and src[r] for the Adam moments and the densification statistics.  No tensor changes
//                      size or storage, so a captured CUDA graph of the training step stays valid.
//   k_mcmc_noise       the per-step SGLD move xyz += Sigma eps gate(o) step_scale, eps ~ N(0, I3) from an in-kernel
//                      Philox4x32-10 keyed by the seed with counter (g, step): a pure function of (seed, step, g).
#include "dgs_b200.h"
#include "dgs_internal.cuh"

#include <cmath>
#include <cstring>

namespace dgs {

#define MCMC_N_MAX 51
#define MCMC_MIN_OPACITY 0.0050000004f   // the smallest float above 0.005 (0x3BA3D70B)

// D(o', N) = sum_{i=1..N} sum_{k=0..i-1} C(i-1,k) (-1)^k o'^(k+1) / sqrt(k+1).  Summing over i first with the
// hockey-stick identity sum_{i=k+1..N} C(i-1,k) = C(N,k+1) leaves one alternating sum,
//   D = sum_{j=1..N} (-1)^(j-1) C(N,j) o'^j / sqrt(j),
// whose largest term is ~ (1 + o')^N: at most ~2e5 for the o' this formula is fed (o' = 1 - (1 - o)^(1/N), o < 1), so
// fp64 keeps ~10 significant digits where the original fp32 loop keeps ~2.  C(N,j) <= C(51,25) ~ 2.5e14 is exact in
// fp64, and so is every partial product C(N,j-1) (N-j+1) below.
__host__ __device__ inline void mcmc_relocation_coeffs(double o, int N, double& o_new, double& c)
{
    N = N < 1 ? 1 : (N > MCMC_N_MAX ? MCMC_N_MAX : N);
    o = o < 0.0 ? 0.0 : (o > 1.0 ? 1.0 : o);
    o_new = -expm1(log1p(-o) / N);          // 1 - (1 - o)^(1/N) without the cancellation for small o
    double binom = 1.0, pw = 1.0, d = 0.0;
    for (int j = 1; j <= N; j++) {
        binom = binom * (double)(N - j + 1) / (double)j;
        pw *= o_new;
        const double t = binom * pw / sqrt((double)j);
        d += (j & 1) ? t : -t;
    }
    c = o / d;
}

// scratch record of entry r: {raw opacity, raw scaling x, y, z} of the relocated source (and its copies)
__global__ void __launch_bounds__(256) k_mcmc_relocation(long long n, const long long* __restrict__ src,
                                                         const int* __restrict__ ratio,
                                                         const float* __restrict__ opacity,
                                                         const float* __restrict__ scaling, float scale_lb,
                                                         int isotropic, float4* __restrict__ scratch)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const long long s = src[r];
    double o_new, c;
    // the store's opacity activation is a clamp: the raw value is the activated one
    mcmc_relocation_coeffs((double)opacity[s], ratio[r], o_new, c);
    // stored opacity clamped to [0.005, 1 - 2^-23], the lower bound being the smallest float above 0.005 (the float
    // nearest to 0.005 lies below it, and a relocated Gaussian must not be dead by the `<= 0.005` rule); the scale
    // coefficient uses the unclamped o', as the original does
    const float op = fmaxf((float)fmin(o_new, 1.0 - 1.0 / 8388608.0), MCMC_MIN_OPACITY);
    float out[3];
    const double lb = (double)scale_lb;
    for (int i = 0; i < 3; i++) {
        const double raw = (double)scaling[3 * s + (isotropic ? 0 : i)];
        if (scale_lb == 0.f)
            out[i] = (float)(raw + log(c));                                  // log(c exp(raw)), exact
        else
            out[i] = (float)log(fmax(c * (exp(raw) + lb) - lb, 0.001));      // LowerBoundLog inverse, as split
    }
    scratch[r] = make_float4(op, out[0], out[1], out[2]);
}

struct RelocTensor { float* t; int width; int kind; long long first_block; };
struct RelocBatch { RelocTensor t[DGS_GATHER_MAX_TENSORS]; int count; long long n; };

// Race-free by construction: opacity / scaling values come from the scratch record only; destination rows are disjoint
// from each other and from every source row (PRECONDITION: sources are drawn from live rows, destinations are the dead
// or appended ones); entries that share a source write identical bits there, because the caller gives all of them the
// same ratio N = 1 + (number of entries sharing the source), hence the same scratch record.
__global__ void __launch_bounds__(256) k_rows_relocate(const RelocBatch b, const long long* __restrict__ dst,
                                                       const long long* __restrict__ src,
                                                       const float4* __restrict__ scratch)
{
    int ti = 0;
#pragma unroll 1
    for (int k = 1; k < b.count; k++)
        if ((long long)blockIdx.x >= b.t[k].first_block) ti = k;
    const RelocTensor& t = b.t[ti];
    const long long i = ((long long)blockIdx.x - t.first_block) * 256 + threadIdx.x;   // (entry, float) index
    if (i >= b.n * t.width) return;
    const long long r = i / t.width;
    const int c = (int)(i - r * t.width);
    const long long d = dst[r] * t.width + c, s = src[r] * t.width + c;
    switch (t.kind) {
    case DGS_RELOCATE_COPY:
        t.t[d] = t.t[s];
        break;
    case DGS_RELOCATE_OPACITY: {
        const float v = scratch[r].x;
        t.t[d] = v; t.t[s] = v;
        break;
    }
    case DGS_RELOCATE_SCALING: {
        const float4 q = scratch[r];
        const float v = c == 0 ? q.y : (c == 1 ? q.z : q.w);
        t.t[d] = v; t.t[s] = v;
        break;
    }
    default:   // DGS_RELOCATE_ZERO
        t.t[d] = 0.f; t.t[s] = 0.f;
        break;
    }
}

// ---- SGLD noise --------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11; Random123's constants): 4 x 32-bit counter, 2 x 32-bit key.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int round = 0; round < 10; round++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}

// (0, 1): the top 24 bits, centred in their interval (never 0, so the log below is finite)
__device__ __forceinline__ float mcmc_uniform(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// eps ~ N(0, I3) of Gaussian g at `step`: Box-Muller on two pairs of the 4 Philox outputs; the fourth normal is unused
__device__ __forceinline__ float3 mcmc_normals(unsigned long long seed, long long step, long long g)
{
    const uint4 x = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)((unsigned long long)g >> 32), (uint32_t)step,
                                             (uint32_t)((unsigned long long)step >> 32)),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float r0 = sqrtf(-2.f * logf(mcmc_uniform(x.x))), r1 = sqrtf(-2.f * logf(mcmc_uniform(x.z)));
    float s0, c0, s1, c1;
    sincospif(2.f * mcmc_uniform(x.y), &s0, &c0);
    sincospif(2.f * mcmc_uniform(x.w), &s1, &c1);
    return make_float3(r0 * c0, r0 * s0, r1 * c1);
}

// xyz += Sigma eps gate step_scale, Sigma = R diag(s^2) R^T with s = exp(raw) + lb (isotropic: column 0) and R =
// build_rotation(normalize(q)) (w first), gate = 1 / (1 + exp(-k ((1 - clamp(o, 0, 1)) - x0))).  56 B per Gaussian.
__global__ void __launch_bounds__(256) k_mcmc_noise(long long P, float* __restrict__ xyz,
                                                    const float* __restrict__ scaling,
                                                    const float* __restrict__ rotation,
                                                    const float* __restrict__ opacity, float scale_lb, int isotropic,
                                                    float step_scale, float k, float x0, unsigned long long seed,
                                                    long long step)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= P) return;
    const float o = fminf(fmaxf(opacity[g], 0.f), 1.f);
    const float gate = 1.f / (1.f + expf(-k * ((1.f - o) - x0)));
    const float e0 = expf(scaling[3 * g]);
    const float s0 = e0 + scale_lb, s1 = (isotropic ? e0 : expf(scaling[3 * g + 1])) + scale_lb,
                s2 = (isotropic ? e0 : expf(scaling[3 * g + 2])) + scale_lb;
    const float4 q = reinterpret_cast<const float4*>(rotation)[g];
    const float nq = fmaxf(sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w), 1e-12f);
    const float w = q.x / nq, x = q.y / nq, y = q.z / nq, z = q.w / nq;
    const float R00 = 1.f - 2.f * (y * y + z * z), R01 = 2.f * (x * y - w * z), R02 = 2.f * (x * z + w * y);
    const float R10 = 2.f * (x * y + w * z), R11 = 1.f - 2.f * (x * x + z * z), R12 = 2.f * (y * z - w * x);
    const float R20 = 2.f * (x * z - w * y), R21 = 2.f * (y * z + w * x), R22 = 1.f - 2.f * (x * x + y * y);
    const float3 e = mcmc_normals(seed, step, g);
    // v = diag(s^2) R^T eps, then R v
    const float f = gate * step_scale;
    const float v0 = s0 * s0 * (R00 * e.x + R10 * e.y + R20 * e.z) * f;
    const float v1 = s1 * s1 * (R01 * e.x + R11 * e.y + R21 * e.z) * f;
    const float v2 = s2 * s2 * (R02 * e.x + R12 * e.y + R22 * e.z) * f;
    xyz[3 * g] += R00 * v0 + R01 * v1 + R02 * v2;
    xyz[3 * g + 1] += R10 * v0 + R11 * v1 + R12 * v2;
    xyz[3 * g + 2] += R20 * v0 + R21 * v1 + R22 * v2;
}

__global__ void __launch_bounds__(256) k_mcmc_normals(long long P, unsigned long long seed, long long step,
                                                      float* __restrict__ out)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= P) return;
    const float3 e = mcmc_normals(seed, step, g);
    out[3 * g] = e.x; out[3 * g + 1] = e.y; out[3 * g + 2] = e.z;
}

}  // namespace dgs

extern "C" {

size_t dgs_mcmc_relocate_scratch_bytes(int64_t n)
{
    return n > 0 ? (size_t)n * sizeof(float4) : 0;
}

int dgs_mcmc_relocate(int n_tensors, float* const* tensors, const int* width, const int* kind, int64_t n,
                      const int64_t* dst_rows, const int64_t* src_rows, const int32_t* ratio, float scale_lower_bound,
                      int isotropic, void* scratch, void* stream)
{
    if (n_tensors < 0 || n_tensors > DGS_GATHER_MAX_TENSORS || n < 0 || !(scale_lower_bound >= 0.f))
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_relocate: invalid argument");
    if (n == 0) return DGS_OK;
    if (!tensors || !width || !kind || !dst_rows || !src_rows || !ratio || !scratch)
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_relocate: null argument");
    dgs::RelocBatch b;
    memset(&b, 0, sizeof(b));
    b.n = n;
    const float* opacity = nullptr;
    const float* scaling = nullptr;
    long long blocks = 0;
    for (int k = 0; k < n_tensors; k++) {
        if (width[k] <= 0 || !tensors[k] || kind[k] < DGS_RELOCATE_COPY || kind[k] > DGS_RELOCATE_ZERO)
            return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_relocate: bad tensor");
        if (kind[k] == DGS_RELOCATE_OPACITY) {
            if (opacity || width[k] != 1) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_relocate: needs one opacity tensor of width 1");
            opacity = tensors[k];
        }
        if (kind[k] == DGS_RELOCATE_SCALING) {
            if (scaling || width[k] != 3) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_relocate: needs one scaling tensor of width 3");
            scaling = tensors[k];
        }
        dgs::RelocTensor& t = b.t[b.count++];
        t.t = tensors[k]; t.width = width[k]; t.kind = kind[k]; t.first_block = blocks;
        blocks += ((long long)n * width[k] + 255) / 256;
    }
    if (!opacity || !scaling)
        return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_relocate: needs one opacity and one scaling tensor");
    if (blocks > 0x7fffffffLL) return dgs::fail(DGS_ERR_UNSUPPORTED, "dgs_mcmc_relocate: size not supported");
    {
        dgs::StageTimer timer(dgs::ST_DENSIFY, (cudaStream_t)stream, 2);
        dgs::k_mcmc_relocation<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
            n, (const long long*)src_rows, ratio, opacity, scaling, scale_lower_bound, isotropic, (float4*)scratch);
        dgs::k_rows_relocate<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            b, (const long long*)dst_rows, (const long long*)src_rows, (const float4*)scratch);
    }
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_mcmc_relocate"); }
}

int dgs_mcmc_noise(int64_t P, float* xyz, const float* scaling, const float* rotation, const float* opacity,
                   float scale_lower_bound, int isotropic, float step_scale, float k, float x0, uint64_t seed,
                   int64_t step, void* stream)
{
    if (P < 0 || step < 0) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_noise: invalid argument");
    if (P == 0) return DGS_OK;
    if (!xyz || !scaling || !rotation || !opacity) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_mcmc_noise: null argument");
    const long long blocks = (P + 255) / 256;
    if (blocks > 0x7fffffffLL) return dgs::fail(DGS_ERR_UNSUPPORTED, "dgs_mcmc_noise: size not supported");
    {
        dgs::StageTimer timer(dgs::ST_ADAM, (cudaStream_t)stream, 1);   // the optimizer's position update
        dgs::k_mcmc_noise<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            P, xyz, scaling, rotation, opacity, scale_lower_bound, isotropic, step_scale, k, x0, seed, step);
    }
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_mcmc_noise"); }
}

int dgs_debug_mcmc_normals(int64_t P, uint64_t seed, int64_t step, float* out, void* stream)
{
    if (P < 0 || step < 0) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_debug_mcmc_normals: invalid argument");
    if (P == 0) return DGS_OK;
    if (!out) return dgs::fail(DGS_ERR_INVALID_ARGUMENT, "dgs_debug_mcmc_normals: null argument");
    const long long blocks = (P + 255) / 256;
    if (blocks > 0x7fffffffLL) return dgs::fail(DGS_ERR_UNSUPPORTED, "dgs_debug_mcmc_normals: size not supported");
    dgs::k_mcmc_normals<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(P, seed, step, out);
    { const cudaError_t e = cudaGetLastError(); return e == cudaSuccess ? DGS_OK : dgs::fail_cuda(e, "dgs_debug_mcmc_normals"); }
}

}  // extern "C"
