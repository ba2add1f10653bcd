// C-ABI of libdgs_b200.so (see include/dgs_b200.h for the contract and the reference
// interfaces each entry point replaces).  Host-side orchestration only: buffer carving,
// kernel launches, all on the caller's stream (no library kernels: scan and sorts are dgs_binning.cu).
#include "dgs_b200.h"
#include "dgs_internal.cuh"

#include <atomic>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

namespace dgs {

static thread_local std::string g_last_error;

int fail(int code, const char* what)
{
    g_last_error = what;
    return code;
}
int fail_cuda(cudaError_t e, const char* where)
{
    g_last_error = std::string(where) + ": " + cudaGetErrorString(e);
    return DGS_ERR_CUDA;
}
#define DGS_CUDA(call, where)                                   \
    do {                                                        \
        cudaError_t e__ = (call);                               \
        if (e__ != cudaSuccess) return fail_cuda(e__, where);   \
    } while (0)

// ---- stage profiling ---------------------------------------------------------------------
// Process-wide measurement state; every access is under g_prof_mutex (host threads may drive different
// devices / streams through the library concurrently), the launch counter is atomic.
struct ProfRec { cudaEvent_t a, b; int stage; };
static std::mutex g_prof_mutex;
static std::atomic<bool> g_prof_on{false};
static std::vector<ProfRec> g_prof;
static std::vector<cudaEvent_t> g_event_pool;
static double g_stage_ms[ST_COUNT];
static long long g_stage_calls[ST_COUNT];
static std::atomic<long long> g_own_launches{0};
static const char* kStageNames[ST_COUNT] = {"preprocess_fwd", "depth_sort", "scan", "tile_sort",
                                            "render_fwd", "blur_mean", "bwd_memset", "render_bwd",
                                            "preprocess_bwd", "pose_fwd", "pose_bwd", "activate_fwd",
                                            "activate_bwd", "adam", "densify"};
static cudaEvent_t get_event()   // g_prof_mutex held
{
    if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
StageTimer::StageTimer(int stage, cudaStream_t st_, int own_kernels) : st(st_), on(false)
{
    g_own_launches.fetch_add(own_kernels, std::memory_order_relaxed);
    if (!g_prof_on.load(std::memory_order_relaxed)) return;
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    ProfRec r;
    r.a = get_event(); r.b = get_event(); r.stage = stage;
    cudaEventRecord(r.a, st);
    g_prof.push_back(r);
    end_event = r.b;
    on = true;
}
StageTimer::~StageTimer()
{
    if (on) cudaEventRecord(end_event, st);   // the event handle is ours until dgs_profile_read recycles it
}

static int bits_for(uint32_t n)  // number of bits needed to hold values 0..n-1 (>= 1)
{
    int b = 1;
    while ((1ull << b) < n) b++;
    return b;
}
// The reference sorts bits [0, 32 + getHigherMsb(tiles)) (rasterizer_impl.cu:35-50,306):
// getHigherMsb(n) = position of the MSB of n, plus one.
static int ref_tile_bits(uint32_t tiles)
{
    int b = 0;
    while (tiles >> b) b++;
    return b < 1 ? 1 : b;
}

GeomLayout geom_layout(size_t P, size_t F)
{
    GeomLayout L;
    const size_t N = P * F;
    const size_t Pp = (P + SORT_CHUNK - 1) / SORT_CHUNK * SORT_CHUNK;
    const size_t Np = Pp * F;
    const size_t nb = (P + 1023) / 1024;          // blocks of the entry gather / offsets kernels
    L.stride = Pp;
    size_t o = 0;
    // read by the backward (depends on P and F only)
    L.geo0 = o; o = align_up(o + N * sizeof(float4));
    L.geo1 = o; o = align_up(o + N * sizeof(float4));
    L.geo2 = o; o = align_up(o + N * sizeof(float4));
    L.cmask = o; o = align_up(o + N);
    // binning state
    L.status = o; o = align_up(o + sizeof(BinStatus));
    L.seg_start = o; o = align_up(o + (F + 1) * sizeof(uint32_t));
    L.seg_len = o; o = align_up(o + (F + 1) * sizeof(uint32_t));
    L.seg_adj = o; o = align_up(o + (F + 1) * sizeof(uint32_t));
    L.seg_total = o; o = align_up(o + (F + 1) * sizeof(unsigned long long));
    L.ticket = o; o = align_up(o + sizeof(uint32_t));
    L.rect = o; o = align_up(o + N * sizeof(uint2));
    L.dkeys = o; o = align_up(o + N * sizeof(uint32_t));
    L.keys_a = o; o = align_up(o + Np * sizeof(uint32_t));
    L.keys_b = o; o = align_up(o + Np * sizeof(uint32_t));
    L.vals_a = o; o = align_up(o + Np * sizeof(uint32_t));
    L.vals_b = o; o = align_up(o + Np * sizeof(uint32_t));
    L.cnt_sorted = L.keys_a;                      // the depth sort is finished when the scan stage runs
    L.off = L.keys_b;
    L.rec = o; o = align_up(o + Np * sizeof(uint2));
    L.block_sums = o; o = align_up(o + F * nb * sizeof(unsigned long long));
    L.block_excl = o; o = align_up(o + F * nb * sizeof(uint32_t));
    L.sort_scratch = o; o = align_up(o + sort_scratch_bytes((uint32_t)(Np / SORT_CHUNK), 8));
    L.total = o + 128;
    return L;
}
// capacity: slots of the duplicate arrays (rounded up to the sort's chunk here)
BinLayout bin_layout(size_t capacity, size_t F, size_t tiles)
{
    BinLayout L;
    (void)F;
    const size_t C = (capacity + SORT_CHUNK - 1) / SORT_CHUNK * SORT_CHUNK;
    L.capacity = C;
    L.passes = sort_pass_plan(bits_for((uint32_t)(tiles > 1 ? tiles : 1)), &L.bits);
    const size_t chunks = C / SORT_CHUNK;
    size_t o = 128;                       // BinHeader
    L.point_list = o; o = align_up(o + C * sizeof(uint32_t));
    L.wmask = o; o = align_up(o + C);
    L.keys_a = o; if (L.passes >= 2) o = align_up(o + C * sizeof(uint32_t));
    L.vals_a = o; if (L.passes >= 2) o = align_up(o + C * sizeof(uint32_t));
    L.keys_b = o; if (L.passes >= 3) o = align_up(o + C * sizeof(uint32_t));
    L.vals_b = o; if (L.passes >= 3) o = align_up(o + C * sizeof(uint32_t));
    L.chunk_first = o; o = align_up(o + (chunks + 1) * sizeof(uint2));
    L.sort_scratch = o; o = align_up(o + sort_scratch_bytes((uint32_t)chunks, L.bits));
    L.total = o + 128;
    return L;
}
ImgLayout img_layout(size_t F, size_t tiles, size_t pixels)
{
    ImgLayout L;
    size_t o = 0;
    L.ranges = o; o = align_up(o + F * tiles * sizeof(uint2));
    L.final_T = o; o = align_up(o + F * pixels * sizeof(float));
    L.n_contrib = o; o = align_up(o + F * pixels * sizeof(uint32_t));
    L.total = o + 128;
    return L;
}

static char* aligned128(char* p) { return (char*)(((uintptr_t)p + 127) & ~(uintptr_t)127); }

static int fill_params(FwdParams& p, int P, int F, int M, const float* background, int W, int H,
                       const float* means3D, const float* shs, const float* colors_precomp,
                       const float* opacities, const float* scales, float scale_modifier,
                       const float* rotations, const float* cov3D_precomp, const float* view,
                       const float* proj, const float* campos, float tan_fovx, float tan_fovy,
                       float z_near, float z_far, int prefiltered, int use_sigmoid)
{
    if (P < 0 || F < 0 || W < 0 || H < 0) return fail(DGS_ERR_INVALID_ARGUMENT, "negative size");
    if (F > DGS_MAX_SUBFRAMES) return fail(DGS_ERR_INVALID_ARGUMENT, "too many sub-frames (max 256)");
    if (P > 0 && F > 0) {
        if ((shs == nullptr) == (colors_precomp == nullptr))
            return fail(DGS_ERR_INVALID_ARGUMENT, "provide exactly one of SHs or precomputed colors");
        const bool has_sr = scales != nullptr && rotations != nullptr;
        if (has_sr == (cov3D_precomp != nullptr) || ((scales != nullptr) != (rotations != nullptr)))
            return fail(DGS_ERR_INVALID_ARGUMENT,
                        "provide exactly one of scale/rotation pair or precomputed 3D covariance");
        if (!means3D || !opacities || !view || !proj || !background)
            return fail(DGS_ERR_INVALID_ARGUMENT, "null required input");
        if (shs != nullptr && campos == nullptr) return fail(DGS_ERR_INVALID_ARGUMENT, "campos required with SHs");
    }
    p.P = P; p.F = F; p.M = M; p.W = W; p.H = H;
    p.tiles_x = (W + DGS_TILE_X - 1) / DGS_TILE_X;
    p.tiles_y = (H + DGS_TILE_Y - 1) / DGS_TILE_Y;
    p.tile_bits = ref_tile_bits((uint32_t)(p.tiles_x * p.tiles_y));
    p.tan_fovx = tan_fovx; p.tan_fovy = tan_fovy;
    p.focal_y = H / (2.0f * tan_fovy);
    p.focal_x = W / (2.0f * tan_fovx);
    p.scale_modifier = scale_modifier;
    p.z_near = z_near; p.z_far = z_far;
    p.prefiltered = prefiltered; p.use_sigmoid = use_sigmoid;
    p.means3D = means3D; p.shs = shs; p.colors_precomp = colors_precomp; p.opacities = opacities;
    p.scales = scales; p.rotations = rotations; p.cov3D_precomp = cov3D_precomp;
    p.view = view; p.proj = proj; p.campos = campos; p.background = background;
    return DGS_OK;
}

static void bind_geom(FwdParams& p, char* geom, const GeomLayout& G)
{
    p.geo0 = (float4*)(geom + G.geo0);
    p.geo1 = (float4*)(geom + G.geo1);
    p.geo2 = (float4*)(geom + G.geo2);
    p.cmask = (uint8_t*)(geom + G.cmask);
    p.rect = (uint2*)(geom + G.rect);
    p.dkeys = (uint32_t*)(geom + G.dkeys);
}
static BinState bind_bin_state(char* geom, const GeomLayout& G)
{
    BinState b;
    b.stride = (uint32_t)G.stride;
    b.order = (const uint32_t*)(geom + G.vals_b);
    b.cnt_sorted = (uint32_t*)(geom + G.cnt_sorted);
    b.off = (uint32_t*)(geom + G.off);
    b.rec = (uint2*)(geom + G.rec);
    b.block_sums = (unsigned long long*)(geom + G.block_sums);
    b.block_excl = (uint32_t*)(geom + G.block_excl);
    b.status = (BinStatus*)(geom + G.status);
    b.seg_start = (uint32_t*)(geom + G.seg_start);
    b.seg_len = (uint32_t*)(geom + G.seg_len);
    b.seg_adj = (uint32_t*)(geom + G.seg_adj);
    b.seg_total = (unsigned long long*)(geom + G.seg_total);
    b.ticket = (uint32_t*)(geom + G.ticket);
    return b;
}

__global__ void k_write_u64(unsigned long long* dst, unsigned long long v) { *dst = v; }

// Pinned host landing zone of the asynchronous status read-back (one per host thread) and its event.
struct StatusMailbox {
    BinStatus* host = nullptr;
    cudaEvent_t ev[64] = {};
    cudaEvent_t event()   // of the current device (an event belongs to the device it was created on)
    {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
        if (!host && cudaHostAlloc((void**)&host, sizeof(BinStatus), cudaHostAllocPortable) != cudaSuccess) return nullptr;
        if (!ev[dev] && cudaEventCreateWithFlags(&ev[dev], cudaEventDisableTiming) != cudaSuccess) return nullptr;
        return ev[dev];
    }
};
static thread_local StatusMailbox g_mailbox;

}  // namespace dgs

using namespace dgs;

extern "C" {

const char* dgs_last_error(void) { return g_last_error.c_str(); }
int dgs_version(void) { return 100; }
int dgs_compiled_arch(void) { return 1000; }

int dgs_key_bits(int width, int height, int F, int* tile_bits, int* subframe_bits)
{
    const int tx = (width + DGS_TILE_X - 1) / DGS_TILE_X, ty = (height + DGS_TILE_Y - 1) / DGS_TILE_Y;
    if (tile_bits) *tile_bits = ref_tile_bits((uint32_t)(tx * ty));
    if (subframe_bits) *subframe_bits = F > 1 ? bits_for((uint32_t)F) : 0;
    return DGS_OK;
}

/* Shared implementation of dgs_blur_forward / dgs_blur_forward_hint / dgs_blur_forward_aa / dgs_blur_forward_contrib.
 *   contrib_wsum != NULL  the blend is the scoring kernel (contribution scores accumulated into contrib_wsum / _wmax).
 *   capacity_hint == 0  exact mode: the host waits for D after the scan stage (one synchronisation, like the
 *                       reference's rasterizer_impl.cu:287) and sizes the binning buffer from it.
 *   capacity_hint  > 0  speculative mode: the binning buffer is sized from the hint and every kernel of the view is
 *                       enqueued without waiting; D and an overflow flag stay on the device.  With num_rendered !=
 *                       NULL the host then waits for the small status read-back that was enqueued right after the
 *                       scan stage (the GPU keeps working on the blend meanwhile) and, if the hint was too small,
 *                       re-runs the tile sort and the blend with the exact size.  With num_rendered == NULL nothing
 *                       is waited for (CUDA-graph capturable); query dgs_blur_forward_status afterwards. */
static int blur_forward_impl(
    dgs_alloc_fn geom_alloc, void* geom_ctx, dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t capacity_hint, int64_t* num_rendered, int antialiasing, void* stream,
    unsigned long long* contrib_wsum = nullptr, uint32_t* contrib_wmax = nullptr)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (antialiasing != 0 && antialiasing != 1) return fail(DGS_ERR_INVALID_ARGUMENT, "antialiasing must be 0 or 1");
    FwdParams p;
    memset(&p, 0, sizeof(p));
    int rc = fill_params(p, P, F, sh_coeffs, background, width, height, means3D, shs, colors_precomp,
                         opacities, scales, scale_modifier, rotations, cov3D_precomp, viewmatrix,
                         projmatrix, campos, tan_fovx, tan_fovy, z_near, z_far, prefiltered, use_sigmoid);
    if (rc != DGS_OK) return rc;
    if (!geom_alloc || !binning_alloc || !image_alloc) return fail(DGS_ERR_INVALID_ARGUMENT, "null allocator");
    if (F > 0 && width * height > 0 && (!out_color || !out_depth)) return fail(DGS_ERR_INVALID_ARGUMENT, "null output");
    if (shs != nullptr && (sh_degree < 0 || sh_degree > 3 || sh_coeffs < (sh_degree + 1) * (sh_degree + 1)))
        return fail(DGS_ERR_INVALID_ARGUMENT, "bad SH degree / coefficient count");
    if (P > 0 && F > 0 && !radii) return fail(DGS_ERR_INVALID_ARGUMENT, "null radii");
    if (capacity_hint < 0) return fail(DGS_ERR_INVALID_ARGUMENT, "negative binning capacity");
    p.radii = radii;

    const size_t N = (size_t)P * F;
    const size_t tiles = (size_t)p.tiles_x * p.tiles_y;
    const size_t pixels = (size_t)width * height;
    const GeomLayout G = geom_layout((size_t)P, (size_t)F);
    if (G.stride * (size_t)F >= (1ull << 32)) return fail(DGS_ERR_UNSUPPORTED, "P*F must be < 2^32");
    // the packed tile rectangle of the duplicate generator holds 10 bits per coordinate
    if (p.tiles_x > 1024 || p.tiles_y > 1024) return fail(DGS_ERR_UNSUPPORTED, "image larger than 16384 pixels per side");

    const ImgLayout I = img_layout(F, tiles, pixels);
    char* geom = geom_alloc(geom_ctx, G.total);
    char* img = image_alloc(image_ctx, I.total);
    if (!geom || !img) return fail(DGS_ERR_ALLOC, "state buffer allocation failed");
    geom = aligned128(geom);
    img = aligned128(img);
    bind_geom(p, geom, G);
    const BinState bs = bind_bin_state(geom, G);
    uint2* ranges = (uint2*)(img + I.ranges);
    float* final_T = (float*)(img + I.final_T);
    uint32_t* n_contrib = (uint32_t*)(img + I.n_contrib);
    uint32_t* ticket = (uint32_t*)(geom + G.ticket);

    int64_t D = 0;
    const size_t pad = (size_t)F * SORT_CHUNK;          // every sub-frame's list is padded to the sort's chunk
    size_t capacity = capacity_hint > 0 ? (size_t)capacity_hint + pad : 0;
    cudaEvent_t ev = nullptr;
    const bool speculative = capacity_hint > 0;
    if (N > 0) {
        DGS_CUDA(cudaMemsetAsync(geom + G.status, 0, G.rect - G.status, st), "status memset");   // status .. ticket
        { StageTimer t(ST_PREPROCESS_FWD, st, 1); launch_preprocess_fwd(p, sh_degree, antialiasing != 0, st); }
        {
            // stage 1: depth order of the Gaussians of every sub-frame (segmented sort on the 32 depth bits)
            StageTimer t(ST_DEPTH_SORT, st, 12);
            const SortScratch sc = bind_sort_scratch(geom + G.sort_scratch, (uint32_t)(G.stride * F / SORT_CHUNK), 8, ticket);
            sort_uniform_u32(F, (uint32_t)P, (uint32_t)G.stride, p.dkeys, (uint32_t*)(geom + G.keys_a),
                             (uint32_t*)(geom + G.vals_a), (uint32_t*)(geom + G.keys_b), (uint32_t*)(geom + G.vals_b),
                             sc, 32, st);
        }
        if (!speculative) {
            // exact mode: D is needed on the host to size the binning buffer
            { StageTimer t(ST_SCAN, st, 2); launch_entry_scan(p, bs, ~0ull, st); }
            BinStatus h;
            DGS_CUDA(cudaMemcpyAsync(&h, bs.status, sizeof(h), cudaMemcpyDeviceToHost, st), "num_rendered copy");
            DGS_CUDA(cudaStreamSynchronize(st), "num_rendered sync");
            if (h.padded + SORT_CHUNK >= (1ull << 32))
                return fail(DGS_ERR_UNSUPPORTED, "more than 2^32 (Gaussian, tile) duplicates in one batched view");
            D = (int64_t)h.num_rendered;
            capacity = (size_t)h.padded;
            // the status words were computed against an unlimited capacity: overflow = 0, n_chunks = padded / chunk
        } else {
            if (capacity + SORT_CHUNK >= (1ull << 32)) capacity = (1ull << 32) - 2 * SORT_CHUNK;
            { StageTimer t(ST_SCAN, st, 2); launch_entry_scan(p, bs, (unsigned long long)(capacity / SORT_CHUNK * SORT_CHUNK), st); }
            if (num_rendered) {
                ev = g_mailbox.event();
                if (!ev) return fail(DGS_ERR_CUDA, "status mailbox allocation failed");
                DGS_CUDA(cudaMemcpyAsync(g_mailbox.host, bs.status, sizeof(BinStatus), cudaMemcpyDeviceToHost, st), "status copy");
                DGS_CUDA(cudaEventRecord(ev, st), "status event");
            }
        }
    }

    char* bin = nullptr;
    for (int attempt = 0; attempt < 2; attempt++) {
        const BinLayout B = bin_layout(capacity, F, tiles);
        bin = binning_alloc(binning_ctx, B.total);
        if (!bin) return fail(DGS_ERR_ALLOC, "binning buffer allocation failed");
        bin = aligned128(bin);
        uint32_t* point_list = (uint32_t*)(bin + B.point_list);
        uint8_t* wmask = (uint8_t*)(bin + B.wmask);
        uint2* chunk_tab = (uint2*)(bin + B.chunk_first);
        {   // header: where the backward finds the capacity-dependent arrays (a memset node: capture-safe, no host source)
            static_assert(sizeof(BinHeader) == 8, "header is one 64-bit word");
            DGS_CUDA(cudaMemsetAsync(bin, 0, 128, st), "header memset");
            k_write_u64<<<1, 1, 0, st>>>((unsigned long long*)bin, (unsigned long long)B.wmask);
        }

        if (F > 0 && tiles > 0)
            DGS_CUDA(cudaMemsetAsync(ranges, 0, (size_t)F * tiles * sizeof(uint2), st), "ranges memset");
        if (N > 0 && B.capacity > 0) {
            { StageTimer t(ST_SCAN, st, 1); launch_entry_offsets(p, bs, chunk_tab, st); }
            // stage 2: duplicates generated from the depth-ordered entries and sorted by tile id inside every
            // sub-frame's segment; the last pass writes point_list and the per-tile ranges
            StageTimer t(ST_TILE_SORT, st, 3 * B.passes);
            SegTable tab;
            memset(&tab, 0, sizeof(tab));
            tab.seg_start = bs.seg_start; tab.seg_len = bs.seg_len; tab.seg_adj = bs.seg_adj;
            tab.n_chunks = &bs.status->n_chunks; tab.chunk_tab = chunk_tab; tab.nseg = F;
            GenParams gp;
            gp.off = bs.off; gp.rec = bs.rec;
            gp.entries_per_seg = (uint32_t)P; gp.entry_stride = bs.stride; gp.tiles_x = p.tiles_x;
            const uint32_t max_chunks = (uint32_t)(B.capacity / SORT_CHUNK);
            const SortScratch sc = bind_sort_scratch(bin + B.sort_scratch, max_chunks, B.bits, ticket);
            uint32_t* ka = (uint32_t*)(bin + B.keys_a); uint32_t* va = (uint32_t*)(bin + B.vals_a);
            uint32_t* kb = (uint32_t*)(bin + B.keys_b); uint32_t* vb = (uint32_t*)(bin + B.vals_b);
            const uint32_t* kin = nullptr; const uint32_t* vin = nullptr;
            for (int pass = 0; pass < B.passes; pass++) {
                const bool last = pass == B.passes - 1;
                uint32_t* ko = last ? nullptr : (pass == 0 ? ka : kb);
                uint32_t* vo = last ? point_list : (pass == 0 ? va : vb);
                sort_pass(tab, max_chunks, B.bits, B.bits * pass, kin, vin, 0, ko, vo, sc, pass == 0 ? &gp : nullptr,
                          last ? ranges : nullptr, (uint32_t)tiles, st);
                kin = ko; vin = vo;
            }
        }
        if (F > 0 && pixels > 0) {
            { StageTimer t(ST_RENDER_FWD, st, 1); launch_render_fwd(p, ranges, point_list, wmask, final_T, n_contrib, out_color, out_depth, contrib_wsum, contrib_wmax, st); }
            if (out_blur) { StageTimer t(ST_BLUR_MEAN, st, 1); launch_blur_mean(out_color, F, 3 * pixels, blur_denominator, out_blur, st); }
        }
        DGS_CUDA(cudaGetLastError(), "forward launch");
        if (!ev) break;
        // speculative mode with a host-visible result: the status was copied right after the scan stage
        DGS_CUDA(cudaEventSynchronize(ev), "status wait");
        const BinStatus h = *g_mailbox.host;
        ev = nullptr;
        D = (int64_t)h.num_rendered;
        if (!h.overflow) break;
        if (h.padded + SORT_CHUNK >= (1ull << 32))
            return fail(DGS_ERR_UNSUPPORTED, "more than 2^32 (Gaussian, tile) duplicates in one batched view");
        // the hint was too small: the tile sort did nothing.  Redo the scan stage against the exact size.
        capacity = (size_t)h.padded;
        { StageTimer t(ST_SCAN, st, 2); launch_entry_scan(p, bs, ~0ull, st); }
    }
    if (num_rendered) *num_rendered = D;
    return DGS_OK;
}

int dgs_blur_forward(
    dgs_alloc_fn geom_alloc, void* geom_ctx, dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t* num_rendered, void* stream)
{
    return blur_forward_impl(geom_alloc, geom_ctx, binning_alloc, binning_ctx, image_alloc, image_ctx, P, F, sh_degree,
                             sh_coeffs, background, width, height, means3D, shs, colors_precomp, opacities, scales,
                             scale_modifier, rotations, cov3D_precomp, viewmatrix, projmatrix, campos, tan_fovx,
                             tan_fovy, z_near, z_far, prefiltered, use_sigmoid, out_color, out_depth, radii, out_blur,
                             blur_denominator, 0, num_rendered, 0, stream);
}

int dgs_blur_forward_hint(
    dgs_alloc_fn geom_alloc, void* geom_ctx, dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t binning_capacity, int64_t* num_rendered, void* stream)
{
    return blur_forward_impl(geom_alloc, geom_ctx, binning_alloc, binning_ctx, image_alloc, image_ctx, P, F, sh_degree,
                             sh_coeffs, background, width, height, means3D, shs, colors_precomp, opacities, scales,
                             scale_modifier, rotations, cov3D_precomp, viewmatrix, projmatrix, campos, tan_fovx,
                             tan_fovy, z_near, z_far, prefiltered, use_sigmoid, out_color, out_depth, radii, out_blur,
                             blur_denominator, binning_capacity, num_rendered, 0, stream);
}

int dgs_blur_forward_aa(
    dgs_alloc_fn geom_alloc, void* geom_ctx, dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t binning_capacity, int64_t* num_rendered, int antialiasing, void* stream)
{
    return blur_forward_impl(geom_alloc, geom_ctx, binning_alloc, binning_ctx, image_alloc, image_ctx, P, F, sh_degree,
                             sh_coeffs, background, width, height, means3D, shs, colors_precomp, opacities, scales,
                             scale_modifier, rotations, cov3D_precomp, viewmatrix, projmatrix, campos, tan_fovx,
                             tan_fovy, z_near, z_far, prefiltered, use_sigmoid, out_color, out_depth, radii, out_blur,
                             blur_denominator, binning_capacity, num_rendered, antialiasing, stream);
}

int dgs_blur_forward_contrib(
    dgs_alloc_fn geom_alloc, void* geom_ctx, dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t binning_capacity, int64_t* num_rendered, int antialiasing,
    uint64_t* contrib_wsum, uint32_t* contrib_wmax, void* stream)
{
    if (P > 0 && F > 0 && (!contrib_wsum || !contrib_wmax))
        return fail(DGS_ERR_INVALID_ARGUMENT, "null contribution score array");
    return blur_forward_impl(geom_alloc, geom_ctx, binning_alloc, binning_ctx, image_alloc, image_ctx, P, F, sh_degree,
                             sh_coeffs, background, width, height, means3D, shs, colors_precomp, opacities, scales,
                             scale_modifier, rotations, cov3D_precomp, viewmatrix, projmatrix, campos, tan_fovx,
                             tan_fovy, z_near, z_far, prefiltered, use_sigmoid, out_color, out_depth, radii, out_blur,
                             blur_denominator, binning_capacity, num_rendered, antialiasing, stream,
                             (unsigned long long*)contrib_wsum, contrib_wmax);
}

size_t dgs_blur_forward_status_offset(int P, int F)
{
    return geom_layout((size_t)(P > 0 ? P : 0), (size_t)(F > 0 ? F : 0)).status;
}

int dgs_blur_forward_status(const char* geom_buffer, int P, int F, int64_t* num_rendered, int* overflow, void* stream)
{
    if (num_rendered) *num_rendered = 0;
    if (overflow) *overflow = 0;
    if ((size_t)P * (size_t)F == 0) return DGS_OK;
    if (!geom_buffer) return fail(DGS_ERR_INVALID_ARGUMENT, "null geometry buffer");
    const GeomLayout G = geom_layout((size_t)P, (size_t)F);
    BinStatus h;
    DGS_CUDA(cudaMemcpyAsync(&h, aligned128((char*)geom_buffer) + G.status, sizeof(h), cudaMemcpyDeviceToHost,
                             (cudaStream_t)stream), "status copy");
    DGS_CUDA(cudaStreamSynchronize((cudaStream_t)stream), "status sync");
    if (num_rendered) *num_rendered = (int64_t)h.num_rendered;
    if (overflow) *overflow = (int)h.overflow;
    return DGS_OK;
}

size_t dgs_blur_backward_scratch_bytes(int P, int F)
{
    const size_t N = (size_t)P * (size_t)F;
    return align_up(N * 12 * sizeof(float)) + align_up((size_t)F * 32 * sizeof(double)) + 256;
}

// Shared implementation of dgs_blur_backward_range / dgs_blur_backward_range_aa.
static int blur_backward_impl(
    int P, int F, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth, const float* dL_dblur, float blur_denominator,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, float* densify_stats,
    int64_t g_begin, int64_t g_end, int stages, int antialiasing, void* stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (antialiasing != 0 && antialiasing != 1) return fail(DGS_ERR_INVALID_ARGUMENT, "antialiasing must be 0 or 1");
    if (g_begin < 0 || g_end > P || g_begin > g_end) return fail(DGS_ERR_INVALID_ARGUMENT, "bad Gaussian range");
    BwdParams b;
    memset(&b, 0, sizeof(b));
    int rc = fill_params(b.f, P, F, sh_coeffs, background, width, height, means3D, shs, colors_precomp,
                         opacities, scales, scale_modifier, rotations, cov3D_precomp, viewmatrix,
                         projmatrix, campos, tan_fovx, tan_fovy, z_near, z_far, 0, use_sigmoid);
    if (rc != DGS_OK) return rc;
    if (F == 0) return DGS_OK;
    if (!dL_dviewmatrix || !dL_dprojmatrix) return fail(DGS_ERR_INVALID_ARGUMENT, "null pose gradient output");
    if (P == 0) {
        if (stages & DGS_BWD_FINISH) {
            DGS_CUDA(cudaMemsetAsync(dL_dviewmatrix, 0, (size_t)F * 16 * sizeof(float), st), "memset");
            DGS_CUDA(cudaMemsetAsync(dL_dprojmatrix, 0, (size_t)F * 16 * sizeof(float), st), "memset");
        }
        return DGS_OK;
    }
    if (!geom_buffer || !binning_buffer || !image_buffer || !scratch || !radii)
        return fail(DGS_ERR_INVALID_ARGUMENT, "null state buffer");
    if (!dL_dmeans3D || !dL_dopacity) return fail(DGS_ERR_INVALID_ARGUMENT, "null gradient output");
    if (P >= (1 << 27)) return fail(DGS_ERR_UNSUPPORTED, "the blend backward packs the Gaussian index into 27 bits: P must be < 2^27");
    if (shs && !dL_dsh) return fail(DGS_ERR_INVALID_ARGUMENT, "null dL_dsh");
    if (scales && (!dL_dscales || !dL_drotations)) return fail(DGS_ERR_INVALID_ARGUMENT, "null dL_dscales/dL_drotations");

    const size_t N = (size_t)P * F;
    const size_t tiles = (size_t)b.f.tiles_x * b.f.tiles_y;
    const size_t pixels = (size_t)width * height;
    const GeomLayout G = geom_layout((size_t)P, (size_t)F);
    const ImgLayout I = img_layout(F, tiles, pixels);
    char* geom = aligned128((char*)geom_buffer);
    char* img = aligned128((char*)image_buffer);
    char* bin = aligned128((char*)binning_buffer);
    bind_geom(b.f, geom, G);
    b.f.radii = (int*)radii;
    b.ranges = (const uint2*)(img + I.ranges);
    b.final_T = (const float*)(img + I.final_T);
    b.n_contrib = (const uint32_t*)(img + I.n_contrib);
    b.bin_header = (const BinHeader*)bin;
    b.point_list = (const uint32_t*)(bin + 128);   // point_list follows the 128-B header of the binning buffer
    b.dL_dpix = dL_dpix;
    b.dL_dpixdepth = dL_dpixdepth;
    b.dL_dblur = dL_dblur;
    b.blur_denominator = blur_denominator;
    char* sc = aligned128(scratch);
    b.g0 = (float4*)sc;
    b.g1 = b.g0 + N;
    b.g2 = b.g1 + N;
    b.pose_acc = (double*)(sc + align_up(N * 12 * sizeof(float)));
    b.dL_dmeans2D = dL_dmeans2D; b.dL_dmeans3D = dL_dmeans3D; b.dL_dsh = dL_dsh; b.dL_dopacity = dL_dopacity;
    b.dL_dscales = dL_dscales; b.dL_drotations = dL_drotations;
    b.dL_dcolors_precomp = dL_dcolors_precomp; b.dL_dcov3D_precomp = dL_dcov3D_precomp;
    b.dL_dview = dL_dviewmatrix; b.dL_dproj = dL_dprojmatrix;
    b.densify_stats = densify_stats;
    b.g_begin = (int)g_begin;
    b.g_end = (int)g_end;

    if (stages & DGS_BWD_BLEND) {
        {
            StageTimer t(ST_BWD_MEMSET, st, 0);
            DGS_CUDA(cudaMemsetAsync(sc, 0, align_up(N * 12 * sizeof(float)) + (size_t)F * 32 * sizeof(double), st), "grad memset");
        }
        // num_rendered is informational (the lists are delimited by the per-tile ranges); < 0 = unknown (speculative forward)
        if (num_rendered != 0 && pixels > 0) { StageTimer t(ST_RENDER_BWD, st, 1); launch_render_bwd(b, st); }
    }
    if ((stages & DGS_BWD_GAUSSIANS) && g_end > g_begin) {
        StageTimer t(ST_PREPROCESS_BWD, st, colors_precomp ? 1 : 2);
        launch_preprocess_bwd(b, sh_degree, antialiasing != 0, st);
    }
    if (stages & DGS_BWD_FINISH) { StageTimer t(ST_PREPROCESS_BWD, st, 1); launch_pose_finalize(b, st); }
    DGS_CUDA(cudaGetLastError(), "backward launch");
    return DGS_OK;
}

int dgs_blur_backward_range(
    int P, int F, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth, const float* dL_dblur, float blur_denominator,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, float* densify_stats,
    int64_t g_begin, int64_t g_end, int stages, void* stream)
{
    return blur_backward_impl(P, F, sh_degree, sh_coeffs, num_rendered, background, width, height, means3D, shs,
                              colors_precomp, opacities, scales, scale_modifier, rotations, cov3D_precomp, viewmatrix,
                              projmatrix, campos, tan_fovx, tan_fovy, z_near, z_far, use_sigmoid, radii, geom_buffer,
                              binning_buffer, image_buffer, dL_dpix, dL_dpixdepth, dL_dblur, blur_denominator, scratch,
                              dL_dmeans2D, dL_dmeans3D, dL_dsh, dL_dopacity, dL_dscales, dL_drotations,
                              dL_dcolors_precomp, dL_dcov3D_precomp, dL_dviewmatrix, dL_dprojmatrix, densify_stats,
                              g_begin, g_end, stages, 0, stream);
}

int dgs_blur_backward_range_aa(
    int P, int F, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth, const float* dL_dblur, float blur_denominator,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, float* densify_stats,
    int64_t g_begin, int64_t g_end, int stages, int antialiasing, void* stream)
{
    return blur_backward_impl(P, F, sh_degree, sh_coeffs, num_rendered, background, width, height, means3D, shs,
                              colors_precomp, opacities, scales, scale_modifier, rotations, cov3D_precomp, viewmatrix,
                              projmatrix, campos, tan_fovx, tan_fovy, z_near, z_far, use_sigmoid, radii, geom_buffer,
                              binning_buffer, image_buffer, dL_dpix, dL_dpixdepth, dL_dblur, blur_denominator, scratch,
                              dL_dmeans2D, dL_dmeans3D, dL_dsh, dL_dopacity, dL_dscales, dL_drotations,
                              dL_dcolors_precomp, dL_dcov3D_precomp, dL_dviewmatrix, dL_dprojmatrix, densify_stats,
                              g_begin, g_end, stages, antialiasing, stream);
}

int dgs_blur_backward(
    int P, int F, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth, const float* dL_dblur, float blur_denominator,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, float* densify_stats, void* stream)
{
    return dgs_blur_backward_range(P, F, sh_degree, sh_coeffs, num_rendered, background, width, height, means3D, shs,
                                   colors_precomp, opacities, scales, scale_modifier, rotations, cov3D_precomp,
                                   viewmatrix, projmatrix, campos, tan_fovx, tan_fovy, z_near, z_far, use_sigmoid, radii,
                                   geom_buffer, binning_buffer, image_buffer, dL_dpix, dL_dpixdepth, dL_dblur,
                                   blur_denominator, scratch, dL_dmeans2D, dL_dmeans3D, dL_dsh, dL_dopacity, dL_dscales,
                                   dL_drotations, dL_dcolors_precomp, dL_dcov3D_precomp, dL_dviewmatrix, dL_dprojmatrix,
                                   densify_stats, 0, P, DGS_BWD_ALL, stream);
}

int dgs_forward(
    dgs_alloc_fn geom_alloc, void* geom_ctx, dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    int64_t* num_rendered, void* stream)
{
    return dgs_blur_forward(geom_alloc, geom_ctx, binning_alloc, binning_ctx, image_alloc, image_ctx, P, 1,
                            sh_degree, sh_coeffs, background, width, height, means3D, shs, colors_precomp,
                            opacities, scales, scale_modifier, rotations, cov3D_precomp, viewmatrix,
                            projmatrix, campos, tan_fovx, tan_fovy, z_near, z_far, prefiltered, use_sigmoid,
                            out_color, out_depth, radii, nullptr, 1.0f, num_rendered, stream);
}

int dgs_backward(
    int P, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, void* stream)
{
    return dgs_blur_backward(P, 1, sh_degree, sh_coeffs, num_rendered, background, width, height, means3D, shs,
                             colors_precomp, opacities, scales, scale_modifier, rotations, cov3D_precomp,
                             viewmatrix, projmatrix, campos, tan_fovx, tan_fovy, z_near, z_far, use_sigmoid,
                             radii, geom_buffer, binning_buffer, image_buffer, dL_dpix, dL_dpixdepth, nullptr, 1.0f, scratch,
                             dL_dmeans2D, dL_dmeans3D, dL_dsh, dL_dopacity, dL_dscales, dL_drotations,
                             dL_dcolors_precomp, dL_dcov3D_precomp, dL_dviewmatrix, dL_dprojmatrix, nullptr, stream);
}

// ---- profiling / measurement ------------------------------------------------------------
int dgs_profile_enable(int on)
{
    g_prof_on.store(on != 0);
    return DGS_OK;
}
int dgs_profile_num_stages(void) { return ST_COUNT; }
const char* dgs_profile_stage_name(int i) { return (i >= 0 && i < ST_COUNT) ? kStageNames[i] : ""; }
int dgs_profile_read(double* ms, int64_t* calls, int n, int reset)
{
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    for (auto& r : g_prof) {
        float t = 0.f;
        cudaError_t e = cudaEventSynchronize(r.b);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&t, r.a, r.b);
        if (e != cudaSuccess) return fail_cuda(e, "profile read");
        g_stage_ms[r.stage] += t;
        g_stage_calls[r.stage] += 1;
        g_event_pool.push_back(r.a);
        g_event_pool.push_back(r.b);
    }
    g_prof.clear();
    for (int i = 0; i < n && i < ST_COUNT; i++) {
        if (ms) ms[i] = g_stage_ms[i];
        if (calls) calls[i] = g_stage_calls[i];
    }
    if (reset) {
        for (int i = 0; i < ST_COUNT; i++) { g_stage_ms[i] = 0.0; g_stage_calls[i] = 0; }
    }
    return DGS_OK;
}
int64_t dgs_launch_count(int reset)
{
    return reset ? g_own_launches.exchange(0) : g_own_launches.load();
}

int dgs_debug_workload(const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
                       int P, int F, int width, int height, int64_t num_rendered, uint64_t* out_dev,
                       void* stream)
{
    if (F == 0 || P == 0) return DGS_OK;
    if (!geom_buffer || !binning_buffer || !image_buffer || !out_dev) return fail(DGS_ERR_INVALID_ARGUMENT, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    FwdParams p;
    memset(&p, 0, sizeof(p));
    p.P = P; p.F = F; p.W = width; p.H = height;
    p.tiles_x = (width + DGS_TILE_X - 1) / DGS_TILE_X;
    p.tiles_y = (height + DGS_TILE_Y - 1) / DGS_TILE_Y;
    const size_t tiles = (size_t)p.tiles_x * p.tiles_y, pixels = (size_t)width * height;
    (void)num_rendered;
    const GeomLayout G = geom_layout((size_t)P, (size_t)F);
    const ImgLayout I = img_layout(F, tiles, pixels);
    char* geom = aligned128((char*)geom_buffer);
    char* img = aligned128((char*)image_buffer);
    char* bin = aligned128((char*)binning_buffer);
    bind_geom(p, geom, G);
    DGS_CUDA(cudaMemsetAsync(out_dev, 0, 3 * sizeof(uint64_t), st), "workload memset");
    launch_workload(p, (const uint2*)(img + I.ranges), (const uint32_t*)(bin + 128),
                    (const uint32_t*)(img + I.n_contrib), (unsigned long long*)out_dev, st);
    DGS_CUDA(cudaGetLastError(), "workload");
    return DGS_OK;
}

// ---- debug / parity accessors ---------------------------------------------------------
__global__ void k_debug_geometry(int P, int F, uint32_t stride, const float4* g0, const float4* g1, const float4* g2,
                                 const uint2* rect, const uint32_t* off, float* depths,
                                 float* means2D, float* conic_opacity, float* rgb, float* clamped,
                                 uint32_t* tiles_out, uint32_t* offsets_out)
{
    const size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= (size_t)P * F) return;
    const uint2 r = rect[n];
    const uint32_t cnt = (r.y & 0xFFFFu) * (r.y >> 16);
    const bool vis = cnt > 0;
    float4 a = make_float4(0, 0, 0, 0), b = a, c = a;
    if (vis) { a = g0[n]; b = g1[n]; c = g2[n]; }
    if (depths) depths[n] = a.z;
    if (means2D) { means2D[2 * n] = a.x; means2D[2 * n + 1] = a.y; }
    if (conic_opacity) { conic_opacity[4 * n] = b.x; conic_opacity[4 * n + 1] = b.y; conic_opacity[4 * n + 2] = b.z; conic_opacity[4 * n + 3] = b.w; }
    if (rgb) { rgb[3 * n] = c.x; rgb[3 * n + 1] = c.y; rgb[3 * n + 2] = c.z; }
    if (clamped) {
        const unsigned m = vis ? __float_as_uint(c.w) : 0u;
        clamped[3 * n] = (m & 1u) ? 1.f : 0.f; clamped[3 * n + 1] = (m & 2u) ? 1.f : 0.f; clamped[3 * n + 2] = (m & 4u) ? 1.f : 0.f;
    }
    if (tiles_out) tiles_out[n] = cnt;
    if (offsets_out) { const size_t s = n / P, i = n - s * P; offsets_out[n] = off[s * stride + i]; }
}

int dgs_debug_geometry(const char* geom_buffer, int P, int F, float* depths, float* means2D,
                       float* conic_opacity, float* rgb, float* clamped, uint32_t* tiles_touched,
                       uint32_t* point_offsets, void* stream)
{
    const size_t N = (size_t)P * F;
    if (N == 0) return DGS_OK;
    if (!geom_buffer) return fail(DGS_ERR_INVALID_ARGUMENT, "null geometry buffer");
    const GeomLayout G = geom_layout((size_t)P, (size_t)F);
    char* geom = aligned128((char*)geom_buffer);
    k_debug_geometry<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        P, F, (uint32_t)G.stride, (const float4*)(geom + G.geo0), (const float4*)(geom + G.geo1),
        (const float4*)(geom + G.geo2), (const uint2*)(geom + G.rect), (const uint32_t*)(geom + G.off), depths,
        means2D, conic_opacity, rgb, clamped, tiles_touched, point_offsets);
    DGS_CUDA(cudaGetLastError(), "debug geometry");
    return DGS_OK;
}

int dgs_debug_binning(const char* geom_buffer, const char* binning_buffer, const char* image_buffer, int P, int F,
                      int width, int height, int64_t num_rendered, uint64_t* keys, uint32_t* point_list,
                      uint32_t* ranges, void* stream)
{
    if (F <= 0 || P <= 0) return DGS_OK;
    if (!binning_buffer || !geom_buffer || !image_buffer) return fail(DGS_ERR_INVALID_ARGUMENT, "null state buffer");
    (void)num_rendered;
    const int tx = (width + DGS_TILE_X - 1) / DGS_TILE_X, ty = (height + DGS_TILE_Y - 1) / DGS_TILE_Y;
    const size_t tiles = (size_t)tx * ty, pixels = (size_t)width * height;
    const GeomLayout G = geom_layout((size_t)P, (size_t)F);
    const ImgLayout I = img_layout(F, tiles, pixels);
    char* geom = aligned128((char*)geom_buffer);
    char* img = aligned128((char*)image_buffer);
    char* bin = aligned128((char*)binning_buffer);
    launch_debug_lists(P, F, (int)tiles, ref_tile_bits((uint32_t)tiles), (const uint2*)(img + I.ranges),
                       (const uint32_t*)(bin + 128), (const float4*)(geom + G.geo0), (const uint32_t*)(geom + G.seg_start),
                       (const uint32_t*)(geom + G.seg_adj), keys, point_list, ranges, (cudaStream_t)stream);
    DGS_CUDA(cudaGetLastError(), "debug lists");
    return DGS_OK;
}

int dgs_debug_image(const char* image_buffer, int F, int width, int height, float* final_T, uint32_t* n_contrib,
                    void* stream)
{
    const size_t tiles = (size_t)((width + DGS_TILE_X - 1) / DGS_TILE_X) * ((height + DGS_TILE_Y - 1) / DGS_TILE_Y);
    const size_t pixels = (size_t)width * height;
    if (F == 0) return DGS_OK;
    if (!image_buffer) return fail(DGS_ERR_INVALID_ARGUMENT, "null image buffer");
    const ImgLayout I = img_layout(F, tiles, pixels);
    char* img = aligned128((char*)image_buffer);
    cudaStream_t st = (cudaStream_t)stream;
    if (final_T && pixels) DGS_CUDA(cudaMemcpyAsync(final_T, img + I.final_T, F * pixels * sizeof(float), cudaMemcpyDeviceToDevice, st), "copy T");
    if (n_contrib && pixels) DGS_CUDA(cudaMemcpyAsync(n_contrib, img + I.n_contrib, F * pixels * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st), "copy n_contrib");
    return DGS_OK;
}

/* Debug entry of the segmented radix sort (dgs_binning.cu): sorts keys [nseg][len] (device, u32) on their low
 * key_bits bits, segment by segment, stable; writes the sorted keys and the source index inside the segment.
 * scratch: dgs_debug_sort_scratch_bytes(nseg, len). */
size_t dgs_debug_sort_scratch_bytes(int nseg, int64_t len)
{
    const size_t stride = ((size_t)len + SORT_CHUNK - 1) / SORT_CHUNK * SORT_CHUNK;
    const size_t Np = stride * (size_t)(nseg > 0 ? nseg : 0);
    return 4 * align_up(Np * 4) + sort_scratch_bytes((uint32_t)(Np / SORT_CHUNK), 8) + 512;
}
__global__ void k_debug_unpad(int nseg, uint32_t len, uint32_t stride, const uint32_t* a, const uint32_t* b,
                              uint32_t* out_a, uint32_t* out_b)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)nseg * len) return;
    const size_t s = i / len, j = i - s * len;
    if (out_a) out_a[i] = a[s * stride + j];
    if (out_b) out_b[i] = b[s * stride + j];
}
int dgs_debug_sort(int nseg, int64_t len, int key_bits, const uint32_t* keys, uint32_t* keys_sorted,
                   uint32_t* index_sorted, char* scratch, void* stream)
{
    if (nseg <= 0 || len <= 0) return DGS_OK;
    if (!keys || !scratch || key_bits < 1 || key_bits > 32) return fail(DGS_ERR_INVALID_ARGUMENT, "dgs_debug_sort: invalid argument");
    const size_t stride = ((size_t)len + SORT_CHUNK - 1) / SORT_CHUNK * SORT_CHUNK;
    const size_t Np = stride * (size_t)nseg;
    if (Np >= (1ull << 32)) return fail(DGS_ERR_UNSUPPORTED, "dgs_debug_sort: too many items");
    cudaStream_t st = (cudaStream_t)stream;
    char* sc = aligned128(scratch);
    uint32_t* ka = (uint32_t*)sc; sc += align_up(Np * 4);
    uint32_t* kb = (uint32_t*)sc; sc += align_up(Np * 4);
    uint32_t* va = (uint32_t*)sc; sc += align_up(Np * 4);
    uint32_t* vb = (uint32_t*)sc; sc += align_up(Np * 4);
    uint32_t* ticket = (uint32_t*)sc; sc += 128;
    DGS_CUDA(cudaMemsetAsync(ticket, 0, sizeof(uint32_t), st), "ticket memset");
    const SortScratch ss = bind_sort_scratch(sc, (uint32_t)(Np / SORT_CHUNK), 8, ticket);
    sort_uniform_u32(nseg, (uint32_t)len, (uint32_t)stride, keys, ka, va, kb, vb, ss, key_bits, st);
    const size_t n = (size_t)nseg * len;
    k_debug_unpad<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(nseg, (uint32_t)len, (uint32_t)stride, kb, vb, keys_sorted, index_sorted);
    DGS_CUDA(cudaGetLastError(), "dgs_debug_sort");
    return DGS_OK;
}

// ---- FP32 FMA throughput of this GPU (denominator of the blend kernels' roofline) -------------------
__global__ void __launch_bounds__(256) k_fma_peak(float* sink, int iters, float a, float b)
{
    // 16 independent FMA chains per thread: enough ILP to fill the FP32 pipes from 8 warps per scheduler
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = (float)(threadIdx.x + i) * 1e-3f;
    for (int k = 0; k < iters; k++) {
#pragma unroll
        for (int i = 0; i < 16; i++) v[i] = fmaf(v[i], a, b);
    }
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 16; i++) acc += v[i];
    if (acc == 123.456f) sink[0] = acc;   // never true: keeps the chains alive
}

int dgs_measure_fp32_peak(double* tflops, double* sm_clock_mhz_hint, void* stream)
{
    if (!tflops) return fail(DGS_ERR_INVALID_ARGUMENT, "dgs_measure_fp32_peak: null output");
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 0;
    DGS_CUDA(cudaGetDevice(&dev), "get device");
    DGS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev), "sm count");
    float* sink = nullptr;
    DGS_CUDA(cudaMalloc(&sink, sizeof(float)), "fp32 peak sink");
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int blocks = sms * 8, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {         // first repetitions warm the clocks up
        cudaEventRecord(e0, st);
        k_fma_peak<<<blocks, 256, 0, st>>>(sink, iters, 1.0000001f, 1e-7f);
        cudaEventRecord(e1, st);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double flops = 2.0 * 16.0 * (double)iters * 256.0 * (double)blocks;
        if (ms > 0.f && flops / (ms * 1e-3) / 1e12 > best) best = flops / (ms * 1e-3) / 1e12;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    DGS_CUDA(cudaGetLastError(), "fp32 peak");
    *tflops = best;
    if (sm_clock_mhz_hint) *sm_clock_mhz_hint = best * 1e12 / (2.0 * 128.0 * sms) / 1e6;   // clock this rate implies
    return DGS_OK;
}

// ---- mark_visible ----------------------------------------------------------------------
__global__ void k_mark_visible(int P, const float* __restrict__ means, const float* __restrict__ V,
                               uint8_t* __restrict__ present)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= P) return;
    const float3 m = {means[3 * g], means[3 * g + 1], means[3 * g + 2]};
    const float3 pv = xform_point_4x3(m, V);
    present[g] = pv.z > 0.2f ? 1 : 0;
}

int dgs_mark_visible(int P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                     uint8_t* present, void* stream)
{
    (void)projmatrix;
    if (P == 0) return DGS_OK;
    if (!means3D || !viewmatrix || !present) return fail(DGS_ERR_INVALID_ARGUMENT, "null argument");
    k_mark_visible<<<(P + 255) / 256, 256, 0, (cudaStream_t)stream>>>(P, means3D, viewmatrix, present);
    DGS_CUDA(cudaGetLastError(), "mark_visible");
    return DGS_OK;
}

}  // extern "C"
