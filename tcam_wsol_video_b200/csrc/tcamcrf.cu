// tcamcrf.cu -- kernels + C ABI of libtcamcrf.so (see include/tcamcrf.h).
//
// Pipeline for one chunk of frames (all launches on the caller's stream, chained by programmatic dependent
// launch: each kernel runs what does not depend on its predecessor ahead of griddepcontrol.wait):
//
//   -- lattice stages (need the images only) --
//   prepare_kernel       clears the primary tier of the frame tables (and the overflow
//                        tier only if the previous use spilled into it), zeroes counters
//   build_kernel<D>      per pixel: features -> embedding -> d+1 packed keys ->
//                        warp-deduplicated (runs of equal keys) insert into the frame's two-tier table
//                        (all first probes issued before any is consumed);
//                        warp-aggregated allocation of dense, per-frame-contiguous ids
//   neighbour_kernel<D>  per (vertex, axis): two table lookups (n1, n2), one 8-byte store of the link
//                        pair; the axis-0 item clears the vertex' value row
//   -- value stages (any number of times on one lattice) --
//   vertex_init_kernel   (host path / lattice re-use only) zeroes the value rows again
//   splat_kernel<V>      per pixel: entry -> dense id (kept, tagged, for slice and later splats), vector
//                        RED.ADD of w * seg[k] into values[id][0..Kp)
//   blur_kernel<V> x(d+1) per (vertex, k-vector): new = old + 0.5*(old[n1]+old[n2])
//   slice_kernel<V>      per pixel: AS[k] = sum_r (bary_r*alpha) * values[id_r][k];
//                        block partial of seg . AS; the last block folds the partials into the loss
//
// Reference functions replaced: bilateralfilter_batch / bilateralfilter /
// initializePermutohedral (bilateralfilter.cpp:4-55), the colour variants
// (colorbilateralfilter.cpp:4-54), Permutohedral::init / compute
// (permutohedral.cpp:115-297, 507-572), DenseCRFLossFunction.forward/backward
// arithmetic (dlib/crf/dense_crf_loss.py:56-74).
//
// Differences from the reference that are deliberate:
//   * all K classes go through the lattice in one pass (values[v][K]); the
//     reference runs K scalar passes (bilateralfilter.cpp:31-37) -- per channel
//     the arithmetic is identical;
//   * vertex ids are a relabelling of the reference's first-seen order;
//   * splat accumulates with floating-point RED atomics, so the summation order
//     inside one vertex differs from the reference's pixel order (parity budget
//     rel 1e-4; measured ~1e-6).  Blur and slice round exactly like the SSE code.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <type_traits>
#include <utility>
#include <vector>

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>   // header-only; ranges cost a pointer check when no tool is attached

#include "../../include/tcamcrf.h"
#include "lattice.cuh"
#include "seed.cuh"

namespace tcamcrf {

// ---------------------------------------------------------------------------
// error handling
// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return fail(TCAMCRF_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                    \
    } while (0)

// ---------------------------------------------------------------------------
// tuning knobs: read from the environment ONCE (first use), changeable at run time through
// tcamcrf_set_tuning() -- no getenv on the call path.  0 / -1 = library default.
// ---------------------------------------------------------------------------
struct Tuning {
    int dense = -1;           // TCAMCRF_DENSE: force the row-cooperative splat on (1) / off (0); -1 = density hint
    int build_dedup = -1;     // TCAMCRF_BUILD_DEDUP: force the shared-memory dedup build on (1) / off (0); -1 = density hint
    int himg_sections = 0;    // TCAMCRF_HIMG_SECTIONS: sections of a chunk on the host-frames path
    int host_groups = 0;      // TCAMCRF_HOST_GROUPS: value-stage groups per chunk on the host-pointer path
    int host_section0 = 0;    // TCAMCRF_HOST_SECTION0: frames of the first section on the host-pointer path
    int host_trace = 0;       // TCAMCRF_HOST_TRACE: print the timeline of host_run
    int host_grow = 0;        // TCAMCRF_HOST_GROW: each section of the host-pointer path is this many times the one before
};
static int env_int(const char *name, int dflt)
{
    const char *v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}
static Tuning &tuning()
{
    static Tuning t = [] {
        Tuning x;
        x.dense = env_int("TCAMCRF_DENSE", -1);
        x.build_dedup = env_int("TCAMCRF_BUILD_DEDUP", -1);
        x.himg_sections = env_int("TCAMCRF_HIMG_SECTIONS", 0);
        x.host_groups = env_int("TCAMCRF_HOST_GROUPS", 0);
        x.host_section0 = env_int("TCAMCRF_HOST_SECTION0", 0);
        x.host_trace = getenv("TCAMCRF_HOST_TRACE") != nullptr;
        x.host_grow = env_int("TCAMCRF_HOST_GROW", 0);
        return x;
    }();
    return t;
}

// ---------------------------------------------------------------------------
// workspace layout
// ---------------------------------------------------------------------------
constexpr int kThreads = 256;
constexpr int kFlagLogits = 1;        // segs holds logits, softmax on the fly
constexpr int kFlagReverseBlur = 2;   // blur axes d..0: the transposed filter
constexpr int kFlagLowp = 4;          // with kFlagLogits: the logits are 2-byte (fp16, or bf16 with kFlagBF16)
constexpr int kFlagBF16 = 8;



// ctrl words (ints).  [0,16) are reset by the host at the start of every call; MAGIC/DIRTY persist
// with the workspace; per-frame vertex counters follow at kCtrlCounts.
constexpr int kCtrlStatus = 0;      // TCAMCRF_DEV_* bits
constexpr int kCtrlLastCount = 1;   // vertices of the last chunk (sum over frames)
constexpr int kCtrlDirtyNew = 2;    // the build of the current chunk spilled into the overflow tier
constexpr int kCtrlTicket = 3;      // blocks of the slice kernel that have published their partial sum
constexpr int kCtrlAccInts = 8;      // a double: running sum of seg . AS over the chunks of the call
constexpr int kCtrlResetInts = 16;
constexpr int kCtrlMagic = 16;      // signature of the plan that last initialised the tables
constexpr int kCtrlDirty = 17;      // overflow tier holds keys (must be cleared before reuse)
constexpr int kCtrlEffSlots = 18;   // primary-tier size in use by the current call (effective_geom)
constexpr int kCtrlPrevMax = 19;    // largest per-frame vertex count of the last build on this workspace
constexpr int kCtrlCounts = 32;     // [chunk] vertices per frame

struct Plan {
    int D, K, Kp, H, W, P;
    int chunk;              // frames per pass
    TableGeom geom;         // per-frame table geometry
    unsigned int slots;     // geom.slots1 + geom.slots2
    int stride;             // vertex ids per frame (ids of frame n: [n*stride, n*stride + M_n))
    long long pool;         // chunk * stride
    int blocks_per_frame;   // pixel blocks per frame
    int sig;                // plan signature stored in the workspace
    float loss_weight;      // cfg->loss_weight (0 -> 1)
    // byte offsets into the workspace
    size_t off_ctrl, off_acc, off_partial, off_table, off_offset, off_bary, off_vkey, off_nbr, off_val0, off_val1,
        total;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static int feature_dim(const tcamcrf_config *cfg)
{
    if (!cfg) return -1;
    if (cfg->channels < 1) return -1;
    if (cfg->feat == TCAMCRF_FEAT_XY_RGB) return 2 + cfg->channels;
    if (cfg->feat == TCAMCRF_FEAT_COLOR) return cfg->channels;
    return -1;
}

static unsigned int pow2_at_least(double need, unsigned int lo)
{
    unsigned long long v = lo;
    while ((double)v < need) v <<= 1;
    return v > (1ull << 30) ? 0u : (unsigned int)v;
}

static int make_plan(const tcamcrf_config *cfg, int N, int K, int H, int W, Plan &pl)
{
    const int D = feature_dim(cfg);
    if (D < 1 || D > kMaxD) return fail(TCAMCRF_ERR_INVALID, "unsupported lattice dimension %d (1..%d)", D, kMaxD);
    if (N < 1 || K < 1 || H < 1 || W < 1) return fail(TCAMCRF_ERR_INVALID, "N,K,H,W must be positive");
    if ((long long)H * W > (1ll << 26)) return fail(TCAMCRF_ERR_INVALID, "image too large");
    // stride < channels: consecutive frames read overlapping windows of the image buffer -- what the reference's
    // colour batch loop does for DIM > 3 (a fixed stride of 3 planes, colorbilateralfilter.cpp:50)
    if (cfg->image_stride_planes < 1)
        return fail(TCAMCRF_ERR_INVALID, "image_stride_planes (%d) must be positive", cfg->image_stride_planes);
    if (!(cfg->sigma_rgb > 0.f) || (cfg->feat == TCAMCRF_FEAT_XY_RGB && !(cfg->sigma_xy > 0.f)))
        return fail(TCAMCRF_ERR_INVALID, "sigmas must be positive");
    pl.D = D;
    pl.loss_weight = cfg->loss_weight != 0.f ? cfg->loss_weight : 1.0f;
    pl.K = K;
    pl.Kp = K <= 2 ? K : (K + 3) / 4 * 4;  // value rows padded to whole float4s
    pl.H = H;
    pl.W = W;
    pl.P = H * W;
    int chunk = cfg->chunk_frames > 0 ? cfg->chunk_frames : 64;
    if (chunk > 256) chunk = 256;  // kMaxChunk: the vertex kernels keep a per-frame prefix sum in shared memory
    pl.chunk = chunk < N ? chunk : N;
    // every pixel (+ the ghost pixel) contributes at most d+1 distinct vertices
    const double worst = (double)(D + 1) * (pl.P + 1);
    // primary tier: hash_load is the load it would have with 1.2 vertices per pixel (iid-noise frames at
    // 224^2 have 1.12, natural frames ~0.06); overflow tier: worst case at load 0.75
    float load = cfg->hash_load > 0.f ? cfg->hash_load : 0.25f;
    pl.geom.slots1 = pow2_at_least(1.2 * (pl.P + 1) / load, 256);
    pl.geom.slots2 = pow2_at_least(worst / 0.75, 256);
    if (!pl.geom.slots1 || !pl.geom.slots2) return fail(TCAMCRF_ERR_INVALID, "hash table too large");
    pl.geom.window = pl.geom.slots1 < 128 ? pl.geom.slots1 : 128;
    auto log2u = [](unsigned int v) { int l = 0; while ((1u << l) < v) l++; return (unsigned int)l; };
    pl.geom.shift1 = 32 - log2u(pl.geom.slots1);
    pl.geom.shift2 = 32 - log2u(pl.geom.slots2);
    pl.geom.base2 = pl.geom.slots1;
    pl.slots = pl.geom.slots1 + pl.geom.slots2;
    float pf = cfg->pool_factor > 0.f ? cfg->pool_factor : 1.0f;
    if (pf > 1.f) pf = 1.f;
    if (worst * pf + 64 > (double)0x7fffff00) return fail(TCAMCRF_ERR_INVALID, "image too large");
    pl.stride = ((int)(worst * pf) + 32 + 31) / 32 * 32;
    // vertex ids, link indices ((d+1) * pool) and table entry indices (chunk * slots) are 32-bit: large frames get
    // a smaller chunk instead of an error (the reference takes any size; frames are independent, so the chunk
    // size never changes a result)
    {
        const long long lim = 0x7fffff00ll;
        long long most = lim / ((long long)pl.stride * (D + 1));
        if (lim / (long long)pl.slots < most) most = lim / (long long)pl.slots;
        if (most < 1) return fail(TCAMCRF_ERR_INVALID, "image too large");
        if (pl.chunk > most) pl.chunk = (int)most;
    }
    if (cfg->chunk_frames <= 0) {
        // default chunk: keep the workspace of large frames within ~16 GiB (64 frames of 1024x1024 would take 47)
        const double per_frame = (double)pl.slots * sizeof(Entry) + 2.0 * (D + 1) * pl.P * 4.0 +
                                 (double)pl.stride * (8.0 + (D + 1) * 8.0 + 2.0 * pl.Kp * 4.0);
        long long most = (long long)(16.0 * 1024 * 1024 * 1024 / per_frame);
        if (most < 1) most = 1;
        if (pl.chunk > most) pl.chunk = (int)most;
    }
    pl.pool = (long long)pl.stride * pl.chunk;
    // + 1: the ghost pixel that stands for the reference's zero-feature padding (see build_kernel)
    pl.blocks_per_frame = (pl.P + 1 + kThreads - 1) / kThreads;
    unsigned int sig = 0x9e3779b9u;
    for (unsigned int v : {(unsigned)D, (unsigned)pl.chunk, pl.geom.slots1, pl.geom.slots2, (unsigned)pl.stride,
                           (unsigned)pl.Kp, (unsigned)pl.P})
        sig = (sig ^ v) * 0x01000193u + 0x7f4a7c15u;
    pl.sig = (int)(sig | 1u);

    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t at = o;
        o = align_up(o + bytes, 256);
        return at;
    };
    pl.off_ctrl = take((size_t)(kCtrlCounts + pl.chunk) * sizeof(int));
    pl.off_acc = pl.off_ctrl + kCtrlAccInts * sizeof(int);   // inside the per-call reset region
    pl.off_partial = take((size_t)pl.chunk * pl.blocks_per_frame * sizeof(float));
    pl.off_table = take((size_t)pl.chunk * pl.slots * sizeof(Entry));
    pl.off_offset = take((size_t)pl.chunk * (D + 1) * pl.P * sizeof(int));
    pl.off_bary = take((size_t)pl.chunk * (D + 1) * pl.P * sizeof(float));
    pl.off_vkey = take((size_t)pl.pool * sizeof(unsigned long long));
    pl.off_nbr = take((size_t)(D + 1) * pl.pool * sizeof(int2));
    pl.off_val0 = take((size_t)pl.pool * pl.Kp * sizeof(float) + 64);
    pl.off_val1 = take((size_t)pl.pool * pl.Kp * sizeof(float) + 64);
    pl.total = o;
    return TCAMCRF_OK;
}

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
// Programmatic dependent launch.  The kernels of one chunk form a chain on the caller's stream; each is
// launched with cudaLaunchAttributeProgrammaticStreamSerialization, so its blocks may become resident while
// the previous kernel drains, run the part of their work that does not depend on it, and then block in
// pdl_wait() until the previous grid has completed and its writes are visible.  Every kernel calls
// pdl_launch_dependents() only AFTER its own pdl_wait(): when kernel X+1 starts, all blocks of X are past their
// wait, hence X-1 and everything before it is complete.  So, ahead of its wait, a kernel may READ what kernels
// up to X-2 (and the caller) produced, and must not write anything.
__device__ __forceinline__ void pdl_wait()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
__device__ __forceinline__ void pdl_launch_dependents()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

struct BuildParams {
    const void *images;     // [N, stride_planes, P] float or u8
    Entry *table;           // [n][slots1 + slots2]
    int *offset;            // [n][r][p] : global entry index (n*slots + s)
    float *bary;            // [n][r][p]
    unsigned long long *vkey;   // [pool] key of each vertex
    int *ctrl;
    int P, W, H;
    int stride_planes, channels, feat;
    TableGeom geom;
    unsigned int slots;
    int stride;             // ids per frame
    long long pool;
    float sigma_rgb, sigma_xy;
    int frame0;             // frame of block index 0 (sections of a chunk, host path)
    EmbedConsts ec;
};

template <typename T>
__device__ __forceinline__ float load_pixel(const void *base, size_t idx);
template <>
__device__ __forceinline__ float load_pixel<float>(const void *base, size_t idx)
{
    return __ldg((const float *)base + idx);
}
template <>
__device__ __forceinline__ float load_pixel<uint8_t>(const void *base, size_t idx)
{
    return (float)__ldg((const uint8_t *)base + idx);
}

// primary-tier slots per vertex of the previous call (rounded up to a power of two).  Measured, noise K=10, 32 frames:
// 4 -> build 0.206 / neighbour 0.130 / clear 0.028 ms; 2 (tables of all frames fit the L2) -> 0.211 / 0.159 / 0.016;
// 1 -> 0.343 / 0.481 / 0.036: the probe count matters, not where the table lives.
constexpr unsigned int kTableHeadroom = 4;
// Clears the tables of `nc` frames: always the primary tier, the overflow tier only when the workspace is
// new (magic mismatch) or the previous use spilled into it.  Also zeroes the per-frame vertex counters.
__global__ void __launch_bounds__(kThreads) prepare_kernel(Entry *table, int *ctrl, int frame0, int nc, int chunk,
                                                           TableGeom geom, int sig)
{
    pdl_wait();
    pdl_launch_dependents();
    // frame0 > 0: a later section of a chunk whose first section has already dealt with the overflow tiers
    const bool full = frame0 == 0 && ((ctrl[kCtrlMagic] != sig) || (ctrl[kCtrlDirty] != 0));
    // primary-tier size for this call (see effective_geom); later sections of a chunk take the first one's
    unsigned int eff = geom.slots1;
    if (frame0 > 0) {
        eff = (unsigned int)ctrl[kCtrlEffSlots];
    } else if (!full) {
        const unsigned int want = kTableHeadroom * (unsigned int)ctrl[kCtrlPrevMax];
        unsigned int e = geom.slots1 >> 4;   // floor: bounds what a bad guess costs (window-long probe chains)
        if (e < 4096u) e = 4096u;
        while (e < want && e < geom.slots1) e <<= 1;
        eff = e < geom.slots1 ? e : geom.slots1;
    }
    const unsigned int slots = geom.base2 + geom.slots2;
    geom.slots1 = eff;
    const long long n_primary = (long long)nc * geom.slots1;
    // the overflow tiers of ALL frames of the workspace are cleared together: the dirty flag is per workspace
    const long long total = n_primary + (full ? (long long)chunk * geom.slots2 : 0);
    const long long stride = (long long)gridDim.x * kThreads;
    const long long tid = (long long)blockIdx.x * kThreads + threadIdx.x;
    const uint4 empty = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0u);  // key EMPTY, id -1
    uint4 *t4 = reinterpret_cast<uint4 *>(table);
    for (long long i = tid; i < total; i += stride) {
        long long n, s;
        if (i < n_primary) {
            n = i / geom.slots1;
            s = i - n * geom.slots1;
            n += frame0;
        } else {
            const long long o = i - n_primary;
            n = o / geom.slots2;
            s = geom.base2 + (o - n * geom.slots2);
        }
        t4[n * slots + s] = empty;
    }
    if (tid < nc) ctrl[kCtrlCounts + frame0 + tid] = 0;
    if (tid == 0 && frame0 == 0) {
        ctrl[kCtrlLastCount] = 0;
        ctrl[kCtrlEffSlots] = (int)eff;
    }
}

// Occupancy target of the build kernel: 5 blocks of 256 threads per SM caps it at 48 registers (a few
// spills).  Measured on B200 (K=2, noise / natural frames, ms per 32-frame batch): 3 blocks 0.250 / 0.143,
// 4 blocks 0.221 / 0.119, 5 blocks 0.214 / 0.109, 6 blocks 0.218 / 0.107, 8 blocks 0.235 / 0.107.
constexpr int kBuildMinBlocks = 5;
// Front end shared by the two build kernels: the pixel's features (initializePermutohedral, bilateralfilter.cpp:4-19 /
// colorbilateralfilter.cpp:4-15), its embedding, the d+1 packed keys of its simplex, and the barycentric weights,
// which leave the registers right here.  Reads the caller's images only, so it runs ahead of griddepcontrol.wait (the
// kernel in front of a build kernel is prepare_kernel, an ordinary launch: every earlier reader of bary[] has
// completed before any block of this grid runs).  Returns false when a lattice coordinate leaves the key range.
template <int D, typename ImgT>
__device__ __forceinline__ bool build_front(const BuildParams &p, int n, int pix, bool valid, bool ghost,
                                            unsigned long long (&key)[D + 1])
{
    using Codec = KeyCodec<D>;
    float f[D];
    const size_t img0 = (size_t)n * p.stride_planes * p.P + pix;
    if (ghost) {
#pragma unroll
        for (int c = 0; c < D; c++) f[c] = 0.0f;
    } else if (p.feat == TCAMCRF_FEAT_XY_RGB) {
        const int row = pix / p.W, col = pix - row * p.W;
        f[0] = __fdiv_rn((float)col, p.sigma_xy);
        if (D > 1) f[1 < D ? 1 : 0] = __fdiv_rn((float)row, p.sigma_xy);
#pragma unroll
        for (int c = 2; c < D; c++) f[c] = __fdiv_rn(load_pixel<ImgT>(p.images, img0 + (size_t)(c - 2) * p.P), p.sigma_rgb);
    } else {
#pragma unroll
        for (int c = 0; c < D; c++) f[c] = __fdiv_rn(load_pixel<ImgT>(p.images, img0 + (size_t)c * p.P), p.sigma_rgb);
    }
    int z[D + 1], rank[D + 1];
    float bary[D + 1];
    const bool ok = embed_point<D>(f, p.ec, z, rank, bary);
    if (!ok) {
        // keep the fields well-formed; the whole call is poisoned through the status word
#pragma unroll
        for (int i = 0; i <= D; i++) {
            z[i] = 0;
            rank[i] = i;
        }
    }
    Codec::pack_simplex(z, rank, key);
    if (valid) {
        const size_t base = (size_t)n * (D + 1) * p.P + pix;
#pragma unroll
        for (int r = 0; r <= D; r++) p.bary[base + (size_t)r * p.P] = bary[r];
    }
    return ok;
}

template <int D, typename ImgT>
__global__ void __launch_bounds__(kThreads, kBuildMinBlocks) build_kernel(const BuildParams p)
{
    const int n = p.frame0 + blockIdx.x;
    const int pix = blockIdx.y * kThreads + threadIdx.x;
    const bool valid = pix < p.P;
    // The reference embeds pixels four at a time and also inserts the zero-feature padding pixels of the
    // last partial block (permutohedral.cpp:173,238-251).  Those vertices are never splatted to, but they
    // exist, pick up values during the blur and hand them on -- so they change the result.  All padding
    // pixels share one feature vector, hence one ghost pixel per frame reproduces them.
    const bool ghost = (pix == p.P) && (p.P & 3) != 0;
    const bool active = valid || ghost;
    const int lane = threadIdx.x & 31;

    unsigned long long key[D + 1];
    unsigned int wonmask = 0;
    bool ok = true;

    if (active) {
        ok = build_front<D, ImgT>(p, n, pix, valid, ghost, key);
    } else {
#pragma unroll
        for (int r = 0; r <= D; r++) key[r] = kEmptyKey;
    }
    // everything above reads the caller's images only; the tables are cleared by the previous kernel
    pdl_wait();
    pdl_launch_dependents();
    if (!ok) atomicOr(p.ctrl + kCtrlStatus, TCAMCRF_DEV_KEY_RANGE);
    // the primary-tier size this call works with (chosen by prepare_kernel)
    const TableGeom geom = effective_geom(p.geom, (unsigned int)p.ctrl[kCtrlEffSlots]);

    // Warp-cooperative insertion.  A warp holds 32 neighbouring pixels of one image row; in real frames
    // most of them fall on the same lattice vertices.  Lanes whose key equals their left neighbour's form a
    // run; only the head of a run touches the table and the result is broadcast back to the run
    // (one SHFL + one ballot per key -- MATCH.ANY.U64 measured ~3x the short-scoreboard stalls; equal keys
    // that are not adjacent are simply inserted twice, the second insert finds the first).  A head probes
    // for all the keys it leads in lock step: every round issues one load per pending key before any result
    // is consumed, so the d+1 dependent probe chains overlap instead of running one after the other.
    //
    // Vertex ids at build time.  A probe is ONE 16-byte load of {key, id}: when the key is already there and its
    // creator has published the id (blocks are interleaved across frames, so most keys are found by later waves
    // with plain loads), the pixel gets the dense vertex id right here and the splat never has to translate the
    // entry index -- up to 6 random look-ups and 6 stores per pixel less.  Where the id is not visible yet (-1)
    // the entry index is kept and the splat resolves it as before.
    Entry *tab = p.table + (size_t)n * p.slots;
    const unsigned int mask1 = geom.slots1 - 1;
    unsigned int pend = 0;
    // 5 bits per remainder: the lane that heads this lane's run (7 remainders at D = 6 need 35 bits)
    using LeaderWord = typename std::conditional<(D + 1) * 5 <= 32, unsigned int, unsigned long long>::type;
    LeaderWord leaders = 0;
    int slot[D + 1];                 // the slot being probed; once the key is resolved, the slot it lives in
    int vid[D + 1];                  // id field of the entry last probed = the vertex id once resolved (-1: unknown)
    unsigned long long cur[D + 1];
#pragma unroll
    for (int r = 0; r <= D; r++) {
        const unsigned long long left = __shfl_up_sync(0xffffffffu, key[r], 1);
        const bool head = lane == 0 || left != key[r];
        const unsigned int heads = __ballot_sync(0xffffffffu, head);
        leaders |= (LeaderWord)(unsigned int)(31 - __clz(heads & (0xffffffffu >> (31 - lane)))) << (5 * r);   // nearest head at or below
        slot[r] = -1;
        vid[r] = -1;
        cur[r] = 0;
        if (active && head) {
            pend |= 1u << r;
            slot[r] = (int)hash_primary(key[r], geom);
            load_entry_cg(tab + slot[r], cur[r], vid[r]);
        }
    }
    constexpr int kLockstepRounds = 6;
    int rounds = 0;
    for (; rounds < kLockstepRounds && pend; rounds++) {
        // every claim of the round is issued before any result is looked at: with the compare-and-swap and the test of
        // its result in one branch per key, a warp went through up to d+1 atomic round trips one after the other
        unsigned int tried = 0;
#pragma unroll
        for (int r = 0; r <= D; r++) {
            if ((pend & (1u << r)) && cur[r] == kEmptyKey) {
                tried |= 1u << r;
                cur[r] = atomicCAS(&tab[slot[r]].key, kEmptyKey, key[r]);
            }
        }
#pragma unroll
        for (int r = 0; r <= D; r++) {
            if (!(pend & (1u << r))) continue;
            unsigned long long c = cur[r];
            if (tried & (1u << r)) {
                vid[r] = -1;   // ours to allocate below, or created this instant by another thread
                if (c == kEmptyKey) {
                    wonmask |= 1u << r;
                    c = key[r];
                }
            }
            if (c == key[r])
                pend &= ~(1u << r);
            else
                slot[r] = (int)(((unsigned int)slot[r] + 1u) & mask1);
        }
#pragma unroll
        for (int r = 0; r <= D; r++)
            if (pend & (1u << r)) load_entry_cg(tab + slot[r], cur[r], vid[r]);
    }
    bool table_full = false, spilled_any = false;
#pragma unroll
    for (int r = 0; r <= D; r++) {
        if (pend & (1u << r)) {  // stragglers: long probe chains, overflow tier
            bool won, spilled;
            slot[r] = table_insert_from(tab, geom, key[r], (unsigned int)slot[r], (unsigned int)rounds, cur[r], won,
                                        spilled);
            vid[r] = -1;
            if (won) wonmask |= 1u << r;
            if (slot[r] < 0) table_full = true;
            spilled_any |= spilled;
        }
    }
    __syncwarp();
    if (table_full) atomicOr(p.ctrl + kCtrlStatus, TCAMCRF_DEV_TABLE_FULL);
    if (spilled_any) p.ctrl[kCtrlDirtyNew] = 1;

    // warp-aggregated allocation of dense vertex ids: one atomic per warp on the frame's counter (no block
    // barrier: a warp that is done does not wait for the slowest warp of its block)
    const int nwin = __popc(wonmask);
    int incl = nwin;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    int wbase = 0;
    if (lane == 31 && incl > 0) wbase = atomicAdd(p.ctrl + kCtrlCounts + n, incl);
    wbase = __shfl_sync(0xffffffffu, wbase, 31);
    int local = wbase + incl - nwin;
    bool pool_full = false;
#pragma unroll
    for (int r = 0; r <= D; r++) {
        if (wonmask & (1u << r)) {
            Entry *e = tab + slot[r];
            if (local < p.stride) {
                const int id = n * p.stride + local;
                e->id = id;
                p.vkey[id] = key[r];
                vid[r] = id;
            } else {
                pool_full = true;  // e->id stays -1
            }
            local++;
        }
    }
    if (pool_full) atomicOr(p.ctrl + kCtrlStatus, TCAMCRF_DEV_POOL_FULL);

    // what the pixel kernels find in offset[]: -2 - id (vertex id known), the entry index (>= 0: the first splat
    // looks the id up) or -1 (no vertex: table full).  Heads hand theirs to the lanes of their run.
    const size_t base = (size_t)n * (D + 1) * p.P + pix;
#pragma unroll
    for (int r = 0; r <= D; r++) {
        const int mine = vid[r] >= 0 ? -2 - vid[r] : (slot[r] < 0 ? -1 : (int)(n * p.slots + slot[r]));
        const int ref = __shfl_sync(0xffffffffu, mine, (int)((leaders >> (5 * r)) & 31u));
        if (valid) p.offset[base + (size_t)r * p.P] = ref;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Build kernel for SPARSE lattices (real frames: ~0.06 vertices per pixel, ~100 pixels per vertex).
//
// build_kernel spends most of its time between the embedding and the offset store: run detection, d+1 hashes,
// lock-step probes of the frame table in L2, id allocation -- and on real frames nearly all of that work finds a key
// some neighbouring pixel has just handled (the +-4 sensor noise makes equal keys ALTERNATE along a row, so runs of
// equal keys are only ~2.5 lanes long while a block of 256 pixels holds a few dozen distinct vertices).  Here the
// 256 x (d+1) keys of a block are first deduplicated in a shared-memory table (a hit is one LDS.64 and a compare),
// only the block's DISTINCT keys go to the frame table in L2 (one thread per key, first probe inline), and the pixels
// pick their result up from shared memory.  All of the shared-memory phase runs ahead of griddepcontrol.wait, i.e.
// while prepare_kernel is still clearing the tables.  Same table protocol and the same results as build_kernel (ids
// are a relabelling); the host picks per call from the density hint, like the splat variant.
constexpr int kTileW = 32, kTileH = 8;   // pixel tile of a build_dedup_kernel block
constexpr int kTileThreads = kTileW * kTileH;
static_assert(kTileW == 8 || kTileW == 16 || kTileW == 32, "a warp covers whole row segments of the tile");
static_assert(kTileThreads % 32 == 0 && kTileThreads <= 256, "tile = one thread block");

constexpr int ceil_log2(int v) { return v <= 1 ? 0 : 1 + ceil_log2((v + 1) / 2); }

template <int D>
struct DedupTable {
    // threads x (D+1) keys at most; the power of two >= that (load <= 0.875 in the worst case: 256 threads, D = 6)
    static constexpr int kBits = ceil_log2(kTileThreads * (D + 1));
    static constexpr int kSlots = 1 << kBits;
    static constexpr unsigned int kShift = 32 - kBits;
};

constexpr int kDedupMinBlocks = 8;
template <int D, typename ImgT>
__global__ void __launch_bounds__(kTileThreads, kDedupMinBlocks) build_dedup_kernel(const BuildParams p)
{
    constexpr int kSlots = DedupTable<D>::kSlots;
    __shared__ __align__(16) unsigned long long s_key[kSlots];
    __shared__ int s_val[kSlots];                         // what offset[] gets for the key in the same slot
    __shared__ unsigned short s_list[kTileThreads * (D + 1)];   // occupied slots, in insertion order
    __shared__ int s_count;
    static_assert(kSlots >= kTileThreads * (D + 1), "the embedding scratch lives in s_val");
    // A block is a TILE of 32 x 8 pixels (a warp = 32 neighbouring pixels of one row: coalesced like the linear
    // mapping), not 256 consecutive pixels: a row sweeps through many lattice cells, a compact tile through few (the
    // synthetic natural frames: 77 distinct keys per tile against 293 per 256-pixel run).  grid = (frames, tile rows
    // [+ 1], tile columns); block (ty = tile rows, tx = 0) carries the ghost pixel (see build_kernel) when there is one.
    const int n = p.frame0 + blockIdx.x;
    const int lane = threadIdx.x & 31;
    const int px = blockIdx.z * kTileW + (threadIdx.x % kTileW), py = blockIdx.y * kTileH + (threadIdx.x / kTileW);
    const bool ghost_block = (int)blockIdx.y * kTileH >= p.H;
    if (ghost_block && blockIdx.z != 0) return;
    const bool valid = !ghost_block && px < p.W && py < p.H;
    const bool ghost = ghost_block && threadIdx.x == 0;
    const bool active = valid || ghost;
    const int pix = valid ? py * p.W + px : p.P;

    // the pixel's features (initializePermutohedral, bilateralfilter.cpp:4-19 / colorbilateralfilter.cpp:4-15)
    float f[D];
#pragma unroll
    for (int c = 0; c < D; c++) f[c] = 0.0f;
    if (valid) {
        const size_t img0 = (size_t)n * p.stride_planes * p.P + pix;
        if (p.feat == TCAMCRF_FEAT_XY_RGB) {
            f[0] = __fdiv_rn((float)px, p.sigma_xy);
            if (D > 1) f[1 < D ? 1 : 0] = __fdiv_rn((float)py, p.sigma_xy);
#pragma unroll
            for (int c = 2; c < D; c++)
                f[c] = __fdiv_rn(load_pixel<ImgT>(p.images, img0 + (size_t)(c - 2) * p.P), p.sigma_rgb);
        } else {
#pragma unroll
            for (int c = 0; c < D; c++) f[c] = __fdiv_rn(load_pixel<ImgT>(p.images, img0 + (size_t)c * p.P), p.sigma_rgb);
        }
    }
    {   // clear the key table, two slots per store
        const ulonglong2 empty2 = make_ulonglong2(kEmptyKey, kEmptyKey);
        for (int i = threadIdx.x; i < kSlots / 2; i += kTileThreads) reinterpret_cast<ulonglong2 *>(s_key)[i] = empty2;
        if (threadIdx.x == 0) s_count = 0;
    }
    // embedding, keys and weights; s_val / s_list are free until the barrier below and serve as the per-thread
    // scratch columns of embed_simplex_scratch.  The weights leave the registers right here: the kernel in front of
    // this one (prepare_kernel) is an ordinary launch, so every earlier reader of bary[] has completed.
    unsigned long long key[D + 1];
    bool ok = true;
    if (active) {
        float bary[D + 1];
        ok = embed_simplex_scratch<D>(f, p.ec, reinterpret_cast<float *>(s_val) + threadIdx.x, s_list + threadIdx.x,
                                      kTileThreads, key, bary);
        if (valid) {
            const size_t base = (size_t)n * (D + 1) * p.P + pix;
#pragma unroll
            for (int r = 0; r <= D; r++) p.bary[base + (size_t)r * p.P] = bary[r];
        }
    }
    __syncthreads();

    // phase 1: the block's distinct keys (shared memory only)
    int myslot[D + 1];
#pragma unroll
    for (int r = 0; r <= D; r++) {
        unsigned int h = 0;
        bool won = false;
        if (active) {
            h = hash_slot(key[r], kHashMul1, DedupTable<D>::kShift);
            while (true) {
                unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(s_key + h);
                if (cur == kEmptyKey) {
                    cur = atomicCAS(s_key + h, kEmptyKey, key[r]);
                    won = cur == kEmptyKey;
                    if (won) break;
                }
                if (cur == key[r]) break;
                h = (h + 1) & (kSlots - 1);
            }
        }
        myslot[r] = (int)h;
        // the slots this warp has just filled join the block's list: one shared-memory atomic per warp
        const unsigned int w = __ballot_sync(0xffffffffu, won);
        if (w) {
            const int leader = __ffs(w) - 1;
            int at = 0;
            if (lane == leader) at = atomicAdd(&s_count, __popc(w));   // one lane: nothing for the compiler to aggregate
            at = __shfl_sync(0xffffffffu, at, leader);
            if (won) s_list[at + __popc(w & ((1u << lane) - 1u))] = (unsigned short)h;
        }
    }
    __syncthreads();
    const int count = s_count;

    // everything above reads the caller's images only; the tables are cleared by the previous kernel
    pdl_wait();
    pdl_launch_dependents();
    if (!ok) atomicOr(p.ctrl + kCtrlStatus, TCAMCRF_DEV_KEY_RANGE);
    const TableGeom geom = effective_geom(p.geom, (unsigned int)p.ctrl[kCtrlEffSlots]);
    Entry *tab = p.table + (size_t)n * p.slots;

    // phase 2: one thread per distinct key goes to the frame table (the loop bound is uniform over the block)
    bool table_full = false, spilled_any = false, pool_full = false;
    for (int base = 0; base < count; base += kTileThreads) {
        const int i = base + threadIdx.x;
        const bool on = i < count;
        int hs = 0, slot = -1, vid = -1;
        unsigned long long k = kEmptyKey;
        bool won = false;
        if (on) {
            hs = s_list[i];
            k = s_key[hs];
            const unsigned int h = hash_primary(k, geom);
            unsigned long long cur;
            load_entry_cg(tab + h, cur, vid);   // {key, id} in one 16-byte load
            if (cur == k) {
                slot = (int)h;   // the common case on real frames: an earlier block of the frame created it
            } else {
                bool spilled;
                slot = table_insert_from(tab, geom, k, h, 0, cur, won, spilled);
                vid = -1;        // ours to allocate below, or not looked at: the splat resolves the entry index
                table_full |= slot < 0;
                spilled_any |= spilled;
            }
        }
        // warp-aggregated allocation of dense vertex ids: one atomic per warp on the frame's counter
        const unsigned int winners = __ballot_sync(0xffffffffu, won);
        if (winners) {
            const int leader = __ffs(winners) - 1;
            int wbase = 0;
            if (lane == leader) wbase = atomicAdd(p.ctrl + kCtrlCounts + n, __popc(winners));
            wbase = __shfl_sync(0xffffffffu, wbase, leader);
            if (won) {
                const int local = wbase + __popc(winners & ((1u << lane) - 1u));
                if (local < p.stride) {
                    vid = n * p.stride + local;
                    tab[slot].id = vid;
                    p.vkey[vid] = k;
                } else {
                    pool_full = true;   // the entry's id stays -1
                }
            }
        }
        // -2 - id (vertex id known), the entry index (>= 0: the first splat looks the id up) or -1 (table full)
        if (on) s_val[hs] = vid >= 0 ? -2 - vid : (slot < 0 ? -1 : (int)(n * p.slots + slot));
    }
    if (table_full) atomicOr(p.ctrl + kCtrlStatus, TCAMCRF_DEV_TABLE_FULL);
    if (spilled_any) p.ctrl[kCtrlDirtyNew] = 1;
    if (pool_full) atomicOr(p.ctrl + kCtrlStatus, TCAMCRF_DEV_POOL_FULL);
    __syncthreads();

    // phase 3: every pixel picks up the results for its keys
    if (valid) {
        const size_t base = (size_t)n * (D + 1) * p.P + pix;
#pragma unroll
        for (int r = 0; r <= D; r++) p.offset[base + (size_t)r * p.P] = s_val[myslot[r]];
    }
}

struct VertexParams {
    const Entry *table;
    const unsigned long long *vkey;
    int2 *nbr;              // [axis][pool]
    float *values;          // rows of the vertices in use are zeroed here
    int *ctrl;
    TableGeom geom;
    unsigned int slots;
    int stride;
    long long pool;
    int Kp;
    int sig;
    int frame0;             // first frame of the chunk this launch works on (0 unless the host path runs the
                            // value stages group by group on a lattice built for the whole batch)
    int zero_values;        // neighbour_kernel: also clear the value rows
};

// The vertex kernels are persistent 1-D grids over the FLAT list of vertices of all frames of the chunk
// (frame 0's vertices first, then frame 1's, ...): the per-frame counts are turned into a prefix sum in
// shared memory once per block, and a flat index is mapped back to (frame, local vertex) by binary search.
// Frames are therefore swept in order, and the grid works on neighbouring frames at any moment.
constexpr int kMaxChunk = 256;

__device__ __forceinline__ int load_frame_prefix(const int *ctrl, int frame0, int nc, int stride, int *s_prefix)
{
    __shared__ int s_total;
    for (int n = threadIdx.x; n < nc; n += blockDim.x) {
        int m = ctrl[kCtrlCounts + frame0 + n];
        s_prefix[n + 1] = m > stride ? stride : m;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        s_prefix[0] = 0;
        for (int n = 0; n < nc; n++) {
            run += s_prefix[n + 1];
            s_prefix[n + 1] = run;
        }
        s_total = run;
    }
    __syncthreads();
    return s_total;
}

// largest n with prefix[n] <= t  (t < prefix[nc])
__device__ __forceinline__ int find_frame(const int *s_prefix, int nc, int t)
{
    int lo = 0, hi = nc;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (s_prefix[mid] <= t)
            lo = mid;
        else
            hi = mid;
    }
    return lo;
}

// A thread's flat index only grows from one loop iteration to the next, so the frame can be tracked with a
// cursor that moves forward (amortised O(1)) instead of a binary search per item.
__device__ __forceinline__ int advance_frame(const int *s_prefix, int nc, int n, int t)
{
    while (n + 1 < nc && t >= s_prefix[n + 1]) n++;
    return n;
}

// Zeroes the value rows of the vertices in use (host path and lattice re-use: the neighbour kernel clears them
// only once, right after the build).
__global__ void __launch_bounds__(kThreads) vertex_init_kernel(const VertexParams p, int nc)
{
    __shared__ int s_prefix[kMaxChunk + 1];
    pdl_wait();
    pdl_launch_dependents();
    load_frame_prefix(p.ctrl, p.frame0, nc, p.stride, s_prefix);
    const int stride = gridDim.x * kThreads;
    const int tid = blockIdx.x * kThreads + threadIdx.x;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    // pure streaming stores: walk the frames one after the other (the counts sit in shared memory), 16 bytes
    // per store; a frame's rows start 16-byte aligned (stride is a multiple of 32) and a store may run up to
    // 12 bytes past the last vertex in use, into rows nothing reads
    for (int n = 0; n < nc; n++) {
        const int M = s_prefix[n + 1] - s_prefix[n];
        const size_t id0 = (size_t)(p.frame0 + n) * p.stride;
        float4 *v4 = reinterpret_cast<float4 *>(p.values + id0 * p.Kp);
        const int quads = (M * p.Kp + 3) >> 2;
        for (int i = tid; i < quads; i += stride) v4[i] = zero4;
    }
}

// Blur neighbours: two table lookups per (vertex, axis), one coalesced 8-byte store of the link pair; the axis-0
// item also clears the vertex' value row for the splat.  (n1(v, j) = u <=> n2(u, j) = v, so one lookup could fill
// both directions, but the scattered 4-byte store into the other vertex' links and the preset pass it needs cost
// more than the second probe: 0.190 -> 0.150 ms per 32 noise frames, 0.049 -> 0.019 on natural frames.  Keeping
// several items per thread in flight measured no faster: profiles/README.md.)
template <int D>
__global__ void __launch_bounds__(kThreads) neighbour_kernel(const VertexParams p, int nc)
{
    using Codec = KeyCodec<D>;
    __shared__ int s_prefix[kMaxChunk + 1];
    pdl_wait();   // the vertex counts come from the build kernel, the launch right before this one
    pdl_launch_dependents();
    const int total = load_frame_prefix(p.ctrl, p.frame0, nc, p.stride, s_prefix);
    const int stride = gridDim.x * kThreads;
    const int tid = blockIdx.x * kThreads + threadIdx.x;
    const TableGeom geom = effective_geom(p.geom, (unsigned int)p.ctrl[kCtrlEffSlots]);
    const int work = total * (D + 1);   // < 2^31: pool * (D+1) is checked in make_plan
    // items are ordered frame by frame (so the grid probes one or two frame tables at a time and they stay
    // in L2), axis-major inside a frame: adjacent lanes handle adjacent vertices of one axis (coalesced key
    // loads and link stores)
    int n = 0;
    for (int i = tid; i < work; i += stride) {
        n = advance_frame(s_prefix, nc, n, i / (D + 1));   // prefix[n]*(D+1) <= i
        const int m = s_prefix[n + 1] - s_prefix[n];
        const int local = i - s_prefix[n] * (D + 1);
        const int axis = local / m;
        const int id = (p.frame0 + n) * p.stride + (local - axis * m);
        const Entry *tab = p.table + (size_t)(p.frame0 + n) * p.slots;
        const unsigned long long key = __ldg(p.vkey + id);
        unsigned long long k1, k2;
        Codec::neighbour_keys(key, axis, k1, k2);
        // both neighbours are looked up (their first probes are issued together) and the link pair is written
        // with one coalesced 8-byte store: no scattered 4-byte store into another vertex' links, and no
        // "missing" preset pass over the link table
        const unsigned int h1 = hash_primary(k1, geom);
        const unsigned int h2 = hash_primary(k2, geom);
        const uint4 e1 = __ldg(reinterpret_cast<const uint4 *>(tab + h1));
        const uint4 e2 = __ldg(reinterpret_cast<const uint4 *>(tab + h2));
        if (p.zero_values && axis == 0) {   // the value row of this vertex, cleared for the splat
            float4 *row4 = reinterpret_cast<float4 *>(p.values + (size_t)id * p.Kp);
            if ((p.Kp & 3) == 0) {
                for (int q = 0; q < (p.Kp >> 2); q++) row4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
            } else {
                for (int q = 0; q < p.Kp; q++) p.values[(size_t)id * p.Kp + q] = 0.f;
            }
        }
        const int nb1 = table_lookup_from(tab, geom, k1, h1, 0, e1);
        const int nb2 = table_lookup_from(tab, geom, k2, h2, 0, e2);
        p.nbr[(size_t)axis * p.pool + id] = make_int2(nb1, nb2);
    }
    if (tid == 0) {
        // sections of one chunk run one after the other on the stream: plain read-modify-write is enough
        p.ctrl[kCtrlLastCount] = (p.frame0 == 0 ? 0 : p.ctrl[kCtrlLastCount]) + total;
        // hand the spill state of this chunk over to the next prepare_kernel
        p.ctrl[kCtrlDirty] = (p.frame0 == 0 ? 0 : p.ctrl[kCtrlDirty]) | p.ctrl[kCtrlDirtyNew];
        p.ctrl[kCtrlDirtyNew] = 0;
        p.ctrl[kCtrlMagic] = p.sig;
        // the next call sizes its primary tier from this (effective_geom)
        int mx = p.frame0 == 0 ? 0 : p.ctrl[kCtrlPrevMax];
        for (int f = 0; f < nc; f++) mx = max(mx, s_prefix[f + 1] - s_prefix[f]);
        p.ctrl[kCtrlPrevMax] = mx;
    }
}

// vector helpers -------------------------------------------------------------
__device__ __forceinline__ void red_add(float *addr, const float (&v)[1]) { atomicAdd(addr, v[0]); }
__device__ __forceinline__ void red_add(float *addr, const float (&v)[2])
{
    atomicAdd(reinterpret_cast<float2 *>(addr), make_float2(v[0], v[1]));
}
__device__ __forceinline__ void red_add(float *addr, const float (&v)[4])
{
    atomicAdd(reinterpret_cast<float4 *>(addr), make_float4(v[0], v[1], v[2], v[3]));
}

template <int V>
__device__ __forceinline__ void load_vec(const float *addr, float (&v)[V])
{
    if (V == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(addr));
        v[0] = t.x;
        v[1 % V] = t.y;
        v[2 % V] = t.z;
        v[3 % V] = t.w;
    } else if (V == 2) {
        const float2 t = __ldg(reinterpret_cast<const float2 *>(addr));
        v[0] = t.x;
        v[1 % V] = t.y;
    } else {
        v[0] = __ldg(addr);
    }
}

template <int V>
__device__ __forceinline__ void store_vec(float *addr, const float (&v)[V])
{
    if (V == 4)
        *reinterpret_cast<float4 *>(addr) = make_float4(v[0], v[1 % V], v[2 % V], v[3 % V]);
    else if (V == 2)
        *reinterpret_cast<float2 *>(addr) = make_float2(v[0], v[1 % V]);
    else
        *addr = v[0];
}

struct PixelParams {
    const void *segs;       // [n][K][P]: float32 class probabilities, or logits when `logits` is set (2-byte
                            // logits for the *_lowp kernels)
    int logits;             // 1: segs holds logits; softmax over K is taken on the fly (never stored)
    float *as_out;          // [n][K][P]
    int *offset;            // [n][r][P]; entry index on entry to splat, dense id afterwards
    const float *bary;      // [n][r][P]
    const Entry *table;
    float *values;          // [pool][Kp]
    float *partial;         // [n][blocks_per_frame]; null when no loss is wanted
    int *ctrl;
    double *acc;            // running sum of seg . AS over the chunks of this call
    float *loss_out;        // non-null on the last chunk: receives -acc / n_norm
    float n_norm;
    float loss_scale;       // the module's weight, folded in: loss = loss_scale * (-acc / n_norm)
    int P, K, Kp;
    int frame0;             // workspace frame of blockIdx.y == 0 (segs / as_out already point at that frame)
    int dense;              // host-side hint: the lattices of this workspace have been dense lately (splat variant)
    long long pool;
    float alpha;
    int bf16;               // *_lowp kernels: the logits are bf16 (1) or fp16 (0)
};

// The segmentations of a launch as the body of a pixel kernel reads them: float32, or 2-byte logits (*_lowp kernels)
template <typename Z>
__device__ __forceinline__ Z segs_of(const PixelParams &p);
template <>
__device__ __forceinline__ const float *segs_of<const float *>(const PixelParams &p)
{
    return static_cast<const float *>(p.segs);
}
template <>
__device__ __forceinline__ Logits16 segs_of<Logits16>(const PixelParams &p)
{
    return Logits16{static_cast<const unsigned short *>(p.segs), p.bf16};
}

// softmax over the K planes of one pixel without storing it: max and sum first, then
// prob_k = exp(z_k - max) / sum, the order of operations of torch's softmax forward
struct SoftmaxStat {
    float zmax, sum;
};
// (Z: const float * or Logits16, see ld_logit)
template <typename Z>
__device__ __forceinline__ SoftmaxStat softmax_stat(Z z, int K, int P)
{
    SoftmaxStat s;
    s.zmax = -INFINITY;
    for (int k = 0; k < K; k++) s.zmax = fmaxf(s.zmax, ld_logit(z + (size_t)k * P));
    s.sum = 0.f;
    for (int k = 0; k < K; k++) s.sum += expf(ld_logit(z + (size_t)k * P) - s.zmax);
    return s;
}
template <bool L, typename Z>
__device__ __forceinline__ float seg_value(Z z, int k, int P, const SoftmaxStat &st)
{
    const float v = ld_logit(z + (size_t)k * P);
    return L ? __fdiv_rn(expf(v - st.zmax), st.sum) : v;
}

// Two classes (what TCAM trains with: fg / bg) with the softmax fused in: both probabilities of a pixel are formed
// once and kept in registers -- two loads, two expf, two divisions instead of softmax_stat's two passes plus
// seg_value's recomputation per use (six loads, four to six expf: expf is ~28 instructions, and the gradient kernel
// spent 388 instructions per pixel this way).  Same operations in the same order as softmax_stat + seg_value, hence
// the same bits.
struct Prob2 {
    float p0, p1;
    template <typename Z>
    __device__ __forceinline__ void load(Z z, int P)
    {
        const float z0 = ld_logit(z), z1 = ld_logit(z + P);
        const float zmax = fmaxf(fmaxf(-INFINITY, z0), z1);
        const float e0 = expf(z0 - zmax), e1 = expf(z1 - zmax);
        const float sum = (0.f + e0) + e1;
        p0 = __fdiv_rn(e0, sum);
        p1 = __fdiv_rn(e1, sum);
    }
    __device__ __forceinline__ float get(int k) const { return k == 0 ? p0 : p1; }
};

// Pixel-kernel bodies shared by the float32 kernels and their *_lowp twins (Z: the logits' source, see segs_of).
// `tid` is threadIdx.x read by the kernel itself, where __launch_bounds__ bounds it: read inside the inlined body the
// bound is lost and the index arithmetic compiles to other (slower to issue) instructions.
template <int D, int V, bool L, typename Z>
__device__ __forceinline__ void splat_body(const PixelParams p, unsigned int tid)
{
    const int n = blockIdx.y;
    const int pix = blockIdx.x * kThreads + tid;
    const bool valid = pix < p.P;
    const int lane = tid & 31;
    const size_t base = (size_t)(p.frame0 + n) * (D + 1) * p.P + (valid ? pix : 0);
    int id[D + 1];
    float w[D + 1];
    // Runs of neighbouring lanes that hit the same vertex (the common case in real frames: ~100 pixels per
    // vertex) are summed in registers first and only the head of a run issues the RED -- same-address atomics
    // serialise in L2.  run[r] = lanes above this one (bit i = lane+1+i) up to the end of its run.
    unsigned int heads[D + 1];
    unsigned int fresh = 0;   // bit r: offset[r] still held the entry index
    bool any_run = false;
    // ahead of the wait: entry indices, weights and ids come from the build kernel (two launches back), the
    // segmentations from the caller
#pragma unroll
    for (int r = 0; r <= D; r++) {
        int v = -1;
        if (valid) {
            // offset[] holds a table entry index (>= 0) until the first splat on this lattice has turned it into
            // the dense vertex id, stored as -2 - id (so a lattice can be applied any number of times); -1 = none
            const int s = p.offset[base + (size_t)r * p.P];
            if (s >= 0) {
                v = __ldg(&p.table[s].id);
                fresh |= 1u << r;
            } else if (s <= -2) {
                v = -2 - s;
            }
            w[r] = p.bary[base + (size_t)r * p.P];
        } else {
            w[r] = 0.f;
        }
        id[r] = v;
    }
    const Z seg = segs_of<Z>(p) + (size_t)n * p.K * p.P + (valid ? pix : 0);
    SoftmaxStat sm = {0.f, 1.f};
    Prob2 p2 = {0.f, 0.f};
    const bool two = L && p.K == 2;
    if (L && valid) {
        if (two)
            p2.load(seg, p.P);
        else
            sm = softmax_stat(seg, p.K, p.P);
    }
    pdl_wait();   // the value rows are cleared by the previous kernel
    pdl_launch_dependents();
#pragma unroll
    for (int r = 0; r <= D; r++) {
        const int v = id[r];
        if (fresh & (1u << r)) p.offset[base + (size_t)r * p.P] = v < 0 ? -1 : -2 - v;
        const int left = __shfl_up_sync(0xffffffffu, v, 1);
        const bool head = lane == 0 || left != v;
        heads[r] = __ballot_sync(0xffffffffu, head);
        any_run |= heads[r] != 0xffffffffu;
    }
    for (int k = 0; k < p.Kp; k += V) {
        float s[V];
#pragma unroll
        for (int e = 0; e < V; e++)
            s[e] = (valid && k + e < p.K) ? ((L && two) ? p2.get(k + e) : seg_value<L>(seg, k + e, p.P, sm)) : 0.f;
#pragma unroll
        for (int r = 0; r <= D; r++) {
            float t[V];
#pragma unroll
            for (int e = 0; e < V; e++) t[e] = __fmul_rn(w[r], s[e]);
            bool issue = id[r] >= 0;
            if (any_run && heads[r] != 0xffffffffu) {   // warp-uniform: some run of this remainder is longer than 1
                // segmented suffix sum over the run: lane i adds lane i+o when no head lies in (i, i+o]
                const unsigned int above = heads[r] >> 1 >> lane;   // bit j = head flag of lane+1+j
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const bool take = (lane + o < 32) && ((above & ((1u << o) - 1u)) == 0u);
#pragma unroll
                    for (int e = 0; e < V; e++) {
                        const float other = __shfl_down_sync(0xffffffffu, t[e], o);
                        if (take) t[e] += other;
                    }
                }
                issue = issue && ((heads[r] >> lane) & 1u);
            }
            if (issue) red_add(p.values + (size_t)id[r] * p.Kp + k, t);
        }
    }
}

template <int D, int V, bool L>
__global__ void __launch_bounds__(kThreads) splat_kernel(const PixelParams p)
{
    splat_body<D, V, L, const float *>(p, threadIdx.x);
}

// the same from fp16 / bf16 logits
template <int D, int V>
__global__ void __launch_bounds__(kThreads) splat_lowp_kernel(const PixelParams p)
{
    splat_body<D, V, true, Logits16>(p, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------------------
// Row-cooperative splat for value rows of 2..4 float4s (K = 5..16), used on DENSE lattices.
//
// splat_kernel touches a vertex row with KV separate 16-byte REDs per thread: 32 lanes x KV instructions =
// 32*KV requests to L2 per remainder, and on iid-noise frames (every pixel on its own vertices) the request rate of
// the L2 (~180 G/s, profiles/README.md) is what bounds the kernel.  Here KV neighbouring lanes share one pixel and
// each handles one float4 column of the row, so the KV REDs of a row sit in one instruction and leave the SM as ONE
// request (two when the row straddles a 128-byte line): a third of the requests at K = 10 (0.205 -> 0.177 ms per 32
// noise frames).  Per-pixel inputs are fetched with coalesced accesses and handed to the (pixel, column) lanes
// through shared memory.  On real frames the pixel kernel wins (runs of equal vertices merge over the 32 pixels of
// a warp instead of 32 / KV, no block barrier: 0.135 against 0.152 ms), so the host picks per call from the vertex
// density of the previous calls on the workspace (density_hint below): a hint, never a correctness matter.
template <int KV>
__host__ __device__ constexpr unsigned int stride_bits(int count)   // bits KV, 2*KV, ..., count*KV
{
    unsigned int m = 0;
    for (int i = 1; i <= count; i++) m |= 1u << (i * KV);
    return m;
}

template <int KV>
struct RowMap {
    static constexpr int kPpw = 32 / KV;                       // pixels per warp
    static constexpr int kPpb = (kThreads / 32) * kPpw;        // pixels per block
};

template <int D, int KV, bool L, typename Z>
__device__ __forceinline__ void splat_rows_body(const PixelParams p, unsigned int tid)
{
    constexpr int kPpw = RowMap<KV>::kPpw, kPpb = RowMap<KV>::kPpb;
    constexpr int Kp = 4 * KV;
    __shared__ int s_raw[D + 1][kPpb];     // offset[] as stored (entry index, tagged id or -1)
    __shared__ int s_id[D + 1][kPpb];
    __shared__ float s_w[D + 1][kPpb];
    __shared__ float s_seg[4 * KV][kPpb];
    const int n = blockIdx.y;
    const int pix0 = blockIdx.x * kPpb;
    const int npix = min(kPpb, p.P - pix0);
    const size_t base = (size_t)(p.frame0 + n) * (D + 1) * p.P + pix0;
    // ahead of the wait (see splat_kernel): coalesced loads, id look-ups
    for (int t = tid; t < (D + 1) * kPpb; t += kThreads) {
        const int r = t / kPpb, q = t - r * kPpb;
        int raw = -1, v = -1;
        float w = 0.f;
        if (q < npix) {
            raw = p.offset[base + (size_t)r * p.P + q];
            if (raw >= 0)
                v = __ldg(&p.table[raw].id);
            else if (raw <= -2)
                v = -2 - raw;
            w = p.bary[base + (size_t)r * p.P + q];
        }
        s_raw[r][q] = raw;
        s_id[r][q] = v;
        s_w[r][q] = w;
    }
    const Z seg = segs_of<Z>(p) + (size_t)n * p.K * p.P + pix0;
    for (int t = tid; t < Kp * kPpb; t += kThreads) {
        const int k = t / kPpb, q = t - k * kPpb;
        s_seg[k][q] = (k < p.K && q < npix) ? ld_logit(seg + (size_t)k * p.P + q) : 0.f;
    }
    __syncthreads();
    const int lane = tid & 31, warp = tid >> 5;
    const int j = lane / KV, c = lane - j * KV;                // pixel slot within the warp, float4 column
    const bool lane_on = j < kPpw;
    const int q = warp * kPpw + (lane_on ? j : 0);             // pixel slot within the block
    const bool valid = lane_on && q < npix;
    int id[D + 1];
    float w[D + 1];
#pragma unroll
    for (int r = 0; r <= D; r++) {
        id[r] = valid ? s_id[r][q] : -1;
        w[r] = valid ? s_w[r][q] : 0.f;
    }
    float s[4];
    if (L) {   // softmax over the K planes of this pixel, torch's order of operations (see softmax_stat)
        float zmax = -INFINITY, sum = 0.f;
        for (int k = 0; k < p.K; k++) zmax = fmaxf(zmax, s_seg[k][q]);
        for (int k = 0; k < p.K; k++) sum += expf(s_seg[k][q] - zmax);
#pragma unroll
        for (int e = 0; e < 4; e++)
            s[e] = (valid && 4 * c + e < p.K) ? __fdiv_rn(expf(s_seg[4 * c + e][q] - zmax), sum) : 0.f;
    } else {
#pragma unroll
        for (int e = 0; e < 4; e++) s[e] = valid ? s_seg[4 * c + e][q] : 0.f;
    }
    pdl_wait();   // the value rows are cleared by the previous kernel
    pdl_launch_dependents();
    // entry indices become tagged vertex ids (coalesced write-back of the fresh ones)
    for (int t = tid; t < (D + 1) * kPpb; t += kThreads) {
        const int r = t / kPpb, qq = t - r * kPpb;
        if (s_raw[r][qq] >= 0) {
            const int v = s_id[r][qq];
            p.offset[base + (size_t)r * p.P + qq] = v < 0 ? -1 : -2 - v;
        }
    }
    unsigned int heads[D + 1];
    bool any_run = false;
#pragma unroll
    for (int r = 0; r <= D; r++) {
        // runs of neighbouring PIXELS on the same vertex (lanes KV apart); idle lanes end every run
        const int v = id[r];
        const int left = __shfl_up_sync(0xffffffffu, v, KV);
        const bool head = j == 0 || left != v || !lane_on;
        heads[r] = __ballot_sync(0xffffffffu, head);
        any_run |= heads[r] != 0xffffffffu;
    }
#pragma unroll
    for (int r = 0; r <= D; r++) {
        float t[4];
#pragma unroll
        for (int e = 0; e < 4; e++) t[e] = __fmul_rn(w[r], s[e]);
        bool issue = id[r] >= 0;
        if (any_run && heads[r] != 0xffffffffu) {   // warp-uniform
            // segmented suffix sum over the run: pixel j adds pixel j+o when no head lies in (j, j+o]
            const unsigned int above = heads[r] >> lane;   // bit i*KV = head flag of pixel j+i (same column)
#pragma unroll
            for (int o = 1; o < kPpw; o <<= 1) {
                const bool take = (j + o < kPpw) && ((above & stride_bits<KV>(o)) == 0u);
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const float other = __shfl_down_sync(0xffffffffu, t[e], o * KV);
                    if (take) t[e] += other;
                }
            }
            issue = issue && ((heads[r] >> lane) & 1u);
        }
        if (issue) red_add(p.values + (size_t)id[r] * Kp + 4 * c, t);
    }
}

template <int D, int KV, bool L>
__global__ void __launch_bounds__(kThreads) splat_rows_kernel(const PixelParams p)
{
    splat_rows_body<D, KV, L, const float *>(p, threadIdx.x);
}

// the same from fp16 / bf16 logits
template <int D, int KV>
__global__ void __launch_bounds__(kThreads) splat_rows_lowp_kernel(const PixelParams p)
{
    splat_rows_body<D, KV, true, Logits16>(p, threadIdx.x);
}

struct BlurParams {
    const float *src;
    float *dst;
    const int2 *nbr;        // this axis: [pool]
    const int *ctrl;
    int Kp, stride;
    int frame0;
};

// persistent 1-D grid over the flat, frame-ordered vertex list (see the note above load_frame_prefix).
// Work item = (vertex, vector column); KV = Kp / V columns per vertex (0: run-time value).  The kernel is
// issue-sensitive (ncu: 0.6 IPC per scheduler with the first version, ~140 instructions per item, most of them
// a 64-bit division), so the (vertex, column) pair of a thread is advanced incrementally: no division in the loop.
template <int V, int KV>
__global__ void __launch_bounds__(kThreads) blur_kernel(const BlurParams p, int nc)
{
    __shared__ int s_prefix[kMaxChunk + 1];
    // ahead of the wait: vertex counts (build) and links (neighbour) are older than the previous launch
    const int total = load_frame_prefix(p.ctrl, p.frame0, nc, p.stride, s_prefix);
    const int kv = KV > 0 ? KV : p.Kp / V;
    const unsigned int nthreads = gridDim.x * kThreads;
    const unsigned int tid = blockIdx.x * kThreads + threadIdx.x;
    // thread `tid` handles items tid, tid + nthreads, ...; item i = vertex i / kv, column i % kv
    const int dt = (int)(nthreads / (unsigned)kv), dc = (int)(nthreads % (unsigned)kv);
    int t = (int)(tid / (unsigned)kv), c = (int)(tid % (unsigned)kv);
    int n = 0;
    const int Kp = KV > 0 ? KV * V : p.Kp;
    // the links of the NEXT item are fetched while the rows of the current one are in flight: one dependent
    // round trip per item instead of two
    int v = 0;
    int2 nb = make_int2(-1, -1);
    if (t < total) {
        n = advance_frame(s_prefix, nc, n, t);
        v = (p.frame0 + n) * p.stride + (t - s_prefix[n]);
        nb = __ldg(p.nbr + v);
    }
    pdl_wait();
    pdl_launch_dependents();
    while (t < total) {
        const int col = c * V;
        float own[V], a[V], b[V];
#pragma unroll
        for (int e = 0; e < V; e++) a[e] = b[e] = 0.f;
        load_vec<V>(p.src + (size_t)v * Kp + col, own);
        if (nb.x >= 0) load_vec<V>(p.src + (size_t)nb.x * Kp + col, a);
        if (nb.y >= 0) load_vec<V>(p.src + (size_t)nb.y * Kp + col, b);
        float *dst = p.dst + (size_t)v * Kp + col;
        t += dt;
        c += dc;
        if (c >= kv) {
            c -= kv;
            t++;
        }
        if (t < total) {
            n = advance_frame(s_prefix, nc, n, t);
            v = (p.frame0 + n) * p.stride + (t - s_prefix[n]);
            nb = __ldg(p.nbr + v);
        }
        float out[V];
        // new = old + 0.5*(n1 + n2), rounded after every operation (permutohedral.cpp:547)
#pragma unroll
        for (int e = 0; e < V; e++) out[e] = __fadd_rn(own[e], __fmul_rn(0.5f, __fadd_rn(a[e], b[e])));
        store_vec<V>(dst, out);
    }
}

// The last block to arrive folds the block partials of seg . AS (fixed order => deterministic given AS) into the
// running total and, when p.loss_out is set (last chunk), writes the loss: no separate reduction launches.
// Call with all threads of the block, after the block's partial has been written.
__device__ __forceinline__ void fold_loss_partials(const PixelParams &p)
{
    __shared__ bool s_last;
    __shared__ double s_sum[kThreads / 32];
    const int nblocks = gridDim.x * gridDim.y;
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(p.ctrl + kCtrlTicket, 1) == nblocks - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double sum = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += kThreads) sum += (double)__ldcg(p.partial + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        double total = p.acc[0];
        for (int w = 0; w < kThreads / 32; w++) total += s_sum[w];
        p.acc[0] = total;
        p.ctrl[kCtrlTicket] = 0;
        if (p.loss_out) {
            // loss = -(sum)/n_norm, NaN when the device status is set (dense_crf_loss.py:63-64)
            const float s = (float)total;
            // weight * loss as two separately rounded operations, like `self.weight * Function.apply(...)`
            // (dense_crf_loss.py:118-122); loss_scale = 1 leaves the bits of the plain loss untouched
            p.loss_out[0] = p.ctrl[kCtrlStatus] != 0 ? __int_as_float(0x7fc00000)
                                                     : __fmul_rn(p.loss_scale, __fdiv_rn(-s, p.n_norm));
        }
    }
}

template <int D, int V, bool L, typename Z>
__device__ __forceinline__ void slice_body(const PixelParams p)
{
    __shared__ float s_red[kThreads / 32];
    const int n = blockIdx.y;
    const int pix = blockIdx.x * kThreads + threadIdx.x;
    float dot = 0.f;
    int id[D + 1];
    float w[D + 1];
    const Z seg = segs_of<Z>(p) + (size_t)n * p.K * p.P + pix;
    SoftmaxStat sm = {0.f, 1.f};
    Prob2 p2 = {0.f, 0.f};
    const bool two = L && p.K == 2;
    // ahead of the wait: vertex ids (splat), weights (build) and segmentations (caller) are all older than
    // the previous launch (the last blur pass)
    if (pix < p.P) {
        const size_t base = (size_t)(p.frame0 + n) * (D + 1) * p.P + pix;
#pragma unroll
        for (int r = 0; r <= D; r++) {
            const int s = p.offset[base + (size_t)r * p.P];
            id[r] = s <= -2 ? -2 - s : -1;   // see splat_kernel
            // (bary * alpha) first, then * value (permutohedral.cpp:562-564)
            w[r] = __fmul_rn(p.bary[base + (size_t)r * p.P], p.alpha);
        }
        if (L) {
            if (two)
                p2.load(seg, p.P);
            else
                sm = softmax_stat(seg, p.K, p.P);
        }
    }
    pdl_wait();
    pdl_launch_dependents();
    const bool poisoned = p.ctrl[kCtrlStatus] != 0;
    if (pix < p.P) {
        float *out = p.as_out + (size_t)n * p.K * p.P + pix;
        for (int k = 0; k < p.Kp; k += V) {
            float acc[V];
#pragma unroll
            for (int e = 0; e < V; e++) acc[e] = 0.f;
#pragma unroll
            for (int r = 0; r <= D; r++) {
                float val[V];
                if (id[r] >= 0)
                    load_vec<V>(p.values + (size_t)id[r] * p.Kp + k, val);
                else {
#pragma unroll
                    for (int e = 0; e < V; e++) val[e] = 0.f;
                }
#pragma unroll
                for (int e = 0; e < V; e++) acc[e] = __fadd_rn(acc[e], __fmul_rn(w[r], val[e]));
            }
#pragma unroll
            for (int e = 0; e < V; e++) {
                if (k + e < p.K) {
                    const float o = poisoned ? __int_as_float(0x7fc00000) : acc[e];
                    out[(size_t)(k + e) * p.P] = o;
                    dot = fmaf((L && two) ? p2.get(k + e) : seg_value<L>(seg, k + e, p.P, sm), o, dot);
                }
            }
        }
    }
    // block partial of seg . AS
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = dot;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = threadIdx.x < kThreads / 32 ? s_red[threadIdx.x] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (threadIdx.x == 0 && p.partial) p.partial[(size_t)n * gridDim.x + blockIdx.x] = t;
    }
    if (!p.partial) return;
    fold_loss_partials(p);
}

template <int D, int V, bool L>
__global__ void __launch_bounds__(kThreads) slice_kernel(const PixelParams p)
{
    slice_body<D, V, L, const float *>(p);
}

// the same from fp16 / bf16 logits
template <int D, int V>
__global__ void __launch_bounds__(kThreads) slice_lowp_kernel(const PixelParams p)
{
    slice_body<D, V, true, Logits16>(p);
}

// grad = ((-2*g) * AS) / n  with the reference's rounding order (dense_crf_loss.py:73)
__global__ void __launch_bounds__(kThreads) loss_backward_kernel(const float *__restrict__ as,
                                                                 const float *__restrict__ grad_out,
                                                                 float *__restrict__ grad, size_t count, float n_norm,
                                                                 float weight)
{
    // grad_out * weight first: what autograd hands DenseCRFLossFunction.backward for `weight * loss`
    const float t = __fmul_rn(-2.0f, __fmul_rn(__ldg(grad_out), weight));
    // vector path only when both buffers are 16-byte aligned (sub-batches of odd-sized frames are not)
    const bool aligned = ((reinterpret_cast<uintptr_t>(as) | reinterpret_cast<uintptr_t>(grad)) & 15) == 0;
    const size_t n4 = aligned ? count / 4 : 0;
    const size_t stride = (size_t)gridDim.x * kThreads;
    const size_t tid = (size_t)blockIdx.x * kThreads + threadIdx.x;
    const float4 *as4 = reinterpret_cast<const float4 *>(as);
    float4 *g4 = reinterpret_cast<float4 *>(grad);
    for (size_t i = tid; i < n4; i += stride) {
        const float4 a = __ldcs(as4 + i);
        float4 g;
        g.x = __fdiv_rn(__fmul_rn(t, a.x), n_norm);
        g.y = __fdiv_rn(__fmul_rn(t, a.y), n_norm);
        g.z = __fdiv_rn(__fmul_rn(t, a.z), n_norm);
        g.w = __fdiv_rn(__fmul_rn(t, a.w), n_norm);
        __stcs(g4 + i, g);
    }
    for (size_t i = n4 * 4 + tid; i < count; i += stride) grad[i] = __fdiv_rn(__fmul_rn(t, as[i]), n_norm);
}

// Backward through the CRF loss AND the softmax that produced its input, for one pixel:
//   g_k = ((-2*g) * AS_k) / n   (dense_crf_loss.py:73),   dz_k = p_k * (g_k - sum_j p_j g_j)
// out(k, dz_k, p_k) receives each class's gradient and probability; z / a point at class 0 of the pixel (stride P).
template <typename Z, typename Out>
__device__ __forceinline__ void softmax_crf_grad(Z z, const float *a, int K, int P, float t, float n_norm, Out &&out)
{
    if (K == 2) {   // fg / bg: everything loaded once, the four loads in flight together
        const float a0 = __ldg(a), a1 = __ldg(a + P);
        Prob2 p2;
        p2.load(z, P);
        const float g0 = __fdiv_rn(__fmul_rn(t, a0), n_norm), g1 = __fdiv_rn(__fmul_rn(t, a1), n_norm);
        const float inner2 = fmaf(p2.p1, g1, fmaf(p2.p0, g0, 0.f));
        out(0, p2.p0 * (g0 - inner2), p2.p0);
        out(1, p2.p1 * (g1 - inner2), p2.p1);
        return;
    }
    const SoftmaxStat sm = softmax_stat(z, K, P);
    float inner = 0.f;
    for (int k = 0; k < K; k++) {
        const float pk = __fdiv_rn(expf(ld_logit(z + (size_t)k * P) - sm.zmax), sm.sum);
        inner = fmaf(pk, __fdiv_rn(__fmul_rn(t, __ldg(a + (size_t)k * P)), n_norm), inner);
    }
    for (int k = 0; k < K; k++) {
        const float pk = __fdiv_rn(expf(ld_logit(z + (size_t)k * P) - sm.zmax), sm.sum);
        const float gk = __fdiv_rn(__fmul_rn(t, __ldg(a + (size_t)k * P)), n_norm);
        out(k, pk * (gk - inner), pk);
    }
}

// T *__restrict__ for a pointer type T *, T itself otherwise
template <typename T>
struct Restrict {
    using type = T;
};
template <typename T>
struct Restrict<T *> {
    using type = T *__restrict__;
};

// thread per pixel; logits / AS / grad planar [n][K][P]; G: float * or Grad16 (the logits' 2-byte type)
template <typename Z, typename G>
__device__ __forceinline__ void loss_backward_logits_body(const float *__restrict__ as,
                                                          typename Restrict<Z>::type logits,
                                                          const float *__restrict__ grad_out,
                                                          typename Restrict<G>::type grad, int K, int P,
                                                          long long pixels, float n_norm, float weight,
                                                          unsigned int tid)
{
    const float t = __fmul_rn(-2.0f, __fmul_rn(__ldg(grad_out), weight));
    const long long stride = (long long)gridDim.x * kThreads;
    for (long long i = (long long)blockIdx.x * kThreads + tid; i < pixels; i += stride) {
        // (32-bit division when the pixel index fits: a 64-bit one is ~25 instructions more per pixel)
        const long long n = pixels <= 0x7fffffffll ? (long long)((unsigned int)i / (unsigned int)P) : i / P;
        const size_t base = (size_t)n * K * P + (i - n * P);
        softmax_crf_grad(logits + base, as + base, K, P, t, n_norm,
                         [&](int k, float v, float) { st_grad(grad + (base + (size_t)k * P), v); });
    }
}

__global__ void __launch_bounds__(kThreads) loss_backward_logits_kernel(const float *__restrict__ as,
                                                                        const float *__restrict__ logits,
                                                                        const float *__restrict__ grad_out,
                                                                        float *__restrict__ grad, int K, int P,
                                                                        long long pixels, float n_norm, float weight)
{
    loss_backward_logits_body<const float *, float *>(as, logits, grad_out, grad, K, P, pixels, n_norm, weight,
                                                      threadIdx.x);
}

// the same on fp16 / bf16 logits; the gradient is written in their type, rounded once from the float32 value
__global__ void __launch_bounds__(kThreads) loss_backward_logits_lowp_kernel(const float *__restrict__ as,
                                                                             Logits16 logits,
                                                                             const float *__restrict__ grad_out,
                                                                             Grad16 grad, int K, int P,
                                                                             long long pixels, float n_norm,
                                                                             float weight)
{
    loss_backward_logits_body<Logits16, Grad16>(as, logits, grad_out, grad, K, P, pixels, n_norm, weight, threadIdx.x);
}

// seed_ce_backward_kernel (seed.cuh) on fp16 / bf16 logits, with the gradient in their type.  Each labelled pixel's
// gradient is formed in float32 and rounded ONCE: base + coef * (p_k - [k == label]), where base is
//   as == NULL: the gradient already in `grad`, widened (exact; zero for SeedCrossEntropyFunction)
//   as != NULL: the float32 CRF gradient of the pixel, recomputed by softmax_crf_grad exactly as
//               loss_backward_logits_lowp_kernel formed it before rounding (t = -2 * (g * crf_weight)):
// the float32 sequence "CRF gradient, then the cross-entropy added in place" rounded once, where adding onto the
// already rounded value would round twice.
__global__ void __launch_bounds__(256) seed_ce_backward_lowp_kernel(Logits16 logits, const int *__restrict__ sel,
                                                                    Grad16 grad, const float *__restrict__ count,
                                                                    const float *__restrict__ grad_out, float scale,
                                                                    int K, int H, int W, int kmax, int ksz,
                                                                    const float *__restrict__ as, float n_norm,
                                                                    float crf_weight)
{
    const int b = blockIdx.x;
    const int HW = H * W;
    const int *sel_b = sel + (size_t)b * 2 * kmax;
    const Logits16 z = logits + (size_t)b * K * HW;
    const Grad16 g = grad + (size_t)b * K * HW;
    const float coef = __fdiv_rn(__fmul_rn(__ldg(grad_out), scale), __ldg(count));
    const float t = __fmul_rn(-2.0f, __fmul_rn(__ldg(grad_out), crf_weight));
    const int win = ksz * ksz, items = 2 * kmax * win;
    for (int it = threadIdx.x; it < items; it += 256) {
        const int side = it / (kmax * win), rest = it - side * kmax * win;
        int pix;
        const int label = seed_window_label(sel_b, kmax, ksz, H, W, side, rest / win, rest % win, pix);
        if (label < 0) continue;
        // (same expression as seed_ce_backward_kernel's `g += coef * (pk - onehot)`, contracted to one fma)
        auto add_ce = [&](int k, float base, float pk) {
            st_grad(g + ((size_t)k * HW + pix), fmaf(coef, pk - (k == label ? 1.f : 0.f), base));
        };
        if (as) {
            softmax_crf_grad(z + (size_t)pix, as + (size_t)b * K * HW + pix, K, HW, t, n_norm, add_ce);
        } else {
            const SoftmaxStat sm = softmax_stat(z + (size_t)pix, K, HW);
            for (int k = 0; k < K; k++)
                add_ce(k, ld_grad(g + ((size_t)k * HW + pix)), seg_value<true>(z + (size_t)pix, k, HW, sm));
        }
    }
}

// out[b][i] = max_t cams[b][t][i], NaN-propagating like torch.maximum
// (dlib/datasets/wsol_loader.py:591-600)
__global__ void __launch_bounds__(kThreads) temporal_max_kernel(const float *__restrict__ cams,
                                                                float *__restrict__ out, int T, int HW,
                                                                long long total)
{
    const long long stride = (long long)gridDim.x * kThreads;
    for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < total; i += stride) {
        const long long b = i / HW;
        const int px = (int)(i - b * HW);
        const float *src = cams + (size_t)b * T * HW + px;
        float m = __ldg(src);
        for (int t = 1; t < T; t++) {
            const float v = __ldg(src + (size_t)t * HW);
            // torch.maximum: if either is NaN the result is NaN
            m = (m != m) ? m : ((v != v) ? v : (v > m ? v : m));
        }
        out[i] = m;
    }
}

// ---------------------------------------------------------------------------
// host-side drivers
// ---------------------------------------------------------------------------

// Vertex density of the recent calls, per workspace (density_hint below).
struct DensityHints {
    struct Slot {
        void *ws;
        int *word;            // pinned
        unsigned int calls;   // calls seen on this workspace
    };
    std::mutex mu;
    std::vector<Slot> slots;   // a handful of workspaces per process
    cudaStream_t side = nullptr;                   // the copies run here, off the caller's stream
    cudaEvent_t ev = nullptr;
    // caller holds `mu`
    Slot *find(void *ws, bool create)
    {
        for (auto &s : slots)
            if (s.ws == ws) return &s;
        if (!create) return nullptr;
        int *p = nullptr;
        if (cudaHostAlloc((void **)&p, sizeof(int), cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        *p = 0;
        slots.push_back({ws, p, 0u});
        return &slots.back();
    }
};

// The copy stream of the host-frames path (run_chunk_host_frames) and the events that fork and join it.
struct CopyLane {
    std::mutex mu;
    cudaStream_t stream = nullptr;
    std::vector<cudaEvent_t> events;
    size_t next = 0;
    int ready()   // this device's copy stream, created on first use
    {
        if (stream) return TCAMCRF_OK;
        CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        return TCAMCRF_OK;
    }
    int event(cudaEvent_t *ev)
    {
        if (events.size() < 64) {
            cudaEvent_t e = nullptr;
            CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            events.push_back(e);
            *ev = e;
            return TCAMCRF_OK;
        }
        *ev = events[next++ % events.size()];   // a waiter keeps the record it was given: re-recording is safe
        return TCAMCRF_OK;
    }
};

// Cached buffers, streams and events of the host-pointer path (host_run).
struct HostCtx {
    std::mutex mu;
    void *buf = nullptr;
    size_t cap = 0;
    cudaStream_t stream = nullptr;   // compute
    cudaStream_t s_in = nullptr;     // host -> device copies
    cudaStream_t s_out = nullptr;    // device -> host copies
    std::vector<cudaEvent_t> events;
    void *pin = nullptr;             // pinned staging: grad_out in, per-group losses and status words out
    size_t pin_cap = 0;
};

// Captured schedules of host_run, a handful per device (a trainer alternates between a few pinned buffers).
struct HostGraphs {
    struct Key {
        tcamcrf_config cfg;
        int N, K, H, W;
        const void *images, *segs, *as_host, *grad_host, *buf, *pin;
        int want_loss, dedup, dense, groups_knob, sec0_knob, grow_knob;
        bool operator==(const Key &o) const { return memcmp(this, &o, sizeof(Key)) == 0; }
    };
    struct Item {
        Key key;
        cudaGraphExec_t exec;
        int groups;
        long long launches;      // kernels of one replay (for tcamcrf_launch_count)
        unsigned long long used;
    };
    std::vector<Item> items;
    unsigned long long tick = 0;
    void clear()
    {
        for (auto &it : items) cudaGraphExecDestroy(it.exec);
        items.clear();
    }
};

// What the library keeps per CUDA device: a process may drive several (threads of DataParallel, or alternating
// cuda:0 / cuda:1), and each gets its own limits, kernel attributes, streams, events and buffers.
struct Device {
    std::once_flag once;
    int sms = 148;                           // multiprocessors
    int select_smem = 0;                     // dynamic shared memory of seed_select_smem_kernel (0: opt-in refused)
    int fused_smem = 0;                      // the same for seed_fused_kernel
    DensityHints hints;
    CopyLane lane;
    HostCtx host;
    HostGraphs graphs;                       // guarded by host.mu
    std::vector<cudaEvent_t> timing_events;  // free events of the stage profiler, guarded by g_prof.mu

    void init(int ordinal)   // runs once, with this device current
    {
        int v = 0, optin = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, ordinal) == cudaSuccess && v > 0) sms = v;
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ordinal);
        cudaFuncAttributes fa;
        int stat = 12 * 1024;
        if (cudaFuncGetAttributes(&fa, seed_fused_kernel) == cudaSuccess) stat = (int)fa.sharedSizeBytes;
        const int sel = optin - 2048, fused = optin - stat - 1024;   // 2 KB: seed_select_smem_kernel's static smem
        const cudaFuncAttribute smem = cudaFuncAttributeMaxDynamicSharedMemorySize;
        if (sel > 0 && cudaFuncSetAttribute(seed_select_smem_kernel, smem, sel) == cudaSuccess) select_smem = sel;
        if (fused > 0 && cudaFuncSetAttribute(seed_fused_kernel, smem, fused) == cudaSuccess) fused_smem = fused;
        cudaGetLastError();   // a refused opt-in leaves the kernel at the default limit: not an error of any call
    }
    cudaEvent_t timing_event()
    {
        cudaEvent_t e = nullptr;
        if (timing_events.empty()) {
            cudaEventCreate(&e);
            return e;
        }
        e = timing_events.back();
        timing_events.pop_back();
        return e;
    }
};
constexpr int kMaxDevices = 64;
static Device g_devices[kMaxDevices];

// The context of the current device, set up on its first use.
static int this_device(Device **out)
{
    int ordinal = 0;
    CUDA_TRY(cudaGetDevice(&ordinal));
    if (ordinal < 0 || ordinal >= kMaxDevices)
        return fail(TCAMCRF_ERR_INVALID, "device %d: the library serves devices 0..%d", ordinal, kMaxDevices - 1);
    Device &dev = g_devices[ordinal];
    std::call_once(dev.once, [&] { dev.init(ordinal); });
    *out = &dev;
    return TCAMCRF_OK;
}

// persistent kernels: one wave of resident CTAs (8 x 256 threads per SM)
static int persistent_grid(const Device &dev) { return dev.sms * 8; }

// Exactly one resident wave of `kernel` (what its register use allows), so that the frame-ordered sweep of
// the vertex kernels really has all blocks on the same frame at the same time.
template <typename Kernel>
static int resident_grid(const Device &dev, Kernel kernel)
{
    static const int per_sm = [kernel] {   // one instance per kernel type; depends on the architecture only
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, kThreads, 0) != cudaSuccess || n < 1) {
            cudaGetLastError();
            n = 4;
        }
        return n;
    }();
    return per_sm * dev.sms;
}

// ---------------------------------------------------------------------------
// optional per-stage timing (CUDA events on the caller's stream) + launch counter
// ---------------------------------------------------------------------------
enum Stage { kStBuild = 0, kStNeighbour, kStSplat, kStBlur, kStSlice, kStLoss, kStBackward, kStPrepare, kStSeed, kStCount };
static_assert(kStCount == TCAMCRF_STAGES, "stage list and header disagree");

struct Profiler {
    std::mutex mu;
    bool enabled = false;
    struct Span {
        int stage;
        int launches;
        Device *dev;   // whose pool the events go back to
        cudaEvent_t a, b;
    };
    std::vector<Span> spans;
    double ms[kStCount] = {0};
    long long launches[kStCount] = {0};
    long long total_launches = 0;
};
static Profiler g_prof;

// Brackets the launches of one stage.  When profiling is off it only counts launches.
struct StageScope {
    int stage, launches;
    cudaStream_t st;
    Device *dev = nullptr;
    cudaEvent_t a = nullptr;
    StageScope(int stage_, int launches_, cudaStream_t st_) : stage(stage_), launches(launches_), st(st_)
    {
        static const char *const names[kStCount] = {"tcamcrf:build", "tcamcrf:neighbour", "tcamcrf:splat", "tcamcrf:blur",
                                                    "tcamcrf:slice", "tcamcrf:loss", "tcamcrf:backward",
                                                    "tcamcrf:prepare", "tcamcrf:seed"};
        nvtxRangePushA(names[stage]);   // host-side range around the launches of the stage (nsys / ncu --nvtx)
        std::lock_guard<std::mutex> lock(g_prof.mu);
        g_prof.total_launches += launches;
        if (g_prof.enabled && this_device(&dev) == TCAMCRF_OK) {
            a = dev->timing_event();
            cudaEventRecord(a, st);
        }
    }
    ~StageScope()
    {
        nvtxRangePop();
        if (!a) return;
        std::lock_guard<std::mutex> lock(g_prof.mu);
        cudaEvent_t b = dev->timing_event();
        cudaEventRecord(b, st);
        g_prof.spans.push_back({stage, launches, dev, a, b});
    }
};

static void scale_factors(int d, EmbedConsts &ec)
{
    // evaluated exactly like the reference: float inv_std_dev, double expression, narrowed to float
    // (permutohedral.cpp:156-159)
    const float inv_std_dev = (float)(sqrt(2.0 / 3.0) * (d + 1));
    for (int i = 0; i < kMaxD; i++) ec.scale[i] = 0.f;
    for (int i = 0; i < d; i++) ec.scale[i] = (float)(1.0 / sqrt((double)((i + 2) * (i + 1))) * inv_std_dev);
}

// Launches `kernel` as a programmatic dependent of the previous kernel on `st` (see pdl_wait above).
template <typename... KArgs, typename... Args>
static void launch_chained_block(void (*kernel)(KArgs...), dim3 grid, int threads, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = grid;
    lc.blockDim = dim3(threads);
    lc.dynamicSmemBytes = 0;
    lc.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    cudaLaunchKernelEx(&lc, kernel, std::forward<Args>(args)...);
}
template <typename... KArgs, typename... Args>
static void launch_chained(void (*kernel)(KArgs...), dim3 grid, cudaStream_t st, Args &&...args)
{
    launch_chained_block(kernel, grid, kThreads, st, std::forward<Args>(args)...);
}

template <int D, typename ImgT>
static void launch_build(const BuildParams &bp, dim3 grid, bool dedup, cudaStream_t st)
{
    if (dedup)
        launch_chained_block(build_dedup_kernel<D, ImgT>, grid, kTileThreads, st, bp);
    else
        launch_chained(build_kernel<D, ImgT>, grid, st, bp);
}

template <int D, int V>
static void launch_pixel_v(bool splat, bool lowp, const PixelParams &pp, dim3 grid, cudaStream_t st)
{
    if constexpr (V > 1) {   // (2-byte logits always have K >= 2, hence V >= 2)
        if (lowp) {
            if (splat)
                launch_chained(splat_lowp_kernel<D, V>, grid, st, pp);
            else
                launch_chained(slice_lowp_kernel<D, V>, grid, st, pp);
            return;
        }
    }
    if (splat) {
        if (pp.logits)
            launch_chained(splat_kernel<D, V, true>, grid, st, pp);
        else
            launch_chained(splat_kernel<D, V, false>, grid, st, pp);
    } else {
        if (pp.logits)
            launch_chained(slice_kernel<D, V, true>, grid, st, pp);
        else
            launch_chained(slice_kernel<D, V, false>, grid, st, pp);
    }
}

template <int D, int KV>
static void launch_splat_rows(bool lowp, const PixelParams &pp, int frames, cudaStream_t st)
{
    const dim3 grid((pp.P + RowMap<KV>::kPpb - 1) / RowMap<KV>::kPpb, frames);
    if (lowp)
        launch_chained(splat_rows_lowp_kernel<D, KV>, grid, st, pp);
    else if (pp.logits)
        launch_chained(splat_rows_kernel<D, KV, true>, grid, st, pp);
    else
        launch_chained(splat_rows_kernel<D, KV, false>, grid, st, pp);
}

// lowp: the logits are 2-byte (pp.bf16 says which type)
template <int D>
static void launch_pixel(bool splat, bool lowp, int V, const PixelParams &pp, dim3 grid, cudaStream_t st)
{
    if (splat && pp.dense && V == 4) {
        switch (pp.Kp / 4) {   // rows of 2..4 float4s (K = 5..16)
        case 2: return launch_splat_rows<D, 2>(lowp, pp, grid.y, st);
        case 3: return launch_splat_rows<D, 3>(lowp, pp, grid.y, st);
        case 4: return launch_splat_rows<D, 4>(lowp, pp, grid.y, st);
        default: break;
        }
    }
    if (V == 4)
        launch_pixel_v<D, 4>(splat, lowp, pp, grid, st);
    else if (V == 2)
        launch_pixel_v<D, 2>(splat, lowp, pp, grid, st);
    else
        launch_pixel_v<D, 1>(splat, lowp, pp, grid, st);
}

template <int V, int KV>
static void launch_blur_kv(const Device &dev, const BlurParams &bp, int nc, cudaStream_t st)
{
    launch_chained(blur_kernel<V, KV>, dim3(resident_grid(dev, blur_kernel<V, KV>)), st, bp, nc);
}

static void launch_blur(const Device &dev, int V, const BlurParams &bp, int nc, cudaStream_t st)
{
    const int kv = bp.Kp / V;
    if (V == 4) {
        switch (kv) {
        case 1: return launch_blur_kv<4, 1>(dev, bp, nc, st);
        case 2: return launch_blur_kv<4, 2>(dev, bp, nc, st);
        case 3: return launch_blur_kv<4, 3>(dev, bp, nc, st);   // K = 9..12
        case 4: return launch_blur_kv<4, 4>(dev, bp, nc, st);
        case 6: return launch_blur_kv<4, 6>(dev, bp, nc, st);   // K = 21..24 (VOC's 21 classes)
        default: return launch_blur_kv<4, 0>(dev, bp, nc, st);
        }
    }
    if (V == 2) return launch_blur_kv<2, 1>(dev, bp, nc, st);   // Kp = 2 is the only even, non-multiple-of-4 row width
    return launch_blur_kv<1, 1>(dev, bp, nc, st);               // Kp = 1
}

static int density_hint(Device &dev, void *ws);   // largest per-frame vertex count lately on ws (0: unknown); below

// "Dense" lattice: more than one vertex per four pixels in the fullest frame lately (iid-noise frames have ~1.1 per
// pixel, real frames ~0.06).  Selects kernel variants that are both correct for every input.
static bool lattice_is_dense(int hint, int P) { return (long long)hint * 4 > (long long)P; }

// Stage 1 of a chunk: the lattice of `nc` frames (tables, per-pixel vertices and weights, blur links).  Needs
// only the images.  `zero_values`: also clear the value rows in the same launch (the device path does; the
// host path clears them group by group in value_stages).
template <int D>
static int lattice_stages(Device &dev, const tcamcrf_config *cfg, const Plan &pl, bool u8, const void *images,
                          int frame0, int nc, char *ws, bool zero_values, cudaStream_t st)
{
    int *ctrl = (int *)(ws + pl.off_ctrl);
    Entry *table = (Entry *)(ws + pl.off_table);
    {
        StageScope scope(kStPrepare, 1, st);
        prepare_kernel<<<persistent_grid(dev), kThreads, 0, st>>>(table, ctrl, frame0, nc, pl.chunk, pl.geom, pl.sig);
    }
    {
        StageScope scope(kStBuild, 1, st);
        BuildParams bp;
        bp.images = images;
        bp.table = table;
        bp.offset = (int *)(ws + pl.off_offset);
        bp.bary = (float *)(ws + pl.off_bary);
        bp.vkey = (unsigned long long *)(ws + pl.off_vkey);
        bp.ctrl = ctrl;
        bp.P = pl.P;
        bp.W = pl.W;
        bp.H = pl.H;
        bp.stride_planes = cfg->image_stride_planes;
        bp.channels = cfg->channels;
        bp.feat = cfg->feat;
        bp.geom = pl.geom;
        bp.slots = pl.slots;
        bp.stride = pl.stride;
        bp.pool = pl.pool;
        bp.sigma_rgb = cfg->sigma_rgb;
        bp.sigma_xy = cfg->sigma_xy;
        bp.frame0 = frame0;
        scale_factors(D, bp.ec);
        dim3 bgrid(nc, pl.blocks_per_frame);
        // sparse lattice lately (or nothing known yet): deduplicate the block's keys in shared memory first
        bool dedup = !lattice_is_dense(density_hint(dev, ws), pl.P);
        if (tuning().build_dedup >= 0) dedup = tuning().build_dedup != 0;   // tests and sweeps: force either way
        if (dedup)   // one block per 32 x 8 tile; one more row of blocks for the ghost pixel's block
            bgrid = dim3(nc, (pl.H + kTileH - 1) / kTileH + ((pl.P & 3) != 0 ? 1 : 0), (pl.W + kTileW - 1) / kTileW);
        if (u8)
            launch_build<D, uint8_t>(bp, bgrid, dedup, st);
        else
            launch_build<D, float>(bp, bgrid, dedup, st);
    }
    VertexParams vp;
    vp.table = table;
    vp.vkey = (unsigned long long *)(ws + pl.off_vkey);
    vp.nbr = (int2 *)(ws + pl.off_nbr);
    vp.values = (float *)(ws + pl.off_val0);
    vp.ctrl = ctrl;
    vp.geom = pl.geom;
    vp.slots = pl.slots;
    vp.stride = pl.stride;
    vp.pool = pl.pool;
    vp.Kp = pl.Kp;
    vp.sig = pl.sig;
    vp.frame0 = frame0;
    vp.zero_values = zero_values ? 1 : 0;
    {
        StageScope scope(kStNeighbour, 1, st);
        launch_chained(neighbour_kernel<D>, dim3(resident_grid(dev, neighbour_kernel<D>)), st, vp, nc);
    }
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

// (the density hint is refreshed by the callers AFTER the value stages: an asynchronous copy between the
// neighbour kernel and the splat would break the programmatic launch chain)

// Vertex density of the recent calls on a workspace, for the HOST: after every lattice build the largest per-frame
// vertex count (kCtrlPrevMax) is copied into a pinned word with an asynchronous device-to-host copy on the caller's
// stream -- no synchronisation; the next calls read whatever has arrived (one or two calls old).  It only selects
// between kernels that are both correct for every input.
static bool stream_is_capturing(cudaStream_t st)
{
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &status) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return status != cudaStreamCaptureStatusNone;
}

// largest per-frame vertex count seen lately on this workspace (0: unknown)
static int density_hint(Device &dev, void *ws)
{
    std::lock_guard<std::mutex> lock(dev.hints.mu);
    DensityHints::Slot *slot = dev.hints.find(ws, false);
    return slot ? *(volatile int *)slot->word : 0;
}

// Queue the refresh of the hint behind the work already on `st`, on a side stream: the caller's stream never waits
// for the copy (in-stream it costs ~5 us per call, more than the hint is worth on short steps).  Nothing is done
// while a graph is being captured (an unjoined fork is not capturable; the hint then keeps its last value).
static void density_hint_refresh(Device &dev, const Plan &pl, char *ws, cudaStream_t st)
{
    if (stream_is_capturing(st)) return;   // (also: no pinned allocation while a capture is open)
    std::lock_guard<std::mutex> lock(dev.hints.mu);
    DensityHints::Slot *slot = dev.hints.find(ws, true);
    if (!slot) return;
    // every 8th call is plenty for a hint (the three driver calls below cost ~10 us of host time, which shows on
    // 0.25 ms steps); the first two calls on a workspace always refresh
    const unsigned int c = slot->calls++;
    if (c >= 2 && (c & 7u) != 0) return;
    if (!dev.hints.side) {   // this device's side stream, created on first use
        if (cudaStreamCreateWithFlags(&dev.hints.side, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&dev.hints.ev, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            dev.hints.side = nullptr;
            return;
        }
    }
    cudaEventRecord(dev.hints.ev, st);
    cudaStreamWaitEvent(dev.hints.side, dev.hints.ev, 0);
    cudaMemcpyAsync(slot->word, ws + pl.off_ctrl + kCtrlPrevMax * sizeof(int), sizeof(int), cudaMemcpyDeviceToHost,
                    dev.hints.side);
}

// Stage 2: splat -> blur x(d+1) -> slice (+ loss) for the frames [frame0, frame0 + nc) of a chunk whose lattice
// is built.  segs / as_out point at frame0.  `zero_values`: the value rows were not cleared by lattice_stages.
template <int D>
static int value_stages(Device &dev, const Plan &pl, const void *segs, float *as_out, int frame0, int nc, char *ws,
                        bool zero_values, bool want_loss, float *loss_final, float n_norm, int flags, cudaStream_t st)
{
    int *ctrl = (int *)(ws + pl.off_ctrl);
    int2 *nbr = (int2 *)(ws + pl.off_nbr);
    float *val0 = (float *)(ws + pl.off_val0);
    float *val1 = (float *)(ws + pl.off_val1);
    if (zero_values) {
        VertexParams vp;
        memset(&vp, 0, sizeof(vp));
        vp.nbr = nbr;
        vp.values = val0;
        vp.ctrl = ctrl;
        vp.stride = pl.stride;
        vp.pool = pl.pool;
        vp.Kp = pl.Kp;
        vp.frame0 = frame0;
        vp.zero_values = 1;
        StageScope scope(kStSplat, 1, st);
        vertex_init_kernel<<<resident_grid(dev, vertex_init_kernel), kThreads, 0, st>>>(vp, nc);
    }
    const dim3 pgrid(pl.blocks_per_frame, nc);
    const int V = (pl.Kp % 4 == 0) ? 4 : (pl.Kp % 2 == 0) ? 2 : 1;
    PixelParams pp;
    pp.segs = segs;
    pp.logits = flags & kFlagLogits;
    pp.bf16 = (flags & kFlagBF16) ? 1 : 0;
    const bool lowp = (flags & kFlagLowp) != 0;
    pp.as_out = as_out;
    pp.offset = (int *)(ws + pl.off_offset);
    pp.bary = (float *)(ws + pl.off_bary);
    pp.table = (Entry *)(ws + pl.off_table);
    pp.values = val0;
    pp.partial = want_loss ? (float *)(ws + pl.off_partial) : nullptr;
    pp.ctrl = ctrl;
    pp.acc = (double *)(ws + pl.off_acc);
    pp.loss_out = loss_final;
    pp.n_norm = n_norm;
    pp.loss_scale = pl.loss_weight;
    pp.P = pl.P;
    pp.K = pl.K;
    pp.Kp = pl.Kp;
    pp.frame0 = frame0;
    // dense lattice lately (more than one vertex per four pixels in the fullest frame): row-cooperative splat
    pp.dense = lattice_is_dense(density_hint(dev, ws), pl.P) ? 1 : 0;
    if (tuning().dense >= 0) pp.dense = tuning().dense != 0;   // tests and sweeps: force either way
    pp.pool = pl.pool;
    pp.alpha = 1.0f / (1 + powf(2, -D));
    {
        StageScope scope(kStSplat, 1, st);
        launch_pixel<D>(true, lowp, V, pp, pgrid, st);
    }

    float *src = val0, *dst = val1;
    {
        StageScope scope(kStBlur, D + 1, st);
        for (int j = 0; j <= D; j++) {
            BlurParams bl;
            bl.src = src;
            bl.dst = dst;
            // axes 0..d like the reference (permutohedral.cpp:537); d..0 gives the transposed filter, because
            // every single-axis blur is symmetric
            bl.nbr = nbr + (size_t)((flags & kFlagReverseBlur) ? D - j : j) * pl.pool;
            bl.ctrl = ctrl;
            bl.Kp = pl.Kp;
            bl.stride = pl.stride;
            bl.frame0 = frame0;
            launch_blur(dev, V, bl, nc, st);
            float *t = src;
            src = dst;
            dst = t;
        }
    }

    pp.values = src;
    {
        StageScope scope(kStSlice, 1, st);
        launch_pixel<D>(false, lowp, V, pp, pgrid, st);
    }
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

#define TCAMCRF_DISPATCH_D(dim, call)                                                   \
    switch (dim) {                                                                      \
    case 1: { constexpr int D = 1; return call; }                                       \
    case 2: { constexpr int D = 2; return call; }                                       \
    case 3: { constexpr int D = 3; return call; }                                       \
    case 4: { constexpr int D = 4; return call; }                                       \
    case 5: { constexpr int D = 5; return call; }                                       \
    case 6: { constexpr int D = 6; return call; }                                       \
    }                                                                                   \
    return fail(TCAMCRF_ERR_INVALID, "unsupported lattice dimension %d", dim)

// `images` points at frame 0 of the chunk; the lattice of frames [frame0, frame0 + nc) is built.
static int run_lattice(Device &dev, const tcamcrf_config *cfg, const Plan &pl, bool u8, const void *images, int frame0,
                       int nc, char *ws, bool zero_values, cudaStream_t st)
{
    TCAMCRF_DISPATCH_D(pl.D, lattice_stages<D>(dev, cfg, pl, u8, images, frame0, nc, ws, zero_values, st));
}

static int run_values(Device &dev, const Plan &pl, const void *segs, float *as_out, int frame0, int nc, char *ws,
                      bool zero_values, bool want_loss, float *loss_final, float n_norm, int flags, cudaStream_t st)
{
    TCAMCRF_DISPATCH_D(pl.D, value_stages<D>(dev, pl, segs, as_out, frame0, nc, ws, zero_values, want_loss, loss_final,
                                             n_norm, flags, st));
}

static int run_chunk(Device &dev, const tcamcrf_config *cfg, const Plan &pl, bool u8, const void *images,
                     const void *segs, float *as_out, int nc, char *ws, bool want_loss, float *loss_final,
                     float n_norm, int flags, cudaStream_t st)
{
    int rc = run_lattice(dev, cfg, pl, u8, images, 0, nc, ws, true, st);
    if (rc) return rc;
    rc = run_values(dev, pl, segs, as_out, 0, nc, ws, false, want_loss, loss_final, n_norm, flags, st);
    density_hint_refresh(dev, pl, ws, st);
    return rc;
}

// Frames that are still in HOST memory (the reference's trainer keeps raw_img on the CPU, train_wsol.py:1128, and
// hands it to DenseCRFLoss.forward every step): they are copied section by section on a copy stream of the
// library while the lattice of the sections that have arrived is being built on the caller's stream, instead of
// one copy followed by one build.  Fork/join with events only: nothing synchronises, and the pattern can be
// captured in a CUDA graph (pinned source).
//
// One chunk whose frames come from the host: `img_host` / `img_dev` point at frame 0 of the chunk.
static int run_chunk_host_frames(Device &dev, const tcamcrf_config *cfg, const Plan &pl, bool u8, const char *img_host,
                                 char *img_dev, const void *segs, float *as_out, int nc, bool first_chunk,
                                 bool last_chunk, char *ws, bool want_loss, float *loss_final, float n_norm, int flags,
                                 cudaStream_t st)
{
    // sections of at least 4 frames, 4 per chunk by default (32 frames: 8 + 8 + 8 + 8)
    int nsec = 4;
    if (tuning().himg_sections >= 1 && tuning().himg_sections <= 64) nsec = tuning().himg_sections;
    int per = (nc + nsec - 1) / nsec;
    if (per < 4) per = nc < 4 ? nc : 4;
    const size_t elem = u8 ? 1 : sizeof(float);
    const size_t frame = (size_t)cfg->image_stride_planes * pl.P;   // elements per image
    std::lock_guard<std::mutex> lock(dev.lane.mu);
    int rc = dev.lane.ready();
    if (rc) return rc;
    cudaEvent_t ev;
    if (first_chunk) {
        // the staging buffer may still be read by work queued earlier on the caller's stream; later chunks of the
        // call use other parts of it, and their copies simply queue behind the first chunk's on the copy stream
        rc = dev.lane.event(&ev);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(ev, st));
        CUDA_TRY(cudaStreamWaitEvent(dev.lane.stream, ev, 0));
    }
    for (int f0 = 0; f0 < nc; f0 += per) {
        const int fn = nc - f0 < per ? nc - f0 : per;
        size_t elems = (size_t)fn * frame;
        // the very last image of the batch may be shorter than the stride (see host_run)
        if (last_chunk && f0 + fn == nc) elems = ((size_t)(fn - 1) * cfg->image_stride_planes + cfg->channels) * pl.P;
        CUDA_TRY(cudaMemcpyAsync(img_dev + (size_t)f0 * frame * elem, img_host + (size_t)f0 * frame * elem, elems * elem,
                                 cudaMemcpyHostToDevice, dev.lane.stream));
        rc = dev.lane.event(&ev);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(ev, dev.lane.stream));
        CUDA_TRY(cudaStreamWaitEvent(st, ev, 0));
        rc = run_lattice(dev, cfg, pl, u8, img_dev, f0, fn, ws, true, st);
        if (rc) return rc;
    }
    rc = run_values(dev, pl, segs, as_out, 0, nc, ws, false, want_loss, loss_final, n_norm, flags, st);
    density_hint_refresh(dev, pl, ws, st);
    return rc;
}

// `images_host` != NULL: the frames are there (same element type) and `images` is the device buffer they are
// staged in.  `segs` holds float32 values, or 2-byte logits with kFlagLowp.
static int run_filter(const tcamcrf_config *cfg, bool u8, const void *images, const void *segs, float *as_out,
                      float *loss, int N, int K, int H, int W, float n_norm, void *workspace, size_t ws_bytes,
                      cudaStream_t st, int flags = 0, const void *images_host = nullptr)
{
    if (!cfg || !images || !segs || !as_out || !workspace) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    Plan pl;
    int rc = make_plan(cfg, N, K, H, W, pl);
    if (rc) return rc;
    if (ws_bytes < pl.total)
        return fail(TCAMCRF_ERR_WORKSPACE, "workspace too small: %zu < %zu bytes", ws_bytes, pl.total);
    if (((uintptr_t)workspace & 255) != 0) return fail(TCAMCRF_ERR_WORKSPACE, "workspace must be 256-byte aligned");
    const size_t seg_elem = (flags & kFlagLowp) ? 2 : 4;
    if (((uintptr_t)segs & (seg_elem - 1)) || ((uintptr_t)as_out & 3) || (!u8 && ((uintptr_t)images & 3)))
        return fail(TCAMCRF_ERR_INVALID, "buffers must be aligned to their element size");
    Device *dev = nullptr;
    rc = this_device(&dev);
    if (rc) return rc;
    char *ws = (char *)workspace;
    // status word + loss accumulator start clean for this call (MAGIC / DIRTY persist with the workspace)
    CUDA_TRY(cudaMemsetAsync(ws + pl.off_ctrl, 0, kCtrlResetInts * sizeof(int), st));
    const size_t img_elem = u8 ? 1 : 4;
    for (int n0 = 0; n0 < N; n0 += pl.chunk) {
        const int nc = (N - n0) < pl.chunk ? (N - n0) : pl.chunk;
        const char *img = (const char *)images + (size_t)n0 * cfg->image_stride_planes * pl.P * img_elem;
        const bool last = n0 + nc >= N;
        if (images_host)
            rc = run_chunk_host_frames(*dev, cfg, pl, u8,
                                       (const char *)images_host + (size_t)n0 * cfg->image_stride_planes * pl.P * img_elem,
                                       const_cast<char *>(img), (const char *)segs + (size_t)n0 * K * pl.P * seg_elem,
                                       as_out + (size_t)n0 * K * pl.P, nc, n0 == 0, last, ws, loss != nullptr,
                                       last ? loss : nullptr, n_norm, flags, st);
        else
            rc = run_chunk(*dev, cfg, pl, u8, img, (const char *)segs + (size_t)n0 * K * pl.P * seg_elem, as_out + (size_t)n0 * K * pl.P, nc, ws,
                           loss != nullptr, last ? loss : nullptr, n_norm, flags, st);
        if (rc) return rc;
    }
    return TCAMCRF_OK;
}

// ---------------------------------------------------------------------------
// host-pointer (drop-in) path: cached device buffers, chunk-pipelined copies
// ---------------------------------------------------------------------------
static int host_pin_reserve(HostCtx &g_host, size_t bytes)
{
    if (g_host.pin_cap >= bytes) return TCAMCRF_OK;
    if (g_host.pin) cudaFreeHost(g_host.pin);
    g_host.pin = nullptr;
    g_host.pin_cap = 0;
    CUDA_TRY(cudaHostAlloc(&g_host.pin, bytes * 2, cudaHostAllocDefault));
    g_host.pin_cap = bytes * 2;
    return TCAMCRF_OK;
}

static int host_reserve(HostCtx &g_host, size_t bytes, char **out)
{
    for (cudaStream_t *s : {&g_host.stream, &g_host.s_in, &g_host.s_out})
        if (!*s) CUDA_TRY(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
    if (g_host.cap < bytes) {
        if (g_host.buf) cudaFree(g_host.buf);
        g_host.buf = nullptr;
        g_host.cap = 0;
        CUDA_TRY(cudaMalloc(&g_host.buf, bytes));
        g_host.cap = bytes;
    }
    *out = (char *)g_host.buf;
    return TCAMCRF_OK;
}

static int host_event(HostCtx &g_host, size_t i, cudaEvent_t *ev)
{
    while (g_host.events.size() <= i) {
        cudaEvent_t e = nullptr;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        g_host.events.push_back(e);
    }
    *ev = g_host.events[i];
    return TCAMCRF_OK;
}

// TCAMCRF_HOST_TRACE=1: timeline of one host_run call (timing events on the three streams), printed to stderr.
struct HostTrace {
    bool on = false;
    struct Mark { const char *what; int idx; cudaEvent_t ev; };
    std::vector<Mark> marks;
    cudaEvent_t t0 = nullptr;
    struct timespec h0;
    void begin(cudaStream_t s)
    {
        on = tuning().host_trace != 0;
        if (!on) return;
        cudaEventCreate(&t0);
        cudaEventRecord(t0, s);
        clock_gettime(CLOCK_MONOTONIC, &h0);
    }
    // host wall clock since begin(): how long the CPU took to get here (enqueueing is not free)
    void host_mark(const char *what)
    {
        if (!on) return;
        struct timespec h1;
        clock_gettime(CLOCK_MONOTONIC, &h1);
        fprintf(stderr, "[host trace] %-12s host %7.3f ms\n", what, (h1.tv_sec - h0.tv_sec) * 1e3 + (h1.tv_nsec - h0.tv_nsec) * 1e-6);
    }
    void mark(const char *what, int idx, cudaStream_t s)
    {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        marks.push_back({what, idx, e});
    }
    void end()
    {
        if (!on) return;
        for (auto &m : marks) {
            float ms = 0.f;
            cudaEventSynchronize(m.ev);
            cudaEventElapsedTime(&ms, t0, m.ev);
            fprintf(stderr, "[host trace] %-12s %2d  %7.3f ms\n", m.what, m.idx, ms);
            cudaEventDestroy(m.ev);
        }
        cudaEventDestroy(t0);
    }
};

static int check_device()
{
    int n = tcamcrf_device_count();
    if (n <= 0) return fail(TCAMCRF_ERR_NO_DEVICE, "no sm_100 (B200) device visible; this library has no CPU path");
    return TCAMCRF_OK;
}

// Filter (and optionally loss + gradient) with host buffers, pipelined over three streams (host->device
// copies, kernels, device->host copies; truly asynchronous when the host buffers are pinned, pageable buffers
// still work, the copies are then staged by the driver).
//
// The lattice depends on the images only, and the images are the small input (12 bytes per pixel against 4K
// for the segmentations).  So the images go first, the lattice is built while the segmentations are still on the
// wire, and only the value stages (splat, blur, slice, gradient) run group by group as the segmentations of a group
// arrive; the results of a group go back while the next group computes.  The PCIe link is the bound of this path
// (one step's bytes in, one step's bytes out): what is left on top of it is the tail -- value stages and copy back
// of the LAST group -- so the groups shrink towards the end of the batch.
//
// One call is ~200 driver calls (copies, events, ~130 launches): about as long on the CPU as the link needs for the
// bytes.  With pinned buffers the whole schedule is therefore captured ONCE into a CUDA graph, keyed by the problem
// and the buffer addresses, and a call is one graph launch (HostGraphs).
struct HostJob {
    tcamcrf_config cfg;
    Plan pl;
    const float *images, *segs;
    float *as_host, *grad_host;
    bool want_loss;
    int N, K, H, W;
    // device buffers (inside g_host.buf) and pinned staging (g_host.pin)
    float *d_img, *d_seg, *d_as, *d_grad, *d_scal, *d_loss;
    int *d_status;
    char *d_ws;
    float *h_gout;      // pinned: grad_out of this call
    float *h_loss;      // pinned: per-group losses
    int *h_status;      // pinned: per-group status words
    int max_groups;
    bool dedup_hint, dense_hint;   // part of the graph key: the kernel variants are chosen at enqueue time
};

// group sizes of the value stages for `frames` frames: groups of `size` frames, the last one shorter
static void host_groups(int frames, int size, std::vector<int> &out)
{
    out.clear();
    for (int left = frames; left > 0; left -= size) out.push_back(size < left ? size : left);
}

// Queues the whole call on the three streams.  `st` is the origin: s_in / s_out fork from it and join it again, so
// the same code runs eagerly or under stream capture.  `groups_out`: number of groups (entries of h_loss / h_status).
static int host_enqueue(Device &dev, const HostJob &j, HostTrace &trace, int *groups_out)
{
    HostCtx &g_host = dev.host;
    const Plan &pl = j.pl;
    const int N = j.N, K = j.K;
    cudaStream_t st = g_host.stream, s_in = g_host.s_in, s_out = g_host.s_out;
    const size_t P = (size_t)j.H * j.W;
    const size_t img_frame = (size_t)j.cfg.image_stride_planes * P;   // floats per image
    const size_t seg_frame = (size_t)K * P;
    size_t ev_i = 0;
    int rc;
    cudaEvent_t ev_fork;
    rc = host_event(g_host, ev_i++, &ev_fork);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(ev_fork, st));
    CUDA_TRY(cudaStreamWaitEvent(s_in, ev_fork, 0));
    CUDA_TRY(cudaStreamWaitEvent(s_out, ev_fork, 0));
    if (j.grad_host) CUDA_TRY(cudaMemcpyAsync(j.d_scal, j.h_gout, sizeof(float), cudaMemcpyHostToDevice, s_in));
    // Value-stage groups (measured on B200, tools/r2_host_sweep.sh, 32 frames): wide batches (K >= 6: the
    // segmentations are most of the bytes) in groups of 2 frames, so that results flow back almost as soon as their
    // inputs are in (K=10: 2.18 -> 2.06 ms per call); narrow ones in groups of a quarter chunk.  TCAMCRF_HOST_GROUPS
    // = groups per chunk.
    int group = K >= 6 ? 2 : (pl.chunk + 3) / 4;
    if (tuning().host_groups >= 1 && tuning().host_groups <= 64)
        group = (pl.chunk + tuning().host_groups - 1) / tuning().host_groups;
    if (group < 1) group = 1;
    std::vector<int> sizes;
    int gi = 0;   // running group index
    for (int c0 = 0; c0 < N; c0 += pl.chunk) {
        const int cn = (N - c0) < pl.chunk ? (N - c0) : pl.chunk;
        // status word + loss accumulator start clean (MAGIC / DIRTY persist with the workspace)
        CUDA_TRY(cudaMemsetAsync(j.d_ws + pl.off_ctrl, 0, kCtrlResetInts * sizeof(int), st));
        // Sections: the lattice of a first, small section is built as soon as its images are in, so that the first
        // results start their way back early (the link carries ~55 GB/s one way but only ~88 GB/s both ways together:
        // every millisecond in which nothing flows back is lost); later sections grow by `grow` (their lattices are
        // built at greater width while the segmentations of the section before are on the wire).
        // Measured (32 frames): K=10: first section 4 frames, doubling (4, 8, 16, 4); K=2: four equal sections.
        int sec0 = cn >= 16 ? (K >= 6 ? (cn + 7) / 8 : (cn + 3) / 4) : cn;
        if (tuning().host_section0 >= 1) sec0 = tuning().host_section0 < cn ? tuning().host_section0 : cn;
        const int grow = tuning().host_grow >= 1 ? tuning().host_grow : (K >= 6 ? 2 : 1);
        for (int f0 = 0, fn = 0, want = sec0; f0 < cn; f0 += fn) {
            fn = want < cn - f0 ? want : cn - f0;
            want = (long long)want * grow > cn ? cn : want * grow;
            cudaEvent_t ev_img;
            rc = host_event(g_host, ev_i++, &ev_img);
            if (rc) return rc;
            // only the planes the kernels read: the very last image may be shorter than the stride
            // (the reference reads `channels` planes at a stride of 3, colorbilateralfilter.cpp:50)
            size_t img_floats = (size_t)fn * img_frame;
            size_t img_skip = 0;   // floats at the head of the section that the section before has already brought
            if (c0 + f0 + fn == N || j.cfg.channels > j.cfg.image_stride_planes)
                img_floats = ((size_t)(fn - 1) * j.cfg.image_stride_planes + j.cfg.channels) * P;
            if (j.cfg.channels > j.cfg.image_stride_planes && c0 + f0 > 0)   // overlapping windows (see make_plan)
                img_skip = (size_t)(j.cfg.channels - j.cfg.image_stride_planes) * P;
            CUDA_TRY(cudaMemcpyAsync(j.d_img + (size_t)(c0 + f0) * img_frame + img_skip,
                                     j.images + (size_t)(c0 + f0) * img_frame + img_skip,
                                     (img_floats - img_skip) * sizeof(float), cudaMemcpyHostToDevice, s_in));
            CUDA_TRY(cudaEventRecord(ev_img, s_in));
            trace.mark("images in", c0 + f0, s_in);
            CUDA_TRY(cudaStreamWaitEvent(st, ev_img, 0));
            rc = run_lattice(dev, &j.cfg, pl, false, j.d_img + (size_t)c0 * img_frame, f0, fn, j.d_ws, false, st);
            if (rc) return rc;
            trace.mark("lattice", c0 + f0, st);
            host_groups(fn, group, sizes);
            if (f0 == 0 && fn < cn && fn <= group) sizes.assign(1, fn);   // a small first section stays whole
            int g0 = f0;
            for (size_t si = 0; si < sizes.size(); si++, gi++) {
                const int nc = sizes[si];
                const int n0 = c0 + g0;
                if (gi >= j.max_groups) return fail(TCAMCRF_ERR_INVALID, "internal: group count");
                cudaEvent_t ev_in, ev_done;
                rc = host_event(g_host, ev_i++, &ev_in);
                if (rc) return rc;
                rc = host_event(g_host, ev_i++, &ev_done);
                if (rc) return rc;
                CUDA_TRY(cudaMemcpyAsync(j.d_seg + n0 * seg_frame, j.segs + n0 * seg_frame,
                                         (size_t)nc * seg_frame * sizeof(float), cudaMemcpyHostToDevice, s_in));
                CUDA_TRY(cudaEventRecord(ev_in, s_in));
                trace.mark("segs in", gi, s_in);
                CUDA_TRY(cudaStreamWaitEvent(st, ev_in, 0));
                // every group reports its own share of the loss (already divided by the full batch size N)
                CUDA_TRY(cudaMemsetAsync(j.d_ws + pl.off_acc, 0, sizeof(double), st));
                rc = run_values(dev, pl, j.d_seg + n0 * seg_frame, j.d_as + n0 * seg_frame, g0, nc, j.d_ws, true,
                                j.want_loss, j.want_loss ? j.d_loss + gi : nullptr, (float)N, 0, st);
                if (rc) return rc;
                CUDA_TRY(cudaMemcpyAsync(j.d_status + gi, j.d_ws + pl.off_ctrl, sizeof(int), cudaMemcpyDeviceToDevice, st));
                if (j.grad_host) {
                    StageScope scope(kStBackward, 1, st);
                    const size_t count = (size_t)nc * seg_frame;
                    size_t blocks = (count / 4 + kThreads - 1) / kThreads;
                    if (blocks > (size_t)persistent_grid(dev)) blocks = (size_t)persistent_grid(dev);
                    if (blocks < 1) blocks = 1;
                    loss_backward_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(j.d_as + n0 * seg_frame, j.d_scal,
                                                                                j.d_grad + n0 * seg_frame, count, (float)N,
                                                                                1.0f);
                }
                CUDA_TRY(cudaGetLastError());
                CUDA_TRY(cudaEventRecord(ev_done, st));
                trace.mark("computed", gi, st);
                CUDA_TRY(cudaStreamWaitEvent(s_out, ev_done, 0));
                if (j.as_host)
                    CUDA_TRY(cudaMemcpyAsync(j.as_host + n0 * seg_frame, j.d_as + n0 * seg_frame,
                                             (size_t)nc * seg_frame * sizeof(float), cudaMemcpyDeviceToHost, s_out));
                if (j.grad_host)
                    CUDA_TRY(cudaMemcpyAsync(j.grad_host + n0 * seg_frame, j.d_grad + n0 * seg_frame,
                                             (size_t)nc * seg_frame * sizeof(float), cudaMemcpyDeviceToHost, s_out));
                trace.mark("results out", gi, s_out);
                g0 += nc;
            }
        }
    }
    // per-group losses and status words into pinned staging, then join the copy streams
    if (j.want_loss) CUDA_TRY(cudaMemcpyAsync(j.h_loss, j.d_loss, gi * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(j.h_status, j.d_status, gi * sizeof(int), cudaMemcpyDeviceToHost, st));
    cudaEvent_t ev_join_in, ev_join_out;
    rc = host_event(g_host, ev_i++, &ev_join_in);
    if (rc) return rc;
    rc = host_event(g_host, ev_i++, &ev_join_out);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(ev_join_in, s_in));
    CUDA_TRY(cudaEventRecord(ev_join_out, s_out));
    CUDA_TRY(cudaStreamWaitEvent(st, ev_join_in, 0));
    CUDA_TRY(cudaStreamWaitEvent(st, ev_join_out, 0));
    *groups_out = gi;
    return TCAMCRF_OK;
}

static bool host_pinned(const void *p)
{
    if (!p) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

static int host_run(const tcamcrf_config *cfg_in, const float *images, const float *segs, float *as_host,
                    float *loss_host, float *grad_host, int N, int K, int H, int W, float grad_out)
{
    int rc = check_device();
    if (rc) return rc;
    if (!cfg_in || !images || !segs) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    HostJob j;
    j.cfg = *cfg_in;
    if (j.cfg.chunk_frames <= 0 || j.cfg.chunk_frames > 64) j.cfg.chunk_frames = 64;
    rc = make_plan(&j.cfg, N, K, H, W, j.pl);
    if (rc) return rc;
    const Plan &pl = j.pl;
    Device *dev = nullptr;
    rc = this_device(&dev);
    if (rc) return rc;
    HostCtx &g_host = dev->host;
    HostGraphs &graphs = dev->graphs;
    std::lock_guard<std::mutex> lock(g_host.mu);
    const int ngroups = N + 8;   // upper bound: a group holds at least one frame
    const size_t P = (size_t)H * W;
    const size_t img_frame = (size_t)j.cfg.image_stride_planes * P;
    const size_t seg_frame = (size_t)K * P;
    const size_t img_over = j.cfg.channels > j.cfg.image_stride_planes
                                ? (size_t)(j.cfg.channels - j.cfg.image_stride_planes) * P : 0;   // overlapping windows
    const size_t img_bytes = align_up(((size_t)N * img_frame + img_over) * sizeof(float), 256);
    const size_t seg_bytes = align_up((size_t)N * seg_frame * sizeof(float), 256);
    const size_t scal_bytes = align_up((size_t)(2 * ngroups + 2) * sizeof(float), 256);
    char *base = nullptr;
    const void *old_buf = g_host.buf;
    rc = host_reserve(g_host, img_bytes + 3 * seg_bytes + scal_bytes + pl.total, &base);
    if (rc) return rc;
    if (old_buf != g_host.buf) graphs.clear();   // the captured schedules point into the old buffer
    rc = host_pin_reserve(g_host, (size_t)(2 * ngroups + 2) * sizeof(float));
    if (rc) return rc;   // (a new staging block changes the graph key: stale schedules age out of the cache)
    j.images = images;
    j.segs = segs;
    j.as_host = as_host;
    j.grad_host = grad_host;
    j.want_loss = loss_host != nullptr;
    j.N = N;
    j.K = K;
    j.H = H;
    j.W = W;
    j.d_img = (float *)base;
    j.d_seg = (float *)(base + img_bytes);
    j.d_as = (float *)(base + img_bytes + seg_bytes);
    j.d_grad = (float *)(base + img_bytes + 2 * seg_bytes);
    j.d_scal = (float *)(base + img_bytes + 3 * seg_bytes);  // [0]=grad_out, [1..]=loss per group, then status
    j.d_loss = j.d_scal + 1;
    j.d_status = (int *)(j.d_scal + 1 + ngroups);
    j.d_ws = base + img_bytes + 3 * seg_bytes + scal_bytes;
    j.h_gout = (float *)g_host.pin;
    j.h_loss = j.h_gout + 1;
    j.h_status = (int *)(j.h_loss + ngroups);
    j.max_groups = ngroups;
    const int hint = density_hint(*dev, j.d_ws);
    j.dedup_hint = !lattice_is_dense(hint, pl.P);
    j.dense_hint = lattice_is_dense(hint, pl.P);
    *j.h_gout = grad_out;
    cudaStream_t st = g_host.stream;

    HostTrace trace;
    int gi = 0;
    // the captured schedule needs pinned buffers (a copy from pageable memory cannot be captured), and neither the
    // per-stage profiler nor the trace (both record timing events between the kernels)
    const bool graph_ok = !g_prof.enabled && tuning().host_trace == 0 &&
                          host_pinned(images) && host_pinned(segs) && host_pinned(as_host) && host_pinned(grad_host);
    HostGraphs::Key key;
    memset(&key, 0, sizeof(key));
    HostGraphs::Item *hit = nullptr;
    if (graph_ok) {
        key.cfg = j.cfg;
        key.N = N; key.K = K; key.H = H; key.W = W;
        key.images = images; key.segs = segs; key.as_host = as_host; key.grad_host = grad_host;
        key.buf = g_host.buf; key.pin = g_host.pin;
        key.want_loss = j.want_loss; key.dedup = j.dedup_hint; key.dense = j.dense_hint;
        key.groups_knob = tuning().host_groups; key.sec0_knob = tuning().host_section0; key.grow_knob = tuning().host_grow;
        for (auto &it : graphs.items)
            if (it.key == key) hit = &it;
    }
    if (hit) {
        hit->used = ++graphs.tick;
        gi = hit->groups;
        CUDA_TRY(cudaGraphLaunch(hit->exec, st));
        std::lock_guard<std::mutex> plock(g_prof.mu);
        g_prof.total_launches += hit->launches;
    } else {
        trace.begin(g_host.s_in);
        rc = host_enqueue(*dev, j, trace, &gi);
        if (rc) return rc;
        trace.host_mark("enqueued");
    }
    density_hint_refresh(*dev, pl, j.d_ws, st);
    CUDA_TRY(cudaStreamSynchronize(st));
    trace.host_mark("synced");
    trace.end();
    int st_bits = 0;
    double total = 0.0;
    for (int g = 0; g < gi; g++) {
        st_bits |= j.h_status[g];
        total += (double)j.h_loss[g];
    }
    if (loss_host) *loss_host = (float)total;
    if (graph_ok && !hit && !st_bits) {
        // First call with these buffers: it ran eagerly (every helper object now exists and the streams are idle);
        // capture the same schedule for the calls to come.  A failure here only means the next call is eager again.
        if (graphs.items.size() >= 8) {   // drop the least recently used schedule
            size_t lru = 0;
            for (size_t i = 1; i < graphs.items.size(); i++)
                if (graphs.items[i].used < graphs.items[lru].used) lru = i;
            cudaGraphExecDestroy(graphs.items[lru].exec);
            graphs.items.erase(graphs.items.begin() + lru);
        }
        long long launches0;
        {
            std::lock_guard<std::mutex> plock(g_prof.mu);
            launches0 = g_prof.total_launches;
        }
        cudaGraph_t graph = nullptr;
        int groups = 0;
        if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            HostTrace off;
            const int crc = host_enqueue(*dev, j, off, &groups);
            const cudaError_t ce = cudaStreamEndCapture(st, &graph);
            cudaGraphExec_t exec = nullptr;
            if (!crc && ce == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
                std::lock_guard<std::mutex> plock(g_prof.mu);
                graphs.items.push_back({key, exec, groups, g_prof.total_launches - launches0, ++graphs.tick});
                g_prof.total_launches = launches0;   // capturing launched nothing
            }
            if (graph) cudaGraphDestroy(graph);
        }
        cudaGetLastError();
    }
    if (st_bits)
        return fail(TCAMCRF_ERR_DEVICE_STATUS, "device status 0x%x (%s%s%s)", st_bits,
                    (st_bits & TCAMCRF_DEV_TABLE_FULL) ? "hash table full " : "",
                    (st_bits & TCAMCRF_DEV_POOL_FULL) ? "vertex pool full " : "",
                    (st_bits & TCAMCRF_DEV_KEY_RANGE) ? "lattice coordinate out of key range" : "");
    return TCAMCRF_OK;
}

static tcamcrf_config ref_config(int feat, int channels, int stride, float srgb, float sxy)
{
    tcamcrf_config c;
    memset(&c, 0, sizeof(c));
    c.feat = feat;
    c.channels = channels;
    c.image_stride_planes = stride;
    c.sigma_rgb = srgb;
    c.sigma_xy = sxy;
    c.loss_weight = 0.f;
    return c;
}

// |lattice coordinate quotient| a frame can reach when every image plane lies in [0, max_value] (features are
// non-negative): el[0] = sum_i cf_i and el[j] = sum_{i >= j} cf_i - j * cf_{j-1} with cf_i = f_i * scale_i
// (embed_point), so |el| <= max(sum_i cf_i, max_j j * cf_{j-1}); the quotient is el / (d+1) rounded, moved by at
// most one by the rank fix-up, and needs room for one neighbour step on either side.
template <int D>
static bool key_range_ok(const float (&fmax)[kMaxD])
{
    EmbedConsts ec;
    scale_factors(D, ec);
    double sum = 0.0, worst = 0.0;
    for (int i = 0; i < D; i++) {
        const double cf = (double)fmax[i] * (double)ec.scale[i];
        sum += cf;
        if ((i + 1) * cf > worst) worst = (i + 1) * cf;
    }
    if (sum > worst) worst = sum;
    return worst / (D + 1) + 3.0 <= (double)KeyCodec<D>::kQMax;
}

}  // namespace tcamcrf

// ===========================================================================
// C ABI
// ===========================================================================
using namespace tcamcrf;

extern "C" {

int tcamcrf_version(void) { return TCAMCRF_VERSION; }

const char *tcamcrf_last_error(void) { return g_err; }

int tcamcrf_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int i = 0; i < n; i++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

size_t tcamcrf_workspace_bytes(const tcamcrf_config *cfg, int N, int K, int H, int W)
{
    Plan pl;
    if (make_plan(cfg, N, K, H, W, pl)) return 0;
    return pl.total;
}

int tcamcrf_filter(const tcamcrf_config *cfg, const float *images_dev, const float *segs_dev, float *as_dev, int N,
                   int K, int H, int W, void *workspace, size_t workspace_bytes, void *cuda_stream)
{
    return run_filter(cfg, false, images_dev, segs_dev, as_dev, nullptr, N, K, H, W, 1.f, workspace,
                      workspace_bytes, (cudaStream_t)cuda_stream);
}

int tcamcrf_filter_transposed(const tcamcrf_config *cfg, const void *images_dev, int images_u8, const float *segs_dev,
                               float *ats_dev, int N, int K, int H, int W, void *workspace, size_t workspace_bytes,
                               void *cuda_stream)
{
    return run_filter(cfg, images_u8 != 0, images_dev, segs_dev, ats_dev, nullptr, N, K, H, W, 1.f, workspace,
                      workspace_bytes, (cudaStream_t)cuda_stream, kFlagReverseBlur);
}

// Checks shared by the two lattice entry points (the plan must describe ONE chunk holding all N frames), and the
// current device's context.
static int lattice_plan(const tcamcrf_config *cfg, int N, int K, int H, int W, void *workspace, size_t ws_bytes,
                        Plan &pl, Device **dev)
{
    if (!cfg || !workspace) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    int rc = make_plan(cfg, N, K, H, W, pl);
    if (rc) return rc;
    if (N > pl.chunk)
        return fail(TCAMCRF_ERR_INVALID, "a lattice holds at most chunk_frames (%d) frames, got %d", pl.chunk, N);
    if (ws_bytes < pl.total)
        return fail(TCAMCRF_ERR_WORKSPACE, "workspace too small: %zu < %zu bytes", ws_bytes, pl.total);
    if (((uintptr_t)workspace & 255) != 0) return fail(TCAMCRF_ERR_WORKSPACE, "workspace must be 256-byte aligned");
    return this_device(dev);
}

int tcamcrf_key_range_ok(const tcamcrf_config *cfg, int H, int W, float max_value)
{
    const int D = feature_dim(cfg);
    if (D < 1 || D > kMaxD || H < 1 || W < 1 || !(cfg->sigma_rgb > 0.f)) return 0;
    float fmax[kMaxD] = {0};
    int c0 = 0;
    if (cfg->feat == TCAMCRF_FEAT_XY_RGB) {
        if (!(cfg->sigma_xy > 0.f)) return 0;
        fmax[0] = (float)(W - 1) / cfg->sigma_xy;
        if (D > 1) fmax[1] = (float)(H - 1) / cfg->sigma_xy;
        c0 = 2;
    }
    for (int c = c0; c < D; c++) fmax[c] = max_value / cfg->sigma_rgb;
    switch (D) {
    case 1: return key_range_ok<1>(fmax);
    case 2: return key_range_ok<2>(fmax);
    case 3: return key_range_ok<3>(fmax);
    case 4: return key_range_ok<4>(fmax);
    case 5: return key_range_ok<5>(fmax);
    case 6: return key_range_ok<6>(fmax);
    }
    return 0;
}

int tcamcrf_chunk_frames(const tcamcrf_config *cfg, int N, int K, int H, int W)
{
    if (!cfg) return 0;
    Plan pl;
    if (make_plan(cfg, N, K, H, W, pl)) return 0;
    return pl.chunk;
}

int tcamcrf_lattice_build(const tcamcrf_config *cfg, const void *images_dev, int images_u8, int N, int K, int H,
                          int W, void *workspace, size_t workspace_bytes, void *cuda_stream)
{
    if (!images_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    Plan pl;
    Device *dev = nullptr;
    int rc = lattice_plan(cfg, N, K, H, W, workspace, workspace_bytes, pl, &dev);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    CUDA_TRY(cudaMemsetAsync((char *)workspace + pl.off_ctrl, 0, kCtrlResetInts * sizeof(int), st));
    return run_lattice(*dev, cfg, pl, images_u8 != 0, images_dev, 0, N, (char *)workspace, false, st);
}

int tcamcrf_lattice_apply(const tcamcrf_config *cfg, const float *segs_dev, float *out_dev, float *loss_dev, int N,
                          int K, int H, int W, float n_norm, int transposed, void *workspace, size_t workspace_bytes,
                          void *cuda_stream)
{
    if (!segs_dev || !out_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    Plan pl;
    Device *dev = nullptr;
    int rc = lattice_plan(cfg, N, K, H, W, workspace, workspace_bytes, pl, &dev);
    if (rc) return rc;
    if (((uintptr_t)segs_dev & 3) || ((uintptr_t)out_dev & 3))
        return fail(TCAMCRF_ERR_INVALID, "float buffers must be 4-byte aligned");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    // the loss accumulator starts at zero; the status word of the build is kept (a poisoned lattice stays poisoned)
    if (loss_dev) CUDA_TRY(cudaMemsetAsync((char *)workspace + pl.off_acc, 0, sizeof(double), st));
    return run_values(*dev, pl, segs_dev, out_dev, 0, N, (char *)workspace, true, loss_dev != nullptr, loss_dev, n_norm,
                      transposed ? kFlagReverseBlur : 0, st);
}

int tcamcrf_filter_u8(const tcamcrf_config *cfg, const uint8_t *images_dev, const float *segs_dev, float *as_dev,
                      int N, int K, int H, int W, void *workspace, size_t workspace_bytes, void *cuda_stream)
{
    return run_filter(cfg, true, images_dev, segs_dev, as_dev, nullptr, N, K, H, W, 1.f, workspace, workspace_bytes,
                      (cudaStream_t)cuda_stream);
}

int tcamcrf_loss_forward(const tcamcrf_config *cfg, const float *images_dev, const float *segs_dev, float *as_dev,
                         float *loss_dev, int N, int K, int H, int W, float n_norm, void *workspace,
                         size_t workspace_bytes, void *cuda_stream)
{
    if (!loss_dev) return fail(TCAMCRF_ERR_INVALID, "null loss pointer");
    return run_filter(cfg, false, images_dev, segs_dev, as_dev, loss_dev, N, K, H, W, n_norm, workspace,
                      workspace_bytes, (cudaStream_t)cuda_stream);
}

// run_filter flags for logits of TCAMCRF_DTYPE_* `dtype`, or -1 (with an error set) for an unknown code
static int logits_flags(int dtype)
{
    switch (dtype) {
    case TCAMCRF_DTYPE_F32: return kFlagLogits;
    case TCAMCRF_DTYPE_F16: return kFlagLogits | kFlagLowp;
    case TCAMCRF_DTYPE_BF16: return kFlagLogits | kFlagLowp | kFlagBF16;
    }
    fail(TCAMCRF_ERR_INVALID, "unknown logits dtype code %d", dtype);
    return -1;
}

static int host_frames_forward(const tcamcrf_config *cfg, const void *images_host, void *images_stage_dev,
                               int images_u8, const void *segs_dev, float *as_dev, float *loss_dev, int flags, int N,
                               int K, int H, int W, float n_norm, void *workspace, size_t workspace_bytes,
                               void *cuda_stream)
{
    if (!images_host || !images_stage_dev) return fail(TCAMCRF_ERR_INVALID, "null image pointer");
    if (cfg && cfg->channels > cfg->image_stride_planes)
        return fail(TCAMCRF_ERR_INVALID, "overlapping image windows (stride < channels) need device frames or the "
                    "host-pointer API");
    const bool logits = (flags & kFlagLogits) != 0;
    if (logits && K < 2) return fail(TCAMCRF_ERR_INVALID, "softmax needs at least two classes");
    if (logits && !loss_dev) return fail(TCAMCRF_ERR_INVALID, "null loss pointer");
    return run_filter(cfg, images_u8 != 0, images_stage_dev, segs_dev, as_dev, loss_dev, N, K, H, W, n_norm, workspace,
                      workspace_bytes, (cudaStream_t)cuda_stream, flags, images_host);
}

int tcamcrf_loss_forward_host_frames(const tcamcrf_config *cfg, const void *images_host, void *images_stage_dev,
                                     int images_u8, const float *segs_dev, float *as_dev, float *loss_dev, int logits,
                                     int N, int K, int H, int W, float n_norm, void *workspace,
                                     size_t workspace_bytes, void *cuda_stream)
{
    return host_frames_forward(cfg, images_host, images_stage_dev, images_u8, segs_dev, as_dev, loss_dev,
                               logits ? kFlagLogits : 0, N, K, H, W, n_norm, workspace, workspace_bytes, cuda_stream);
}

int tcamcrf_loss_forward_host_frames_typed(const tcamcrf_config *cfg, const void *images_host, void *images_stage_dev,
                                           int images_u8, const void *logits_dev, int logits_dtype, float *as_dev,
                                           float *loss_dev, int N, int K, int H, int W, float n_norm, void *workspace,
                                           size_t workspace_bytes, void *cuda_stream)
{
    const int flags = logits_flags(logits_dtype);
    if (flags < 0) return TCAMCRF_ERR_INVALID;
    return host_frames_forward(cfg, images_host, images_stage_dev, images_u8, logits_dev, as_dev, loss_dev, flags, N,
                               K, H, W, n_norm, workspace, workspace_bytes, cuda_stream);
}

int tcamcrf_loss_forward_u8(const tcamcrf_config *cfg, const uint8_t *images_dev, const float *segs_dev,
                            float *as_dev, float *loss_dev, int N, int K, int H, int W, float n_norm,
                            void *workspace, size_t workspace_bytes, void *cuda_stream)
{
    if (!loss_dev) return fail(TCAMCRF_ERR_INVALID, "null loss pointer");
    return run_filter(cfg, true, images_dev, segs_dev, as_dev, loss_dev, N, K, H, W, n_norm, workspace,
                      workspace_bytes, (cudaStream_t)cuda_stream);
}

int tcamcrf_loss_forward_logits(const tcamcrf_config *cfg, const void *images_dev, int images_u8,
                                const float *logits_dev, float *as_dev, float *loss_dev, int N, int K, int H, int W,
                                float n_norm, void *workspace, size_t workspace_bytes, void *cuda_stream)
{
    return tcamcrf_loss_forward_logits_typed(cfg, images_dev, images_u8, logits_dev, TCAMCRF_DTYPE_F32, as_dev,
                                             loss_dev, N, K, H, W, n_norm, workspace, workspace_bytes, cuda_stream);
}

int tcamcrf_loss_forward_logits_typed(const tcamcrf_config *cfg, const void *images_dev, int images_u8,
                                      const void *logits_dev, int logits_dtype, float *as_dev, float *loss_dev, int N,
                                      int K, int H, int W, float n_norm, void *workspace, size_t workspace_bytes,
                                      void *cuda_stream)
{
    const int flags = logits_flags(logits_dtype);
    if (flags < 0) return TCAMCRF_ERR_INVALID;
    if (!loss_dev) return fail(TCAMCRF_ERR_INVALID, "null loss pointer");
    if (K < 2) return fail(TCAMCRF_ERR_INVALID, "softmax needs at least two classes");
    return run_filter(cfg, images_u8 != 0, images_dev, logits_dev, as_dev, loss_dev, N, K, H, W, n_norm, workspace,
                      workspace_bytes, (cudaStream_t)cuda_stream, flags);
}

int tcamcrf_loss_backward_logits(const float *as_dev, const float *logits_dev, const float *grad_out_dev,
                                 float *grad_logits_dev, int N, int K, int H, int W, float n_norm, void *cuda_stream)
{
    return tcamcrf_loss_backward_logits_weighted(as_dev, logits_dev, grad_out_dev, grad_logits_dev, N, K, H, W, n_norm,
                                                 1.0f, cuda_stream);
}

int tcamcrf_loss_backward_logits_weighted(const float *as_dev, const float *logits_dev, const float *grad_out_dev,
                                          float *grad_logits_dev, int N, int K, int H, int W, float n_norm,
                                          float weight, void *cuda_stream)
{
    return tcamcrf_loss_backward_logits_typed(as_dev, logits_dev, TCAMCRF_DTYPE_F32, grad_out_dev, grad_logits_dev, N,
                                              K, H, W, n_norm, weight, cuda_stream);
}

int tcamcrf_loss_backward_logits_typed(const float *as_dev, const void *logits_dev, int logits_dtype,
                                       const float *grad_out_dev, void *grad_logits_dev, int N, int K, int H, int W,
                                       float n_norm, float weight, void *cuda_stream)
{
    if (logits_flags(logits_dtype) < 0) return TCAMCRF_ERR_INVALID;
    if (!as_dev || !logits_dev || !grad_out_dev || !grad_logits_dev)
        return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (N < 1 || K < 2 || H < 1 || W < 1) return fail(TCAMCRF_ERR_INVALID, "N,H,W must be positive and K >= 2");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    const long long pixels = (long long)N * H * W;
    long long blocks = (pixels + kThreads - 1) / kThreads;
    if (blocks > persistent_grid(*dev)) blocks = persistent_grid(*dev);
    StageScope scope(kStBackward, 1, (cudaStream_t)cuda_stream);
    if (logits_dtype == TCAMCRF_DTYPE_F32) {
        loss_backward_logits_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)cuda_stream>>>(
            as_dev, (const float *)logits_dev, grad_out_dev, (float *)grad_logits_dev, K, H * W, pixels, n_norm, weight);
    } else {
        const int bf16 = logits_dtype == TCAMCRF_DTYPE_BF16;
        loss_backward_logits_lowp_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)cuda_stream>>>(
            as_dev, Logits16{(const unsigned short *)logits_dev, bf16}, grad_out_dev,
            Grad16{(unsigned short *)grad_logits_dev, bf16}, K, H * W, pixels, n_norm, weight);
    }
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcamcrf_loss_backward(const float *as_dev, const float *grad_out_dev, float *grad_seg_dev, size_t count,
                          float n_norm, void *cuda_stream)
{
    return tcamcrf_loss_backward_weighted(as_dev, grad_out_dev, grad_seg_dev, count, n_norm, 1.0f, cuda_stream);
}

int tcamcrf_loss_backward_weighted(const float *as_dev, const float *grad_out_dev, float *grad_seg_dev, size_t count,
                                   float n_norm, float weight, void *cuda_stream)
{
    if (!as_dev || !grad_out_dev || !grad_seg_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (count == 0) return TCAMCRF_OK;
    if (((uintptr_t)as_dev & 3) || ((uintptr_t)grad_seg_dev & 3))
        return fail(TCAMCRF_ERR_INVALID, "buffers must be 4-byte aligned");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    size_t blocks = (count / 4 + kThreads - 1) / kThreads;
    if (blocks > (size_t)persistent_grid(*dev)) blocks = persistent_grid(*dev);
    if (blocks < 1) blocks = 1;
    StageScope scope(kStBackward, 1, (cudaStream_t)cuda_stream);
    loss_backward_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)cuda_stream>>>(as_dev, grad_out_dev,
                                                                                       grad_seg_dev, count, n_norm,
                                                                                       weight);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcamcrf_workspace_status(void *workspace, void *cuda_stream, int *dev_status, int *vertices)
{
    if (!workspace || !dev_status) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    int host[kCtrlResetInts];
    CUDA_TRY(cudaMemcpyAsync(host, workspace, sizeof(host), cudaMemcpyDeviceToHost, (cudaStream_t)cuda_stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)cuda_stream));
    *dev_status = host[kCtrlStatus];
    if (vertices) *vertices = host[kCtrlLastCount];
    return TCAMCRF_OK;
}

int tcamcrf_debug_lattice(const tcamcrf_config *cfg, const float *image_host, int H, int W, int32_t *offset_host,
                          float *bary_host, int *vertices, int32_t *nbr_host, size_t nbr_cap)
{
    int rc = check_device();
    if (rc) return rc;
    if (!cfg || !image_host || !offset_host || !bary_host || !vertices)
        return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    tcamcrf_config c = *cfg;
    c.image_stride_planes = c.channels;
    Plan pl;
    rc = make_plan(&c, 1, 1, H, W, pl);
    if (rc) return rc;
    const size_t P = (size_t)H * W;
    const int dp1 = pl.D + 1;
    Device *dev = nullptr;
    rc = this_device(&dev);
    if (rc) return rc;
    HostCtx &g_host = dev->host;
    std::lock_guard<std::mutex> lock(g_host.mu);
    const size_t img_bytes = align_up((size_t)c.channels * P * sizeof(float), 256);
    const size_t seg_bytes = align_up(P * sizeof(float), 256);
    char *base = nullptr;
    rc = host_reserve(g_host, img_bytes + 2 * seg_bytes + pl.total, &base);
    if (rc) return rc;
    float *d_img = (float *)base, *d_seg = (float *)(base + img_bytes), *d_as = (float *)(base + img_bytes + seg_bytes);
    char *d_ws = base + img_bytes + 2 * seg_bytes;
    cudaStream_t st = g_host.stream;
    CUDA_TRY(cudaMemcpyAsync(d_img, image_host, (size_t)c.channels * P * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(d_seg, 0, P * sizeof(float), st));
    rc = run_filter(&c, false, d_img, d_seg, d_as, nullptr, 1, 1, H, W, 1.f, d_ws, pl.total, st);
    if (rc) return rc;
    std::vector<int> off((size_t)dp1 * P);
    std::vector<float> bar((size_t)dp1 * P);
    int ctrl[kCtrlResetInts];
    CUDA_TRY(cudaMemcpyAsync(off.data(), d_ws + pl.off_offset, off.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(bar.data(), d_ws + pl.off_bary, bar.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(ctrl, d_ws + pl.off_ctrl, sizeof(ctrl), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (ctrl[kCtrlStatus]) return fail(TCAMCRF_ERR_DEVICE_STATUS, "device status 0x%x", ctrl[kCtrlStatus]);
    const int M = ctrl[kCtrlLastCount];
    *vertices = M;
    // device layout is [r][p]; the reference's offset_/barycentric_ are [p][r]
    for (size_t px = 0; px < P; px++)
        for (int r = 0; r < dp1; r++) {
            const int sv = off[(size_t)r * P + px];
            offset_host[px * dp1 + r] = sv <= -2 ? -2 - sv : -1;   // stored as -2 - id after the splat
            bary_host[px * dp1 + r] = bar[(size_t)r * P + px];
        }
    if (nbr_host && nbr_cap >= (size_t)dp1 * M * 2) {
        std::vector<int2> nb((size_t)M);
        for (int j = 0; j < dp1; j++) {
            CUDA_TRY(cudaMemcpy(nb.data(), d_ws + pl.off_nbr + (size_t)j * pl.pool * sizeof(int2), (size_t)M * sizeof(int2),
                                cudaMemcpyDeviceToHost));
            for (int v = 0; v < M; v++) {
                nbr_host[((size_t)j * M + v) * 2 + 0] = nb[v].x;
                nbr_host[((size_t)j * M + v) * 2 + 1] = nb[v].y;
            }
        }
    }
    return TCAMCRF_OK;
}

int tcam_debug_seed_draws(const unsigned int *rng_dev, int B, int HW, unsigned int *words_dev, float *draws_dev,
                          void *cuda_stream)
{
    if (!rng_dev || !words_dev || !draws_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || HW < 1) return fail(TCAMCRF_ERR_INVALID, "B,HW must be positive");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    long long blocks = ((long long)B * 2 * HW + 255) / 256;
    if (blocks > persistent_grid(*dev)) blocks = persistent_grid(*dev);
    seed_debug_draws_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(rng_dev, B, HW, words_dev, draws_dev);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcam_debug_exp_draws(const unsigned int *words_dev, int n, float *draws_dev, void *cuda_stream)
{
    if (!words_dev || !draws_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (n < 1) return fail(TCAMCRF_ERR_INVALID, "n must be positive");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    long long blocks = ((long long)n + 255) / 256;
    if (blocks > persistent_grid(*dev)) blocks = persistent_grid(*dev);
    seed_debug_exp_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(words_dev, n, draws_dev);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

// ---- drop-in host API ------------------------------------------------------

int bilateralfilter(float *image, int len_image, float *in, int len_in, float *out, int len_out, int H, int W,
                    float sigmargb, float sigmaxy)
{
    (void)len_image;
    (void)len_out;
    if (H < 1 || W < 1) return fail(TCAMCRF_ERR_INVALID, "H,W must be positive");
    const int K = len_in / W / H;  // class count is inferred (bilateralfilter.cpp:27)
    if (K < 1) return TCAMCRF_OK;  // the reference's loop runs zero times
    tcamcrf_config c = ref_config(TCAMCRF_FEAT_XY_RGB, 3, 3, sigmargb, sigmaxy);
    return host_run(&c, image, in, out, nullptr, nullptr, 1, K, H, W, 0.f);
}

int bilateralfilter_batch(float *images, int len_images, float *ins, int len_ins, float *outs, int len_outs, int N,
                          int K, int H, int W, float sigmargb, float sigmaxy)
{
    (void)len_images;
    (void)len_ins;
    (void)len_outs;
    if (N < 1 || K < 1) return TCAMCRF_OK;  // empty batch: nothing to do, like the reference's loop
    tcamcrf_config c = ref_config(TCAMCRF_FEAT_XY_RGB, 3, 3, sigmargb, sigmaxy);
    return host_run(&c, images, ins, outs, nullptr, nullptr, N, K, H, W, 0.f);
}

int colorbilateralfilter(float *image, int len_image, float *in, int len_in, float *out, int len_out, int H, int W,
                         float sigmargb, int DIM)
{
    (void)len_image;
    (void)len_out;
    if (H < 1 || W < 1) return fail(TCAMCRF_ERR_INVALID, "H,W must be positive");
    const int K = len_in / W / H;
    if (K < 1) return TCAMCRF_OK;
    tcamcrf_config c = ref_config(TCAMCRF_FEAT_COLOR, DIM, DIM, sigmargb, 1.f);
    return host_run(&c, image, in, out, nullptr, nullptr, 1, K, H, W, 0.f);
}

int colorbilateralfilter_batch(float *images, int len_images, float *ins, int len_ins, float *outs, int len_outs,
                               int N, int K, int H, int W, float sigmargb, int DIM)
{
    (void)len_ins;
    (void)len_outs;
    if (N < 1 || K < 1) return TCAMCRF_OK;
    // the reference strides images by 3 planes whatever DIM is (colorbilateralfilter.cpp:50); with DIM > 3 that
    // reads overlapping windows of `images`, which needs len_images >= ((N-1)*3 + DIM)*H*W.
    if (DIM > 3 && (long long)len_images < ((long long)(N - 1) * 3 + DIM) * H * W)
        return fail(TCAMCRF_ERR_INVALID, "images too short for DIM=%d with the reference's 3-plane stride", DIM);
    // stride 3 whatever DIM is: for DIM > 3 frame n reads planes [3n, 3n + DIM), like the reference
    tcamcrf_config c = ref_config(TCAMCRF_FEAT_COLOR, DIM, 3, sigmargb, 1.f);
    return host_run(&c, images, ins, outs, nullptr, nullptr, N, K, H, W, 0.f);
}

int tcamcrf_loss_fwd_bwd_host(const tcamcrf_config *cfg, const float *images_host, const float *segs_host,
                              float *loss_host, float *grad_host, int N, int K, int H, int W, float grad_out)
{
    if (!loss_host || !grad_host) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    return host_run(cfg, images_host, segs_host, nullptr, loss_host, grad_host, N, K, H, W, grad_out);
}

int tcamcrf_set_tuning(const char *name, int value)
{
    if (!name) return fail(TCAMCRF_ERR_INVALID, "null knob name");
    if (strncmp(name, "TCAMCRF_", 8) == 0) name += 8;
    Tuning &t = tuning();
    if (!strcmp(name, "DENSE")) t.dense = value < 0 ? -1 : (value != 0);
    else if (!strcmp(name, "BUILD_DEDUP")) t.build_dedup = value < 0 ? -1 : (value != 0);
    else if (!strcmp(name, "HIMG_SECTIONS")) t.himg_sections = value > 0 ? value : 0;
    else if (!strcmp(name, "HOST_GROUPS")) t.host_groups = value > 0 ? value : 0;
    else if (!strcmp(name, "HOST_SECTION0")) t.host_section0 = value > 0 ? value : 0;
    else if (!strcmp(name, "HOST_TRACE")) t.host_trace = value > 0;
    else if (!strcmp(name, "HOST_GROW")) t.host_grow = value > 0 ? value : 0;
    else return fail(TCAMCRF_ERR_INVALID, "unknown tuning knob '%s'", name);
    return TCAMCRF_OK;
}

void tcamcrf_profile_enable(int on)
{
    std::lock_guard<std::mutex> lock(g_prof.mu);
    g_prof.enabled = on != 0;
}

int tcamcrf_profile_read(double *ms, long long *launches, int reset)
{
    std::lock_guard<std::mutex> lock(g_prof.mu);
    for (auto &sp : g_prof.spans) {
        float t = 0.f;
        if (cudaEventSynchronize(sp.b) == cudaSuccess && cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess) {
            g_prof.ms[sp.stage] += t;
            g_prof.launches[sp.stage] += sp.launches;
        }
        sp.dev->timing_events.push_back(sp.a);
        sp.dev->timing_events.push_back(sp.b);
    }
    g_prof.spans.clear();
    for (int i = 0; i < kStCount; i++) {
        if (ms) ms[i] = g_prof.ms[i];
        if (launches) launches[i] = g_prof.launches[i];
        if (reset) {
            g_prof.ms[i] = 0;
            g_prof.launches[i] = 0;
        }
    }
    return TCAMCRF_OK;
}

long long tcamcrf_launch_count(void)
{
    std::lock_guard<std::mutex> lock(g_prof.mu);
    return g_prof.total_launches;
}

int tcam_seed_select(const float *cams_dev, int T, const int64_t *roi_dev, const float *q_dev,
                     const int *q_offset_dev, const int *n_cand_dev, int k_fg, int k_bg, int weighted_fg, int B, int HW,
                     float *cam_max_dev, float *scratch_dev, int *sel_dev, int kmax, void *cuda_stream)
{
    if (!cams_dev || !q_dev || !q_offset_dev || !n_cand_dev || !cam_max_dev || !scratch_dev || !sel_dev)
        return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || T < 1 || HW < 1 || kmax < 1 || k_fg < 0 || k_bg < 0)
        return fail(TCAMCRF_ERR_INVALID, "B,T,HW,kmax must be positive and k_fg,k_bg non-negative");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    SeedParams sp;
    sp.cams = cams_dev;
    sp.roi = reinterpret_cast<const long long *>(roi_dev);
    sp.q = q_dev;
    sp.q_offset = q_offset_dev;
    sp.n_cand = n_cand_dev;
    sp.cam_max = cam_max_dev;
    sp.scratch = scratch_dev;
    sp.sel = sel_dev;
    sp.T = T;
    sp.HW = HW;
    sp.kmax = kmax;
    sp.k_fg = k_fg;
    sp.k_bg = k_bg;
    sp.weighted_fg = weighted_fg;
    {
        StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
        // keys of a sample in shared memory when the frame fits (4 bytes per pixel of the 227 KB an SM has)
        const size_t smem = (size_t)HW * sizeof(unsigned int);
        if (smem <= (size_t)dev->select_smem)
            seed_select_smem_kernel<<<dim3(2, B), kSeedThreads, smem, (cudaStream_t)cuda_stream>>>(sp);
        else
            seed_select_kernel<<<dim3(2, B), kSeedThreads, 0, (cudaStream_t)cuda_stream>>>(sp);
    }
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

static int seed_fused_slice(int HW) { return ((HW + kSeedCluster - 1) / kSeedCluster + 3) / 4 * 4; }

int tcam_seed_fused_supported(int HW, int kmax)
{
    if (HW < 1 || kmax < 1 || kmax > kSeedFusedMaxK) return 0;
    Device *dev = nullptr;
    if (this_device(&dev)) return 0;
    return (size_t)seed_fused_slice(HW) * 2 * sizeof(unsigned int) <= (size_t)dev->fused_smem ? 1 : 0;
}

int tcam_seed_fused(const float *cams_dev, int T, const int64_t *roi_dev, const float *q_dev, const int *q_offset_dev,
                    const int *n_cand_dev, const unsigned int *rng_dev, float max_p, int n_fg_fixed, int n_bg, int k_fg,
                    int k_bg, int weighted_fg, int B, int H, int W, int ksz, long long ignore_idx, float *cam_max_dev,
                    int *sel_dev, int kmax, int64_t *labels_dev, void *cuda_stream)
{
    if (!cams_dev || !cam_max_dev || !sel_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || T < 1 || H < 1 || W < 1 || kmax < 1 || k_fg < 0 || k_bg < 0 || ksz < 1)
        return fail(TCAMCRF_ERR_INVALID, "B,T,H,W,kmax,ksz must be positive and k_fg,k_bg non-negative");
    if ((long long)H * W > (1ll << 26)) return fail(TCAMCRF_ERR_INVALID, "image too large");
    if (q_dev ? (!q_offset_dev || !n_cand_dev) : !rng_dev)
        return fail(TCAMCRF_ERR_INVALID, "draws need q_offset and n_cand; without draws the Philox key words are needed");
    const int HW = H * W;
    if (!tcam_seed_fused_supported(HW, kmax))
        return fail(TCAMCRF_ERR_INVALID, "tcam_seed_fused: frame too large for shared memory or kmax > %d "
                    "(use tcam_seed_select + tcam_seed_labels)", kSeedFusedMaxK);
    if (B > 65535) return fail(TCAMCRF_ERR_INVALID, "batch too large");
    SeedFusedParams sp;
    sp.cams = cams_dev;
    sp.roi = reinterpret_cast<const long long *>(roi_dev);
    sp.q = q_dev;
    sp.q_offset = q_offset_dev;
    sp.n_cand = n_cand_dev;
    sp.rng = rng_dev;
    sp.cam_max = cam_max_dev;
    sp.sel = sel_dev;
    sp.labels = reinterpret_cast<long long *>(labels_dev);
    sp.T = T;
    sp.HW = HW;
    sp.H = H;
    sp.W = W;
    sp.kmax = kmax;
    sp.k_fg = k_fg;
    sp.k_bg = k_bg;
    sp.weighted_fg = weighted_fg;
    sp.max_p = max_p;
    sp.n_fg_fixed = n_fg_fixed;
    sp.n_bg = n_bg;
    sp.ksz = ksz;
    sp.ignore_idx = ignore_idx;
    sp.slice = seed_fused_slice(HW);
    StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = dim3(kSeedCluster, B);
    lc.blockDim = dim3(kSeedFusedThreads);
    lc.dynamicSmemBytes = (size_t)sp.slice * 2 * sizeof(unsigned int);
    lc.stream = (cudaStream_t)cuda_stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kSeedCluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&lc, seed_fused_kernel, sp));
    return TCAMCRF_OK;
}

int tcam_seed_ce_forward(const float *logits_dev, const int *sel_dev, int kmax, int B, int K, int H, int W, int ksz,
                         float *scratch_dev, float *loss_dev, float *count_dev, const float *add_dev, float weight,
                         float *total_dev, void *cuda_stream)
{
    return tcam_seed_ce_forward_typed(logits_dev, TCAMCRF_DTYPE_F32, sel_dev, kmax, B, K, H, W, ksz, scratch_dev,
                                      loss_dev, count_dev, add_dev, weight, total_dev, cuda_stream);
}

int tcam_seed_ce_forward_typed(const void *logits_dev, int logits_dtype, const int *sel_dev, int kmax, int B, int K,
                               int H, int W, int ksz, float *scratch_dev, float *loss_dev, float *count_dev,
                               const float *add_dev, float weight, float *total_dev, void *cuda_stream)
{
    if (logits_flags(logits_dtype) < 0) return TCAMCRF_ERR_INVALID;
    if (!logits_dev || !sel_dev || !scratch_dev || !loss_dev || !count_dev)
        return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || K < 2 || H < 1 || W < 1 || kmax < 1 || ksz < 1)
        return fail(TCAMCRF_ERR_INVALID, "B,H,W,kmax,ksz must be positive and K >= 2");
    SeedCeParams sp;
    sp.logits = logits_dev;
    sp.sel = sel_dev;
    sp.partial = scratch_dev + 1;
    sp.ticket = reinterpret_cast<int *>(scratch_dev);
    sp.loss_out = loss_dev;
    sp.count_out = count_dev;
    sp.add = add_dev;
    sp.total_out = total_dev;
    sp.weight = weight;
    sp.B = B;
    sp.K = K;
    sp.H = H;
    sp.W = W;
    sp.kmax = kmax;
    sp.ksz = ksz;
    sp.bf16 = logits_dtype == TCAMCRF_DTYPE_BF16;
    StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
    if (logits_dtype == TCAMCRF_DTYPE_F32)
        seed_ce_forward_kernel<<<B, 256, 0, (cudaStream_t)cuda_stream>>>(sp);
    else
        seed_ce_forward_lowp_kernel<<<B, 256, 0, (cudaStream_t)cuda_stream>>>(sp);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcam_seed_ce_backward(const float *logits_dev, const int *sel_dev, int kmax, int B, int K, int H, int W, int ksz,
                          const float *count_dev, const float *grad_out_dev, float scale, float *grad_logits_dev,
                          void *cuda_stream)
{
    return tcam_seed_ce_backward_typed(logits_dev, TCAMCRF_DTYPE_F32, sel_dev, kmax, B, K, H, W, ksz, count_dev,
                                       grad_out_dev, scale, grad_logits_dev, cuda_stream);
}

// the cross-entropy's share of the backward pass; crf_as_dev != NULL: grad_logits_dev holds the CRF gradient of
// loss_backward_logits_lowp_kernel, which the labelled pixels recompute in float32 (seed_ce_backward_lowp_kernel)
static int seed_ce_backward_any(const void *logits_dev, int logits_dtype, const int *sel_dev, int kmax, int B, int K,
                                int H, int W, int ksz, const float *count_dev, const float *grad_out_dev, float scale,
                                void *grad_logits_dev, const float *crf_as_dev, float n_norm, float crf_weight,
                                cudaStream_t st)
{
    if (!logits_dev || !sel_dev || !count_dev || !grad_out_dev || !grad_logits_dev)
        return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || K < 2 || H < 1 || W < 1 || kmax < 1 || ksz < 1)
        return fail(TCAMCRF_ERR_INVALID, "B,H,W,kmax,ksz must be positive and K >= 2");
    StageScope scope(kStSeed, 1, st);
    if (logits_dtype == TCAMCRF_DTYPE_F32) {
        seed_ce_backward_kernel<<<B, 256, 0, st>>>((const float *)logits_dev, sel_dev, (float *)grad_logits_dev,
                                                   count_dev, grad_out_dev, scale, K, H, W, kmax, ksz);
    } else {
        const int bf16 = logits_dtype == TCAMCRF_DTYPE_BF16;
        seed_ce_backward_lowp_kernel<<<B, 256, 0, st>>>(
            Logits16{(const unsigned short *)logits_dev, bf16}, sel_dev, Grad16{(unsigned short *)grad_logits_dev, bf16},
            count_dev, grad_out_dev, scale, K, H, W, kmax, ksz, crf_as_dev, n_norm, crf_weight);
    }
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcam_seed_ce_backward_typed(const void *logits_dev, int logits_dtype, const int *sel_dev, int kmax, int B, int K,
                                int H, int W, int ksz, const float *count_dev, const float *grad_out_dev, float scale,
                                void *grad_logits_dev, void *cuda_stream)
{
    if (logits_flags(logits_dtype) < 0) return TCAMCRF_ERR_INVALID;
    return seed_ce_backward_any(logits_dev, logits_dtype, sel_dev, kmax, B, K, H, W, ksz, count_dev, grad_out_dev,
                                scale, grad_logits_dev, nullptr, 0.f, 0.f, (cudaStream_t)cuda_stream);
}

int tcam_crf_seed_ce_backward_typed(const float *as_dev, const void *logits_dev, int logits_dtype, const int *sel_dev,
                                    int kmax, int ksz, const float *count_dev, const float *grad_out_dev, int B, int K,
                                    int H, int W, float n_norm, float crf_weight, float ce_weight,
                                    void *grad_logits_dev, void *cuda_stream)
{
    int rc = tcamcrf_loss_backward_logits_typed(as_dev, logits_dev, logits_dtype, grad_out_dev, grad_logits_dev, B, K,
                                                H, W, n_norm, crf_weight, cuda_stream);
    if (rc) return rc;
    // float32: the cross-entropy is added in place onto the float32 CRF gradient, exactly as before
    return seed_ce_backward_any(logits_dev, logits_dtype, sel_dev, kmax, B, K, H, W, ksz, count_dev, grad_out_dev,
                                ce_weight, grad_logits_dev, logits_dtype == TCAMCRF_DTYPE_F32 ? nullptr : as_dev,
                                n_norm, crf_weight, (cudaStream_t)cuda_stream);
}

int tcam_seed_labels(const int *sel_dev, int kmax, int B, int H, int W, int ksz, long long ignore_idx,
                     int64_t *out_dev, void *cuda_stream)
{
    if (!sel_dev || !out_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || H < 1 || W < 1 || kmax < 1 || ksz < 1) return fail(TCAMCRF_ERR_INVALID, "B,H,W,kmax,ksz must be positive");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    const long long total = (long long)B * H * W;
    long long blocks = (total + 255) / 256;
    if (blocks > persistent_grid(*dev)) blocks = persistent_grid(*dev);
    {
        StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
        seed_labels_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(
            sel_dev, kmax, B, H, W, ksz, ignore_idx, reinterpret_cast<long long *>(out_dev));
    }
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcam_otsu_roi(const float *cams_dev, int64_t *roi_dev, float *thresh_dev, int B, int HW, void *cuda_stream)
{
    if (!cams_dev || !roi_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || HW < 1) return fail(TCAMCRF_ERR_INVALID, "B,HW must be positive");
    {
        StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
        otsu_roi_kernel<<<B, kSeedThreads, 0, (cudaStream_t)cuda_stream>>>(
            cams_dev, reinterpret_cast<long long *>(roi_dev), thresh_dev, HW);
    }
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcam_temporal_max(const float *cams_dev, float *out_dev, int B, int T, int HW, void *cuda_stream)
{
    if (!cams_dev || !out_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || T < 1 || HW < 1) return fail(TCAMCRF_ERR_INVALID, "B,T,HW must be positive");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    const long long total = (long long)B * HW;
    long long blocks = (total + kThreads - 1) / kThreads;
    if (blocks > persistent_grid(*dev)) blocks = persistent_grid(*dev);
    StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
    temporal_max_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)cuda_stream>>>(cams_dev, out_dev, T, HW, total);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

size_t tcam_roi_components_scratch_bytes(int B, int H, int W)
{
    if (B < 1 || H < 1 || W < 1) return 0;
    return (size_t)B * H * W * (2 * sizeof(int) + sizeof(double)) + 256;
}

int tcam_roi_components(const float *cams_dev, const float *thresh_dev, long long *roi_dev, float *bbox_mask_dev,
                        int *bbox_dev, int B, int H, int W, int largest_only, double p_min_area, void *scratch_dev,
                        size_t scratch_bytes, void *cuda_stream)
{
    if (!cams_dev || !thresh_dev || !roi_dev || !bbox_mask_dev || !bbox_dev || !scratch_dev)
        return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || H < 1 || W < 1) return fail(TCAMCRF_ERR_INVALID, "B,H,W must be positive");
    if ((long long)H * W > (1ll << 26)) return fail(TCAMCRF_ERR_INVALID, "image too large");
    if (scratch_bytes < tcam_roi_components_scratch_bytes(B, H, W))
        return fail(TCAMCRF_ERR_WORKSPACE, "scratch too small");
    const size_t n = (size_t)B * H * W;
    char *base = (char *)(((uintptr_t)scratch_dev + 255) / 256 * 256);
    double *sum = (double *)base;
    int *labels = (int *)(base + n * sizeof(double));
    int *area = labels + n;
    StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
    // min_area = (h * w) * p_min_area_roi in float64 (tcam_seeding.py:364)
    roi_components_kernel<<<B, kSeedThreads, 0, (cudaStream_t)cuda_stream>>>(
        cams_dev, thresh_dev, roi_dev, bbox_mask_dev, bbox_dev, labels, area, sum, H, W, largest_only ? 1 : 0,
        (double)((long long)H * W) * p_min_area);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcam_temporal_max_renorm(const float *cams_dev, float *out_dev, int B, int T, int HW, float h, void *cuda_stream)
{
    if (!cams_dev || !out_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || T < 1 || HW < 1) return fail(TCAMCRF_ERR_INVALID, "B,T,HW must be positive");
    if (!(h > 0.f)) return tcam_temporal_max(cams_dev, out_dev, B, T, HW, cuda_stream);   // wsol_loader.py:594
    StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
    temporal_max_renorm_kernel<<<B, kSeedThreads, 0, (cudaStream_t)cuda_stream>>>(cams_dev, out_dev, T, HW, h);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

int tcam_prepare_std_cams(const float *cams_dev, float *out_dev, int B, int h, int w, int H, int W, void *cuda_stream)
{
    if (!cams_dev || !out_dev) return fail(TCAMCRF_ERR_INVALID, "null pointer argument");
    if (B < 1 || h < 1 || w < 1 || H < 1 || W < 1) return fail(TCAMCRF_ERR_INVALID, "sizes must be positive");
    Device *dev = nullptr;
    if (const int rc = this_device(&dev)) return rc;
    const long long total = (long long)B * H * W;
    long long blocks = (total + 255) / 256;
    if (blocks > persistent_grid(*dev)) blocks = persistent_grid(*dev);
    StageScope scope(kStSeed, 1, (cudaStream_t)cuda_stream);
    // ATen: scale = (float)input_size / output_size when no scale factor is given (upsample with size=)
    prepare_std_cams_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(
        cams_dev, out_dev, h, w, H, W, (float)h / (float)H, (float)w / (float)W, total);
    CUDA_TRY(cudaGetLastError());
    return TCAMCRF_OK;
}

}  // extern "C"
