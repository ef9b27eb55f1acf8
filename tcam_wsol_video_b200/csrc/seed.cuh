// seed.cuh -- temporal-CAM max fused with fg/bg seed selection, and the seed-label map.
// Included by tcamcrf.cu (one translation unit, one .so).
//
// What it replaces in the reference:
//   tcam_seed_select  <- the chain of torch.maximum over the frames' CAMs (dlib/datasets/wsol_loader.py:591-600)
//                        + _SFG.forward / _SBG.forward for every sample of the batch
//                        (dlib/cams/tcam_seeding.py:498-592): `cam*roi + 1e-8`, stable sort, top-n mask,
//                        row-major candidates, multinomial without replacement
//   tcam_seed_labels  <- TCAMSeeder.forward's tail (tcam_seeding.py:239-254): kornia flat ksz x ksz dilation
//                        of the fg and bg one-hot maps, fg/bg conflict -> ignore, labels {ignore, 0, 1}
//
// The reference sorts all H*W values twice per sample only to find which pixels are the n largest /
// smallest; here ONE thread block per (sample, fg|bg) finds the n-th value with a 4-pass radix select and
// breaks ties by pixel index, which is what a stable sort does.  torch.multinomial without replacement is
// argmax / top-k of p / q with q ~ Exp(1) drawn in candidate (row-major) order; the draws are an INPUT, so
// the selection is bit-exact given the same draws.
#pragma once
#include <cstdint>
#include <cooperative_groups.h>
#include <cuda_runtime.h>

namespace tcamcrf {

constexpr int kSeedThreads = 1024;

// ascending-order key of a float (NaN sorts last, like torch.sort); -0.0 is folded onto +0.0
__device__ __forceinline__ unsigned int float_order_key(float v)
{
    v = v + 0.0f;
    const unsigned int b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// block-wide exclusive scan of one int per thread (kSeedThreads threads); returns the exclusive prefix and the
// block total through `total`
__device__ __forceinline__ int block_exclusive_scan(int v, int *s_warp, int &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();  // s_warp may still be read from the previous scan
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        s_warp[lane] = wi - w;          // exclusive warp offsets
        if (lane == 31) s_warp[32] = wi;  // block total
    }
    __syncthreads();
    total = s_warp[32];
    return s_warp[warp] + incl - v;
}

struct SeedParams {
    const float *cams;      // [B][T][HW]
    const long long *roi;   // [B][HW] or null
    const float *q;         // exponential draws, all samples concatenated
    const int *q_offset;    // [B][2] start of the (sample, fg|bg) draws in q
    const int *n_cand;      // [B][2] candidates (0 -> no seed: degenerate cam, n == 0, or min_/max_ == 0)
    float *cam_max;         // [B][HW] out: temporal max (before roi / epsilon)
    float *scratch;         // [B][2][HW] scores
    int *sel;               // [B][2][kmax] out: selected pixel indices, -1 = unused
    int T, HW, kmax;
    int k_fg, k_bg;
    int weighted_fg;
};

// grid (2, B): blockIdx.x = 0 foreground, 1 background
__global__ void __launch_bounds__(kSeedThreads) seed_select_kernel(const SeedParams p)
{
    __shared__ int s_hist[256];
    __shared__ int s_warp[33];
    __shared__ unsigned int s_prefix;
    __shared__ int s_need;
    __shared__ float s_best_v[32];
    __shared__ int s_best_i[32];

    const int b = blockIdx.y;
    const bool fg = blockIdx.x == 0;
    const int tid = threadIdx.x;
    const int HW = p.HW;
    const float *cam0 = p.cams + (size_t)b * p.T * HW;
    float *cmax = p.cam_max + (size_t)b * HW;
    const long long *roi = (fg && p.roi) ? p.roi + (size_t)b * HW : nullptr;
    float *score = p.scratch + ((size_t)b * 2 + (fg ? 0 : 1)) * HW;
    int *sel = p.sel + ((size_t)b * 2 + (fg ? 0 : 1)) * p.kmax;
    const int n = p.n_cand[b * 2 + (fg ? 0 : 1)];
    int k = fg ? p.k_fg : p.k_bg;
    if (k > n) k = n;
    if (k > p.kmax) k = p.kmax;

    // pass 0 (foreground block only writes it): temporal max, float4 over the T planes where HW allows
    if (fg) {
        if ((HW & 3) == 0) {
            for (int i = tid; i < HW / 4; i += kSeedThreads) {
                float4 m = __ldg(reinterpret_cast<const float4 *>(cam0) + i);
                for (int t = 1; t < p.T; t++) {
                    const float4 v = __ldg(reinterpret_cast<const float4 *>(cam0 + (size_t)t * HW) + i);
                    // torch.maximum: NaN if either operand is NaN
                    m.x = (m.x != m.x) ? m.x : ((v.x != v.x) ? v.x : (v.x > m.x ? v.x : m.x));
                    m.y = (m.y != m.y) ? m.y : ((v.y != v.y) ? v.y : (v.y > m.y ? v.y : m.y));
                    m.z = (m.z != m.z) ? m.z : ((v.z != v.z) ? v.z : (v.z > m.z ? v.z : m.z));
                    m.w = (m.w != m.w) ? m.w : ((v.w != v.w) ? v.w : (v.w > m.w ? v.w : m.w));
                }
                reinterpret_cast<float4 *>(cmax)[i] = m;
            }
        } else {
            for (int i = tid; i < HW; i += kSeedThreads) {
                float m = __ldg(cam0 + i);
                for (int t = 1; t < p.T; t++) {
                    const float v = __ldg(cam0 + (size_t)t * HW + i);
                    m = (m != m) ? m : ((v != v) ? v : (v > m ? v : m));
                }
                cmax[i] = m;
            }
        }
    }
    for (int i = tid; i < p.kmax; i += kSeedThreads) sel[i] = -1;
    if (n <= 0 || k <= 0) return;

    // value of pixel i as the reference scores it: cam*roi + 1e-8 (fg with roi) or cam + 1e-8
    // (tcam_seeding.py:511-517,564-565).  The background block recomputes the max instead of waiting for
    // the foreground block's cam_max.
    auto value_at = [&](int i) -> float {
        float m = __ldg(cam0 + i);
        for (int t = 1; t < p.T; t++) {
            const float v = __ldg(cam0 + (size_t)t * HW + i);
            m = (m != m) ? m : ((v != v) ? v : (v > m ? v : m));
        }
        if (roi) m = __fmul_rn(m, (float)__ldg(roi + i));
        return __fadd_rn(m, 1e-8f);
    };
    // selection key: the n SMALLEST keys are the candidates (descending order for the foreground)
    auto key_at = [&](int i) -> unsigned int {
        const unsigned int u = float_order_key(value_at(i));
        return fg ? ~u : u;
    };

    // radix select, 8 bits at a time from the top: after 4 passes `prefix` is the n-th smallest key
    unsigned int prefix = 0;
    int need = n;  // rank of the wanted key among the keys that share the current prefix
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += kSeedThreads) s_hist[i] = 0;
        __syncthreads();
        const unsigned int himask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
        for (int i = tid; i < HW; i += kSeedThreads) {
            const unsigned int key = key_at(i);
            if ((key & himask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255u], 1);
        }
        __syncthreads();
        if (tid == 0) {
            int run = 0, bin = 0;
            for (; bin < 256; bin++) {
                if (run + s_hist[bin] >= need) break;
                run += s_hist[bin];
            }
            s_prefix = prefix | ((unsigned int)bin << shift);
            s_need = need - run;
        }
        __syncthreads();
        prefix = s_prefix;
        need = s_need;
        __syncthreads();
    }
    const unsigned int kth = prefix;   // keys < kth are candidates; of the keys == kth the first `need` by index

    // candidates in row-major order -> their draw q[rank]; score = p / q  (torch.multinomial without replacement)
    const float *q = p.q + p.q_offset[b * 2 + (fg ? 0 : 1)];
    const bool weighted = fg && p.weighted_fg;
    int ties_before = 0, cands_before = 0;
    for (int base = 0; base < HW; base += kSeedThreads) {
        const int i = base + tid;
        unsigned int key = 0xffffffffu;
        float val = 0.f;
        if (i < HW) {
            val = value_at(i);
            const unsigned int u = float_order_key(val);
            key = fg ? ~u : u;
        }
        const int is_tie = (i < HW && key == kth) ? 1 : 0;
        int tie_total, cand_total;
        const int tie_rank = ties_before + block_exclusive_scan(is_tie, s_warp, tie_total);
        const int is_cand = (i < HW && (key < kth || (is_tie && tie_rank < need))) ? 1 : 0;
        const int cand_rank = cands_before + block_exclusive_scan(is_cand, s_warp, cand_total);
        if (i < HW) {
            float sc = -INFINITY;
            if (is_cand) sc = __fdiv_rn(weighted ? val : 1.0f, __ldg(q + cand_rank));
            score[i] = sc;
        }
        ties_before += tie_total;
        cands_before += cand_total;
    }
    __syncthreads();

    // k rounds of block argmax (lowest index wins ties); a selected pixel is retired with -inf
    for (int round = 0; round < k; round++) {
        float bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int i = tid; i < HW; i += kSeedThreads) {
            const float s = score[i];
            if (s > bv || (s == bv && i < bi && s != -INFINITY)) {
                bv = s;
                bi = i;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) {
                bv = ov;
                bi = oi;
            }
        }
        if ((tid & 31) == 0) {
            s_best_v[tid >> 5] = bv;
            s_best_i[tid >> 5] = bi;
        }
        __syncthreads();
        if (tid < 32) {
            bv = s_best_v[tid];
            bi = s_best_i[tid];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) {
                    bv = ov;
                    bi = oi;
                }
            }
            if (tid == 0) {
                if (bv > -INFINITY && bi < HW) {
                    sel[round] = bi;
                    score[bi] = -INFINITY;
                }
            }
        }
        __syncthreads();
    }
}

// inverse of float_order_key
__device__ __forceinline__ float float_from_order_key(unsigned int u)
{
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// The same selection with the sample's keys resident in shared memory (HW * 4 bytes of dynamic shared memory, i.e.
// frames up to ~56 k pixels: 224 x 224 fits): the temporal max is taken once instead of in each of the four radix
// passes and in the ranking pass, and the row-major candidate ranks come from TWO block scans over per-thread
// counts -- every thread owns a contiguous chunk of pixels -- instead of two scans per 1024 pixels (~100 scans,
// ~300 barriers at 224 x 224).  Bit-identical results to seed_select_kernel; TCAMSeeder.forward_stack on 32 samples of
// 224 x 224: 0.48 -> 0.30 ms (tools/seed_timing.py).
__global__ void __launch_bounds__(kSeedThreads) seed_select_smem_kernel(const SeedParams p)
{
    extern __shared__ unsigned int s_key[];   // [HW] selection keys, later the scores
    __shared__ int s_hist[256];
    __shared__ int s_warp[33];
    __shared__ unsigned int s_prefix;
    __shared__ int s_need;
    __shared__ float s_best_v[32];
    __shared__ int s_best_i[32];

    const int b = blockIdx.y;
    const bool fg = blockIdx.x == 0;
    const int tid = threadIdx.x;
    const int HW = p.HW;
    const float *cam0 = p.cams + (size_t)b * p.T * HW;
    float *cmax = p.cam_max + (size_t)b * HW;
    const long long *roi = (fg && p.roi) ? p.roi + (size_t)b * HW : nullptr;
    int *sel = p.sel + ((size_t)b * 2 + (fg ? 0 : 1)) * p.kmax;
    const int n = p.n_cand[b * 2 + (fg ? 0 : 1)];
    int k = fg ? p.k_fg : p.k_bg;
    if (k > n) k = n;
    if (k > p.kmax) k = p.kmax;
    const bool active = n > 0 && k > 0;

    // one pass over the T planes: temporal max (written by the foreground block), value = cam*roi + 1e-8 or
    // cam + 1e-8 (tcam_seeding.py:511-517,564-565), key = its order key (complemented for the foreground: the n
    // SMALLEST keys are the candidates)
    for (int i = tid; i < HW; i += kSeedThreads) {
        float m = __ldg(cam0 + i);
        for (int t = 1; t < p.T; t++) {
            const float v = __ldg(cam0 + (size_t)t * HW + i);
            m = (m != m) ? m : ((v != v) ? v : (v > m ? v : m));   // torch.maximum: NaN if either is NaN
        }
        if (fg) cmax[i] = m;
        if (roi) m = __fmul_rn(m, (float)__ldg(roi + i));
        const unsigned int u = float_order_key(__fadd_rn(m, 1e-8f));
        s_key[i] = fg ? ~u : u;
    }
    for (int i = tid; i < p.kmax; i += kSeedThreads) sel[i] = -1;
    if (!active) return;
    __syncthreads();

    // radix select, 8 bits at a time from the top: after 4 passes `prefix` is the n-th smallest key
    unsigned int prefix = 0;
    int need = n;
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += kSeedThreads) s_hist[i] = 0;
        __syncthreads();
        const unsigned int himask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
        for (int i = tid; i < HW; i += kSeedThreads) {
            const unsigned int key = s_key[i];
            if ((key & himask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255u], 1);
        }
        __syncthreads();
        if (tid == 0) {
            int run = 0, bin = 0;
            for (; bin < 256; bin++) {
                if (run + s_hist[bin] >= need) break;
                run += s_hist[bin];
            }
            s_prefix = prefix | ((unsigned int)bin << shift);
            s_need = need - run;
        }
        __syncthreads();
        prefix = s_prefix;
        need = s_need;
        __syncthreads();
    }
    const unsigned int kth = prefix;   // keys < kth are candidates; of the keys == kth the first `need` by index

    // row-major ranks: thread t owns pixels [t*chunk, (t+1)*chunk)
    const int chunk = (HW + kSeedThreads - 1) / kSeedThreads;
    const int lo = min(tid * chunk, HW), hi = min(lo + chunk, HW);
    int my_ties = 0;
    for (int i = lo; i < hi; i++) my_ties += s_key[i] == kth;
    int tie_total;
    int tie_rank = block_exclusive_scan(my_ties, s_warp, tie_total);
    int my_cands = 0;
    {
        int tr = tie_rank;
        for (int i = lo; i < hi; i++) {
            const unsigned int key = s_key[i];
            if (key < kth) my_cands++;
            else if (key == kth) my_cands += (tr++ < need);
        }
    }
    int cand_total;
    int cand_rank = block_exclusive_scan(my_cands, s_warp, cand_total);
    // candidates -> their draw q[rank]; score = p / q (torch.multinomial without replacement); others -inf.
    // The scores replace the keys in shared memory.
    const float *q = p.q + p.q_offset[b * 2 + (fg ? 0 : 1)];
    const bool weighted = fg && p.weighted_fg;
    for (int i = lo; i < hi; i++) {
        const unsigned int key = s_key[i];
        bool is_cand = key < kth;
        if (key == kth) is_cand = tie_rank++ < need;
        float sc = -INFINITY;
        if (is_cand) {
            const float val = float_from_order_key(fg ? ~key : key);
            sc = __fdiv_rn(weighted ? val : 1.0f, __ldg(q + cand_rank));
            cand_rank++;
        }
        s_key[i] = __float_as_uint(sc);
    }
    __syncthreads();

    // k rounds of block argmax (lowest index wins ties); a selected pixel is retired with -inf
    for (int round = 0; round < k; round++) {
        float bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int i = tid; i < HW; i += kSeedThreads) {
            const float sc = __uint_as_float(s_key[i]);
            if (sc > bv || (sc == bv && i < bi && sc != -INFINITY)) {
                bv = sc;
                bi = i;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) {
                bv = ov;
                bi = oi;
            }
        }
        if ((tid & 31) == 0) {
            s_best_v[tid >> 5] = bv;
            s_best_i[tid >> 5] = bi;
        }
        __syncthreads();
        if (tid < 32) {
            bv = s_best_v[tid];
            bi = s_best_i[tid];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) {
                    bv = ov;
                    bi = oi;
                }
            }
            if (tid == 0) {
                if (bv > -INFINITY && bi < HW) {
                    sel[round] = bi;
                    s_key[bi] = __float_as_uint(-INFINITY);
                }
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------
// The whole seeding step of a batch in ONE launch, at GPU width: a thread-block CLUSTER of 8 blocks per sample.
//
// seed_select[_smem]_kernel run one block per (sample, fg|bg): 64 blocks on 148 SMs, the temporal max taken by both
// blocks, four serial 256-bin scans by one thread, candidate counts from five torch reductions, 2*H*W exponential draws
// per sample made by torch (12.8 MB per step) to use a few of them, and a second launch for the label map.  Here:
//   * block r of the cluster owns pixels [r*slice, (r+1)*slice) of the sample: ONE pass over the T planes (float4)
//     gives the temporal max (written out), min / max / roi count for the candidate counts (tcam_seeding.py:465,510,519,
//     567) and the fg and bg selection keys, kept in shared memory (2 x 4 bytes per pixel of the slice);
//   * 4-pass radix select for both sides at once: per-block 256-bin histograms in shared memory, summed across the
//     cluster by reading the other blocks' histograms through distributed shared memory (one cluster barrier per pass,
//     histograms double-buffered), bin scan by one warp per side;
//   * ties at the threshold go to the lowest pixel indices (stable sort), row-major candidate ranks come from block
//     scans + a cluster-wide exclusive prefix -- needed only when the draws are an INPUT (rng_parity: bit-identical to
//     the reference's stream); otherwise the Exp(1) draw of a candidate comes from Philox4x32-10 keyed by two words
//     torch's CUDA generator produced for this call and counted by (sample, side, pixel): only candidates draw;
//   * top-k by score p/q: k rounds of block arg-max + cluster all-gather; then every block writes the label map of its
//     slice (kornia's flat ksz x ksz dilation of the fg / bg seeds, conflicts -> ignore, tcam_seeding.py:239-254).
// Results are bit-identical to seed_select_kernel + seed_labels_kernel when the draws are given.
namespace cg = cooperative_groups;

constexpr int kSeedCluster = 8;          // portable cluster size
#ifndef TCAMCRF_SEED_THREADS
#define TCAMCRF_SEED_THREADS 512
#endif
constexpr int kSeedFusedThreads = TCAMCRF_SEED_THREADS;   // 512 or 1024
static_assert(kSeedFusedThreads >= 512 && kSeedFusedThreads <= 1024 && kSeedFusedThreads % 32 == 0, "one thread per (side, bin)");
constexpr int kSeedFusedMaxK = 32;       // seeds per side this kernel handles (larger k: the two-kernel path)

struct SeedFusedParams {
    const float *cams;          // [B][T][HW]
    const long long *roi;       // [B][HW] or null
    const float *q;             // exponential draws in candidate order, or null -> Philox
    const int *q_offset;        // [B][2] (with q)
    const int *n_cand;          // [B][2] candidate counts computed by the caller, or null -> computed here
    const unsigned int *rng;    // [2] Philox key words (with q == null)
    float *cam_max;             // [B][HW]
    int *sel;                   // [B][2][kmax]
    long long *labels;          // [B][HW] or null
    int T, HW, H, W, kmax, k_fg, k_bg, weighted_fg;
    float max_p;                // float32(max_p): n_fg = int(max_p * roi.sum()) as a float32 product
    int n_fg_fixed;             // n_fg without a roi: int(max_p * H * W)
    int n_bg;                   // int(min_p * H * W)
    int ksz;
    long long ignore_idx;
    int slice;                  // pixels per block of the cluster (multiple of 4)
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned int hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned int hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// random word of (sample, side, pixel): first output word of Philox4x32-10 at counter (pixel, 2b + side, 0x5eed, 0)
__device__ __forceinline__ unsigned int seed_philox_word(uint2 key, int b, int side, int pixel)
{
    return philox4x32_10(make_uint4((unsigned int)pixel, (unsigned int)(b * 2 + side), 0x5eedu, 0u), key).x;
}

// Exp(1) draw from a 32-bit word: -log(u), u = (2m + 1) * 2^-24 with m = word >> 9.  2m + 1 < 2^24, so u is exact in
// float32 and lies in [2^-24, 1 - 2^-24]: the draw is finite and > 0 (5.96e-8 .. 16.6), and u never rounds to 1 (a
// zero draw would score -inf, the score of a non-candidate).  The smallest draws decide the picks and come from u near
// 1, where __logf's absolute error bound is a few percent of the result; logf is within 1 ulp there.
__device__ __forceinline__ float exp1_from_word(unsigned int word)
{
    const float u = (float)((word >> 9) * 2u + 1u) * (1.0f / 16777216.0f);
    return -logf(u);
}

// test hooks (tcam_debug_seed_draws / tcam_debug_exp_draws): the words and draws seed_fused_kernel makes.
// words / draws [B][2][HW]
__global__ void __launch_bounds__(256) seed_debug_draws_kernel(const unsigned int *__restrict__ rng, int B, int HW,
                                                               unsigned int *__restrict__ words, float *__restrict__ draws)
{
    const uint2 key = make_uint2(__ldg(rng), __ldg(rng + 1));
    const long long total = (long long)B * 2 * HW;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int bs = (int)(i / HW), pixel = (int)(i - (long long)bs * HW);
        const unsigned int w = seed_philox_word(key, bs >> 1, bs & 1, pixel);
        words[i] = w;
        draws[i] = exp1_from_word(w);
    }
}

__global__ void __launch_bounds__(256) seed_debug_exp_kernel(const unsigned int *__restrict__ words, int n,
                                                             float *__restrict__ draws)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) draws[i] = exp1_from_word(words[i]);
}

__device__ __forceinline__ float nanmax(float m, float v)   // torch.maximum: NaN if either is NaN
{
    return (m != m) ? m : ((v != v) ? v : (v > m ? v : m));
}

// block-wide exclusive scan for kSeedFusedThreads threads (same contract as block_exclusive_scan)
__device__ __forceinline__ int fused_exclusive_scan(int v, int *s_warp, int &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = lane < kSeedFusedThreads / 32 ? s_warp[lane] : 0;
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        s_warp[lane] = wi - w;
        if (lane == 31) s_warp[32] = wi;
    }
    __syncthreads();
    total = s_warp[32];
    return s_warp[warp] + incl - v;
}

__global__ void __launch_bounds__(kSeedFusedThreads) seed_fused_kernel(const SeedFusedParams p)
{
    extern __shared__ unsigned int s_key[];           // [2][slice]: keys, later scores (fg first)
    __shared__ int s_hist[2][2][256];                 // [buffer][side][bin]
    __shared__ int s_tot[2][256];
    __shared__ int s_gi[2][kSeedCluster][4];          // small all-gathers across the cluster, double-buffered
    __shared__ float s_gf[2][kSeedCluster][2];
    __shared__ int s_warp[33];
    __shared__ float s_rf[2][kSeedFusedThreads / 32];
    __shared__ int s_ri[2][kSeedFusedThreads / 32];
    __shared__ unsigned int s_prefix[2];
    __shared__ int s_need[2];
    __shared__ int s_sel[2][kSeedFusedMaxK];

    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int HW = p.HW, slice = p.slice;
    const int lo = min(rank * slice, HW), hi = min(lo + slice, HW);
    const int cnt = hi - lo;
    const float *cam0 = p.cams + (size_t)b * p.T * HW;
    float *cmax = p.cam_max + (size_t)b * HW;
    const long long *roi = p.roi ? p.roi + (size_t)b * HW : nullptr;
    unsigned int *key_fg = s_key, *key_bg = s_key + slice;
    int gbuf = 0;   // which gather buffer the next all-gather uses

    // every block of the cluster writes `vals` into slot [rank] of EVERY block's gather buffer
    auto gather_put_i = [&](int buf, int v0, int v1, int v2, int v3) {
        if (tid < kSeedCluster) {
            int *dst = cluster.map_shared_rank(&s_gi[buf][rank][0], tid);
            dst[0] = v0; dst[1] = v1; dst[2] = v2; dst[3] = v3;
        }
    };

    // ---- pass 0: temporal max, keys, statistics of the slice
    float mn = INFINITY, mx = -INFINITY;
    int has_nan = 0, roi_sum = 0;
    auto take = [&](int i, float m) {   // i: index within the slice
        has_nan |= (m != m);
        mn = fminf(mn, m);
        mx = fmaxf(mx, m);
        float vfg = m;
        if (roi) {
            const long long r = __ldg(roi + lo + i);
            roi_sum += (int)r;
            vfg = __fmul_rn(m, (float)r);
        }
        key_fg[i] = ~float_order_key(__fadd_rn(vfg, 1e-8f));   // the n SMALLEST keys are the candidates
        key_bg[i] = float_order_key(__fadd_rn(m, 1e-8f));
    };
    if ((HW & 3) == 0) {   // slice and HW are multiples of 4: whole float4s
        for (int i4 = tid; i4 < cnt / 4; i4 += kSeedFusedThreads) {
            float4 m = __ldg(reinterpret_cast<const float4 *>(cam0 + lo) + i4);
            for (int t = 1; t < p.T; t++) {
                const float4 v = __ldg(reinterpret_cast<const float4 *>(cam0 + (size_t)t * HW + lo) + i4);
                m.x = nanmax(m.x, v.x);
                m.y = nanmax(m.y, v.y);
                m.z = nanmax(m.z, v.z);
                m.w = nanmax(m.w, v.w);
            }
            reinterpret_cast<float4 *>(cmax + lo)[i4] = m;
            take(4 * i4 + 0, m.x);
            take(4 * i4 + 1, m.y);
            take(4 * i4 + 2, m.z);
            take(4 * i4 + 3, m.w);
        }
    } else {
        for (int i = tid; i < cnt; i += kSeedFusedThreads) {
            float m = __ldg(cam0 + lo + i);
            for (int t = 1; t < p.T; t++) m = nanmax(m, __ldg(cam0 + (size_t)t * HW + lo + i));
            cmax[lo + i] = m;
            take(i, m);
        }
    }
    for (int i = tid; i < 2 * kSeedFusedMaxK; i += kSeedFusedThreads) (&s_sel[0][0])[i] = -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        has_nan |= __shfl_xor_sync(0xffffffffu, has_nan, o);
        roi_sum += __shfl_xor_sync(0xffffffffu, roi_sum, o);
    }
    if (lane == 0) {
        s_rf[0][warp] = mn;
        s_rf[1][warp] = mx;
        s_ri[0][warp] = has_nan;
        s_ri[1][warp] = roi_sum;
    }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < kSeedFusedThreads / 32; w++) {
            mn = fminf(mn, s_rf[0][w]);
            mx = fmaxf(mx, s_rf[1][w]);
            has_nan |= s_ri[0][w];
            roi_sum += s_ri[1][w];
        }
        s_rf[0][0] = mn;
        s_rf[1][0] = mx;
        s_ri[0][0] = has_nan;
        s_ri[1][0] = roi_sum;
    }
    __syncthreads();
    gather_put_i(gbuf, __float_as_int(s_rf[0][0]), __float_as_int(s_rf[1][0]), s_ri[0][0], s_ri[1][0]);
    cluster.sync();
    int n[2], k[2];
    {
        float gmn = INFINITY, gmx = -INFINITY;
        int gnan = 0, gsum = 0;
        for (int r = 0; r < kSeedCluster; r++) {
            gmn = fminf(gmn, __int_as_float(s_gi[gbuf][r][0]));
            gmx = fmaxf(gmx, __int_as_float(s_gi[gbuf][r][1]));
            gnan |= s_gi[gbuf][r][2];
            gsum += s_gi[gbuf][r][3];
        }
        // flat CAM: no seeds at all (cam.min() == cam.max(), tcam_seeding.py:465; NaN compares unequal)
        const bool alive = gnan || gmn != gmx;
        n[0] = roi ? (int)__fmul_rn(p.max_p, (float)gsum) : p.n_fg_fixed;   // tcam_seeding.py:510,515,519
        n[1] = p.n_bg;                                                       // tcam_seeding.py:567
        if (p.k_fg <= 0 || !alive) n[0] = 0;
        if (p.k_bg <= 0 || !alive) n[1] = 0;
        if (p.n_cand) {   // the caller's counts (sized its draws with them)
            n[0] = p.n_cand[b * 2];
            n[1] = p.n_cand[b * 2 + 1];
        }
        n[0] = min(n[0], HW);
        n[1] = min(n[1], HW);
        k[0] = min(min(p.k_fg, n[0]), p.kmax);
        k[1] = min(min(p.k_bg, n[1]), p.kmax);
    }
    gbuf ^= 1;
    const bool on[2] = {n[0] > 0 && k[0] > 0, n[1] > 0 && k[1] > 0};

    if (on[0] || on[1]) {
        // ---- radix select, 8 bits at a time from the top, both sides at once
        if (tid < 2) {
            s_prefix[tid] = 0;
            s_need[tid] = n[tid];
        }
        for (int pass = 0; pass < 4; pass++) {
            const int shift = 24 - 8 * pass;
            const int hb = pass & 1;
            for (int i = tid; i < 512; i += kSeedFusedThreads) (&s_hist[hb][0][0])[i] = 0;
            __syncthreads();
            const unsigned int himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
#pragma unroll
            for (int side = 0; side < 2; side++) {
                if (!on[side]) continue;
                const unsigned int prefix = s_prefix[side];
                const unsigned int *keys = side ? key_bg : key_fg;
                for (int i = tid; i < cnt; i += kSeedFusedThreads) {
                    const unsigned int key = keys[i];
                    if ((key & himask) == prefix) atomicAdd(&s_hist[hb][side][(key >> shift) & 255u], 1);
                }
            }
            cluster.sync();   // every block's histogram of this pass is complete
            if (tid < 512) {   // thread (side, bin): the bin summed over the cluster
                const int side = tid >> 8, bin = tid & 255;
                int sum = 0;
                for (int r = 0; r < kSeedCluster; r++) sum += *cluster.map_shared_rank(&s_hist[hb][side][bin], r);
                s_tot[side][bin] = sum;
            }
            __syncthreads();
            if (warp < 2 && on[warp]) {   // one warp per side: which bin holds the need-th key
                const int side = warp;
                int c[8], mine = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    c[j] = s_tot[side][lane * 8 + j];
                    mine += c[j];
                }
                int incl = mine;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                const int need = s_need[side];
                const int excl = incl - mine;
                const unsigned int holds = __ballot_sync(0xffffffffu, excl < need && need <= incl);
                __syncwarp();
                if (holds && lane == __ffs(holds) - 1) {
                    int run = excl, bin = lane * 8;
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        if (run + c[j] >= need) break;
                        run += c[j];
                        bin++;
                    }
                    s_prefix[side] |= (unsigned int)bin << shift;
                    s_need[side] = need - run;
                }
            }
            __syncthreads();
        }
        // keys < kth are candidates; of the keys == kth the first `need` by pixel index
        // ---- row-major ranks: thread t owns pixels [t*chunk, (t+1)*chunk) of the slice
        const int chunk = (slice + kSeedFusedThreads - 1) / kSeedFusedThreads;
        const int clo = min(tid * chunk, cnt), chi = min(clo + chunk, cnt);
        int tie_rank[2] = {0, 0}, cand_rank[2] = {0, 0};
        {
            int my_ties[2] = {0, 0}, tot[2];
#pragma unroll
            for (int side = 0; side < 2; side++) {
                if (on[side]) {
                    const unsigned int *keys = side ? key_bg : key_fg;
                    const unsigned int kth = s_prefix[side];
                    for (int i = clo; i < chi; i++) my_ties[side] += keys[i] == kth;
                }
                tie_rank[side] = fused_exclusive_scan(my_ties[side], s_warp, tot[side]);
            }
            gather_put_i(gbuf, tot[0], tot[1], 0, 0);
            cluster.sync();
            for (int r = 0; r < rank; r++) {
                tie_rank[0] += s_gi[gbuf][r][0];
                tie_rank[1] += s_gi[gbuf][r][1];
            }
            gbuf ^= 1;
        }
        if (p.q) {   // the draws are an input, in row-major candidate order: global candidate ranks
            int my_c[2] = {0, 0}, tot[2];
#pragma unroll
            for (int side = 0; side < 2; side++) {
                if (on[side]) {
                    const unsigned int *keys = side ? key_bg : key_fg;
                    const unsigned int kth = s_prefix[side];
                    const int need = s_need[side];
                    int tr = tie_rank[side];
                    for (int i = clo; i < chi; i++) {
                        const unsigned int key = keys[i];
                        if (key < kth) my_c[side]++;
                        else if (key == kth) my_c[side] += (tr++ < need);
                    }
                }
                cand_rank[side] = fused_exclusive_scan(my_c[side], s_warp, tot[side]);
            }
            gather_put_i(gbuf, tot[0], tot[1], 0, 0);
            cluster.sync();
            for (int r = 0; r < rank; r++) {
                cand_rank[0] += s_gi[gbuf][r][0];
                cand_rank[1] += s_gi[gbuf][r][1];
            }
            gbuf ^= 1;
        }
        // ---- scores replace the keys: p / q for candidates (torch.multinomial without replacement), -inf otherwise
        uint2 rkey = make_uint2(0u, 0u);
        if (!p.q) rkey = make_uint2(__ldg(p.rng), __ldg(p.rng + 1));
#pragma unroll
        for (int side = 0; side < 2; side++) {
            if (!on[side]) continue;
            unsigned int *keys = side ? key_bg : key_fg;
            const unsigned int kth = s_prefix[side];
            const int need = s_need[side];
            const bool weighted = side == 0 && p.weighted_fg;
            const float *q = p.q ? p.q + p.q_offset[b * 2 + side] : nullptr;
            int tr = tie_rank[side], cr = cand_rank[side];
            for (int i = clo; i < chi; i++) {
                const unsigned int key = keys[i];
                bool is_cand = key < kth;
                if (key == kth) is_cand = tr++ < need;
                float sc = -INFINITY;
                if (is_cand) {
                    const float val = float_from_order_key(side ? key : ~key);
                    const float draw = q ? __ldg(q + cr++) : exp1_from_word(seed_philox_word(rkey, b, side, lo + i));
                    sc = __fdiv_rn(weighted ? val : 1.0f, draw);
                }
                keys[i] = __float_as_uint(sc);
            }
        }
        __syncthreads();
        // ---- top-k: k rounds of arg-max over the sample (lowest index wins ties), the winner retires with -inf
        const int rounds = max(on[0] ? k[0] : 0, on[1] ? k[1] : 0);
        for (int round = 0; round < rounds; round++) {
            float bv[2] = {-INFINITY, -INFINITY};
            int bi[2] = {0x7fffffff, 0x7fffffff};
#pragma unroll
            for (int side = 0; side < 2; side++) {
                if (!(on[side] && round < k[side])) continue;
                const unsigned int *keys = side ? key_bg : key_fg;
                for (int i = tid; i < cnt; i += kSeedFusedThreads) {
                    const float sc = __uint_as_float(keys[i]);
                    if (sc > bv[side] || (sc == bv[side] && lo + i < bi[side] && sc != -INFINITY)) {
                        bv[side] = sc;
                        bi[side] = lo + i;
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const float ov = __shfl_xor_sync(0xffffffffu, bv[side], o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi[side], o);
                    if (ov > bv[side] || (ov == bv[side] && oi < bi[side])) {
                        bv[side] = ov;
                        bi[side] = oi;
                    }
                }
                if (lane == 0) {
                    s_rf[side][warp] = bv[side];
                    s_ri[side][warp] = bi[side];
                }
            }
            __syncthreads();
            if (tid < 2) {
                const int side = tid;
                float v = -INFINITY;
                int ix = 0x7fffffff;
                if (on[side] && round < k[side])
                    for (int w = 0; w < kSeedFusedThreads / 32; w++) {
                        const float ov = s_rf[side][w];
                        const int oi = s_ri[side][w];
                        if (ov > v || (ov == v && oi < ix)) {
                            v = ov;
                            ix = oi;
                        }
                    }
                for (int r = 0; r < kSeedCluster; r++) {   // all-gather of (value, index) of this block
                    *cluster.map_shared_rank(&s_gf[gbuf][rank][side], r) = v;
                    *cluster.map_shared_rank(&s_gi[gbuf][rank][side], r) = ix;
                }
            }
            cluster.sync();
            if (tid < 2) {
                const int side = tid;
                if (on[side] && round < k[side]) {
                    float v = -INFINITY;
                    int ix = 0x7fffffff;
                    for (int r = 0; r < kSeedCluster; r++) {
                        const float ov = s_gf[gbuf][r][side];
                        const int oi = s_gi[gbuf][r][side];
                        if (ov > v || (ov == v && oi < ix)) {
                            v = ov;
                            ix = oi;
                        }
                    }
                    if (v > -INFINITY && ix < HW) {
                        s_sel[side][round] = ix;
                        if (ix >= lo && ix < hi) (side ? key_bg : key_fg)[ix - lo] = __float_as_uint(-INFINITY);
                    }
                }
            }
            gbuf ^= 1;
            __syncthreads();
        }
    }
    // ---- outputs: the selected pixels, and the label map of this block's slice
    if (rank == 0)
        for (int i = tid; i < 2 * p.kmax; i += kSeedFusedThreads) {
            const int side = i / p.kmax, j = i - side * p.kmax;
            p.sel[((size_t)b * 2 + side) * p.kmax + j] = j < kSeedFusedMaxK ? s_sel[side][j] : -1;
        }
    if (p.labels) {
        // kornia 0.6.4 dilation with a flat ksz x ksz kernel (see seed_labels_kernel).  The windows of the seeds are
        // worked out once per block (rows / columns a seed reaches); a pixel then only compares.
        __shared__ short s_win[2][kSeedFusedMaxK][4];   // y0, y1, x0, x1 (inclusive); y0 > y1: unused
        const int origin = p.ksz / 2, back = p.ksz - 1 - origin;
        const int kk = min(p.kmax, kSeedFusedMaxK);
        for (int i = tid; i < 2 * kSeedFusedMaxK; i += kSeedFusedThreads) {
            const int c = i / kSeedFusedMaxK, j = i - c * kSeedFusedMaxK;
            const int sp = j < kk ? s_sel[c][j] : -1;
            const int sy = sp >= 0 ? sp / p.W : 0, sx = sp >= 0 ? sp - sy * p.W : 0;
            s_win[c][j][0] = (short)(sp >= 0 ? max(sy - back, -1) : 1);
            s_win[c][j][1] = (short)(sp >= 0 ? min(sy + origin, 32766) : 0);
            s_win[c][j][2] = (short)max(sx - back, -1);
            s_win[c][j][3] = (short)min(sx + origin, 32766);
        }
        __syncthreads();
        // rows of the frame any window reaches: outside them (nearly everywhere) a pixel is ignore without a look
        int ymin = 0x7fffffff, ymax = -1;
        for (int c = 0; c < 2; c++)
            for (int j = 0; j < kk; j++)
                if (s_win[c][j][0] <= s_win[c][j][1]) {
                    ymin = min(ymin, (int)s_win[c][j][0]);
                    ymax = max(ymax, (int)s_win[c][j][1]);
                }
        long long *out = p.labels + (size_t)b * HW;
        int y = (lo + tid) / p.W, x = (lo + tid) - y * p.W;
        const int dy = kSeedFusedThreads / p.W, dx = kSeedFusedThreads - dy * p.W;   // one division per thread, not per pixel
        for (int i = lo + tid; i < hi; i += kSeedFusedThreads) {
            bool near[2] = {false, false};
            if (y >= ymin && y <= ymax) {
#pragma unroll
                for (int c = 0; c < 2; c++)
                    for (int j = 0; j < kk; j++) {
                        if (s_win[c][j][0] > s_win[c][j][1]) break;   // seeds are filled from slot 0 on
                        if (y >= s_win[c][j][0] && y <= s_win[c][j][1] && x >= s_win[c][j][2] && x <= s_win[c][j][3])
                            near[c] = true;
                    }
            }
            long long label = p.ignore_idx;
            if (near[0] != near[1]) label = near[0] ? 1 : 0;   // claimed by both -> neither (tcam_seeding.py:247-250)
            out[i] = label;
            y += dy;
            x += dx;
            if (x >= p.W) {
                x -= p.W;
                y++;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Cross-entropy on the seeds WITHOUT the label map (SelfLearningTcams, dlib/losses/tcam.py:48-77:
// CrossEntropyLoss(ignore_index)(fcams, seeds), reduction 'mean' over the labelled pixels).
//
// The label map TCAMSeeder hands to the loss is ignore everywhere except the ksz x ksz windows around the
// 2 x k selected seeds: 18 labelled pixels of 50 176 with the README recipe.  torch's cross-entropy still runs
// log-softmax, NLL and both backward passes over the whole [B,K,H,W] tensor (12.8 MB at K = 2: 0.076 ms of a 0.41 ms
// step).  Here the labelled pixels are enumerated from the selected seeds themselves: work item = (sample, side, seed,
// window offset); a pixel counts once per side (the first seed whose window covers it) and is dropped when both
// sides cover it -- exactly seed_labels_kernel's rule (tcam_seeding.py:239-254).  Same value and gradient as torch's
// call on the label map; the sums run in a fixed order (one block per sample, ticketed final fold): deterministic.
struct SeedCeParams {
    const float *logits;   // [B][K][HW]
    const int *sel;        // [B][2][kmax]
    float *partial;        // [B][2]: loss sum, labelled pixels of the sample
    int *ticket;           // [1], zero before the first call; left at zero
    float *loss_out;       // [1]: mean over the labelled pixels of the batch (NaN when there is none, like torch)
    float *count_out;      // [1]: labelled pixels of the batch
    const float *add;      // optional [1]: another loss term (the CRF's), already on the stream
    float *total_out;      // optional [1]: add + weight * loss
    float weight;
    int B, K, H, W, kmax, ksz;
};

// label of window pixel `off` of seed j on `side`, or -1 when the item does not count (outside the frame, an earlier
// seed of the side already covers the pixel, or the other side covers it too); `pix` receives the pixel index
__device__ __forceinline__ int seed_window_label(const int *sel_b, int kmax, int ksz, int H, int W, int side, int j,
                                                 int off, int &pix)
{
    const int origin = ksz / 2, back = ksz - 1 - origin;
    const int sp = sel_b[side * kmax + j];
    if (sp < 0) return -1;
    const int sy = sp / W, sx = sp - sy * W;
    const int y = sy - back + off / ksz, x = sx - back + off % ksz;   // a seed at sy reaches [sy - back, sy + origin]
    if (y < 0 || y >= H || x < 0 || x >= W) return -1;
    pix = y * W + x;
    auto covers = [&](int sd, int jj) {
        const int q = sel_b[sd * kmax + jj];
        if (q < 0) return false;
        const int qy = q / W, qx = q - qy * W;
        return y >= qy - back && y <= qy + origin && x >= qx - back && x <= qx + origin;
    };
    for (int jj = 0; jj < j; jj++)
        if (covers(side, jj)) return -1;          // counted with the earlier seed
    for (int jj = 0; jj < kmax; jj++)
        if (covers(1 - side, jj)) return -1;      // claimed by both sides -> ignore
    return side == 0 ? 1 : 0;                     // side 0 = foreground seeds -> class 1
}

__global__ void __launch_bounds__(256) seed_ce_forward_kernel(const SeedCeParams p)
{
    __shared__ float s_l[8];
    __shared__ int s_c[8];
    __shared__ bool s_last;
    const int b = blockIdx.x;
    const int HW = p.H * p.W;
    const int *sel_b = p.sel + (size_t)b * 2 * p.kmax;
    const float *z = p.logits + (size_t)b * p.K * HW;
    const int win = p.ksz * p.ksz, items = 2 * p.kmax * win;
    float lsum = 0.f;
    int cnt = 0;
    for (int it = threadIdx.x; it < items; it += 256) {
        const int side = it / (p.kmax * win), rest = it - side * p.kmax * win;
        int pix;
        const int label = seed_window_label(sel_b, p.kmax, p.ksz, p.H, p.W, side, rest / win, rest % win, pix);
        if (label < 0) continue;
        float zmax = -INFINITY;
        for (int k = 0; k < p.K; k++) zmax = fmaxf(zmax, __ldg(z + (size_t)k * HW + pix));
        float sum = 0.f;
        for (int k = 0; k < p.K; k++) sum += expf(__ldg(z + (size_t)k * HW + pix) - zmax);
        lsum += (logf(sum) + zmax) - __ldg(z + (size_t)label * HW + pix);   // -log_softmax(z)[label]
        cnt++;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_l[threadIdx.x >> 5] = lsum;
        s_c[threadIdx.x >> 5] = cnt;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) {
            lsum += s_l[w];
            cnt += s_c[w];
        }
        p.partial[b * 2 + 0] = lsum;
        p.partial[b * 2 + 1] = (float)cnt;
        __threadfence();
        s_last = atomicAdd(p.ticket, 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    float total = 0.f, n = 0.f;
    for (int i = 0; i < p.B; i++) {   // fixed order
        total += __ldcg(p.partial + i * 2);
        n += __ldcg(p.partial + i * 2 + 1);
    }
    const float ce = __fdiv_rn(total, n);   // 0 / 0 = NaN: torch's mean over no element
    p.loss_out[0] = ce;
    p.count_out[0] = n;
    if (p.total_out) p.total_out[0] = __fadd_rn(p.add ? p.add[0] : 0.f, __fmul_rn(ce, p.weight));
    *p.ticket = 0;
}

// grad[b][k][pix] += (g * scale) * (softmax_k - [k == label]) / count   on the labelled pixels (every labelled pixel
// belongs to exactly one work item: plain read-modify-write)
__global__ void __launch_bounds__(256) seed_ce_backward_kernel(const float *__restrict__ logits,
                                                               const int *__restrict__ sel, float *grad,
                                                               const float *__restrict__ count,
                                                               const float *__restrict__ grad_out, float scale, int K,
                                                               int H, int W, int kmax, int ksz)
{
    const int b = blockIdx.x;
    const int HW = H * W;
    const int *sel_b = sel + (size_t)b * 2 * kmax;
    const float *z = logits + (size_t)b * K * HW;
    float *g = grad + (size_t)b * K * HW;
    const float coef = __fdiv_rn(__fmul_rn(__ldg(grad_out), scale), __ldg(count));
    const int win = ksz * ksz, items = 2 * kmax * win;
    for (int it = threadIdx.x; it < items; it += 256) {
        const int side = it / (kmax * win), rest = it - side * kmax * win;
        int pix;
        const int label = seed_window_label(sel_b, kmax, ksz, H, W, side, rest / win, rest % win, pix);
        if (label < 0) continue;
        float zmax = -INFINITY;
        for (int k = 0; k < K; k++) zmax = fmaxf(zmax, __ldg(z + (size_t)k * HW + pix));
        float sum = 0.f;
        for (int k = 0; k < K; k++) sum += expf(__ldg(z + (size_t)k * HW + pix) - zmax);
        for (int k = 0; k < K; k++) {
            const float pk = __fdiv_rn(expf(__ldg(z + (size_t)k * HW + pix) - zmax), sum);
            g[(size_t)k * HW + pix] += coef * (pk - (k == label ? 1.f : 0.f));
        }
    }
}

// out[b][y][x] = 1 if a fg seed dilates onto the pixel, 0 if a bg seed does, ignore if none or both
__global__ void __launch_bounds__(256) seed_labels_kernel(const int *__restrict__ sel, int kmax, int B, int H, int W,
                                                          int ksz, long long ignore_idx, long long *__restrict__ out)
{
    // kornia 0.6.4 dilation with a flat ksz x ksz kernel: out[y] = max_{d in [0,ksz)} in[y + d - origin],
    // origin = ksz / 2  =>  a seed at sy reaches y in [sy - (ksz-1-origin), sy + origin]
    const int origin = ksz / 2;
    const int back = ksz - 1 - origin;
    const long long total = (long long)B * H * W;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int b = (int)(i / ((long long)H * W));
        const int px = (int)(i - (long long)b * H * W);
        const int y = px / W, x = px - y * W;
        bool near[2] = {false, false};
#pragma unroll
        for (int c = 0; c < 2; c++) {
            const int *s = sel + ((size_t)b * 2 + c) * kmax;
            for (int j = 0; j < kmax; j++) {
                const int sp = __ldg(s + j);
                if (sp < 0) break;
                const int sy = sp / W, sx = sp - sy * W;
                if (y >= sy - back && y <= sy + origin && x >= sx - back && x <= sx + origin) near[c] = true;
            }
        }
        long long label = ignore_idx;
        if (near[0] != near[1]) label = near[0] ? 1 : 0;   // claimed by both -> neither (tcam_seeding.py:247-250)
        out[i] = label;
    }
}

// ROI of a CAM by Otsu's threshold, one thread block per sample.  Restates, on the GPU,
//   GetRoiSingleCam.get_thresh + __call__ with roi_method == 'roi_all' (dlib/cams/tcam_seeding.py:337-345,419-430):
//     cam_ = floor(cam * 255.);  th = 0 if flat else skimage.filters.threshold_otsu(cam_);  roi = cam*255. >= th
//   skimage 0.17.2 threshold_otsu (third-party, requirements.txt:83): 256-bin np.histogram over [min, max],
//     bin centres, between-class variance in float64, threshold = centre of the arg-max bin.
// np.histogram's float32 arithmetic is reproduced step by step: edges[i] = fl(fl(i*step) + first) (np.linspace),
// index = trunc(((v - first) / (last - first)) * 256) with the +-1 corrections against the edges.
__global__ void __launch_bounds__(kSeedThreads) otsu_roi_kernel(const float *__restrict__ cams,
                                                                long long *__restrict__ roi,
                                                                float *__restrict__ thresh_out, int HW)
{
    __shared__ float s_edge[257];
    __shared__ int s_hist[256];
    __shared__ float s_red[2][32];
    __shared__ float s_th;
    const int b = blockIdx.x, tid = threadIdx.x;
    const float *cam = cams + (size_t)b * HW;

    float lo = INFINITY, hi = -INFINITY;
    for (int i = tid; i < HW; i += kSeedThreads) {
        const float v = floorf(__fmul_rn(__ldg(cam + i), 255.0f));
        lo = fminf(lo, v);
        hi = fmaxf(hi, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((tid & 31) == 0) {
        s_red[0][tid >> 5] = lo;
        s_red[1][tid >> 5] = hi;
    }
    __syncthreads();
    lo = s_red[0][0];
    hi = s_red[1][0];
    for (int w = 1; w < kSeedThreads / 32; w++) {
        lo = fminf(lo, s_red[0][w]);
        hi = fmaxf(hi, s_red[1][w]);
    }
    const bool flat = !(lo < hi);
    if (!flat) {
        const float step = __fdiv_rn(__fsub_rn(hi, lo), 256.0f);
        for (int i = tid; i < 257; i += kSeedThreads)
            s_edge[i] = i == 256 ? hi : __fadd_rn(__fmul_rn((float)i, step), lo);
        for (int i = tid; i < 256; i += kSeedThreads) s_hist[i] = 0;
        __syncthreads();
        const float denom = __fsub_rn(hi, lo);
        for (int i = tid; i < HW; i += kSeedThreads) {
            const float v = floorf(__fmul_rn(__ldg(cam + i), 255.0f));
            int idx = (int)__fmul_rn(__fdiv_rn(__fsub_rn(v, lo), denom), 256.0f);
            if (idx == 256) idx = 255;
            if (v < s_edge[idx]) idx -= 1;
            if (v >= s_edge[idx + 1] && idx != 255) idx += 1;
            atomicAdd(&s_hist[idx], 1);
        }
        __syncthreads();
        if (tid == 0) {
            // sequential float64 cumulative sums, like np.cumsum
            double w2_after[257], m2_after[257];   // suffix sums from bin i on
            double run_w = 0.0, run_m = 0.0;
            w2_after[256] = 0.0;
            m2_after[256] = 0.0;
            for (int i = 255; i >= 0; i--) {
                const float centre = __fdiv_rn(__fadd_rn(s_edge[i], s_edge[i + 1]), 2.0f);
                run_w += (double)s_hist[i];
                run_m += (double)s_hist[i] * (double)centre;
                w2_after[i] = run_w;
                m2_after[i] = run_m / run_w;          // mean2[i]
            }
            double w1 = 0.0, m1 = 0.0, best = -1.0;
            int best_i = 0;
            for (int i = 0; i < 255; i++) {
                const float centre = __fdiv_rn(__fadd_rn(s_edge[i], s_edge[i + 1]), 2.0f);
                w1 += (double)s_hist[i];
                m1 += (double)s_hist[i] * (double)centre;
                const double mean1 = m1 / w1;
                const double d = mean1 - m2_after[i + 1];
                const double var = (w1 * w2_after[i + 1]) * (d * d);
                if (var > best) {                     // np.argmax: first maximum
                    best = var;
                    best_i = i;
                }
            }
            s_th = __fdiv_rn(__fadd_rn(s_edge[best_i], s_edge[best_i + 1]), 2.0f);
        }
    } else if (tid == 0) {
        s_th = 0.0f;
    }
    __syncthreads();
    const float th = s_th;
    if (tid == 0 && thresh_out) thresh_out[b] = th;
    long long *out = roi + (size_t)b * HW;
    for (int i = tid; i < HW; i += kSeedThreads) out[i] = __fmul_rn(__ldg(cam + i), 255.0f) >= th ? 1 : 0;
}


// ---------------------------------------------------------------------------------------------------------
// ROI by connected components: GetRoiSingleCam.__call__ with roi_method 'roi_high_density' / 'roi_largest'
// (dlib/cams/tcam_seeding.py:347-412).  The reference runs on the CPU per sample:
//   blobs = cam*255 >= thresh;  skimage.measure.label(blobs, connectivity=1)   (4-connected components)
//   per component: area, density = sum(cam over the component) / area          (float64)
//   high density: the densest component, unless its area < p_min_area*H*W -> the largest one;  largest: the largest
//   final_roi = that component;  bbox = cv2.boundingRect of its (single) external contour, x1/y1 clamped
//   (dlib/utils/wsol.py:133-137);  bbox_mask[y0:y1, x0:x1] = 1
// Here: one thread block per sample.  Components by union-find on the pixel grid (label = smallest pixel index of
// the component, merged with atomicMin like ECL-CC), so "first label" ties resolve like skimage's raster-order
// numbering; areas with integer atomics, sums with float64 atomics (the order of the additions is not the
// reference's pairwise one: densities agree to ~1e-15 relative; exact ties go to the first component).
// scratch: labels int[B*HW], area int[B*HW], sum double[B*HW].
__device__ __forceinline__ int cc_find(const int *label, int x)
{
    int p = label[x];
    while (p != x) {
        x = p;
        p = label[x];
    }
    return x;
}

__device__ __forceinline__ void cc_union(int *label, int a, int b)
{
    while (true) {
        a = cc_find(label, a);
        b = cc_find(label, b);
        if (a == b) return;
        if (a < b) {
            const int t = a;
            a = b;
            b = t;
        }
        // hang the larger root under the smaller one; if somebody re-rooted `a` meanwhile, retry from there
        const int old = atomicMin(label + a, b);
        if (old == a) return;
        a = old;
    }
}

struct RoiBest {
    double key;   // density or area
    int idx;      // root pixel index; smaller wins ties
};
__device__ __forceinline__ RoiBest roi_better(RoiBest x, RoiBest y)
{
    if (y.idx < 0) return x;
    if (x.idx < 0) return y;
    if (y.key > x.key || (y.key == x.key && y.idx < x.idx)) return y;
    return x;
}

__global__ void __launch_bounds__(kSeedThreads) roi_components_kernel(const float *__restrict__ cams,
                                                                      const float *__restrict__ thresh,
                                                                      long long *__restrict__ roi,
                                                                      float *__restrict__ bbox_mask,
                                                                      int *__restrict__ bbox, int *labels, int *area,
                                                                      double *sum, int H, int W, int largest_only,
                                                                      double min_area)
{
    __shared__ RoiBest s_best[2][kSeedThreads / 32];
    __shared__ int s_sel;
    __shared__ int s_box[4][kSeedThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int HW = H * W;
    const float *cam = cams + (size_t)b * HW;
    int *lab = labels + (size_t)b * HW;
    int *ar = area + (size_t)b * HW;
    double *sm = sum + (size_t)b * HW;
    const float th = thresh[b];

    for (int i = tid; i < HW; i += kSeedThreads) {
        lab[i] = __fmul_rn(cam[i], 255.0f) >= th ? i : -1;
        ar[i] = 0;
        sm[i] = 0.0;
    }
    __syncthreads();
    // 4-connectivity: merge with the left and the upper neighbour
    for (int i = tid; i < HW; i += kSeedThreads) {
        if (lab[i] < 0) continue;
        const int y = i / W, x = i - y * W;
        if (x > 0 && lab[i - 1] >= 0) cc_union(lab, i, i - 1);
        if (y > 0 && lab[i - W] >= 0) cc_union(lab, i, i - W);
    }
    __syncthreads();
    // flatten + per-component statistics
    for (int i = tid; i < HW; i += kSeedThreads) {
        if (lab[i] < 0) continue;
        const int r = cc_find(lab, i);
        lab[i] = r;   // only shortens paths: concurrent finds stay correct
        atomicAdd(ar + r, 1);
        atomicAdd(sm + r, (double)cam[i]);
    }
    __syncthreads();
    // best component by density and by area (ties: first in raster order)
    RoiBest dens = {0.0, -1}, big = {0.0, -1};
    for (int i = tid; i < HW; i += kSeedThreads) {
        if (lab[i] != i) continue;
        const double a = (double)ar[i];
        dens = roi_better(dens, RoiBest{sm[i] / a, i});
        big = roi_better(big, RoiBest{a, i});
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        RoiBest od, ob;
        od.key = __shfl_xor_sync(0xffffffffu, dens.key, o);
        od.idx = __shfl_xor_sync(0xffffffffu, dens.idx, o);
        ob.key = __shfl_xor_sync(0xffffffffu, big.key, o);
        ob.idx = __shfl_xor_sync(0xffffffffu, big.idx, o);
        dens = roi_better(dens, od);
        big = roi_better(big, ob);
    }
    if ((tid & 31) == 0) {
        s_best[0][tid >> 5] = dens;
        s_best[1][tid >> 5] = big;
    }
    __syncthreads();
    if (tid == 0) {
        dens = s_best[0][0];
        big = s_best[1][0];
        for (int w = 1; w < kSeedThreads / 32; w++) {
            dens = roi_better(dens, s_best[0][w]);
            big = roi_better(big, s_best[1][w]);
        }
        int sel = largest_only ? big.idx : dens.idx;
        // tcam_seeding.py:381-384: a dense but tiny component gives way to the largest one
        if (!largest_only && sel >= 0 && (double)ar[sel] < min_area) sel = big.idx;
        s_sel = sel;
    }
    __syncthreads();
    const int sel = s_sel;
    int x0 = W, y0 = H, x1 = -1, y1 = -1;
    long long *out = roi + (size_t)b * HW;
    for (int i = tid; i < HW; i += kSeedThreads) {
        const bool in = sel >= 0 && lab[i] == sel;
        out[i] = in ? 1 : 0;
        if (in) {
            const int y = i / W, x = i - y * W;
            x0 = min(x0, x);
            y0 = min(y0, y);
            x1 = max(x1, x);
            y1 = max(y1, y);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        x0 = min(x0, __shfl_xor_sync(0xffffffffu, x0, o));
        y0 = min(y0, __shfl_xor_sync(0xffffffffu, y0, o));
        x1 = max(x1, __shfl_xor_sync(0xffffffffu, x1, o));
        y1 = max(y1, __shfl_xor_sync(0xffffffffu, y1, o));
    }
    if ((tid & 31) == 0) {
        s_box[0][tid >> 5] = x0;
        s_box[1][tid >> 5] = y0;
        s_box[2][tid >> 5] = x1;
        s_box[3][tid >> 5] = y1;
    }
    __syncthreads();
    x0 = s_box[0][0];
    y0 = s_box[1][0];
    x1 = s_box[2][0];
    y1 = s_box[3][0];
    for (int w = 1; w < kSeedThreads / 32; w++) {
        x0 = min(x0, s_box[0][w]);
        y0 = min(y0, s_box[1][w]);
        x1 = max(x1, s_box[2][w]);
        y1 = max(y1, s_box[3][w]);
    }
    int bx0 = 0, by0 = 0, bx1 = 0, by1 = 0;   // no contour: [[0, 0, 0, 0]] (wsol.py:125-126)
    if (x1 >= 0) {
        // cv2.boundingRect: (x, y, w, h) = (min, min, max-min+1, max-min+1); x1 = min(x + w, W - 1) (wsol.py:133-136)
        bx0 = x0;
        by0 = y0;
        bx1 = min(x1 + 1, W - 1);
        by1 = min(y1 + 1, H - 1);
    }
    if (tid == 0) {
        bbox[b * 4 + 0] = bx0;
        bbox[b * 4 + 1] = by0;
        bbox[b * 4 + 2] = bx1;
        bbox[b * 4 + 3] = by1;
    }
    float *mask = bbox_mask + (size_t)b * HW;
    for (int i = tid; i < HW; i += kSeedThreads) {
        const int y = i / W, x = i - y * W;
        mask[i] = (x >= bx0 && x < bx1 && y >= by0 && y < by1) ? 1.0f : 0.0f;   // bbox_mask[y0:y1, x0:x1] = 1
    }
}

// torch.nan_to_num(x, nan=0.0, posinf=1.0, neginf=0.0)  (wsol_loader.py:634, train_wsol.py:426,431)
__device__ __forceinline__ float nan_to_num01(float v)
{
    if (v != v) return 0.0f;
    if (v == INFINITY) return 1.0f;
    if (v == -INFINITY) return 0.0f;
    return v;
}

// Temporal max with the loader's optional re-normalisation of every frame's CAM first
// (dlib/datasets/wsol_loader.py:591-600 + re_normalize_cam :630-635):
//   e = exp((cam + 1e-6) * h);  e = e / e.max();  e = nan_to_num(e, 0, 1, 0);  out = maximum(out, e)
// One thread block per sample; cams [B,T,HW], out [B,HW].  e.max() is torch's NaN-propagating max over the frame.
__global__ void __launch_bounds__(kSeedThreads) temporal_max_renorm_kernel(const float *__restrict__ cams,
                                                                           float *__restrict__ out, int T, int HW,
                                                                           float h)
{
    __shared__ float s_red[kSeedThreads / 32];
    __shared__ int s_nan[kSeedThreads / 32];
    __shared__ float s_max;
    __shared__ int s_anynan;
    const int b = blockIdx.x;
    const float *src = cams + (size_t)b * T * HW;
    float *dst = out + (size_t)b * HW;
    for (int t = 0; t < T; t++) {
        const float *frame = src + (size_t)t * HW;
        float m = -INFINITY;
        int nan = 0;
        for (int i = threadIdx.x; i < HW; i += kSeedThreads) {
            const float e = expf(__fmul_rn(__fadd_rn(frame[i], 1e-6f), h));
            nan |= (e != e);
            m = fmaxf(m, e);   // NaN handled through the flag
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
            nan |= __shfl_xor_sync(0xffffffffu, nan, o);
        }
        if ((threadIdx.x & 31) == 0) {
            s_red[threadIdx.x >> 5] = m;
            s_nan[threadIdx.x >> 5] = nan;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            float mm = -INFINITY;
            int nn = 0;
            for (int w = 0; w < kSeedThreads / 32; w++) {
                mm = fmaxf(mm, s_red[w]);
                nn |= s_nan[w];
            }
            s_max = mm;
            s_anynan = nn;
        }
        __syncthreads();
        const float emax = s_anynan ? __int_as_float(0x7fc00000) : s_max;
        for (int i = threadIdx.x; i < HW; i += kSeedThreads) {
            const float e = expf(__fmul_rn(__fadd_rn(frame[i], 1e-6f), h));
            const float v = nan_to_num01(__fdiv_rn(e, emax));
            if (t == 0) {
                dst[i] = v;
            } else {
                const float cur = dst[i];
                dst[i] = (cur != cur) ? cur : ((v != v) ? v : (v > cur ? v : cur));
            }
        }
        __syncthreads();
    }
}

// Trainer.prepare_std_cams_disq (dlib/learning/train_wsol.py:417-432) in one pass:
//   nan_to_num -> F.interpolate(size, mode='bilinear', align_corners=False) -> nan_to_num
// in [B,h,w] -> out [B,H,W].  Source index and weights as in ATen's upsample_bilinear2d (area_pixel_compute_source_index
// with align_corners=False: src = scale * (dst + 0.5) - 0.5 clamped at 0, scale = in / out).
__global__ void __launch_bounds__(256) prepare_std_cams_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                               int h, int w, int H, int W, float scale_h,
                                                               float scale_w, long long total)
{
    const long long stride = (long long)gridDim.x * 256;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += stride) {
        const int x = (int)(i % W);
        const long long r = i / W;
        const int y = (int)(r % H);
        const long long b = r / H;
        float sy = scale_h * ((float)y + 0.5f) - 0.5f;
        float sx = scale_w * ((float)x + 0.5f) - 0.5f;
        sy = sy < 0.f ? 0.f : sy;
        sx = sx < 0.f ? 0.f : sx;
        const int y0 = min((int)sy, h - 1), x0 = min((int)sx, w - 1);
        const int yp = y0 < h - 1 ? 1 : 0, xp = x0 < w - 1 ? 1 : 0;
        const float ly1 = sy - (float)y0, ly0 = 1.f - ly1;
        const float lx1 = sx - (float)x0, lx0 = 1.f - lx1;
        const float *p = in + (size_t)b * h * w + (size_t)y0 * w + x0;
        const float v00 = nan_to_num01(__ldg(p)), v01 = nan_to_num01(__ldg(p + xp));
        const float v10 = nan_to_num01(__ldg(p + (size_t)yp * w)), v11 = nan_to_num01(__ldg(p + (size_t)yp * w + xp));
        const float v = ly0 * (lx0 * v00 + lx1 * v01) + ly1 * (lx0 * v10 + lx1 * v11);
        out[i] = nan_to_num01(v);
    }
}

}  // namespace tcamcrf
