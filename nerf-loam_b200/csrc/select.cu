// Per-iteration ray selection on the device: N distinct points of a scan, uniformly at random, in the scan's point order --
// the distribution of LidarFrame.sample_rays / sampling_without_replacement (src/lidarFrame.py:55-57, src/utils/sample_util.py:4-19:
// Gumbel top-k over constant weights = a uniform N-subset, returned as a mask, i.e. in point order) -- plus the gather of the
// selected rays' direction / range / cosine, as ONE launch.
//
// The torch formulation of the same thing (rand -> top-k of 131 072 keys -> sort -> three gathers) is ~10 kernels and 140-160 us,
// a third of a 2048-ray tracking iteration whose other 20 kernels take 270 us.  Here one 8-CTA cluster per frame gives every point an
// independent 32-bit key from a counter-based generator (seed, frame, point index) and selects the N smallest keys with a
// three-pass radix select (11 + 11 + 10 bits, histograms in shared memory, summed across the cluster through DSMEM): that is exactly "top-k of iid keys", i.e. a uniform
// N-subset, it is deterministic for a given seed (ties between equal keys go to the lower point index), and the last pass walks
// the points in order, so the output is in point order without a sort.  A thread hashes its (strided) points once and keeps the keys in registers for the three
// histogram passes; the ordered emission re-hashes the thread's contiguous run.  Nothing but the histograms is stored.
#include "nl_cuda.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace {

__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ uint32_t point_key(uint32_t seed, uint32_t i) { return mix32(seed ^ mix32(i * 0x9E3779B1u + 0x7F4A7C15u)); }

constexpr int SEL_THREADS = 1024;
constexpr int SEL_BINS = 2048;
constexpr int SEL_CLUSTER = 8;     // CTAs per scan: each hashes an eighth of the points, histograms are summed over distributed shared memory
constexpr int SEL_KEYS = 16;        // keys a thread keeps in registers between the passes (covers scans of up to 8 x 1024 x 16 = 131 072 points)

// Among this scan's keys that pass `match`, find the bin (of `digit`) in which the `want`-th smallest key (1-based) lies, and the
// number of matching keys in lower bins.  Every CTA of the cluster histograms its own points [p0, p1), reads the other CTAs'
// histograms through DSMEM and finds the bin redundantly.  hist: SEL_BINS ints of shared memory (same offset in every CTA).
template <class Match, class Digit>
__device__ void find_bin(cg::cluster_group &cluster, int p0, int p1, uint32_t seed, const uint32_t (&keys)[SEL_KEYS], bool cached, int want, Match match,
                         Digit digit, int *hist, int *s_scan, int &bin, int &below) {
    const int t = threadIdx.x;
    for (int i = t; i < SEL_BINS; i += SEL_THREADS) hist[i] = 0;
    __syncthreads();
    if (cached) {
#pragma unroll
        for (int j = 0; j < SEL_KEYS; ++j)
            if (p0 + t + j * SEL_THREADS < p1 && match(keys[j])) atomicAdd(&hist[digit(keys[j])], 1);
    } else {
        for (int i = p0 + t; i < p1; i += SEL_THREADS) {
            const uint32_t k = point_key(seed, (uint32_t)i);
            if (match(k)) atomicAdd(&hist[digit(k)], 1);
        }
    }
    cluster.sync();
    int a = 0, b = 0;
#pragma unroll
    for (int q = 0; q < SEL_CLUSTER; ++q) {
        const int2 h = *reinterpret_cast<const int2 *>(cluster.map_shared_rank(hist, q) + 2 * t);
        a += h.x; b += h.y;
    }
    // inclusive scan over the 2048 bins: 2 per thread + block scan of the pair sums
    int incl = a + b;
    const int lane = t & 31, w = t >> 5;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += y;
    }
    if (lane == 31) s_scan[w] = incl;
    __syncthreads();
    int pre = 0;
    for (int q = 0; q < w; ++q) pre += s_scan[q];
    const int upto_a = pre + incl - b, upto_b = pre + incl;        // keys in bins <= 2t and <= 2t+1
    const int before = upto_a - a;                                 // keys in bins < 2t
    if (before < want && want <= upto_a) { s_scan[32] = 2 * t; s_scan[33] = before; }
    else if (upto_a < want && want <= upto_b) { s_scan[32] = 2 * t + 1; s_scan[33] = upto_a; }
    __syncthreads();
    bin = s_scan[32];
    below = s_scan[33];
    __syncthreads();                                               // s_scan is reused by the next pass
    // (no cluster barrier here: every pass has its own histogram, so a CTA may start the next pass while a peer still reads this one)
}

__global__ void __launch_bounds__(SEL_THREADS)
    k_select_rays(int cap, int n_select, const int64_t *__restrict__ n_points, const uint32_t *__restrict__ seed_dev, uint32_t seed_host,
                  const float *__restrict__ dirs_all, const float *__restrict__ gt_all, const float *__restrict__ cos_all, float *__restrict__ dirs,
                  float *__restrict__ gt, float *__restrict__ cosv, int32_t *__restrict__ idx_out) {
    __shared__ __align__(8) int hist[3][SEL_BINS];          // one histogram per pass: no barrier needed before re-use
    __shared__ int s_scan[36];
    __shared__ unsigned long long s_w[SEL_THREADS / 32];
    __shared__ unsigned long long s_total;
    cg::cluster_group cluster = cg::this_cluster();
    const int f = blockIdx.x / SEL_CLUSTER, c = (int)cluster.block_rank(), t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int n = (int)min((long long)n_points[f], (long long)cap);
    const int N = min(n_select, n);
    uint32_t seed = seed_dev ? *seed_dev : seed_host;
    seed = mix32(seed ^ 0x9E3779B9u * (uint32_t)(f + 1));
    // this CTA's contiguous share of the scan, and inside it every thread's contiguous run (for the ordered emission)
    const int share = (n + SEL_CLUSTER - 1) / SEL_CLUSTER;
    const int c0 = min(c * share, n), c1 = min(c0 + share, n);
    // threshold key T = the N-th smallest key; `ties` = how many of the keys equal to T belong to the N smallest
    uint32_t T = 0xffffffffu;
    int ties = 0;
    // the three histogram passes look at the same keys: hash them once (strided over the CTA's share), keep them in registers
    uint32_t keys[SEL_KEYS];
    const bool cached = (c1 - c0) <= SEL_KEYS * SEL_THREADS;
    if (cached && N < n && N > 0) {
#pragma unroll
        for (int j = 0; j < SEL_KEYS; ++j) {
            const int i = c0 + t + j * SEL_THREADS;
            keys[j] = i < c1 ? point_key(seed, (uint32_t)i) : 0u;
        }
    }
    if (N < n && N > 0) {
        int bA, bB, bC, below;
        find_bin(cluster, c0, c1, seed, keys, cached, N, [](uint32_t) { return true; }, [](uint32_t k) { return (int)(k >> 21); }, hist[0], s_scan, bA, below);
        int want = N - below;
        find_bin(cluster, c0, c1, seed, keys, cached, want, [bA](uint32_t k) { return (int)(k >> 21) == bA; }, [](uint32_t k) { return (int)((k >> 10) & 2047u); }, hist[1],
                 s_scan, bB, below);
        want -= below;
        const uint32_t top22 = ((uint32_t)bA << 11) | (uint32_t)bB;
        find_bin(cluster, c0, c1, seed, keys, cached, want, [top22](uint32_t k) { return (k >> 10) == top22; }, [](uint32_t k) { return (int)(k & 1023u); }, hist[2], s_scan,
                 bC, below);
        T = (top22 << 10) | (uint32_t)bC;
        ties = want - below;
    }
    const int per = (c1 - c0 + SEL_THREADS - 1) / SEL_THREADS;
    const int p0 = min(c0 + t * per, c1), p1 = min(p0 + per, c1);
    int lt = 0, eq = 0;
    for (int i = p0; i < p1; ++i) {
        const uint32_t k = point_key(seed, (uint32_t)i);
        lt += (N == n) || (k < T);
        eq += (N < n) && (k == T);
    }
    // two exclusive scans (below-threshold counts and tie counts) packed into one 64-bit scan: over the block, then over the cluster
    const unsigned long long pk = ((unsigned long long)(unsigned)eq << 32) | (unsigned)lt;
    unsigned long long incl = pk;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += y;
    }
    if (lane == 31) s_w[w] = incl;
    __syncthreads();
    unsigned long long pre = 0;
    for (int q = 0; q < w; ++q) pre += s_w[q];
    if (t == SEL_THREADS - 1) s_total = pre + incl;
    cluster.sync();
    for (int q = 0; q < c; ++q) pre += *cluster.map_shared_rank(&s_total, q);
    const unsigned long long excl = pre + incl - pk;
    const int lt_before = (int)(excl & 0xffffffffULL);
    int eq_before = (int)(excl >> 32);
    int slot = lt_before + min(eq_before, ties);                  // selected points in front of this thread's run
    const size_t in0 = (size_t)f * cap, out0 = (size_t)f * n_select;
    for (int i = p0; i < p1; ++i) {
        const uint32_t k = point_key(seed, (uint32_t)i);
        bool take = (N == n) || (k < T);
        if (!take && k == T) take = eq_before++ < ties;           // equal keys: the lower point index wins
        if (!take) continue;
        const size_t o = out0 + (size_t)slot++;
        dirs[o * 3] = dirs_all[(in0 + i) * 3]; dirs[o * 3 + 1] = dirs_all[(in0 + i) * 3 + 1]; dirs[o * 3 + 2] = dirs_all[(in0 + i) * 3 + 2];
        gt[o] = gt_all[in0 + i];
        cosv[o] = cos_all[in0 + i];
        if (idx_out) idx_out[o] = i;
    }
    cluster.sync();                                                // nobody leaves while its totals may still be read
}

}  // namespace

extern "C" int nl_select_rays(int n_frames, int cap, int n_select, const int64_t *d_n_points, const uint32_t *d_seed, uint32_t seed,
                              const float *d_dirs_all, const float *d_gt_all, const float *d_cos_all, float *d_dirs, float *d_gt, float *d_cos,
                              int32_t *d_idx, void *stream) {
    if (n_frames <= 0 || cap <= 0 || n_select <= 0) return nl_set_error("nl_select_rays: sizes must be positive");
    if (!d_n_points || !d_dirs_all || !d_gt_all || !d_cos_all || !d_dirs || !d_gt || !d_cos) return nl_set_error("nl_select_rays: null pointer");
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_frames * SEL_CLUSTER);
    cfg.blockDim = dim3(SEL_THREADS);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = SEL_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, k_select_rays, cap, n_select, d_n_points, d_seed, seed, d_dirs_all, d_gt_all, d_cos_all,
                                             d_dirs, d_gt, d_cos, d_idx);
    if (e != cudaSuccess) return nl_set_error_code(NL_ERR_CUDA, cudaGetErrorString(e));
    NL_CHECK_LAUNCH("nl_select_rays");
    return NL_OK;
}
