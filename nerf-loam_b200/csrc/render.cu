// Fused renderer front end: rays -> sorted/clipped voxel hits -> inverse-CDF samples -> compact
// sample list + loss-mask statistics, with no host synchronisation and no padded [R, S_max] tensors.
//
// Replaces, for the hot path (SURVEY.md section 8 a-2 .. a-5):
//   src/variations/voxel_helpers.py:92-137, 530-567   svo_ray_intersect wrapper + ray_intersect
//   src/variations/voxel_helpers.py:262-344, 570-598  InverseCDFRaySampling wrapper + ray_sample
//   src/variations/render_helpers.py:207-257          hit/sample masking and `ray()` of render_rays
//   src/criterion.py:67-88                            get_masks (the masks depend on depths only)
//
// Kernel chain (all on one stream):
//   k_traverse_sort : 1 thread/ray  DFS + stable sort by min_depth + distance clipping  -> hit planes [20][R]
//   k_scan<HITS>    : 1 block       exclusive scan of hit flags -> rank of every hit ray, R_hit
//   k_sample<false> : 1 thread/hit ray  sampler dry run -> samples per ray, S_max, loss-mask counters
//   k_scan<SAMPLES> : 1 block       exclusive scan of samples per ray -> offsets, M
//   k_sample<true>  : 1 thread/hit ray  sampler again, writes the compact sample list
// The reference keeps every intermediate as a padded dense tensor and syncs the host 6 times to size them.
#include "loss.cuh"
#include "sampler.cuh"
#include "traverse.cuh"

namespace {

struct Workspace {
    int32_t *h_idx;   // [20][R]
    float *h_min;     // [20][R]
    float *h_max;     // [20][R]
    int32_t *nvalid;  // [R]
    int32_t *hitray;  // [R] ray index of the q-th hit ray
    unsigned long long *scan;   // [2][SCAN_SCRATCH]: tile ticket + per-tile (ready << 32 | total) of the two chained scans; zeroed per call
};
constexpr int SCAN_MAX_TILES = 1024;                 // tiles of 4096 elements: up to 4 M rays per call in one wave of look-back
constexpr int SCAN_SCRATCH = SCAN_MAX_TILES + 8;     // words per scan: [0] = ticket counter, [8 + tile] = published tile total

__host__ __device__ inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

inline Workspace carve(void *base, int R) {
    char *p = (char *)base;
    Workspace w;
    w.h_idx = (int32_t *)p; p += align256(sizeof(int32_t) * NL_MAX_HITS * (size_t)R);
    w.h_min = (float *)p; p += align256(sizeof(float) * NL_MAX_HITS * (size_t)R);
    w.h_max = (float *)p; p += align256(sizeof(float) * NL_MAX_HITS * (size_t)R);
    w.nvalid = (int32_t *)p; p += align256(sizeof(int32_t) * (size_t)R);
    w.hitray = (int32_t *)p; p += align256(sizeof(int32_t) * (size_t)R);
    w.scan = (unsigned long long *)p; p += align256(sizeof(unsigned long long) * 2 * SCAN_SCRATCH);
    return w;
}

__device__ __forceinline__ int warp_max(int v) { return __reduce_max_sync(0xffffffffu, v); }

// ------------------------------------------------------------------------------------------------
// k_traverse_sort: svo_intersect + ray_intersect (voxel_helpers.py:530-567) for one ray per thread.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) k_traverse_sort(int R, float voxel_size, float max_distance,
                                                        const float *__restrict__ centres,
                                                        const int32_t *__restrict__ structure,
                                                        const float *__restrict__ ray_o, const float *__restrict__ ray_d,
                                                        Workspace ws, int32_t *__restrict__ ray_nsamp, nl_render_stats *stats) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int nv = 0;
    if (r < R) {
        int32_t idx[NL_MAX_HITS];
        float mn[NL_MAX_HITS], mx[NL_MAX_HITS];
        mn[0] = 0.f;   // never read before the first insertion (the loop guard tests p > 0 first); keeps the compiler quiet
        const NlRay ray = nl_make_ray(ray_o[r * 3], ray_o[r * 3 + 1], ray_o[r * 3 + 2], ray_d[r * 3], ray_d[r * 3 + 1], ray_d[r * 3 + 2]);
        int cnt = 0;
        const int rc = nl_traverse(ray, centres, structure, voxel_size * 0.5f, NL_MAX_HITS, [&](int k, float lo, float hi) {
            // stable insertion by min_depth (ties keep DFS emission order; torch.sort at voxel_helpers.py:546
            // leaves the order of equal keys unspecified)
            int p = cnt;
            while (p > 0 && mn[p - 1] > lo) { idx[p] = idx[p - 1]; mn[p] = mn[p - 1]; mx[p] = mx[p - 1]; --p; }
            idx[p] = k; mn[p] = lo; mx[p] = hi;
            ++cnt;
        });
        if (rc < 0) atomicOr(&stats->error, 4);
        const float two_md = 2.0f * max_distance;
#pragma unroll
        for (int c = 0; c < NL_MAX_HITS; ++c) {
            int32_t i = -1;
            float a = max_distance, b = max_distance;
            if (c < cnt && !(mx[c] > two_md) && !(mn[c] > max_distance)) { i = idx[c]; a = mn[c]; b = mx[c]; ++nv; }
            ws.h_idx[(size_t)c * R + r] = i;
            ws.h_min[(size_t)c * R + r] = a;
            ws.h_max[(size_t)c * R + r] = b;
        }
        ws.nvalid[r] = nv;
        ray_nsamp[r] = 0;
    }
    const int wm = warp_max(nv);
    if ((threadIdx.x & 31) == 0 && wm > 0) atomicMax(&stats->max_hits, wm);
}

// ------------------------------------------------------------------------------------------------
// k_traverse_coop<LANES>: the same traversal, LANES (4 or 8) lanes per ray, 32/LANES rays per warp.
//   The thread-per-ray kernel above is latency-bound: 83 k rays give 17 warps per SM, each walking a chain of dependent
//   loads (ncu: 0.65 IPC/SM, stalls = long scoreboard).  Here every node expansion is one step of a lane group: lane u loads
//   record u of the node's packed child list (the group reads one 64/128-byte piece of a 128-byte line), slab-tests it, a
//   warp ballot yields the group's hit mask, and the hit children are pushed onto the ray's stack in SHARED memory at
//   positions given by the popcount of the lower mask bits.  Many more warps hide the latency; the stack and the hit lists
//   never touch local memory.
//   The packed list holds the node's EXISTING children, compacted (terminated by id -1): in ascending slot order for inner
//   nodes -- so pushes are in slot order 0..7 and pop 7..0 like the reference -- and in DESCENDING slot order for nodes of
//   side 2, whose children are leaves: those are recorded right away, in exactly the order in which the reference pops them
//   (it pushes slots 0..7, pops 7..0, and a leaf pushes nothing, so those pops are consecutive), and the 20-hit cut-off drops
//   the same tail.  With 4 lanes a node with more than 4 children takes a second pass (octree nodes here have 2.8 children on
//   average), which halves the predicated-off slab tests of the 8-lane variant.  A node's side is carried on the stack as
//   log2(side) (children have half the side).  Then a rank-by-counting stable sort by min_depth inside the group, distance
//   clipping, and a block-wide transposed write of the [20][R] planes.
// ------------------------------------------------------------------------------------------------
constexpr int CO_HPAD = NL_MAX_HITS + 1;    // row padding: conflict-free column reads in the transposed write

template <int LANES>
__global__ void __launch_bounds__(256) k_traverse_coop(int R, float voxel_size, float max_distance, const float *__restrict__ centres,
                                                        const int32_t *__restrict__ structure, const float4 *__restrict__ packed,
                                                        const float *__restrict__ ray_o, const float *__restrict__ ray_d, Workspace ws,
                                                        int32_t *__restrict__ ray_nsamp, nl_render_stats *stats) {
    constexpr int CO_RAYS = 256 / LANES;        // rays per block
    constexpr int STK = NL_STACK_CAP;           // same bound as the thread-per-ray kernel (1 + 7 x 18 levels)
    constexpr int NE = (NL_MAX_HITS + LANES - 1) / LANES;   // hit-list entries per lane in the sort
    __shared__ int s_stk[CO_RAYS][STK];
    __shared__ int s_idx[CO_RAYS][CO_HPAD];
    __shared__ float s_mn[CO_RAYS][CO_HPAD];
    __shared__ float s_mx[CO_RAYS][CO_HPAD];
    __shared__ int s_nv[CO_RAYS];
    const int tid = threadIdx.x, lane = tid & 31, o = tid / LANES, u = tid % LANES, gb = lane & ~(LANES - 1);
    const unsigned gmask = (LANES == 8 ? 0xffu : 0xfu);
    const int r = blockIdx.x * CO_RAYS + o;
    const float half_voxel = voxel_size * 0.5f;
    NlRay ray = nl_make_ray(0.f, 0.f, 0.f, 1.f, 1.f, 1.f);
    int ptr = -1, cnt = 0;
    bool overflow = false;
    if (r < R) {
        ray = nl_make_ray(ray_o[r * 3], ray_o[r * 3 + 1], ray_o[r * 3 + 2], ray_d[r * 3], ray_d[r * 3 + 1], ray_d[r * 3 + 2]);
        const int root_side = structure[8];
        float lo, hi;
        if (nl_slab(ray, centres[0], centres[1], centres[2], __fmul_rn(half_voxel, (float)root_side), lo, hi)) {
            if (root_side == 1) {      // degenerate one-voxel tree: the root is the only leaf
                if (u == 0) { s_idx[o][0] = 0; s_mn[o][0] = lo; s_mx[o][0] = hi; }
                cnt = 1;
            } else {
                if (u == 0) s_stk[o][0] = (31 - __clz(root_side)) << 26;
                ptr = 0;
            }
        }
    }
    __syncwarp();
    bool alive = ptr >= 0;
    while (__any_sync(0xffffffffu, alive)) {
        int lg = 0;
        const float4 *rec = packed;
        if (alive) {
            const int e = s_stk[o][ptr];
            lg = e >> 26;
            rec = packed + (size_t)(e & 0x3ffffff) * 8;
        }
        const float half = __fmul_rn(__fmul_rn(half_voxel, (float)(1 << lg)), 0.5f);
        __syncwarp();                                           // every lane of the group has read the stack top
        if (alive) --ptr;
        bool more = alive;                                      // this group still has records of the node to look at
#pragma unroll
        for (int pass = 0; pass < 8 / LANES; ++pass) {
            bool hit = false;
            float lo = 0.f, hi = 0.f;
            int id = -1;
            if (more) {
                const float4 c = rec[pass * LANES + u];
                id = __float_as_int(c.w);
                if (id > -1) hit = nl_slab(ray, c.x, c.y, c.z, half, lo, hi);
            }
            const unsigned mg = (__ballot_sync(0xffffffffu, hit) >> gb) & gmask;
            const int last_id = __shfl_sync(0xffffffffu, id, gb + LANES - 1);
            if (more) {
                const int nh = __popc(mg), below = __popc(mg & ((1u << u) - 1u));
                if (lg == 1) {
                    if (hit && cnt + below < NL_MAX_HITS) { s_idx[o][cnt + below] = id; s_mn[o][cnt + below] = lo; s_mx[o][cnt + below] = hi; }
                    cnt = min(cnt + nh, NL_MAX_HITS);
                } else if (ptr + nh >= STK) {
                    overflow = true;
                    ptr = -1;
                    more = false;
                } else {
                    if (hit) s_stk[o][ptr + 1 + below] = id | ((lg - 1) << 26);
                    ptr += nh;
                }
                more = more && last_id > -1 && cnt < NL_MAX_HITS;   // the list may continue in the next pass
            }
            if (pass + 1 < 8 / LANES && !__any_sync(0xffffffffu, more)) break;
        }
        if (alive) alive = !overflow && ptr >= 0 && cnt < NL_MAX_HITS;
        __syncwarp();                                           // pushes visible before the next pop
    }
    if (overflow && u == 0) atomicOr(&stats->error, 4);
    // ---- stable sort by min_depth (rank by counting; ties keep emission order), clipping (voxel_helpers.py:546-556) ----
    const float two_md = 2.0f * max_distance;
    int e_idx[NE], e_pos[NE];
    float e_mn[NE], e_mx[NE];
#pragma unroll
    for (int t = 0; t < NE; ++t) {
        const int i = u + t * LANES;
        e_pos[t] = -1;
        if (i < cnt) {
            const float key = s_mn[o][i];
            int pos = 0;
            for (int j = 0; j < cnt; ++j) {
                const float kj = s_mn[o][j];
                pos += (kj < key || (kj == key && j < i)) ? 1 : 0;
            }
            e_pos[t] = pos; e_idx[t] = s_idx[o][i]; e_mn[t] = key; e_mx[t] = s_mx[o][i];
        }
    }
    __syncwarp();                                               // every entry is in registers: permute in place
#pragma unroll
    for (int t = 0; t < NE; ++t)
        if (e_pos[t] >= 0) { s_idx[o][e_pos[t]] = e_idx[t]; s_mn[o][e_pos[t]] = e_mn[t]; s_mx[o][e_pos[t]] = e_mx[t]; }
    __syncwarp();
    int nv = 0;
#pragma unroll
    for (int t = 0; t < NE; ++t) {
        const int c = u + t * LANES;
        if (c < NL_MAX_HITS) {
            int32_t i = -1;
            float a = max_distance, b = max_distance;
            if (c < cnt) {
                const float mn = s_mn[o][c], mx = s_mx[o][c];
                if (!(mx > two_md) && !(mn > max_distance)) { i = s_idx[o][c]; a = mn; b = mx; ++nv; }
            }
            s_idx[o][c] = i; s_mn[o][c] = a; s_mx[o][c] = b;
        }
    }
#pragma unroll
    for (int off = 1; off < LANES; off <<= 1) nv += __shfl_xor_sync(0xffffffffu, nv, off);
    if (u == 0) s_nv[o] = nv;
    const int wm = warp_max(r < R ? nv : 0);
    if (lane == 0 && wm > 0) atomicMax(&stats->max_hits, wm);
    __syncthreads();
    // ---- transposed, coalesced write of the hit planes ----
    const int r0 = blockIdx.x * CO_RAYS;
    for (int e = tid; e < NL_MAX_HITS * CO_RAYS; e += 256) {
        const int c = e / CO_RAYS, ol = e % CO_RAYS;
        if (r0 + ol < R) {
            const size_t off = (size_t)c * R + r0 + ol;
            ws.h_idx[off] = s_idx[ol][c];
            ws.h_min[off] = s_mn[ol][c];
            ws.h_max[off] = s_mx[ol][c];
        }
    }
    if (tid < CO_RAYS && r0 + tid < R) {
        ws.nvalid[r0 + tid] = s_nv[tid];
        ray_nsamp[r0 + tid] = 0;
    }
}

__global__ void k_pack_children(int n_nodes, const int32_t *__restrict__ ids, const float *__restrict__ centres,
                                const int32_t *__restrict__ structure, float4 *__restrict__ packed) {
    // one thread per node: the existing children compacted to the front of the node's 8 records (terminated by id -1), in
    // ascending slot order for inner nodes (push order) and DESCENDING slot order for nodes of side 2, whose children are
    // leaves and are recorded in the order the reference pops them
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n_nodes) return;
    const int n = ids ? ids[slot] : slot;        // ids: re-pack only the listed nodes (incremental map update)
    const int32_t *st = structure + (size_t)n * 9;
    const bool leaf_parent = st[8] == 2;
    float4 *rec = packed + (size_t)n * 8;
    int j = 0;
    for (int i = 0; i < 8; ++i) {
        const int c = st[leaf_parent ? 7 - i : i];
        if (c > -1) rec[j++] = make_float4(centres[(size_t)c * 3], centres[(size_t)c * 3 + 1], centres[(size_t)c * 3 + 2], __int_as_float(c));
    }
    for (; j < 8; ++j) rec[j] = make_float4(0.f, 0.f, 0.f, __int_as_float(-1));
}

// ------------------------------------------------------------------------------------------------
// k_scan: single-block exclusive scan over n <= 2^31 ints (n is ~1e5..1e6; ~10 us).
//   HITS:    in = nvalid (flag = nvalid > 0) -> hit_rank[r] (or -1), hitray[rank] = r, total -> n_hit_rays
//   SAMPLES: in = ray_nsamp                  -> ray_offset[r],                         total -> n_samples
// ------------------------------------------------------------------------------------------------
enum { SCAN_HITS = 0, SCAN_SAMPLES = 1 };

template <int MODE>
__global__ void __launch_bounds__(1024) k_scan(int n, const int32_t *__restrict__ in, int32_t *__restrict__ out,
                                                int32_t *__restrict__ hitray, nl_render_stats *stats, int sample_capacity) {
    // tiles of 4096 elements: every thread owns 4 consecutive ones (one 16-byte load, issued one tile ahead so that its
    // latency hides behind the previous tile), warp shuffle scan, then every warp scans the 32 warp totals redundantly:
    // one __syncthreads per tile (the totals are double-buffered) and the running carry stays in registers
    __shared__ int wsum[2][32];
    __shared__ int compact[MODE == SCAN_HITS ? 4096 : 1];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    auto load4 = [&](int i0) {
        int4 x = make_int4(0, 0, 0, 0);
        if (i0 + 3 < n) {
            x = *reinterpret_cast<const int4 *>(in + i0);
        } else {
            if (i0 < n) x.x = in[i0];
            if (i0 + 1 < n) x.y = in[i0 + 1];
            if (i0 + 2 < n) x.z = in[i0 + 2];
        }
        return x;
    };
    int carry = 0;
    int4 nxt = load4(t * 4);
    for (int base = 0, par = 0; base < n; base += 4096, par ^= 1) {
        const int i0 = base + t * 4;
        const int4 x = nxt;
        if (base + 4096 < n) nxt = load4(i0 + 4096);
        int v[4] = {x.x, x.y, x.z, x.w};
        if (MODE == SCAN_HITS) {
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = v[k] > 0;
        }
        const int mine = v[0] + v[1] + v[2] + v[3];
        int incl = mine;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += y;
        }
        if (lane == 31) wsum[par][w] = incl;
        __syncthreads();
        const int ws = wsum[par][lane];
        int wi = ws;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, wi, off);
            if (lane >= off) wi += y;
        }
        const int wexcl = __shfl_sync(0xffffffffu, wi - ws, w);      // exclusive prefix of this warp's total
        const int tile_total = __shfl_sync(0xffffffffu, wi, 31);
        int run = carry + wexcl + incl - mine;
        if (MODE == SCAN_HITS) {
            // ranks as one 16-byte store; the compacted ray list of this tile is contiguous in the output, so it is staged in
            // shared memory and written back coalesced
            int4 o;
            o.x = v[0] ? run : -1;
            o.y = v[1] ? run + v[0] : -1;
            o.z = v[2] ? run + v[0] + v[1] : -1;
            o.w = v[3] ? run + v[0] + v[1] + v[2] : -1;
            if (i0 + 3 < n) {
                *reinterpret_cast<int4 *>(out + i0) = o;
            } else {
                if (i0 < n) out[i0] = o.x;
                if (i0 + 1 < n) out[i0 + 1] = o.y;
                if (i0 + 2 < n) out[i0 + 2] = o.z;
            }
            int loc = run - carry;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (v[k]) compact[loc] = i0 + k;     // v[k] is 0 for i0 + k >= n
                loc += v[k];
            }
            __syncthreads();
            for (int j = t; j < tile_total; j += 1024) hitray[carry + j] = compact[j];
            // the next tile's writes to compact[] come after its own __syncthreads (warp totals), which every thread reaches
            // only after finishing this copy
        } else {
            const int4 o = make_int4(run, run + v[0], run + v[0] + v[1], run + v[0] + v[1] + v[2]);
            if (i0 + 3 < n) {
                *reinterpret_cast<int4 *>(out + i0) = o;
            } else {
                if (i0 < n) out[i0] = o.x;
                if (i0 + 1 < n) out[i0 + 1] = o.y;
                if (i0 + 2 < n) out[i0 + 2] = o.z;
            }
        }
        carry += tile_total;
    }
    if (t == 0) {
        const int total = carry;
        if (MODE == SCAN_HITS) {
            stats->n_hit_rays = total;
        } else {
            stats->n_samples = total;
            if (total > sample_capacity) atomicOr(&stats->error, 2);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_scan_chained: the same two scans over many blocks (one 4096-element tile each) in a single pass.  A block takes a ticket
// (so that every tile it may have to wait for belongs to a block that is already running), scans its tile, publishes the tile
// total, and adds up the totals of the tiles before it -- one thread per predecessor, spinning until that total is published.
// At 83 k rays that is 21 blocks and ~5 us instead of 17-30 us for the single-block loop above (which stays as the fallback for
// more than 4 M rays).  scratch: [0] ticket, [8 + tile] (1 << 32 | total); zeroed by nl_render_samples before the chain starts.
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(1024) k_scan_chained(int n, const int32_t *__restrict__ in, int32_t *__restrict__ out,
                                                        int32_t *__restrict__ hitray, nl_render_stats *stats, int sample_capacity,
                                                        unsigned long long *scratch) {
    __shared__ int s_warp[32];
    __shared__ int s_tile, s_carry;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) s_tile = (int)atomicAdd(&scratch[0], 1ULL);
    __syncthreads();
    const int tile = s_tile;
    const int i0 = tile * 4096 + t * 4;
    int4 x = make_int4(0, 0, 0, 0);
    if (i0 + 3 < n) {
        x = *reinterpret_cast<const int4 *>(in + i0);
    } else {
        if (i0 < n) x.x = in[i0];
        if (i0 + 1 < n) x.y = in[i0 + 1];
        if (i0 + 2 < n) x.z = in[i0 + 2];
    }
    int v[4] = {x.x, x.y, x.z, x.w};
    if (MODE == SCAN_HITS) {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = v[k] > 0;
    }
    const int mine = v[0] + v[1] + v[2] + v[3];
    int incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += y;
    }
    if (lane == 31) s_warp[w] = incl;
    __syncthreads();
    const int ws_ = s_warp[lane];
    int wi = ws_;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, wi, off);
        if (lane >= off) wi += y;
    }
    const int wexcl = __shfl_sync(0xffffffffu, wi - ws_, w);
    const int tile_total = __shfl_sync(0xffffffffu, wi, 31);
    if (t == 0) {
        __threadfence();
        atomicExch(&scratch[8 + tile], (1ULL << 32) | (unsigned long long)(unsigned)tile_total);
    }
    // totals of the tiles before this one (gridDim.x <= 1024 = one thread per predecessor)
    int prev = 0;
    if (t < tile) {
        unsigned long long a;
        do { a = *((volatile unsigned long long *)&scratch[8 + t]); } while ((a >> 32) == 0ULL);
        prev = (int)(unsigned)(a & 0xffffffffULL);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) prev += __shfl_down_sync(0xffffffffu, prev, off);
    __syncthreads();                       // s_warp is reused
    if (lane == 0) s_warp[w] = prev;
    __syncthreads();
    if (t == 0) {
        int c = 0;
        for (int k = 0; k < 32; ++k) c += s_warp[k];
        s_carry = c;
    }
    __syncthreads();
    const int carry = s_carry;
    const int run = carry + wexcl + incl - mine;
    if (MODE == SCAN_HITS) {
        int4 o;
        o.x = v[0] ? run : -1;
        o.y = v[1] ? run + v[0] : -1;
        o.z = v[2] ? run + v[0] + v[1] : -1;
        o.w = v[3] ? run + v[0] + v[1] + v[2] : -1;
        if (i0 + 3 < n) {
            *reinterpret_cast<int4 *>(out + i0) = o;
        } else {
            if (i0 < n) out[i0] = o.x;
            if (i0 + 1 < n) out[i0 + 1] = o.y;
            if (i0 + 2 < n) out[i0 + 2] = o.z;
        }
        int loc = run;                     // positions ascend with the thread index: a warp's writes fall into one short range
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (v[k]) hitray[loc] = i0 + k;
            loc += v[k];
        }
    } else {
        const int4 o = make_int4(run, run + v[0], run + v[0] + v[1], run + v[0] + v[1] + v[2]);
        if (i0 + 3 < n) {
            *reinterpret_cast<int4 *>(out + i0) = o;
        } else {
            if (i0 < n) out[i0] = o.x;
            if (i0 + 1 < n) out[i0 + 1] = o.y;
            if (i0 + 2 < n) out[i0 + 2] = o.z;
        }
    }
    if (tile == (int)gridDim.x - 1 && t == 0) {
        const int total = carry + tile_total;
        if (MODE == SCAN_HITS) {
            stats->n_hit_rays = total;
        } else {
            stats->n_samples = total;
            if (total > sample_capacity) atomicOr(&stats->error, 2);
        }
    }
}

// counter-based uniform noise in (0,1) for the stochastic sampler when no noise tensor is passed in
__device__ __forceinline__ float hash_uniform(uint32_t seed, uint32_t ray, uint32_t step) {
    uint32_t x = seed ^ (ray * 0x9E3779B1u) ^ (step * 0x85EBCA77u);
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    const float u = (float)(x >> 8) * (1.0f / 16777216.0f);
    return fminf(fmaxf(u, 0.001f), 0.999f);  // voxel_helpers.py:301 clamp
}

struct SampleParams {
    int R, sample_capacity, compat;
    float step_size, truncation, max_depth;
    const float *ray_o, *ray_d, *gt_depth, *cosv, *noise;
    int noise_stride;
    uint32_t rng_seed;
    const uint32_t *rng_seed_dev;
    int32_t *s_ray, *s_vox;
    float *s_depth, *s_xyz;
    uint8_t *s_flag;
    int32_t *ray_nsamp;
    const int32_t *ray_offset;
};

// criterion.py:67-82 for one cell: bit0 front_mask, bit1 sdf_mask
__device__ __forceinline__ uint32_t loss_flags(float z, float d, float trunc, float max_depth) {
    const bool front = z < __fsub_rn(d, trunc);
    const bool back = z > __fadd_rn(d, trunc);
    const bool dm = (d > 0.0f) && (d < max_depth);
    return (front ? 1u : 0u) | ((!front && !back && dm) ? 2u : 0u);
}

// ------------------------------------------------------------------------------------------------
// k_sample: ray_sample + InverseCDFRaySampling.forward + inverse_cdf_sampling_kernel for the q-th hit ray.
// The [200, K', P] padding / 800-ray chunking of the reference wrapper only matters through the two
// index quirks of the kernel tail (SURVEY A.3); they are reproduced from (q, R_hit, P) directly.
// ------------------------------------------------------------------------------------------------
template <bool FILL>
__global__ void __launch_bounds__(128) k_sample(SampleParams p, Workspace ws, nl_render_stats *stats) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int R_hit = stats->n_hit_rays;
    const int R = p.R;
    long long c_fs = 0, c_sdf = 0;
    int nsamp = 0, steps_ceil = 0;
    if (q < R_hit) {
        const int r = ws.hitray[q];
        const int P = stats->max_hits;
        int32_t bidx[NL_MAX_HITS];
        float bmin[NL_MAX_HITS], bmax[NL_MAX_HITS], prob[NL_MAX_HITS];
        float tot = 0.f;
#pragma unroll
        for (int c = 0; c < NL_MAX_HITS; ++c) {
            if (c < P) {
                bidx[c] = ws.h_idx[(size_t)c * R + r];
                bmin[c] = ws.h_min[(size_t)c * R + r];
                bmax[c] = ws.h_max[(size_t)c * R + r];
                prob[c] = (bidx[c] == -1) ? 0.f : __fsub_rn(bmax[c], bmin[c]);  // voxel_helpers.py:572-575
                tot = __fadd_rn(tot, prob[c]);                                   // left-to-right fp32 sum
            }
        }
#pragma unroll
        for (int c = 0; c < NL_MAX_HITS; ++c)
            if (c < P) prob[c] = __fdiv_rn(prob[c], tot);                        // :576
        const float steps = __fdiv_rn(tot, p.step_size);                         // :577
        if (!FILL) {
            if (tot > 10.0f * NL_MAX_DEPTH_FILL) atomicOr(&stats->error, 1);      // :579
            steps_ceil = (int)ceilf(steps);
        }
        // position of this ray in the reference's [200, K', P] layout and 800-wide launches (voxel_helpers.py:274-316)
        const int Kp = (R_hit + NL_SAMPLE_G - 1) / NL_SAMPLE_G;
        const int b = q / Kp, j0 = q - b * Kp;
        const int ch = j0 / NL_SAMPLE_CHUNK, j = j0 - ch * NL_SAMPLE_CHUNK;
        const int num_rays = min(NL_SAMPLE_CHUNK, Kp - ch * NL_SAMPLE_CHUNK);
        const int r_lead = ws.hitray[b * Kp + ch * NL_SAMPLE_CHUNK];            // ray 0 of this (batch, chunk)
        const int H = j * P;

        const float cosr = p.cosv ? p.cosv[r] : 1.0f;
        const float gd = p.gt_depth ? p.gt_depth[r] : 0.0f;
        const bool with_loss = p.gt_depth != nullptr;
        const float ox = p.ray_o[r * 3], oy = p.ray_o[r * 3 + 1], oz = p.ray_o[r * 3 + 2];
        const float dx = p.ray_d[r * 3], dy = p.ray_d[r * 3 + 1], dz = p.ray_d[r * 3 + 2];
        const int base = FILL ? p.ray_offset[r] : 0;

        auto emit = [&](int vox, float depth) {
            uint32_t fl = 0;
            if (with_loss) fl = loss_flags(__fmul_rn(depth, cosr), gd, p.truncation, p.max_depth);
            if (FILL) {
                const int m = base + nsamp;
                if (m < p.sample_capacity) {
                    p.s_ray[m] = r;
                    p.s_vox[m] = vox;
                    p.s_depth[m] = depth;
                    p.s_xyz[(size_t)m * 3 + 0] = __fadd_rn(ox, __fmul_rn(dx, depth));  // ray(): mul then add (render_helpers.py:9-10)
                    p.s_xyz[(size_t)m * 3 + 1] = __fadd_rn(oy, __fmul_rn(dy, depth));
                    p.s_xyz[(size_t)m * 3 + 2] = __fadd_rn(oz, __fmul_rn(dz, depth));
                    p.s_flag[m] = (uint8_t)fl;
                }
            } else {
                c_fs += (fl & 1u);
                c_sdf += (fl >> 1) & 1u;
            }
            ++nsamp;
        };

        // ---- the walk (sampler.cuh).  Tail quirks of the reference's batched launch, in terms of this ray's slot j in its
        //      (batch, chunk) of num_rays rays: flush only while num_rays > j*P + bin; continuation test on the chunk's leader ray ----
        uint32_t seed = p.rng_seed;
        if (p.rng_seed_dev) { seed = *p.rng_seed_dev; seed = seed ? seed : 1u; }
        struct {
            const int32_t *i; const float *a, *b, *pr;
            __device__ __forceinline__ int idx(int c) const { return i[c]; }
            __device__ __forceinline__ float lo(int c) const { return a[c]; }
            __device__ __forceinline__ float hi(int c) const { return b[c]; }
            __device__ __forceinline__ float prob(int c) const { return pr[c]; }
        } bins = {bidx, bmin, bmax, prob};
        nl_inverse_cdf_walk(
            P, bins, steps, -1.0f,
            [&](int i) {
                if (p.noise) return p.noise[(size_t)q * p.noise_stride + i];
                return seed ? hash_uniform(seed, (uint32_t)r, (uint32_t)i) : 0.5f;
            },
            [&](int vox, float z0, float z1) { emit(vox, __fmul_rn(__fadd_rn(z1, z0), 0.5f)); },
            [&](int bin) { return !p.compat || num_rays > (H + bin); },
            [&](int bin) { return p.compat ? ws.h_idx[(size_t)bin * R + r_lead] : bidx[bin]; });

        if (!FILL) {
            p.ray_nsamp[r] = nsamp;
            if (with_loss) {  // padded cells of this row: z_vals = MAX_DEPTH (voxel_helpers.py:590), sdf = 1, valid = 0
                const uint32_t fl = loss_flags(__fmul_rn(NL_MAX_DEPTH_FILL, cosr), gd, p.truncation, p.max_depth);
                if (fl & 1u) {
                    atomicAdd((unsigned long long *)&stats->pad_fs_rays, 1ULL);
                    atomicAdd((unsigned long long *)&stats->pad_fs_nsamp, (unsigned long long)nsamp);
                }
                if (fl & 2u) {
                    atomicAdd((unsigned long long *)&stats->pad_sdf_rays, 1ULL);
                    atomicAdd((unsigned long long *)&stats->pad_sdf_nsamp, (unsigned long long)nsamp);
                    atomicAdd(&stats->pad_sdf_d2, (double)gd * (double)gd);
                    atomicAdd(&stats->pad_sdf_d2_nsamp, (double)gd * (double)gd * (double)nsamp);
                }
            }
        }
    }
    if (!FILL) {
        const int wm = warp_max(nsamp);
        const int wsc = warp_max(steps_ceil);
        for (int off = 16; off > 0; off >>= 1) {
            c_fs += __shfl_down_sync(0xffffffffu, c_fs, off);
            c_sdf += __shfl_down_sync(0xffffffffu, c_sdf, off);
        }
        if ((threadIdx.x & 31) == 0) {
            if (wm > 0) atomicMax(&stats->max_samples, wm);
            if (wsc > 0) atomicMax(&stats->max_steps_ceil, wsc);
            if (c_fs) atomicAdd((unsigned long long *)&stats->cnt_fs_valid, (unsigned long long)c_fs);
            if (c_sdf) atomicAdd((unsigned long long *)&stats->cnt_sdf_valid, (unsigned long long)c_sdf);
        }
    }
}

// criterion.py:84-88 and the mean() denominators of :97-100
__global__ void k_loss_prepare(nl_render_stats *s, float fs_weight, float sdf_weight) {
    const long long S = s->max_samples;
    const long long n_fs = s->cnt_fs_valid + s->pad_fs_rays * S - s->pad_fs_nsamp;
    const long long n_sdf = s->cnt_sdf_valid + s->pad_sdf_rays * S - s->pad_sdf_nsamp;
    const float nfs = (float)n_fs, nsdf = (float)n_sdf;
    const float num = __fadd_rn(nsdf, nfs);
    s->n_fs = nfs;
    s->n_sdf = nsdf;
    s->w_fs = __fsub_rn(1.0f, __fdiv_rn(nfs, num));
    s->w_sdf = __fsub_rn(1.0f, __fdiv_rn(nsdf, num));
    const float N = (float)((long long)s->n_hit_rays * S);
    const bool ok = (N > 0.f) && (num > 0.f);   // no hit rays: nothing to optimise, keep the constants finite
    s->g_fs = ok ? fs_weight * s->w_fs / N : 0.f;
    s->g_sdf = ok ? sdf_weight * s->w_sdf / N : 0.f;
    s->pad_fs_sum = (float)(s->pad_fs_rays * S - s->pad_fs_nsamp);           // each padded front cell: (0 - 1)^2
    s->pad_sdf_sum = (float)(s->pad_sdf_d2 * (double)S - s->pad_sdf_d2_nsamp); // each padded sdf cell: (0 - depth)^2
    s->fs_sum = 0.0;
    s->sdf_sum = 0.0;
    s->loss = s->fs_loss = s->sdf_loss = 0.f;
}

__global__ void k_loss_finalize(nl_render_stats *s, float fs_weight, float sdf_weight) { nl_loss_finalize_dev(s, fs_weight, sdf_weight); }

// Fold one iteration's statistics into the call-wide control block (include/nerfloam_b200.h section 8).
__global__ void k_iter_status(const nl_render_stats *s, const int32_t *prev, int32_t *ctl) {
    for (int i = 0; i < NL_CTL_WORDS; ++i) ctl[i] = prev[i];
    const int err = s->error;
    const int skip = (s->n_hit_rays <= 0) || (err & 1);   // render_rays -> None (render_helpers.py:216, voxel_helpers.py:579); global values
                                                          // after the multi-GPU exchange, so every rank decides alike
    ctl[NL_CTL_ERROR] |= err;
    ctl[NL_CTL_SKIPPED] += skip;
    ctl[NL_CTL_SKIP_NOW] = skip;
    ctl[NL_CTL_ADAM_STEP] += skip ? 0 : 1;
    ctl[NL_CTL_MIN_HIT] = min(ctl[NL_CTL_MIN_HIT], s->n_hit_rays);
    ctl[NL_CTL_ITERS] += 1;
    ctl[NL_CTL_MAX_SAMPLES] = max(ctl[NL_CTL_MAX_SAMPLES], s->n_samples);
}

// Statistics exchange, packed (section 9): every value that must become global travels in one f64 vector reduced with SUM.
__global__ void k_stats_pack(const nl_render_stats *s, void *buf_, int rank, int world, int phase) {
    if (phase == 0) {
        double *b = (double *)buf_;
        const int t = threadIdx.x;
        if (t == 0) {
            b[0] = (double)s->cnt_fs_valid; b[1] = (double)s->cnt_sdf_valid; b[2] = (double)s->pad_fs_rays; b[3] = (double)s->pad_fs_nsamp;
            b[4] = (double)s->pad_sdf_rays; b[5] = (double)s->pad_sdf_nsamp; b[6] = s->pad_sdf_d2; b[7] = s->pad_sdf_d2_nsamp;
            b[8] = (double)s->n_hit_rays; b[9] = 0.0;
        }
        for (int r = t; r < world; r += blockDim.x) {
            b[NL_STATS_PACK_FIXED + r] = (r == rank) ? (double)s->max_samples : 0.0;          // SUM of one-hot slots, MAX on unpack
            b[NL_STATS_PACK_FIXED + world + r] = (r == rank) ? (double)s->error : 0.0;        // OR on unpack
        }
    } else if (threadIdx.x == 0) {
        float *b = (float *)buf_;
        const float fh = (float)s->fs_sum, sh = (float)s->sdf_sum;
        b[0] = fh; b[1] = (float)(s->fs_sum - (double)fh); b[2] = sh; b[3] = (float)(s->sdf_sum - (double)sh);
    }
}

__global__ void k_stats_unpack(nl_render_stats *s, const void *buf_, int world, int phase) {
    if (phase == 0) {
        const double *b = (const double *)buf_;
        s->cnt_fs_valid = (long long)b[0]; s->cnt_sdf_valid = (long long)b[1]; s->pad_fs_rays = (long long)b[2]; s->pad_fs_nsamp = (long long)b[3];
        s->pad_sdf_rays = (long long)b[4]; s->pad_sdf_nsamp = (long long)b[5]; s->pad_sdf_d2 = b[6]; s->pad_sdf_d2_nsamp = b[7];
        s->n_hit_rays = (int32_t)b[8];
        int smax = 0, err = 0;
        for (int r = 0; r < world; ++r) {
            smax = max(smax, (int)b[NL_STATS_PACK_FIXED + r]);
            err |= (int)b[NL_STATS_PACK_FIXED + world + r];
        }
        s->max_samples = smax;
        s->error = err;
    } else {
        const float *b = (const float *)buf_;
        s->fs_sum = (double)b[0] + (double)b[1];
        s->sdf_sum = (double)b[2] + (double)b[3];
    }
}

// phase-0 unpack straight from every rank's packed vector in symmetric memory (P2P loads, summed in rank order on every rank):
// the statistics exchange without a collective library call -- pack, cross-rank barrier, this kernel.
__global__ void k_stats_unpack_peers(nl_render_stats *s, const double *const *peers, int world) {
    __shared__ double b[NL_STATS_PACK_FIXED];
    const int t = threadIdx.x;
    if (t < NL_STATS_PACK_FIXED) {
        double acc = 0.0;
        for (int q = 0; q < world; ++q) acc += peers[q][t];
        b[t] = acc;
    }
    __syncthreads();
    if (t == 0) {
        s->cnt_fs_valid = (long long)b[0]; s->cnt_sdf_valid = (long long)b[1]; s->pad_fs_rays = (long long)b[2]; s->pad_fs_nsamp = (long long)b[3];
        s->pad_sdf_rays = (long long)b[4]; s->pad_sdf_nsamp = (long long)b[5]; s->pad_sdf_d2 = b[6]; s->pad_sdf_d2_nsamp = b[7];
        s->n_hit_rays = (int32_t)b[8];
        int smax = 0, err = 0;
        for (int q = 0; q < world; ++q) {               // slot q of rank q's own vector (the other slots of a vector are zero)
            smax = max(smax, (int)peers[q][NL_STATS_PACK_FIXED + q]);
            err |= (int)peers[q][NL_STATS_PACK_FIXED + world + q];
        }
        s->max_samples = smax;
        s->error = err;
    }
}

}  // namespace

extern "C" int nl_stats_unpack_peers(nl_render_stats *d_stats, const double *const *d_peer_bufs, int world, float fs_weight, float sdf_weight,
                                     void *stream) {
    if (!d_stats || !d_peer_bufs || world < 1) return nl_set_error("nl_stats_unpack_peers: bad arguments");
    k_stats_unpack_peers<<<1, 32, 0, (cudaStream_t)stream>>>(d_stats, d_peer_bufs, world);
    k_loss_prepare<<<1, 1, 0, (cudaStream_t)stream>>>(d_stats, fs_weight, sdf_weight);
    NL_CHECK_LAUNCH("nl_stats_unpack_peers");
    return NL_OK;
}

extern "C" int nl_iter_status(const nl_render_stats *d_stats, const int32_t *d_ctl_prev, int32_t *d_ctl, void *stream) {
    if (!d_stats || !d_ctl || !d_ctl_prev) return nl_set_error("nl_iter_status: null pointer");
    k_iter_status<<<1, 1, 0, (cudaStream_t)stream>>>(d_stats, d_ctl_prev, d_ctl);
    NL_CHECK_LAUNCH("nl_iter_status");
    return NL_OK;
}

extern "C" int nl_stats_pack(const nl_render_stats *d_stats, void *d_buf, int rank, int world, int phase, void *stream) {
    if (!d_stats || !d_buf) return nl_set_error("nl_stats_pack: null pointer");
    if (world < 1 || rank < 0 || rank >= world || (phase != 0 && phase != 1)) return nl_set_error("nl_stats_pack: bad rank / world / phase");
    k_stats_pack<<<1, 32, 0, (cudaStream_t)stream>>>(d_stats, d_buf, rank, world, phase);
    NL_CHECK_LAUNCH("nl_stats_pack");
    return NL_OK;
}

extern "C" int nl_stats_unpack(nl_render_stats *d_stats, const void *d_buf, int world, int phase, float fs_weight, float sdf_weight, void *stream) {
    if (!d_stats || !d_buf) return nl_set_error("nl_stats_unpack: null pointer");
    if (world < 1 || (phase != 0 && phase != 1)) return nl_set_error("nl_stats_unpack: bad world / phase");
    k_stats_unpack<<<1, 1, 0, (cudaStream_t)stream>>>(d_stats, d_buf, world, phase);
    if (phase == 0) k_loss_prepare<<<1, 1, 0, (cudaStream_t)stream>>>(d_stats, fs_weight, sdf_weight);
    NL_CHECK_LAUNCH("nl_stats_unpack");
    return NL_OK;
}

extern "C" int64_t nl_octree_packed_bytes(int32_t n_nodes) { return n_nodes < 0 ? -1 : (int64_t)n_nodes * 128; }

extern "C" int nl_octree_pack_children(int32_t n_nodes, const float *d_centres, const int32_t *d_structure, void *d_packed, void *stream) {
    if (n_nodes <= 0) return nl_set_error("nl_octree_pack_children: n_nodes must be positive");
    if (n_nodes >= (1 << 26)) return nl_set_error("nl_octree_pack_children: at most 2^26 nodes (the traversal stack packs id and level)");
    if (!d_centres || !d_structure || !d_packed) return nl_set_error("nl_octree_pack_children: null pointer");
    if (((uintptr_t)d_packed & 15u) != 0) return nl_set_error("nl_octree_pack_children: d_packed must be 16-byte aligned");
    k_pack_children<<<nl_div_up(n_nodes, 128), 128, 0, (cudaStream_t)stream>>>(n_nodes, nullptr, d_centres, d_structure, (float4 *)d_packed);
    NL_CHECK_LAUNCH("nl_octree_pack_children");
    return NL_OK;
}

extern "C" int nl_octree_pack_children_rows(int32_t n_ids, const int32_t *d_ids, const float *d_centres, const int32_t *d_structure, void *d_packed,
                                            void *stream) {
    if (n_ids < 0) return nl_set_error("nl_octree_pack_children_rows: negative count");
    if (n_ids == 0) return NL_OK;
    if (!d_ids || !d_centres || !d_structure || !d_packed) return nl_set_error("nl_octree_pack_children_rows: null pointer");
    if (((uintptr_t)d_packed & 15u) != 0) return nl_set_error("nl_octree_pack_children_rows: d_packed must be 16-byte aligned");
    k_pack_children<<<nl_div_up(n_ids, 128), 128, 0, (cudaStream_t)stream>>>(n_ids, d_ids, d_centres, d_structure, (float4 *)d_packed);
    NL_CHECK_LAUNCH("nl_octree_pack_children_rows");
    return NL_OK;
}

extern "C" int64_t nl_render_workspace_bytes(int32_t n_rays) {
    if (n_rays < 0) return -1;
    const size_t R = (size_t)(n_rays > 0 ? n_rays : 1);
    return (int64_t)(3 * align256(4 * NL_MAX_HITS * R) + 2 * align256(4 * R) + align256(8 * 2 * SCAN_SCRATCH) + 256);
}

extern "C" int nl_render_samples(const nl_render_args *a, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!a) return nl_set_error("nl_render_samples: null args");
    if (a->n_rays <= 0 || a->n_nodes <= 0) return nl_set_error("nl_render_samples: n_rays and n_nodes must be positive");
    if (!a->d_centres || !a->d_structure || !a->d_ray_o || !a->d_ray_d || !a->d_stats || !a->d_hit_rank || !a->d_s_ray ||
        !a->d_s_vox || !a->d_s_depth || !a->d_s_xyz || !a->d_s_flag || !a->d_ray_nsamp || !a->d_ray_offset || !a->d_workspace)
        return nl_set_error("nl_render_samples: null pointer");
    if (a->workspace_bytes < nl_render_workspace_bytes(a->n_rays)) return nl_set_error("nl_render_samples: workspace too small");
    if (!(a->step_size > 0.f) || !(a->voxel_size > 0.f)) return nl_set_error("nl_render_samples: step_size and voxel_size must be > 0");
    if (a->d_noise && a->noise_stride <= 0) return nl_set_error("nl_render_samples: noise_stride must be > 0 with d_noise");
    if ((((uintptr_t)a->d_ray_nsamp | (uintptr_t)a->d_ray_offset | (uintptr_t)a->d_hit_rank | (uintptr_t)a->d_workspace) & 15u) != 0)
        return nl_set_error("nl_render_samples: d_ray_nsamp, d_ray_offset, d_hit_rank and d_workspace must be 16-byte aligned");
    const int R = a->n_rays;
    Workspace ws = carve(a->d_workspace, R);
    cudaMemsetAsync(a->d_stats, 0, sizeof(nl_render_stats), stream);
    const int blocks = nl_div_up(R, 128);
    // lanes per ray: 8 (one per child) while the launch is latency-bound -- a tracking / real-size mapping iteration has 2-10 k rays,
    // far fewer than the GPU holds threads for (B200: 5.99 -> 5.53 ms per 25-iteration scan, 15.8 -> 15.2 ms per 5-frame mapping call);
    // 4 once the rays alone fill the SMs (83 k rays: 1.575 vs 1.617 ms per step).
    if (a->d_packed_children && R <= 32768)
        k_traverse_coop<8><<<nl_div_up(R, 32), 256, 0, stream>>>(R, a->voxel_size, a->max_distance, a->d_centres, a->d_structure,
                                                                  (const float4 *)a->d_packed_children, a->d_ray_o, a->d_ray_d, ws,
                                                                  a->d_ray_nsamp, a->d_stats);
    else if (a->d_packed_children)
        k_traverse_coop<4><<<nl_div_up(R, 64), 256, 0, stream>>>(R, a->voxel_size, a->max_distance, a->d_centres, a->d_structure,
                                                                  (const float4 *)a->d_packed_children, a->d_ray_o, a->d_ray_d, ws,
                                                                  a->d_ray_nsamp, a->d_stats);
    else
        k_traverse_sort<<<nl_div_up(R, 64), 64, 0, stream>>>(R, a->voxel_size, a->max_distance, a->d_centres, a->d_structure, a->d_ray_o,
                                                              a->d_ray_d, ws, a->d_ray_nsamp, a->d_stats);
    // the single-block scans are the fallback for more than 4 M rays
    const int scan_tiles = nl_div_up(R, 4096);
    const bool chained = scan_tiles <= SCAN_MAX_TILES;
    if (chained) {
        cudaMemsetAsync(ws.scan, 0, sizeof(unsigned long long) * 2 * SCAN_SCRATCH, stream);
        k_scan_chained<SCAN_HITS><<<scan_tiles, 1024, 0, stream>>>(R, ws.nvalid, a->d_hit_rank, ws.hitray, a->d_stats, 0, ws.scan);
    } else {
        k_scan<SCAN_HITS><<<1, 1024, 0, stream>>>(R, ws.nvalid, a->d_hit_rank, ws.hitray, a->d_stats, 0);
    }
    SampleParams p;
    p.R = R; p.sample_capacity = a->sample_capacity; p.compat = a->reference_compat;
    p.step_size = a->step_size; p.truncation = a->truncation; p.max_depth = a->max_depth;
    p.ray_o = a->d_ray_o; p.ray_d = a->d_ray_d; p.gt_depth = a->d_gt_depth; p.cosv = a->d_cos; p.noise = a->d_noise;
    p.noise_stride = a->noise_stride; p.rng_seed = a->rng_seed; p.rng_seed_dev = a->d_noise ? nullptr : a->d_rng_seed;
    p.s_ray = a->d_s_ray; p.s_vox = a->d_s_vox; p.s_depth = a->d_s_depth; p.s_xyz = a->d_s_xyz; p.s_flag = a->d_s_flag;
    p.ray_nsamp = a->d_ray_nsamp; p.ray_offset = a->d_ray_offset;
    k_sample<false><<<blocks, 128, 0, stream>>>(p, ws, a->d_stats);
    if (chained) k_scan_chained<SCAN_SAMPLES><<<scan_tiles, 1024, 0, stream>>>(R, a->d_ray_nsamp, a->d_ray_offset, nullptr, a->d_stats, a->sample_capacity, ws.scan + SCAN_SCRATCH);
    else k_scan<SCAN_SAMPLES><<<1, 1024, 0, stream>>>(R, a->d_ray_nsamp, a->d_ray_offset, nullptr, a->d_stats, a->sample_capacity);
    k_sample<true><<<blocks, 128, 0, stream>>>(p, ws, a->d_stats);
    if (a->d_gt_depth) k_loss_prepare<<<1, 1, 0, stream>>>(a->d_stats, a->fs_weight, a->sdf_weight);
    NL_CHECK_LAUNCH("nl_render_samples");
    return NL_OK;
}

extern "C" int nl_loss_prepare(nl_render_stats *d_stats, float fs_weight, float sdf_weight, void *stream) {
    if (!d_stats) return nl_set_error("nl_loss_prepare: null stats");
    k_loss_prepare<<<1, 1, 0, (cudaStream_t)stream>>>(d_stats, fs_weight, sdf_weight);
    NL_CHECK_LAUNCH("nl_loss_prepare");
    return NL_OK;
}

extern "C" int nl_loss_finalize(nl_render_stats *d_stats, float fs_weight, float sdf_weight, void *stream) {
    if (!d_stats) return nl_set_error("nl_loss_finalize: null stats");
    k_loss_finalize<<<1, 1, 0, (cudaStream_t)stream>>>(d_stats, fs_weight, sdf_weight);
    NL_CHECK_LAUNCH("nl_loss_finalize");
    return NL_OK;
}
