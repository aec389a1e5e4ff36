// Embedding gather + trilinear interpolation and its backward scatter (SURVEY.md section 8 a-6, a-7).
//
// Replaces get_features / get_embeddings / trilinear_interp / offset_points
// (src/variations/render_helpers.py:40-93): four chained F.embedding gathers with a GPU->CPU->GPU
// detour through an 8 GB id table, ~12 elementwise kernels with [M,8,3] / [M,8,16] temporaries, and
// autograd's mirror image of all that.  Here: one thread per sample, the voxel -> 8 embedding rows
// indirection is a single flat i32[n,8] table, each bf16 row is two 16-byte loads (16 independent
// loads in flight per thread), weights and the 16 output features never leave registers.
//
// Algorithmic HBM bytes per sample (BASELINE.md): forward 312 B (voxel id 4, xyz 12 [depth 4 + centre
// lookup], 8 row ids 32, 8 x 32 B bf16 rows 256, output is 64 B of features here instead of 4 B sdf
// because the MLP is a separate kernel), backward 1116 - 312 = 804 B (ids 32, rows 256, 512 B of
// fp32 atomic adds, dfeats 64 in).
//
// Numerics follow render_helpers.py:65: p = (xyz - centre) / voxel_size + 0.5 with a true division;
// corner k = 4*kx + 2*ky + kz; w_k = (ax * ay) * az with a = p or 1-p.
#include "nl_cuda.cuh"

namespace {

struct Tri {
    float px, py, pz;
};

__device__ __forceinline__ Tri tri_coords(const float *__restrict__ xyz, const float *__restrict__ centre, float voxel_size) {
    Tri t;
    t.px = __fadd_rn(__fdiv_rn(__fsub_rn(xyz[0], centre[0]), voxel_size), 0.5f);
    t.py = __fadd_rn(__fdiv_rn(__fsub_rn(xyz[1], centre[1]), voxel_size), 0.5f);
    t.pz = __fadd_rn(__fdiv_rn(__fsub_rn(xyz[2], centre[2]), voxel_size), 0.5f);
    return t;
}

__device__ __forceinline__ float corner_weight(const Tri &t, int k) {
    const float ax = (k & 4) ? t.px : __fsub_rn(1.0f, t.px);
    const float ay = (k & 2) ? t.py : __fsub_rn(1.0f, t.py);
    const float az = (k & 1) ? t.pz : __fsub_rn(1.0f, t.pz);
    return __fmul_rn(__fmul_rn(ax, ay), az);
}

__device__ __forceinline__ void unpack8(const uint4 &v, float *f) {
    f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
}

__global__ void __launch_bounds__(128) k_gather_fwd(long long M_host, const int32_t *__restrict__ M_dev,
                                                     const float *__restrict__ xyz, const int32_t *__restrict__ vox,
                                                     const float *__restrict__ centres, const int32_t *__restrict__ vox2row,
                                                     const uint4 *__restrict__ emb, float voxel_size, float4 *__restrict__ feats) {
    const long long M = M_dev ? min((long long)*M_dev, M_host) : M_host;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (long long)gridDim.x * blockDim.x) {
        const int v = vox[i];
        const int4 r0 = *reinterpret_cast<const int4 *>(vox2row + (size_t)v * 8);
        const int4 r1 = *reinterpret_cast<const int4 *>(vox2row + (size_t)v * 8 + 4);
        const int rows[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
        uint4 raw[16];
#pragma unroll
        for (int k = 0; k < 8; ++k) {  // issue all 16 row loads before using any; a vertex without a row reads as zeros
            const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
            raw[2 * k] = rows[k] >= 0 ? __ldg(emb + (size_t)rows[k] * 2) : z4;
            raw[2 * k + 1] = rows[k] >= 0 ? __ldg(emb + (size_t)rows[k] * 2 + 1) : z4;
        }
        const Tri t = tri_coords(xyz + i * 3, centres + (size_t)v * 3, voxel_size);
        float acc[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) acc[e] = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float w = corner_weight(t, k);
            float f[16];
            unpack8(raw[2 * k], f);
            unpack8(raw[2 * k + 1], f + 8);
#pragma unroll
            for (int e = 0; e < 16; ++e) acc[e] = __fadd_rn(acc[e], __fmul_rn(w, f[e]));  // (weights * feats).sum(1)
        }
        float4 *o = feats + i * 4;
        o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
        o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
        o[2] = make_float4(acc[8], acc[9], acc[10], acc[11]);
        o[3] = make_float4(acc[12], acc[13], acc[14], acc[15]);
    }
}

// Backward: autograd of the forward above w.r.t. the embedding rows (scatter-add) and xyz (-> pose).
// Consecutive samples of a ray usually sit in the same voxel (step = voxel/2) and therefore scatter to the same 8 rows.  Runs
// of equal voxel ids inside a warp are merged in groups of up to four: lanes at even positions of a run add their right
// neighbour's (already bf16-rounded) contributions with one shuffle per value, lanes at positions 0 mod 4 then add the pair
// sum two lanes to their right and issue the atomics for the group, the other lanes issue none.
__global__ void __launch_bounds__(128) k_gather_bwd(long long M_host, const int32_t *__restrict__ M_dev,
                                                     const float *__restrict__ xyz, const int32_t *__restrict__ vox,
                                                     const float *__restrict__ centres, const int32_t *__restrict__ vox2row,
                                                     const uint4 *__restrict__ emb, float voxel_size,
                                                     const float4 *__restrict__ dfeats, int round_bf16,
                                                     float *__restrict__ grad_emb, float *__restrict__ dxyz_out,
                                                     const int32_t *__restrict__ s_ray, const float *__restrict__ s_depth,
                                                     const float *__restrict__ dir_local, const int32_t *__restrict__ ray_frame,
                                                     int n_frames, float *__restrict__ pose_acc) {
    extern __shared__ float s_acc[];  // [n_frames][12]
    const bool want_pose = pose_acc != nullptr;
    if (want_pose) {
        for (int i = threadIdx.x; i < n_frames * 12; i += blockDim.x) s_acc[i] = 0.f;
        __syncthreads();
    }
    const long long M = M_dev ? min((long long)*M_dev, M_host) : M_host;
    const bool want_x = want_pose || dxyz_out != nullptr;
    const int lane = threadIdx.x & 31;
    for (long long base = (long long)blockIdx.x * blockDim.x; base < M; base += (long long)gridDim.x * blockDim.x) {
        const long long i = base + threadIdx.x;
        const bool active = i < M;
        float gx = 0.f, gy = 0.f, gz = 0.f;
        int frame = -1;
        int v = -1;
        int rows[8];
        float g[16];
        Tri t;
        t.px = t.py = t.pz = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) rows[k] = -1;
#pragma unroll
        for (int e = 0; e < 16; ++e) g[e] = 0.f;
        if (active) {
            v = vox[i];
            const int4 r0 = *reinterpret_cast<const int4 *>(vox2row + (size_t)v * 8);
            const int4 r1 = *reinterpret_cast<const int4 *>(vox2row + (size_t)v * 8 + 4);
            rows[0] = r0.x; rows[1] = r0.y; rows[2] = r0.z; rows[3] = r0.w; rows[4] = r1.x; rows[5] = r1.y; rows[6] = r1.z; rows[7] = r1.w;
            const float4 *gp = dfeats + i * 4;
            const float4 g0 = gp[0], g1 = gp[1], g2 = gp[2], g3 = gp[3];
            g[0] = g0.x; g[1] = g0.y; g[2] = g0.z; g[3] = g0.w; g[4] = g1.x; g[5] = g1.y; g[6] = g1.z; g[7] = g1.w;
            g[8] = g2.x; g[9] = g2.y; g[10] = g2.z; g[11] = g2.w; g[12] = g3.x; g[13] = g3.y; g[14] = g3.z; g[15] = g3.w;
            t = tri_coords(xyz + i * 3, centres + (size_t)v * 3, voxel_size);
        }
        // run structure inside the warp: emitters = positions 0 mod 4 of a run of equal voxel ids
        bool emit = true, take = false, take2 = false;
        if (grad_emb) {
            const int vprev = __shfl_up_sync(0xffffffffu, v, 1);
            const bool head = (lane == 0) || (vprev != v) || (v < 0);
            const unsigned hf = __ballot_sync(0xffffffffu, head);
            const int head_lane = 31 - __clz(hf & (0xffffffffu >> (31 - lane)));
            const int pos = lane - head_lane;
            take = (pos & 1) == 0 && lane < 31 && !((hf >> (lane + 1)) & 1u);   // the right neighbour continues this run
            emit = (pos & 3) == 0;
            take2 = emit && lane < 30 && !((hf >> (lane + 1)) & 3u);   // so does the lane after it (which holds a pair sum)
        }
        const float inv_vs = 1.0f / voxel_size;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float ax = (k & 4) ? t.px : __fsub_rn(1.0f, t.px);
            const float ay = (k & 2) ? t.py : __fsub_rn(1.0f, t.py);
            const float az = (k & 1) ? t.pz : __fsub_rn(1.0f, t.pz);
            const float w = __fmul_rn(__fmul_rn(ax, ay), az);
            const bool has_row = rows[k] >= 0;
            if (grad_emb) {
                // d(emb row): grad_out * w, rounded to bf16 where autograd casts it for a bf16 table
                float c[16];
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    c[e] = has_row ? g[e] * w : 0.f;
                    if (round_bf16) c[e] = nl_round_bf16(c[e]);
                    const float nb = __shfl_down_sync(0xffffffffu, c[e], 1);
                    if (take) c[e] += nb;
                    const float nb2 = __shfl_down_sync(0xffffffffu, c[e], 2);
                    if (take2) c[e] += nb2;
                }
                if (has_row && emit) {
                    float4 *dst = reinterpret_cast<float4 *>(grad_emb + (size_t)rows[k] * 16);
                    atomicAdd(dst + 0, make_float4(c[0], c[1], c[2], c[3]));
                    atomicAdd(dst + 1, make_float4(c[4], c[5], c[6], c[7]));
                    atomicAdd(dst + 2, make_float4(c[8], c[9], c[10], c[11]));
                    atomicAdd(dst + 3, make_float4(c[12], c[13], c[14], c[15]));
                }
            }
            if (want_x && has_row) {
                float f[16];
                unpack8(__ldg(emb + (size_t)rows[k] * 2), f);
                unpack8(__ldg(emb + (size_t)rows[k] * 2 + 1), f + 8);
                float dot = 0.f;  // d loss / d w_k = sum_e grad_out[e] * emb_k[e]
#pragma unroll
                for (int e = 0; e < 16; ++e) dot = fmaf(g[e], f[e], dot);
                gx += dot * ((k & 4) ? 1.f : -1.f) * ay * az;
                gy += dot * ((k & 2) ? 1.f : -1.f) * ax * az;
                gz += dot * ((k & 1) ? 1.f : -1.f) * ax * ay;
            }
        }
        if (active) {
            gx *= inv_vs; gy *= inv_vs; gz *= inv_vs;  // d p / d xyz = 1 / voxel_size
            if (dxyz_out) { dxyz_out[i * 3] = gx; dxyz_out[i * 3 + 1] = gy; dxyz_out[i * 3 + 2] = gz; }
            if (want_pose) frame = ray_frame ? ray_frame[s_ray[i]] : 0;
        }
        if (want_pose) {
            // xyz = t_f + depth * R_f * d_local  =>  dL/dt_f += g,  dL/dR_f[a][b] += g[a] * depth * d_local[b]
            float v12[12];
            if (active) {
                const int r = s_ray[i];
                const float dep = s_depth[i];
                const float lx = dir_local[r * 3] * dep, ly = dir_local[r * 3 + 1] * dep, lz = dir_local[r * 3 + 2] * dep;
                v12[0] = gx; v12[1] = gy; v12[2] = gz;
                v12[3] = gx * lx; v12[4] = gx * ly; v12[5] = gx * lz;
                v12[6] = gy * lx; v12[7] = gy * ly; v12[8] = gy * lz;
                v12[9] = gz * lx; v12[10] = gz * ly; v12[11] = gz * lz;
            } else {
#pragma unroll
                for (int c = 0; c < 12; ++c) v12[c] = 0.f;
            }
            // samples of a warp nearly always share a frame: reduce in the warp, one smem atomic per value
            const unsigned act = __ballot_sync(0xffffffffu, active);
            const int f0 = __shfl_sync(0xffffffffu, frame, act ? (__ffs(act) - 1) : 0);
            const bool uniform = __all_sync(0xffffffffu, !active || frame == f0);
            if (uniform) {
#pragma unroll
                for (int c = 0; c < 12; ++c) {
                    float s = v12[c];
                    for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
                    if ((threadIdx.x & 31) == 0 && act) atomicAdd(&s_acc[f0 * 12 + c], s);
                }
            } else if (active) {
#pragma unroll
                for (int c = 0; c < 12; ++c) atomicAdd(&s_acc[frame * 12 + c], v12[c]);
            }
        }
    }
    if (want_pose) {
        __syncthreads();
        for (int i = threadIdx.x; i < n_frames * 12; i += blockDim.x)
            if (s_acc[i] != 0.f) atomicAdd(&pose_acc[i], s_acc[i]);
    }
}

inline int persistent_blocks(long long M, int threads, int per_sm) {
    long long need = (M + threads - 1) / threads;
    long long cap = (long long)nl_num_sms() * per_sm;
    return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}

}  // namespace

extern "C" int nl_gather_trilinear_fwd(int64_t M, const int32_t *d_M_dev, const float *xyz, const int32_t *vox,
                                       const float *centres, const int32_t *vox2row, const uint16_t *emb, float voxel_size,
                                       float *feats, void *stream) {
    if (M < 0) return nl_set_error("nl_gather_trilinear_fwd: negative M");
    if (M == 0) return NL_OK;
    if (!xyz || !vox || !centres || !vox2row || !emb || !feats) return nl_set_error("nl_gather_trilinear_fwd: null pointer");
    if (!(voxel_size > 0.f)) return nl_set_error("nl_gather_trilinear_fwd: voxel_size must be > 0");
    k_gather_fwd<<<persistent_blocks(M, 128, 16), 128, 0, (cudaStream_t)stream>>>(
        M, d_M_dev, xyz, vox, centres, vox2row, reinterpret_cast<const uint4 *>(emb), voxel_size, reinterpret_cast<float4 *>(feats));
    NL_CHECK_LAUNCH("nl_gather_trilinear_fwd");
    return NL_OK;
}

extern "C" int nl_gather_trilinear_bwd(int64_t M, const int32_t *d_M_dev, const float *xyz, const int32_t *vox,
                                       const float *centres, const int32_t *vox2row, const uint16_t *emb, float voxel_size,
                                       const float *dfeats, int round_bf16, float *grad_emb, float *dxyz,
                                       const int32_t *s_ray, const float *s_depth, const float *ray_dir_local,
                                       const int32_t *ray_frame, int n_frames, float *pose_acc, void *stream) {
    if (M < 0) return nl_set_error("nl_gather_trilinear_bwd: negative M");
    if (M == 0) return NL_OK;
    if (!xyz || !vox || !centres || !vox2row || !emb || !dfeats) return nl_set_error("nl_gather_trilinear_bwd: null pointer");
    if (pose_acc && (!s_ray || !s_depth || !ray_dir_local || n_frames <= 0 || n_frames > 1024))
        return nl_set_error("nl_gather_trilinear_bwd: pose accumulation needs s_ray, s_depth, ray_dir_local, 0 < n_frames <= 1024");
    const size_t smem = pose_acc ? sizeof(float) * 12 * (size_t)n_frames : 0;
    k_gather_bwd<<<persistent_blocks(M, 128, 16), 128, smem, (cudaStream_t)stream>>>(
        M, d_M_dev, xyz, vox, centres, vox2row, reinterpret_cast<const uint4 *>(emb), voxel_size,
        reinterpret_cast<const float4 *>(dfeats), round_bf16, grad_emb, dxyz, s_ray, s_depth, ray_dir_local, ray_frame, n_frames,
        pose_acc);
    NL_CHECK_LAUNCH("nl_gather_trilinear_bwd");
    return NL_OK;
}
