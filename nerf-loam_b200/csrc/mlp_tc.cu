// Tensor-core version of the SDF decoder MLP (16 -> 256 -> 256 -> 1, ReLU) for sm_100a:
// tcgen05.mma kind::tf32 with a 3-term hi/lo split (3xTF32: a*b ~= ah*bh + ah*bl + al*bh, fp32
// accumulation in TMEM), which keeps the result within ~1e-6 of an fp32 evaluation -- single-pass
// TF32/BF16 (1e-3) would break the 1e-5 SDF parity bar.
//
// One persistent CTA per SM, 6 warps:
//   warp 0   producer : streams pre-swizzled weight panels (hi+lo, 64 KB per K-block of 32) from L2 into a
//                       2-stage shared-memory ring with cp.async.bulk (1-D TMA) + mbarrier complete_tx
//   warp 1   MMA      : one elected thread issues tcgen05.mma (M=128 samples, N=256, K=8 per instruction),
//                       releases ring stages with tcgen05.commit; owns the TMEM allocation (512 columns:
//                       D1 = layer-1 accumulator, D2 = layer-2 accumulator)
//   warps 2-5 epilogue: thread = sample row (TMEM lane).  Loads x, and for every K-block of layer 2 pulls 32
//                       columns of D1 out of TMEM (tcgen05.ld), applies bias+ReLU, splits into tf32 hi/lo and
//                       writes the A operand tile straight into the 128B-swizzled K-major layout the tensor
//                       core reads; finally reduces relu(D2 + b1) . w2 + b2 per row.
// Layer 1 (K = 16) runs through the same ring as one extra K-block with 2 k-steps.
// Shared memory: 2 x 64 KB weight stages + 2 x 32 KB activation stages = 192 KB.
#include <cstdlib>
#include <mutex>

#include "nl_cuda.cuh"

namespace tc {

constexpr int TM = 128;               // samples per tile (UMMA M)
constexpr int WN = 256;               // hidden width (UMMA N)
constexpr int PANEL_A = TM * 128;     // 16 KB : 128 rows x 128 B (32 tf32 of K)
constexpr int PANEL_B = WN * 128;     // 32 KB : 256 rows x 128 B
constexpr int STAGE_A = 2 * PANEL_A;  // hi + lo
constexpr int STAGE_B = 2 * PANEL_B;
constexpr int NSTAGE = 2;
constexpr int STEPS_FWD = 9;          // layer 1 + 8 K-blocks of layer 2
constexpr int STEPS_TRAIN = 25;       // + 8 K-blocks of backward layer 2 + 8 of backward layer 1
constexpr int PANEL_B16 = 16 * 128;   // 2 KB: the 16-row panels of backward layer 1
constexpr int SMEM_DATA = NSTAGE * (STAGE_A + STAGE_B);
constexpr int SMEM_TOTAL = SMEM_DATA + 8192 + 1024;  // + biases/barriers/exchange + alignment slack
constexpr int NTHREADS_TRAIN = 320;   // producer warp, MMA warp, 2 groups of 4 epilogue warps
constexpr int NTHREADS = 192;

// byte offset of 16-byte chunk c (0..7) of row r inside a K-major SWIZZLE_128B panel
__host__ __device__ __forceinline__ int panel_off(int r, int c) { return (r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4); }

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ float tf32_rna(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}

// ---- mbarrier helpers -------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("{ .reg .b64 st; mbarrier.arrive.shared::cta.b64 st, [%0]; }" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("{ .reg .b64 st; mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1; }" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30)
// (ignored for swizzled K-major, set to 1), SBO>>4 = 1024>>4 [32,46), version 1 [46,48), layout SWIZZLE_128B = 2 [61,64)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 = 1 [4,6), a/b_format TF32 = 2 [7,10)/[10,13),
// a/b K-major = 0, N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc),
        "r"(accumulate) : "memory");
}
// One lane of a converged warp.  The single-thread roles (MMA issue, bulk copies) run their loops warp-uniformly and
// predicate only the issuing instruction: every operand then lives in uniform registers and the compiler emits a plain
// UTCHMMA / UBLKCP instead of a per-thread serialisation loop (R2UR + ELECT + BRA.U.ANY, ~100 cycles per MMA).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// all MMAs of one K-block: NTERM tf32 terms (hi*hi, hi*lo, lo*hi) x NK k-steps of 8, fully unrolled
template <int NK, int NTERM>
__device__ __forceinline__ void issue_kblock(uint32_t d, uint32_t a_hi, uint32_t b_hi, uint32_t idesc, uint32_t acc) {
    const uint64_t adh = make_desc(a_hi), adl = make_desc(a_hi + PANEL_A), bdh = make_desc(b_hi), bdl = make_desc(b_hi + PANEL_B);
#pragma unroll
    for (int term = 0; term < NTERM; ++term) {
        const uint64_t ad = (term == 2) ? adl : adh, bd = (term == 1) ? bdl : bdh;
#pragma unroll
        for (int ks = 0; ks < NK; ++ks) {
            mma_tf32(d, ad + 2 * ks, bd + 2 * ks, idesc, acc);
            acc = 1u;
        }
    }
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,"
        "%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// Weight panels: the exact shared-memory image (K-major, 128B swizzle, tf32 hi then lo) of every weight
// K-block, laid out contiguously in global memory so one bulk copy fills a ring stage.
//   stage 0       : W0  [256 x 16]  (row j, k = e; only the first 64 B of each 128 B row are meaningful)
//   stage 1 + kb  : W1[:, 32kb : 32kb+32]              forward layer 2
//   stage 9 + jb  : (diag(w2) W1)^T[:, 32jb : 32jb+32] backward layer 2 (d h1 = dsdf * relu'(h2) . diag(w2) W1, see k_mlp_tc_train)
//   stage 17 + kb : W0^T[:, 32kb : 32kb+32] (16 rows)  backward layer 1 (d x  = d h1 . W0)
// ------------------------------------------------------------------------------------------------
__global__ void k_tc_prepare(const float *__restrict__ W0, const float *__restrict__ W1, const float *__restrict__ w2,
                             uint8_t *__restrict__ panels) {
    const int stage = blockIdx.y;                         // 0..24
    const int t = blockIdx.x * blockDim.x + threadIdx.x;  // (row, chunk)
    if (t >= WN * 8) return;
    const int r = t >> 3, c = t & 7;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (stage == 0) {                                     // layer 1:   B[j][e] = W0[j][e]
        if (c < 4) for (int i = 0; i < 4; ++i) v[i] = W0[r * 16 + c * 4 + i];
    } else if (stage <= 8) {                              // layer 2:   B[j][k] = W1[j][k],      k in K-block stage-1
        const int k0 = (stage - 1) * 32 + c * 4;
        for (int i = 0; i < 4; ++i) v[i] = W1[(size_t)r * WN + k0 + i];
    } else if (stage <= 16) {                             // bwd layer 2: B[k][j] = w2[j] W1[j][k], j in K-block stage-9
        const int j0 = (stage - 9) * 32 + c * 4;
        for (int i = 0; i < 4; ++i) v[i] = __fmul_rn(w2[j0 + i], W1[(size_t)(j0 + i) * WN + r]);
    } else {                                              // bwd layer 1: B[e][k] = W0[k][e],    k in K-block stage-17 (16 rows)
        if (r >= 16) return;
        const int k0 = (stage - 17) * 32 + c * 4;
        for (int i = 0; i < 4; ++i) v[i] = W0[(size_t)(k0 + i) * 16 + r];
    }
    float hi[4], lo[4];
    for (int i = 0; i < 4; ++i) { hi[i] = tf32_rna(v[i]); lo[i] = tf32_rna(v[i] - hi[i]); }
    uint8_t *base = panels + (size_t)stage * STAGE_B;
    *reinterpret_cast<float4 *>(base + panel_off(r, c)) = make_float4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<float4 *>(base + PANEL_B + panel_off(r, c)) = make_float4(lo[0], lo[1], lo[2], lo[3]);
}

struct FwdParams {
    long long M_host;
    const int32_t *M_dev;
    const float *feats;       // [M,16]
    const uint8_t *panels;    // 9 stages x 64 KB
    const float *b0, *b1, *w2, *b2;
    float *sdf;
};

__global__ void __launch_bounds__(NTHREADS, 1) k_mlp_tc_fwd(FwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;  // SWIZZLE_128B panels need 1024-byte alignment
    uint8_t *sm = smem_raw + (base - raw);
    const uint32_t sB = base, sA = base + NSTAGE * STAGE_B;
    uint8_t *A_gen = sm + NSTAGE * STAGE_B;        // generic pointer to the activation stages
    float *b0s = reinterpret_cast<float *>(sm + SMEM_DATA);
    float *b1s = b0s + WN;
    float *w2s = b1s + WN;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm + SMEM_DATA + 3 * WN * 4);
    // barriers: 0,1 b_full  2,3 b_empty  4,5 a_full  6,7 a_empty  8 d1_full  9 d2_full  10 d2_empty
    const uint32_t bar0 = smem_u32(bars);
    auto BAR = [&](int i) { return bar0 + 8u * i; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 12);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long M = p.M_dev ? min((long long)*p.M_dev, p.M_host) : p.M_host;
    const long long ntiles = (M + TM - 1) / TM;

    for (int i = tid; i < WN; i += NTHREADS) { b0s[i] = p.b0[i]; b1s[i] = p.b1[i]; w2s[i] = p.w2[i]; }
    if (tid == 0) {
        mbar_init(BAR(0), 1); mbar_init(BAR(1), 1);      // b_full: producer's expect_tx arrive
        mbar_init(BAR(2), 1); mbar_init(BAR(3), 1);      // b_empty: tcgen05.commit
        mbar_init(BAR(4), 4); mbar_init(BAR(5), 4);      // a_full: one arrive per epilogue warp
        mbar_init(BAR(6), 1); mbar_init(BAR(7), 1);      // a_empty: tcgen05.commit
        mbar_init(BAR(8), 1); mbar_init(BAR(9), 1);      // d1_full, d2_full: tcgen05.commit
        mbar_init(BAR(10), 4);                           // d2_empty: one arrive per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: all 512 columns (D1 at column 0, D2 at column 256)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t D1 = tmem, D2 = tmem + 256;

    if (warp == 0) {
        // ===================== producer: weight panels -> ring =====================
        uint32_t it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            for (int step = 0; step < STEPS_FWD; ++step, ++it) {
                const uint32_t s = it & 1, ph = (it >> 1) & 1;
                mbar_wait(BAR(2 + s), ph ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(BAR(0 + s), STAGE_B);
                    const uint8_t *src = p.panels + (size_t)step * STAGE_B;
                    bulk_g2s(sB + s * STAGE_B, src, PANEL_B, BAR(0 + s));
                    bulk_g2s(sB + s * STAGE_B + PANEL_B, src + PANEL_B, PANEL_B, BAR(0 + s));
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (warp-uniform loop, one elected lane issues) =====================
        constexpr uint32_t idesc = make_idesc(TM, WN);
        uint32_t it = 0, tl = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tl) {
            for (int step = 0; step < STEPS_FWD; ++step, ++it) {
                const uint32_t s = it & 1, ph = (it >> 1) & 1;
                if (step == 1) mbar_wait(BAR(10), (tl & 1) ^ 1);   // D2 of the previous tile fully read
                mbar_wait(BAR(0 + s), ph);                          // weights landed
                mbar_wait(BAR(4 + s), ph);                          // activations written
                tc_fence_after();
                const uint32_t a_hi = sA + s * STAGE_A, b_hi = sB + s * STAGE_B;
                if (elect_one()) {
                    if (step == 0) issue_kblock<2, 3>(D1, a_hi, b_hi, idesc, 0u);          // K = 16: 2 k-steps of 8
                    else issue_kblock<4, 3>(D2, a_hi, b_hi, idesc, step == 1 ? 0u : 1u);   // first MMA of a layer overwrites
                    tc_commit(BAR(2 + s));                              // ring stages free once these MMAs retire
                    tc_commit(BAR(6 + s));
                    if (step == 0) tc_commit(BAR(8));                   // D1 complete
                    if (step == STEPS_FWD - 1) tc_commit(BAR(9));       // D2 complete
                }
                __syncwarp();
            }
        }
    } else {
        // ===================== epilogue warps: thread = sample row =====================
        const int q = warp & 3;                       // TMEM lane quarter this warp may access
        const int row = q * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        const float b2 = p.b2[0];
        uint32_t it = 0, tl = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tl) {
            const long long m = tile * TM + row;
            // ---- step 0: x (16 features = 4 chunks) -> A stage ----
            {
                const uint32_t s = it & 1, ph = (it >> 1) & 1;
                mbar_wait(BAR(6 + s), ph ^ 1);
                uint8_t *dst = A_gen + s * STAGE_A;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (m < M) v = *reinterpret_cast<const float4 *>(p.feats + (size_t)m * 16 + c * 4);
                    const float4 hi = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
                    const float4 lo = make_float4(tf32_rna(v.x - hi.x), tf32_rna(v.y - hi.y), tf32_rna(v.z - hi.z), tf32_rna(v.w - hi.w));
                    *reinterpret_cast<float4 *>(dst + panel_off(row, c)) = hi;
                    *reinterpret_cast<float4 *>(dst + PANEL_A + panel_off(row, c)) = lo;
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(4 + s));
                ++it;
            }
            // ---- steps 1..8: h1 K-block kb = relu(D1[:, 32kb:32kb+32] + b0) -> A stage ----
            mbar_wait(BAR(8), tl & 1);
            tc_fence_after();
            for (int kb = 0; kb < 8; ++kb, ++it) {
                const uint32_t s = it & 1, ph = (it >> 1) & 1;
                uint32_t v[32];
                tmem_ld32(D1 + lane_addr + kb * 32, v);
                mbar_wait(BAR(6 + s), ph ^ 1);
                uint8_t *dst = A_gen + s * STAGE_A;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    float h[4], hi[4], lo[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        h[i] = fmaxf(__uint_as_float(v[c * 4 + i]) + b0s[kb * 32 + c * 4 + i], 0.f);
                        hi[i] = tf32_rna(h[i]);
                        lo[i] = tf32_rna(h[i] - hi[i]);
                    }
                    *reinterpret_cast<float4 *>(dst + panel_off(row, c)) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<float4 *>(dst + PANEL_A + panel_off(row, c)) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(4 + s));
            }
            // ---- output layer: sdf = relu(D2 + b1) . w2 + b2 ----
            mbar_wait(BAR(9), tl & 1);
            tc_fence_after();
            float acc4[4] = {0.f, 0.f, 0.f, 0.f};
            for (int cb = 0; cb < 8; ++cb) {
                uint32_t v[32];
                tmem_ld32(D2 + lane_addr + cb * 32, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float h = fmaxf(__uint_as_float(v[i]) + b1s[cb * 32 + i], 0.f);
                    acc4[i & 3] = fmaf(h, w2s[cb * 32 + i], acc4[i & 3]);
                }
            }
            const float acc = (acc4[0] + acc4[1]) + (acc4[2] + acc4[3]);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(BAR(10));
            if (m < M) p.sdf[m] = acc + b2;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}


// ================================================================================================
// Training kernel: forward + loss + backward w.r.t. the input features in one pass per 128-sample tile.
//   steps  0      layer 1            D1 = x . W0^T                      (TMEM cols 0..255)
//          1..8   layer 2            D2 = relu(D1+b0) . W1^T            (TMEM cols 256..511)
//                 epilogue: sdf = relu(D2+b1).w2 + b2, loss terms, d loss/d sdf (all thread-local: thread = sample)
//          9..16  backward layer 2   D3 = relu'(h2) . (diag(w2) W1)     (reuses D1's columns)
//          17..24 backward layer 1   D4 = (dsdf * D3 * relu'(h1)) . W0  (N = 16, reuses D2's first 16 columns) = d loss / d x
// The output layer has ONE unit, so d h2 = dsdf (per sample) x w2 (per column) x relu'(h2) is rank-1 up to the mask:
// the per-sample factor is pulled out of the GEMM (applied when D3 is read back), the per-column factor is folded into
// the weight panels, and the A operand of backward layer 2 is the 0/1 mask itself -- exact in tf32, so that GEMM needs
// two terms (mask x hi, mask x lo) instead of three and no lo panel.  ReLU masks are 2 x 256 bits per thread in registers.
// With WGRAD the kernel writes h1 and dh1 to HBM in 16 KB "panel" blocks [(tile*8 + kblock)][row][32] (bulk copies of the
// A stages) plus the relu'(h2) bits (32 B/sample) and dsdf; the same factorisation lets k_dw1_tc / k_dw0_tc / k_mask_colsum rebuild
// everything that used to need dh2 and h2 panels (see there).
// ================================================================================================
struct TrainParams {
    long long M_host;
    const int32_t *M_dev;
    const float *feats;
    const uint8_t *panels;     // 25 stages x 64 KB
    const float *b0, *b1, *w2, *b2;
    float *sdf, *dfeats;
    const uint8_t *s_flag;
    const float *s_depth;
    const int32_t *s_ray;
    const float *cosv, *gt_depth;
    nl_render_stats *stats;
    float truncation;
    const float *dsdf_ext;
    float *act_h1, *act_dh1;             // WGRAD: panel-major [ntiles*8][128][32]
    float *act_dsdf;                     // WGRAD: d loss / d sdf per sample [ntiles*128]
    uint32_t *act_mask2;                 // WGRAD: relu'(h2) bits per sample [ntiles*128][8], word g*4+kk = columns 32(2kk+g)..+31
    float *gb2;                          // WGRAD
    long long *dbg;                      // optional timeline stamps (NL_TC_TIMELINE=1), else nullptr
};

// registers -> TMEM, 32 lanes x 32 columns per warp (thread = lane/row); completion via tmem_wait_st()
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,"
        "%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
        "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]),
        "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// A operand from TMEM (lane = row, one 32-bit column per tf32 element, K = 8 columns per instruction), B from shared memory
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc),
        "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// smem -> global bulk copy (1-D TMA store) of this warp's rows of an activation panel; one instruction per warp and
// chunk instead of 8 partially-coalesced STG.128 per thread
__device__ __forceinline__ void bulk_s2g(void *gdst, uint32_t ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

__device__ __forceinline__ void st_shared_v4(uint32_t addr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// tf32 hi/lo split of an A-operand value computed in the epilogue.  The tensor core TRUNCATES its fp32 inputs to tf32.  "hi" is
// therefore simply the raw fp32 bits (which also keeps the stored activation panels exact: the hi tile is what gets bulk-copied
// to HBM for the weight-gradient kernels), and lo = x - trunc(x), exact in fp32.  What matters is how lo reaches 11 bits: left
// to the hardware it is truncated too -- an error of up to 2^-21 |x| that always points towards zero, i.e. a BIAS shared by every
// sample.  Gradients that are sums of 10^4..10^5 strongly cancelling per-sample terms (the pose gradient near convergence:
// cancellation ~10^4) turned that into 10^-3 relative error, 100x what fp32 arithmetic gives (measured against an fp64 run of
// the same function, tests/test_gpu_pipeline.py).  Rounding lo to nearest instead (integer add of half an ulp, then mask) makes
// the hardware truncation of lo a no-op and the residual <= 2^-22 |x| with random sign.
__device__ __forceinline__ float tf32_lo_part(float x) {
    const float lo = x - __uint_as_float(__float_as_uint(x) & 0xffffe000u);
    return __uint_as_float((__float_as_uint(lo) + 0x1000u) & 0xffffe000u);
}
// One 128 B row (32 fp32) of an A-operand K-block as hi and lo tiles.  off[c] = swizzled byte offset of chunk c for this thread's
// row (loop invariant).
__device__ __forceinline__ void store_a_row_fast(uint32_t stage, const uint32_t (&off)[8], const float (&h)[32]) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        st_shared_v4(stage + off[c], h[c * 4], h[c * 4 + 1], h[c * 4 + 2], h[c * 4 + 3]);
        st_shared_v4(stage + PANEL_A + off[c], tf32_lo_part(h[c * 4]), tf32_lo_part(h[c * 4 + 1]), tf32_lo_part(h[c * 4 + 2]), tf32_lo_part(h[c * 4 + 3]));
    }
}

// Warp roles (NTHREADS_TRAIN = 320): warps 0-7 epilogue (group g = warp >> 2, TMEM lane quarter q = warp & 3), warp 8
// producer, warp 9 MMA issuer + TMEM owner.  The two single-thread roles get the HIGHEST warp ids: the per-SMSP arbiter
// prefers the highest warp id, so the busy epilogue warps cannot starve the thread that feeds the tensor core.
// Only the forward steps 0..8 take their A operand from the shared-memory activation stages.  The A operands of both backward
// GEMMs come from TMEM: the 0/1 mask of backward layer 2 is written (tcgen05.st) over the dead layer-2 accumulator right where
// each thread read its pre-activations, so those 8 K-blocks need no activation stage, no smem stores and no per-chunk
// hand-shake; the dh1 chunks of backward layer 1 go through two 64-column TMEM slots (hi | lo), one per epilogue group.
// Shared-memory traffic of those 16 steps is the weight panels alone, and the tiny N = 16 MMAs fetch no A tile from smem.
// Every CTA streams each weight stage from L2 itself; backward layer 2 is bound by that stream (64 KB per K-block and SM).
template <bool WGRAD>
__global__ void __launch_bounds__(NTHREADS_TRAIN, 1) k_mlp_tc_train(TrainParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t *sm = smem_raw + (base - raw);
    const uint32_t sB = base, sA = base + NSTAGE * STAGE_B;
    float *b0s = reinterpret_cast<float *>(sm + SMEM_DATA);
    float *b1s = b0s + WN;
    float *w2s = b1s + WN;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm + SMEM_DATA + 3 * WN * 4);
    // barriers: 0,1 b_full  2,3 b_empty  4,5 a_full  6,7 a_empty  8 d1_full  9 d2_full  10 d3_full  11 d4_full  12 d4_empty
    //           14,15 slot_full[g]  16,17 slot_empty[g]  18..25 mask_full[K-block]
    const uint32_t bar0 = smem_u32(bars);
    auto BAR = [&](int i) { return bar0 + 8u * i; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 28);
    float *sdf_part = reinterpret_cast<float *>(sm + SMEM_DATA + 4096);   // [tile parity][group][row]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    long long *dbg = (blockIdx.x == 0) ? p.dbg : nullptr;   // [role 0..3][step 0..24][4 stamps]
#define NL_STAMP(role, step, k) do { if (dbg && tl == 1 && (threadIdx.x & 31) == 0) dbg[((role) * 25 + (step)) * 8 + (k)] = clock64(); } while (0)
    const long long M = p.M_dev ? min((long long)*p.M_dev, p.M_host) : p.M_host;
    const long long ntiles = (M + TM - 1) / TM;

    for (int i = tid; i < WN; i += NTHREADS_TRAIN) { b0s[i] = p.b0[i]; b1s[i] = p.b1[i]; w2s[i] = p.w2[i]; }
    if (tid == 0) {
        mbar_init(BAR(0), 1); mbar_init(BAR(1), 1);
        mbar_init(BAR(2), 1); mbar_init(BAR(3), 1);
        mbar_init(BAR(4), 4); mbar_init(BAR(5), 4);      // a_full: the 4 warps of the group that owns the chunk
        mbar_init(BAR(6), 1); mbar_init(BAR(7), 1);
        mbar_init(BAR(8), 1); mbar_init(BAR(9), 1); mbar_init(BAR(10), 1); mbar_init(BAR(11), 1);
        mbar_init(BAR(12), 4);
        for (int i = 0; i < 8; ++i) mbar_init(BAR(18 + i), 4);   // mask_full[K-block]: the 4 warps of the group that owns it
        mbar_init(BAR(14), 4); mbar_init(BAR(15), 4);    // slot_full: the 4 warps of the group
        mbar_init(BAR(16), 1); mbar_init(BAR(17), 1);    // slot_empty: tcgen05.commit
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 9) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t D1 = tmem, D2 = tmem + 256;   // D3 aliases D1, D4 aliases D2[0:16]
    // mask2 overwrites D2 (all 256 columns) for steps 9..16; dh1 slot g = D2[64 + 64g, +64) (hi | lo) for steps 17..24
    auto SLOT = [&](int g) { return D2 + 64u + 64u * (uint32_t)g; };
    // activation-stage use index: only steps 0..8 of each tile use a stage
    auto AIT = [&](uint32_t tl, int step) { return tl * 9u + (uint32_t)step; };

    if (warp == 8) {
        // ===== producer (warp-uniform loop, one elected lane issues the copies) =====
        uint32_t it = 0, tl = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tl) {
            for (int step = 0; step < STEPS_TRAIN; ++step, ++it) {
                const uint32_t s = it & 1, ph = (it >> 1) & 1;
                const uint32_t bytes = (step < 17) ? PANEL_B : PANEL_B16;
                NL_STAMP(0, step, 0);
                mbar_wait(BAR(2 + s), ph ^ 1);
                NL_STAMP(0, step, 1);
                if (elect_one()) {
                    mbar_expect_tx(BAR(0 + s), 2 * bytes);            // hi + lo
                    const uint8_t *src = p.panels + (size_t)step * STAGE_B;
                    bulk_g2s(sB + s * STAGE_B, src, bytes, BAR(0 + s));
                    bulk_g2s(sB + s * STAGE_B + PANEL_B, src + PANEL_B, bytes, BAR(0 + s));
                }
                __syncwarp();
            }
        }
    } else if (warp == 9) {
        // ===== MMA issuer (warp-uniform loop, one elected lane issues) =====
        constexpr uint32_t idesc256 = make_idesc(TM, WN), idesc16 = make_idesc(TM, 16);
        uint32_t it = 0, tl = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tl) {
            for (int step = 0; step < STEPS_TRAIN; ++step, ++it) {
                const uint32_t s = it & 1, ph = (it >> 1) & 1;
                NL_STAMP(1, step, 0);
                if (step == 1) mbar_wait(BAR(12), (tl & 1) ^ 1);   // D4 (in D2's columns) of the previous tile fully read
                mbar_wait(BAR(0 + s), ph);
                NL_STAMP(1, step, 1);
                const uint32_t b_hi = sB + s * STAGE_B;
                if (step <= 8) {
                    const uint32_t ai = AIT(tl, step), as = ai & 1, aph = (ai >> 1) & 1;
                    mbar_wait(BAR(4 + as), aph);
                    NL_STAMP(1, step, 2);
                    tc_fence_after();
                    const uint32_t a_hi = sA + as * STAGE_A;
                    if (elect_one()) {
                        if (step == 0) issue_kblock<2, 3>(D1, a_hi, b_hi, idesc256, 0u);                      // layer 1 (K = 16)
                        else issue_kblock<4, 3>(D2, a_hi, b_hi, idesc256, step == 1 ? 0u : 1u);               // layer 2
                        tc_commit(BAR(2 + s));
                        tc_commit(BAR(6 + as));
                        if (step == 0) tc_commit(BAR(8));
                        if (step == 8) tc_commit(BAR(9));
                    }
                } else if (step <= 16) {
                    // ---- backward layer 2: A = mask2 columns of K-block jb in TMEM (0/1, exact in tf32: no lo term) ----
                    mbar_wait(BAR(18 + (step - 9)), tl & 1);
                    NL_STAMP(1, step, 2);
                    tc_fence_after();
                    const uint32_t a_t = D2 + (uint32_t)(step - 9) * 32u;
                    if (elect_one()) {
                        const uint64_t bdh = make_desc(b_hi), bdl = make_desc(b_hi + PANEL_B);
                        uint32_t acc = step == 9 ? 0u : 1u;
#pragma unroll
                        for (int term = 0; term < 2; ++term) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                mma_tf32_ts(D1, a_t + 8 * ks, (term ? bdl : bdh) + 2 * ks, idesc256, acc);
                                acc = 1u;
                            }
                        }
                        tc_commit(BAR(2 + s));
                        if (step == 16) tc_commit(BAR(10));
                    }
                } else {
                    // ---- backward layer 1 (N = 16): A = dh1 chunk (hi | lo) in the TMEM slot of the group that owns K-block kb ----
                    const int kb = step - 17, g = kb & 1;
                    const uint32_t u = tl * 4u + (uint32_t)(kb >> 1);
                    mbar_wait(BAR(14 + g), u & 1);
                    NL_STAMP(1, step, 2);
                    tc_fence_after();
                    const uint32_t a_t = SLOT(g);
                    if (elect_one()) {
                        const uint64_t bdh = make_desc(b_hi), bdl = make_desc(b_hi + PANEL_B);
                        uint32_t acc = step == 17 ? 0u : 1u;
#pragma unroll
                        for (int term = 0; term < 3; ++term) {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                mma_tf32_ts(D2, a_t + (term == 2 ? 32u : 0u) + 8 * ks, (term == 1 ? bdl : bdh) + 2 * ks, idesc16, acc);
                                acc = 1u;
                            }
                        }
                        tc_commit(BAR(2 + s));
                        tc_commit(BAR(16 + g));
                        if (step == 24) tc_commit(BAR(11));
                    }
                }
                __syncwarp();
                NL_STAMP(1, step, 3);
            }
        }
    } else {
        // ===== epilogue: 2 groups x 4 warps; thread = (sample row, group); group g owns the K-blocks with (kb & 1) == g =====
        const int q = warp & 3;                        // TMEM lane quarter this warp may access
        const int g = warp >> 2;                       // 0: warps 0-3, 1: warps 4-7
        const int row = q * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        uint32_t offc[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) offc[c] = (uint32_t)panel_off(row, c);
        const float b2 = p.b2[0];
        float g_fs = 0.f, g_sdf = 0.f;
        if (!p.dsdf_ext) { g_fs = p.stats->g_fs; g_sdf = p.stats->g_sdf; }
        double loss_fs = 0.0, loss_sdf = 0.0;
        float gb2r = 0.f;
        // per-sample inputs of the next tile are fetched one tile ahead (their latency hides behind a whole tile)
        float4 xn[4];
        uint32_t fl_n = 0u;
        float z_n = 0.f, dgt_n = 0.f, dext_n = 0.f;
        auto prefetch = [&](long long tile) {
            const long long mm = tile * TM + row;
            const bool lv = tile < ntiles && mm < M;
#pragma unroll
            for (int c = 0; c < 4; ++c) xn[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            fl_n = 0u; z_n = 0.f; dgt_n = 0.f; dext_n = 0.f;
            if (lv) {
                if (g == 0) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) xn[c] = *reinterpret_cast<const float4 *>(p.feats + (size_t)mm * 16 + c * 4);
                }
                if (p.dsdf_ext) {
                    dext_n = p.dsdf_ext[mm];
                } else {
                    fl_n = p.s_flag[mm];
                    const int r = p.s_ray[mm];
                    z_n = __fmul_rn(p.s_depth[mm], p.cosv ? p.cosv[r] : 1.0f);
                    dgt_n = p.gt_depth[r];
                }
            }
        };
        prefetch(blockIdx.x);
        uint32_t tl = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tl) {
            const long long m = tile * TM + row;
            const bool live = m < M;
            const uint32_t fl = fl_n;
            const float z = z_n, dgt = dgt_n, dext = dext_n;
            uint32_t mask1[4], mask2[4];
            // ---- step 0: x -> A (group 0).  The activation stages are idle during the backward steps, so every later tile's x
            // is staged at the end of the tile before it (below) ----
            if (g == 0 && tl == 0) {
                const uint32_t it = AIT(tl, 0), s = it & 1, ph = (it >> 1) & 1;
                if (WGRAD) { if (lane == 0) bulk_wait_read(); __syncwarp(); }
                mbar_wait(BAR(6 + s), ph ^ 1);
                const uint32_t dst = sA + s * STAGE_A;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 v = xn[c];
                    const float4 hi = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
                    st_shared_v4(dst + offc[c], hi.x, hi.y, hi.z, hi.w);
                    st_shared_v4(dst + PANEL_A + offc[c], tf32_rna(v.x - hi.x), tf32_rna(v.y - hi.y), tf32_rna(v.z - hi.z), tf32_rna(v.w - hi.w));
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(4 + s));
            }
            // ---- steps 1..8: h1 chunks ----
            mbar_wait(BAR(8), tl & 1);
            tc_fence_after();
#pragma unroll 1
            for (int kk = 0; kk < 4; ++kk) {
                const int kb = 2 * kk + g;
                const uint32_t it = AIT(tl, 1 + kb), s = it & 1, ph = (it >> 1) & 1;
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 0);
                uint32_t v[32];
                tmem_ld32(D1 + lane_addr + kb * 32, v);
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 4);
                float h[32];
                uint32_t mk = 0u;
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float t = __uint_as_float(v[i]) + b0s[kb * 32 + i];
                    const bool on = t > 0.f;
                    h[i] = on ? t : 0.f;
                    mk |= on ? (1u << i) : 0u;
                }
                mask1[kk] = mk;
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 5);
                if (WGRAD) { if (lane == 0) bulk_wait_read(); __syncwarp(); }   // previous panel store of this warp left the stage
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 1);
                mbar_wait(BAR(6 + s), ph ^ 1);
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 2);
                store_a_row_fast(sA + s * STAGE_A, offc, h);
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 6);
                fence_proxy_async();
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 7);
                __syncwarp();
                if (WGRAD && lane == 0) bulk_s2g(p.act_h1 + ((size_t)(tile * 8 + kb) * TM + q * 32) * 32, sA + s * STAGE_A + q * 4096, 4096);
                if (lane == 0) mbar_arrive(BAR(4 + s));
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 1 + kb, 3);
            }
            // ---- output layer + loss: each group reduces its 4 column blocks, partial sums exchanged through smem ----
            if (q == 0 && lane == 0) NL_STAMP(2 + g, 0, 0);
            mbar_wait(BAR(9), tl & 1);
            tc_fence_after();
            if (q == 0 && lane == 0) NL_STAMP(2 + g, 0, 1);
            float acc4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
            for (int kk = 0; kk < 4; ++kk) {
                const int cb = 2 * kk + g;
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 0, 2 + kk);
                uint32_t v[32];
                tmem_ld32(D2 + lane_addr + cb * 32, v);
                uint32_t mk = 0u;
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float t = __uint_as_float(v[i]) + b1s[cb * 32 + i];
                    const bool on = t > 0.f;
                    mk |= on ? (1u << i) : 0u;
                    acc4[i & 3] = fmaf(on ? t : 0.f, w2s[cb * 32 + i], acc4[i & 3]);
                    v[i] = on ? 0x3f800000u : 0u;               // 1.0f / 0.0f: the A operand of backward layer 2
                }
                mask2[kk] = mk;
                // same lanes / columns this thread just read; backward layer 2 may start on this K-block right away
                tmem_st32(D2 + lane_addr + cb * 32, v);
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(18 + cb));
            }
            float *part = sdf_part + (tl & 1) * 256;
            part[g * 128 + row] = (acc4[0] + acc4[1]) + (acc4[2] + acc4[3]);
            if (q == 0 && lane == 0) NL_STAMP(2 + g, 0, 6);
            asm volatile("bar.sync 1, 256;" ::: "memory");          // the 8 epilogue warps
            if (q == 0 && lane == 0) NL_STAMP(2 + g, 0, 7);
            const float sdf = (part[row] + part[128 + row]) + b2;
            float dsdf = 0.f;
            if (live) {
                if (g == 0) p.sdf[m] = sdf;
                if (p.dsdf_ext) {
                    dsdf = dext;
                } else {
                    if (fl & 1u) {
                        const float e = sdf - 1.0f;
                        if (g == 0) loss_fs += (double)e * (double)e;
                        dsdf += 2.0f * g_fs * e;
                    }
                    if (fl & 2u) {
                        const float e = __fsub_rn(__fadd_rn(z, __fmul_rn(sdf, p.truncation)), dgt);
                        if (g == 0) loss_sdf += (double)e * (double)e;
                        dsdf += 2.0f * g_sdf * p.truncation * e;
                    }
                }
            }
            if (WGRAD) {
                if (g == 0) {
                    gb2r += dsdf;
                    p.act_dsdf[tile * TM + row] = dsdf;
                }
                *reinterpret_cast<uint4 *>(p.act_mask2 + (size_t)(tile * TM + row) * 8 + g * 4) = make_uint4(mask2[0], mask2[1], mask2[2], mask2[3]);
            }
            // steps 9..16 (backward layer 2) need nothing more from the epilogue: their 0/1 mask operand is already in TMEM
            prefetch(tile + gridDim.x);                 // next tile's x / loss inputs: a whole backward pass to arrive
            // ---- steps 17..24: dh1 (masked) chunks from D3 ----
            mbar_wait(BAR(10), tl & 1);
            tc_fence_after();
#pragma unroll 1
            for (int kk = 0; kk < 4; ++kk) {
                const int kb = 2 * kk + g;
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 17 + kb, 0);
                uint32_t v[32];
                tmem_ld32(D1 + lane_addr + kb * 32, v);
                float h[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) h[i] = ((mask1[kk] >> i) & 1u) ? dsdf * __uint_as_float(v[i]) : 0.f;
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 17 + kb, 1);
                // hi = the fp32 bits (the tensor core truncates to tf32), lo = x - trunc(x) rounded to tf32 (tf32_lo_part); both into this group's TMEM slot
                const uint32_t u = tl * 4u + (uint32_t)kk;
                mbar_wait(BAR(16 + g), (u & 1) ^ 1);               // the MMAs of this group's previous chunk retired
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 17 + kb, 2);
                uint32_t w[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) w[i] = __float_as_uint(h[i]);
                tmem_st32(SLOT(g) + lane_addr, w);
#pragma unroll
                for (int i = 0; i < 32; ++i) w[i] = __float_as_uint(tf32_lo_part(h[i]));
                tmem_st32(SLOT(g) + lane_addr + 32, w);
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(14 + g));
                if (WGRAD) {   // panel store for gW0 / gb0: staged through the activation stage this group used in steps 1..8
                    const uint32_t sg = sA + ((tl + 1u + (uint32_t)g) & 1u) * STAGE_A;
                    if (lane == 0) bulk_wait_read();
                    __syncwarp();
#pragma unroll
                    for (int c = 0; c < 8; ++c) st_shared_v4(sg + offc[c], h[c * 4], h[c * 4 + 1], h[c * 4 + 2], h[c * 4 + 3]);
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) bulk_s2g(p.act_dh1 + ((size_t)(tile * 8 + kb) * TM + q * 32) * 32, sg + q * 4096, 4096);
                }
                if (q == 0 && lane == 0) NL_STAMP(2 + g, 17 + kb, 3);
            }
            if (WGRAD) {   // stages change hands between the groups at the tile boundary: all panel stores must have left smem
                if (lane == 0) bulk_wait_read();
                asm volatile("bar.sync 2, 256;" ::: "memory");
            }
            // x of the next tile (prefetched above) -> its activation stage now: the MMA warp can issue the next layer 1
            // right behind this tile's last backward MMAs instead of waiting for the d x read-back below
            if (g == 0 && tile + gridDim.x < ntiles) {
                const uint32_t it = AIT(tl + 1, 0), s = it & 1, ph = (it >> 1) & 1;
                if (WGRAD) { if (lane == 0) bulk_wait_read(); __syncwarp(); }
                mbar_wait(BAR(6 + s), ph ^ 1);
                const uint32_t dst = sA + s * STAGE_A;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 v = xn[c];
                    const float4 hi = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
                    st_shared_v4(dst + offc[c], hi.x, hi.y, hi.z, hi.w);
                    st_shared_v4(dst + PANEL_A + offc[c], tf32_rna(v.x - hi.x), tf32_rna(v.y - hi.y), tf32_rna(v.z - hi.z), tf32_rna(v.w - hi.w));
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(4 + s));
            }
            // ---- d loss / d x (group 0) ----
            if (g == 0) {
                mbar_wait(BAR(11), tl & 1);
                tc_fence_after();
                uint32_t v[16];
                tmem_ld16(D2 + lane_addr, v);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(BAR(12));
                if (live) {
                    float4 *o = reinterpret_cast<float4 *>(p.dfeats + (size_t)m * 16);
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        o[c] = make_float4(__uint_as_float(v[c * 4]), __uint_as_float(v[c * 4 + 1]), __uint_as_float(v[c * 4 + 2]),
                                           __uint_as_float(v[c * 4 + 3]));
                }
            }
        }
        if (!p.dsdf_ext && g == 0) {
            for (int off = 16; off > 0; off >>= 1) {
                loss_fs += __shfl_down_sync(0xffffffffu, loss_fs, off);
                loss_sdf += __shfl_down_sync(0xffffffffu, loss_sdf, off);
            }
            if (lane == 0) {
                if (loss_fs != 0.0) atomicAdd(&p.stats->fs_sum, loss_fs);
                if (loss_sdf != 0.0) atomicAdd(&p.stats->sdf_sum, loss_sdf);
            }
        }
        if (WGRAD && g == 0) {
            for (int off = 16; off > 0; off >>= 1) gb2r += __shfl_down_sync(0xffffffffu, gb2r, off);
            if (lane == 0) atomicAdd(p.gb2, gb2r);
        }
        if (WGRAD && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // panel stores complete before exit
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 9) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

// ================================================================================================
// Weight gradients of the hidden and output layers on tensor cores.  With m2 = relu'(h2) (0/1) and d = dsdf:
//   G[j][k]  = sum_s m2[s][j] * (d[s] h1[s][k])                 (256 x 256, fp32 in TMEM: 2 accumulators x 256 columns)
//   gW1[j][k] += w2[j] G[j][k]                                   (= sum_s dh2[s][j] h1[s][k])
//   gW2[j]    += sum_k W1[j][k] G[j][k]   (+ b1[j] c[j], added by k_mask_colsum;  = sum_s d[s] h2[s][j] because
//                                            h2 = m2 * (h1 . W1^T + b1), c[j] = sum_s m2[s][j] d[s])
//   K = samples, streamed in K-blocks of 16 rows.  Both operands are MN-major (SWIZZLE_128B_BASE32B, the only layout
//   tcgen05 takes for MN-major tf32).  Per K-block the producer bulk-copies the 16 rows of the h1 panels (16 KB, the
//   K-major image k_mlp_tc_train stored), 512 B of mask bits and 64 B of dsdf; 8 converter warps expand the bits into
//   the 0/1 A operand (exact in tf32: one term fewer than 3xTF32) and write hi/lo of d*h1 as the B operand.
//   4-deep raw ring (17 KB stages) + 3-deep converted ring (48 KB stages), 219 KB of shared memory.  Every CTA finally adds
//   its partial sums with atomics.
// ================================================================================================
constexpr int DW_KROWS = 16;
constexpr int DW_PANEL = DW_KROWS * 128;        // 2 KB: 16 sample rows x 128 B
constexpr int DW_OPER = 8 * DW_PANEL;           // 16 KB: all 256 columns of one operand
constexpr int DW_BITS = DW_KROWS * 32;          // 512 B of relu'(h2) bits
constexpr int DW_RAW = DW_OPER + 1024;          // h1 raw (K-major SWIZZLE_128B image as stored in HBM) | bits | dsdf
constexpr int DW_CONV = 3 * DW_OPER;            // 48 KB: A mask | B hi | B lo (MN-major SWIZZLE_128B_BASE32B)
constexpr int DW_NCW = 8;                       // converter warps of k_dw1_tc and k_dw0_tc (warps 2..9)
constexpr int DW_NCT = 32 * DW_NCW;             // converter threads
constexpr int DW_THREADS = 64 + DW_NCT;         // + producer warp and MMA warp
constexpr int DW_NRAW = 4, DW_NCONV = 3;        // ring depths of k_dw1_tc
constexpr int DW_SMEM = DW_NRAW * DW_RAW + DW_NCONV * DW_CONV + 1024 + 1024;

// MN-major SWIZZLE_128B_BASE32B descriptor (layout type 1): LBO = byte stride between 32-element MN groups (= one 2 KB
// panel), SBO = byte stride between groups of 4 K rows (512 B); one k-step (K = 8) spans two such groups
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(DW_PANEL >> 4) << 16) | (32ull << 32) | (1ull << 46) | (1ull << 61);
}

__global__ void __launch_bounds__(DW_THREADS, 1) k_dw1_tc(long long M_host, const int32_t *__restrict__ M_dev, const uint32_t *__restrict__ act_mask2,
                                                       const float *__restrict__ act_dsdf, const float *__restrict__ act_h1,
                                                       const float *__restrict__ W1, const float *__restrict__ w2, float *__restrict__ gW1,
                                                       float *__restrict__ gW2) {
    constexpr int NRAW = DW_NRAW, NCONV = DW_NCONV;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t *sm = smem_raw + (base - raw);
    // converted stages first: their operand tiles need 1024-byte alignment, the raw stages only 16
    const uint32_t sConv = base, sRaw = base + NCONV * DW_CONV;
    uint8_t *conv_gen = sm, *raw_gen = sm + NCONV * DW_CONV;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm + NCONV * DW_CONV + NRAW * DW_RAW);
    // barriers: 0..3 raw_full  4..7 raw_empty  8..10 conv_full  11..13 conv_empty  14 d_full
    const uint32_t bar0 = smem_u32(bars);
    auto BAR = [&](int i) { return bar0 + 8u * i; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long M = M_dev ? min((long long)*M_dev, M_host) : M_host;
    const long long nkb = ((M + TM - 1) / TM) * (TM / DW_KROWS);   // K-blocks of 16 rows (whole tiles: padded rows have dsdf = 0)
    if (tid == 0) {
        for (int i = 0; i < NRAW; ++i) { mbar_init(BAR(i), 1); mbar_init(BAR(4 + i), DW_NCW); }
        for (int i = 0; i < NCONV; ++i) { mbar_init(BAR(8 + i), DW_NCW); mbar_init(BAR(11 + i), 1); }
        mbar_init(BAR(14), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const bool has_work = (long long)blockIdx.x < nkb;

    if (warp == 0) {
        uint32_t it = 0;
        for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x, ++it) {
            const uint32_t s = it % NRAW, ph = (it / NRAW) & 1;
            mbar_wait(BAR(4 + s), ph ^ 1);
            if (elect_one()) {
                mbar_expect_tx(BAR(0 + s), DW_OPER + DW_BITS + DW_KROWS * 4);
                const long long tile = kb >> 3;
                const int r0 = (int)(kb & 7) * DW_KROWS;
                const uint32_t dst = sRaw + s * DW_RAW;
#pragma unroll
                for (int pnl = 0; pnl < 8; ++pnl)
                    bulk_g2s(dst + pnl * DW_PANEL, act_h1 + ((size_t)(tile * 8 + pnl) * TM + r0) * 32, DW_PANEL, BAR(0 + s));
                bulk_g2s(dst + DW_OPER, act_mask2 + (size_t)(tile * TM + r0) * 8, DW_BITS, BAR(0 + s));
                bulk_g2s(dst + DW_OPER + DW_BITS, act_dsdf + tile * TM + r0, DW_KROWS * 4, BAR(0 + s));
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        if (has_work) {
            // M = 128 (rows j), N = 256 (columns k), both operands MN-major (bits 15, 16)
            constexpr uint32_t idesc = make_idesc(TM, WN) | (1u << 15) | (1u << 16);
            uint32_t it = 0;
            for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x, ++it) {
                const uint32_t s = it % NCONV, ph = (it / NCONV) & 1;
                mbar_wait(BAR(8 + s), ph);
                tc_fence_after();
                const uint32_t a_m = sConv + s * DW_CONV, b_hi = a_m + DW_OPER, b_lo = a_m + 2 * DW_OPER;
                if (elect_one()) {
#pragma unroll
                    for (int jt = 0; jt < 2; ++jt) {
                        uint32_t acc = it > 0 ? 1u : 0u;
#pragma unroll
                        for (int term = 0; term < 2; ++term) {
                            const uint32_t a0 = a_m + jt * 4 * DW_PANEL;
                            const uint32_t b0 = (term == 1 ? b_lo : b_hi);
#pragma unroll
                            for (int ks = 0; ks < DW_KROWS / 8; ++ks) {
                                mma_tf32(tmem + jt * 256, make_desc_mn(a0 + ks * 1024), make_desc_mn(b0 + ks * 1024), idesc, acc);
                                acc = 1u;
                            }
                        }
                    }
                    tc_commit(BAR(11 + s));
                }
                __syncwarp();
            }
            if (elect_one()) tc_commit(BAR(14));
            __syncwarp();
        }
    } else {
        // converters (256 threads).  Stored h1 image: K-major SWIZZLE_128B (16 B chunk c of row r at c ^ (r & 7)); operand
        // tiles: MN-major SWIZZLE_128B_BASE32B (32 B chunk c of row r at c ^ (r & 3)).  hi = the fp32 bits of d*h1
        // (truncated to tf32 by the hardware), lo = tf32(x - trunc(x)).
        constexpr int NCT = DW_NCT;
        const int ct = tid - 64;
        // mask expansion: one (column block, sample row) per group of NCT/128 threads, 8 / (NCT/128) float4 each
        constexpr int MSPLIT = NCT / 128;
        const int m_pair = ct / MSPLIT, m_part = ct % MSPLIT;
        const int m_pnl = m_pair >> 4, m_lr = m_pair & 15;
        const int m_word = (m_pnl & 1) * 4 + (m_pnl >> 1);         // storage order of k_mlp_tc_train: [group][kk]
        uint32_t it = 0;
        for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x, ++it) {
            const uint32_t rs = it % NRAW, rph = (it / NRAW) & 1;
            const uint32_t cs = it % NCONV, cph = (it / NCONV) & 1;
            mbar_wait(BAR(0 + rs), rph);          // raw tiles landed
            mbar_wait(BAR(11 + cs), cph ^ 1);     // converted stage free (its MMAs retired)
            const uint8_t *rawp = raw_gen + rs * DW_RAW;
            const float4 *src = reinterpret_cast<const float4 *>(rawp);
            const uint32_t *bits = reinterpret_cast<const uint32_t *>(rawp + DW_OPER);
            const float *dsd = reinterpret_cast<const float *>(rawp + DW_OPER + DW_BITS);
            float4 *am = reinterpret_cast<float4 *>(conv_gen + cs * DW_CONV);
            float4 *hi = reinterpret_cast<float4 *>(conv_gen + cs * DW_CONV + DW_OPER);
            float4 *lo = reinterpret_cast<float4 *>(conv_gen + cs * DW_CONV + 2 * DW_OPER);
            {
                const uint32_t mk = bits[m_lr * 8 + m_word];
#pragma unroll
                for (int cc = 0; cc < 8 / MSPLIT; ++cc) {
                    const int c16 = m_part * (8 / MSPLIT) + cc;
                    const int d16 = (((c16 >> 1) ^ (m_lr & 3)) << 1) | (c16 & 1);
                    am[(m_pnl << 7) | (m_lr << 3) | d16] =
                        make_float4((mk >> (4 * c16)) & 1u ? 1.f : 0.f, (mk >> (4 * c16 + 1)) & 1u ? 1.f : 0.f,
                                    (mk >> (4 * c16 + 2)) & 1u ? 1.f : 0.f, (mk >> (4 * c16 + 3)) & 1u ? 1.f : 0.f);
                }
            }
#pragma unroll 4
            for (int f = ct; f < DW_OPER / 16; f += NCT) {        // f: float4 index = (panel, local row, stored chunk)
                const int pnl = f >> 7, lr = (f >> 3) & 15, p16 = f & 7;
                const int c16 = p16 ^ (lr & 7);                   // logical 16 B chunk (r0 is a multiple of 16: r & 7 == lr & 7)
                const int d16 = (((c16 >> 1) ^ (lr & 3)) << 1) | (c16 & 1);
                const float d = dsd[lr];
                float4 v = src[f];
                v.x *= d; v.y *= d; v.z *= d; v.w *= d;
                float4 l;
                l.x = tf32_rna(v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u));
                l.y = tf32_rna(v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u));
                l.z = tf32_rna(v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u));
                l.w = tf32_rna(v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u));
                const int o = (pnl << 7) | (lr << 3) | d16;
                hi[o] = v;
                lo[o] = l;
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) { mbar_arrive(BAR(8 + cs)); mbar_arrive(BAR(4 + rs)); }
        }
        // epilogue: thread = row j of each accumulator; add the CTA's partial sums into gW1 (scaled by w2[j]) and gW2
        if (has_work) {
            mbar_wait(BAR(14), 0);
            tc_fence_after();
            const int q = warp & 3;
            const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
            // each accumulator half is drained by its own 4 converter warps.  All CTAs finish at about the same time: start
            // each one at a different column block so the 148 partial sums do not hammer the same L2 lines simultaneously.
            const int jt = (warp - 2) >> 2;
            const int j = jt * 128 + q * 32 + lane;
            const float w2j = w2[j];
            float dot = 0.f;
            for (int cc = 0; cc < 8; ++cc) {
                const int cb = (cc + blockIdx.x) & 7;
                uint32_t v[32];
                tmem_ld32(tmem + lane_addr + jt * 256 + cb * 32, v);
                float4 *o = reinterpret_cast<float4 *>(gW1 + (size_t)j * WN + cb * 32);
                const float4 *wr = reinterpret_cast<const float4 *>(W1 + (size_t)j * WN + cb * 32);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float4 w = wr[c];
                    const float g0 = __uint_as_float(v[c * 4]), g1 = __uint_as_float(v[c * 4 + 1]), g2 = __uint_as_float(v[c * 4 + 2]),
                                g3 = __uint_as_float(v[c * 4 + 3]);
                    dot = fmaf(w.x, g0, fmaf(w.y, g1, fmaf(w.z, g2, fmaf(w.w, g3, dot))));
                    atomicAdd(o + c, make_float4(w2j * g0, w2j * g1, w2j * g2, w2j * g3));
                }
            }
            atomicAdd(gW2 + j, dot);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

// ================================================================================================
// Weight gradient of the first layer on tensor cores:  gW0[k][e] += sum_s dh1[s][k] x[s][e],  gb0[k] += sum_s dh1[s][k]
//   Same streaming skeleton as k_dw1_tc (K = samples in K-blocks of 16 rows, MN-major operands).  A = dh1^T from the
//   stored panels (hi = fp32 bits, lo = x - trunc(x)), B = one 32-column panel [x (16) | 1 | 0 ...] (hi/lo), so column 16 of
//   the accumulator is the bias gradient.  D = 256 x 32 fp32 in TMEM (2 x 32 columns), 3 tf32 terms, N = 32 MMAs.
// ================================================================================================
constexpr int D0_RAW = DW_OPER + 1024;          // dh1 raw (16 KB) | x rows (16 x 64 B)
constexpr int D0_CONV = 2 * DW_OPER + 2 * DW_PANEL;   // A hi | A lo | B hi | B lo = 36 KB
constexpr int D0_NRAW = 4, D0_NCONV = 4;        // ring depths: 219 KB of shared memory
constexpr int D0_SMEM = D0_NRAW * D0_RAW + D0_NCONV * D0_CONV + 1024 + 1024;

__global__ void __launch_bounds__(DW_THREADS, 1) k_dw0_tc(long long M_host, const int32_t *__restrict__ M_dev, const float *__restrict__ act_dh1,
                                                       const float *__restrict__ feats, float *__restrict__ gW0, float *__restrict__ gb0) {
    constexpr int NRAW = D0_NRAW, NCONV = D0_NCONV;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t *sm = smem_raw + (base - raw);
    const uint32_t sConv = base, sRaw = base + NCONV * D0_CONV;
    uint8_t *conv_gen = sm, *raw_gen = sm + NCONV * D0_CONV;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm + NCONV * D0_CONV + NRAW * D0_RAW);
    // barriers: 0..3 raw_full  4..7 raw_empty  8..11 conv_full  12..15 conv_empty  16 d_full
    const uint32_t bar0 = smem_u32(bars);
    auto BAR = [&](int i) { return bar0 + 8u * i; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 18);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long M = M_dev ? min((long long)*M_dev, M_host) : M_host;
    const long long nkb = ((M + TM - 1) / TM) * (TM / DW_KROWS);
    if (tid == 0) {
        for (int i = 0; i < NRAW; ++i) { mbar_init(BAR(i), 1); mbar_init(BAR(4 + i), DW_NCW); }
        for (int i = 0; i < NCONV; ++i) { mbar_init(BAR(8 + i), DW_NCW); mbar_init(BAR(12 + i), 1); }
        mbar_init(BAR(16), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(64u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const bool has_work = (long long)blockIdx.x < nkb;

    if (warp == 0) {
        uint32_t it = 0;
        for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x, ++it) {
            const uint32_t s = it % NRAW, ph = (it / NRAW) & 1;
            mbar_wait(BAR(4 + s), ph ^ 1);
            if (elect_one()) {
                const long long tile = kb >> 3;
                const int r0 = (int)(kb & 7) * DW_KROWS;
                const long long left = M - (tile * TM + r0);                       // feature rows that exist (the panels are tile-padded,
                const uint32_t xrows = left >= DW_KROWS ? DW_KROWS : (left > 0 ? (uint32_t)left : 0u);   // the feature array is not)
                mbar_expect_tx(BAR(0 + s), DW_OPER + xrows * 64);
                const uint32_t dst = sRaw + s * D0_RAW;
#pragma unroll
                for (int pnl = 0; pnl < 8; ++pnl)
                    bulk_g2s(dst + pnl * DW_PANEL, act_dh1 + ((size_t)(tile * 8 + pnl) * TM + r0) * 32, DW_PANEL, BAR(0 + s));
                if (xrows) bulk_g2s(dst + DW_OPER, feats + (size_t)(tile * TM + r0) * 16, xrows * 64, BAR(0 + s));
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        if (has_work) {
            constexpr uint32_t idesc = make_idesc(TM, 32) | (1u << 15) | (1u << 16);   // both operands MN-major
            uint32_t it = 0;
            for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x, ++it) {
                const uint32_t s = it % NCONV, ph = (it / NCONV) & 1;
                mbar_wait(BAR(8 + s), ph);
                tc_fence_after();
                const uint32_t a_hi = sConv + s * D0_CONV, a_lo = a_hi + DW_OPER, b_hi = a_hi + 2 * DW_OPER, b_lo = b_hi + DW_PANEL;
                if (elect_one()) {
#pragma unroll
                    for (int jt = 0; jt < 2; ++jt) {
                        uint32_t acc = it > 0 ? 1u : 0u;
#pragma unroll
                        for (int term = 0; term < 3; ++term) {
                            const uint32_t a0 = (term == 2 ? a_lo : a_hi) + jt * 4 * DW_PANEL;
                            const uint32_t b0 = (term == 1 ? b_lo : b_hi);
#pragma unroll
                            for (int ks = 0; ks < DW_KROWS / 8; ++ks) {
                                mma_tf32(tmem + jt * 32, make_desc_mn(a0 + ks * 1024), make_desc_mn(b0 + ks * 1024), idesc, acc);
                                acc = 1u;
                            }
                        }
                    }
                    tc_commit(BAR(12 + s));
                }
                __syncwarp();
            }
            if (elect_one()) tc_commit(BAR(16));
            __syncwarp();
        }
    } else {
        const int ct = tid - 64;
        uint32_t it = 0;
        for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x, ++it) {
            const uint32_t rs = it % NRAW, rph = (it / NRAW) & 1;
            const uint32_t cs = it % NCONV, cph = (it / NCONV) & 1;
            mbar_wait(BAR(0 + rs), rph);
            mbar_wait(BAR(12 + cs), cph ^ 1);
            const uint8_t *rawp = raw_gen + rs * D0_RAW;
            const float4 *src = reinterpret_cast<const float4 *>(rawp);
            float4 *hi = reinterpret_cast<float4 *>(conv_gen + cs * D0_CONV);
            float4 *lo = reinterpret_cast<float4 *>(conv_gen + cs * D0_CONV + DW_OPER);
            float4 *bh = reinterpret_cast<float4 *>(conv_gen + cs * D0_CONV + 2 * DW_OPER);
            float4 *bl = reinterpret_cast<float4 *>(conv_gen + cs * D0_CONV + 2 * DW_OPER + DW_PANEL);
            if (ct < 128) {   // B panel: row lr = [x (16 floats) | 1 | 0 x 15], 32-byte chunk c stored at c ^ (lr & 3)
                const int lr = (ct & 63) >> 2, j = ct & 3;
                const long long m = (kb >> 3) * TM + (kb & 7) * DW_KROWS + lr;
                float4 v, l = make_float4(0.f, 0.f, 0.f, 0.f);
                int chunk;
                if (ct < 64) {
                    chunk = j >> 1;
                    v = (m < M) ? reinterpret_cast<const float4 *>(rawp + DW_OPER)[lr * 4 + j] : make_float4(0.f, 0.f, 0.f, 0.f);
                    l.x = tf32_rna(v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u));
                    l.y = tf32_rna(v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u));
                    l.z = tf32_rna(v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u));
                    l.w = tf32_rna(v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u));
                } else {
                    chunk = 2 + (j >> 1);
                    v = make_float4(j == 0 ? 1.f : 0.f, 0.f, 0.f, 0.f);
                }
                const int o = (lr << 3) | ((chunk ^ (lr & 3)) << 1) | (j & 1);
                bh[o] = v;
                bl[o] = l;
            }
#pragma unroll 4
            for (int f = ct; f < DW_OPER / 16; f += DW_NCT) {
                const int pnl = f >> 7, lr = (f >> 3) & 15, p16 = f & 7;
                const int c16 = p16 ^ (lr & 7);
                const int d16 = (((c16 >> 1) ^ (lr & 3)) << 1) | (c16 & 1);
                const float4 v = src[f];
                float4 l;
                l.x = tf32_rna(v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u));
                l.y = tf32_rna(v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u));
                l.z = tf32_rna(v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u));
                l.w = tf32_rna(v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u));
                const int o = (pnl << 7) | (lr << 3) | d16;
                hi[o] = v;
                lo[o] = l;
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) { mbar_arrive(BAR(8 + cs)); mbar_arrive(BAR(4 + rs)); }
        }
        if (has_work) {
            mbar_wait(BAR(16), 0);
            tc_fence_after();
            const int q = warp & 3;
            const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
            const int jt = (warp - 2) >> 2;             // each accumulator half is drained by its own 4 converter warps
            const int k = jt * 128 + q * 32 + lane;
            uint32_t v[32];
            tmem_ld32(tmem + lane_addr + jt * 32, v);
            float4 *o = reinterpret_cast<float4 *>(gW0 + (size_t)k * 16);
#pragma unroll
            for (int c = 0; c < 4; ++c)
                atomicAdd(o + c, make_float4(__uint_as_float(v[c * 4]), __uint_as_float(v[c * 4 + 1]), __uint_as_float(v[c * 4 + 2]),
                                             __uint_as_float(v[c * 4 + 3])));
            atomicAdd(gb0 + k, __uint_as_float(v[16]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(64u) : "memory");
    }
}

// c[j] = sum_m relu'(h2)[m][j] dsdf[m]  ->  gb1[j] += w2[j] c[j],  gW2[j] += b1[j] c[j]  (the other part of gW2 comes from
// k_dw1_tc).  thread = (storage word w = tid & 7, row lane tid >> 3); 36 B/sample, a few tens of microseconds
__global__ void __launch_bounds__(256) k_mask_colsum(long long M_host, const int32_t *__restrict__ M_dev, const uint32_t *__restrict__ mask2,
                                                      const float *__restrict__ dsdf, const float *__restrict__ b1, const float *__restrict__ w2,
                                                      float *__restrict__ gb1, float *__restrict__ gW2) {
    const long long M = M_dev ? min((long long)*M_dev, M_host) : M_host;
    const int w = threadIdx.x & 7, rl = threadIdx.x >> 3;
    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    const long long stride = (long long)gridDim.x * 32;
    for (long long m0 = (long long)blockIdx.x * 32 + rl; m0 < M; m0 += 4 * stride) {   // 4 independent rows in flight per thread
        uint32_t mk[4];
        float d[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const long long m = m0 + u * stride;
            mk[u] = m < M ? mask2[(size_t)m * 8 + w] : 0u;
            d[u] = m < M ? dsdf[m] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] += (mk[u] >> i) & 1u ? d[u] : 0.f;
    }
    __shared__ float red[32][257];
    const int cb = 2 * (w & 3) + (w >> 2);               // storage word g*4+kk holds columns 32(2kk+g)..+31
#pragma unroll
    for (int i = 0; i < 32; ++i) red[rl][cb * 32 + i] = acc[i];
    __syncthreads();
    const int j = threadIdx.x;
    float c = 0.f;
#pragma unroll 8
    for (int r = 0; r < 32; ++r) c += red[r][j];
    atomicAdd(gb1 + j, w2[j] * c);
    atomicAdd(gW2 + j, b1[j] * c);
}

}  // namespace tc

extern "C" int64_t nl_mlp_tc_panel_bytes(void) { return (int64_t)tc::STEPS_TRAIN * tc::STAGE_B; }

extern "C" int nl_mlp_tc_prepare(const float *W0, const float *W1, const float *w2, void *panels, void *stream) {
    if (!W0 || !W1 || !w2 || !panels) return nl_set_error("nl_mlp_tc_prepare: null pointer");
    dim3 grid(nl_div_up(tc::WN * 8, 256), tc::STEPS_TRAIN);
    tc::k_tc_prepare<<<grid, 256, 0, (cudaStream_t)stream>>>(W0, W1, w2, (uint8_t *)panels);
    NL_CHECK_LAUNCH("nl_mlp_tc_prepare");
    return NL_OK;
}

extern "C" int nl_mlp_tc_forward(int64_t M, const int32_t *d_M_dev, const float *feats, const void *panels, const float *b0,
                                 const float *b1, const float *w2, const float *b2, float *sdf, void *stream) {
    if (M < 0) return nl_set_error("nl_mlp_tc_forward: negative M");
    if (M == 0) return NL_OK;
    if (!feats || !panels || !b0 || !b1 || !w2 || !b2 || !sdf) return nl_set_error("nl_mlp_tc_forward: null pointer");
    static NlPerDevice configured;
    const cudaError_t e0 = configured.once([] { return cudaFuncSetAttribute(tc::k_mlp_tc_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_TOTAL); });
    if (e0 != cudaSuccess) return nl_set_error_code(NL_ERR_CUDA, cudaGetErrorString(e0));
    tc::FwdParams p;
    p.M_host = M; p.M_dev = d_M_dev; p.feats = feats; p.panels = (const uint8_t *)panels;
    p.b0 = b0; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.sdf = sdf;
    const long long ntiles = (M + tc::TM - 1) / tc::TM;
    const int grid = (int)(ntiles < (long long)nl_num_sms() ? ntiles : (long long)nl_num_sms());
    tc::k_mlp_tc_fwd<<<grid, tc::NTHREADS, tc::SMEM_TOTAL, (cudaStream_t)stream>>>(p);
    NL_CHECK_LAUNCH("nl_mlp_tc_forward");
    return NL_OK;
}

// per 128-sample tile: h1 and dh1 panels (2 x 128 KB), dsdf (512 B), relu'(h2) bits (4 KB)
extern "C" int64_t nl_mlp_tc_act_floats(int64_t M) { return ((M + tc::TM - 1) / tc::TM) * (2 * 8 * tc::TM * 32 + tc::TM + tc::TM * 8); }

extern "C" int nl_mlp_tc_train(int64_t M, const int32_t *d_M_dev, const float *feats, const void *panels, const float *W1, const float *b0,
                               const float *b1, const float *w2, const float *b2, const uint8_t *s_flag, const float *s_depth,
                               const int32_t *s_ray, const float *cosv, const float *gt_depth, nl_render_stats *stats,
                               float truncation, float *sdf, float *dfeats, const nl_mlp_grads *grads, float *act,
                               const float *dsdf_ext, void *wgrad_stream_, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (M < 0) return nl_set_error("nl_mlp_tc_train: negative M");
    if (M == 0) return NL_OK;
    if (!feats || !panels || !W1 || !b0 || !b1 || !w2 || !b2 || !sdf || !dfeats) return nl_set_error("nl_mlp_tc_train: null pointer");
    if (!dsdf_ext && (!s_flag || !s_depth || !s_ray || !gt_depth || !stats))
        return nl_set_error("nl_mlp_tc_train: the loss needs s_flag, s_depth, s_ray, gt_depth and stats");
    if (grads && (!grads->gW0 || !grads->gb0 || !grads->gW1 || !grads->gb1 || !grads->gW2 || !grads->gb2 || !act))
        return nl_set_error("nl_mlp_tc_train: decoder gradients requested but a buffer is null");
    // per-device one-time state (kernel attributes are per device; so is the event that orders the weight-gradient stream)
    constexpr int NL_MAX_DEV = 64;
    static std::mutex dev_mu;
    static bool configured_dev[NL_MAX_DEV] = {};
    static cudaEvent_t ev_dev[NL_MAX_DEV] = {};
    int cur_dev = 0;
    if (cudaGetDevice(&cur_dev) != cudaSuccess || cur_dev < 0 || cur_dev >= NL_MAX_DEV) return nl_set_error_code(NL_ERR_CUDA, "nl_mlp_tc_train: cudaGetDevice");
    std::lock_guard<std::mutex> dev_lock(dev_mu);
    bool &configured = configured_dev[cur_dev];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(tc::k_mlp_tc_train<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_TOTAL);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::k_mlp_tc_train<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_TOTAL);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::k_dw1_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::DW_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tc::k_dw0_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::D0_SMEM);
        if (e != cudaSuccess) return nl_set_error_code(NL_ERR_CUDA, cudaGetErrorString(e));
        configured = true;
    }
    tc::TrainParams p = {};
    p.M_host = M; p.M_dev = d_M_dev; p.feats = feats; p.panels = (const uint8_t *)panels;
    p.b0 = b0; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.sdf = sdf; p.dfeats = dfeats;
    p.s_flag = s_flag; p.s_depth = s_depth; p.s_ray = s_ray; p.cosv = cosv; p.gt_depth = gt_depth; p.stats = stats;
    p.truncation = truncation; p.dsdf_ext = dsdf_ext;
    const long long ntiles = (M + tc::TM - 1) / tc::TM;
    const int sms = nl_num_sms();
    const int grid = (int)(ntiles < (long long)sms ? ntiles : (long long)sms);
    static long long *dbg_dev = nullptr;
    static int dbg_calls = 0;
    const bool want_dbg = getenv("NL_TC_TIMELINE") != nullptr;
    if (want_dbg && !dbg_dev) { cudaMalloc(&dbg_dev, 4 * 25 * 8 * sizeof(long long)); cudaMemset(dbg_dev, 0, 4 * 25 * 8 * sizeof(long long)); }
    p.dbg = want_dbg ? dbg_dev : nullptr;
    if (grads) {
        const size_t panel = (size_t)ntiles * 8 * tc::TM * 32;   // capacity-based carve (M is the host-side bound)
        p.act_h1 = act; p.act_dh1 = act + panel; p.act_dsdf = act + 2 * panel;
        p.act_mask2 = reinterpret_cast<uint32_t *>(act + 2 * panel + (size_t)ntiles * tc::TM);
        p.gb2 = grads->gb2;
        tc::k_mlp_tc_train<true><<<grid, tc::NTHREADS_TRAIN, tc::SMEM_TOTAL, stream>>>(p);
        // The weight-gradient kernels only need what the kernel above wrote; on a second stream they overlap with whatever the
        // caller enqueues next on `stream` (the embedding scatter, which is L2-atomic bound and leaves the SMs mostly idle).
        cudaStream_t ws = wgrad_stream_ ? (cudaStream_t)wgrad_stream_ : stream;
        if (ws != stream) {
            cudaEvent_t &ev = ev_dev[cur_dev];
            if (!ev && cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) return nl_set_error_code(NL_ERR_CUDA, "cudaEventCreate");
            if (cudaEventRecord(ev, stream) != cudaSuccess || cudaStreamWaitEvent(ws, ev, 0) != cudaSuccess)
                return nl_set_error_code(NL_ERR_CUDA, "nl_mlp_tc_train: could not order the weight-gradient stream behind the decoder kernel");
        }
        // back to back on all SMs: k_dw0_tc streams 1 KB/sample and is limited per SM by its converter warps, so it needs every SM
        tc::k_dw1_tc<<<sms, tc::DW_THREADS, tc::DW_SMEM, ws>>>(M, d_M_dev, p.act_mask2, p.act_dsdf, p.act_h1, W1, w2, grads->gW1, grads->gW2);
        tc::k_dw0_tc<<<sms, tc::DW_THREADS, tc::D0_SMEM, ws>>>(M, d_M_dev, p.act_dh1, feats, grads->gW0, grads->gb0);
        tc::k_mask_colsum<<<sms * 8, 256, 0, ws>>>(M, d_M_dev, p.act_mask2, p.act_dsdf, b1, w2, grads->gb1, grads->gW2);
    } else {
        tc::k_mlp_tc_train<false><<<grid, tc::NTHREADS_TRAIN, tc::SMEM_TOTAL, stream>>>(p);
    }
    NL_CHECK_LAUNCH("nl_mlp_tc_train");
    if (want_dbg && ++dbg_calls == 8) {   // debug only: dump one steady-state tile timeline of CTA 0 (synchronises)
        long long h[800];
        cudaStreamSynchronize(stream);
        cudaMemcpy(h, dbg_dev, sizeof(h), cudaMemcpyDeviceToHost);
        long long t0 = h[0];
        for (int i = 0; i < 800; ++i) if (h[i] && h[i] < t0) t0 = h[i];
        const char *roles[4] = {"producer", "mma", "epi_g0", "epi_g1"};
        for (int r = 0; r < 4; ++r)
            for (int st = 0; st < 25; ++st) {
                long long *q = h + (r * 25 + st) * 8;
                if (q[0] || q[1] || q[2] || q[3]) {
                    fprintf(stderr, "TL %-8s step %2d :", roles[r], st);
                    for (int k = 0; k < 8; ++k) fprintf(stderr, " %7lld", q[k] ? q[k] - t0 : -1);
                    fprintf(stderr, "\n");
                }
            }
    }
    return NL_OK;
}
