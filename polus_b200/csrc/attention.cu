// Fused multi-head self-attention for S <= 512, head_dim = 64 (BERT-base/large heads), forward and backward.
// The S x S score / probability tensors never leave the SM: scores live in TMEM, probabilities go through shared
// memory straight into the second tcgen05.mma.  Replaces, per layer, three batched GEMM launches + the softmax
// kernel in forward and five launches in backward (the unfused path of ops.attention, kept for longer sequences),
// i.e. the TF ops behind HF TFBertSelfAttention: matmul(q,k^T)/sqrt(dh) + (1-mask)*-10000 (polus/models.py:175-195)
// -> softmax -> dropout -> matmul(p, v), and their gradients.
//
// Forward, one CTA per (batch, head, 128-query tile), 32 + 128 NSEG threads (NSEG = 2 for S <= 256, 4 for S <= 512):
//   warp 0 / lane 0 : TMA loads of Q [128x64], K and V [128 NSEG x 64] from the packed [B,S,3H] projection (4-D tensor
//                     map (dh, s, slot, b), slot = {q,k,v} x head); tcgen05.mma  S = Q K^T (M128 N256 K64 per 256 keys)
//                     into TMEM cols 0..128 NSEG-1; later O = P V (M128 N64 K = 128 NSEG) into cols 0..63.
//   other warps     : thread = (query row, 128-key segment).  Two passes over its TMEM columns: max, then
//                     e = 2^((x - max) log2 e) (sum kept in fp32), dropout with the same Philox counters as the unfused
//                     softmax kernel (decisions made, and written out for the backward, while the tiles are in flight),
//                     bf16 e -> 128B-swizzled smem (K-major A operand) over the dead Q / K tiles.  After the second MMA:
//                     O * (1/(1-p)) / sum -> bf16 -> smem -> TMA store into ctx [B,S,H].  Saves L = max + log(sum).
//
// Backward, one CTA per (batch, head, 256-query half): blocks (query tile i, key block j) of 128x128; K / V stream
// through two 128-key stages; with two halves (S > 256) dK / dV partial sums are reduce-added in bf16 by the TMA unit.
//   TMEM: S_ij 0..127 | dP_ij 128..255 | dQ_0 256..319 | dK_j 320..383 | dV_j 384..447 | dQ_1 448..511.
//   smem: Q, K, V, dO (32 KB each), Pd_ij and dS_ij (32 KB each; ONE copy of dS serves both dQ += dS K (K-major A)
//   and dK += dS^T Q (MN-major A): the two canonical layouts coincide byte for byte).
//   P is recomputed from the saved L; delta_row = sum_d dO*O.
#include "common.cuh"
#include "ptx.cuh"
#include <cuda.h>
#include <atomic>

extern std::atomic<long long> g_launch_count;
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

namespace {

constexpr int DH = 64;
constexpr float kLog2e = 1.4426950408889634f;

struct AttnParams {
    int B, S, nh;
    float scale;           // 1/sqrt(dh)
    uint32_t thresh16;     // dropout threshold (0 = off)
    float inv_keep;
    unsigned long long seed;
    uint32_t site;
    const uint32_t* d_step;
    const int32_t* mask;   // [B,S] or null
    float* lse;            // [B,nh,S]
    uint32_t* keepbits;    // [B*nh*S][S/32] dropout keep bits (forward writes, backward reads); null when p = 0
    float* gbias;          // backward: [3H] bias gradient of the QKV projection += column sums of dqkv; may be null
    int pf_stride;         // backward: CTA i warms the L2 with the tiles of CTA i + pf_stride (0 = off)
};

// 2^x as ONE MUFU.EX2.  exp2f() costs four issue slots per value -- compare against -126, pre-scale by 0.5, MUFU, square --
// to return denormal results; here x <= 0 always and a probability below 2^-126 is 0 in the bf16 P tile anyway.
__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// barrier + OR-reduction of a predicate over the `nthreads` threads of named barrier `id`
__device__ __forceinline__ bool named_bar_or(int id, int nthreads, bool pred) {
    int r;
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.s32 p, %1, 0;\n"
        "bar.red.or.pred q, %2, %3, p;\n"
        "selp.s32 %0, 1, 0, q;\n"
        "}\n"
        : "=r"(r) : "r"((int)pred), "r"(id), "r"(nthreads) : "memory");
    return r != 0;
}

// ================================================================================================ forward
// NSEG = number of 128-key segments the kernel covers: 2 for S <= 256 (288 threads, 2 CTAs per SM), 4 for S <= 512
// (544 threads, one CTA per SM: the 128 x 512 score tile fills the SM's 512 TMEM columns).
// warp 0 = TMA + MMA issue, warps 1..4*NSEG = softmax (thread = (query row, 128-key segment)).
template <int NSEG> struct FwdCfg {
    static constexpr int THREADS = 32 + 128 * NSEG;
    static constexpr int SM_THREADS = 128 * NSEG;
    static constexpr int SQ = 0;                      // 16 KB  Q tile                  } P (NSEG x 32 KB) overlays Q, K and
    static constexpr int SK = 16384;                  // NSEG x 16 KB  K                } the pad behind them once S = Q K^T
    static constexpr int SV = NSEG * 32768;           // NSEG x 16 KB  V                  retired; O staging reuses 16 KB of it
    static constexpr int MISC = SV + NSEG * 16384;    // mask [128 NSEG] f32 | red [NSEG][128] f32 | barriers
    static constexpr int SMEM = 1024 + MISC + NSEG * 1024 + 64;
};

template <int NSEG>
__global__ void __launch_bounds__(FwdCfg<NSEG>::THREADS, NSEG == 2 ? 2 : 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmO, const AttnParams p) {
    using Cfg = FwdCfg<NSEG>;
    constexpr int SMT = Cfg::SM_THREADS;
    // 1024-byte alignment (128B-swizzle atoms) comes from the declaration, which also keeps the pointer in the shared
    // address space for the compiler: LDS / STS instead of generic LD / ST on every staging access
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((ptx::smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* sQ = smem + Cfg::SQ;
    uint8_t* sK = smem + Cfg::SK;
    uint8_t* sV = smem + Cfg::SV;
    uint8_t* sP = smem;  // overlay
    float* sMask = reinterpret_cast<float*>(smem + Cfg::MISC);
    float* sRed = reinterpret_cast<float*>(smem + Cfg::MISC + NSEG * 512);        // [NSEG segments][128 rows]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::MISC + NSEG * 1024);  // 0 load, 1 S ready, 2 P ready, 3 O ready
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q_tiles = (p.S + 127) / 128;
    const int qt = blockIdx.x % q_tiles;
    const int h = (blockIdx.x / q_tiles) % p.nh;
    const int b = blockIdx.x / (q_tiles * p.nh);
    const int q0 = qt * 128;

    pdl_trigger();
    // (1) the additive key mask of this thread's key slot: a graph input, never written inside the step, so the load may
    //     start before pdl_wait() and overlaps the whole prologue (it used to be a fully exposed global load in front of
    //     the first named barrier: 7 % of the kernel's stall samples at p = 0, profiles/r02_ncu_attn_fwd_p0.txt)
    float my_mask = -INFINITY;
    if (warp > 0) {
        const int t = threadIdx.x - 32;
        if (t < p.S) my_mask = p.mask ? (1.0f - (float)__ldg(p.mask + (long long)b * p.S + t)) * -10000.0f : 0.f;
    }
    // (2) the first thread of warp 1 owns the load barrier and issues the TMA loads at once, while warp 0 initialises the
    //     other barriers and allocates TMEM: allocation and the block-wide barrier run UNDER the loads, not in front of them
    if (threadIdx.x == 32) {
        ptx::prefetch_tensormap(&tmQKV);
        ptx::mbar_init(&bars[0], 1);
        ptx::fence_barrier_init();
        pdl_wait();  // qkv is the previous kernel's output
        ptx::mbar_expect_tx(&bars[0], 16384 + NSEG * 32768);
        ptx::tma_load_4d(sQ, &tmQKV, &bars[0], 0, q0, h, b);
#pragma unroll
        for (int g = 0; g < NSEG; ++g) {
            ptx::tma_load_4d(sK + g * 16384, &tmQKV, &bars[0], 0, g * 128, p.nh + h, b);
            ptx::tma_load_4d(sV + g * 16384, &tmQKV, &bars[0], 0, g * 128, 2 * p.nh + h, b);
        }
    }
    if (threadIdx.x == 0) {
        ptx::prefetch_tensormap(&tmO);
        ptx::mbar_init(&bars[1], 1);
        ptx::mbar_init(&bars[2], SMT);
        ptx::mbar_init(&bars[3], 1);
        ptx::fence_barrier_init();
    }
    __syncwarp();
    if (warp == 0) ptx::tmem_alloc<128 * NSEG>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    pdl_wait();

    if (warp == 0) {
        if (lane == 0) {
            ptx::mbar_wait(&bars[0], 0);
            ptx::tc_fence_after();
            {   // S = Q K^T : A = Q (K-major), B = K (K-major), M128 N256 per 256 keys, K = 64 in 4 steps
                constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 256, 0, 0);
                const uint64_t base = ptx::umma_desc_base(16, 1024);
                const uint32_t a = ptx::smem_u32(sQ), bb = ptx::smem_u32(sK);
#pragma unroll
                for (int g = 0; g < NSEG / 2; ++g)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        ptx::umma_bf16(tmem + g * 256, ptx::umma_desc(base, a + k * 32), ptx::umma_desc(base, bb + g * 32768 + k * 32),
                                       idesc, k > 0);
                ptx::umma_commit(&bars[1]);
            }
            ptx::mbar_wait(&bars[2], 0);
            ptx::tc_fence_after();
            {   // O = P V : A = P (K-major, 2 NSEG k-blocks of 64 keys), B = V ([key][d] => MN-major), M128 N64 K(128 NSEG) -> cols 0..63
                constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 64, 0, 1);
                const uint64_t abase = ptx::umma_desc_base(16, 1024);
                const uint64_t bbase = ptx::umma_desc_base(64 * 128, 1024);
                const uint32_t a = ptx::smem_u32(sP), bb = ptx::smem_u32(sV);
#pragma unroll
                for (int k = 0; k < 8 * NSEG; ++k)
                    ptx::umma_bf16(tmem, ptx::umma_desc(abase, a + (k >> 2) * 16384 + (k & 3) * 32),
                                   ptx::umma_desc(bbase, bb + k * 2048), idesc, k > 0);
                ptx::umma_commit(&bars[3]);
            }
        }
    } else {
        // ---------------------------------------------------------------- softmax / epilogue: thread = (row, key segment)
        const int t = threadIdx.x - 32;          // 0..128 NSEG - 1
        const int e = warp - 1;                  // 0..4 NSEG - 1
        const int quad = warp & 3;               // TMEM lane quadrant this warp may access
        const int half = e >> 2;                 // key segment: keys [128*half, 128*half + 128)
        const int row = quad * 32 + lane;        // row inside the tile (== TMEM lane)
        const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
        // additive key mask, staged once: (1 - m) * -10000 for real keys, -inf for keys beyond S (loaded at the top)
        sMask[t] = my_mask;
        // Dropout decisions of this thread's 128 probabilities, made (and written out for the backward kernel) while the
        // Q/K/V tiles are still in flight and the first MMA runs: 16 Philox blocks that used to sit between the two
        // softmax passes (attention_fwd p=0.1 vs p=0: +50 % time, profiles/r01_kernel_times_v9_b64.log).
        const uint32_t step = p.thresh16 ? *p.d_step : 0u;
        const bool qvalid = q0 + row < p.S;
        const long long grow = ((long long)(b * p.nh + h) * p.S + (q0 + row));  // row of the [B*nh*S, S] probability matrix
        const int chunks_per_row = p.S >> 3;
        uint32_t kbits[4] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
        if (p.thresh16) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int kc = half * 128 + c * 32;
                if (qvalid && kc < p.S) {
                    uint32_t bits = 0;
#pragma unroll
                    for (int g8 = 0; g8 < 4; ++g8) {
                        const int key0 = kc + g8 * 8;
                        uint32_t keep = 0xFFu;
                        if (key0 < p.S)
                            keep = dropout_keep8(p.seed, p.site, step, (unsigned long long)grow * chunks_per_row + (key0 >> 3), p.thresh16);
                        bits |= keep << (8 * g8);
                    }
                    p.keepbits[grow * (p.S >> 5) + (kc >> 5)] = bits;  // reused by the backward kernel
                    kbits[c] = bits;
                }
            }
        }
        // (barrier for sMask) + is any of the 128 NSEG key slots masked?  Sequences without padding take the branch that
        // never reads the mask: two instructions per score fewer in each pass, and identical results (x * s + 0 == x * s)
        const bool masked = named_bar_or(1, SMT, my_mask != 0.f);
        ptx::mbar_wait(&bars[1], 0);
        ptx::tc_fence_after();
        const float sc = p.scale;
        // Both passes keep the NEXT 32-column chunk's tcgen05.ld in flight while the current one is processed (the load
        // used to sit, fully exposed, at the head of every chunk) and run four independent max / sum chains instead of one
        // 128-long dependent chain per thread.
        float va[32], vb[32];
        float mx;
        {
            float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
            ptx::tmem_ld32(lane_addr + half * 128, va);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float* cur = (c & 1) ? vb : va;
                float* nxt = (c & 1) ? va : vb;
                ptx::tmem_ld_wait();
                // chunk c + 1 of this pass, or chunk 0 of the exp pass (the same columns are read twice)
                ptx::tmem_ld32(lane_addr + half * 128 + ((c + 1) & 3) * 32, nxt);
                if (masked) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        m0 = fmaxf(m0, fmaf(cur[j], sc, sMask[half * 128 + c * 32 + j]));
                        m1 = fmaxf(m1, fmaf(cur[j + 1], sc, sMask[half * 128 + c * 32 + j + 1]));
                        m2 = fmaxf(m2, fmaf(cur[j + 2], sc, sMask[half * 128 + c * 32 + j + 2]));
                        m3 = fmaxf(m3, fmaf(cur[j + 3], sc, sMask[half * 128 + c * 32 + j + 3]));
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        m0 = fmaxf(m0, cur[j]);
                        m1 = fmaxf(m1, cur[j + 1]);
                        m2 = fmaxf(m2, cur[j + 2]);
                        m3 = fmaxf(m3, cur[j + 3]);
                    }
                }
            }
            mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
        }
        if (!masked) mx *= sc;  // sc > 0: max(x_j * sc) == max(x_j) * sc, rounding included
        sRed[half * 128 + row] = mx;
        named_bar_sync(1, SMT);
#pragma unroll
        for (int g = 1; g < NSEG; ++g) mx = fmaxf(mx, sRed[((half + g) % NSEG) * 128 + row]);  // keys beyond S are -inf, real keys finite: mx is finite
        named_bar_sync(1, SMT);                        // sRed is reused for the sums below
        float sum;
        const float mxl = mx * kLog2e;
        const float scl = sc * kLog2e;
        {
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float* v = (c & 1) ? vb : va;      // chunk 0 was requested at the end of the max pass into va
                float* nxt = (c & 1) ? va : vb;
                ptx::tmem_ld_wait();
                if (c < 3) ptx::tmem_ld32(lane_addr + half * 128 + (c + 1) * 32, nxt);
                const int kc = half * 128 + c * 32;  // first key of this chunk
                if (masked) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        v[j] = fast_exp2(fmaf(v[j], scl, fmaf(sMask[kc + j], kLog2e, -mxl)));
                        v[j + 1] = fast_exp2(fmaf(v[j + 1], scl, fmaf(sMask[kc + j + 1], kLog2e, -mxl)));
                        v[j + 2] = fast_exp2(fmaf(v[j + 2], scl, fmaf(sMask[kc + j + 2], kLog2e, -mxl)));
                        v[j + 3] = fast_exp2(fmaf(v[j + 3], scl, fmaf(sMask[kc + j + 3], kLog2e, -mxl)));
                        s0 += v[j];
                        s1 += v[j + 1];
                        s2 += v[j + 2];
                        s3 += v[j + 3];
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        v[j] = fast_exp2(fmaf(v[j], scl, -mxl));
                        v[j + 1] = fast_exp2(fmaf(v[j + 1], scl, -mxl));
                        v[j + 2] = fast_exp2(fmaf(v[j + 2], scl, -mxl));
                        v[j + 3] = fast_exp2(fmaf(v[j + 3], scl, -mxl));
                        s0 += v[j];
                        s1 += v[j + 1];
                        s2 += v[j + 2];
                        s3 += v[j + 3];
                    }
                }
                if (p.thresh16) {
                    const uint32_t bits = kbits[c];
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = ((bits >> j) & 1u) ? v[j] : 0.f;  // (the 1/(1-p) factor rides on 1/sum below)
                }
                // keys [kc, kc+32) -> k-block kc/64, 16-byte chunks ((kc/32)&1)*4 .. +3 of row `row`
                uint8_t* blk = sP + (kc >> 6) * 16384 + row * 128;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int chunk = (((kc >> 5) & 1) * 4 + j) ^ (row & 7);
                    *reinterpret_cast<bf16x8*>(blk + chunk * 16) = pack8(v + 8 * j);
                }
            }
            sum = (s0 + s1) + (s2 + s3);
        }
        sRed[half * 128 + row] = sum;
        ptx::fence_proxy_async_smem();
        ptx::tc_fence_before();
        ptx::mbar_arrive(&bars[2]);
        named_bar_sync(1, SMT);
        if (NSEG == 2) {
            sum += sRed[(half ^ 1) * 128 + row];
        } else {  // the same order in every thread of the row: identical 1/sum across the row's O columns
            sum = 0.f;
#pragma unroll
            for (int g = 0; g < NSEG; ++g) sum += sRed[g * 128 + row];
        }
        if (qvalid && half == 0) p.lse[grow] = mx + logf(sum);
        const float inv = p.inv_keep / sum;  // O = (keep o e) V * (1/(1-p)) / sum: one multiply per output instead of one per score
        ptx::mbar_wait(&bars[3], 0);
        ptx::tc_fence_after();
        {   // O columns [OC*half, +OC) of this row -> staging tile [128 rows][128 B] at the start of the P region
            constexpr int OC = 64 / NSEG;
            float v[OC];
            if (NSEG == 2) ptx::tmem_ld32(lane_addr + half * OC, v);
            else ptx::tmem_ld16(lane_addr + half * OC, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < OC; ++j) v[j] *= inv;
            uint8_t* stg = smem + row * 128;
#pragma unroll
            for (int j = 0; j < OC / 8; ++j) {
                const int chunk = (half * (OC / 8) + j) ^ (row & 7);
                *reinterpret_cast<bf16x8*>(stg + chunk * 16) = pack8(v + 8 * j);
            }
        }
        ptx::fence_proxy_async_smem();
        named_bar_sync(1, SMT);
        if (half == 0 && lane == 0) {
            ptx::tma_store_4d(&tmO, smem + quad * 4096, 0, q0 + quad * 32, h, b);  // rows >= S clipped
            ptx::tma_store_commit();
            ptx::tma_store_wait_read<0>();
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<128 * NSEG>(tmem);
    }
}

// ================================================================================================ backward
// 544 threads: warp 0 = TMA + MMA issue, warps 1-16: thread = (query row, 32-key quarter of the 128-key block).
// Sixteen softmax warps (four per scheduler): with eight, the exp / dS arithmetic of a block ran at a fraction of the
// issue rate -- two warps per scheduler cannot cover TMEM-load, MUFU and shared-memory latency -- and the kernel's time
// was the sum of its serial phases (profiles/r01_attn_bwd_stalls_v10.txt).
constexpr int BWD_SM_WARPS = 16;
constexpr int BWD_SM_THREADS = BWD_SM_WARPS * 32;
constexpr int BWD_THREADS = 32 + BWD_SM_THREADS;
constexpr int B_SQ = 0;                   // 32 KB: Q rows 0..255
constexpr int B_SK = B_SQ + 32768;        // 32 KB: two 128-key stages of K (key block j lives in stage j & 1)
constexpr int B_SV = B_SK + 32768;        // 32 KB: the same for V
constexpr int B_SDO = B_SV + 32768;
constexpr int B_SPD = B_SDO + 32768;      // 32 KB: Pd_ij  [2 key groups][128 q][64 keys]; also the drain staging tile
constexpr int B_SDS = B_SPD + 32768;      // 32 KB: dS_ij  same layout
constexpr int B_SO1 = B_SDS + 32768;      // 16 KB: O rows 128..255 (O rows 0..127 land in the Pd region, idle until block 0 stores)
constexpr int B_MISC = B_SO1 + 16384;     // mask [512] floats | delta exchange [2 tiles][4 quarters][128 rows] floats | barriers
constexpr int B_SMEM = 1024 + B_MISC + 2048 + 4096 + 128;

// NKB = key blocks the instantiation can walk: 2 (S <= 256, the whole head in one CTA) or 4 (S <= 512)
template <int NKB>
__global__ void __launch_bounds__(BWD_THREADS, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                const __grid_constant__ CUtensorMap tmDQKV, const __grid_constant__ CUtensorMap tmO, const AttnParams p) {
    // 1024-byte alignment (128B-swizzle atoms) comes from the declaration, which also keeps the pointer in the shared
    // address space for the compiler: LDS / STS instead of generic LD / ST on every staging access
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((ptx::smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* sQ = smem + B_SQ;
    uint8_t* sK = smem + B_SK;
    uint8_t* sV = smem + B_SV;
    uint8_t* sDO = smem + B_SDO;
    uint8_t* sPd = smem + B_SPD;
    uint8_t* sDS = smem + B_SDS;
    float* sMask = reinterpret_cast<float*>(smem + B_MISC);
    uint8_t* sO1 = smem + B_SO1;
    float* sEx = reinterpret_cast<float*>(smem + B_MISC + 2048);
    // 0 first load group, 1 S/dP ready, 2 Pd/dS ready, 3 block MMAs done, 4/5 K,V stage 0/1 reloaded (S > 256 only),
    // 6 second query tile loaded (Q, dO, O rows 128..255), 7 second key block loaded (K, V rows 128..255)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + B_MISC + 2048 + 4096);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // one CTA per (batch, head, 256-query half): S <= 256 has one half and the CTA owns the whole head; for S <= 512 the
    // two halves of a head each walk all key blocks and their dK / dV partial sums meet in global memory (bf16 TMA
    // reduce-add into a zeroed dqkv, see polus_attention_bwd)
    const int n_half = (p.S + 255) / 256;
    const int qh = blockIdx.x % n_half;
    const int h = (blockIdx.x / n_half) % p.nh;
    const int b = blockIdx.x / (n_half * p.nh);
    const int qbase = qh * 256;                          // first query row of this CTA
    const int n_qt = min(2, (p.S - qbase + 127) / 128);  // query tiles of this CTA (1 or 2)
    const int n_kh = (p.S + 127) / 128;                  // 128-key blocks (1..4)
    const bool partial_kv = n_half > 1;

    pdl_trigger();
    // The first thread of warp 1 owns the three load barriers and issues every initial TMA load at once; warp 0 meanwhile
    // initialises the other barriers and allocates TMEM, so allocation and the block-wide barrier run under the loads.
    // O (the forward output) comes through TMA as well: delta = rowsum(dO * O) is computed from shared memory, so dO is
    // read from HBM once and no thread-issued global load sits in the prologue.  Three load groups, in the order of
    // first use: block (0,0) starts when the first 80 KB have landed; the second query tile and the second key block
    // (another 80 KB) arrive under its arithmetic (every CTA of a wave starts at the same time: the prologue is
    // bandwidth-bound, profiles/r01_attn_bwd_timeline_v11.txt)
    if (threadIdx.x == 32) {
        ptx::prefetch_tensormap(&tmQKV);
        ptx::prefetch_tensormap(&tmDO);
        ptx::prefetch_tensormap(&tmO);
        ptx::mbar_init(&bars[0], 1);
        ptx::mbar_init(&bars[6], 1);
        ptx::mbar_init(&bars[7], 1);
        ptx::fence_barrier_init();
        pdl_wait();  // qkv / ctx / dctx are earlier kernels' outputs
        ptx::mbar_expect_tx(&bars[0], 5 * 16384);
        ptx::tma_load_4d(sQ, &tmQKV, &bars[0], 0, qbase, h, b);
        ptx::tma_load_4d(sK, &tmQKV, &bars[0], 0, 0, p.nh + h, b);
        ptx::tma_load_4d(sDO, &tmDO, &bars[0], 0, qbase, h, b);
        ptx::tma_load_4d(sV, &tmQKV, &bars[0], 0, 0, 2 * p.nh + h, b);
        ptx::tma_load_4d(sPd, &tmO, &bars[0], 0, qbase, h, b);
        if (n_qt > 1) {
            ptx::mbar_expect_tx(&bars[6], 3 * 16384);
            ptx::tma_load_4d(sQ + 16384, &tmQKV, &bars[6], 0, qbase + 128, h, b);
            ptx::tma_load_4d(sDO + 16384, &tmDO, &bars[6], 0, qbase + 128, h, b);
            ptx::tma_load_4d(sO1, &tmO, &bars[6], 0, qbase + 128, h, b);
        }
        if (n_kh > 1) {
            ptx::mbar_expect_tx(&bars[7], 2 * 16384);
            ptx::tma_load_4d(sK + 16384, &tmQKV, &bars[7], 0, 128, p.nh + h, b);
            ptx::tma_load_4d(sV + 16384, &tmQKV, &bars[7], 0, 128, 2 * p.nh + h, b);
        }
    }
    if (threadIdx.x == 0) {
        ptx::prefetch_tensormap(&tmDQKV);
        ptx::mbar_init(&bars[1], 1);
        ptx::mbar_init(&bars[2], BWD_SM_THREADS);
        ptx::mbar_init(&bars[3], 1);
        ptx::mbar_init(&bars[4], 1);
        ptx::mbar_init(&bars[5], 1);
        ptx::fence_barrier_init();
    }
    if (warp == 0) ptx::tmem_alloc<512>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    pdl_wait();
    constexpr uint32_t C_S = 0, C_DP = 128, C_DQ0 = 256, C_DK = 320, C_DV = 384, C_DQ1 = 448;

    if (warp == 0) {
        if (lane == 0) {
            ptx::mbar_wait(&bars[0], 0);
            ptx::tc_fence_after();
            const uint64_t kbase = ptx::umma_desc_base(16, 1024);            // K-major, one 64-wide k-block
            const uint64_t mn1 = ptx::umma_desc_base(128 * 128, 1024);       // MN-major, 64-wide groups 16 KB apart (128 k-rows)
            const uint32_t aQ = ptx::smem_u32(sQ), aK = ptx::smem_u32(sK), aV = ptx::smem_u32(sV), aDO = ptx::smem_u32(sDO);
            const uint32_t aPd = ptx::smem_u32(sPd), aDS = ptx::smem_u32(sDS);
            uint32_t ph2 = 0;
            // S_ij = Q_i K_j^T ; dP_ij = dO_i V_j^T   (M128 N128 K64) -> bars[1]
            auto issue_scores = [&](int i, int j) {
                constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 128, 0, 0);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    ptx::umma_bf16(tmem + C_S, ptx::umma_desc(kbase, aQ + i * 16384 + k * 32),
                                   ptx::umma_desc(kbase, aK + (j & 1) * 16384 + k * 32), idesc, k > 0);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    ptx::umma_bf16(tmem + C_DP, ptx::umma_desc(kbase, aDO + i * 16384 + k * 32),
                                   ptx::umma_desc(kbase, aV + (j & 1) * 16384 + k * 32), idesc, k > 0);
                ptx::umma_commit(&bars[1]);
            };
            issue_scores(0, 0);
            const int n_blk = n_kh * n_qt;
            for (int blk = 0; blk < n_blk; ++blk) {
                const int j = blk / n_qt, i = blk % n_qt;
                // Pd_ij / dS_ij are in shared memory and every softmax thread has read S_ij / dP_ij out of TMEM
                ptx::mbar_wait(&bars[2], ph2);
                ph2 ^= 1;
                if (blk > 0) {
                    // (the softmax threads waited for the previous block's products before they stored: already complete)
                    ptx::mbar_wait(&bars[3], (blk - 1) & 1);
                    // that block was the last reader of its key block's K / V stage: refill it with key block jr + 2
                    const int jr = (blk - 1) / n_qt;
                    if (NKB > 2 && (blk - 1) % n_qt == n_qt - 1 && jr + 2 < n_kh) {
                        uint64_t* lb = &bars[4 + (jr & 1)];
                        ptx::mbar_expect_tx(lb, 32768);
                        ptx::tma_load_4d(sK + (jr & 1) * 16384, &tmQKV, lb, 0, (jr + 2) * 128, p.nh + h, b);
                        ptx::tma_load_4d(sV + (jr & 1) * 16384, &tmQKV, lb, 0, (jr + 2) * 128, 2 * p.nh + h, b);
                    }
                }
                ptx::tc_fence_after();
                // the NEXT block's scores first: they only need the S / dP columns, so the softmax threads can start on
                // them while the three accumulating products of this block are still running (they wait for bars[3] of
                // this block only before overwriting Pd / dS)
                if (blk + 1 < n_blk) {
                    const int ni = (blk + 1) % n_qt, nj = (blk + 1) / n_qt;
                    if (NKB > 2 && ni == 0 && nj >= 2) {  // first use of a refilled stage
                        ptx::mbar_wait(&bars[4 + (nj & 1)], ((nj >> 1) - 1) & 1);
                        ptx::tc_fence_after();
                    }
                    if (ni == 1 && nj == 0) {  // first use of the second query tile
                        ptx::mbar_wait(&bars[6], 0);
                        ptx::tc_fence_after();
                    }
                    if (ni == 0 && nj == 1) {  // first use of the second key block
                        ptx::mbar_wait(&bars[7], 0);
                        ptx::tc_fence_after();
                    }
                    issue_scores(ni, nj);
                }
                {   // dV_j += Pd_ij^T dO_i ; dK_j += dS_ij^T Q_i   (A MN-major over keys, B MN-major over d; M128 N64 K128)
                    constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 64, 1, 1);
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        ptx::umma_bf16(tmem + C_DV, ptx::umma_desc(mn1, aPd + k * 2048),
                                       ptx::umma_desc(mn1, aDO + i * 16384 + k * 2048), idesc, (i > 0 || k > 0));
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        ptx::umma_bf16(tmem + C_DK, ptx::umma_desc(mn1, aDS + k * 2048),
                                       ptx::umma_desc(mn1, aQ + i * 16384 + k * 2048), idesc, (i > 0 || k > 0));
                }
                {   // dQ_i += dS_ij K_j   (A K-major: 2 k-blocks of 64 keys; B = K_j rows as MN-major over d; M128 N64 K128)
                    constexpr uint32_t idesc = ptx::umma_idesc_bf16(128, 64, 0, 1);
                    const uint32_t cdq = i == 0 ? C_DQ0 : C_DQ1;
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        ptx::umma_bf16(tmem + cdq, ptx::umma_desc(kbase, aDS + (k >> 2) * 16384 + (k & 3) * 32),
                                       ptx::umma_desc(mn1, aK + (j & 1) * 16384 + k * 2048), idesc, (j > 0 || k > 0));
                }
                ptx::umma_commit(&bars[3]);
            }
        }
    } else {
        const int t = threadIdx.x - 32;   // 0..511
        const int e = warp - 1;           // 0..15
        const int quad = warp & 3;        // TMEM lane quadrant this warp may access
        const int q4 = e >> 2;            // keys [32*q4, +32) of the current 128-key block
        const int row = quad * 32 + lane;
        const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
        float my_mask = -INFINITY;  // thread t stages key t (512 slots)
        if (t < p.S) my_mask = p.mask ? (1.0f - (float)p.mask[(long long)b * p.S + t]) * (-10000.0f * kLog2e) : 0.f;
        sMask[t] = my_mask;
        if (t >= n_kh * 128) my_mask = 0.f;  // slots of key blocks that are never visited do not count as "masked"
        // L_row and the dropout keep bits of every block this thread will process (4 words): global loads issued first,
        // consumed after the tiles have landed, so that none sits on the per-block critical path
        float delta0 = 0.f, delta1 = 0.f, L0 = 0.f, L1 = 0.f;
        uint32_t kbits[NKB][2];
        {
            const uint32_t* kbuf = p.thresh16 ? p.keepbits : nullptr;
            bool ok[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) ok[i] = (i < n_qt) && (qbase + i * 128 + row < p.S);
#pragma unroll
            for (int j = 0; j < NKB; ++j)
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int q = qbase + i * 128 + row, kc = j * 128 + q4 * 32;
                    uint32_t bits = 0xFFFFFFFFu;
                    if (p.thresh16 && i < n_qt && j < n_kh && q < p.S && kc < p.S)
                        bits = kbuf[((long long)(b * p.nh + h) * p.S + q) * (p.S >> 5) + (kc >> 5)];
                    kbits[j][i] = bits;
                }
            if (ok[0]) L0 = p.lse[(long long)(b * p.nh + h) * p.S + qbase + row];
            if (ok[1]) L1 = p.lse[(long long)(b * p.nh + h) * p.S + qbase + 128 + row];
            ptx::mbar_wait(&bars[0], 0);
        }
        // One CTA per SM: every CTA of a wave starts together and their 176 KB prologues are HBM-bound while the tensor
        // cores idle; then HBM idles while they compute (profiles/r01_attn_bwd_timeline_v11.txt).  Once this CTA's first
        // load group has landed, one thread asks the TMA unit to pull the tiles of the CTA that runs one wave later
        // (block index + number of SMs) into L2: that traffic runs under this CTA's arithmetic, and the later CTA's
        // prologue is served from L2.
        if (t == 0 && p.pf_stride > 0) {
            const long long nbk = (long long)blockIdx.x + p.pf_stride;
            if (nbk < (long long)gridDim.x) {
                const int nb = (int)nbk;
                const int nqh = nb % n_half, nh_ = (nb / n_half) % p.nh, nbb = nb / (n_half * p.nh);
                const int nq0 = nqh * 256;
                const int nqt = min(2, (p.S - nq0 + 127) / 128);
                ptx::tma_prefetch_l2_4d(&tmQKV, 0, nq0, nh_, nbb);
                ptx::tma_prefetch_l2_4d(&tmQKV, 0, 0, p.nh + nh_, nbb);
                ptx::tma_prefetch_l2_4d(&tmDO, 0, nq0, nh_, nbb);
                ptx::tma_prefetch_l2_4d(&tmQKV, 0, 0, 2 * p.nh + nh_, nbb);
                ptx::tma_prefetch_l2_4d(&tmO, 0, nq0, nh_, nbb);
                if (nqt > 1) {
                    ptx::tma_prefetch_l2_4d(&tmQKV, 0, nq0 + 128, nh_, nbb);
                    ptx::tma_prefetch_l2_4d(&tmDO, 0, nq0 + 128, nh_, nbb);
                    ptx::tma_prefetch_l2_4d(&tmO, 0, nq0 + 128, nh_, nbb);
                }
                if (n_kh > 1) {
                    ptx::tma_prefetch_l2_4d(&tmQKV, 0, 128, p.nh + nh_, nbb);
                    ptx::tma_prefetch_l2_4d(&tmQKV, 0, 128, 2 * p.nh + nh_, nbb);
                }
            }
        }
        // delta_row = sum_d dO[row,d] * O[row,d]: the four threads sharing a row split the 64 columns (two 16-byte chunks
        // each) of the swizzled dO / O tiles and exchange their quarters through shared memory
        auto delta_part = [&](const uint8_t* o_tile, const uint8_t* do_tile, int i) {
            float part = 0.f;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int off = row * 128 + (((q4 * 2 + c) ^ (row & 7)) << 4);
                float a[8], d8[8];
                unpack8(*reinterpret_cast<const bf16x8*>(o_tile + off), a);
                unpack8(*reinterpret_cast<const bf16x8*>(do_tile + off), d8);
#pragma unroll
                for (int x = 0; x < 8; ++x) part = fmaf(a[x], d8[x], part);
            }
            sEx[(i * 4 + q4) * 128 + row] = part;
        };
        auto delta_sum = [&](int i) {
            float d = 0.f;
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) d += sEx[(i * 4 + qq) * 128 + row];
            return d;
        };
        delta_part(sPd, sDO, 0);
        const bool masked = named_bar_or(1, BWD_SM_THREADS, my_mask != 0.f);  // (also the barrier behind sMask and the delta exchange)
        delta0 = delta_sum(0);
        const float sc = p.scale;
        uint32_t ph1 = 0;
        int blk = 0;
        // bias gradient of the QKV projection = column sums of dQ | dK | dV: thread (w = lane, rg = e) adds the column pair
        // (2w, 2w+1) over rows [8 rg, 8 rg + 8) of every drained tile, from the staged bf16 values
        float bsum[3][2] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
        // TMEM accumulator columns `col` (this thread: row `row`, 16 of the 64 columns) -> bf16 -> swizzled staging tile
        auto stage_acc = [&](uint32_t col, uint8_t* tile) {
            float v[16];
            ptx::tmem_ld16(lane_addr + col + q4 * 16, v);
            ptx::tmem_ld_wait();
            uint8_t* stg = tile + row * 128;
#pragma unroll
            for (int x = 0; x < 2; ++x) {
                const int chunk = (q4 * 2 + x) ^ (row & 7);
                *reinterpret_cast<bf16x8*>(stg + chunk * 16) = pack8(v + 8 * x);
            }
        };
        auto colsum_tile = [&](const uint8_t* tile, int row0, float* bs) {
            const int nrows = min(128, p.S - row0);  // (may be <= 0 for a tile beyond S: nothing is added)
#pragma unroll
            for (int rr = 0; rr < 8; ++rr) {
                const int r = e * 8 + rr;
                if (r < nrows) {
                    const uint32_t w = *reinterpret_cast<const uint32_t*>(tile + r * 128 + (((lane >> 2) ^ (r & 7)) << 4) + (lane & 3) * 4);
                    bs[0] += __uint_as_float(w << 16);
                    bs[1] += __uint_as_float(w & 0xFFFF0000u);
                }
            }
        };
#pragma unroll
        for (int j = 0; j < NKB; ++j) {
            if (j >= n_kh) break;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i >= n_qt) break;
                ptx::mbar_wait(&bars[1], ph1);
                ph1 ^= 1;
                ptx::tc_fence_after();
                const int q = qbase + i * 128 + row;
                const bool qvalid = q < p.S;
                const float Ll = qvalid ? (i == 0 ? L0 : L1) * kLog2e : INFINITY;  // rows beyond S: p = exp2(-inf) = 0
                const float dl = i == 0 ? delta0 : delta1;
                const float scl = sc * kLog2e;
                const int kl = q4 * 32;              // key offset inside the 128-key block
                const int kc = j * 128 + kl;         // absolute first key
                const uint32_t bits = kbits[j][i];  // keep bits written by the forward kernel (same Philox stream)
                bf16x8 pdq[4], dsq[4];              // results stay packed (16 registers) until the stores are allowed
#pragma unroll
                for (int sub = 0; sub < 2; ++sub) {  // 16 keys at a time: 96 registers per thread
                    float s[16], dp[16];
                    ptx::tmem_ld16(lane_addr + C_S + kl + 16 * sub, s);
                    ptx::tmem_ld16(lane_addr + C_DP + kl + 16 * sub, dp);
                    ptx::tmem_ld_wait();
                    if (masked) {
#pragma unroll
                        for (int x = 0; x < 16; ++x) s[x] = fmaf(s[x], scl, sMask[kc + 16 * sub + x]) - Ll;  // sMask holds mask * log2(e)
                    } else {  // no padded key in this sequence: the mask is never read
#pragma unroll
                        for (int x = 0; x < 16; ++x) s[x] = fmaf(s[x], scl, -Ll);
                    }
#pragma unroll
                    for (int x = 0; x < 16; ++x) {
                        const float pr = fast_exp2(s[x]);
                        const float m = ((bits >> (16 * sub + x)) & 1u) ? p.inv_keep : 0.f;      // dropout multiplier
                        s[x] = pr * m;                                                           // dropped probability (for dV)
                        dp[x] = (pr * sc) * fmaf(dp[x], m, -dl);                                 // dS = P (dP - delta) / sqrt(dh)
                    }
                    pdq[2 * sub] = pack8(s);
                    pdq[2 * sub + 1] = pack8(s + 8);
                    dsq[2 * sub] = pack8(dp);
                    dsq[2 * sub + 1] = pack8(dp + 8);
                }
                if (blk > 0) {
                    // the previous block's accumulating products read Pd / dS from shared memory: they must have
                    // retired before these stores (S / dP of THIS block were issued ahead of them)
                    ptx::mbar_wait(&bars[3], (blk - 1) & 1);
                    if (i == 0) {
                        // ... and with them dK / dV of the previous key block are final.  Drained HERE, after this block's
                        // arithmetic, so that the wait for those MMAs is already over (draining right behind the block
                        // that produced them exposed ~2500 cycles of it, profiles/r01_attn_bwd_timeline_v11.txt); this
                        // block's own accumulations, which restart dK / dV, are only issued after its arrive below.
                        ptx::tc_fence_after();
                        stage_acc(C_DK, sPd);
                        stage_acc(C_DV, sDS);
                        ptx::fence_proxy_async_smem();
                        named_bar_sync(1, BWD_SM_THREADS);
                        if (q4 == 0 && lane == 0) {
                            if (partial_kv) {
                                ptx::tma_reduce_add_4d(&tmDQKV, sPd + quad * 4096, 0, (j - 1) * 128 + quad * 32, p.nh + h, b);
                                ptx::tma_reduce_add_4d(&tmDQKV, sDS + quad * 4096, 0, (j - 1) * 128 + quad * 32, 2 * p.nh + h, b);
                            } else {
                                ptx::tma_store_4d(&tmDQKV, sPd + quad * 4096, 0, (j - 1) * 128 + quad * 32, p.nh + h, b);
                                ptx::tma_store_4d(&tmDQKV, sDS + quad * 4096, 0, (j - 1) * 128 + quad * 32, 2 * p.nh + h, b);
                            }
                            ptx::tma_store_commit();
                        }
                        if (p.gbias != nullptr) {
                            colsum_tile(sPd, (j - 1) * 128, bsum[1]);
                            colsum_tile(sDS, (j - 1) * 128, bsum[2]);
                        }
                        if (q4 == 0 && lane == 0) ptx::tma_store_wait_read<0>();
                        named_bar_sync(1, BWD_SM_THREADS);  // staging tiles free again
                        ptx::tc_fence_before();
                    }
                }
                {   // keys [kl, kl+32) -> key group kl/64, 16-byte chunks ((kl/32)&1)*4 .. +3 of row `row`
                    uint8_t* bp = sPd + (q4 >> 1) * 16384 + row * 128;
                    uint8_t* bs = sDS + (q4 >> 1) * 16384 + row * 128;
#pragma unroll
                    for (int x = 0; x < 4; ++x) {
                        const int chunk = ((q4 & 1) * 4 + x) ^ (row & 7);
                        *reinterpret_cast<bf16x8*>(bp + chunk * 16) = pdq[x];
                        *reinterpret_cast<bf16x8*>(bs + chunk * 16) = dsq[x];
                    }
                }
                ptx::fence_proxy_async_smem();
                ptx::tc_fence_before();
                ptx::mbar_arrive(&bars[2]);
                if (j == 0 && i == 0 && n_qt > 1) {
                    // delta of the second query tile, in the shadow of the hand-off to the MMA thread (its tiles were
                    // loaded behind block 0's)
                    ptx::mbar_wait(&bars[6], 0);
                    delta_part(sO1, sDO + 16384, 1);
                    named_bar_sync(1, BWD_SM_THREADS);
                    delta1 = delta_sum(1);
                }
                if (j == n_kh - 1 && i == n_qt - 1) {
                    // last block: everything that is still in TMEM -- dK / dV of this key block and every dQ tile
                    ptx::mbar_wait(&bars[3], blk & 1);
                    ptx::tc_fence_after();
                    stage_acc(C_DK, sPd);
                    stage_acc(C_DV, sDS);
                    stage_acc(C_DQ0, sPd + 16384);
                    if (n_qt > 1) stage_acc(C_DQ1, sDS + 16384);
                    ptx::fence_proxy_async_smem();
                    named_bar_sync(1, BWD_SM_THREADS);
                    if (q4 == 0 && lane == 0) {
                        if (partial_kv) {
                            ptx::tma_reduce_add_4d(&tmDQKV, sPd + quad * 4096, 0, j * 128 + quad * 32, p.nh + h, b);
                            ptx::tma_reduce_add_4d(&tmDQKV, sDS + quad * 4096, 0, j * 128 + quad * 32, 2 * p.nh + h, b);
                        } else {
                            ptx::tma_store_4d(&tmDQKV, sPd + quad * 4096, 0, j * 128 + quad * 32, p.nh + h, b);
                            ptx::tma_store_4d(&tmDQKV, sDS + quad * 4096, 0, j * 128 + quad * 32, 2 * p.nh + h, b);
                        }
                        ptx::tma_store_4d(&tmDQKV, sPd + 16384 + quad * 4096, 0, qbase + quad * 32, h, b);
                        if (n_qt > 1) ptx::tma_store_4d(&tmDQKV, sDS + 16384 + quad * 4096, 0, qbase + 128 + quad * 32, h, b);
                        ptx::tma_store_commit();
                    }
                    if (p.gbias != nullptr) {
                        colsum_tile(sPd, j * 128, bsum[1]);
                        colsum_tile(sDS, j * 128, bsum[2]);
                        colsum_tile(sPd + 16384, qbase, bsum[0]);
                        if (n_qt > 1) colsum_tile(sDS + 16384, qbase + 128, bsum[0]);
                    }
                    if (q4 == 0 && lane == 0) ptx::tma_store_wait_read<0>();
                    named_bar_sync(1, BWD_SM_THREADS);  // the bias-sum scratch below reuses Pd
                    ptx::tc_fence_before();
                }
                ++blk;
            }
        }
        if (p.gbias != nullptr) {
            // 16 warps x 3 slots x 64 columns of partial sums -> one fp32 atomic per column per CTA
            float* red = reinterpret_cast<float*>(sPd);  // [16][3][64]
#pragma unroll
            for (int s3 = 0; s3 < 3; ++s3) {
                red[(e * 3 + s3) * 64 + 2 * lane] = bsum[s3][0];
                red[(e * 3 + s3) * 64 + 2 * lane + 1] = bsum[s3][1];
            }
            named_bar_sync(1, BWD_SM_THREADS);
            if (t < 192) {
                float acc = 0.f;
#pragma unroll
                for (int w = 0; w < BWD_SM_WARPS; ++w) acc += red[w * 192 + t];
                atomicAdd(p.gbias + ((t >> 6) * p.nh + h) * DH + (t & 63), acc);
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<512>(tmem);
    }
}

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(f);
    }
    return fn;
}

// (dh, s, slot, b) view of a [B, S, slots*dh] bf16 tensor; box = {64, box_rows, 1, 1}, 128B swizzle
int head_map(CUtensorMap* m, const void* ptr, int B, int S, int slots, int box_rows) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) {
        polus_set_error("cuTensorMapEncodeTiled entry point not found");
        return POLUS_ERR_CUDA;
    }
    const cuuint64_t row = (cuuint64_t)slots * DH * 2;
    cuuint64_t dims[4] = {DH, (cuuint64_t)S, (cuuint64_t)slots, (cuuint64_t)B};
    cuuint64_t strides[3] = {row, DH * 2, row * (cuuint64_t)S};
    cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        polus_set_error("attention: cuTensorMapEncodeTiled failed (%d)", (int)r);
        return POLUS_ERR_INVALID;
    }
    return 0;
}

AttnParams make_params(int B, int S, int nh, float p_drop, uint64_t seed, uint32_t site, const uint32_t* d_step,
                       const int32_t* mask, float* lse, uint32_t* keepbits, float* gbias = nullptr) {
    AttnParams p;
    p.B = B; p.S = S; p.nh = nh;
    p.scale = 1.0f / sqrtf((float)DH);
    p.thresh16 = p_drop > 0.f ? (uint32_t)lrintf(p_drop * 65536.0f) : 0u;
    p.inv_keep = p_drop > 0.f ? 1.0f / (1.0f - p_drop) : 1.0f;
    p.seed = seed; p.site = site; p.d_step = d_step; p.mask = mask; p.lse = lse; p.keepbits = keepbits;
    p.gbias = gbias;
    p.pf_stride = 0;
    return p;
}

}  // namespace

extern "C" int polus_attention_supported(int S, int dh) { return (dh == DH && S >= 32 && S <= 512 && S % 32 == 0) ? 1 : 0; }
extern "C" size_t polus_attention_keepbits_words(int B, int S, int nh) { return (size_t)B * nh * S * (S / 32); }

extern "C" int polus_attention_fwd(const polus_bf16_t* qkv, const int32_t* mask, int B, int S, int nh, int dh, float p_drop,
                                   uint64_t seed, uint32_t site, const uint32_t* d_step, polus_bf16_t* ctx, float* lse,
                                   uint32_t* keepbits, void* stream) {
    POLUS_REQUIRE(polus_attention_supported(S, dh), "polus_attention_fwd: needs head_dim 64 and S <= 512, S %% 32 == 0 (got S=%d dh=%d)", S, dh);
    POLUS_REQUIRE(p_drop == 0.f || (d_step != nullptr && keepbits != nullptr), "polus_attention_fwd: dropout needs d_step and keepbits");
    if (B == 0) return 0;
    CUtensorMap tq, to;
    int rc = head_map(&tq, qkv, B, S, 3 * nh, 128);
    if (rc) return rc;
    rc = head_map(&to, ctx, B, S, nh, 32);
    if (rc) return rc;
    static bool set = false;
    if (!set) {
        POLUS_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdCfg<2>::SMEM));
        POLUS_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, FwdCfg<4>::SMEM));
        set = true;
    }
    AttnParams p = make_params(B, S, nh, p_drop, seed, site, d_step, mask, lse, keepbits);
    const int q_tiles = (S + 127) / 128;
    if (S <= 256)
        POLUS_CHECK_CUDA(polus_launch_pdl(attn_fwd_kernel<2>, dim3(B * nh * q_tiles), dim3(FwdCfg<2>::THREADS), FwdCfg<2>::SMEM, (cudaStream_t)stream, tq, to, p));
    else
        POLUS_CHECK_CUDA(polus_launch_pdl(attn_fwd_kernel<4>, dim3(B * nh * q_tiles), dim3(FwdCfg<4>::THREADS), FwdCfg<4>::SMEM, (cudaStream_t)stream, tq, to, p));
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

extern "C" int polus_attention_bwd(const polus_bf16_t* qkv, const int32_t* mask, const polus_bf16_t* ctx,
                                   const polus_bf16_t* dctx, const float* lse, int B, int S, int nh, int dh, float p_drop,
                                   uint64_t seed, uint32_t site, const uint32_t* d_step, const uint32_t* keepbits,
                                   polus_bf16_t* dqkv, float* gbias_qkv, void* stream) {
    POLUS_REQUIRE(polus_attention_supported(S, dh), "polus_attention_bwd: needs head_dim 64 and S <= 512, S %% 32 == 0 (got S=%d dh=%d)", S, dh);
    POLUS_REQUIRE(p_drop == 0.f || keepbits != nullptr, "polus_attention_bwd: dropout needs the forward's keepbits");
    if (B == 0) return 0;
    CUtensorMap tq, tdo, tdq, to;
    int rc = head_map(&tq, qkv, B, S, 3 * nh, 128);
    if (rc) return rc;
    rc = head_map(&tdo, dctx, B, S, nh, 128);
    if (rc) return rc;
    rc = head_map(&to, ctx, B, S, nh, 128);
    if (rc) return rc;
    rc = head_map(&tdq, dqkv, B, S, 3 * nh, 32);
    if (rc) return rc;
    static bool set = false;
    if (!set) {
        POLUS_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
        POLUS_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, B_SMEM));
        set = true;
    }
    POLUS_REQUIRE(p_drop == 0.f || d_step != nullptr, "polus_attention_bwd: dropout needs d_step");
    AttnParams p = make_params(B, S, nh, p_drop, seed, site, d_step, mask, const_cast<float*>(lse), const_cast<uint32_t*>(keepbits), gbias_qkv);
    p.pf_stride = polus_num_sms();   // CTA i warms the L2 for CTA i + (number of SMs): one wave ahead
    const int n_half = (S + 255) / 256;
    if (n_half > 1) {
        // two CTAs per head (one per 256-query half) add their dK / dV partial sums into dqkv with bf16 TMA reduce-adds:
        // the K and V column blocks [H, 3H) of every row start from zero (the dQ block is stored, not accumulated)
        const size_t H2 = (size_t)nh * DH * sizeof(polus_bf16_t);
        POLUS_CHECK_CUDA(cudaMemset2DAsync(reinterpret_cast<uint8_t*>(dqkv) + H2, 3 * H2, 0, 2 * H2, (size_t)B * S, (cudaStream_t)stream));
        attn_bwd_kernel<4><<<dim3(B * nh * n_half), dim3(BWD_THREADS), B_SMEM, (cudaStream_t)stream>>>(tq, tdo, tdq, to, p);
        POLUS_CHECK_CUDA(cudaGetLastError());
    } else {
        POLUS_CHECK_CUDA(polus_launch_pdl(attn_bwd_kernel<2>, dim3(B * nh), dim3(BWD_THREADS), B_SMEM, (cudaStream_t)stream, tq, tdo, tdq, to, p));
    }
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}
