// Batched bf16 GEMM on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM, operands staged
// by TMA with 128-byte swizzle).  C[b] = act(alpha * A[b] . B[b]^T + bias), fp32 accumulate.
//
// Replaces the cuBLAS calls TensorFlow makes on behalf of HF TFBertLayer (reference
// polus/models.py:205-213), the NER head Dense (polus/ner/models.py:36) and every gradient GEMM that
// tf.GradientTape derives from them (polus/training.py:185).
//
// Two variants of one kernel template:
//   CG = 2 (default for M > 128): a CTA PAIR (cluster 2x1x1, two SMs of one TPC) owns a 256 x BN tile and
//           issues tcgen05.mma.cta_group::2 (M = 256).  Each CTA stages its own 128 rows of A and HALF of the
//           B tile; the tensor cores read both halves.
//   CG = 1: one CTA owns a 128 x BN tile (small M, odd shapes).
// Kernel shape (persistent, warp-specialised, one CTA per SM, 384 threads):
//   warp 0      TMA producer       global -> smem ring (kStages x {A 128x64, B (BN/CG)x64} bf16)
//   warp 1      MMA issuer         one thread issues 4 x tcgen05.mma (K=16) per stage
//   warp 2      TMEM alloc/dealloc 2 x BN fp32 columns: accumulator double buffer
//   warps 4-11  epilogue           warp e owns TMEM lanes 32*(e%4).. and column half e/4:
//                                  tcgen05.ld -> alpha/bias/activation -> bf16 into a 128B-swizzled smem
//                                  staging block -> TMA store (coalesced, OOB-clipped); fp32 outputs
//                                  (split-K wgrad, atomics) are written straight from registers.
// Three mbarrier pipelines: smem full/empty, TMEM full/empty; tiles = batch x M/(128*CG) x N/BN x split_k.
// Either operand may be K-major (reduction dim contiguous) or MN-major (the other dim contiguous), so
// forward (X.W), dgrad (dY.W^T) and wgrad (X^T.dY) all read row-major tensors with no transposes.
//
// Round-1 measurement that shaped the epilogue: with per-thread row stores (each lane writing 16 B into a
// different row) a 128x256 tile took ~19 us to drain vs ~3 us of MMA for K=768 (profiles/r01_gemm_shapes_v2.log).
#include "common.cuh"
#include "ptx.cuh"
#include <cuda.h>
#include <atomic>

extern std::atomic<long long> g_launch_count;

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = one 128-byte swizzle row
constexpr int kEpiWarps = 8;
constexpr int A_STAGE_BYTES = BM * BK * 2;
constexpr int STG_BLOCK = 32 * 128;                       // one staging block: 32 rows x 64 bf16, swizzled
// Epilogue staging: ONE buffer per epilogue warp, 4 KB (a 32-row x 64-column bf16 block) or 8 KB when the launch also
// needs a second block (C2 output, the Emul multiplier tile, or the second 32-column half of an fp32 block).  Every byte
// not spent here is operand-ring depth, which is what the main loop lives on: with the former 2 x 8 KB per warp the
// 256-wide pair tile had 3 stages; 5-6 stages run the same shapes 1.2-1.35x faster (profiles/r01_gemm_stage_raster_exp.log).
constexpr int kSmemTotal = 227 * 1024;
constexpr int kBarBytes = 512;
constexpr int kMaxStages = 8;
constexpr int kGroupM = 8;  // m-tiles per rasterisation group (TcParams::group_m)

struct TcParams {
    int M, N, K;
    int batch0;
    int m_tiles, n_tiles, split_k, kb_total, kb_per_split;
    int num_tiles;
    int n_stages;     // operand-ring depth (<= kMaxStages)
    int stg_warp;     // staging bytes per epilogue warp: STG_BLOCK or 2 * STG_BLOCK
    int group_m;      // rasterisation: tiles are ordered in groups of group_m m-tiles x all n-tiles (m fastest inside a group)
    void* C;
    long long ldc, cbs0, cbs1;
    const float* bias;
    float alpha;
    int act;
    int c_f32;
    int accumulate;
    int has_c2;
    int c2_grad;      // C2 = act'(pre-activation) instead of the pre-activation
    int has_emul;     // C = (alpha A.B^T + bias) * Emul, Emul read through tmC2
    float* colsum;    // colsum[n] += sum_m C[m,n]
    int c2_u8;        // C2 (forward) / Emul (backward) holds gelu' as 8-bit fixed point (common.cuh d8_pack4): 16-warp kernel only
};

template <int BN, int CG>
struct Cfg {
    static_assert(BN == 64 || BN == 128 || BN == 256, "tile widths: 64, 128, 256");
    static_assert(CG == 1 || (CG == 2 && BN >= 128), "one CTA, or a pair that splits the B tile into 64-column multiples");
    static constexpr int BN_LOCAL = BN / CG;  // rows of the B tile this CTA stages
    static constexpr int B_GROUPS = BN_LOCAL / 64;  // MN-major B arrives in 64-column groups (one 128-byte swizzle atom wide)
    static constexpr int B_STAGE_BYTES = BN_LOCAL * BK * 2;
    static constexpr int kStageBytes = A_STAGE_BYTES + B_STAGE_BYTES;
    static constexpr int kTmemCols = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    static int stages(int stg_warp) {
        const int n = (kSmemTotal - 1024 - kEpiWarps * stg_warp - kBarBytes) / kStageBytes;
        return n > kMaxStages ? kMaxStages : n;
    }
    static int smem_bytes(int stg_warp) { return 1024 + stages(stg_warp) * kStageBytes + kEpiWarps * stg_warp + kBarBytes; }
    static constexpr int kColBlocks = BN / 64;                       // 64-column blocks per tile
    static constexpr int kEpiActive = kColBlocks >= 2 ? 8 : 4;        // epilogue warps that do work
    static constexpr int kBlocksPerWarp = kColBlocks >= 2 ? kColBlocks / 2 : 1;
};

__device__ __forceinline__ void red_add_v2(float* addr, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int ACT>
__device__ __forceinline__ void apply_act32(float* v) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = act_fwd(ACT, v[j]);
}
__device__ __forceinline__ void apply_act(int act, float* v) {
    switch (act) {  // one warp-uniform branch per 32 values, bodies fully unrolled
        case POLUS_ACT_GELU: apply_act32<POLUS_ACT_GELU>(v); break;
        case POLUS_ACT_RELU: apply_act32<POLUS_ACT_RELU>(v); break;
        case POLUS_ACT_SWISH: apply_act32<POLUS_ACT_SWISH>(v); break;
        case POLUS_ACT_TANH: apply_act32<POLUS_ACT_TANH>(v); break;
        case POLUS_ACT_MISH: apply_act32<POLUS_ACT_MISH>(v); break;
        default: break;
    }
}

// y = act(x) and d = act'(x), 32 values, sharing the transcendental work (GELU: one rcp + one ex2 for both)
template <int ACT>
__device__ __forceinline__ void act_fwd_grad32(float* v, float* d) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const float x = v[j];
        if (ACT == POLUS_ACT_GELU) {
            float cdf, pdf;
            gelu_cdf_pdf(x, cdf, pdf);
            v[j] = x * cdf;
            d[j] = fmaf(x, pdf, cdf);
        } else {
            v[j] = act_fwd(ACT, x);
            d[j] = act_grad(ACT, x);
        }
    }
}
__device__ __forceinline__ void apply_act_grad(int act, float* v, float* d) {
    switch (act) {
        case POLUS_ACT_GELU: act_fwd_grad32<POLUS_ACT_GELU>(v, d); break;
        case POLUS_ACT_RELU: act_fwd_grad32<POLUS_ACT_RELU>(v, d); break;
        case POLUS_ACT_SWISH: act_fwd_grad32<POLUS_ACT_SWISH>(v, d); break;
        case POLUS_ACT_TANH: act_fwd_grad32<POLUS_ACT_TANH>(v, d); break;
        case POLUS_ACT_MISH: act_fwd_grad32<POLUS_ACT_MISH>(v, d); break;
        default:
#pragma unroll
            for (int j = 0; j < 32; ++j) d[j] = 1.0f;
            break;
    }
}

// 32 fp32 -> 32 bf16 into row `lane` of a swizzled [32 rows][128 B] block; `half` selects the 64-byte half.
__device__ __forceinline__ void stage_row(uint8_t* block, int lane, int half, const float* v) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int chunk = (half * 4 + j) ^ (lane & 7);  // 128B swizzle: 16-byte chunk index XOR row%8
        *reinterpret_cast<bf16x8*>(block + lane * 128 + chunk * 16) = pack8(v + 8 * j);
    }
}

// 8 fp32 -> 8 bf16 into 16-byte chunk `chunk` (0..7) of row `lane`
__device__ __forceinline__ void stage8(uint8_t* block, int lane, int chunk, const float* v8) {
    *reinterpret_cast<bf16x8*>(block + lane * 128 + ((chunk ^ (lane & 7)) << 4)) = pack8(v8);
}
// y = act(x), d = act'(x) for 8 values
__device__ __forceinline__ void act_fwd_grad8(int act, float* v, float* d) {
    if (act == POLUS_ACT_GELU) {  // the case that matters (warp-uniform branch): two values per instruction
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            float2 y2, d2;
            gelu_fwd_grad2(make_float2(v[j], v[j + 1]), y2, d2);
            v[j] = y2.x;
            v[j + 1] = y2.y;
            d[j] = d2.x;
            d[j + 1] = d2.y;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float x = v[j];
            v[j] = act_fwd(act, x);
            d[j] = act_grad(act, x);
        }
    }
}

// 32 fp32 (one 128-byte row) into row `lane` of a swizzled [32 rows][128 B] block
__device__ __forceinline__ void stage_row_f32(uint8_t* block, int lane, const float* v) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int chunk = j ^ (lane & 7);
        *reinterpret_cast<float4*>(block + lane * 128 + chunk * 16) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
}

template <int BN, bool A_MN, bool B_MN, int CG, int EPI>
__global__ void __launch_bounds__(128 + 32 * EPI, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmC2, const TcParams p) {
    using C = Cfg<BN, CG>;
    const int kStages = p.n_stages;
    constexpr int BN_LOCAL = C::BN_LOCAL;
    constexpr int B_STAGE_BYTES = C::B_STAGE_BYTES;
    constexpr uint32_t kStageTx = C::kStageBytes * CG;  // bytes landing on the leader's barrier per k-block
    const uint32_t cta_rank = CG == 2 ? ptx::cluster_ctarank() : 0u;  // position inside the pair
    const bool is_leader = cta_rank == 0;
    const int tile0 = (int)(blockIdx.x / CG);
    const int tile_step = (int)(gridDim.x / CG);

    // 1024-byte alignment (128B-swizzle atoms) comes from the declaration, which also keeps the pointer in the shared
    // address space for the compiler (LDS / STS instead of generic LD / ST in the staging code)
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((ptx::smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* sA = smem;
    uint8_t* sB = smem + kStages * A_STAGE_BYTES;
    uint8_t* sStage = smem + kStages * (A_STAGE_BYTES + B_STAGE_BYTES);  // 1024-aligned (stage sizes are multiples of 4 KB)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(sStage + kEpiWarps * p.stg_warp);
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tfull_bar = empty_bar + kMaxStages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* emul_bar = tempty_bar + 2;  // [epilogue warp]: Emul tile landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(emul_bar + 4 * kEpiWarps);  // (16-warp kernel, 8-bit multipliers: two barriers per warp)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    pdl_trigger();  // the next kernel may start its own prologue as soon as SMs free up
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tmA);
        ptx::prefetch_tensormap(&tmB);
        ptx::prefetch_tensormap(&tmC);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            ptx::mbar_init(&tfull_bar[s], 1);
            ptx::mbar_init(&tempty_bar[s], (EPI == 16 ? 16 : C::kEpiActive) * CG);  // one arrive per working epilogue warp of the group
        }
        for (int s = 0; s < 4 * kEpiWarps; ++s) ptx::mbar_init(&emul_bar[s], 1);
        ptx::fence_barrier_init();
    }
    if (warp == 2) {
        if (CG == 2) ptx::tmem_alloc_2sm<C::kTmemCols>(tmem_slot);
        else ptx::tmem_alloc<C::kTmemCols>(tmem_slot);
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (CG > 1) ptx::cluster_sync();  // peer barriers initialised before any remote arrive / multicast commit
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();  // operands / outputs of earlier kernels are touched only from here on

    auto decode = [&](int t, int& mt, int& nt, int& sp, int& b0, int& b1) {
        const int mn = p.m_tiles * p.n_tiles;
        const int r = t % mn;
        t /= mn;
        const int per_group = p.group_m * p.n_tiles;
        const int g = r / per_group;
        const int gm = min(p.group_m, p.m_tiles - g * p.group_m);  // the last group may be narrower
        const int rr = r - g * per_group;
        mt = g * p.group_m + rr % gm;
        nt = rr / gm;
        sp = t % p.split_k;
        t /= p.split_k;
        b0 = t % p.batch0;
        b1 = t / p.batch0;
    };

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            auto load = [&](void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
                if (CG == 2) ptx::tma_load_4d_2sm(dst, map, bar, c0, c1, c2, c3);
                else ptx::tma_load_4d(dst, map, bar, c0, c1, c2, c3);
            };
            for (int t = tile0; t < p.num_tiles; t += tile_step) {
                int mt, nt, sp, b0, b1;
                decode(t, mt, nt, sp, b0, b1);
                const int kb0 = sp * p.kb_per_split;
                const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
                const int m0 = (mt * CG + (int)cta_rank) * BM;      // this CTA's 128 rows of A / C
                const int n0 = nt * BN + (int)cta_rank * BN_LOCAL;  // this CTA's share of the B tile
                for (int kb = kb0; kb < kb1; ++kb) {
                    ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (is_leader) ptx::mbar_expect_tx(&full_bar[stage], kStageTx);
                    uint8_t* a = sA + stage * A_STAGE_BYTES;
                    uint8_t* b = sB + stage * B_STAGE_BYTES;
                    if (!A_MN) {
                        load(a, &tmA, &full_bar[stage], kb * BK, m0, b0, b1);
                    } else {
#pragma unroll
                        for (int g = 0; g < BM / 64; ++g)
                            load(a + g * (BK * 128), &tmA, &full_bar[stage], m0 + g * 64, kb * BK, b0, b1);
                    }
                    if (!B_MN) {
                        load(b, &tmB, &full_bar[stage], kb * BK, n0, b0, b1);
                    } else {
#pragma unroll
                        for (int g = 0; g < C::B_GROUPS; ++g)
                            load(b + g * (BK * 128), &tmB, &full_bar[stage], n0 + g * 64, kb * BK, b0, b1);
                    }
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        if (lane == 0 && is_leader) {
            constexpr uint32_t idesc = ptx::umma_idesc_bf16(BM * CG, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
            const uint64_t adesc_base = A_MN ? ptx::umma_desc_base(BK * 128, 1024) : ptx::umma_desc_base(16, 1024);
            const uint64_t bdesc_base = B_MN ? ptx::umma_desc_base(BK * 128, 1024) : ptx::umma_desc_base(16, 1024);
            constexpr uint32_t a_kstep = A_MN ? 2048 : 32;  // bytes per UMMA_K=16 step
            constexpr uint32_t b_kstep = B_MN ? 2048 : 32;
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int t = tile0; t < p.num_tiles; t += tile_step) {
                int mt, nt, sp, b0, b1;
                decode(t, mt, nt, sp, b0, b1);
                const int kb0 = sp * p.kb_per_split;
                const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
                ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                ptx::tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = kb0; kb < kb1; ++kb) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t a_addr = ptx::smem_u32(sA + stage * A_STAGE_BYTES);
                    const uint32_t b_addr = ptx::smem_u32(sB + stage * B_STAGE_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        const uint64_t ad = ptx::umma_desc(adesc_base, a_addr + k * a_kstep);
                        const uint64_t bd = ptx::umma_desc(bdesc_base, b_addr + k * b_kstep);
                        const uint32_t accum = (kb > kb0 || k > 0) ? 1u : 0u;
                        if (CG == 2) ptx::umma_bf16_2sm(tmem_d, ad, bd, idesc, accum);
                        else ptx::umma_bf16(tmem_d, ad, bd, idesc, accum);
                    }
                    // smem slot reusable (in both CTAs of the pair) once these MMAs retire
                    if (CG == 2) ptx::umma_commit_2sm(&empty_bar[stage]);
                    else ptx::umma_commit(&empty_bar[stage]);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                // accumulator complete -> epilogue warps of both CTAs
                if (CG == 2) ptx::umma_commit_2sm(&tfull_bar[acc]);
                else ptx::umma_commit(&tfull_bar[acc]);
                if (++acc == 2) {
                    acc = 0;
                    acc_phase ^= 1;
                }
            }
        }
    } else if (EPI == 16 && warp >= 4) {
        // ------------------------------------------------------------ epilogue, 16 warps (bf16 outputs with per-element
        // math: activation + derivative, multiplier tile + column sums).  With 8 warps those epilogues ran at IPC 0.28 per
        // scheduler -- two resident warps cannot cover MUFU / TMEM-load / shared-memory latency -- and paced the whole GEMM.
        // Every warp works alone on 32-row x 32-column blocks (TMEM lanes 32*quad.., column chunks (e/4)*kCPW + i of the
        // tile): its own 2 KB staging tile for C and 2 KB for C2 / the multiplier tile, 64-byte-swizzled, moved by TMA boxes
        // of 32 x 32.  No barrier between warps: the first 16-warp version paired warps on 64-column blocks and spent 19 %
        // of its samples in the pair's bar.sync (profiles/r01_ncu_summary_v13_emul.txt).
        const int e = warp - 4;
        const int quad = e & 3;
        const int csub = e >> 2;
        constexpr int kCPW = (BN / 32) / 4 > 0 ? (BN / 32) / 4 : 1;  // 32-column chunks per warp per tile
        const uint32_t sC = ptx::smem_u32(sStage) + (uint32_t)e * 4096u;  // [32 rows][64 B] C
        const uint32_t sX = sC + 2048u;                                    // [32 rows][64 B] C2 or multiplier
        const uint32_t swz = (uint32_t)((lane >> 1) & 3);                 // 64B swizzle: 16-byte chunk index ^ (row/2)%4
        int acc = 0;
        uint32_t acc_phase = 0;
        bool store_pending = false;
        int nblk = 0;
        auto blk_valid = [&](int t, int i) -> bool {
            if (t >= p.num_tiles || i >= kCPW) return false;
            int mt, nt, sp, b0, b1;
            decode(t, mt, nt, sp, b0, b1);
            return nt * BN + (csub * kCPW + i) * 32 < p.N;
        };
        auto advance = [&](int& t, int& i) {
            ++i;
            while (t < p.num_tiles && !blk_valid(t, i)) {
                t += tile_step;
                i = 0;
            }
        };
        // Multiplier tiles.  bf16: one 2 KB tile per warp, fetched one block ahead.  8-bit: the same 2 KB hold TWO 1 KB
        // tiles with a barrier each, fetched two blocks ahead -- the bf16 path waits on this load at every block (halving
        // its bytes alone changed nothing: 157.0 vs 156.3 us, profiles/r02_gemm_d8.log).
        auto emul_issue = [&](int t, int i, int buf) {
            if (lane == 0) {
                int mt, nt, sp, b0, b1;
                decode(t, mt, nt, sp, b0, b1);
                uint64_t* ebar = &emul_bar[buf * 16 + e];
                const uint32_t dstX = sX + (uint32_t)buf * 1024u;
                ptx::mbar_expect_tx(ebar, p.c2_u8 ? 1024 : 2048);   // 32 x 32 multipliers, bf16 or 8-bit
                asm volatile(
                    "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                    ::"r"(dstX), "l"(reinterpret_cast<uint64_t>(&tmC2)), "r"(ptx::smem_u32(ebar)),
                    "r"(nt * BN + (csub * kCPW + i) * 32), "r"((mt * CG + (int)cta_rank) * BM + quad * 32), "r"(b0), "r"(b1)
                    : "memory");
            }
        };
        auto sts16 = [&](uint32_t tile, int chunk, const float* v8) {  // 8 values -> 16-byte chunk `chunk` of row `lane`
            const bf16x8 q = pack8(v8);
            const uint32_t* u = reinterpret_cast<const uint32_t*>(&q);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(tile + (uint32_t)lane * 64u + (((uint32_t)chunk ^ swz) << 4)),
                         "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]) : "memory");
        };
        auto tma_store32 = [&](const CUtensorMap* map, uint32_t tile, int c0, int c1, int c2, int c3) {
            asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                         ::"l"(reinterpret_cast<uint64_t>(map)), "r"(tile), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
        };
        int pf_t = tile0, pf_i = -1;
        if (p.has_emul) {
            advance(pf_t, pf_i);
            if (pf_t < p.num_tiles) emul_issue(pf_t, pf_i, 0);
            if (p.c2_u8) {
                advance(pf_t, pf_i);
                if (pf_t < p.num_tiles) emul_issue(pf_t, pf_i, 1);
            }
        }
        for (int t = tile0; t < p.num_tiles; t += tile_step) {
            int mt, nt, sp, b0, b1;
            decode(t, mt, nt, sp, b0, b1);
            ptx::mbar_wait(&tfull_bar[acc], acc_phase);
            ptx::tc_fence_after();
            const int row0 = (mt * CG + (int)cta_rank) * BM + quad * 32;
            const bool add_bias = (p.bias != nullptr) && (sp == 0);
#pragma unroll 1
            for (int i = 0; i < kCPW; ++i) {
                const int cc = csub * kCPW + i;
                const int col0 = nt * BN + cc * 32;
                if (col0 >= p.N) break;  // warp-uniform
                if (store_pending) {
                    if (lane == 0) ptx::tma_store_wait_read<0>();  // the previous block's stores have read the tiles
                    __syncwarp();
                    store_pending = false;
                }
                const uint32_t tcol = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + cc * 32;
                const bool full32 = p.N - col0 >= 32;
                if (p.has_c2 && p.c2_grad && full32) {
                    // activation + derivative (the FFN-up GEMM): 16 accumulator columns at a time; the second half's
                    // tcgen05.ld is in flight while the first half is processed (21 % of this path's stall samples were
                    // long-scoreboard waits behind the loads, profiles/r02_ncu_gemm_ffn1.txt)
                    float va[16], vb[16];
                    ptx::tmem_ld16(tcol, va);
#pragma unroll
                    for (int sub = 0; sub < 2; ++sub) {
                        float* v = sub == 0 ? va : vb;
                        ptx::tmem_ld_wait();
                        if (sub == 0) ptx::tmem_ld16(tcol + 16, vb);
                        if (p.alpha != 1.0f) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) v[j] *= p.alpha;
                        }
                        if (add_bias) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + sub * 16) + j);
                                v[4 * j] += bv.x;
                                v[4 * j + 1] += bv.y;
                                v[4 * j + 2] += bv.z;
                                v[4 * j + 3] += bv.w;
                            }
                        }
                        uint32_t dq[4];  // 8-bit derivative: this half's 16 values = one 16-byte store into the [32][32 B] tile
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            float d8[8];
                            act_fwd_grad8(p.act, v + 8 * j, d8);
                            if (p.c2_u8) {
                                dq[2 * j] = d8_pack4(d8[0], d8[1], d8[2], d8[3]);
                                dq[2 * j + 1] = d8_pack4(d8[4], d8[5], d8[6], d8[7]);
                            } else {
                                sts16(sX, sub * 2 + j, d8);
                            }
                            sts16(sC, sub * 2 + j, v + 8 * j);
                        }
                        if (p.c2_u8)
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sX + (uint32_t)lane * 32u + (uint32_t)sub * 16u),
                                         "r"(dq[0]), "r"(dq[1]), "r"(dq[2]), "r"(dq[3]) : "memory");
                    }
                } else {
                    float v[32];
                    ptx::tmem_ld32(tcol, v);
                    ptx::tmem_ld_wait();
                    const int nvalid = min(32, p.N - col0);
                    if (p.alpha != 1.0f) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] *= p.alpha;
                    }
                    if (add_bias) {
                        if (full32) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + j);
                                v[4 * j] += bv.x;
                                v[4 * j + 1] += bv.y;
                                v[4 * j + 2] += bv.z;
                                v[4 * j + 3] += bv.w;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < nvalid) v[j] += __ldg(p.bias + col0 + j);
                        }
                    }
                    if (p.has_emul) {
                        const int ebuf = p.c2_u8 ? (nblk & 1) : 0;
                        ptx::mbar_wait(&emul_bar[ebuf * 16 + e], p.c2_u8 ? (((uint32_t)nblk >> 1) & 1u) : ((uint32_t)nblk & 1u));
                        if (p.c2_u8) {   // [32 rows][32 bytes], not swizzled: row `lane` = two 16-byte loads
#pragma unroll
                            for (int j = 0; j < 2; ++j) {
                                uint32_t u[4];
                                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3])
                                             : "r"(sX + (uint32_t)ebuf * 1024u + (uint32_t)lane * 32u + (uint32_t)j * 16u));
#pragma unroll
                                for (int w = 0; w < 4; ++w) {
                                    float m4[4];
                                    d8_unpack4(u[w], m4);
#pragma unroll
                                    for (int x = 0; x < 4; ++x) v[16 * j + 4 * w + x] *= m4[x];
                                }
                            }
                        } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            bf16x8 q;
                            uint32_t* u = reinterpret_cast<uint32_t*>(&q);
                            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3])
                                         : "r"(sX + (uint32_t)lane * 64u + (((uint32_t)j ^ swz) << 4)));
                            float m8[8];
                            unpack8(q, m8);
#pragma unroll
                            for (int x = 0; x < 8; ++x) v[8 * j + x] *= m8[x];
                        }
                        }
                        __syncwarp();  // every lane has its multipliers: the tile may be refilled
                        advance(pf_t, pf_i);
                        if (pf_t < p.num_tiles) emul_issue(pf_t, pf_i, ebuf);
                    } else {
                        if (p.has_c2) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) sts16(sX, j, v + 8 * j);  // pre-activation copy
                        }
                        apply_act(p.act, v);
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) sts16(sC, j, v + 8 * j);
                }
                ptx::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    tma_store32(&tmC, sC, col0, row0, b0, b1);  // rows >= M / columns >= N are clipped by the tensor map
                    if (p.has_c2) tma_store32(&tmC2, sX, col0, row0, b0, b1);
                    ptx::tma_store_commit();
                }
                store_pending = true;
                if (p.colsum != nullptr) {
                    // column sums of the staged (bf16-rounded) 32 x 32 block: lane L = column L, four independent chains
                    const int nrows = min(32, p.M - row0);
                    float s[4] = {0.f, 0.f, 0.f, 0.f};
                    const uint32_t cb16 = (uint32_t)(lane >> 3), off = (uint32_t)(lane & 7) * 2u;
#pragma unroll
                    for (int r = 0; r < 32; ++r) {
                        uint32_t w;
                        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(w) : "r"(sC + (uint32_t)r * 64u + ((cb16 ^ (uint32_t)((r >> 1) & 3)) << 4) + off));
                        if (r < nrows) s[r & 3] += __uint_as_float(w << 16);
                    }
                    if (col0 + lane < p.N) atomicAdd(p.colsum + col0 + lane, (s[0] + s[1]) + (s[2] + s[3]));
                }
                ++nblk;
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CG == 2) ptx::mbar_arrive_remote(&tempty_bar[acc], 0);
                else ptx::mbar_arrive(&tempty_bar[acc]);
            }
            if (++acc == 2) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
        if (lane == 0) ptx::tma_store_wait_all();  // smem must outlive the bulk stores
    } else if (EPI == 8 && warp >= 4 && (warp - 4) < C::kEpiActive) {
        // ------------------------------------------------------------ epilogue (TMEM lane = row)
        const int e = warp - 4;
        const int quad = e & 3;   // TMEM lanes [32*quad, 32*quad+32)  (hardware: warp_id % 4)
        const int half = e >> 2;  // which half of the tile's 64-column blocks
        uint8_t* stg = sStage + e * p.stg_warp;  // [C | C2 or Emul or second fp32 half]
        int acc = 0;
        uint32_t acc_phase = 0;
        int stores_in_flight = 0;
        int nblk = 0;  // blocks staged so far (phase of this warp's Emul barrier)
        // ---- Emul prefetch: the multiplier tile of block n+1 is fetched by TMA into the second half of the staging
        // buffer as soon as block n's has been consumed into registers.
        auto blk_valid = [&](int t, int i) -> bool {
            if (t >= p.num_tiles || i >= C::kBlocksPerWarp) return false;
            int mt, nt, sp, b0, b1;
            decode(t, mt, nt, sp, b0, b1);
            return half * C::kBlocksPerWarp + i < C::kColBlocks && nt * BN + (half * C::kBlocksPerWarp + i) * 64 < p.N;
        };
        auto advance = [&](int& t, int& i) {
            ++i;
            while (t < p.num_tiles && !blk_valid(t, i)) {
                t += tile_step;
                i = 0;
            }
        };
        auto emul_issue = [&](int t, int i) {
            if (lane == 0) {
                int mt, nt, sp, b0, b1;
                decode(t, mt, nt, sp, b0, b1);
                uint64_t* bar = &emul_bar[e];
                ptx::mbar_expect_tx(bar, STG_BLOCK);
                ptx::tma_load_4d(stg + STG_BLOCK, &tmC2, bar, nt * BN + (half * C::kBlocksPerWarp + i) * 64,
                                 (mt * CG + (int)cta_rank) * BM + quad * 32, b0, b1);
            }
        };
        int pf_t = tile0, pf_i = -1;
        if (p.has_emul) {
            advance(pf_t, pf_i);
            if (pf_t < p.num_tiles) emul_issue(pf_t, pf_i);
        }
        for (int t = tile0; t < p.num_tiles; t += tile_step) {
            int mt, nt, sp, b0, b1;
            decode(t, mt, nt, sp, b0, b1);
            ptx::mbar_wait(&tfull_bar[acc], acc_phase);
            ptx::tc_fence_after();
            const int row0 = (mt * CG + (int)cta_rank) * BM + quad * 32;
            const bool add_bias = (p.bias != nullptr) && (sp == 0);
#pragma unroll 1
            for (int i = 0; i < C::kBlocksPerWarp; ++i) {
                const int cb = half * C::kBlocksPerWarp + i;
                const int colb = nt * BN + cb * 64;
                if (cb >= C::kColBlocks || colb >= p.N) break;  // warp-uniform
                uint8_t* blkC = stg;
                uint8_t* blkC2 = stg + STG_BLOCK;
                if (stores_in_flight) {
                    // the TMA store of the previous block must be done reading the staging buffer
                    if (lane == 0) ptx::tma_store_wait_read<0>();
                    __syncwarp();
                    stores_in_flight = 0;
                }
                if (p.has_emul) ptx::mbar_wait(&emul_bar[e], (uint32_t)nblk & 1u);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int col0 = colb + h * 32;
                    if (col0 < p.N) {  // warp-uniform; columns >= N of a staged block are clipped by the TMA store
                        float v[32];
                        ptx::tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + cb * 64 + h * 32, v);
                        ptx::tmem_ld_wait();
                        const int nvalid = min(32, p.N - col0);
                        if (p.alpha != 1.0f) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] *= p.alpha;
                        }
                        if (add_bias) {
                            if (nvalid == 32) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) {
                                    const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + j);
                                    v[4 * j] += bv.x;
                                    v[4 * j + 1] += bv.y;
                                    v[4 * j + 2] += bv.z;
                                    v[4 * j + 3] += bv.w;
                                }
                            } else {
#pragma unroll
                                for (int j = 0; j < 32; ++j)
                                    if (j < nvalid) v[j] += __ldg(p.bias + col0 + j);
                            }
                        }
                        if (p.c_f32) {
                            // fp32 output: the two 32-column chunks of this block use the buffer's two 4 KB halves
                            apply_act(p.act, v);
                            stage_row_f32(h == 0 ? blkC : blkC2, lane, v);
                        } else if (p.has_emul) {
                            // multiplier tile (rows >= M / columns >= N arrive as zeros): same swizzled layout as the staging block
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                float m8[8];
                                unpack8(*reinterpret_cast<const bf16x8*>(blkC2 + lane * 128 + (((h * 4 + j) ^ (lane & 7)) << 4)), m8);
#pragma unroll
                                for (int x = 0; x < 8; ++x) v[8 * j + x] *= m8[x];
                            }
                            stage_row(blkC, lane, h, v);
                        } else if (p.has_c2 && p.c2_grad) {
                            float d[32];
                            apply_act_grad(p.act, v, d);
                            stage_row(blkC2, lane, h, d);  // act'(z): the next layer's dgrad multiplies by it
                            stage_row(blkC, lane, h, v);
                        } else {
                            if (p.has_c2) stage_row(blkC2, lane, h, v);  // pre-activation copy
                            apply_act(p.act, v);
                            stage_row(blkC, lane, h, v);
                        }
                    }
                }
                ptx::fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA engine
                __syncwarp();
                if (p.has_emul) {
                    // every lane has consumed this block's multiplier tile (program order + the fence/syncwarp above):
                    // fetch the next block's now, so that it lands while this warp waits for its next accumulator
                    advance(pf_t, pf_i);
                    if (pf_t < p.num_tiles) emul_issue(pf_t, pf_i);
                }
                if (lane == 0) {
                    // rows >= M and columns >= N are clipped by the tensor map
                    if (p.c_f32) {
                        if (p.accumulate) {  // split-K / shared-variable gradients: fp32 add performed by the TMA unit at L2
                            ptx::tma_reduce_add_4d(&tmC, blkC, colb, row0, b0, b1);
                            if (colb + 32 < p.N) ptx::tma_reduce_add_4d(&tmC, blkC2, colb + 32, row0, b0, b1);
                        } else {
                            ptx::tma_store_4d(&tmC, blkC, colb, row0, b0, b1);
                            if (colb + 32 < p.N) ptx::tma_store_4d(&tmC, blkC2, colb + 32, row0, b0, b1);
                        }
                    } else {
                        ptx::tma_store_4d(&tmC, blkC, colb, row0, b0, b1);
                        if (p.has_c2) ptx::tma_store_4d(&tmC2, blkC2, colb, row0, b0, b1);
                    }
                    ptx::tma_store_commit();
                }
                if (p.colsum != nullptr && !p.c_f32) {
                    // column sums of the staged (bf16-rounded) block: lane L owns columns 2L, 2L+1 -- word L of every row,
                    // so each row is read as one conflict-free 128-byte wavefront
                    const int nrows = min(32, p.M - row0);
                    float s0 = 0.f, s1 = 0.f;
#pragma unroll 8
                    for (int r = 0; r < 32; ++r) {
                        if (r < nrows) {
                            const uint32_t w = *reinterpret_cast<const uint32_t*>(blkC + r * 128 + ((((lane >> 2) ^ (r & 7))) << 4) + (lane & 3) * 4);
                            s0 += __uint_as_float(w << 16);
                            s1 += __uint_as_float(w & 0xFFFF0000u);
                        }
                    }
                    const int c = colb + 2 * lane;
                    if (c < p.N) atomicAdd(p.colsum + c, s0);
                    if (c + 1 < p.N) atomicAdd(p.colsum + c + 1, s1);
                }
                ++stores_in_flight;
                ++nblk;
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CG == 2) ptx::mbar_arrive_remote(&tempty_bar[acc], 0);  // the pair leader's MMA thread waits on it
                else ptx::mbar_arrive(&tempty_bar[acc]);
            }
            if (++acc == 2) {
                acc = 0;
                acc_phase ^= 1;
            }
        }
        if (lane == 0) ptx::tma_store_wait_all();  // smem must outlive the bulk stores
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (CG > 1) ptx::cluster_sync();  // the peer may still be reading our smem / arriving on our barriers
    if (warp == 2) {
        ptx::tc_fence_after();
        if (CG == 2) ptx::tmem_dealloc_2sm<C::kTmemCols>(tmem_base);
        else ptx::tmem_dealloc<C::kTmemCols>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(f);
    }
    return fn;
}

// 4-D bf16 view (dim0 contiguous, rows, batch0, batch1); box = {64, box_rows, 1, 1}, 128-byte swizzle.
int encode_map(CUtensorMap* map, const void* ptr, long long inner, long long rows, long long ld, int batch0,
               long long bs0, int batch1, long long bs1, int box_rows, int esize = 2, int box_bytes = 128) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) {
        polus_set_error("cuTensorMapEncodeTiled entry point not found (driver too old?)");
        return POLUS_ERR_CUDA;
    }
    cuuint64_t dims[4] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)batch0, (cuuint64_t)batch1};
    cuuint64_t strides[3];
    cuuint32_t box[4] = {(cuuint32_t)(box_bytes / esize), (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    strides[0] = (cuuint64_t)ld * esize;
    strides[1] = (cuuint64_t)(batch0 > 1 ? bs0 * esize : rows * ld * esize);
    strides[2] = (cuuint64_t)(batch1 > 1 ? bs1 * esize : strides[1] * (cuuint64_t)batch0);
    CUresult r = enc(map, esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : (esize == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16), 4,
                     const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     box_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_NONE : (box_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B),
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        polus_set_error("cuTensorMapEncodeTiled failed (%d): ptr=%p inner=%lld rows=%lld ld=%lld b0=%d/%lld b1=%d/%lld",
                        (int)r, ptr, inner, rows, ld, batch0, bs0, batch1, bs1);
        return POLUS_ERR_INVALID;
    }
    return 0;
}

int make_map(CUtensorMap* map, const polus_operand_t& op, long long mn_len, long long k_len, int batch0, int batch1,
             int box_mn) {
    const long long inner = op.mn_major ? mn_len : k_len;
    const long long rows = op.mn_major ? k_len : mn_len;
    return encode_map(map, op.ptr, inner, rows, op.ld, batch0, op.bs0, batch1, op.bs1, op.mn_major ? BK : box_mn);
}

template <int BN, bool A_MN, bool B_MN, int CG, int EPI = 8>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tc2,
           const TcParams& p_in, cudaStream_t st) {
    auto kern = gemm_tc_kernel<BN, A_MN, B_MN, CG, EPI>;
    using C = Cfg<BN, CG>;
    static bool attr_set = false;
    if (!attr_set) {
        POLUS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal));
        attr_set = true;
    }
    TcParams p = p_in;
    p.n_stages = C::stages(p.stg_warp);
    POLUS_REQUIRE(p.n_stages >= 2, "polus_gemm_tc: operand ring needs at least two stages");
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(128 + 32 * EPI);
    cfg.dynamicSmemBytes = C::smem_bytes(p.stg_warp);
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    int groups = polus_num_sms() / CG;
    if (p.num_tiles < groups) groups = p.num_tiles;
    cfg.gridDim = dim3(groups * CG);
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    POLUS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, tc2, p));
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

template <int BN, int CG>
int launch_major(int a_mn, int b_mn, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
                 const CUtensorMap& tc2, const TcParams& p, cudaStream_t st) {
    if (!a_mn && !b_mn) return launch<BN, false, false, CG>(ta, tb, tc, tc2, p, st);
    if (!a_mn && b_mn) return launch<BN, false, true, CG>(ta, tb, tc, tc2, p, st);
    if (a_mn && !b_mn) return launch<BN, true, false, CG>(ta, tb, tc, tc2, p, st);
    return launch<BN, true, true, CG>(ta, tb, tc, tc2, p, st);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct TilePlan {
    int CG;      // CTAs per tile: 2 = a CTA pair on a 256-row tile, 1 = one CTA on a 128-row tile
    int BN;      // tile width: 64, 128 or 256
    int split;   // K splits (before clamping to the number of k-blocks)
    bool epi16;  // 16-epilogue-warp kernel
};

// The one place that picks the kernel for a problem: the dispatch in polus_gemm_tc launches what this returns, and
// why_unsupported accepts the 8-bit derivative only where it returns the 16-warp kernel.
TilePlan plan_tiles(const polus_gemm_t* g, int sms) {
    const int batch0 = g->batch0 < 1 ? 1 : g->batch0;
    const int batch1 = g->batch1 < 1 ? 1 : g->batch1;
    TilePlan t;
    // CTA pairs (cta_group::2, 256-row tiles) whenever there are at least two 128-row tiles to pair up
    t.CG = (g->M > BM && g->N > 64) ? 2 : 1;
    const long long mt = cdiv(g->M, BM * t.CG);
    const long long nb = (long long)batch0 * batch1;
    const int kb_total = cdiv(g->K, BK);
    const long long groups = sms / t.CG;
    // Tile width and split-K.
    //  * accumulate GEMMs with split_k == 0 (wgrad: few output tiles, very long K): 256-wide tiles whenever N allows
    //    (a 128-wide pair tile needs 96 B/clk/SM of operand traffic, more than L2 delivers) and the split that
    //    minimises waves x (k-blocks per split + fixed tile overhead).
    //  * everything else: the widest tile that still yields one full wave of CTAs.
    const bool wgrad = g->split_k == 0 && g->accumulate && g->act == POLUS_ACT_NONE && g->C2 == nullptr;
    t.split = g->split_k < 1 ? 1 : g->split_k;
    if (g->N <= 64) t.BN = 64;
    else if (g->N <= 128) t.BN = 128;
    else if (wgrad) t.BN = 256;
    else t.BN = mt * cdiv(g->N, 256) * nb * t.split * t.CG >= sms ? 256 : 128;
    if (wgrad) {
        const long long tiles = mt * cdiv(g->N, t.BN) * nb;
        const int max_split = kb_total / 4 > 1 ? kb_total / 4 : 1;  // >= 4 k-blocks per split
        long long best_cost = -1;
        for (int sp = 1; sp <= max_split && sp <= 32; ++sp) {
            const long long waves = (tiles * sp + groups - 1) / groups;
            const long long cost = waves * (cdiv(kb_total, sp) + 8);
            if (best_cost < 0 || cost < best_cost) {
                best_cost = cost;
                t.split = sp;
            }
        }
    }
    // epilogues with per-element math run on the 16-epilogue-warp instantiation (256-wide pair tiles, A K-major:
    // the FFN-up forward GEMM and the dgrad GEMM that applies act' and sums the bias gradient)
    t.epi16 = t.CG == 2 && t.BN == 256 && g->c_dtype != POLUS_F32 && !g->A.mn_major &&
              (g->act != POLUS_ACT_NONE || g->Emul != nullptr || g->C2 != nullptr);
    return t;
}

const char* why_unsupported(const polus_gemm_t* g) {
    if (g->A.dtype != POLUS_BF16 || g->B.dtype != POLUS_BF16) return "operands must be bf16";
    if (g->M < 1 || g->N < 1 || g->K < 1) return "empty problem";
    if (!aligned16(g->A.ptr) || !aligned16(g->B.ptr) || !aligned16(g->C)) return "pointers must be 16-byte aligned";
    if (g->A.ld % 8 || g->B.ld % 8) return "operand leading dims must be multiples of 8 elements";
    if ((g->batch0 > 1 && (g->A.bs0 % 8 || g->B.bs0 % 8)) || (g->batch1 > 1 && (g->A.bs1 % 8 || g->B.bs1 % 8)))
        return "batch strides must be multiples of 8 elements";
    const int cvec = g->c_dtype == POLUS_F32 ? 4 : 8;
    if (g->ldc % cvec || g->cbs0 % cvec || g->cbs1 % cvec) return "C strides must be 16-byte multiples";
    // N % 8 != 0 (vocabulary projections): the TMA loads of a K-major B zero-fill rows >= N, the epilogue's bias loads
    // stop at N, and the C tensor map has N columns; C2, Emul, colsum and activations assume whole 8-column groups
    if (g->N % 8 && (g->B.mn_major || g->C2 || g->Emul || g->colsum || g->c2_kind != 0 || g->act != POLUS_ACT_NONE))
        return "N not a multiple of 8: only plain or bias-only problems with a K-major B";
    if (g->C2 && (g->c_dtype != POLUS_BF16 || !aligned16(g->C2))) return "C2 requires bf16 C";
    if (g->bias && !aligned16(g->bias)) return "bias must be 16-byte aligned";
    if (g->accumulate && g->c_dtype != POLUS_F32) return "accumulate requires fp32 C";
    if (g->split_k > 1 && (!g->accumulate || g->act != POLUS_ACT_NONE || g->C2)) return "split_k needs accumulate, no activation";
    if (g->c_dtype != POLUS_F32 && g->c_dtype != POLUS_BF16) return "C dtype";
    if (g->Emul && (g->c_dtype != POLUS_BF16 || g->C2 || g->act != POLUS_ACT_NONE || !aligned16(g->Emul)))
        return "Emul requires bf16 C, no C2 and no activation";
    if (g->colsum && g->c_dtype != POLUS_BF16) return "colsum requires bf16 C";
    if (g->c2_kind < 0 || g->c2_kind > 2) return "c2_kind";
    if (g->c2_kind == 2) {
        // 8-bit gelu' (C2 of a GELU forward, or the Emul tile of the dgrad that consumes it): only the 16-epilogue-warp
        // kernel implements it
        if (!(g->C2 != nullptr && g->act == POLUS_ACT_GELU) && g->Emul == nullptr) return "8-bit derivative: GELU forward with C2, or Emul";
        if (!plan_tiles(g, polus_num_sms()).epi16) return "8-bit derivative needs the 16-warp pair kernel";
        if (g->N % 32) return "8-bit derivative: N must be a multiple of 32";
        if (g->ldc % 16 || g->cbs0 % 16 || g->cbs1 % 16) return "8-bit derivative: strides must be multiples of 16";
    }
    return nullptr;
}

}  // namespace

extern "C" int polus_gemm_tc_supported(const polus_gemm_t* g) { return why_unsupported(g) == nullptr ? 1 : 0; }

extern "C" int polus_gemm_tc(const polus_gemm_t* g, void* stream) {
    const char* why = why_unsupported(g);
    POLUS_REQUIRE(why == nullptr, "polus_gemm_tc: unsupported problem (%s) M=%d N=%d K=%d", why, g->M, g->N, g->K);
    const int batch0 = g->batch0 < 1 ? 1 : g->batch0;
    const int batch1 = g->batch1 < 1 ? 1 : g->batch1;
    const TilePlan plan = plan_tiles(g, polus_num_sms());
    const int CG = plan.CG, BN = plan.BN;
    const long long mt = cdiv(g->M, BM * CG);
    const long long nb = (long long)batch0 * batch1;
    int split = plan.split;

    TcParams p;
    p.M = g->M;
    p.N = g->N;
    p.K = g->K;
    p.batch0 = batch0;
    p.m_tiles = (int)mt;
    p.n_tiles = cdiv(g->N, BN);
    p.kb_total = cdiv(g->K, BK);
    if (split > p.kb_total) split = p.kb_total;
    p.kb_per_split = cdiv(p.kb_total, split);
    p.split_k = cdiv(p.kb_total, p.kb_per_split);
    p.num_tiles = (int)(mt * p.n_tiles * p.split_k * nb);
    // Rasterisation: concurrently running tiles form (about) an 8 x 9 patch of the tile grid instead of a 74 x 1 column
    // strip, so each A row block and each B column block in flight is shared by 8-9 clusters (measured 1.05-1.15x).
    p.group_m = kGroupM < p.m_tiles ? kGroupM : p.m_tiles;
    p.C = g->C;
    p.ldc = g->ldc;
    p.cbs0 = g->cbs0;
    p.cbs1 = g->cbs1;
    p.bias = g->bias;
    p.alpha = g->alpha;
    p.act = g->act;
    p.c_f32 = g->c_dtype == POLUS_F32;
    p.accumulate = g->accumulate;
    p.has_c2 = g->C2 != nullptr;
    p.c2_grad = g->c2_kind >= 1;
    p.has_emul = g->Emul != nullptr;
    p.colsum = g->colsum;
    p.c2_u8 = g->c2_kind == 2;
    p.stg_warp = (p.c_f32 || p.has_c2 || p.has_emul) ? 2 * STG_BLOCK : STG_BLOCK;
    p.n_stages = 0;  // set per instantiation in launch()

    CUtensorMap ta, tb, tc, tc2;
    int rc = make_map(&ta, g->A, g->M, g->K, batch0, batch1, BM);
    if (rc) return rc;
    rc = make_map(&tb, g->B, g->N, g->K, batch0, batch1, BN / CG);
    if (rc) return rc;
    if (!p.c_f32) {  // bf16 outputs leave through TMA stores of 32-row x 64-column blocks
        rc = encode_map(&tc, g->C, g->N, g->M, g->ldc, batch0, g->cbs0, batch1, g->cbs1, 32);
        if (rc) return rc;
        if (p.has_c2 || p.has_emul) {
            rc = encode_map(&tc2, p.has_c2 ? g->C2 : const_cast<void*>(g->Emul), g->N, g->M, g->ldc, batch0, g->cbs0, batch1, g->cbs1, 32);
            if (rc) return rc;
        } else {
            tc2 = tc;
        }
    } else {  // fp32 outputs: 32-row x 32-column blocks, stored or reduce-added by the TMA unit
        rc = encode_map(&tc, g->C, g->N, g->M, g->ldc, batch0, g->cbs0, batch1, g->cbs1, 32, 4);
        if (rc) return rc;
        tc2 = tc;
    }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (plan.epi16) {
        // 16 warps x (2 KB C + 2 KB C2 / multiplier), 32 x 32 TMA boxes with the 64-byte swizzle
        p.stg_warp = 2 * STG_BLOCK;
        rc = encode_map(&tc, g->C, g->N, g->M, g->ldc, batch0, g->cbs0, batch1, g->cbs1, 32, 2, 64);
        if (rc) return rc;
        tc2 = tc;
        if (p.has_c2 || p.has_emul) {
            void* x2 = p.has_c2 ? g->C2 : const_cast<void*>(g->Emul);
            if (p.c2_u8) rc = encode_map(&tc2, x2, g->N, g->M, g->ldc, batch0, g->cbs0, batch1, g->cbs1, 32, 1, 32);  // [32][32 B] boxes, no swizzle
            else rc = encode_map(&tc2, x2, g->N, g->M, g->ldc, batch0, g->cbs0, batch1, g->cbs1, 32, 2, 64);
            if (rc) return rc;
        }
        if (g->B.mn_major) return launch<256, false, true, 2, 16>(ta, tb, tc, tc2, p, st);
        return launch<256, false, false, 2, 16>(ta, tb, tc, tc2, p, st);
    }
    if (CG == 2) {
        if (BN == 128) return launch_major<128, 2>(g->A.mn_major, g->B.mn_major, ta, tb, tc, tc2, p, st);
        return launch_major<256, 2>(g->A.mn_major, g->B.mn_major, ta, tb, tc, tc2, p, st);
    }
    if (BN == 64) return launch_major<64, 1>(g->A.mn_major, g->B.mn_major, ta, tb, tc, tc2, p, st);
    if (BN == 128) return launch_major<128, 1>(g->A.mn_major, g->B.mn_major, ta, tb, tc, tc2, p, st);
    return launch_major<256, 1>(g->A.mn_major, g->B.mn_major, ta, tb, tc, tc2, p, st);
}
