// LayerNorm family (HBM-bound): fused residual + dropout + LayerNorm forward/backward, and the BERT
// embedding block (gather x3 + sum + LayerNorm + dropout; backward with scatter-add).
//
// Replaces, per call, the ~7 Eigen kernels TF runs for HF TFBertSelfOutput/TFBertOutput
// (`LayerNorm(dropout(dense(x)) + residual)`, eps 1e-12) and the ~8 it runs for TFBertEmbeddings;
// reached from the reference through polus/models.py:205-213 and polus/data.py:526-545.
//
// Layout: one warp per row, each lane owns 16-byte chunks `lane + 32*i`; row statistics by warp
// shuffles; no shared memory on the forward path.  Parameter gradients use a deterministic two-stage
// reduction (per-CTA partials in a workspace, then a column-sum kernel) instead of global atomics.
#include "common.cuh"
#include "ptx.cuh"
#include <atomic>
#include <stdlib.h>
extern std::atomic<long long> g_launch_count;
int polus_launch_colsum_reduce(const float* partial, int rows, int cols, float* out0, float* out1, int split, cudaStream_t st);

namespace {

constexpr int kWarps = 8;            // warps per CTA
constexpr int kBwdBlocks = 148 * 2;  // CTAs of the backward kernels (partials per CTA)

struct DropCfg {
    unsigned long long seed;
    uint32_t site;
    uint32_t thresh16;  // 0 => dropout off
    float inv_keep;
};

inline DropCfg make_drop(float p, uint64_t seed, uint32_t site) {
    DropCfg d;
    d.seed = seed;
    d.site = site;
    d.thresh16 = p > 0.f ? (uint32_t)lrintf(p * 65536.0f) : 0u;
    d.inv_keep = p > 0.f ? 1.0f / (1.0f - p) : 1.0f;
    return d;
}

// ------------------------------------------------------------------------------ forward
// NC = 16-byte chunks per lane (H <= 256*NC); FULL: H == 256*NC exactly (no bounds checks: BERT-base 768, large 1024).
// Instruction-bound as much as HBM-bound (ablation: profiles/r01_ablation_v8_marginal_costs.txt), so the code is
// written for instruction count: all global loads of a row issued first, 128-bit accesses only, dropout applied straight
// from the Philox words (keep bits saved, one byte per chunk, so that backward does not run Philox again), deviations
// d = v - mean kept in place of v, gamma/beta staged in shared memory once per CTA.
template <int NC, bool FULL>
__global__ void __launch_bounds__(128, NC <= 3 ? 6 : (NC == 4 ? 4 : 1))
ln_res_fwd_kernel(bf16* __restrict__ x, const bf16* __restrict__ res, const float* __restrict__ gamma,
                  const float* __restrict__ beta, int M, int H, float eps, DropCfg dc,
                  const uint32_t* __restrict__ d_step, bf16* __restrict__ y, float* __restrict__ mean_out,
                  float* __restrict__ rstd_out, uint8_t* __restrict__ keepbits) {
    extern __shared__ float sgb[];  // gamma [H] | beta [H]
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int chunks = H >> 3;
    pdl_trigger();
    // parameters are last written by the optimizer of the PREVIOUS step: safe to stage before the dependency wait
    for (int i = threadIdx.x; i < (H >> 2); i += blockDim.x) {
        reinterpret_cast<float4*>(sgb)[i] = __ldg(reinterpret_cast<const float4*>(gamma) + i);
        reinterpret_cast<float4*>(sgb + H)[i] = __ldg(reinterpret_cast<const float4*>(beta) + i);
    }
    pdl_wait();
    __syncthreads();
    const uint32_t step = dc.thresh16 ? *d_step : 0u;
    const float inv_h = 1.0f / (float)H;
    for (int row = blockIdx.x * 4 + warp; row < M; row += gridDim.x * 4) {
        const long long base = (long long)row * H;
        bf16x8 xr[NC], rr[NC];
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            if (FULL || c < chunks) {
                xr[i] = ld_stream8(x + base + c * 8);
                if (res != nullptr) rr[i] = ld_global16(res + base + c * 8);
            }
        }
        float v[NC][8];
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            if (FULL || c < chunks) {
                unpack8(xr[i], v[i]);
                if (dc.thresh16) {
                    const uint32_t bits = dropout_apply8(dc.seed, dc.site, step, (unsigned long long)row * chunks + c, dc.thresh16, dc.inv_keep, v[i]);
                    if (keepbits != nullptr) keepbits[(long long)row * chunks + c] = (uint8_t)bits;
                }
                if (res != nullptr) {
                    float rv[8];
                    unpack8(rr[i], rv);
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[i][j] += rv[j];
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) sum += v[i][j];
                st_global16(x + base + c * 8, pack8(v[i]));  // z, kept for backward
            }
        }
        const float mean = warp_sum(sum) * inv_h;
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            if (FULL || lane + 32 * i < chunks) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    v[i][j] -= mean;
                    sq = fmaf(v[i][j], v[i][j], sq);
                }
            }
        }
        const float rstd = rsqrtf(warp_sum(sq) * inv_h + eps);
        if (lane == 0) {
            mean_out[row] = mean;
            rstd_out[row] = rstd;
        }
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            if (FULL || c < chunks) {
                float o[8];
                const float4 g0 = reinterpret_cast<const float4*>(sgb + c * 8)[0], g1 = reinterpret_cast<const float4*>(sgb + c * 8)[1];
                const float4 b0 = reinterpret_cast<const float4*>(sgb + H + c * 8)[0], b1 = reinterpret_cast<const float4*>(sgb + H + c * 8)[1];
                const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] = fmaf(v[i][j] * rstd, g[j], b[j]);
                st_global16(y + base + c * 8, pack8(o));
            }
        }
    }
}

// ------------------------------------------------------------------------------ backward
// dz = rstd * (g - mean(g) - xhat * mean(g*xhat)), g = dy*gamma.  Writes dres = dz and dx = dropout'(dz).
// dy and z stay PACKED (bf16) in registers between the two passes (xhat and g are recomputed), which keeps the
// kernel at <= 128 registers => two 8-warp CTAs per SM.  Per-warp register partials of dgamma = sum dy*xhat,
// dbeta = sum dy and (optionally) dbias = sum dx -- the bias gradient of the Dense layer that produced x -- are
// reduced per CTA in shared memory and added to the gradient arena with one fp32 atomic per column per CTA.
// keepbits: the forward kernel's dropout decisions (one byte per chunk); NULL => regenerated with Philox.
template <int NC>
__global__ void __launch_bounds__(kWarps * 32, NC <= 4 ? 2 : 1)
ln_res_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ dy2, const bf16* __restrict__ z, const float* __restrict__ mean_in,
                  const float* __restrict__ rstd_in, const float* __restrict__ gamma, int M, int H, DropCfg dc,
                  const uint32_t* __restrict__ d_step, bf16* __restrict__ dx, bf16* __restrict__ dres,
                  float* __restrict__ ggamma, float* __restrict__ gbeta, float* __restrict__ gbias,
                  const uint8_t* __restrict__ keepbits) {
    extern __shared__ float red[];  // [kWarps][H] reduction scratch | gamma [H]
    float* sg = red + kWarps * H;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int chunks = H >> 3;
    pdl_trigger();
    for (int i = threadIdx.x; i < (H >> 2); i += blockDim.x)
        reinterpret_cast<float4*>(sg)[i] = __ldg(reinterpret_cast<const float4*>(gamma) + i);
    float dg[NC][8], db[NC][8], dxs[NC][8];
#pragma unroll
    for (int i = 0; i < NC; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) dg[i][j] = db[i][j] = dxs[i][j] = 0.f;
    pdl_wait();
    __syncthreads();
    const uint32_t step = dc.thresh16 ? *d_step : 0u;
    const float inv_h = 1.0f / (float)H;
    for (int row = blockIdx.x * kWarps + warp; row < M; row += gridDim.x * kWarps) {
        const long long base = (long long)row * H;
        bf16x8 dyr[NC], zr[NC];
        uint32_t kb[NC];
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
                dyr[i] = ld_stream8(dy + base + c * 8);
                zr[i] = ld_stream8(z + base + c * 8);
                if (dc.thresh16 && keepbits != nullptr) kb[i] = keepbits[(long long)row * chunks + c];
            }
        }
        if (dy2 != nullptr) {  // second contribution to d(y) (residual stream): summed here, no add kernel
#pragma unroll
            for (int i = 0; i < NC; ++i) {
                const int c = lane + 32 * i;
                if (c < chunks) {
                    float a[8], b2[8];
                    unpack8(dyr[i], a);
                    unpack8(ld_stream8(dy2 + base + c * 8), b2);
#pragma unroll
                    for (int j = 0; j < 8; ++j) a[j] += b2[j];
                    dyr[i] = pack8(a);  // bf16 sum, as the separate add kernel produced
                }
            }
        }
        const float rstd = rstd_in[row];
        const float nmr = -mean_in[row] * rstd;
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
                float dyv[8], zv[8];
                unpack8(dyr[i], dyv);
                unpack8(zr[i], zv);
                const float4 g0 = reinterpret_cast<const float4*>(sg + c * 8)[0], g1 = reinterpret_cast<const float4*>(sg + c * 8)[1];
                const float gam[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float xh = fmaf(zv[j], rstd, nmr);
                    const float g = dyv[j] * gam[j];
                    s1 += g;
                    s2 = fmaf(g, xh, s2);
                    dg[i][j] = fmaf(dyv[j], xh, dg[i][j]);
                    db[i][j] += dyv[j];
                }
            }
        }
        const float c1 = warp_sum(s1) * inv_h * rstd;
        const float c2 = warp_sum(s2) * inv_h * rstd;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
                float dyv[8], zv[8], dz[8];
                unpack8(dyr[i], dyv);
                unpack8(zr[i], zv);
                const float4 g0 = reinterpret_cast<const float4*>(sg + c * 8)[0], g1 = reinterpret_cast<const float4*>(sg + c * 8)[1];
                const float gam[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float xh = fmaf(zv[j], rstd, nmr);
                    dz[j] = fmaf(-xh, c2, fmaf(dyv[j] * gam[j], rstd, -c1));  // rstd * (g - mean(g) - xhat * mean(g xhat))
                }
                if (dres != nullptr && dres != dx) st_global16(dres + base + c * 8, pack8(dz));
                if (dc.thresh16) {
                    if (keepbits != nullptr) dropout_apply8_bits(kb[i], dc.inv_keep, dz);
                    else dropout_apply8(dc.seed, dc.site, step, (unsigned long long)row * chunks + c, dc.thresh16, dc.inv_keep, dz);
                }
                st_global16(dx + base + c * 8, pack8(dz));
                if (gbias != nullptr) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) dxs[i][j] += dz[j];
                }
            }
        }
    }
    // CTA reduction of the parameter-gradient partials, one quantity at a time (red is [kWarps][H])
#pragma unroll
    for (int which = 0; which < 3; ++which) {
        float* out = which == 0 ? ggamma : (which == 1 ? gbeta : gbias);
        if (out == nullptr) continue;  // uniform
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
                float* r8 = red + warp * H + c * 8;
                const float* src = which == 0 ? dg[i] : (which == 1 ? db[i] : dxs[i]);
                reinterpret_cast<float4*>(r8)[0] = make_float4(src[0], src[1], src[2], src[3]);
                reinterpret_cast<float4*>(r8)[1] = make_float4(src[4], src[5], src[6], src[7]);
            }
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < H; idx += blockDim.x) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += red[w * H + idx];
            atomicAdd(out + idx, s);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------ backward, rows prefetched by bulk copies
// Same arithmetic as ln_res_bwd_kernel for H = 256 * NC.  ncu on that kernel: IPC 0.30 per scheduler, "long scoreboard"
// the dominant stall, 16 resident warps (128 registers each hold the three column accumulators) -- every warp loads a
// row, waits out the DRAM latency, computes, and only then asks for its next row.  Here each warp owns two shared-memory
// row slots (dy | dy2 | z, 3 x 2H bytes); lane 0 posts the bulk copies of row k+1 before the warp starts on row k, so a
// CTA keeps 2 x 8 rows in flight without a single extra register and the loads overlap the arithmetic.
// NC = 4 (H = 1024, the BERT-large-sized configuration): 137 KB of shared memory per CTA, one CTA per SM, and therefore the
// whole register file for its 256 threads -- the register-resident kernel needs ~250 registers per thread for four
// column chunks and spilled 520 bytes per thread under its two-CTA bound (csrc/build/layernorm.ptxas.log, round 1).
template <int NC>
__global__ void __launch_bounds__(kWarps * 32, NC <= 3 ? 2 : 1)
ln_res_bwd_pf_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ dy2, const bf16* __restrict__ z, const float* __restrict__ mean_in,
                     const float* __restrict__ rstd_in, const float* __restrict__ gamma, int M, DropCfg dc,
                     const uint32_t* __restrict__ d_step, bf16* __restrict__ dx, bf16* __restrict__ dres,
                     float* __restrict__ ggamma, float* __restrict__ gbeta, float* __restrict__ gbias,
                     const uint8_t* __restrict__ keepbits) {
    constexpr int H = NC * 256;
    constexpr int ROWB = H * 2;  // bytes of one bf16 row
    extern __shared__ __align__(128) uint8_t ln_smem[];
    float* red = reinterpret_cast<float*>(ln_smem);            // [kWarps][H] reduction scratch
    float* sg = red + kWarps * H;                               // gamma [H]
    constexpr int SLOT = 3 * ROWB + 128;                        // dy | dy2 | z rows + the row's dropout keep bytes (H / 8 <= 128)
    uint8_t* rows = reinterpret_cast<uint8_t*>(sg + H);         // [kWarps][2 slots][SLOT]
    uint64_t* bars = reinterpret_cast<uint64_t*>(rows + kWarps * 2 * SLOT);  // [kWarps][2]
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    constexpr int chunks = H >> 3;
    pdl_trigger();
    for (int i = threadIdx.x; i < (H >> 2); i += blockDim.x)
        reinterpret_cast<float4*>(sg)[i] = __ldg(reinterpret_cast<const float4*>(gamma) + i);
    if (lane == 0) {
        ptx::mbar_init(&bars[warp * 2], 1);
        ptx::mbar_init(&bars[warp * 2 + 1], 1);
        ptx::fence_barrier_init();
    }
    float dg[NC][8], db[NC][8], dxs[NC][8];
#pragma unroll
    for (int i = 0; i < NC; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) dg[i][j] = db[i][j] = dxs[i][j] = 0.f;
    pdl_wait();
    __syncthreads();
    const uint32_t step = dc.thresh16 ? *d_step : 0u;
    constexpr float inv_h = 1.0f / (float)H;
    const int row_step = gridDim.x * kWarps;
    // The keep bytes of the row ride on the same bulk copy as the row itself (H / 8 bytes, a 16-byte multiple for the three
    // widths this kernel is built for).  They used to be prefetched into registers with LDG.U8: with 72 accumulator
    // registers per thread ptxas spilled them, and the spill STORE right behind the load waited for the load -- 12 % of
    // the kernel's stall samples sat on that one instruction (profiles/r02_ncu_ln_bwd.txt).
    const bool kb_smem = dc.thresh16 && keepbits != nullptr;
    const uint32_t tx = (dy2 != nullptr ? 3u : 2u) * ROWB + (kb_smem ? (uint32_t)chunks : 0u);
    uint8_t* my = rows + warp * (2 * SLOT);
    auto post = [&](int row, int slot) {  // lane 0 only
        uint8_t* dst = my + slot * SLOT;
        uint64_t* bar = &bars[warp * 2 + slot];
        ptx::mbar_expect_tx(bar, tx);
        ptx::bulk_load(dst, dy + (long long)row * H, ROWB, bar);
        ptx::bulk_load(dst + 2 * ROWB, z + (long long)row * H, ROWB, bar);
        if (dy2 != nullptr) ptx::bulk_load(dst + ROWB, dy2 + (long long)row * H, ROWB, bar);
        if (kb_smem) ptx::bulk_load(dst + 3 * ROWB, keepbits + (long long)row * chunks, chunks, bar);
    };
    int row = blockIdx.x * kWarps + warp;
    if (row < M && lane == 0) post(row, 0);
    float rstd_n = 0.f, mean_n = 0.f;
    if (row < M) {
        rstd_n = rstd_in[row];
        mean_n = mean_in[row];
    }
    for (int k = 0; row < M; row += row_step, ++k) {
        const int slot = k & 1;
        const int next = row + row_step;
        const float rstd = rstd_n;
        const float nmr = -mean_n * rstd;
        ptx::fence_proxy_async_smem();  // the dy + dy2 sums written into the other slot (row k-1) vs the bulk copy about to overwrite it
        __syncwarp();                   // every lane is done with that slot
        if (next < M) {
            if (lane == 0) post(next, slot ^ 1);
            rstd_n = rstd_in[next];
            mean_n = mean_in[next];
        }
        ptx::mbar_wait(&bars[warp * 2 + slot], (uint32_t)(k >> 1) & 1u);
        uint8_t* src = my + slot * SLOT;
        const long long base = (long long)row * H;
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            float dyv[8], zv[8];
            unpack8(*reinterpret_cast<const bf16x8*>(src + c * 16), dyv);
            unpack8(*reinterpret_cast<const bf16x8*>(src + 2 * ROWB + c * 16), zv);
            if (dy2 != nullptr) {  // second contribution to d(y) (residual stream): bf16 sum, as the separate add kernel
                float b2[8];       // produced, written back to the slot so that the second pass reads the same values
                unpack8(*reinterpret_cast<const bf16x8*>(src + ROWB + c * 16), b2);
#pragma unroll
                for (int j = 0; j < 8; ++j) dyv[j] += b2[j];
                const bf16x8 sum = pack8(dyv);
                *reinterpret_cast<bf16x8*>(src + c * 16) = sum;
                unpack8(sum, dyv);
            }
            const float4 g0 = reinterpret_cast<const float4*>(sg + c * 8)[0], g1 = reinterpret_cast<const float4*>(sg + c * 8)[1];
            const float gam[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float xh = fmaf(zv[j], rstd, nmr);
                const float g = dyv[j] * gam[j];
                s1 += g;
                s2 = fmaf(g, xh, s2);
                dg[i][j] = fmaf(dyv[j], xh, dg[i][j]);
                db[i][j] += dyv[j];
            }
        }
        const float c1 = warp_sum(s1) * inv_h * rstd;
        const float c2 = warp_sum(s2) * inv_h * rstd;
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            float dyv[8], zv[8], dz[8];
            unpack8(*reinterpret_cast<const bf16x8*>(src + c * 16), dyv);  // each lane re-reads the chunks it wrote
            unpack8(*reinterpret_cast<const bf16x8*>(src + 2 * ROWB + c * 16), zv);
            const float4 g0 = reinterpret_cast<const float4*>(sg + c * 8)[0], g1 = reinterpret_cast<const float4*>(sg + c * 8)[1];
            const float gam[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float xh = fmaf(zv[j], rstd, nmr);
                dz[j] = fmaf(-xh, c2, fmaf(dyv[j] * gam[j], rstd, -c1));
            }
            if (dres != nullptr && dres != dx) st_global16(dres + base + c * 8, pack8(dz));
            if (dc.thresh16) {
                if (keepbits != nullptr) dropout_apply8_bits(src[3 * ROWB + c], dc.inv_keep, dz);
                else dropout_apply8(dc.seed, dc.site, step, (unsigned long long)row * chunks + c, dc.thresh16, dc.inv_keep, dz);
            }
            st_global16(dx + base + c * 8, pack8(dz));
            if (gbias != nullptr) {
#pragma unroll
                for (int j = 0; j < 8; ++j) dxs[i][j] += dz[j];
            }
        }
    }
    // CTA reduction of the parameter-gradient partials, one quantity at a time (red is [kWarps][H])
#pragma unroll
    for (int which = 0; which < 3; ++which) {
        float* out = which == 0 ? ggamma : (which == 1 ? gbeta : gbias);
        if (out == nullptr) continue;  // uniform
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = lane + 32 * i;
            float* r8 = red + warp * H + c * 8;
            const float* srcp = which == 0 ? dg[i] : (which == 1 ? db[i] : dxs[i]);
            reinterpret_cast<float4*>(r8)[0] = make_float4(srcp[0], srcp[1], srcp[2], srcp[3]);
            reinterpret_cast<float4*>(r8)[1] = make_float4(srcp[4], srcp[5], srcp[6], srcp[7]);
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < H; idx += blockDim.x) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += red[w * H + idx];
            atomicAdd(out + idx, s);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------ embeddings
// RoBERTa position ids (HF create_position_ids_from_input_ids): padding_idx + (number of non-pad tokens up to and
// including s) for a real token, padding_idx for a pad token.  One warp per row; the prefix count runs over 32-token
// slices with a ballot, so any S works and nothing leaves the device.
__global__ void __launch_bounds__(kWarps * 32)
position_ids_kernel(const int32_t* __restrict__ ids, int B, int S, int padding_idx, int32_t* __restrict__ pos) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (row >= B) return;
    const int32_t* r = ids + (long long)row * S;
    int32_t* o = pos + (long long)row * S;
    int count = padding_idx;
    for (int s0 = 0; s0 < S; s0 += 32) {
        const int s = s0 + lane;
        const bool real = s < S && r[s] != padding_idx;
        const uint32_t m = __ballot_sync(0xffffffffu, real);
        if (s < S) o[s] = real ? count + __popc(m & ((2u << lane) - 1u)) : padding_idx;
        count += __popc(m);
    }
}

// POS: the position row of token `row` is pos_ids[row] (clamped to the n_pos rows of the table) instead of row % S.
template <int MAXC, bool POS>
__global__ void __launch_bounds__(kWarps * 32)
embed_ln_fwd_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ tt, const float* __restrict__ word,
                    const float* __restrict__ pos, const float* __restrict__ type, const float* __restrict__ gamma,
                    const float* __restrict__ beta, int M, int S, int H, int vocab, int n_types, float eps, DropCfg dc,
                    const uint32_t* __restrict__ d_step, bf16* __restrict__ y, float* __restrict__ zout,
                    float* __restrict__ mean_out, float* __restrict__ rstd_out, const int32_t* __restrict__ pos_ids,
                    int n_pos) {
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int chunks = H >> 3;
    const uint32_t step = dc.thresh16 ? *d_step : 0u;
    for (int row = blockIdx.x * kWarps + warp; row < M; row += gridDim.x * kWarps) {
        int id = ids[row];
        id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
        int t = tt ? tt[row] : 0;
        t = t < 0 ? 0 : (t >= n_types ? n_types - 1 : t);
        int s;
        if constexpr (POS) {
            s = pos_ids[row];
            s = s < 0 ? 0 : (s >= n_pos ? n_pos - 1 : s);
        } else {
            s = row % S;
        }
        const float* wrow = word + (long long)id * H;
        const float* prow = pos + (long long)s * H;
        const float* trow = type + (long long)t * H;
        float v[MAXC][8];
        float sum = 0.f;
        const long long base = (long long)row * H;
#pragma unroll
        for (int i = 0; i < MAXC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const float4 a = __ldg(reinterpret_cast<const float4*>(wrow + c * 8) + h);
                    const float4 b = __ldg(reinterpret_cast<const float4*>(prow + c * 8) + h);
                    const float4 d = __ldg(reinterpret_cast<const float4*>(trow + c * 8) + h);
                    // TF adds word + type first?  HF: inputs_embeds + position_embeds + token_type_embeds
                    const float4 r = make_float4((a.x + b.x) + d.x, (a.y + b.y) + d.y, (a.z + b.z) + d.z, (a.w + b.w) + d.w);
                    v[i][4 * h + 0] = r.x;
                    v[i][4 * h + 1] = r.y;
                    v[i][4 * h + 2] = r.z;
                    v[i][4 * h + 3] = r.w;
                    reinterpret_cast<float4*>(zout + base + c * 8)[h] = r;
                    sum += (r.x + r.y) + (r.z + r.w);
                }
            }
        }
        const float mean = warp_sum(sum) / (float)H;
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < MAXC; ++i)
            if (lane + 32 * i < chunks) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float d = v[i][j] - mean;
                    sq += d * d;
                }
            }
        const float rstd = rsqrtf(warp_sum(sq) / (float)H + eps);
        if (lane == 0) {
            mean_out[row] = mean;
            rstd_out[row] = rstd;
        }
#pragma unroll
        for (int i = 0; i < MAXC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
                float o[8];
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    o[j] = (v[i][j] - mean) * rstd * __ldg(gamma + c * 8 + j) + __ldg(beta + c * 8 + j);
                if (dc.thresh16) {
                    const uint32_t keep = dropout_keep8(dc.seed, dc.site, step, (unsigned long long)row * chunks + c, dc.thresh16);
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = ((keep >> j) & 1u) ? o[j] * dc.inv_keep : 0.f;
                }
                *reinterpret_cast<bf16x8*>(y + base + c * 8) = pack8(o);
            }
        }
    }
}

// stage A of the embedding backward: dropout' + LayerNorm backward -> dz (fp32) + dgamma/dbeta partials
template <int MAXC>
__global__ void __launch_bounds__(kWarps * 32)
embed_ln_bwd_kernel(const bf16* __restrict__ dy, const float* __restrict__ z, const float* __restrict__ mean_in,
                    const float* __restrict__ rstd_in, const float* __restrict__ gamma, int M, int H, DropCfg dc,
                    const uint32_t* __restrict__ d_step, float* __restrict__ dz_out, float* __restrict__ ggamma,
                    float* __restrict__ gbeta) {
    extern __shared__ float red[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int chunks = H >> 3;
    const uint32_t step = dc.thresh16 ? *d_step : 0u;
    float dg[MAXC][8], db[MAXC][8];
#pragma unroll
    for (int i = 0; i < MAXC; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) dg[i][j] = db[i][j] = 0.f;
    for (int row = blockIdx.x * kWarps + warp; row < M; row += gridDim.x * kWarps) {
        const long long base = (long long)row * H;
        const float mean = mean_in[row], rstd = rstd_in[row];
        float g[MAXC][8], xh[MAXC][8];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < MAXC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
                float dyv[8];
                unpack8(ld_stream8(dy + base + c * 8), dyv);
                if (dc.thresh16) {
                    const uint32_t keep = dropout_keep8(dc.seed, dc.site, step, (unsigned long long)row * chunks + c, dc.thresh16);
#pragma unroll
                    for (int j = 0; j < 8; ++j) dyv[j] = ((keep >> j) & 1u) ? dyv[j] * dc.inv_keep : 0.f;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    xh[i][j] = (z[base + c * 8 + j] - mean) * rstd;
                    g[i][j] = dyv[j] * __ldg(gamma + c * 8 + j);
                    s1 += g[i][j];
                    s2 += g[i][j] * xh[i][j];
                    dg[i][j] += dyv[j] * xh[i][j];
                    db[i][j] += dyv[j];
                }
            }
        }
        s1 = warp_sum(s1) / (float)H;
        s2 = warp_sum(s2) / (float)H;
#pragma unroll
        for (int i = 0; i < MAXC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
#pragma unroll
                for (int j = 0; j < 8; ++j) dz_out[base + c * 8 + j] = rstd * (g[i][j] - s1 - xh[i][j] * s2);
            }
        }
    }
#pragma unroll
    for (int which = 0; which < 2; ++which) {
        float* out = which == 0 ? ggamma : gbeta;
        if (out == nullptr) continue;
#pragma unroll
        for (int i = 0; i < MAXC; ++i) {
            const int c = lane + 32 * i;
            if (c < chunks) {
#pragma unroll
                for (int j = 0; j < 8; ++j) red[warp * H + c * 8 + j] = which == 0 ? dg[i][j] : db[i][j];
            }
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < H; idx += blockDim.x) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += red[w * H + idx];
            atomicAdd(out + idx, s);
        }
        __syncthreads();
    }
}

// stage B: one CTA per position s.  gpos[s] is owned exclusively (no atomics); token-type sums are
// reduced in registers (2 types) and word rows are scatter-added with fp32 atomics (what TF's
// IndexedSlices -> unsorted_segment_sum does for the reference).
// POS: column s of the batch reaches any position row, keyed by pos_ids (TF semantics: pad tokens add to the
// padding_idx row like any other).  Two runs of equal position id stay open in registers, the most recently used
// first; a run is flushed with one atomic per column when a third id evicts it and at the end.  At one s a right- or
// left-padded batch holds the padding row and, right-padded, one real position: every pad token of the column lands
// in one register sum instead of one atomic each.
__device__ __forceinline__ void atomic_add4(float* p, float4 v) {
    atomicAdd(p + 0, v.x); atomicAdd(p + 1, v.y); atomicAdd(p + 2, v.z); atomicAdd(p + 3, v.w);
}

template <bool POS>
__global__ void embed_scatter_kernel(const float* __restrict__ dz, const int32_t* __restrict__ ids,
                                     const int32_t* __restrict__ tt, int B, int S, int H, int vocab, int n_types,
                                     float* __restrict__ gword, float* __restrict__ gpos, float* __restrict__ gtype,
                                     const int32_t* __restrict__ pos_ids, int n_pos) {
    const int s = blockIdx.x;
    for (int col = threadIdx.x * 4; col < H; col += blockDim.x * 4) {
        float4 accp = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 acct0 = accp, acct1 = accp;
        float4 acc1 = accp;  // POS: accp is the run of key k0 (most recent), acc1 the run of key k1
        int k0 = -1, k1 = -1;
        for (int b = 0; b < B; ++b) {
            const long long row = (long long)b * S + s;
            const float4 v = *reinterpret_cast<const float4*>(dz + row * H + col);
            if constexpr (POS) {
                int p = pos_ids[row];
                p = p < 0 ? 0 : (p >= n_pos ? n_pos - 1 : p);
                if (p != k0) {
                    if (p != k1) {
                        if (k1 >= 0 && gpos != nullptr) atomic_add4(gpos + (long long)k1 * H + col, acc1);
                        k1 = p;
                        acc1 = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    const float4 ta = accp;
                    accp = acc1;
                    acc1 = ta;
                    k1 = k0;
                    k0 = p;
                }
            }
            accp.x += v.x; accp.y += v.y; accp.z += v.z; accp.w += v.w;
            if (gword != nullptr) {
                int id = ids[row];
                id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
                float* w = gword + (long long)id * H + col;
                atomicAdd(w + 0, v.x); atomicAdd(w + 1, v.y); atomicAdd(w + 2, v.z); atomicAdd(w + 3, v.w);
            }
            int t = tt ? tt[row] : 0;
            t = t < 0 ? 0 : (t >= n_types ? n_types - 1 : t);
            if (t == 0) { acct0.x += v.x; acct0.y += v.y; acct0.z += v.z; acct0.w += v.w; }
            else if (t == 1) { acct1.x += v.x; acct1.y += v.y; acct1.z += v.z; acct1.w += v.w; }
            else if (gtype != nullptr) {
                float* g = gtype + (long long)t * H + col;
                atomicAdd(g + 0, v.x); atomicAdd(g + 1, v.y); atomicAdd(g + 2, v.z); atomicAdd(g + 3, v.w);
            }
        }
        if constexpr (POS) {
            if (gpos != nullptr) {
                if (k0 >= 0) atomic_add4(gpos + (long long)k0 * H + col, accp);
                if (k1 >= 0) atomic_add4(gpos + (long long)k1 * H + col, acc1);
            }
        } else if (gpos != nullptr) {
            float4* gp = reinterpret_cast<float4*>(gpos + (long long)s * H + col);
            float4 o = *gp;
            o.x += accp.x; o.y += accp.y; o.z += accp.z; o.w += accp.w;
            *gp = o;
        }
        if (gtype != nullptr) {
            float* g0 = gtype + col;
            atomicAdd(g0 + 0, acct0.x); atomicAdd(g0 + 1, acct0.y); atomicAdd(g0 + 2, acct0.z); atomicAdd(g0 + 3, acct0.w);
            if (n_types > 1) {
                float* g1 = gtype + H + col;
                atomicAdd(g1 + 0, acct1.x); atomicAdd(g1 + 1, acct1.y); atomicAdd(g1 + 2, acct1.z); atomicAdd(g1 + 3, acct1.w);
            }
        }
    }
}

int grid_for_rows(int M) {
    int want = cdiv(M, kWarps);
    int cap = polus_num_sms() * 8;
    return want < cap ? want : cap;
}

}  // namespace

#define DISPATCH_MAXC(H, CALL4, CALL16)        \
    if ((H) <= 1024) { CALL4; } else { CALL16; }

extern "C" size_t polus_ln_ws_floats(int H) { return (size_t)kBwdBlocks * 2 * (size_t)H; }

extern "C" int polus_ln_res_fwd(polus_bf16_t* x, const polus_bf16_t* res, const float* gamma, const float* beta, int M,
                                int H, float eps, float p_drop, uint64_t seed, uint32_t site, const uint32_t* d_step,
                                polus_bf16_t* y, float* mean, float* rstd, uint8_t* keepbits, void* stream) {
    POLUS_REQUIRE(M >= 0 && H > 0 && H % 8 == 0 && H <= 4096, "polus_ln_res_fwd: H must be a multiple of 8 and <= 4096 (got %d)", H);
    POLUS_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "polus_ln_res_fwd: bad dropout %f", p_drop);
    POLUS_REQUIRE(p_drop == 0.f || d_step != nullptr, "polus_ln_res_fwd: dropout needs d_step");
    if (M == 0) return 0;
    DropCfg dc = make_drop(p_drop, seed, site);
    cudaStream_t st = (cudaStream_t)stream;
    int grid = cdiv(M, 4);
    const int cap = polus_num_sms() * 16;
    if (grid > cap) grid = cap;
    const int nc = cdiv(H, 256);
    const size_t smem_f = (size_t)2 * H * sizeof(float);
#define LN_FWD(NC_, FULL_) POLUS_CHECK_CUDA(polus_launch_pdl(ln_res_fwd_kernel<NC_, FULL_>, dim3(grid), dim3(128), smem_f, st, (bf16*)x, (const bf16*)res, gamma, beta, M, H, eps, dc, d_step, (bf16*)y, mean, rstd, keepbits))
    if (H == 768) LN_FWD(3, true); else if (H == 1024) LN_FWD(4, true); else if (H == 256) LN_FWD(1, true); else if (H == 512) LN_FWD(2, true);
    else if (nc <= 1) LN_FWD(1, false); else if (nc == 2) LN_FWD(2, false); else if (nc == 3) LN_FWD(3, false); else if (nc == 4) LN_FWD(4, false); else LN_FWD(16, false);
#undef LN_FWD
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

extern "C" int polus_ln_res_bwd(const polus_bf16_t* dy, const polus_bf16_t* dy2, const polus_bf16_t* z, const float* mean,
                                const float* rstd, const float* gamma, int M, int H, float p_drop, uint64_t seed,
                                uint32_t site, const uint32_t* d_step, polus_bf16_t* dx, polus_bf16_t* dres,
                                float* ggamma, float* gbeta, float* gbias_x, const uint8_t* keepbits, void* stream) {
    POLUS_REQUIRE(M >= 0 && H > 0 && H % 8 == 0 && H <= 4096, "polus_ln_res_bwd: H must be a multiple of 8 and <= 4096 (got %d)", H);
    POLUS_REQUIRE(dx != nullptr, "polus_ln_res_bwd: dx required");
    POLUS_REQUIRE(!(p_drop > 0.f && dres == dx), "polus_ln_res_bwd: dres may alias dx only without dropout");
    if (M == 0) return 0;
    DropCfg dc = make_drop(p_drop, seed, site);
    cudaStream_t st = (cudaStream_t)stream;
    int grid = grid_for_rows(M);
    if (grid > kBwdBlocks) grid = kBwdBlocks;
    const size_t smem = (size_t)(kWarps + 1) * H * sizeof(float);
    const int nc = cdiv(H, 256);
#define LN_BWD(NC_)                                                                                                            \
    {                                                                                                                          \
        if (smem > 48 * 1024) POLUS_CHECK_CUDA(cudaFuncSetAttribute(ln_res_bwd_kernel<NC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        POLUS_CHECK_CUDA(polus_launch_pdl(ln_res_bwd_kernel<NC_>, dim3(grid), dim3(kWarps * 32), smem, st, (const bf16*)dy, (const bf16*)dy2, (const bf16*)z, mean, rstd, gamma, M, H, dc, \
                                          d_step, (bf16*)dx, (bf16*)dres, ggamma, gbeta, gbias_x, keepbits));                  \
    }
    // rows prefetched through shared memory (H = 768: 101 KB per CTA, two CTAs per SM)
    const bool aligned = ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dy2) | reinterpret_cast<uintptr_t>(z) |
                           reinterpret_cast<uintptr_t>(keepbits)) & 15) == 0;
    if (aligned && (H == 1024 || H == 768 || H == 512 || H == 256)) {
        const size_t smem_pf = (size_t)(kWarps + 1) * H * sizeof(float) + (size_t)kWarps * 2 * (3 * H * 2 + 128) + kWarps * 2 * sizeof(uint64_t);
#define LN_BWD_PF(NC_)                                                                                                          \
    {                                                                                                                          \
        static bool set = false;                                                                                               \
        if (!set) { POLUS_CHECK_CUDA(cudaFuncSetAttribute(ln_res_bwd_pf_kernel<NC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pf)); set = true; } \
        POLUS_CHECK_CUDA(polus_launch_pdl(ln_res_bwd_pf_kernel<NC_>, dim3(grid), dim3(kWarps * 32), smem_pf, st, (const bf16*)dy, (const bf16*)dy2, (const bf16*)z, mean, rstd, gamma, M, dc, \
                                          d_step, (bf16*)dx, (bf16*)dres, ggamma, gbeta, gbias_x, keepbits));                  \
    }
        if (H == 1024) LN_BWD_PF(4) else if (H == 768) LN_BWD_PF(3) else if (H == 512) LN_BWD_PF(2) else LN_BWD_PF(1)
#undef LN_BWD_PF
        g_launch_count++;
        POLUS_LAUNCH_CHECK();
        return 0;
    }
    if (nc <= 1) LN_BWD(1) else if (nc == 2) LN_BWD(2) else if (nc == 3) LN_BWD(3) else if (nc == 4) LN_BWD(4) else LN_BWD(16)
#undef LN_BWD
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

extern "C" size_t polus_embed_ws_floats(int B, int S, int H) {
    return (size_t)B * S * H + (size_t)kBwdBlocks * 2 * (size_t)H;
}

namespace {

int embed_fwd(const char* fn, const int32_t* ids, const int32_t* tt, const float* word, const float* pos, const float* type,
              const float* gamma, const float* beta, int B, int S, int H, int vocab, int n_types, float eps, float p_drop,
              uint64_t seed, uint32_t site, const uint32_t* d_step, polus_bf16_t* y, float* z, float* mean, float* rstd,
              const int32_t* pos_ids, int n_pos, void* stream) {
    POLUS_REQUIRE(H > 0 && H % 8 == 0 && H <= 4096, "%s: H must be a multiple of 8 and <= 4096 (got %d)", fn, H);
    POLUS_REQUIRE(p_drop == 0.f || d_step != nullptr, "%s: dropout needs d_step", fn);
    const int M = B * S;
    if (M == 0) return 0;
    DropCfg dc = make_drop(p_drop, seed, site);
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = grid_for_rows(M);
#define EMB_FWD(MAXC_, POS_) (embed_ln_fwd_kernel<MAXC_, POS_><<<grid, kWarps * 32, 0, st>>>(ids, tt, word, pos, type, gamma, beta, M, S, H, vocab, n_types, eps, dc, d_step, (bf16*)y, z, mean, rstd, pos_ids, n_pos))
    if (pos_ids != nullptr) {
        DISPATCH_MAXC(H, EMB_FWD(4, true), EMB_FWD(16, true));
    } else {
        DISPATCH_MAXC(H, EMB_FWD(4, false), EMB_FWD(16, false));
    }
#undef EMB_FWD
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

int embed_bwd(const char* fn, const polus_bf16_t* dy, const float* z, const float* mean, const float* rstd, const float* gamma,
              const int32_t* ids, const int32_t* tt, int B, int S, int H, int vocab, int n_types, float p_drop, uint64_t seed,
              uint32_t site, const uint32_t* d_step, float* gword, float* gpos, float* gtype, float* ggamma, float* gbeta,
              float* ws, const int32_t* pos_ids, int n_pos, void* stream) {
    POLUS_REQUIRE(H > 0 && H % 8 == 0 && H <= 4096, "%s: H must be a multiple of 8 and <= 4096 (got %d)", fn, H);
    POLUS_REQUIRE(ws != nullptr, "%s: workspace required (polus_embed_ws_floats)", fn);
    const int M = B * S;
    if (M == 0) return 0;
    DropCfg dc = make_drop(p_drop, seed, site);
    cudaStream_t st = (cudaStream_t)stream;
    float* dz = ws;
    int grid = grid_for_rows(M);
    if (grid > kBwdBlocks) grid = kBwdBlocks;
    const size_t smem = (size_t)kWarps * H * sizeof(float);
    if (H <= 1024) {
        static bool set4 = false;
        if (!set4) { POLUS_CHECK_CUDA(cudaFuncSetAttribute(embed_ln_bwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * 1024 * 4)); set4 = true; }
        embed_ln_bwd_kernel<4><<<grid, kWarps * 32, smem, st>>>((const bf16*)dy, z, mean, rstd, gamma, M, H, dc, d_step, dz, ggamma, gbeta);
    } else {
        static bool set16 = false;
        if (!set16) { POLUS_CHECK_CUDA(cudaFuncSetAttribute(embed_ln_bwd_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * 4096 * 4)); set16 = true; }
        embed_ln_bwd_kernel<16><<<grid, kWarps * 32, smem, st>>>((const bf16*)dy, z, mean, rstd, gamma, M, H, dc, d_step, dz, ggamma, gbeta);
    }
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    if (pos_ids != nullptr)
        embed_scatter_kernel<true><<<S, 192, 0, st>>>(dz, ids, tt, B, S, H, vocab, n_types, gword, gpos, gtype, pos_ids, n_pos);
    else
        embed_scatter_kernel<false><<<S, 192, 0, st>>>(dz, ids, tt, B, S, H, vocab, n_types, gword, gpos, gtype, nullptr, 0);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

}  // namespace

extern "C" int polus_embed_ln_fwd(const int32_t* ids, const int32_t* tt, const float* word, const float* pos,
                                  const float* type, const float* gamma, const float* beta, int B, int S, int H,
                                  int vocab, int n_types, float eps, float p_drop, uint64_t seed, uint32_t site,
                                  const uint32_t* d_step, polus_bf16_t* y, float* z, float* mean, float* rstd, void* stream) {
    return embed_fwd("polus_embed_ln_fwd", ids, tt, word, pos, type, gamma, beta, B, S, H, vocab, n_types, eps, p_drop, seed,
                     site, d_step, y, z, mean, rstd, nullptr, 0, stream);
}

extern "C" int polus_embed_ln_fwd_pos(const int32_t* ids, const int32_t* tt, const float* word, const float* pos,
                                      const float* type, const float* gamma, const float* beta, int B, int S, int H,
                                      int vocab, int n_types, float eps, float p_drop, uint64_t seed, uint32_t site,
                                      const uint32_t* d_step, polus_bf16_t* y, float* z, float* mean, float* rstd,
                                      const int32_t* pos_ids, int n_pos, void* stream) {
    POLUS_REQUIRE(pos_ids != nullptr && n_pos > 0, "polus_embed_ln_fwd_pos: position ids and a table of n_pos > 0 rows required");
    return embed_fwd("polus_embed_ln_fwd_pos", ids, tt, word, pos, type, gamma, beta, B, S, H, vocab, n_types, eps, p_drop,
                     seed, site, d_step, y, z, mean, rstd, pos_ids, n_pos, stream);
}

extern "C" int polus_embed_ln_bwd(const polus_bf16_t* dy, const float* z, const float* mean, const float* rstd,
                                  const float* gamma, const int32_t* ids, const int32_t* tt, int B, int S, int H,
                                  int vocab, int n_types, float p_drop, uint64_t seed, uint32_t site, const uint32_t* d_step,
                                  float* gword, float* gpos, float* gtype, float* ggamma, float* gbeta, float* ws,
                                  void* stream) {
    return embed_bwd("polus_embed_ln_bwd", dy, z, mean, rstd, gamma, ids, tt, B, S, H, vocab, n_types, p_drop, seed, site,
                     d_step, gword, gpos, gtype, ggamma, gbeta, ws, nullptr, 0, stream);
}

extern "C" int polus_embed_ln_bwd_pos(const polus_bf16_t* dy, const float* z, const float* mean, const float* rstd,
                                      const float* gamma, const int32_t* ids, const int32_t* tt, int B, int S, int H,
                                      int vocab, int n_types, float p_drop, uint64_t seed, uint32_t site,
                                      const uint32_t* d_step, float* gword, float* gpos, float* gtype, float* ggamma,
                                      float* gbeta, float* ws, const int32_t* pos_ids, int n_pos, void* stream) {
    POLUS_REQUIRE(pos_ids != nullptr && n_pos > 0, "polus_embed_ln_bwd_pos: position ids and a table of n_pos > 0 rows required");
    return embed_bwd("polus_embed_ln_bwd_pos", dy, z, mean, rstd, gamma, ids, tt, B, S, H, vocab, n_types, p_drop, seed, site,
                     d_step, gword, gpos, gtype, ggamma, gbeta, ws, pos_ids, n_pos, stream);
}

extern "C" int polus_position_ids(const int32_t* ids, int B, int S, int padding_idx, int32_t* pos, void* stream) {
    POLUS_REQUIRE(B >= 0 && S >= 0, "polus_position_ids: bad shape B=%d S=%d", B, S);
    if (B == 0 || S == 0) return 0;
    POLUS_REQUIRE(ids != nullptr && pos != nullptr, "polus_position_ids: ids and pos required");
    position_ids_kernel<<<cdiv(B, kWarps), kWarps * 32, 0, (cudaStream_t)stream>>>(ids, B, S, padding_idx, pos);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}
