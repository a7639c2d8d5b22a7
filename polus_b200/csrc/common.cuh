// Shared device/host helpers for libpolus_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/polus_b200.h"

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------------
// error convention (SURVEY §8b): every entry point returns 0 or a negative class; message kept
// thread-local and returned by polus_last_error().
// ---------------------------------------------------------------------------------------------
void polus_set_error(const char* fmt, ...);

#define POLUS_CHECK_CUDA(expr)                                                            \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            polus_set_error("%s:%d CUDA error %d (%s) in `%s`", __FILE__, __LINE__,       \
                            (int)_e, cudaGetErrorString(_e), #expr);                      \
            return POLUS_ERR_CUDA;                                                        \
        }                                                                                 \
    } while (0)

#define POLUS_REQUIRE(cond, ...)                                                          \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            polus_set_error(__VA_ARGS__);                                                 \
            return POLUS_ERR_INVALID;                                                     \
        }                                                                                 \
    } while (0)

#define POLUS_LAUNCH_CHECK()                                                              \
    do {                                                                                  \
        cudaError_t _e = cudaGetLastError();                                              \
        if (_e != cudaSuccess) {                                                          \
            polus_set_error("%s:%d launch error %d (%s)", __FILE__, __LINE__, (int)_e,    \
                            cudaGetErrorString(_e));                                      \
            return POLUS_ERR_CUDA;                                                        \
        }                                                                                 \
    } while (0)

int polus_num_sms();

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch.  The step is ~260 short kernels (10-60 us) replayed from one CUDA graph; with a
// programmatic edge the next kernel's CTAs are scheduled while the previous kernel drains and run their private
// prologue (barrier init, TMEM allocation, descriptor prefetch, parameter loads) up to pdl_wait().  Rules every
// kernel launched through polus_launch_pdl() follows: (1) pdl_trigger() first thing, (2) EVERY thread executes
// pdl_wait() before its first global-memory access that is not to immutable launch arguments.  pdl_wait() returns
// only when all prerequisite grids have completed and flushed, so ordering stays transitive along the stream.
// ---------------------------------------------------------------------------------------------
template <typename... KArgs, typename... Args>
inline cudaError_t polus_launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                    Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

struct __align__(16) bf16x8 {
    __nv_bfloat162 v[4];
};

__device__ __forceinline__ void unpack8(const bf16x8& p, float* f) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 t = __bfloat1622float2(p.v[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}
__device__ __forceinline__ bf16x8 pack8(const float* f) {
    bf16x8 p;
#pragma unroll
    for (int i = 0; i < 4; ++i) p.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    return p;
}

// streaming (read-once) 16-byte load that does not allocate in L1
__device__ __forceinline__ bf16x8 ld_stream8(const bf16* p) {
    bf16x8 r;
    uint32_t* u = reinterpret_cast<uint32_t*>(&r);
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3])
                 : "l"(p));
    return r;
}

// ---- Philox4x32-10 (Salmon et al. 2011). Counter = (idx_lo, idx_hi, site, step); key = seed.
// The numpy restatement in oracle/philox.py regenerates identical streams, so dropout masks are
// bit-identical between the oracle and the device.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}

// Dropout decisions for 8 consecutive elements starting at element index `idx8*8`.
// keep bit i set <=> 16-bit lane i >= thresh16 (thresh16 = round(p * 65536)).
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t seed, uint32_t site, uint32_t step,
                                                  uint64_t idx8, uint32_t thresh16) {
    uint4 r = philox4x32_10(make_uint4((uint32_t)idx8, (uint32_t)(idx8 >> 32), site, step),
                            make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    uint32_t w[4] = {r.x, r.y, r.z, r.w};
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        m |= ((w[i] & 0xFFFFu) >= thresh16 ? 1u : 0u) << (2 * i);
        m |= ((w[i] >> 16) >= thresh16 ? 1u : 0u) << (2 * i + 1);
    }
    return m;
}

// The same decisions as dropout_keep8, applied directly to 8 fp32 values (v = keep ? v * inv_keep : 0) without building
// the mask first: low lane of word i decides element 2i, high lane element 2i+1;  (w << 16) >= (t << 16)  <=>  lo >= t
// and  w >= (t << 16)  <=>  hi >= t.  Returns the 8 keep bits (dead code unless the caller stores them).
__device__ __forceinline__ uint32_t dropout_apply8(uint64_t seed, uint32_t site, uint32_t step, uint64_t idx8,
                                                   uint32_t thresh16, float inv_keep, float* v) {
    uint4 r = philox4x32_10(make_uint4((uint32_t)idx8, (uint32_t)(idx8 >> 32), site, step),
                            make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    const uint32_t th = thresh16 << 16;
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const bool klo = (w[i] << 16) >= th;
        const bool khi = w[i] >= th;
        v[2 * i] = klo ? v[2 * i] * inv_keep : 0.f;
        v[2 * i + 1] = khi ? v[2 * i + 1] * inv_keep : 0.f;
        bits |= (klo ? 1u : 0u) << (2 * i);
        bits |= (khi ? 1u : 0u) << (2 * i + 1);
    }
    return bits;
}
// dropout from stored keep bits (bit j = element j)
__device__ __forceinline__ void dropout_apply8_bits(uint32_t bits, float inv_keep, float* v) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (bits & (1u << j)) ? v[j] * inv_keep : 0.f;
}

// explicit 128-bit global accesses (the struct-copy form sometimes splits into 32-bit stores)
__device__ __forceinline__ void st_global16(void* p, const bf16x8& v) {
    const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
    asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]) : "memory");
}
__device__ __forceinline__ bf16x8 ld_global16(const void* p) {
    bf16x8 r;
    uint32_t* u = reinterpret_cast<uint32_t*>(&r);
    asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]) : "l"(p));
    return r;
}

// Exact-erf GELU pieces (HF hidden_act="gelu"), written for instruction count -- the FFN-up GEMM epilogue is bound by
// FMA-pipe issue slots, not by MUFU (tools/ubench/alu.cu: FFMA 113/clk/SM, MUFU 16/clk/SM, concurrent).
//   erf by Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7): erf|u| = 1 - (a1 t + .. + a5 t^5) exp(-u^2), t = 1/(1 + p u), u = |x|/sqrt2.
//   phi = exp(-x^2/2)/sqrt(2 pi) comes out of ONE ex2 (its log2 prescale folded into the exponent FFMA) and the
//   polynomial coefficients carry the factor sqrt(2 pi)/2, so that h = poly(t) t phi = (1 - erf|u|)/2 and
//   Phi(x) = 1/2 + copysign(1/2 - h, x).  15 FMA/ALU instructions + 2 MUFU for y = x Phi and y' = Phi + x phi together
//   (was 21; max abs error vs fp64: 5e-7, checked in numpy).
__device__ __forceinline__ void gelu_cdf_pdf(float x, float& cdf, float& pdf) {
    float t, e;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(fabsf(x), 0.3275911f * 0.70710678118654752f, 1.0f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fmaf(x * x, -0.7213475108146667f, -1.325748085975647f)));
    float poly = fmaf(t, 1.3302744626998901f, -1.8212559223175049f);
    poly = fmaf(t, poly, 1.781477928161621f);
    poly = fmaf(t, poly, -0.3565637767314911f);
    poly = fmaf(t, poly, 0.3193815350532532f);
    const float r = fmaf(-poly * t, e, 0.5f);  // 1/2 - h
    cdf = 0.5f + copysignf(r, x);
    pdf = e;
}
// ---- packed fp32x2 arithmetic (Blackwell FFMA2 / FMUL2 / FADD2): one issue slot for two lanes' worth of FMA-pipe work.
// The FMA pipe itself is no faster (tools/ubench/alu.cu: 58.7 FFMA2/clk/SM vs 113 FFMA), but the GEMM epilogues that
// evaluate GELU are bound by ISSUE slots shared with MUFU, ALU, shared-memory and TMEM instructions.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(reinterpret_cast<unsigned long long&>(d))
        : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)), "l"(reinterpret_cast<unsigned long long&>(c)));
    return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    float2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<unsigned long long&>(d))
        : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
    return d;
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
    float2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<unsigned long long&>(d))
        : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
    return d;
}
// gelu_cdf_pdf for two values at once: y = x Phi(x), d = Phi(x) + x phi(x).  Same formula and constants, so each lane's
// result equals the scalar version's up to the fused-multiply rounding of the last two operations.
__device__ __forceinline__ void gelu_fwd_grad2(float2 x, float2& y, float2& d) {
    const float2 ax = make_float2(fabsf(x.x), fabsf(x.y));
    const float2 den = fma2(ax, make_float2(0.3275911f * 0.70710678118654752f, 0.3275911f * 0.70710678118654752f), make_float2(1.0f, 1.0f));
    const float2 arg = fma2(mul2(x, x), make_float2(-0.7213475108146667f, -0.7213475108146667f), make_float2(-1.325748085975647f, -1.325748085975647f));
    float2 t, e;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(den.x));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(den.y));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(arg.x));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(arg.y));
    // the polynomial with all signs flipped, so that  r = 1/2 - poly t e  is one packed FMA
    float2 np = fma2(t, make_float2(-1.3302744626998901f, -1.3302744626998901f), make_float2(1.8212559223175049f, 1.8212559223175049f));
    np = fma2(t, np, make_float2(-1.781477928161621f, -1.781477928161621f));
    np = fma2(t, np, make_float2(0.3565637767314911f, 0.3565637767314911f));
    np = fma2(t, np, make_float2(-0.3193815350532532f, -0.3193815350532532f));
    const float2 r = fma2(mul2(np, t), e, make_float2(0.5f, 0.5f));
    const float2 cdf = add2(make_float2(0.5f, 0.5f), make_float2(copysignf(r.x, x.x), copysignf(r.y, x.y)));
    y = mul2(x, cdf);
    d = fma2(x, e, cdf);
}

// ---- gelu' as 8-bit fixed point (polus_gemm_t.c2_kind = 2).  gelu'(x) lies in [-0.1290, 1.1290]; q = 28 + round(200 x)
// lies in [2, 254], step 0.005: the same aggregate gradient error as a bf16 copy (relative 2^-9 at |x| ~ 1) at half the
// bytes -- the two GEMMs that write / read this tensor are bound by SM store bandwidth and multiplier-tile traffic
// (DESIGN.md section 8).  Encode: one FMA against 1.5 * 2^23 + 28 leaves q in the low mantissa byte (round to nearest
// even done by the FMA); decode: the byte is dropped into the mantissa of 1.5 * 2^23, one subtract, one multiply.
constexpr float kD8Scale = 200.0f, kD8Step = 0.005f, kD8Magic = 12582912.0f, kD8Bias = 28.0f;
__device__ __forceinline__ uint32_t d8_pack4(float a, float b, float c, float d) {
    const uint32_t ya = __float_as_uint(fmaf(a, kD8Scale, kD8Magic + kD8Bias)), yb = __float_as_uint(fmaf(b, kD8Scale, kD8Magic + kD8Bias));
    const uint32_t yc = __float_as_uint(fmaf(c, kD8Scale, kD8Magic + kD8Bias)), yd = __float_as_uint(fmaf(d, kD8Scale, kD8Magic + kD8Bias));
    return __byte_perm(__byte_perm(ya, yb, 0x0040), __byte_perm(yc, yd, 0x0040), 0x5410);
}
__device__ __forceinline__ void d8_unpack4(uint32_t w, float* out) {
    out[0] = (__uint_as_float(__byte_perm(w, 0x4B400000u, 0x7650)) - (kD8Magic + kD8Bias)) * kD8Step;
    out[1] = (__uint_as_float(__byte_perm(w, 0x4B400000u, 0x7651)) - (kD8Magic + kD8Bias)) * kD8Step;
    out[2] = (__uint_as_float(__byte_perm(w, 0x4B400000u, 0x7652)) - (kD8Magic + kD8Bias)) * kD8Step;
    out[3] = (__uint_as_float(__byte_perm(w, 0x4B400000u, 0x7653)) - (kD8Magic + kD8Bias)) * kD8Step;
}

// activations (polus_act_t)
__device__ __forceinline__ float act_fwd(int act, float x) {
    switch (act) {
        case POLUS_ACT_GELU: {
            float cdf, pdf;
            gelu_cdf_pdf(x, cdf, pdf);
            return x * cdf;
        }
        case POLUS_ACT_RELU: return fmaxf(x, 0.0f);
        case POLUS_ACT_SWISH: return x / (1.0f + __expf(-x));
        case POLUS_ACT_TANH: return tanhf(x);
        case POLUS_ACT_MISH: {
            float sp = (x > 20.0f) ? x : log1pf(__expf(x));
            return x * tanhf(sp);
        }
        default: return x;
    }
}
__device__ __forceinline__ float act_grad(int act, float x) {
    switch (act) {
        case POLUS_ACT_GELU: {  // Phi(x) + x phi(x)
            float cdf, pdf;
            gelu_cdf_pdf(x, cdf, pdf);
            return fmaf(x, pdf, cdf);
        }
        case POLUS_ACT_RELU: return x > 0.0f ? 1.0f : 0.0f;
        case POLUS_ACT_SWISH: {
            float s = 1.0f / (1.0f + __expf(-x));
            return s * (1.0f + x * (1.0f - s));
        }
        case POLUS_ACT_TANH: {
            float t = tanhf(x);
            return 1.0f - t * t;
        }
        case POLUS_ACT_MISH: {
            float sp = (x > 20.0f) ? x : log1pf(__expf(x));
            float t = tanhf(sp);
            float s = 1.0f / (1.0f + __expf(-x));
            return t + x * (1.0f - t * t) * s;
        }
        default: return 1.0f;
    }
}

#endif  // __CUDACC__
