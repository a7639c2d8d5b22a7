// Linear-chain CRF: negative log-likelihood with gradients (forward-backward in one launch) and Viterbi
// decode for K <= 128 tags.  K <= 32: one warp per recursion, lane j owns tag j, transitions in shared memory, the T-step
// recurrence kept in registers + warp shuffles (crf_nll_kernel, crf_decode_kernel).  K = 4, the polus.ner tag set:
// one SEQUENCE per lane, the whole K-vector in registers, no cross-lane traffic (crf_nll_lanes_kernel).  33 <= K <= 128,
// and K <= 32 where the [T][K] tables of those kernels do not fit shared memory: one CTA per sequence, thread j owns
// tag j (crf_nll_wide_kernel, crf_decode_wide_kernel; T up to 19 904 / 1 760 steps at K = 128).
//
// Replaces tensorflow_addons.text.crf_log_likelihood / crf_decode, which the reference calls from
// polus/layers.py:78-80 (decode, also run in training), :91-96 and :109-114 (loss); TF executes them
// as a tf.scan / RNN loop of ~6 tiny kernels per time step.
//
// tfa semantics restated here (and in oracle/crf.py):
//   score(b)    = sum_{t<len} x[t,y_t] + sum_{t<len-1} A[y_t,y_{t+1}]
//   alpha_0     = x_0 ; alpha_t[j] = x_t[j] + logsumexp_i(alpha_{t-1}[i] + A[i,j]) ; logZ = logsumexp_j alpha_{len-1}[j]
//   decode      : delta_t[j] = x_t[j] + max_i(delta_{t-1}[i] + A[i,j]), argmax ties -> lowest index,
//                 positions >= len decode to tag 0.
#include "common.cuh"
#include <atomic>
extern std::atomic<long long> g_launch_count;

namespace {

// Scaled forward-backward (Rabiner scaling) instead of per-step log-sum-exp: the recurrences run in the linear
// domain on E = exp(A - max A), each step renormalised, so a time step costs K FMAs + one exp + one reciprocal
// per lane instead of 2K exp + K log.  Warp 0 runs the forward recursion (and the gold-path score), warp 1 the
// backward recursion, concurrently; then all 64 threads turn alpha-hat/beta-hat into marginals = gradients.
//   alpha-hat_t[j] = u_t[j] / c_t,  u_t[j] = (sum_i alpha-hat_{t-1}[i] E[i][j]) * exp(x_t[j] - m_t),  m_t = max_j x_t[j]
//   logZ = sum_t (m_t + log c_t) + (len-1) * max A
//   beta-tilde_t[i] = r_t[i] / d_t, r_t[i] = sum_j E[i][j] w_{t+1}[j],  w_t[j] = exp(x_t[j] - m_t) * beta-tilde_t[j]
//   gamma_t[j]  = alpha-hat_t[j] beta-tilde_t[j] / g_t,                g_t = sum_j alpha-hat_t[j] beta-tilde_t[j]
//   xi_t[i][j]  = alpha-hat_t[i] E[i][j] w_{t+1}[j] / (d_t g_t)        (pair marginal of t -> t+1)
// Shared memory: E [K][K], A [K][K], G [K][K], ah [T][K], ex [T][K] (ex_t[j] = exp(x_t[j] - m_t)), bt [T][K], d [T], c [T].
// reductions over the first kp lanes only (kp = power of two >= K): log2(kp) shuffles instead of 5 on the
// sequential critical path (K = 4 tags => 2)
__device__ __forceinline__ float kmax(float v, int kp) {
    for (int o = kp >> 1; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float ksum(float v, int kp) {
    for (int o = kp >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(64)
crf_nll_kernel(const float* __restrict__ emis, const int32_t* __restrict__ tags, const int32_t* __restrict__ lens,
               const float* __restrict__ trans, const float* __restrict__ weights, int B, int T, int K,
               float* __restrict__ nll_out, float* __restrict__ loss, float* __restrict__ gemis,
               float* __restrict__ gtrans) {
    extern __shared__ float sm[];
    float* sE = sm;
    float* sA = sE + K * K;
    float* sG = sA + K * K;
    float* sAh = sG + K * K;          // [T][K]
    float* sW = sAh + (size_t)T * K;  // [T][K]
    float* sBt = sW + (size_t)T * K;  // [T][K]
    float* sD = sBt + (size_t)T * K;  // [T]
    float* sC = sD + T;               // [T] forward normalisers c_t
    __shared__ float s_logZ, s_score, s_msum[2];
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float amax = -INFINITY;
    for (int i = tid; i < K * K; i += 64) amax = fmaxf(amax, trans[i]);
    amax = warp_max(amax);
    __shared__ float s_amax[2];
    if (lane == 0) s_amax[warp] = amax;
    __syncthreads();
    amax = fmaxf(s_amax[0], s_amax[1]);
    for (int i = tid; i < K * K; i += 64) {
        sA[i] = trans[i];
        sE[i] = expf(trans[i] - amax);
        sG[i] = 0.f;
    }
    __syncthreads();
    int len = lens ? lens[b] : T;
    len = len < 0 ? 0 : (len > T ? T : len);
    const float w_b = (weights ? weights[b] : 1.0f);
    const float gscale = w_b / (float)B;
    const float* x = emis + (long long)b * T * K;
    const int32_t* y = tags + (long long)b * T;
    float* g = gemis + (long long)b * T * K;
    const bool act = lane < K;
    int kp = 1;
    while (kp < K) kp <<= 1;

    if (len == 0) {
        for (int i = tid; i < T * K; i += 64) g[i] = 0.f;
        if (tid == 0 && nll_out) nll_out[b] = 0.f;
        return;
    }
    // ---------------- parallel over t: everything that does not depend on the recurrences.  ex_t[j] = exp(x_t[j] - m_t)
    // goes to sW, sum_t m_t is reduced over the CTA: the exp / max / log work of a time step (~60 dependent instructions
    // in one warp, the loop ran at ~1100 cycles per step) leaves the two sequential loops, which keep K FMAs, the
    // normalising sum and one reciprocal per step.
    {
        float msum = 0.f;
        for (int t = tid; t < len; t += 64) {
            float m = -INFINITY;
            for (int j = 0; j < K; ++j) m = fmaxf(m, x[t * K + j]);
            for (int j = 0; j < K; ++j) sW[t * K + j] = expf(x[t * K + j] - m);
            msum += m;
        }
        msum = warp_sum(msum);
        if (lane == 0) s_msum[warp] = msum;
    }
    __syncthreads();
    if (warp == 0) {
        // ---------------- forward recursion + gold path score
        float u = act ? sW[lane] : 0.f;
        float c = ksum(u, kp);
        float ah = u * __frcp_rn(c);
        if (act) sAh[lane] = ah;
        if (lane == 0) sC[0] = c;
        float exn = (act && 1 < len) ? sW[K + lane] : 0.f;  // next step's factor, loaded one step ahead
        for (int t = 1; t < len; ++t) {
            const float ex = exn;
            exn = (act && t + 1 < len) ? sW[(t + 1) * K + lane] : 0.f;
            float s = 0.f;
            for (int i = 0; i < K; ++i) s = fmaf(__shfl_sync(0xffffffffu, ah, i), act ? sE[i * K + lane] : 0.f, s);
            u = s * ex;
            c = ksum(u, kp);
            ah = u * __frcp_rn(c);
            if (act) sAh[t * K + lane] = ah;
            if (lane == 0) sC[t] = c;
        }
        __syncwarp();
        // logZ = sum_t (m_t + log c_t) + (len - 1) max A, the logs taken in parallel
        float lz = 0.f;
        for (int t = lane; t < len; t += 32) lz += logf(sC[t]);
        lz = warp_sum(lz);
        float sc = 0.f;
        for (int t = lane; t < len; t += 32) {
            const int yt = min(max(y[t], 0), K - 1);
            sc += x[t * K + yt];
            if (t + 1 < len) sc += sA[yt * K + min(max(y[t + 1], 0), K - 1)];
        }
        sc = warp_sum(sc);
        if (lane == 0) {
            s_logZ = lz + (s_msum[0] + s_msum[1]) + (float)(len - 1) * amax;
            s_score = sc;
        }
    } else {
        // ---------------- backward recursion (sW keeps ex_t; w_t[j] = ex_t[j] * beta-tilde_t[j] is rebuilt where it is used)
        float bt = act ? 1.0f : 0.f;  // beta-tilde_{len-1} (any positive constant: marginals renormalise)
        float exn = act ? sW[(len - 1) * K + lane] : 0.f;
        for (int t = len - 1; t >= 0; --t) {
            const float wv = exn * bt;  // w_t[j]
            exn = (act && t > 0) ? sW[(t - 1) * K + lane] : 0.f;
            if (act) sBt[t * K + lane] = bt;
            if (t > 0) {
                float r = 0.f;  // r_{t-1}[i = lane]
                for (int j = 0; j < K; ++j) r = fmaf(act ? sE[lane * K + j] : 0.f, __shfl_sync(0xffffffffu, wv, j), r);
                const float d = ksum(r, kp);
                if (lane == 0) sD[t - 1] = d;
                bt = r * __frcp_rn(d);
            }
        }
    }
    __syncthreads();
    const float nll = s_logZ - s_score;
    if (tid == 0) {
        if (nll_out) nll_out[b] = nll;
        if (loss) atomicAdd(loss, nll * gscale);
    }
    // ---------------- emission gradients: gscale * (gamma_t[j] - [y_t == j]); zero beyond len
    for (int t = tid; t < T; t += 64) {
        if (t < len) {
            float gsum = 0.f;
            for (int j = 0; j < K; ++j) gsum += sAh[t * K + j] * sBt[t * K + j];
            const float inv = 1.0f / gsum;
            const int yt = min(max(y[t], 0), K - 1);
            for (int j = 0; j < K; ++j)
                g[t * K + j] = gscale * (sAh[t * K + j] * sBt[t * K + j] * inv - (j == yt ? 1.0f : 0.f));
            if (t + 1 < len) sD[t] = 1.0f / (sD[t] * gsum);  // -> 1 / (d_t g_t), the pair-marginal normaliser
        } else {
            for (int j = 0; j < K; ++j) g[t * K + j] = 0.f;
        }
    }
    __syncthreads();
    // ---------------- transition gradients: sum_t xi_t[i][j] - counts of gold transitions
    if (gtrans != nullptr) {
        for (int pidx = tid; pidx < K * K; pidx += 64) {
            const int i = pidx / K, j = pidx % K;
            const float e = sE[pidx];
            float acc = 0.f;
            for (int t = 0; t + 1 < len; ++t) acc = fmaf(sAh[t * K + i] * (sW[(t + 1) * K + j] * sBt[(t + 1) * K + j]), sD[t], acc);
            sG[pidx] = acc * e;
        }
        __syncthreads();
        for (int t = tid; t + 1 < len; t += 64) {
            const int yp = min(max(y[t], 0), K - 1), yn = min(max(y[t + 1], 0), K - 1);
            atomicAdd(&sG[yp * K + yn], -1.0f);
        }
        __syncthreads();
        for (int i = tid; i < K * K; i += 64) atomicAdd(gtrans + i, gscale * sG[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// K = 4 (the polus.ner tag set), one sequence per LANE.  In crf_nll_kernel lane j owns tag j, so every time step walks
// a chain of warp shuffles (K broadcasts of alpha-hat, log2 K butterfly steps for the normaliser): ~690 cycles per step
// in ncu for ~35 instructions (profiles/r01_ncu_summary_v18_attn_crf_b128.txt).  Here a lane carries the whole K-vector
// of ONE sequence in registers: a step is 16 FMAs, 3 adds, one reciprocal and 4 multiplies with no cross-lane traffic
// (dependency chain ~75 cycles).  A CTA of 256 threads owns SEQ sequences: lane q of warp 0 runs the forward recursion
// of sequence q, lane q of warp 1 the backward one, concurrently; the exp / max / log work, the gradients and the
// gold-path scores are computed by all eight warps in parallel phases around them.  Same formulas (scaled
// forward-backward, see the top of this file) and the same outputs as crf_nll_kernel.
// Shared memory per sequence: ex [T][4] (+4 pad), alpha-hat [T][4] (+4), beta-tilde [T][4] (+4), m [T] (+1), c [T] (+1),
// d [T] (+1): the pads put the rows of consecutive sequences on different banks for the per-lane row walks.
template <int SEQ>
__global__ void __launch_bounds__(256)
crf_nll_lanes_kernel(const float* __restrict__ emis, const int32_t* __restrict__ tags, const int32_t* __restrict__ lens,
                     const float* __restrict__ trans, const float* __restrict__ weights, int B, int T,
                     float* __restrict__ nll_out, float* __restrict__ loss, float* __restrict__ gemis,
                     float* __restrict__ gtrans) {
    constexpr int K = 4;
    extern __shared__ __align__(16) float sm[];
    const int RS = T * K + K;  // row stride of the [T][4] tables (floats)
    const int CS = T + 1;      // row stride of the [T] tables
    float* sE = sm;                       // [4][4] exp(A - max A)
    float* sA = sE + 16;                  // [4][4] A
    float* sG = sA + 16;                  // [4][4] transition-gradient accumulator of this CTA
    float* sEX = sG + 16;                 // [SEQ][RS]
    float* sAH = sEX + (size_t)SEQ * RS;  // [SEQ][RS]
    float* sBT = sAH + (size_t)SEQ * RS;  // [SEQ][RS]
    float* sM = sBT + (size_t)SEQ * RS;   // [SEQ][CS]
    float* sC = sM + (size_t)SEQ * CS;    // [SEQ][CS]
    float* sD = sC + (size_t)SEQ * CS;    // [SEQ][CS]
    __shared__ int s_len[SEQ];
    __shared__ float s_gscale[SEQ];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b0 = blockIdx.x * SEQ;

    float amax = -INFINITY;
#pragma unroll
    for (int i = 0; i < 16; ++i) amax = fmaxf(amax, trans[i]);
    if (tid < 16) {
        sA[tid] = trans[tid];
        sE[tid] = expf(trans[tid] - amax);
        sG[tid] = 0.f;
    }
    if (tid < SEQ) {
        const int b = b0 + tid;
        int len = 0;
        float gs = 0.f;
        if (b < B) {
            len = lens ? lens[b] : T;
            len = len < 0 ? 0 : (len > T ? T : len);
            gs = (weights ? weights[b] : 1.0f) / (float)B;
        }
        s_len[tid] = len;
        s_gscale[tid] = gs;
    }
    __syncthreads();

    // ---------------- phase A (all threads, one (sequence, t) pair at a time): m_t = max_j x_t[j], ex_t[j] = exp(x_t[j] - m_t)
    for (int it = tid; it < SEQ * T; it += 256) {
        const int q = it / T, t = it - q * T;
        if (t < s_len[q]) {
            const float4 xv = *reinterpret_cast<const float4*>(emis + ((long long)(b0 + q) * T + t) * K);
            const float m = fmaxf(fmaxf(xv.x, xv.y), fmaxf(xv.z, xv.w));
            *reinterpret_cast<float4*>(sEX + (size_t)q * RS + t * K) = make_float4(expf(xv.x - m), expf(xv.y - m), expf(xv.z - m), expf(xv.w - m));
            sM[q * CS + t] = m;
        }
    }
    __syncthreads();

    // ---------------- phase B: the two recursions, one sequence per lane
    if (warp == 0 && lane < SEQ && s_len[lane] > 0) {
        const int len = s_len[lane];
        const float* ex = sEX + (size_t)lane * RS;
        float* ah = sAH + (size_t)lane * RS;
        float* cp = sC + lane * CS;
        float e[16];  // E[i][j], i = previous tag, j = current tag
#pragma unroll
        for (int i = 0; i < 16; ++i) e[i] = sE[i];
        float4 u = *reinterpret_cast<const float4*>(ex);
        float c = (u.x + u.y) + (u.z + u.w);
        float r = __frcp_rn(c);
        float4 a = make_float4(u.x * r, u.y * r, u.z * r, u.w * r);
        *reinterpret_cast<float4*>(ah) = a;
        cp[0] = c;
        float4 nx = 1 < len ? *reinterpret_cast<const float4*>(ex + K) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int t = 1; t < len; ++t) {
            const float4 x4 = nx;
            if (t + 1 < len) nx = *reinterpret_cast<const float4*>(ex + (t + 1) * K);  // one step ahead of its use
            u.x = fmaf(a.x, e[0], fmaf(a.y, e[4], fmaf(a.z, e[8], a.w * e[12]))) * x4.x;
            u.y = fmaf(a.x, e[1], fmaf(a.y, e[5], fmaf(a.z, e[9], a.w * e[13]))) * x4.y;
            u.z = fmaf(a.x, e[2], fmaf(a.y, e[6], fmaf(a.z, e[10], a.w * e[14]))) * x4.z;
            u.w = fmaf(a.x, e[3], fmaf(a.y, e[7], fmaf(a.z, e[11], a.w * e[15]))) * x4.w;
            c = (u.x + u.y) + (u.z + u.w);
            r = __frcp_rn(c);
            a = make_float4(u.x * r, u.y * r, u.z * r, u.w * r);
            *reinterpret_cast<float4*>(ah + t * K) = a;
            cp[t] = c;
        }
    } else if (warp == 1 && lane < SEQ && s_len[lane] > 0) {
        const int len = s_len[lane];
        const float* ex = sEX + (size_t)lane * RS;
        float* btp = sBT + (size_t)lane * RS;
        float* dp = sD + lane * CS;
        float e[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) e[i] = sE[i];
        float4 bt = make_float4(1.f, 1.f, 1.f, 1.f);  // beta-tilde_{len-1} (any positive constant: marginals renormalise)
        float4 nx = *reinterpret_cast<const float4*>(ex + (len - 1) * K);
        for (int t = len - 1; t >= 0; --t) {
            const float4 x4 = nx;
            if (t > 0) nx = *reinterpret_cast<const float4*>(ex + (t - 1) * K);
            *reinterpret_cast<float4*>(btp + t * K) = bt;
            if (t > 0) {
                const float4 w = make_float4(x4.x * bt.x, x4.y * bt.y, x4.z * bt.z, x4.w * bt.w);  // w_t[j]
                float4 rr;  // r_{t-1}[i] = sum_j E[i][j] w_t[j]
                rr.x = fmaf(e[0], w.x, fmaf(e[1], w.y, fmaf(e[2], w.z, e[3] * w.w)));
                rr.y = fmaf(e[4], w.x, fmaf(e[5], w.y, fmaf(e[6], w.z, e[7] * w.w)));
                rr.z = fmaf(e[8], w.x, fmaf(e[9], w.y, fmaf(e[10], w.z, e[11] * w.w)));
                rr.w = fmaf(e[12], w.x, fmaf(e[13], w.y, fmaf(e[14], w.z, e[15] * w.w)));
                const float d = (rr.x + rr.y) + (rr.z + rr.w);
                dp[t - 1] = d;
                const float r = __frcp_rn(d);
                bt = make_float4(rr.x * r, rr.y * r, rr.z * r, rr.w * r);
            }
        }
    }
    __syncthreads();

    // ---------------- phase C1: log-partition and gold-path score, one warp per sequence
    for (int q = warp; q < SEQ; q += 8) {
        const int b = b0 + q, len = s_len[q];
        if (b >= B) continue;  // warp-uniform
        if (len == 0) {
            if (lane == 0 && nll_out) nll_out[b] = 0.f;
            continue;
        }
        const float* x = emis + (long long)b * T * K;
        const int32_t* y = tags + (long long)b * T;
        float lz = 0.f, sc = 0.f;
        for (int t = lane; t < len; t += 32) {
            lz += sM[q * CS + t] + logf(sC[q * CS + t]);
            const int yt = min(max(y[t], 0), K - 1);
            sc += x[t * K + yt];
            if (t + 1 < len) sc += sA[yt * K + min(max(y[t + 1], 0), K - 1)];
        }
        lz = warp_sum(lz);
        sc = warp_sum(sc);
        if (lane == 0) {
            const float nll = lz + (float)(len - 1) * amax - sc;
            if (nll_out) nll_out[b] = nll;
            if (loss) atomicAdd(loss, nll * s_gscale[q]);
        }
    }
    // ---------------- phase C2: emission gradients gscale * (gamma_t[j] - [y_t == j]), zero beyond len;
    //                  d_t -> 1 / (d_t g_t), the pair-marginal normaliser
    for (int it = tid; it < SEQ * T; it += 256) {
        const int q = it / T, t = it - q * T;
        const int b = b0 + q;
        if (b >= B) continue;
        float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < s_len[q]) {
            const float4 a = *reinterpret_cast<const float4*>(sAH + (size_t)q * RS + t * K);
            const float4 bt = *reinterpret_cast<const float4*>(sBT + (size_t)q * RS + t * K);
            const float4 pr = make_float4(a.x * bt.x, a.y * bt.y, a.z * bt.z, a.w * bt.w);
            const float gsum = (pr.x + pr.y) + (pr.z + pr.w);
            const float inv = 1.0f / gsum;
            const float gs = s_gscale[q];
            const int yt = min(max(tags[(long long)b * T + t], 0), K - 1);
            g4.x = gs * (pr.x * inv - (yt == 0 ? 1.0f : 0.f));
            g4.y = gs * (pr.y * inv - (yt == 1 ? 1.0f : 0.f));
            g4.z = gs * (pr.z * inv - (yt == 2 ? 1.0f : 0.f));
            g4.w = gs * (pr.w * inv - (yt == 3 ? 1.0f : 0.f));
            if (t + 1 < s_len[q]) sD[q * CS + t] = 1.0f / (sD[q * CS + t] * gsum);
        }
        *reinterpret_cast<float4*>(gemis + ((long long)b * T + t) * K) = g4;
    }
    __syncthreads();
    // ---------------- phase C3: transition gradients  sum_q gscale_q (E[i][j] sum_t alpha-hat_t[i] w_{t+1}[j] / (d_t g_t) - #gold(i -> j))
    if (gtrans != nullptr) {
        for (int q = warp; q < SEQ; q += 8) {
            const int len = s_len[q];
            if (b0 + q >= B || len < 2) continue;  // warp-uniform
            const int pidx = lane & 15, i = pidx >> 2, j = pidx & 3;
            const float* ah = sAH + (size_t)q * RS;
            const float* ex = sEX + (size_t)q * RS;
            const float* bt = sBT + (size_t)q * RS;
            float acc = 0.f;
            for (int t = lane >> 4; t + 1 < len; t += 2)  // the two half-warps take alternate time steps
                acc = fmaf(ah[t * K + i] * (ex[(t + 1) * K + j] * bt[(t + 1) * K + j]), sD[q * CS + t], acc);
            acc += __shfl_xor_sync(0xffffffffu, acc, 16);
            if (lane < 16) atomicAdd(&sG[pidx], s_gscale[q] * acc * sE[pidx]);
            const int32_t* y = tags + (long long)(b0 + q) * T;
            for (int t = lane; t + 1 < len; t += 32) {
                const int yp = min(max(y[t], 0), K - 1), yn = min(max(y[t + 1], 0), K - 1);
                atomicAdd(&sG[yp * K + yn], -s_gscale[q]);
            }
        }
        __syncthreads();
        if (tid < 16) atomicAdd(gtrans + tid, sG[tid]);
    }
}

__global__ void crf_decode_kernel(const float* __restrict__ emis, const int32_t* __restrict__ lens,
                                  const float* __restrict__ trans, int T, int K, int32_t* __restrict__ tags_out,
                                  float* __restrict__ score_out) {
    extern __shared__ float sm[];
    float* sA = sm;                                              // [K][K]
    uint8_t* bp = reinterpret_cast<uint8_t*>(sm + K * K);        // [T][K] back-pointers
    const int b = blockIdx.x, lane = threadIdx.x;
    for (int i = lane; i < K * K; i += 32) sA[i] = trans[i];
    __syncwarp();
    int len = lens ? lens[b] : T;
    len = len < 0 ? 0 : (len > T ? T : len);
    const float* x = emis + (long long)b * T * K;
    int32_t* out = tags_out + (long long)b * T;
    const bool act = lane < K;
    for (int t = len + lane; t < T; t += 32) out[t] = 0;
    if (len == 0) {
        if (lane == 0 && score_out) score_out[b] = 0.f;
        return;
    }
    float delta = act ? x[lane] : -INFINITY;
    for (int t = 1; t < len; ++t) {
        float best = -INFINITY;
        int arg = 0;
        for (int i = 0; i < K; ++i) {
            const float di = __shfl_sync(0xffffffffu, delta, i);
            if (act) {
                const float c = di + sA[i * K + lane];
                if (c > best) {  // strict: ties keep the lowest i (tf.argmax)
                    best = c;
                    arg = i;
                }
            }
        }
        if (act) {
            bp[t * K + lane] = (uint8_t)arg;
            delta = x[t * K + lane] + best;
        }
    }
    // final argmax over j, ties -> lowest j
    float bv = delta;
    int bi = act ? lane : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
        }
    }
    __syncwarp();
    if (lane == 0) {
        if (score_out) score_out[b] = bv;
        int cur = bi;
        out[len - 1] = cur;
        for (int t = len - 1; t >= 1; --t) {
            cur = bp[t * K + cur];
            out[t - 1] = cur;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Wide tag sets (33 <= K <= 128), and K <= 32 at lengths whose [T][K] tables do not fit crf_nll_kernel's or
// crf_decode_kernel's shared memory (K = 32 at T = 512).  One CTA per sequence, thread j owns tag j (blockDim = K rounded
// up to 32, padding threads carry zeros).  crf_nll_wide_kernel runs the scaled recursions of crf_nll_kernel one after the
// other, so that no per-step table lives in shared memory and the kernel needs no workspace:
//   forward : alpha-hat_t goes to row t of gemis (a [B][T][K] fp32 output anyway); m_t and c_t stay in shared memory.
//   backward: reads alpha-hat_t back, and overwrites row t with gscale * (gamma_t - onehot(y_t)).
// Each step broadcasts an unnormalised vector (u_t forward, v_t = ex_t * r_t backward) through shared memory together with
// the per-warp partial sums of its normaliser, and the reader applies the normaliser: one __syncthreads per step.  The
// backward works with r_t = beta-tilde_t * d_t, so that g_t = h_t / d_t with h_t = sum_i alpha-hat_t[i] r_t[i], and
//   gamma_t[i] = alpha-hat_t[i] r_t[i] / h_t,   xi_t[i][j] = alpha-hat_t[i] E[i][j] v_{t+1}[j] / (h_t d_{t+1}).
// Registers: forward, column j of E (128 floats); backward, row i of sum_t xi_t / E (128 floats), multiplied by E at the end.
// Shared memory: E [KP][129], KP = blockDim (the backward's row i of E as column i, so that a warp's loads are
// conflict-free; at the end the transition gradient), m [T], c [T]: (129 KP + 2T) * 4 bytes, 70 KB at K = 128, T = 512.
constexpr int kWideMaxK = 128;
constexpr int kWideChunks = kWideMaxK / 32;

__global__ void __launch_bounds__(kWideMaxK)
crf_nll_wide_kernel(const float* __restrict__ emis, const int32_t* __restrict__ tags, const int32_t* __restrict__ lens,
                    const float* __restrict__ trans, const float* __restrict__ weights, int B, int T, int K,
                    float* __restrict__ nll_out, float* __restrict__ loss, float* __restrict__ gemis,
                    float* __restrict__ gtrans) {
    extern __shared__ __align__(16) float smw[];
    constexpr int KS = kWideMaxK + 1;  // a constant stride: the backward's loads of a column of E take immediate offsets
    const int KP = blockDim.x;
    float* sE = smw;  // E[i][j] at j * KS + i, zero rows j in [K, KP); after the backward G[i][j] at i * KS + j
    float* sM = sE + KP * KS;  // [T] m_t = max_j x_t[j]
    float* sC = sM + T;       // [T] forward normalisers c_t
    __shared__ __align__(16) float s_vec[3][kWideMaxK];  // broadcast vectors: written at a step, read there and at the next
    __shared__ float2 s_part[3][kWideChunks];            // their per-warp partial sums
    const int b = blockIdx.x, j = threadIdx.x, lane = j & 31, warp = j >> 5, nw = blockDim.x >> 5;
    const bool act = j < K;

    float amax = -INFINITY;
    for (int i = j; i < K * K; i += blockDim.x) amax = fmaxf(amax, trans[i]);
    amax = warp_max(amax);
    if (lane == 0) s_part[2][warp].x = amax;
    __syncthreads();
    amax = s_part[2][0].x;
    for (int w = 1; w < nw; ++w) amax = fmaxf(amax, s_part[2][w].x);
    for (int idx = j; idx < K * K; idx += blockDim.x) sE[(idx % K) * KS + idx / K] = expf(trans[idx] - amax);
    for (int idx = K * KS + j; idx < KP * KS; idx += blockDim.x) sE[idx] = 0.f;
    float e[kWideMaxK];  // E[i][j] for this thread's tag j
#pragma unroll
    for (int i = 0; i < kWideMaxK; ++i) e[i] = (act && i < K) ? expf(trans[i * K + j] - amax) : 0.f;

    int len = lens ? lens[b] : T;
    len = len < 0 ? 0 : (len > T ? T : len);
    const float gscale = (weights ? weights[b] : 1.0f) / (float)B;
    const float* x = emis + (long long)b * T * K;
    const int32_t* y = tags + (long long)b * T;
    float* g = gemis + (long long)b * T * K;
    for (int idx = len * K + j; idx < T * K; idx += blockDim.x) g[idx] = 0.f;
    if (len == 0) {
        if (j == 0 && nll_out) nll_out[b] = 0.f;
        return;
    }
    for (int t = warp; t < len; t += nw) {  // m_t, one warp per row
        float m = -INFINITY;
        for (int q = lane; q < K; q += 32) m = fmaxf(m, x[t * K + q]);
        m = warp_max(m);
        if (lane == 0) sM[t] = m;
    }
    __syncthreads();

    // ---------------- forward: u_0 = ex_0, u_{t+1}[j] = (sum_i u_t[i] E[i][j]) / c_t * ex_{t+1}[j], c_t = sum_j u_t[j]
    float u = act ? expf(x[j] - sM[0]) : 0.f;
    int sl = 0;
    for (int t = 0;; ++t) {
        const bool more = t + 1 < len;
        const float xn = (act && more) ? x[(t + 1) * K + j] : 0.f;  // one step ahead of its use
        s_vec[sl][j] = u;
        const float pu = warp_sum(u);
        if (lane == 0) s_part[sl][warp].x = pu;
        __syncthreads();
        float c = s_part[sl][0].x;
        for (int w = 1; w < nw; ++w) c += s_part[sl][w].x;
        const float rc = __frcp_rn(c);
        if (act) g[t * K + j] = u * rc;  // alpha-hat_t
        if (j == 0) sC[t] = c;
        if (!more) break;
        const float* v = s_vec[sl];
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
        for (int ch = 0; ch < kWideChunks; ++ch) {
            if (ch * 32 < K) {
#pragma unroll
                for (int q = ch * 32; q < ch * 32 + 32; q += 4) {
                    const float4 v4 = *reinterpret_cast<const float4*>(v + q);
                    s0 = fmaf(v4.x, e[q], s0);
                    s1 = fmaf(v4.y, e[q + 1], s1);
                    s2 = fmaf(v4.z, e[q + 2], s2);
                    s3 = fmaf(v4.w, e[q + 3], s3);
                }
            }
        }
        u = act ? ((s0 + s1) + (s2 + s3)) * rc * expf(xn - sM[t + 1]) : 0.f;
        sl = sl == 2 ? 0 : sl + 1;
    }
    __syncthreads();

    // ---------------- logZ = sum_t (m_t + log c_t) + (len - 1) max A, and the gold-path score
    {
        float lz = 0.f, sc = 0.f;
        for (int t = j; t < len; t += blockDim.x) {
            lz += sM[t] + logf(sC[t]);
            const int yt = min(max(y[t], 0), K - 1);
            sc += x[t * K + yt];
            if (t + 1 < len) sc += trans[yt * K + min(max(y[t + 1], 0), K - 1)];
        }
        lz = warp_sum(lz);
        sc = warp_sum(sc);
        if (lane == 0) s_part[0][warp] = make_float2(lz, sc);
        s_vec[2][j] = 0.f;  // v_len: the backward's first step has no pair (t, t + 1)
        __syncthreads();
        if (j == 0) {
            float lzs = s_part[0][0].x, scs = s_part[0][0].y;
            for (int w = 1; w < nw; ++w) {
                lzs += s_part[0][w].x;
                scs += s_part[0][w].y;
            }
            const float nll = lzs + (float)(len - 1) * amax - scs;
            if (nll_out) nll_out[b] = nll;
            if (loss) atomicAdd(loss, nll * gscale);
        }
        __syncthreads();
    }

    // ---------------- backward, thread i = j: r_{len-1} = 1, r_{t-1}[i] = sum_j E[i][j] v_t[j] / d_t, d_t = sum_i r_t[i]
    const int i = j, il = act ? i : 0;  // padding threads load a valid column and discard the result
    float gr[kWideMaxK];  // sum_t alpha-hat_t[i] v_{t+1}[j] / (h_t d_{t+1})
#pragma unroll
    for (int q = 0; q < kWideMaxK; ++q) gr[q] = 0.f;
    float r = act ? 1.f : 0.f;
    float dn = 1.f;  // d_{t+1}
    float ah = act ? g[(len - 1) * K + i] : 0.f;
    float xt = act ? x[(len - 1) * K + i] : 0.f;
    int yt = min(max(y[len - 1], 0), K - 1);
    int cur = 0, nxt = 2;  // s_vec slots of v_t and v_{t+1}
    for (int t = len - 1; t >= 0; --t) {
        float ahp = 0.f, xp = 0.f;
        int yp = 0;
        if (t > 0) {  // one step ahead of their use
            if (act) {
                ahp = g[(t - 1) * K + i];
                xp = x[(t - 1) * K + i];
            }
            yp = min(max(y[t - 1], 0), K - 1);
        }
        s_vec[cur][i] = act ? expf(xt - sM[t]) * r : 0.f;
        const float pd = warp_sum(r), ph = warp_sum(ah * r);
        if (lane == 0) s_part[cur][warp] = make_float2(pd, ph);
        __syncthreads();
        float d = s_part[cur][0].x, h = s_part[cur][0].y;
        for (int w = 1; w < nw; ++w) {
            d += s_part[cur][w].x;
            h += s_part[cur][w].y;
        }
        if (act) g[t * K + i] = gscale * (ah * r * (1.0f / h) - (i == yt ? 1.0f : 0.f));
        const float coef = (act && t + 1 < len) ? ah / (h * dn) : 0.f;
        const float* vc = s_vec[cur];
        const float* vn = s_vec[nxt];
        float r0 = 0.f, r1 = 0.f, r2 = 0.f, r3 = 0.f;
#pragma unroll
        for (int ch = 0; ch < kWideChunks; ++ch) {
            if (ch * 32 < K) {
#pragma unroll
                for (int q = ch * 32; q < ch * 32 + 32; q += 4) {
                    const float4 c4 = *reinterpret_cast<const float4*>(vc + q);
                    r0 = fmaf(sE[q * KS + il], c4.x, r0);
                    r1 = fmaf(sE[(q + 1) * KS + il], c4.y, r1);
                    r2 = fmaf(sE[(q + 2) * KS + il], c4.z, r2);
                    r3 = fmaf(sE[(q + 3) * KS + il], c4.w, r3);
                }
            }
        }
#pragma unroll
        for (int ch = 0; ch < kWideChunks; ++ch) {
            if (ch * 32 < K) {
#pragma unroll
                for (int q = ch * 32; q < ch * 32 + 32; q += 4) {
                    const float4 n4 = *reinterpret_cast<const float4*>(vn + q);
                    gr[q] = fmaf(coef, n4.x, gr[q]);
                    gr[q + 1] = fmaf(coef, n4.y, gr[q + 1]);
                    gr[q + 2] = fmaf(coef, n4.z, gr[q + 2]);
                    gr[q + 3] = fmaf(coef, n4.w, gr[q + 3]);
                }
            }
        }
        r = act ? ((r0 + r1) + (r2 + r3)) * __frcp_rn(d) : 0.f;
        dn = d;
        ah = ahp;
        xt = xp;
        yt = yp;
        nxt = cur;
        cur = cur == 0 ? 2 : cur - 1;
    }

    // ---------------- transition gradients: E[i][j] * sum_t ... - counts of gold transitions
    if (gtrans != nullptr) {
#pragma unroll
        for (int q = 0; q < kWideMaxK; ++q)
            if (act && q < K) gr[q] *= sE[q * KS + i];
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kWideMaxK; ++q)
            if (act && q < K) sE[i * KS + q] = gr[q];
        __syncthreads();
        for (int t = j; t + 1 < len; t += blockDim.x)
            atomicAdd(&sE[min(max(y[t], 0), K - 1) * KS + min(max(y[t + 1], 0), K - 1)], -1.0f);
        __syncthreads();
        for (int idx = j; idx < K * K; idx += blockDim.x) atomicAdd(gtrans + idx, gscale * sE[(idx / K) * KS + idx % K]);
    }
}

// Viterbi for the same shapes: thread j owns tag j, keeps column j of A in registers and broadcasts delta_{t-1} through
// shared memory (one __syncthreads per step).  The max over i runs as four interleaved chains (i mod 4), each keeping its
// first maximum, merged lowest index first: the same tag and value as one ascending scan with a strict compare, as in
// crf_decode_kernel.  Back-pointers: u8 [T][K] in shared memory (64 KB at K = 128, T = 512).
__global__ void __launch_bounds__(kWideMaxK)
crf_decode_wide_kernel(const float* __restrict__ emis, const int32_t* __restrict__ lens, const float* __restrict__ trans,
                       int T, int K, int32_t* __restrict__ tags_out, float* __restrict__ score_out) {
    extern __shared__ uint8_t sbp[];  // [T][K] back-pointers
    __shared__ __align__(16) float s_delta[2][kWideMaxK];
    __shared__ float s_bv[kWideChunks];
    __shared__ int s_bi[kWideChunks];
    const int b = blockIdx.x, j = threadIdx.x, lane = j & 31, warp = j >> 5, nw = blockDim.x >> 5;
    const bool act = j < K;
    int len = lens ? lens[b] : T;
    len = len < 0 ? 0 : (len > T ? T : len);
    const float* x = emis + (long long)b * T * K;
    int32_t* out = tags_out + (long long)b * T;
    for (int t = len + j; t < T; t += blockDim.x) out[t] = 0;
    if (len == 0) {
        if (j == 0 && score_out) score_out[b] = 0.f;
        return;
    }
    float a[kWideMaxK];  // A[i][j]
#pragma unroll
    for (int i = 0; i < kWideMaxK; ++i) a[i] = (act && i < K) ? trans[i * K + j] : 0.f;
    float delta = act ? x[j] : -INFINITY;  // padding tags stay at -inf: never a maximum
    float xn = (act && 1 < len) ? x[K + j] : 0.f;
    for (int t = 1; t < len; ++t) {
        const float xt = xn;
        if (act && t + 1 < len) xn = x[(t + 1) * K + j];
        float* dv = s_delta[t & 1];
        dv[j] = delta;
        __syncthreads();
        float bv[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        int bi[4] = {kWideMaxK, kWideMaxK, kWideMaxK, kWideMaxK};
#pragma unroll
        for (int ch = 0; ch < kWideChunks; ++ch) {
            if (ch * 32 < K) {
#pragma unroll
                for (int q = ch * 32; q < ch * 32 + 32; q += 4) {
                    const float4 d4 = *reinterpret_cast<const float4*>(dv + q);
                    const float c0 = d4.x + a[q], c1 = d4.y + a[q + 1], c2 = d4.z + a[q + 2], c3 = d4.w + a[q + 3];
                    if (c0 > bv[0]) { bv[0] = c0; bi[0] = q; }
                    if (c1 > bv[1]) { bv[1] = c1; bi[1] = q + 1; }
                    if (c2 > bv[2]) { bv[2] = c2; bi[2] = q + 2; }
                    if (c3 > bv[3]) { bv[3] = c3; bi[3] = q + 3; }
                }
            }
        }
#pragma unroll
        for (int k = 1; k < 4; ++k) {
            if (bv[k] > bv[0] || (bv[k] == bv[0] && bi[k] < bi[0])) {
                bv[0] = bv[k];
                bi[0] = bi[k];
            }
        }
        if (act) {
            sbp[t * K + j] = (uint8_t)(bi[0] == kWideMaxK ? 0 : bi[0]);  // nothing above -inf: tag 0, as the scan
            delta = xt + bv[0];
        }
    }
    // final argmax over j, ties -> lowest j
    float bv = delta;
    int bi = act ? j : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
        }
    }
    if (lane == 0) {
        s_bv[warp] = bv;
        s_bi[warp] = bi;
    }
    __syncthreads();
    if (j == 0) {
        for (int w = 1; w < nw; ++w) {
            if (s_bv[w] > bv || (s_bv[w] == bv && s_bi[w] < bi)) {
                bv = s_bv[w];
                bi = s_bi[w];
            }
        }
        if (score_out) score_out[b] = bv;
        int cur = bi;
        out[len - 1] = cur;
        for (int t = len - 1; t >= 1; --t) {
            cur = sbp[t * K + cur];
            out[t - 1] = cur;
        }
    }
}

__global__ void crf_mask_kernel(const float* __restrict__ trans, const float* __restrict__ mask, int n, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = trans[i] * mask[i] + (float)((int)(1.0f - mask[i]) * -10000);
}

// CRF.loss_sample_weights (polus/layers.py:116-121): w_b = any(y*m == 1) + all(y*m == 0) * negative_weight
__global__ void crf_sample_weights_kernel(const float* __restrict__ y, const float* __restrict__ maskpos, float negw,
                                          int T, int K, float* __restrict__ out) {
    const int b = blockIdx.x, lane = threadIdx.x;
    const float* yb = y + (long long)b * T * K;
    int any_one = 0, all_zero = 1;
    for (int i = lane; i < T * K; i += 32) {
        const float v = yb[i] * maskpos[i % K];
        any_one |= (v == 1.0f);
        all_zero &= (v == 0.0f);
    }
    any_one = __any_sync(0xffffffffu, any_one);
    all_zero = __all_sync(0xffffffffu, all_zero);
    if (lane == 0) out[b] = (any_one ? 1.0f : 0.0f) + (all_zero ? negw : 0.0f);
}

}  // namespace

extern "C" int polus_crf_sample_weights(const float* y_true, const float* mask_positive, float negative_weight, int B,
                                        int T, int K, float* out, void* stream) {
    if (B == 0) return 0;
    crf_sample_weights_kernel<<<B, 32, 0, (cudaStream_t)stream>>>(y_true, mask_positive, negative_weight, T, K, out);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

// Dynamic shared memory the wide kernels may use: the 227 KB a block can opt into, less their static arrays.
constexpr size_t kWideSmemMax = 220 * 1024;

extern "C" int polus_crf_nll(const float* emis, const int32_t* tags, const int32_t* lens, const float* trans,
                             const float* weights, int B, int T, int K, float* nll, float* loss, float* gemis,
                             float* gtrans, void* stream) {
    POLUS_REQUIRE(K >= 1 && K <= kWideMaxK, "polus_crf_nll: K must be in [1,%d] (got %d)", kWideMaxK, K);
    POLUS_REQUIRE(gemis != nullptr, "polus_crf_nll: gemis is required");
    POLUS_REQUIRE(T >= 1, "polus_crf_nll: T must be >= 1");
    const size_t smem = ((size_t)3 * K * K + (size_t)3 * T * K + 2 * (size_t)T) * sizeof(float);
    // crf_nll_kernel keeps its [T][K] tables in shared memory; everything else goes to crf_nll_wide_kernel
    const bool narrow = K <= 32 && smem <= 200 * 1024;
    const int wide_threads = cdiv(K, 32) * 32;
    const size_t wide_smem = ((size_t)wide_threads * (kWideMaxK + 1) + 2 * (size_t)T) * sizeof(float);
    POLUS_REQUIRE(narrow || wide_smem <= kWideSmemMax,
                  "polus_crf_nll: T = %d too long for the shared-memory tables at K = %d", T, K);
    if (B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (loss) POLUS_CHECK_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), st));
    // K = 4, the polus.ner tag set (PAD, O, B-, I-: polus/ner/utils.py:9-15): one sequence per lane, when its 16-byte row
    // loads are aligned and four sequences fit in shared memory (T <= 851); otherwise one tag per lane
    const bool lanes_ok = K == 4 && ((reinterpret_cast<uintptr_t>(emis) | reinterpret_cast<uintptr_t>(gemis)) & 15) == 0;
    auto lanes_smem = [&](int seq) { return ((size_t)48 + (size_t)3 * seq * (T * 4 + 4) + (size_t)3 * seq * (T + 1)) * sizeof(float); };
    if (lanes_ok && lanes_smem(4) <= 200 * 1024) {
        if (lanes_smem(8) <= 200 * 1024) {
            const size_t sz = lanes_smem(8);
            if (sz > 48 * 1024) POLUS_CHECK_CUDA(cudaFuncSetAttribute(crf_nll_lanes_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sz));
            crf_nll_lanes_kernel<8><<<cdiv(B, 8), 256, sz, st>>>(emis, tags, lens, trans, weights, B, T, nll, loss, gemis, gtrans);
        } else {
            const size_t sz = lanes_smem(4);
            if (sz > 48 * 1024) POLUS_CHECK_CUDA(cudaFuncSetAttribute(crf_nll_lanes_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sz));
            crf_nll_lanes_kernel<4><<<cdiv(B, 4), 256, sz, st>>>(emis, tags, lens, trans, weights, B, T, nll, loss, gemis, gtrans);
        }
    } else if (narrow) {
        if (smem > 48 * 1024) POLUS_CHECK_CUDA(cudaFuncSetAttribute(crf_nll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        crf_nll_kernel<<<B, 64, smem, st>>>(emis, tags, lens, trans, weights, B, T, K, nll, loss, gemis, gtrans);
    } else {
        if (wide_smem > 48 * 1024)
            POLUS_CHECK_CUDA(cudaFuncSetAttribute(crf_nll_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide_smem));
        crf_nll_wide_kernel<<<B, wide_threads, wide_smem, st>>>(emis, tags, lens, trans, weights, B, T, K, nll, loss, gemis, gtrans);
    }
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

extern "C" int polus_crf_decode(const float* emis, const int32_t* lens, const float* trans, int B, int T, int K,
                                int32_t* tags, float* score, void* stream) {
    POLUS_REQUIRE(K >= 1 && K <= kWideMaxK, "polus_crf_decode: K must be in [1,%d] (got %d)", kWideMaxK, K);
    POLUS_REQUIRE(T >= 1, "polus_crf_decode: T must be >= 1");
    const size_t smem = (size_t)K * K * sizeof(float) + (size_t)T * K;
    // crf_decode_kernel: K <= 32 with A and the back-pointers in shared memory; everything else: crf_decode_wide_kernel
    const bool narrow = K <= 32 && smem <= 200 * 1024;
    const size_t wide_smem = (size_t)T * K;
    POLUS_REQUIRE(narrow || wide_smem <= kWideSmemMax,
                  "polus_crf_decode: T = %d too long for the shared-memory back-pointer table at K = %d", T, K);
    if (B == 0) return 0;
    if (narrow) {
        if (smem > 48 * 1024) POLUS_CHECK_CUDA(cudaFuncSetAttribute(crf_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        crf_decode_kernel<<<B, 32, smem, (cudaStream_t)stream>>>(emis, lens, trans, T, K, tags, score);
    } else {
        if (wide_smem > 48 * 1024)
            POLUS_CHECK_CUDA(cudaFuncSetAttribute(crf_decode_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide_smem));
        crf_decode_wide_kernel<<<B, cdiv(K, 32) * 32, wide_smem, (cudaStream_t)stream>>>(emis, lens, trans, T, K, tags, score);
    }
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

extern "C" int polus_crf_mask_transitions(const float* trans, const float* mask, int K, float* out, void* stream) {
    crf_mask_kernel<<<cdiv(K * K, 128), 128, 0, (cudaStream_t)stream>>>(trans, mask, K * K, out);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}
