// Masked-language-model head (HF BertForMaskedLM / RobertaForMaskedLM, TF BERT's masked_lm_positions format):
//   polus_gather_positions / polus_scatter_positions_add  h[b, pos[b,j], :] <-> rows b*P + j
//   polus_vocab_xent   weighted cross-entropy over a vocabulary row, gradient written over the bf16 logits in place
//   polus_colsum_bf16  column sums of a strided bf16 matrix (the output-bias gradient)
#include "common.cuh"
#include <atomic>
#include <climits>
extern std::atomic<long long> g_launch_count;

namespace {

constexpr int kXentThreads = 512;  // one CTA per SM, one row at a time: 4 x 16 B in flight per thread
constexpr int kXentUnroll = 4;
constexpr int kScatterMaxP = 12288;  // the row's positions in the default 48 KB of shared memory

__device__ __forceinline__ int clamp_pos(int p, int S) { return p < 0 ? 0 : (p >= S ? S - 1 : p); }

// one warp per output row, 16-byte copies (H % 8 == 0)
__global__ void gather_positions_kernel(const bf16* __restrict__ h, const int32_t* __restrict__ pos, int B, int S, int H,
                                        int P, bf16* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= (long long)B * P) return;
    const int b = (int)(row / P);
    const int s = clamp_pos(pos[row], S);
    const bf16x8* src = reinterpret_cast<const bf16x8*>(h + ((long long)b * S + s) * H);
    bf16x8* dst = reinterpret_cast<bf16x8*>(out + row * H);
    for (int c = lane; c < H / 8; c += 32) dst[c] = src[c];
}

// grid (cdiv(H/8, 128), B), P ints of dynamic shared memory.  Thread = 8 columns of one batch row.  Slot j writes only
// when it is the first slot of row b naming its (clamped) position; it then sums every slot of that position in
// ascending j in fp32 and adds the total once: deterministic, and exact up to one bf16 rounding, however often a
// position repeats.  The row's clamped positions are staged in shared memory for the O(P^2) first-occurrence scans.
__global__ void scatter_positions_kernel(const bf16* __restrict__ g, const int32_t* __restrict__ pos, int S, int H, int P,
                                         bf16* __restrict__ dh) {
    extern __shared__ int prow[];
    const int b = blockIdx.y;
    for (int j = threadIdx.x; j < P; j += blockDim.x) prow[j] = clamp_pos(pos[(long long)b * P + j], S);
    __syncthreads();
    const int c8 = blockIdx.x * blockDim.x + threadIdx.x;
    if (c8 * 8 >= H) return;
    for (int j = 0; j < P; ++j) {
        const int s = prow[j];
        bool first = true;
        for (int k = 0; k < j && first; ++k) first = prow[k] != s;
        if (!first) continue;
        float acc[8];
        bf16x8* d = reinterpret_cast<bf16x8*>(dh + ((long long)b * S + s) * H) + c8;
        unpack8(*d, acc);
        for (int k = j; k < P; ++k) {
            if (prow[k] != s) continue;
            float v[8];
            unpack8(reinterpret_cast<const bf16x8*>(g + ((long long)b * P + k) * H)[c8], v);
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[e] += v[e];
        }
        *d = pack8(acc);
    }
}

// L2-allocating 16-byte load (the gradient pass re-reads the row from L2; .nc is not allowed: the row is rewritten)
__device__ __forceinline__ void ld_row8(const bf16* row, int c, int V, float* v) {
    if (c + 8 <= V) {
        bf16x8 q;
        uint32_t* u = reinterpret_cast<uint32_t*>(&q);
        asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]) : "l"(row + c));
        unpack8(q, v);
    } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = c + e < V ? __bfloat162float(row[c + e]) : -INFINITY;
    }
}

struct MaxSum {
    float m, s;
    int idx;  // column of the first occurrence of m
};

__device__ __forceinline__ MaxSum combine(MaxSum a, MaxSum b) {
    MaxSum r;
    r.m = fmaxf(a.m, b.m);
    r.s = (a.m == -INFINITY ? 0.f : a.s * __expf(a.m - r.m)) + (b.m == -INFINITY ? 0.f : b.s * __expf(b.m - r.m));
    r.idx = (a.m > b.m || (a.m == b.m && a.idx < b.idx)) ? a.idx : b.idx;
    return r;
}

__device__ float block_sum(float v, float* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    v = lane < (int)(blockDim.x >> 5) ? red[lane] : 0.f;
    return warp_sum(v);
}

// Persistent: CTA c takes rows c, c + gridDim.x, ...  Pass 1 streams the row once (online max / sum-of-exp / argmax);
// pass 2 re-reads it -- from L2, a wave of rows is one CTA per SM -- and overwrites it with the gradient
// w_r / sum(w) * (softmax - onehot(y_r)).  sum(w) is summed by every CTA in the same order, so all agree bit for bit.
__global__ void __launch_bounds__(kXentThreads, 1)
vocab_xent_kernel(bf16* __restrict__ logits, int R, int V, long long ldl, const int32_t* __restrict__ labels,
                  const float* __restrict__ weights, float* __restrict__ nll, int32_t* __restrict__ argmax) {
    __shared__ float red[32];
    __shared__ MaxSum redm[32];
    __shared__ float row_stat[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float wsum = 0.f;
    if (labels != nullptr) {
        float t = 0.f;
        for (int r = tid; r < R; r += kXentThreads) t += weights[r];
        wsum = block_sum(t, red);
    }
    for (int r = blockIdx.x; r < R; r += gridDim.x) {
        bf16* row = logits + (long long)r * ldl;
        MaxSum ms = {-INFINITY, 0.f, INT_MAX};
        for (int c0 = tid * 8; c0 < V; c0 += kXentThreads * 8 * kXentUnroll) {
            float v[kXentUnroll][8];
#pragma unroll
            for (int u = 0; u < kXentUnroll; ++u) {
                const int c = c0 + u * kXentThreads * 8;
                if (c < V) ld_row8(row, c, V, v[u]);
            }
#pragma unroll
            for (int u = 0; u < kXentUnroll; ++u) {
                const int c = c0 + u * kXentThreads * 8;
                if (c >= V) break;
                float m8 = v[u][0];
                int j8 = 0;
#pragma unroll
                for (int e = 1; e < 8; ++e)
                    if (v[u][e] > m8) { m8 = v[u][e]; j8 = e; }
                if (m8 > ms.m) {  // columns arrive in ascending order: strict > keeps the first occurrence
                    ms.s = ms.m == -INFINITY ? 0.f : ms.s * __expf(ms.m - m8);
                    ms.m = m8;
                    ms.idx = c + j8;
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) ms.s += __expf(v[u][e] - ms.m);  // padding lanes hold -inf: exp = 0
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            MaxSum other = {__shfl_xor_sync(0xffffffffu, ms.m, o), __shfl_xor_sync(0xffffffffu, ms.s, o),
                            __shfl_xor_sync(0xffffffffu, ms.idx, o)};
            ms = combine(ms, other);
        }
        __syncthreads();  // redm / row_stat of the previous row have been read
        if (lane == 0) redm[warp] = ms;
        __syncthreads();
        if (warp == 0) {
            ms = lane < kXentThreads / 32 ? redm[lane] : MaxSum{-INFINITY, 0.f, INT_MAX};
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                MaxSum other = {__shfl_xor_sync(0xffffffffu, ms.m, o), __shfl_xor_sync(0xffffffffu, ms.s, o),
                                __shfl_xor_sync(0xffffffffu, ms.idx, o)};
                ms = combine(ms, other);
            }
            if (lane == 0) {
                if (argmax != nullptr) argmax[r] = ms.idx;
                const float lse = ms.m + logf(ms.s);
                row_stat[0] = lse;
                if (labels != nullptr) {
                    int y = labels[r];
                    y = y < 0 ? 0 : (y >= V ? V - 1 : y);
                    const float nl = lse - __bfloat162float(row[y]);
                    if (nll != nullptr) nll[r] = nl;
                    row_stat[1] = wsum > 0.f ? weights[r] / wsum : 0.f;
                }
            }
        }
        __syncthreads();
        if (labels == nullptr) continue;
        const float lse = row_stat[0], scale = row_stat[1];
        int y = labels[r];
        y = y < 0 ? 0 : (y >= V ? V - 1 : y);
        for (int c0 = tid * 8; c0 < V; c0 += kXentThreads * 8 * kXentUnroll) {
            float v[kXentUnroll][8];
            if (scale != 0.f) {
#pragma unroll
                for (int u = 0; u < kXentUnroll; ++u) {
                    const int c = c0 + u * kXentThreads * 8;
                    if (c < V) ld_row8(row, c, V, v[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < kXentUnroll; ++u) {
                const int c = c0 + u * kXentThreads * 8;
                if (c >= V) break;
                float gv[8];
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    gv[e] = scale == 0.f ? 0.f : (__expf(v[u][e] - lse) - (c + e == y ? 1.f : 0.f)) * scale;
                if (c + 8 <= V) {
                    *reinterpret_cast<bf16x8*>(row + c) = pack8(gv);
                } else {
#pragma unroll
                    for (int e = 0; e < 8; ++e)
                        if (c + e < V) row[c + e] = __float2bfloat16_rn(gv[e]);
                }
            }
        }
    }
}

// loss = sum_r w_r nll_r / sum_r w_r (0 when every weight is 0), one CTA, fixed summation order
__global__ void __launch_bounds__(kXentThreads)
vocab_xent_loss_kernel(const float* __restrict__ nll, const float* __restrict__ weights, int R, float* __restrict__ loss) {
    __shared__ float red[32];
    float a = 0.f, w = 0.f;
    for (int r = threadIdx.x; r < R; r += kXentThreads) {
        a += weights[r] * nll[r];
        w += weights[r];
    }
    a = block_sum(a, red);
    w = block_sum(w, red);
    if (threadIdx.x == 0) *loss = w > 0.f ? a / w : 0.f;
}

constexpr int kColsumRowsPerSlab = 64;
constexpr int kColsumMaxSlabs = 128;

// grid (cdiv(N, 2048), slabs), CTA = 256 threads x 8 columns; one fp32 atomic per column per slab
__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const bf16* __restrict__ x, int R, int N, long long ld, int rows_per_slab, float* __restrict__ out) {
    const int c = (blockIdx.x * 256 + threadIdx.x) * 8;
    if (c >= N) return;
    const int r0 = blockIdx.y * rows_per_slab;
    const int r1 = min(R, r0 + rows_per_slab);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int r = r0; r < r1; ++r) {
        const bf16* p = x + (long long)r * ld + c;
        float v[8];
        if (c + 8 <= N) {
            unpack8(ld_stream8(p), v);
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = c + e < N ? __bfloat162float(p[e]) : 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] += v[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e)
        if (c + e < N) atomicAdd(out + c + e, acc[e]);
}

}  // namespace

extern "C" int polus_gather_positions(const polus_bf16_t* d_h, const int32_t* d_pos, int B, int S, int H, int P,
                                      polus_bf16_t* d_out, void* stream) {
    POLUS_REQUIRE(B >= 0 && P >= 0, "polus_gather_positions: B and P must be >= 0 (got %d, %d)", B, P);
    POLUS_REQUIRE(S >= 1, "polus_gather_positions: S must be >= 1 (got %d)", S);
    POLUS_REQUIRE(H >= 8 && H % 8 == 0, "polus_gather_positions: H must be a positive multiple of 8 (got %d)", H);
    if ((long long)B * P == 0) return 0;
    POLUS_REQUIRE(d_h && d_pos && d_out, "polus_gather_positions: NULL pointer");
    gather_positions_kernel<<<cdiv((long long)B * P, 8), 256, 0, (cudaStream_t)stream>>>(
        (const bf16*)d_h, d_pos, B, S, H, P, (bf16*)d_out);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

extern "C" int polus_scatter_positions_add(const polus_bf16_t* d_g, const int32_t* d_pos, int B, int S, int H, int P,
                                           polus_bf16_t* d_dh, void* stream) {
    POLUS_REQUIRE(B >= 0 && P >= 0, "polus_scatter_positions_add: B and P must be >= 0 (got %d, %d)", B, P);
    POLUS_REQUIRE(S >= 1, "polus_scatter_positions_add: S must be >= 1 (got %d)", S);
    POLUS_REQUIRE(H >= 8 && H % 8 == 0, "polus_scatter_positions_add: H must be a positive multiple of 8 (got %d)", H);
    POLUS_REQUIRE(P <= kScatterMaxP, "polus_scatter_positions_add: P must be <= %d (got %d)", kScatterMaxP, P);
    if ((long long)B * P == 0) return 0;
    POLUS_REQUIRE(d_g && d_pos && d_dh, "polus_scatter_positions_add: NULL pointer");
    scatter_positions_kernel<<<dim3(cdiv(H / 8, 128), B), 128, P * sizeof(int), (cudaStream_t)stream>>>(
        (const bf16*)d_g, d_pos, S, H, P, (bf16*)d_dh);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}

extern "C" int polus_vocab_xent(polus_bf16_t* d_logits, int R, int V, int64_t ldl, const int32_t* d_labels,
                                const float* d_weights, float* d_nll, int32_t* d_argmax, float* d_loss, void* stream) {
    POLUS_REQUIRE(R >= 0, "polus_vocab_xent: R must be >= 0 (got %d)", R);
    POLUS_REQUIRE(V >= 1, "polus_vocab_xent: V must be >= 1 (got %d)", V);
    POLUS_REQUIRE(ldl >= V && ldl % 8 == 0, "polus_vocab_xent: ldl must be >= V and a multiple of 8 (got %lld, V = %d)",
                  (long long)ldl, V);
    POLUS_REQUIRE(d_labels != nullptr || d_argmax != nullptr, "polus_vocab_xent: inference (labels NULL) needs d_argmax");
    POLUS_REQUIRE(d_labels == nullptr || d_weights != nullptr, "polus_vocab_xent: labels need weights");
    POLUS_REQUIRE(d_loss == nullptr || d_nll != nullptr, "polus_vocab_xent: the loss is reduced from d_nll");
    cudaStream_t st = (cudaStream_t)stream;
    if (R == 0) {
        if (d_loss) POLUS_CHECK_CUDA(cudaMemsetAsync(d_loss, 0, sizeof(float), st));
        return 0;
    }
    POLUS_REQUIRE(d_logits != nullptr && ((uintptr_t)d_logits & 15) == 0, "polus_vocab_xent: logits must be 16-byte aligned");
    const int grid = R < polus_num_sms() ? R : polus_num_sms();
    vocab_xent_kernel<<<grid, kXentThreads, 0, st>>>((bf16*)d_logits, R, V, (long long)ldl, d_labels, d_weights, d_nll, d_argmax);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    if (d_labels != nullptr && d_loss != nullptr) {
        vocab_xent_loss_kernel<<<1, kXentThreads, 0, st>>>(d_nll, d_weights, R, d_loss);
        g_launch_count++;
        POLUS_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int polus_colsum_bf16(const polus_bf16_t* d_x, int R, int N, int64_t ld, float* d_out, void* stream) {
    POLUS_REQUIRE(R >= 0 && N >= 1, "polus_colsum_bf16: need R >= 0 and N >= 1 (got %d, %d)", R, N);
    POLUS_REQUIRE(ld >= N && ld % 8 == 0, "polus_colsum_bf16: ld must be >= N and a multiple of 8 (got %lld, N = %d)",
                  (long long)ld, N);
    if (R == 0) return 0;
    POLUS_REQUIRE(d_x && d_out && ((uintptr_t)d_x & 15) == 0, "polus_colsum_bf16: NULL or unaligned pointer");
    int slabs = cdiv(R, kColsumRowsPerSlab);
    if (slabs > kColsumMaxSlabs) slabs = kColsumMaxSlabs;
    const int rows_per_slab = cdiv(R, slabs);
    slabs = cdiv(R, rows_per_slab);
    colsum_bf16_kernel<<<dim3(cdiv(N, 2048), slabs), 256, 0, (cudaStream_t)stream>>>((const bf16*)d_x, R, N, (long long)ld,
                                                                                      rows_per_slab, d_out);
    g_launch_count++;
    POLUS_LAUNCH_CHECK();
    return 0;
}
