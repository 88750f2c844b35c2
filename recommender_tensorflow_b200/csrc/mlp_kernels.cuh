// DNN tower (trainers/deep_fm.py:93-112), head (trainers/deep_fm.py:114-125) and dense optimizer
// kernels.  This file holds the exact-fp32 CUDA-core path: a register-tiled SGEMM with fused
// epilogues (bias+ReLU forward, ReLU-mask backward, FM-gradient add for the input layer) and
// deterministic split-K for the weight gradients.
#pragma once
#include "dfm_types.cuh"
#include "embed_kernels.cuh"

enum { EPI_NONE = 0, EPI_BIAS_RELU = 1, EPI_MASK = 2, EPI_DE = 3 };

// dropout mask of element idx of one layer at one step: keep ? 1/keep : 0   (counter-based, restated by the oracle)
__host__ __device__ __forceinline__ uint64_t dfm_mix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
__host__ __device__ __forceinline__ uint64_t dfm_drop_key(uint64_t seed, uint64_t step, uint64_t layer) {
    return dfm_mix64(dfm_mix64(seed) ^ (step * 64 + layer));
}
__device__ __forceinline__ float dfm_drop(uint64_t key, uint64_t idx, float keep, float inv_keep) {
    const float u = (float)(dfm_mix64(key ^ idx) >> 40) * (1.0f / 16777216.0f);
    return u < keep ? inv_keep : 0.f;
}

// params["activation"] of the reference (trainers/deep_fm.py:22,100).  Forward value and derivative expressed in the
// layer's OUTPUT y (that is what the backward pass has at hand); with dropout the stored output is y * mask / keep:
// a stored zero is a dropped unit (for tanh / identity also the measure-zero case of an exactly zero pre-activation).
__device__ __forceinline__ float act_fwd(int kind, float x) {
    switch (kind) {
        case 1: return tanhf(x);
        case 2: return 1.f / (1.f + expf(-x));
        case 3: return x;
        default: return fmaxf(x, 0.f);
    }
}
__device__ __forceinline__ float act_bwd(int kind, float y_stored, float g, float drop_scale /* 1 / keep, <= 0: no dropout */) {
    if (kind == 0) return y_stored > 0.f ? (drop_scale > 0.f ? g * drop_scale : g) : 0.f;
    float y = y_stored, sc = 1.f;
    if (drop_scale > 0.f) {
        if (y_stored == 0.f) return 0.f;
        y = y_stored / drop_scale; sc = drop_scale;
    }
    const float d = kind == 1 ? 1.f - y * y : kind == 2 ? y * (1.f - y) : 1.f;
    return g * sc * d;
}

struct EpiArgs {
    int      act_kind;   // DFM_ACT_* (0 = ReLU)
    float    drop_keep;  // EPI_BIAS_RELU: > 0 -> dropout after the activation (keep probability)
    float    drop_inv;   //                1 / keep
    uint64_t drop_key;
    int64_t  drop_row0;  // global index of row 0 (sample offset of this rank)
    float    bwd_scale;  // EPI_MASK: gradient scale of the dropout in front (1 / keep), 0 = none
    const float* bias;   // EPI_BIAS_RELU: [N]
    const float* act;    // EPI_MASK: forward activation [M, ld_act]; EPI_DE: h0 [M, ld_act]
    int          ld_act;
    const float* dz;     // EPI_DE: [M]
    const float* s;      // EPI_DE: [M, K] field sums (nullptr when use_mf == 0)
    int          K;      // EPI_DE: embedding size
};

// C[M,N] (+epilogue) = A(M,Kd) * B(Kd,N)
//   A_KC: A stored [M, lda] with k contiguous   (else stored [Kd, lda] with m contiguous)
//   B_KC: B stored [N, ldb] with k contiguous   (else stored [Kd, ldb] with n contiguous)
// blockIdx.z = split over Kd in chunks of k_chunk; split z writes C + z*c_split_stride.
// 128x128x16 tile, 256 threads, 8x8 outputs per thread (two 4-wide strips 64 apart in each dim).
template <bool A_KC, bool B_KC, int EPI, bool VEC>
__global__ void __launch_bounds__(256) sgemm_kernel(const float* __restrict__ A, int lda, const float* __restrict__ Bm,
                                                    int ldb, float* __restrict__ C, int ldc, int M, int N, int Kd,
                                                    int k_chunk, size_t c_split_stride, EpiArgs ep) {
    constexpr int BM = 128, BN = 128, BK = 16;
    __shared__ __align__(16) float As[BK][BM + 4];
    __shared__ __align__(16) float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int kbeg = blockIdx.z * k_chunk;
    const int kend = min(Kd, kbeg + k_chunk);
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    // loader geometry: 128x16 (or 16x128) tile = 512 float4, two per thread
    float4 ra[2], rb[2];
    auto load_a = [&](int k0) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            int q = tid + r * 256;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (A_KC) {  // 128 rows x 4 float4 along k
                int row = q >> 2, kc = (q & 3) * 4;
                int gm = m0 + row, gk = k0 + kc;
                if (gm < M) {
                    const float* p = A + (size_t)gm * lda + gk;
                    if (VEC && gk + 3 < kend) v = __ldg(reinterpret_cast<const float4*>(p));
                    else {
                        if (gk < kend) v.x = __ldg(p);
                        if (gk + 1 < kend) v.y = __ldg(p + 1);
                        if (gk + 2 < kend) v.z = __ldg(p + 2);
                        if (gk + 3 < kend) v.w = __ldg(p + 3);
                    }
                }
            } else {     // 16 k-rows x 32 float4 along m
                int kr = q >> 5, mc = (q & 31) * 4;
                int gk = k0 + kr, gm = m0 + mc;
                if (gk < kend) {
                    const float* p = A + (size_t)gk * lda + gm;
                    if (VEC && gm + 3 < M) v = __ldg(reinterpret_cast<const float4*>(p));
                    else {
                        if (gm < M) v.x = __ldg(p);
                        if (gm + 1 < M) v.y = __ldg(p + 1);
                        if (gm + 2 < M) v.z = __ldg(p + 2);
                        if (gm + 3 < M) v.w = __ldg(p + 3);
                    }
                }
            }
            ra[r] = v;
        }
    };
    auto load_b = [&](int k0) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            int q = tid + r * 256;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (B_KC) {
                int row = q >> 2, kc = (q & 3) * 4;
                int gn = n0 + row, gk = k0 + kc;
                if (gn < N) {
                    const float* p = Bm + (size_t)gn * ldb + gk;
                    if (VEC && gk + 3 < kend) v = __ldg(reinterpret_cast<const float4*>(p));
                    else {
                        if (gk < kend) v.x = __ldg(p);
                        if (gk + 1 < kend) v.y = __ldg(p + 1);
                        if (gk + 2 < kend) v.z = __ldg(p + 2);
                        if (gk + 3 < kend) v.w = __ldg(p + 3);
                    }
                }
            } else {
                int kr = q >> 5, nc = (q & 31) * 4;
                int gk = k0 + kr, gn = n0 + nc;
                if (gk < kend) {
                    const float* p = Bm + (size_t)gk * ldb + gn;
                    if (VEC && gn + 3 < N) v = __ldg(reinterpret_cast<const float4*>(p));
                    else {
                        if (gn < N) v.x = __ldg(p);
                        if (gn + 1 < N) v.y = __ldg(p + 1);
                        if (gn + 2 < N) v.z = __ldg(p + 2);
                        if (gn + 3 < N) v.w = __ldg(p + 3);
                    }
                }
            }
            rb[r] = v;
        }
    };
    auto store_ab = [&]() {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            int q = tid + r * 256;
            if (A_KC) {
                int row = q >> 2, kc = (q & 3) * 4;
                As[kc][row] = ra[r].x; As[kc + 1][row] = ra[r].y; As[kc + 2][row] = ra[r].z; As[kc + 3][row] = ra[r].w;
            } else {
                int kr = q >> 5, mc = (q & 31) * 4;
                *reinterpret_cast<float4*>(&As[kr][mc]) = ra[r];
            }
            if (B_KC) {
                int row = q >> 2, kc = (q & 3) * 4;
                Bs[kc][row] = rb[r].x; Bs[kc + 1][row] = rb[r].y; Bs[kc + 2][row] = rb[r].z; Bs[kc + 3][row] = rb[r].w;
            } else {
                int kr = q >> 5, nc = (q & 31) * 4;
                *reinterpret_cast<float4*>(&Bs[kr][nc]) = rb[r];
            }
        }
    };

    if (kbeg < kend) {
        load_a(kbeg);
        load_b(kbeg);
    }
    for (int k0 = kbeg; k0 < kend; k0 += BK) {
        store_ab();
        __syncthreads();
        if (k0 + BK < kend) {
            load_a(k0 + BK);
            load_b(k0 + BK);
        }
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            float4 a1 = *reinterpret_cast<const float4*>(&As[kk][64 + ty * 4]);
            float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
            float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }

    float* Cz = C + (size_t)blockIdx.z * c_split_stride;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        int gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (gm >= M) continue;
        float dzm = 0.f;
        if (EPI == EPI_DE) dzm = ep.dz[gm];
#pragma unroll
        for (int jh = 0; jh < 2; ++jh) {
            int gn = n0 + jh * 64 + tx * 4;
            float v[4] = {acc[i][jh * 4 + 0], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                int n = gn + c;
                if (n >= N) continue;
                float x = v[c];
                if (EPI == EPI_BIAS_RELU) {
                    x = act_fwd(ep.act_kind, x + ep.bias[n]);
                    if (ep.drop_keep > 0.f) x *= dfm_drop(ep.drop_key, (uint64_t)(ep.drop_row0 + gm) * N + n, ep.drop_keep, ep.drop_inv);
                } else if (EPI == EPI_MASK) x = act_bwd(ep.act_kind, ep.act[(size_t)gm * ep.ld_act + n], x, ep.bwd_scale);
                else if (EPI == EPI_DE) {
                    if (ep.s) x += dzm * (ep.s[(size_t)gm * ep.K + (n % ep.K)] - ep.act[(size_t)gm * ep.ld_act + n]);
                }
                v[c] = x;
            }
            float* cp = Cz + (size_t)gm * ldc + gn;
            if (VEC && gn + 3 < N) *reinterpret_cast<float4*>(cp) = make_float4(v[0], v[1], v[2], v[3]);
            else {
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (gn + c < N) cp[c] = v[c];
            }
        }
    }
}

// out[i] = sum_z partial[z*stride + i]   (fixed order -> deterministic split-K)
static __global__ void reduce_partials_kernel(const float* __restrict__ partial, int nz, size_t stride, int64_t count,
                                       float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    float s = 0.f;
    for (int z = 0; z < nz; ++z) s += partial[(size_t)z * stride + i];
    out[i] = s;
}

// weighted column sums: part[chunk][j] = sum_{b in chunk} w[b] * X[b*ldx + j]   (w == nullptr -> 1)
// block = 32 columns x 8 row phases; rows of a chunk are walked in a fixed order.
static __global__ void __launch_bounds__(256) colsum_partial_kernel(const float* __restrict__ X, int ldx, const float* __restrict__ w,
                                                             int B, int N, int rows_per_chunk, float* __restrict__ part) {
    __shared__ float sm[8][33];
    const int col = blockIdx.x * 32 + (threadIdx.x & 31);
    const int ph = threadIdx.x >> 5;
    const int r0 = blockIdx.y * rows_per_chunk;
    const int r1 = min(B, r0 + rows_per_chunk);
    float s = 0.f;
    if (col < N)
        for (int r = r0 + ph; r < r1; r += 8) s += (w ? w[r] : 1.f) * X[(size_t)r * ldx + col];
    sm[ph][threadIdx.x & 31] = s;
    __syncthreads();
    if (ph == 0 && col < N) {
        float t = 0.f;
#pragma unroll
        for (int p = 0; p < 8; ++p) t += sm[p][threadIdx.x & 31];
        part[(size_t)blockIdx.y * N + col] = t;
    }
}

// numeric-feature gradients (trainers/deep_fm.py:62-67 backward):
//   g_num_emb[j, c] = sum_b x[b,j] * dE[b, (dc+j)*K + c]      g_num_lin[j] = sum_b x[b,j] * dz[b]
// part layout per chunk: [dn*K] then [dn].  One CTA per chunk of rows: the x columns of the chunk are staged in
// shared memory, thread t owns output t and walks the rows in order (deterministic); the numeric part of a dE row
// is contiguous, so the dn*K threads read it coalesced.
static __global__ void __launch_bounds__(256) numeric_grad_partial_kernel(BatchPtrs bp, const float* __restrict__ dE, int dK, int dc, int dn,
                                                                   int K, const float* __restrict__ dz, int B, int rows_per_chunk,
                                                                   float* __restrict__ part) {
    extern __shared__ float xs[];           // [rows_per_chunk][dn + 1]: x columns, then dz
    const int total = dn * K + dn;
    const int r0 = blockIdx.x * rows_per_chunk;
    const int nr = min(B, r0 + rows_per_chunk) - r0;
    const int ldx = dn + 1;
    for (int q = threadIdx.x; q < nr * ldx; q += blockDim.x) {
        int j = q / nr, r = q - j * nr;      // column-major walk: coalesced reads of each x column
        xs[r * ldx + j] = j < dn ? bp.num[j][r0 + r] : dz[r0 + r];
    }
    __syncthreads();
    for (int o = threadIdx.x; o < total; o += blockDim.x) {
        float s = 0.f;
        if (o < dn * K) {
            const int j = o / K;
            if (dE) {
                const float* p = dE + (size_t)r0 * dK + (size_t)dc * K + o;
#pragma unroll 16
                for (int r = 0; r < nr; ++r) s = fmaf(xs[r * ldx + j], __ldg(p + (size_t)r * dK), s);
            }
        } else {
            const int j = o - dn * K;
            for (int r = 0; r < nr; ++r) s = fmaf(xs[r * ldx + j], xs[r * ldx + dn], s);
        }
        part[(size_t)blockIdx.x * total + o] = s;
    }
}

// head: z = zacc + h_L . Wo + bo ; loss_b = max(z,0) - z*y + log1p(exp(-|z|)) ; dz = (sigmoid(z)-y)*scale
// one warp per sample; per-block partial sums of loss and dz (fixed order inside the block).
// WGT: weighted model, loss_b *= w_b and dz = ((sigmoid(z)-y)*scale)*w_b (w = 1 gives the unweighted bits)
// SQ: squared head, loss_b = (y - z)^2 and dz = 2 (z - y) * scale (sq_head), then the weight
template <bool SQ, bool WGT>
__global__ void __launch_bounds__(256) head_kernel(const float* __restrict__ zacc, const float* __restrict__ hL, int H,
                                                   const float* __restrict__ Wo, const float* __restrict__ bo,
                                                   const float* __restrict__ labels, const float* __restrict__ weights, int B, float scale,
                                                   float* __restrict__ logits, float* __restrict__ logits_out,
                                                   float* __restrict__ dz, float* __restrict__ part /*[grid][2]*/) {
    __shared__ float sl[8], sd[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float lsum = 0.f, dsum = 0.f;
    for (int b = blockIdx.x * 8 + warp; b < B; b += gridDim.x * 8) {
        float z = 0.f;
        if (hL) {
            const float* h = hL + (size_t)b * H;
            for (int j = lane; j < H; j += 32) z += h[j] * __ldg(Wo + j);
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) z += __shfl_xor_sync(0xffffffffu, z, o);
            z += bo[0];
        }
        z += zacc ? zacc[b] : 0.f;
        if (lane == 0) {
            logits[b] = z;
            if (logits_out) logits_out[b] = z;
            if (labels) {
                float y = labels[b];
                float l, g;
                if constexpr (SQ) {
                    sq_head(z, y, scale, l, g);
                } else {
                    l = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
                    float sg = 1.f / (1.f + expf(-z));
                    g = (sg - y) * scale;
                }
                if constexpr (WGT) { const float w = weights[b]; g *= w; l *= w; }
                dz[b] = g;
                lsum += l;
                dsum += g;
            }
        }
    }
    if (lane == 0) { sl[warp] = lsum; sd[warp] = dsum; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, c = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) { a += sl[w]; c += sd[w]; }
        part[blockIdx.x * 2] = a;
        part[blockIdx.x * 2 + 1] = c;
    }
}

// Fused head + top of the backward pass for towers whose last hidden layer is H = 32*NH wide (NH <= 8):
// per sample (one warp): z = zacc + h_L . Wo + bo, loss, dz, and immediately dh_L' = dz * Wo * relu'(h_L)
// while h_L is still in registers; per-block partial sums (fixed order) of the loss, dz,
// gWo = h_L^T dz and gb_L = column sums of dh_L'.  Replaces head_kernel + dh_last_kernel + two column-sum
// launches (and one re-read of h_L).   gpart layout: [grid][2*H] = {gWo | gb_L}
// WGT / SQ: as head_kernel
template <int NH, bool SQ, bool WGT>
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ zacc, const float* __restrict__ hL,
                                                       const float* __restrict__ Wo, const float* __restrict__ bo,
                                                       const float* __restrict__ labels, const float* __restrict__ weights, int B, float scale,
                                                       float* __restrict__ logits, float* __restrict__ logits_out,
                                                       float* __restrict__ dz, float* __restrict__ dh,
                                                       float* __restrict__ part /*[grid][2]*/, float* __restrict__ gpart,
                                                       float drop_scale /* 1/keep of the dropout after h_L, or 1 */) {
    constexpr int H = 32 * NH;
    __shared__ float sl[8], sd[8];
    __shared__ float sg[8][2 * H];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float wo[NH], gw[NH], gb[NH];
#pragma unroll
    for (int i = 0; i < NH; ++i) { wo[i] = __ldg(Wo + lane + 32 * i); gw[i] = 0.f; gb[i] = 0.f; }
    const float b0 = bo[0];
    float lsum = 0.f, dsum = 0.f;
    // two samples per warp trip (their loads are independent): the loop is a load -> reduce -> exp -> store chain and
    // was latency-bound at one sample in flight per warp
    const int stride = gridDim.x * 8;
    for (int b = blockIdx.x * 8 + warp; b < B; b += 2 * stride) {
        const int b2 = b + stride;
        const bool two = b2 < B;
        float h[2][NH];
        float z[2] = {0.f, 0.f};
#pragma unroll
        for (int i = 0; i < NH; ++i) {
            h[0][i] = hL[(size_t)b * H + lane + 32 * i];
            h[1][i] = two ? hL[(size_t)b2 * H + lane + 32 * i] : 0.f;
        }
        const float za0 = zacc ? zacc[b] : 0.f, za1 = (zacc && two) ? zacc[b2] : 0.f;
        const float y0 = labels[b], y1 = two ? labels[b2] : 0.f;
        float w0 = 1.f, w1 = 1.f;
        if constexpr (WGT) { w0 = weights[b]; w1 = two ? weights[b2] : 0.f; }
#pragma unroll
        for (int i = 0; i < NH; ++i) { z[0] = fmaf(h[0][i], wo[i], z[0]); z[1] = fmaf(h[1][i], wo[i], z[1]); }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) { z[0] += __shfl_xor_sync(0xffffffffu, z[0], o); z[1] += __shfl_xor_sync(0xffffffffu, z[1], o); }
#pragma unroll
        for (int s2 = 0; s2 < 2; ++s2) {
            if (s2 == 1 && !two) break;
            const int bb = s2 ? b2 : b;
            const float zz = z[s2] + b0 + (s2 ? za1 : za0);
            const float y = s2 ? y1 : y0;
            float g, lsq = 0.f;
            if constexpr (SQ) sq_head(zz, y, scale, lsq, g);
            else g = (1.f / (1.f + expf(-zz)) - y) * scale;
            if constexpr (WGT) g *= s2 ? w1 : w0;
            if (lane == 0) {
                logits[bb] = zz;
                if (logits_out) logits_out[bb] = zz;
                dz[bb] = g;
                float l = SQ ? lsq : fmaxf(zz, 0.f) - zz * y + log1pf(expf(-fabsf(zz)));
                if constexpr (WGT) l *= s2 ? w1 : w0;
                lsum += l;
                dsum += g;
            }
#pragma unroll
            for (int i = 0; i < NH; ++i) {
                const float d = h[s2][i] > 0.f ? g * wo[i] * drop_scale : 0.f;
                dh[(size_t)bb * H + lane + 32 * i] = d;
                gw[i] = fmaf(h[s2][i], g, gw[i]);
                gb[i] += d;
            }
        }
    }
    if (lane == 0) { sl[warp] = lsum; sd[warp] = dsum; }
#pragma unroll
    for (int i = 0; i < NH; ++i) { sg[warp][lane + 32 * i] = gw[i]; sg[warp][H + lane + 32 * i] = gb[i]; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, c = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) { a += sl[w]; c += sd[w]; }
        part[blockIdx.x * 2] = a;
        part[blockIdx.x * 2 + 1] = c;
    }
    for (int j = threadIdx.x; j < 2 * H; j += 256) {
        float a = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) a += sg[w][j];
        gpart[(size_t)blockIdx.x * 2 * H + j] = a;
    }
}

// loss = (sum of block partials) * loss_scale ; dzsum = sum of dz  (single thread block, fixed order)
// o1..o3: further destinations (caller's loss buffer, gradients of the output bias and of the linear bias = sum of dz):
// written here instead of by three 4-byte device-to-device copies on the critical path of the step
static __global__ void head_final_kernel(const float* __restrict__ part, int nblocks, float loss_scale, float* __restrict__ loss_out,
                                  float* __restrict__ dzsum_out, float* __restrict__ loss_copy, float* __restrict__ dz_copy1,
                                  float* __restrict__ dz_copy2) {
    __shared__ float sa[256], sc[256];
    float a = 0.f, c = 0.f;
    for (int i = threadIdx.x; i < nblocks; i += 256) { a += part[i * 2]; c += part[i * 2 + 1]; }
    sa[threadIdx.x] = a; sc[threadIdx.x] = c;
    __syncthreads();
    for (int o = 128; o >= 1; o >>= 1) {
        if (threadIdx.x < o) { sa[threadIdx.x] += sa[threadIdx.x + o]; sc[threadIdx.x] += sc[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (loss_out) *loss_out = sa[0] * loss_scale;
        *dzsum_out = sc[0];
        if (loss_copy) *loss_copy = sa[0] * loss_scale;
        if (dz_copy1) *dz_copy1 = sc[0];
        if (dz_copy2) *dz_copy2 = sc[0];
    }
}

// dh_L'[b,j] = dz[b] * Wo[j] * (h_L[b,j] > 0)
static __global__ void dh_last_kernel(const float* __restrict__ hL, const float* __restrict__ Wo, const float* __restrict__ dz,
                               int64_t total, int H, float* __restrict__ dh, float drop_scale, int act_kind = 0) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) {
        int64_t b = i / H;
        int j = (int)(i - b * H);
        // hL == nullptr: no activation in front (hidden_units == []); drop_scale == 1: no dropout
        dh[i] = !hL ? dz[b] * Wo[j] : act_bwd(act_kind, hL[i], dz[b] * Wo[j], drop_scale != 1.f ? drop_scale : (act_kind ? 0.f : 1.f));
    }
}

// dense optimizer apply over the packed dense-parameter buffer.  Elements [0, n_deep) use the deep
// optimizer, [n_deep, n) the linear one (num_lin, bias).
static __global__ void dense_apply_kernel(float* __restrict__ w, float* __restrict__ s1, float* __restrict__ s2,
                                   const float* __restrict__ g, int64_t n_deep, int64_t n, OptDev od, OptDev ol) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float ww = w[i], a = s1[i], b = s2[i];
    if (i < n_deep) dense_apply(ww, a, b, g[i], od);
    else dense_apply(ww, a, b, g[i], ol);
    w[i] = ww; s1[i] = a; s2[i] = b;
}

// counter-based generator for dfm_init_random (own generator; TF's Philox streams are not reproducible)
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
__device__ __forceinline__ float u01(uint64_t h) { return ((h >> 40) + 0.5f) * (1.0f / 16777216.0f); }

// truncated normal(0, sigma) cut at 2 sigma (rejection on a counter stream), strided destination
// (row_mul, row_add): the stream is keyed on the GLOBAL row g = local * row_mul + row_add, so a row-sharded model
// initialised with seed S holds exactly the rows of the unsharded model initialised with seed S
static __global__ void init_trunc_normal_kernel(float* __restrict__ dst, uint64_t rows, int K, int row_stride, float sigma, uint64_t seed,
                                         uint64_t row_mul, uint64_t row_add) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * (uint64_t)K) return;
    uint64_t r = i / K;
    int c = (int)(i % K);
    const uint64_t gi = (r * row_mul + row_add) * (uint64_t)K + c;
    float z = 0.f;
    for (uint64_t att = 0; att < 64; ++att) {
        uint64_t h1 = splitmix64(seed ^ (gi * 64 + att) * 2);
        uint64_t h2 = splitmix64(seed ^ ((gi * 64 + att) * 2 + 1));
        z = sqrtf(-2.f * logf(u01(h1))) * cospif(2.f * u01(h2));
        if (fabsf(z) <= 2.f) break;
        z = 0.f;
    }
    dst[r * (uint64_t)row_stride + c] = z * sigma;
}
static __global__ void init_uniform_kernel(float* __restrict__ dst, int64_t n, float lim, uint64_t seed) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (2.f * u01(splitmix64(seed ^ (uint64_t)i)) - 1.f) * lim;
}
static __global__ void fill_strided_kernel(float* __restrict__ dst, uint64_t rows, int width, int row_stride, float val) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < rows * (uint64_t)width) dst[(i / width) * (uint64_t)row_stride + (i % width)] = val;
}
