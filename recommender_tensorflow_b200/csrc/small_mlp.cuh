// Fused small-MLP tower (trainers/deep_fm.py:93-112 with the reference default hidden_units
// [16,16] and friends): when every hidden layer is <= 32 wide the tower is ~10 kFLOP/sample and
// not a real GEMM, so it runs on CUDA cores with the weights resident in shared memory
// (BASELINE.json north_star: "tensor cores only when hidden_units make it a real GEMM").
//
//   small_mlp_fwd_bwd_top_kernel   one CTA = 128 samples per tile (persistent over tiles):
//        h1 = relu(h0 W0 + b0) ... z = zacc + h_L Wo + bo, sigmoid-CE loss, dz, then the backward
//        pass through every layer ABOVE the input layer, all without leaving the SM.  Emits
//        logits, dz, dh1' [B,H1] and per-CTA partial gradients of b0, W1, b1, ..., Wo, bo.
//   small_mlp_bwd_input_kernel     grid (sample tiles, 64-column chunks of the input layer):
//        dE = dh1' W0^T + dz (s - E)   and the per-tile partial of   dW0 = h0^T dh1'.
// Partials are reduced in a fixed order afterwards (deterministic).
#pragma once
#include "dfm_types.cuh"
#include "mlp_kernels.cuh"

constexpr int SM_TB = 128;        // samples per tile
constexpr int SM_DC = 32;         // input-layer columns per staged chunk (forward)
constexpr int SM_BC = 64;         // input-layer columns per CTA (backward)
constexpr int SM_MAXH = 32;
constexpr int SM_MAXL = 4;

struct SmallMlpDesc {
    int L;                        // hidden layers (1..SM_MAXL)
    int H[SM_MAXL];               // widths
    int D;                        // input width d*K
    int off_W[SM_MAXL], off_b[SM_MAXL], off_Wo, off_bo;   // offsets in the packed dense buffer
    int up_begin, up_count;       // [b0 .. bo] range (everything above W0) in the packed buffer
    int act_stride;               // floats per sample row in the per-sample scratch (odd)
    float drop_keep, drop_inv;    // dropout after every hidden layer (keep probability, 1/keep); keep == 0 -> off
    uint64_t drop_seed, drop_step;
    int64_t drop_row0;
};

static inline size_t small_mlp_fwd_smem(const SmallMlpDesc& m) {
    size_t f = (size_t)m.D * m.H[0] + 2 * (size_t)m.up_count + (size_t)SM_TB * (SM_DC + 1) + 2 * (size_t)SM_TB * m.act_stride +
               2 * SM_TB + 64;
    return f * sizeof(float);
}

// per-sample scratch row layout: [h_1 | h_2 | ... | h_L]; gradients use a second array of the same shape
// WGT: weighted model, the loss term and dz of sample b are multiplied by weights[b] (after the scale: w = 1 is exact)
// SQ: squared head (sq_head) instead of the sigmoid cross-entropy
template <int H1, bool SQ, bool WGT>
__global__ void __launch_bounds__(256, 2) small_mlp_fwd_bwd_top_kernel(
    SmallMlpDesc m, const float* __restrict__ dw, const float* __restrict__ h0, const float* __restrict__ zacc,
    const float* __restrict__ labels, const float* __restrict__ weights, int B, float scale, int train, float* __restrict__ logits,
    float* __restrict__ logits_out, float* __restrict__ dz_out, float* __restrict__ dh1_out,
    float* __restrict__ up_partial /*[grid][up_count]*/, float* __restrict__ head_part /*[grid][2]*/) {
    extern __shared__ __align__(16) float smem[];
    float* W0s = smem;                                   // [D][H1]
    float* ups = W0s + (size_t)m.D * H1;                 // packed params above W0
    float* gup = ups + m.up_count;                       // per-CTA gradient accumulators (same layout)
    float* hs = gup + m.up_count;                        // [SM_TB][SM_DC+1] staged input chunk
    float* acts = hs + SM_TB * (SM_DC + 1);              // [SM_TB][act_stride]
    float* dacts = acts + SM_TB * m.act_stride;          // [SM_TB][act_stride]
    float* dzs = dacts + SM_TB * m.act_stride;           // [SM_TB]
    float* red = dzs + SM_TB;                            // [SM_TB] loss terms
    const int tid = threadIdx.x;
    const int D = m.D;
    for (int i = tid; i < D * H1; i += 256) W0s[i] = dw[m.off_W[0] + i];
    for (int i = tid; i < m.up_count; i += 256) { ups[i] = dw[m.up_begin + i]; gup[i] = 0.f; }
    __syncthreads();
    auto UP = [&](int packed_off) { return ups + (packed_off - m.up_begin); };
    auto GUP = [&](int packed_off) { return gup + (packed_off - m.up_begin); };
    const int s = tid & (SM_TB - 1), half = tid >> 7;
    constexpr int HJ = H1 / 2;
    const int j0 = half * HJ;
    float loss_acc = 0.f, dz_acc = 0.f;
    const int ntiles = (B + SM_TB - 1) / SM_TB;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int b0 = tile * SM_TB;
        const int b = b0 + s;
        // ---- layer 0: h1 = relu(h0 W0 + b0), input staged chunk by chunk (coalesced)
        float acc[HJ];
#pragma unroll
        for (int j = 0; j < HJ; ++j) acc[j] = 0.f;
        // chunk c+1 is fetched into registers while chunk c is being multiplied (hides the global latency)
        constexpr int NPF = SM_TB * (SM_DC / 4) / 256;
        float4 pf[NPF];
        auto fetch = [&](int c0) {
#pragma unroll
            for (int u = 0; u < NPF; ++u) {
                int q = tid + u * 256;
                int r = q / (SM_DC / 4), cc = (q % (SM_DC / 4)) * 4;
                pf[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (b0 + r < B && c0 + cc < D) pf[u] = __ldg(reinterpret_cast<const float4*>(h0 + (size_t)(b0 + r) * D + c0 + cc));
            }
        };
        fetch(0);
        for (int c0 = 0; c0 < D; c0 += SM_DC) {
            __syncthreads();
#pragma unroll
            for (int u = 0; u < NPF; ++u) {
                int q = tid + u * 256;
                int r = q / (SM_DC / 4), cc = (q % (SM_DC / 4)) * 4;
                float* d = hs + r * (SM_DC + 1) + cc;
                d[0] = pf[u].x; d[1] = pf[u].y; d[2] = pf[u].z; d[3] = pf[u].w;
            }
            __syncthreads();
            if (c0 + SM_DC < D) fetch(c0 + SM_DC);
            const int cmax = min(SM_DC, D - c0);
            const float* hrow = hs + s * (SM_DC + 1);
#pragma unroll 4
            for (int c = 0; c < cmax; ++c) {
                float a = hrow[c];
                const float4* w = reinterpret_cast<const float4*>(W0s + (size_t)(c0 + c) * H1 + j0);
#pragma unroll
                for (int j4 = 0; j4 < HJ / 4; ++j4) {
                    float4 ww = w[j4];
                    acc[j4 * 4 + 0] = fmaf(a, ww.x, acc[j4 * 4 + 0]);
                    acc[j4 * 4 + 1] = fmaf(a, ww.y, acc[j4 * 4 + 1]);
                    acc[j4 * 4 + 2] = fmaf(a, ww.z, acc[j4 * 4 + 2]);
                    acc[j4 * 4 + 3] = fmaf(a, ww.w, acc[j4 * 4 + 3]);
                }
            }
        }
        float* arow = acts + s * m.act_stride;
        float* drow = dacts + s * m.act_stride;
        {
            const float* bb = UP(m.off_b[0]);
#pragma unroll
            for (int j = 0; j < HJ; ++j) arow[j0 + j] = fmaxf(acc[j] + bb[j0 + j], 0.f);
            if (train && m.drop_keep > 0.f) {
                const uint64_t key = dfm_drop_key(m.drop_seed, m.drop_step, 0);
#pragma unroll
                for (int j = 0; j < HJ; ++j)
                    arow[j0 + j] *= dfm_drop(key, (uint64_t)(m.drop_row0 + b) * H1 + j0 + j, m.drop_keep, m.drop_inv);
            }
        }
        __syncthreads();
        // ---- upper layers, head and their backward: one thread per sample
        if (half == 0) {
            int aoff = 0;
            for (int l = 1; l < m.L; ++l) {
                const int Hin = m.H[l - 1], Hout = m.H[l];
                const float* W = UP(m.off_W[l]);
                const float* bb = UP(m.off_b[l]);
                for (int o = 0; o < Hout; ++o) {
                    float a = bb[o];
                    for (int j = 0; j < Hin; ++j) a = fmaf(arow[aoff + j], W[j * Hout + o], a);
                    a = fmaxf(a, 0.f);
                    if (train && m.drop_keep > 0.f)
                        a *= dfm_drop(dfm_drop_key(m.drop_seed, m.drop_step, l), (uint64_t)(m.drop_row0 + b) * Hout + o, m.drop_keep, m.drop_inv);
                    arow[aoff + Hin + o] = a;
                }
                aoff += Hin;
            }
            const int HL = m.H[m.L - 1];
            const float* Wo = UP(m.off_Wo);
            float z = UP(m.off_bo)[0];
            for (int j = 0; j < HL; ++j) z = fmaf(arow[aoff + j], Wo[j], z);
            if (zacc && b < B) z += zacc[b];
            float g = 0.f, lterm = 0.f;
            if (b < B) {
                logits[b] = z;
                if (logits_out) logits_out[b] = z;
                if (train) {
                    float y = labels[b];
                    if constexpr (SQ) {
                        sq_head(z, y, scale, lterm, g);
                    } else {
                        lterm = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
                        g = (1.f / (1.f + expf(-z)) - y) * scale;
                    }
                    if constexpr (WGT) { const float w = weights[b]; g *= w; lterm *= w; }
                    dz_out[b] = g;
                }
            }
            dzs[s] = g;
            red[s] = lterm;
            if (train) {
                // dh_L' = dz * Wo * relu'(h_L); walk down to dh_1'
                const float dsc = m.drop_keep > 0.f ? m.drop_inv : 1.f;   // gradient through the dropout after each ReLU
                for (int j = 0; j < HL; ++j) drow[aoff + j] = arow[aoff + j] > 0.f ? g * Wo[j] * dsc : 0.f;
                for (int l = m.L - 1; l >= 1; --l) {
                    const int Hin = m.H[l - 1], Hout = m.H[l];
                    const float* W = UP(m.off_W[l]);
                    const int in_off = aoff - Hin;
                    for (int j = 0; j < Hin; ++j) {
                        float a = 0.f;
                        for (int o = 0; o < Hout; ++o) a = fmaf(drow[aoff + o], W[j * Hout + o], a);
                        drow[in_off + j] = arow[in_off + j] > 0.f ? a * dsc : 0.f;
                    }
                    aoff = in_off;
                }
                if (b < B) {
                    float4* dst = reinterpret_cast<float4*>(dh1_out + (size_t)b * H1);
#pragma unroll
                    for (int j4 = 0; j4 < H1 / 4; ++j4) dst[j4] = make_float4(drow[j4 * 4], drow[j4 * 4 + 1], drow[j4 * 4 + 2], drow[j4 * 4 + 3]);
                }
            }
        }
        __syncthreads();
        if (train) {
            // ---- per-CTA gradient accumulation for everything above W0 (each output owned by one thread,
            //      samples walked in order -> deterministic)
            int aoff = 0;
            for (int l = 0; l < m.L; ++l) {
                const int Hl = m.H[l];
                // bias l: sum_s dact_l[s][j]
                for (int j = tid; j < Hl; j += 256) {
                    float a = 0.f;
                    for (int r = 0; r < SM_TB; ++r) a += dacts[r * m.act_stride + aoff + j];
                    GUP(m.off_b[l])[j] += a;
                }
                if (l + 1 < m.L) {
                    const int Hn = m.H[l + 1];
                    for (int q = tid; q < Hl * Hn; q += 256) {
                        int j = q / Hn, o = q % Hn;
                        float a = 0.f;
                        for (int r = 0; r < SM_TB; ++r) a = fmaf(acts[r * m.act_stride + aoff + j], dacts[r * m.act_stride + aoff + Hl + o], a);
                        GUP(m.off_W[l + 1])[q] += a;
                    }
                } else {
                    for (int j = tid; j < Hl; j += 256) {
                        float a = 0.f;
                        for (int r = 0; r < SM_TB; ++r) a = fmaf(acts[r * m.act_stride + aoff + j], dzs[r], a);
                        GUP(m.off_Wo)[j] += a;
                    }
                }
                aoff += Hl;
            }
            if (tid == 0) {
                float a = 0.f, c = 0.f;
                for (int r = 0; r < SM_TB; ++r) { a += red[r]; c += dzs[r]; }
                loss_acc += a;
                dz_acc += c;
            }
        }
        __syncthreads();
        // zero the rows for the next tile's out-of-range samples is unnecessary: g = 0 and h = relu(b) only
        // enter sums through dacts (0 when g == 0) and acts * dacts / acts * dzs (0 as well).
    }
    if (train) {
        __syncthreads();
        if (tid == 0) GUP(m.off_bo)[0] = dz_acc;
        __syncthreads();
        for (int i = tid; i < m.up_count; i += 256) up_partial[(size_t)blockIdx.x * m.up_count + i] = gup[i];
        if (tid == 0) { head_part[blockIdx.x * 2] = loss_acc; head_part[blockIdx.x * 2 + 1] = dz_acc; }
    }
}

template <int H1>
constexpr size_t small_mlp_bwd_smem(int K) { return (size_t)(SM_TB * (H1 + 4) + SM_BC * H1 + SM_TB * (SM_BC + 1) + SM_TB * (K + 1) + SM_TB) * sizeof(float); }

// grid (sample groups, ceil(D/SM_BC)).  A CTA walks the sample tiles g, g+G, ... of its group and keeps
// its slice of dW0 = h0^T dh1' in registers; it also writes the dE chunk of every tile it visits.
// The next tile's h0 / dh1' / S rows are fetched into registers while the current tile is processed.
template <int H1>
__global__ void __launch_bounds__(256) small_mlp_bwd_input_kernel(
    const float* __restrict__ W0 /*[D][H1]*/, const float* __restrict__ h0, const float* __restrict__ dh1 /*[B][H1]*/,
    const float* __restrict__ dz, const float* __restrict__ svec /*[B][K] or null*/, int K, int B, int D,
    float* __restrict__ dE, float* __restrict__ w0_partial /*[gridDim.x][D*H1]*/) {
    extern __shared__ __align__(16) float smem_b[];
    float (*ds)[H1 + 4] = reinterpret_cast<float (*)[H1 + 4]>(smem_b);                                  // [SM_TB][H1+4]
    float (*ws)[H1] = reinterpret_cast<float (*)[H1]>(smem_b + SM_TB * (H1 + 4));                        // [SM_BC][H1]
    float (*hs)[SM_BC + 1] = reinterpret_cast<float (*)[SM_BC + 1]>(smem_b + SM_TB * (H1 + 4) + SM_BC * H1);   // [SM_TB][SM_BC+1]
    float* ss = smem_b + SM_TB * (H1 + 4) + SM_BC * H1 + SM_TB * (SM_BC + 1);                            // [SM_TB][K+1] field sums
    float* gs = ss + SM_TB * (K + 1);                                                                    // [SM_TB] dz
    const int tid = threadIdx.x;
    const int c0 = blockIdx.y * SM_BC;
    const int cw = min(SM_BC, D - c0);
    constexpr int TQ = (SM_BC / 4) * (H1 / 4);             // 4x4 register tiles of the dW0 slice
    constexpr int NT = (TQ + 63) / 64;                     // tiles per thread (64 threads per sample quarter)
    constexpr int NH = SM_TB * (SM_BC / 4) / 256;          // h0 float4 per thread per tile (8)
    constexpr int ND = (SM_TB * (H1 / 4) + 255) / 256;     // dh1 float4 per thread per tile
    float wacc[NT][4][4];
#pragma unroll
    for (int u = 0; u < NT; ++u)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) wacc[u][i][j] = 0.f;
    for (int q = tid; q < SM_BC * H1; q += 256) ws[q / H1][q % H1] = (q / H1) < cw ? W0[(size_t)c0 * H1 + q] : 0.f;
    const int ntiles = (B + SM_TB - 1) / SM_TB;
    const int KS = K / 4;                                  // float4 per S row
    float4 ph[NH], pd[ND], ps;
    float pg;
    auto fetch = [&](int tile) {
        const int b0 = tile * SM_TB;
#pragma unroll
        for (int u = 0; u < NH; ++u) {
            int q = tid + u * 256;
            int r = q / (SM_BC / 4), cc = (q % (SM_BC / 4)) * 4;
            ph[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (b0 + r < B && cc < cw) ph[u] = __ldg(reinterpret_cast<const float4*>(h0 + (size_t)(b0 + r) * D + c0 + cc));
        }
#pragma unroll
        for (int u = 0; u < ND; ++u) {
            int q = tid + u * 256;
            int r = q / (H1 / 4), jj = (q % (H1 / 4)) * 4;
            pd[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q < SM_TB * (H1 / 4) && b0 + r < B) pd[u] = __ldg(reinterpret_cast<const float4*>(dh1 + (size_t)(b0 + r) * H1 + jj));
        }
        ps = make_float4(0.f, 0.f, 0.f, 0.f);
        pg = 0.f;
        if (svec) {   // S rows: SM_TB * K/4 float4, at most 2 per thread for K <= 16 -> loop in the store phase for larger K
            if (tid < SM_TB && b0 + tid < B) pg = __ldg(dz + b0 + tid);
        }
    };
    int tile = blockIdx.x;
    if (tile < ntiles) fetch(tile);
    for (; tile < ntiles; tile += gridDim.x) {
        const int b0 = tile * SM_TB;
        __syncthreads();
#pragma unroll
        for (int u = 0; u < NH; ++u) {
            int q = tid + u * 256;
            int r = q / (SM_BC / 4), cc = (q % (SM_BC / 4)) * 4;
            hs[r][cc] = ph[u].x; hs[r][cc + 1] = ph[u].y; hs[r][cc + 2] = ph[u].z; hs[r][cc + 3] = ph[u].w;
        }
#pragma unroll
        for (int u = 0; u < ND; ++u) {
            int q = tid + u * 256;
            int r = q / (H1 / 4), jj = (q % (H1 / 4)) * 4;
            if (q < SM_TB * (H1 / 4)) *reinterpret_cast<float4*>(&ds[r][jj]) = pd[u];
        }
        if (svec) {
            if (tid < SM_TB) gs[tid] = pg;
            for (int q = tid; q < SM_TB * KS; q += 256) {
                int r = q / KS, k4 = (q % KS) * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (b0 + r < B) v = __ldg(reinterpret_cast<const float4*>(svec + (size_t)(b0 + r) * K + k4));
                float* d = ss + r * (K + 1) + k4;
                d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
            }
        }
        __syncthreads();
        if (tile + (int)gridDim.x < ntiles) fetch(tile + gridDim.x);   // in flight during (b) and (a)
        // (b) dW0[c][j] += sum_s h0[s][c] * dh1[s][j].  Register tiles of 4 columns x 4 units; the 128 samples of the
        //     tile are split over 4 thread quarters (32 samples each, walked in order), the quarters are combined in a
        //     fixed order at the end of the kernel -> deterministic.  16 FMA per 5 shared-memory loads.
        {
            const int qs = tid >> 6, t64 = tid & 63;
#pragma unroll
            for (int u = 0; u < NT; ++u) {
                const int tile = t64 + 64 * u;
                if (tile < TQ) {
                    const int c4 = (tile / (H1 / 4)) * 4, j4 = (tile % (H1 / 4)) * 4;
                    float acc[4][4];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc[i][j] = wacc[u][i][j];
#pragma unroll 4
                    for (int r = qs * 32; r < qs * 32 + 32; ++r) {
                        const float a0 = hs[r][c4], a1 = hs[r][c4 + 1], a2 = hs[r][c4 + 2], a3 = hs[r][c4 + 3];
                        const float4 d = *reinterpret_cast<const float4*>(&ds[r][j4]);
                        acc[0][0] = fmaf(a0, d.x, acc[0][0]); acc[0][1] = fmaf(a0, d.y, acc[0][1]); acc[0][2] = fmaf(a0, d.z, acc[0][2]); acc[0][3] = fmaf(a0, d.w, acc[0][3]);
                        acc[1][0] = fmaf(a1, d.x, acc[1][0]); acc[1][1] = fmaf(a1, d.y, acc[1][1]); acc[1][2] = fmaf(a1, d.z, acc[1][2]); acc[1][3] = fmaf(a1, d.w, acc[1][3]);
                        acc[2][0] = fmaf(a2, d.x, acc[2][0]); acc[2][1] = fmaf(a2, d.y, acc[2][1]); acc[2][2] = fmaf(a2, d.z, acc[2][2]); acc[2][3] = fmaf(a2, d.w, acc[2][3]);
                        acc[3][0] = fmaf(a3, d.x, acc[3][0]); acc[3][1] = fmaf(a3, d.y, acc[3][1]); acc[3][2] = fmaf(a3, d.z, acc[3][2]); acc[3][3] = fmaf(a3, d.w, acc[3][3]);
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) wacc[u][i][j] = acc[i][j];
                }
            }
        }
        __syncthreads();
        // (a) dE[s][c] = sum_j dh1[s][j] W0[c][j] + dz[s] * (S[s][c % K] - h0[s][c])   (in place in hs).
        //     Thread = 2 samples (s, s+64) x 16 columns: every W0 row fetched from shared memory feeds 2 x H1 FMAs.
        {
            const int sp = tid & 63, cg = tid >> 6;
            float d0[H1], d1[H1];
#pragma unroll
            for (int j = 0; j < H1; ++j) { d0[j] = ds[sp][j]; d1[j] = ds[sp + 64][j]; }
            const float g0 = svec ? gs[sp] : 0.f, g1 = svec ? gs[sp + 64] : 0.f;
            const float* srow0 = ss + sp * (K + 1);
            const float* srow1 = ss + (sp + 64) * (K + 1);
            int kk = (c0 + cg * (SM_BC / 4)) % K;
#pragma unroll 2
            for (int c = cg * (SM_BC / 4); c < (cg + 1) * (SM_BC / 4); ++c) {
                float x0 = svec ? g0 * (srow0[kk] - hs[sp][c]) : 0.f;
                float x1 = svec ? g1 * (srow1[kk] - hs[sp + 64][c]) : 0.f;
                kk = (kk + 1 == K) ? 0 : kk + 1;
#pragma unroll
                for (int j4 = 0; j4 < H1 / 4; ++j4) {
                    const float4 w = *reinterpret_cast<const float4*>(&ws[c][j4 * 4]);
                    x0 = fmaf(d0[j4 * 4], w.x, x0); x0 = fmaf(d0[j4 * 4 + 1], w.y, x0); x0 = fmaf(d0[j4 * 4 + 2], w.z, x0); x0 = fmaf(d0[j4 * 4 + 3], w.w, x0);
                    x1 = fmaf(d1[j4 * 4], w.x, x1); x1 = fmaf(d1[j4 * 4 + 1], w.y, x1); x1 = fmaf(d1[j4 * 4 + 2], w.z, x1); x1 = fmaf(d1[j4 * 4 + 3], w.w, x1);
                }
                hs[sp][c] = x0;
                hs[sp + 64][c] = x1;
            }
        }
        __syncthreads();
        for (int q = tid; q < SM_TB * (SM_BC / 4); q += 256) {
            int r = q / (SM_BC / 4), cc = (q % (SM_BC / 4)) * 4;
            if (b0 + r < B && cc < cw)
                *reinterpret_cast<float4*>(dE + (size_t)(b0 + r) * D + c0 + cc) = make_float4(hs[r][cc], hs[r][cc + 1], hs[r][cc + 2], hs[r][cc + 3]);
        }
    }
    // combine the four sample quarters in a fixed order (reusing the input tile as scratch) and emit the partial
    __syncthreads();
    {
        float* scratch = &hs[0][0];                        // 4 * SM_BC * H1 floats <= SM_TB * (SM_BC + 1)
        const int qs = tid >> 6, t64 = tid & 63;
#pragma unroll
        for (int u = 0; u < NT; ++u) {
            const int tile = t64 + 64 * u;
            if (tile < TQ) {
                const int c4 = (tile / (H1 / 4)) * 4, j4 = (tile % (H1 / 4)) * 4;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    *reinterpret_cast<float4*>(scratch + (size_t)qs * SM_BC * H1 + (c4 + i) * H1 + j4) =
                        make_float4(wacc[u][i][0], wacc[u][i][1], wacc[u][i][2], wacc[u][i][3]);
            }
        }
        __syncthreads();
        for (int q = tid; q < SM_BC * (H1 / 4); q += 256) {
            const int c = q / (H1 / 4), j4 = (q % (H1 / 4)) * 4;
            float4 a = *reinterpret_cast<const float4*>(scratch + c * H1 + j4);
#pragma unroll
            for (int z = 1; z < 4; ++z) {
                const float4 t = *reinterpret_cast<const float4*>(scratch + (size_t)z * SM_BC * H1 + c * H1 + j4);
                a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
            }
            if (c < cw) *reinterpret_cast<float4*>(w0_partial + (size_t)blockIdx.x * D * H1 + (size_t)(c0 + c) * H1 + j4) = a;
        }
    }
}
