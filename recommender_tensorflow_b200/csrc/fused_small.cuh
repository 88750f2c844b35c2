// Fused forward + top-of-backward kernel for small towers (every hidden layer <= 32 wide; the reference default
// hidden_units [16,16], trainers/deep_fm.py:21): ONE kernel does, per tile of FS_TS samples,
//
//   trainers/deep_fm.py:39      linear_model     gather of the linear weights                       (K2)
//   trainers/deep_fm.py:52-73   input_layer      gather of the embedding rows (+ numeric embeddings) into SHARED memory
//   trainers/deep_fm.py:79-87   FM block         0.5 * sum_k((sum_f E)^2 - sum_f E^2)
//   trainers/deep_fm.py:93-112  DNN block        relu dense stack + dense(1), weights resident in shared memory
//   trainers/deep_fm.py:114-125 head             sigmoid cross-entropy, dz, and the backward pass down to dh1' = dL/d(pre-act 1)
//                                                + the weight gradients dW0 = E^T dh1', dW1.., db.., dWo (per-CTA partials)
//
// so `input_layer` [B, d*K] and its gradient dE are NEVER written to HBM (at the Criteo shape: 164 MB each, written
// once and read two / one times by the unfused path = 0.8 GB of a 0.82 GB algorithmic budget).  The table rows are
// read as stored and the deferred non-lazy Adam decay is replayed in registers (replay.cuh).  What the sparse
// optimizer needs later is tiny and stays in L2: per sample  s = sum_f E [K],  dh1' [H1],  dz;  the gradient of
// lookup (b, f) is rebuilt where it is consumed (GradSrcFused::fetch):
//      dE[b,f,:] = dz_b (s_b - E_row) + dh1'_b . W0[f*K .. f*K+K, :]^T
//
// Thread mapping (256 threads, 2 CTAs per SM so that one CTA's gather overlaps the other's arithmetic; a variant with one
// CTA per SM that staged whole records of 8-sample tiles by cp.async into double buffers removed the memory stalls but
// ran the arithmetic at 2 warps per scheduler and was twice as slow: 0.80 vs 0.40 ms, profiles/r02d):
//   phase 1  warp per sample (FS_TS/8 samples per warp), K/4 lanes per table row, 32/(K/4) fields per round; the ids of
//            the tile were prefetched into shared memory during the previous tile
//   phase 2  layer 0: the warps take the fields round-robin, lane = (sample group, output quad); partial sums combined
//            through shared memory in warp order
//   phase 3  upper layers / head / loss / backward to dh1': thread per (sample, unit)
//   phase 4  dW0 accumulated in REGISTERS across all tiles of the CTA (thread = 4 units x NC input columns, no predicates)
//   phase 5  numeric-feature gradient terms (sum_b x_bj * {dz s, dh1', x dz, dz}) in registers across tiles
// Per-CTA partials are combined in CTA order by fused_reduce_kernel (deterministic).
#pragma once
#include "dfm_types.cuh"
#include "embed_kernels.cuh"
#include "mlp_kernels.cuh"
#include "row_apply.cuh"
#include "small_mlp.cuh"

constexpr int FS_TS = 16;          // samples per tile
constexpr int FS_NC = 12;          // max input columns per thread in the dW0 accumulation (x 4 units)
constexpr int FS_NUMACC = 4;       // numeric-gradient accumulators per thread

struct FusedArgs {
    const int32_t* ids; int B, dc, dn, n_slots;
    const uint32_t* row_off; Table tb; BatchPtrs bp;
    const float* dw;                               // packed dense parameters
    int off_num_emb, off_num_lin, off_bias;        // offsets in dw, -1: absent
    int use_linear, use_mf;
    SmallMlpDesc m;
    const float* labels; float scale; int train;
    RowReplay rr; OptDev od, ol;
    const uint32_t* uidx; const float* rowbuf; int rowbuf_stride;     // sharded: rows were fetched into rowbuf[unique index]
    float *logits, *logits_out, *dz_out, *dh1_out, *s_out;
    float *up_partial, *w0_partial, *num_partial, *head_part;
    int D, es_stride, n_numacc;                    // D = d*K; floats per E row in shared memory; dn * (K + H1 + 2)
};

__host__ __device__ inline int fs_es_stride(int D) { return ((D + 4) / 4) % 2 ? D + 4 : D + 8; }   // multiple of 4, odd number of float4

static inline size_t fused_smem_floats(const SmallMlpDesc& m, int K, int dc, int dn) {
    const int H1 = m.H[0];
    size_t f = (size_t)m.D * H1;                   // W0
    f += 2 * (size_t)m.up_count + 4;               // upper parameters + their per-CTA gradient accumulators
    f += (size_t)FS_TS * fs_es_stride(m.D);        // E tile
    f += (size_t)8 * FS_TS * H1;                   // layer-0 partial sums
    f += (size_t)FS_TS * H1;                       // dh1' (16-byte aligned copy)
    f += 2 * (size_t)FS_TS * m.act_stride;         // activations, their gradients
    f += 3 * (size_t)FS_TS;                        // zacc, dz, loss terms
    f += (size_t)FS_TS * (dn > 0 ? dn : 1) + 4;    // numeric inputs
    f += (size_t)FS_TS * K;                        // field sums s
    f += 4 * (size_t)FS_TS * (dc > 0 ? dc : 1) + 8;    // ids (and unique-row indices) of two tiles
    return f + 16;
}

// NC: input columns per thread in the dW0 accumulation = ceil(d / (CG / K)), CG = 256 / (H1/4)  (compile time so that
// the accumulators stay in registers without per-column predicates)
// WGT: weighted model, the head multiplies the loss term and dz of sample b by a.bp.weights[b] (after the scale: w = 1 is exact)
// SQ: squared head (sq_head) instead of the sigmoid cross-entropy
template <int K, int H1, bool ROWBUF, int NC, bool SQ, bool WGT>
__global__ void __launch_bounds__(256, 2) fused_small_kernel(FusedArgs a) {
    constexpr int LPR = K / 4, FPR = 32 / LPR;
    constexpr int OQ = H1 / 4;                     // output quads
    constexpr int NSG = 32 / OQ;                   // sample groups per warp in phase 2
    constexpr int SPT = (FS_TS + NSG - 1) / NSG;   // samples per thread in phase 2
    constexpr int CG = 256 / OQ;                   // column groups in phase 4
    constexpr int FST = CG / K;                    // fields per column-group step
    static_assert(CG % K == 0, "column groups must cover whole fields");
    extern __shared__ __align__(16) float smem[];
    const SmallMlpDesc& m = a.m;
    const int D = a.D, ES = a.es_stride;
    const int dc = a.dc, dn = a.dn, d = dc + dn;
    float* W0s = smem;                                   // [D][H1]
    float* ups = W0s + (size_t)D * H1;                   // packed parameters above W0
    float* gup = ups + m.up_count;                       // per-CTA gradient accumulators (same layout)
    float* Es = gup + m.up_count + ((4 - ((2 * m.up_count) & 3)) & 3);   // [FS_TS][ES], 16-byte aligned
    float* part = Es + (size_t)FS_TS * ES;               // [8][FS_TS][H1]
    float* dh1s = part + 8 * FS_TS * H1;                 // [FS_TS][H1]
    float* acts = dh1s + FS_TS * H1;                     // [FS_TS][act_stride]
    float* dacts = acts + FS_TS * m.act_stride;          // [FS_TS][act_stride]
    float* zs = dacts + FS_TS * m.act_stride;            // [FS_TS] linear + FM logit
    float* dzs = zs + FS_TS;                             // [FS_TS]
    float* red = dzs + FS_TS;                            // [FS_TS] loss terms
    float* xs = red + FS_TS;                             // [FS_TS][dn]
    float* ss = xs + ((FS_TS * (dn > 0 ? dn : 1) + 3) & ~3);      // [FS_TS][K]
    int32_t* ids_s = reinterpret_cast<int32_t*>(ss + FS_TS * K);  // [2][FS_TS * dc]
    uint32_t* uix_s = reinterpret_cast<uint32_t*>(ids_s + 2 * FS_TS * (dc > 0 ? dc : 1));   // [2][FS_TS * dc] (sharded)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < D * H1; i += 256) W0s[i] = a.dw[m.off_W[0] + i];
    for (int i = tid; i < m.up_count; i += 256) { ups[i] = a.dw[m.up_begin + i]; gup[i] = 0.f; }
    auto UP = [&](int packed_off) { return ups + (packed_off - m.up_begin); };
    auto GUP = [&](int packed_off) { return gup + (packed_off - m.up_begin); };
    const float* num_emb = a.off_num_emb >= 0 ? a.dw + a.off_num_emb : nullptr;
    const float* num_lin = a.off_num_lin >= 0 ? a.dw + a.off_num_lin : nullptr;
    const float bias0 = (a.use_linear && a.off_bias >= 0) ? a.dw[a.off_bias] : 0.f;
    const ReplayStep rs = replay_step_load(a.rr.rd.closed ? a.rr.rd : a.rr.rl, a.rr.upto);
    const int sub = lane % LPR, grp = lane / LPR;
    const int train = a.train;
    const bool drop = train && m.drop_keep > 0.f;
    const int ntiles = (a.B + FS_TS - 1) / FS_TS;
    const int nrows = FS_TS * dc;                  // table rows per tile (<= 512)

    // dW0 accumulators: thread (jq, cg) owns unit quad jq and input columns (f0 + FST*u)*K + kq, u < NC
    const int jq = tid % OQ, cg = tid / OQ, kq = cg % K, f0 = cg / K;
    int ecol[NC];
    float wacc[NC][4];
#pragma unroll
    for (int u = 0; u < NC; ++u) {
        const int f = f0 + FST * u;
        ecol[u] = (f < d ? f * K : 0) + kq;        // columns beyond D accumulate garbage that is never stored
        wacc[u][0] = 0.f; wacc[u][1] = 0.f; wacc[u][2] = 0.f; wacc[u][3] = 0.f;
    }
    // numeric-gradient accumulators: thread owns terms ai = tid + 256 u of [dn][K + H1 + 2]
    float nacc[FS_NUMACC];
    int nj[FS_NUMACC], nr[FS_NUMACC];
#pragma unroll
    for (int u = 0; u < FS_NUMACC; ++u) {
        const int ai = tid + 256 * u, per = K + H1 + 2;
        nacc[u] = 0.f;
        nj[u] = ai < a.n_numacc ? ai / per : -1;
        nr[u] = ai < a.n_numacc ? ai - (ai / per) * per : 0;
    }
    float loss_acc = 0.f, dz_acc = 0.f;

    // ids (and, sharded, the unique-row indices) of the NEXT tile are fetched while this tile is computed: a tile of ids is
    // contiguous ([B][dc] row-major), two coalesced loads per thread, and the gather below starts from shared memory
    // instead of a dependent global load
    int32_t idr[2]; uint32_t uxr[2];
    auto load_ids = [&](int tile) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int r = tid + 256 * q;
            idr[q] = -1; uxr[q] = 0;
            if (tile < ntiles && r < nrows) {
                const int64_t gi = (int64_t)tile * nrows + r;
                if (gi < (int64_t)a.B * dc) {
                    idr[q] = __ldg(a.ids + gi);
                    if (ROWBUF) uxr[q] = __ldg(a.uidx + gi);
                }
            }
        }
    };
    auto store_ids = [&](int bf) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int r = tid + 256 * q;
            if (r < nrows) { ids_s[bf * nrows + r] = idr[q]; if (ROWBUF) uix_s[bf * nrows + r] = uxr[q]; }
        }
    };
    load_ids(blockIdx.x);
    store_ids(0);
    __syncthreads();

    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int bf = it & 1;
        const int b0 = tile * FS_TS;
        load_ids(tile + gridDim.x);                        // next tile's ids: in flight during this tile, stored at its end
        // ------------------------------------------------------------------ phase 1: gather (+ replay) -> E tile, FM, linear
        for (int sl = warp; sl < FS_TS; sl += 8) {
            const int b = b0 + sl;
            const bool live = b < a.B;
            float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
            float lin = 0.f;
            float* erow = Es + (size_t)sl * ES;
            const int32_t* idrow = ids_s + bf * nrows + sl * dc;
            for (int fb = 0; fb < dc; fb += 2 * FPR) {       // two rounds of rows in flight per lane group
                float4 e[2];
                float lw[2];
                int f[2];
                bool on[2];
                size_t row[2];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    f[r] = fb + r * FPR + grp;
                    on[r] = false; row[r] = 0;
                    e[r] = make_float4(0.f, 0.f, 0.f, 0.f); lw[r] = 0.f;
                    if (live && f[r] < dc) {
                        const int32_t id = idrow[f[r]];
                        if (id >= 0) {
                            on[r] = true;
                            if (ROWBUF) row[r] = (size_t)uix_s[bf * nrows + sl * dc + f[r]];
                            else row[r] = (size_t)__ldg(a.row_off + f[r]) + (uint32_t)id;
                        }
                    }
                }
                if (ROWBUF) {
#pragma unroll
                    for (int r = 0; r < 2; ++r)
                        if (on[r]) {
                            const float* rp = a.rowbuf + row[r] * a.rowbuf_stride;
                            e[r] = __ldg(reinterpret_cast<const float4*>(rp) + sub);
                            lw[r] = __ldg(rp + K);
                        }
                } else {
                    // the whole record of both rows is requested before either is used (one dependent-load level)
                    float4 lr[2], mm[2], vv[2];
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        lr[r] = make_float4(0.f, 0.f, 0.f, 0.f); mm[r] = lr[r]; vv[r] = lr[r];
                        if (on[r]) {
                            lr[r] = __ldg(tab_lin(a.tb, row[r]));
                            e[r] = __ldg(tab_w(a.tb, row[r]) + sub);
                            if (a.rr.emb_adam && a.rr.upto >= 0) { mm[r] = __ldg(tab_s1(a.tb, row[r]) + sub); vv[r] = __ldg(tab_s2(a.tb, row[r]) + sub); }
                        }
                    }
#pragma unroll
                    for (int r = 0; r < 2; ++r)
                        if (on[r]) {
                            replay_row(e[r], mm[r], vv[r], lr[r], sub == 0, a.rr, rs, a.od, a.ol);
                            lw[r] = lr[r].x;
                        }
                }
#pragma unroll
                for (int r = 0; r < 2; ++r)
                    if (f[r] < dc) {
                        reinterpret_cast<float4*>(erow + f[r] * K)[sub] = e[r];
                        s.x += e[r].x; s.y += e[r].y; s.z += e[r].z; s.w += e[r].w;
                        q.x = fmaf(e[r].x, e[r].x, q.x); q.y = fmaf(e[r].y, e[r].y, q.y);
                        q.z = fmaf(e[r].z, e[r].z, q.z); q.w = fmaf(e[r].w, e[r].w, q.w);
                        if (sub == 0) lin += lw[r];
                    }
            }
            for (int j0 = 0; j0 < dn; j0 += FPR) {
                const int j = j0 + grp;
                if (j < dn) {
                    const float x = live ? __ldg(a.bp.num[j] + b) : 0.f;
                    float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (num_emb) {
                        const float4 ve = __ldg(reinterpret_cast<const float4*>(num_emb + j * K) + sub);
                        e = make_float4(x * ve.x, x * ve.y, x * ve.z, x * ve.w);
                    }
                    reinterpret_cast<float4*>(erow + (dc + j) * K)[sub] = e;
                    s.x += e.x; s.y += e.y; s.z += e.z; s.w += e.w;
                    q.x = fmaf(e.x, e.x, q.x); q.y = fmaf(e.y, e.y, q.y); q.z = fmaf(e.z, e.z, q.z); q.w = fmaf(e.w, e.w, q.w);
                    if (sub == 0) {
                        xs[sl * dn + j] = x;
                        if (a.use_linear && num_lin) lin = fmaf(x, __ldg(num_lin + j), lin);
                    }
                }
            }
            // combine the FPR field groups (fixed butterfly -> deterministic)
#pragma unroll
            for (int o = LPR; o < 32; o <<= 1) {
                s.x += __shfl_xor_sync(0xffffffffu, s.x, o); s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
                s.z += __shfl_xor_sync(0xffffffffu, s.z, o); s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
                q.x += __shfl_xor_sync(0xffffffffu, q.x, o); q.y += __shfl_xor_sync(0xffffffffu, q.y, o);
                q.z += __shfl_xor_sync(0xffffffffu, q.z, o); q.w += __shfl_xor_sync(0xffffffffu, q.w, o);
            }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) lin += __shfl_xor_sync(0xffffffffu, lin, o);
            float t = (s.x * s.x - q.x) + (s.y * s.y - q.y) + (s.z * s.z - q.z) + (s.w * s.w - q.w);
#pragma unroll
            for (int o = 1; o < LPR; o <<= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            if (grp == 0) {
                reinterpret_cast<float4*>(ss + sl * K)[sub] = s;
                if (live && a.s_out) reinterpret_cast<float4*>(a.s_out + (size_t)b * K)[sub] = s;
            }
            if (lane == 0) {
                float z = 0.f;
                if (a.use_linear) z += lin + bias0;
                if (a.use_mf) z += 0.5f * t;
                zs[sl] = z;
            }
        }
        __syncthreads();
        // ------------------------------------------------------------------ phase 2: layer 0, the warps take the fields round-robin
        {
            const int oq = lane % OQ, sg = lane / OQ;
            float acc[SPT][4];
#pragma unroll
            for (int j = 0; j < SPT; ++j) { acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f; }
            if (sg < FS_TS) {
                for (int f = warp; f < d; f += 8) {
                    const float* wrow = W0s + (size_t)f * K * H1 + oq * 4;
                    const float* ep = Es + (size_t)sg * ES + f * K;
#pragma unroll 4
                    for (int k = 0; k < K; ++k) {
                        const float4 w = *reinterpret_cast<const float4*>(wrow + k * H1);
#pragma unroll
                        for (int j = 0; j < SPT; ++j) {
                            if (sg + j * NSG < FS_TS) {
                                const float x = ep[(size_t)j * NSG * ES + k];
                                acc[j][0] = fmaf(x, w.x, acc[j][0]); acc[j][1] = fmaf(x, w.y, acc[j][1]);
                                acc[j][2] = fmaf(x, w.z, acc[j][2]); acc[j][3] = fmaf(x, w.w, acc[j][3]);
                            }
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < SPT; ++j)
                    if (sg + j * NSG < FS_TS)
                        *reinterpret_cast<float4*>(part + ((size_t)warp * FS_TS + sg + j * NSG) * H1 + oq * 4) =
                            make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
            }
        }
        __syncthreads();
        {
            const float* bb = UP(m.off_b[0]);
            const uint64_t key = drop ? dfm_drop_key(m.drop_seed, m.drop_step, 0) : 0;
            for (int idx = tid; idx < FS_TS * H1; idx += 256) {
                const int sl = idx / H1, o = idx - sl * H1;
                float v = bb[o];
#pragma unroll
                for (int w = 0; w < 8; ++w) v += part[((size_t)w * FS_TS + sl) * H1 + o];
                v = fmaxf(v, 0.f);
                if (drop) v *= dfm_drop(key, (uint64_t)(m.drop_row0 + b0 + sl) * H1 + o, m.drop_keep, m.drop_inv);
                acts[sl * m.act_stride + o] = v;
            }
        }
        __syncthreads();
        // ------------------------------------------------------------------ phase 3: upper layers, head, loss, backward to dh1'
        int aoff = 0;
        for (int l = 1; l < m.L; ++l) {
            const int Hin = m.H[l - 1], Hout = m.H[l];
            const float* W = UP(m.off_W[l]);
            const float* bb = UP(m.off_b[l]);
            const uint64_t key = drop ? dfm_drop_key(m.drop_seed, m.drop_step, l) : 0;
            for (int idx = tid; idx < FS_TS * Hout; idx += 256) {
                const int sl = idx / Hout, o = idx - sl * Hout;
                const float* arow = acts + sl * m.act_stride + aoff;
                float v = bb[o];
                for (int j = 0; j < Hin; ++j) v = fmaf(arow[j], W[j * Hout + o], v);
                v = fmaxf(v, 0.f);
                if (drop) v *= dfm_drop(key, (uint64_t)(m.drop_row0 + b0 + sl) * Hout + o, m.drop_keep, m.drop_inv);
                acts[sl * m.act_stride + aoff + Hin + o] = v;
            }
            aoff += Hin;
            __syncthreads();
        }
        const int HL = m.H[m.L - 1];
        const float* Wo = UP(m.off_Wo);
        if (tid < FS_TS) {
            const int sl = tid, b = b0 + sl;
            const float* arow = acts + sl * m.act_stride + aoff;
            float z = UP(m.off_bo)[0];
            for (int j = 0; j < HL; ++j) z = fmaf(arow[j], Wo[j], z);
            z += zs[sl];
            float g = 0.f, lterm = 0.f;
            if (b < a.B) {
                a.logits[b] = z;
                if (a.logits_out) a.logits_out[b] = z;
                if (train) {
                    const float y = a.labels[b];
                    if constexpr (SQ) {
                        sq_head(z, y, a.scale, lterm, g);
                    } else {
                        lterm = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
                        g = (1.f / (1.f + expf(-z)) - y) * a.scale;
                    }
                    if constexpr (WGT) { const float w = a.bp.weights[b]; g *= w; lterm *= w; }
                    a.dz_out[b] = g;
                }
            }
            dzs[sl] = g;
            red[sl] = lterm;
        }
        __syncthreads();
        if (train) {
            const float dsc = m.drop_keep > 0.f ? m.drop_inv : 1.f;   // gradient through the dropout after each ReLU
            for (int idx = tid; idx < FS_TS * HL; idx += 256) {
                const int sl = idx / HL, j = idx - sl * HL;
                dacts[sl * m.act_stride + aoff + j] = acts[sl * m.act_stride + aoff + j] > 0.f ? dzs[sl] * Wo[j] * dsc : 0.f;
            }
            __syncthreads();
            int ao = aoff;
            for (int l = m.L - 1; l >= 1; --l) {
                const int Hin = m.H[l - 1], Hout = m.H[l];
                const float* W = UP(m.off_W[l]);
                const int in_off = ao - Hin;
                for (int idx = tid; idx < FS_TS * Hin; idx += 256) {
                    const int sl = idx / Hin, j = idx - sl * Hin;
                    const float* drow = dacts + sl * m.act_stride + ao;
                    float v = 0.f;
                    for (int o = 0; o < Hout; ++o) v = fmaf(drow[o], W[j * Hout + o], v);
                    dacts[sl * m.act_stride + in_off + j] = acts[sl * m.act_stride + in_off + j] > 0.f ? v * dsc : 0.f;
                }
                ao = in_off;
                __syncthreads();
            }
            // dh1' -> global (the sparse optimizer rebuilds dE from it) and an aligned copy for phase 4
            for (int idx = tid; idx < FS_TS * H1; idx += 256) {
                const int sl = idx / H1, j = idx - sl * H1;
                const float v = dacts[sl * m.act_stride + j];
                dh1s[idx] = v;
                if (b0 + sl < a.B) a.dh1_out[(size_t)(b0 + sl) * H1 + j] = v;
            }
            // gradients of everything above W0: each output owned by one thread, samples walked in order
            int go = 0;
            for (int l = 0; l < m.L; ++l) {
                const int Hl = m.H[l];
                for (int j = tid; j < Hl; j += 256) {
                    float v = 0.f;
                    for (int r = 0; r < FS_TS; ++r) v += dacts[r * m.act_stride + go + j];
                    GUP(m.off_b[l])[j] += v;
                }
                if (l + 1 < m.L) {
                    const int Hn = m.H[l + 1];
                    for (int qx = tid; qx < Hl * Hn; qx += 256) {
                        const int j = qx / Hn, o = qx - j * Hn;
                        float v = 0.f;
                        for (int r = 0; r < FS_TS; ++r) v = fmaf(acts[r * m.act_stride + go + j], dacts[r * m.act_stride + go + Hl + o], v);
                        GUP(m.off_W[l + 1])[qx] += v;
                    }
                } else {
                    for (int j = tid; j < Hl; j += 256) {
                        float v = 0.f;
                        for (int r = 0; r < FS_TS; ++r) v = fmaf(acts[r * m.act_stride + go + j], dzs[r], v);
                        GUP(m.off_Wo)[j] += v;
                    }
                }
                go += Hl;
            }
            if (tid == 0) {
                float x = 0.f, c = 0.f;
                for (int r = 0; r < FS_TS; ++r) { x += red[r]; c += dzs[r]; }
                loss_acc += x;
                dz_acc += c;
            }
            __syncthreads();
            // -------------------------------------------------------------- phase 4: dW0 += E^T dh1' (registers, no predicates)
#pragma unroll 4
            for (int r = 0; r < FS_TS; ++r) {
                const float4 dv = *reinterpret_cast<const float4*>(dh1s + r * H1 + jq * 4);
                const float* er = Es + (size_t)r * ES;
#pragma unroll
                for (int u = 0; u < NC; ++u) {
                    const float x = er[ecol[u]];
                    wacc[u][0] = fmaf(x, dv.x, wacc[u][0]); wacc[u][1] = fmaf(x, dv.y, wacc[u][1]);
                    wacc[u][2] = fmaf(x, dv.z, wacc[u][2]); wacc[u][3] = fmaf(x, dv.w, wacc[u][3]);
                }
            }
            // -------------------------------------------------------------- phase 5: numeric-feature gradient terms
            if (dn > 0) {
#pragma unroll
                for (int u = 0; u < FS_NUMACC; ++u) {
                    if (nj[u] >= 0) {
                        const int j = nj[u], r = nr[u];
                        float v = nacc[u];
#pragma unroll 4
                        for (int sl = 0; sl < FS_TS; ++sl) {
                            const float x = xs[sl * dn + j];
                            float y;
                            if (r < K) y = dzs[sl] * ss[sl * K + r];            // -> sum_b x dz s[k]
                            else if (r < K + H1) y = dh1s[sl * H1 + (r - K)];   // -> sum_b x dh1'[o]
                            else if (r == K + H1) y = x * dzs[sl];              // -> sum_b x^2 dz
                            else y = dzs[sl];                                   // -> sum_b x dz   (numeric linear weight)
                            v = fmaf(x, y, v);
                        }
                        nacc[u] = v;
                    }
                }
            }
        }
        store_ids(bf ^ 1);             // the next tile's ids (the other half of the double buffer)
        __syncthreads();               // the E tile and the per-tile scratch are reused
    }
    if (train) {
        if (tid == 0) GUP(m.off_bo)[0] = dz_acc;
        __syncthreads();
        for (int i = tid; i < m.up_count; i += 256) a.up_partial[(size_t)blockIdx.x * m.up_count + i] = gup[i];
        {
            float* wp = a.w0_partial + (size_t)blockIdx.x * D * H1;
#pragma unroll
            for (int u = 0; u < NC; ++u) {
                const int f = f0 + FST * u;
                if (f < d)
                    *reinterpret_cast<float4*>(wp + (size_t)(f * K + kq) * H1 + jq * 4) = make_float4(wacc[u][0], wacc[u][1], wacc[u][2], wacc[u][3]);
            }
        }
#pragma unroll
        for (int u = 0; u < FS_NUMACC; ++u)
            if (tid + 256 * u < a.n_numacc) a.num_partial[(size_t)blockIdx.x * a.n_numacc + tid + 256 * u] = nacc[u];
        if (tid == 0) { a.head_part[blockIdx.x * 2] = loss_acc; a.head_part[blockIdx.x * 2 + 1] = dz_acc; }
    }
}

// Combines the per-CTA partials of fused_small_kernel in CTA order (deterministic) into the dense gradient buffer:
//   dg[up_begin ..]  <- b0, W1, b1, ..., Wo, bo        dg[off_W0 ..] <- dW0
//   numeric terms -> scratch, finished by the LAST block to arrive (numeric_embeddings / numeric linear gradients):
//      g_num_emb[j,k] = P[j,k] - V[j,k] Q[j] + sum_o R[j,o] W0[(dc+j)K+k, o]      g_num_lin[j] = S[j]
//   block 0 also reduces the loss / dz partials (loss, gradient of the linear bias)
struct FusedReduceArgs {
    const float *up_partial, *w0_partial, *num_partial, *head_part;
    int n_cta, up_count, up_begin, off_W0, w0_count, n_numacc;
    float* dg; float* num_scratch; unsigned int* done;
    const float* dw; int off_num_emb, off_num_lin, off_bias, dc, dn, K, H1, use_mf;
    float loss_scale; float *loss_out, *loss_copy, *dzsum_out;
    int direct_num;       // fused_rows_kernel: num_partial holds [dn*K | dn] finished numeric gradients per CTA (n_numacc = dn*K + dn)
};

static __global__ void __launch_bounds__(256) fused_reduce_kernel(FusedReduceArgs r) {
    const int total = r.up_count + r.w0_count + r.n_numacc;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < total) {
        const float* p; size_t stride; float* dst;
        if (i < r.up_count) { p = r.up_partial + i; stride = r.up_count; dst = r.dg + r.up_begin + i; }
        else if (i < r.up_count + r.w0_count) { p = r.w0_partial + (i - r.up_count); stride = r.w0_count; dst = r.dg + r.off_W0 + (i - r.up_count); }
        else {
            const int q = i - r.up_count - r.w0_count;
            p = r.num_partial + q; stride = r.n_numacc; dst = r.num_scratch + q;
            if (r.direct_num) {
                if (q < r.dn * r.K) dst = r.off_num_emb >= 0 ? r.dg + r.off_num_emb + q : nullptr;
                else dst = r.off_num_lin >= 0 ? r.dg + r.off_num_lin + (q - r.dn * r.K) : nullptr;
            }
        }
        float s = 0.f;
        int c = 0;
        for (; c + 32 <= r.n_cta; c += 32) {      // 32 independent loads in flight, added in CTA order (the walk over 144 .. 256
            float t[32];                          // CTA partials is a chain of L2 round trips: 8 per round took 11 .. 23 us)
#pragma unroll
            for (int u = 0; u < 32; ++u) t[u] = __ldg(p + (size_t)(c + u) * stride);
#pragma unroll
            for (int u = 0; u < 32; ++u) s += t[u];
        }
        for (; c + 8 <= r.n_cta; c += 8) {
            float t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) t[u] = __ldg(p + (size_t)(c + u) * stride);
#pragma unroll
            for (int u = 0; u < 8; ++u) s += t[u];
        }
        for (; c < r.n_cta; ++c) s += __ldg(p + (size_t)c * stride);
        if (dst) *dst = s;
    }
    __shared__ float sa[256], sc[256];
    __shared__ bool last;
    if (blockIdx.x == 0) {
        float x = 0.f, c = 0.f;
        for (int k = threadIdx.x; k < r.n_cta; k += 256) { x += r.head_part[k * 2]; c += r.head_part[k * 2 + 1]; }
        sa[threadIdx.x] = x; sc[threadIdx.x] = c;
        __syncthreads();
        for (int o = 128; o >= 1; o >>= 1) {
            if (threadIdx.x < o) { sa[threadIdx.x] += sa[threadIdx.x + o]; sc[threadIdx.x] += sc[threadIdx.x + o]; }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            if (r.loss_out) *r.loss_out = sa[0] * r.loss_scale;
            if (r.loss_copy) *r.loss_copy = sa[0] * r.loss_scale;
            if (r.dzsum_out) *r.dzsum_out = sc[0];
            if (r.off_bias >= 0) r.dg[r.off_bias] = sc[0];
        }
    }
    if (r.dn <= 0 || r.direct_num) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(r.done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (threadIdx.x == 0) *r.done = 0;                    // re-armed for the next step
    const int per = r.K + r.H1 + 2;
    const volatile float* ns = r.num_scratch;
    for (int o = threadIdx.x; o < r.dn * r.K + r.dn; o += 256) {
        if (o < r.dn * r.K) {
            if (r.off_num_emb < 0) continue;
            const int j = o / r.K, k = o - j * r.K;
            float v = 0.f;
            if (r.use_mf) v = ns[j * per + k] - r.dw[r.off_num_emb + o] * ns[j * per + r.K + r.H1];
            const float* w0 = r.dw + r.off_W0 + (size_t)((r.dc + j) * r.K + k) * r.H1;
            for (int u = 0; u < r.H1; ++u) v = fmaf(ns[j * per + r.K + u], w0[u], v);
            r.dg[r.off_num_emb + o] = v;
        } else if (r.off_num_lin >= 0) {
            const int j = o - r.dn * r.K;
            r.dg[r.off_num_lin + j] = ns[j * per + r.K + r.H1 + 1];
        }
    }
}

// Gradient source of the sparse optimizer when the step ran through fused_small_kernel: the gradient of lookup
// (b, f) is rebuilt from the per-sample vectors (all L2-resident) instead of being read from a [B, d*K] buffer.
//   fetch -> g = dz_b s_b + dh1'_b . W0[f*K + k, :]^T  (this lane's 4 k),  gl = dz_b;  the caller subtracts sum(dz) * E_row.
template <int K, int H1>
struct GradSrcFused {
    static constexpr bool SUB_E = true;
    const float* dh1;           // [B][H1]
    const float* s;             // [B][K], nullptr without the FM term
    const float* dz;            // [B]
    const float* W0;            // [D][H1] (global; the K x H1 slice of a field stays in L1)
    int n_slots;
    const float* erow; int erow_stride;     // sharded requester: the rows as fetched from their owners (unique order)
    __device__ __forceinline__ bool sub_e() const { return s != nullptr; }
    // staging interface of row_apply_kernel: [dh1' (H1) | s (K) | dz, pad] of the row's first lookup, moved by cp.async
    static constexpr int STAGE_F = H1 + K + 4;
    __device__ __forceinline__ void stage_async(uint32_t val, float* dst, int sub) const {
        constexpr int LPR = K / 4;
        const uint32_t b = payload_sample(val);
        for (int c = sub; c < H1 / 4; c += LPR) cp_async16(dst + c * 4, dh1 + (size_t)b * H1 + c * 4);
        if (s) cp_async16(dst + H1 + sub * 4, s + (size_t)b * K + sub * 4);
        if (sub == LPR - 1) cp_async4(dst + H1 + K, dz + b);
    }
    int n_w0;                   // floats of W0 = D * H1 (copied to shared memory once per CTA by row_apply_kernel)
    int aux_floats() const { return n_w0; }
    __device__ __forceinline__ void aux_load(float* dst, int tid) const {
        for (int i = tid * 4; i < n_w0; i += 256 * 4) *reinterpret_cast<float4*>(dst + i) = __ldg(reinterpret_cast<const float4*>(W0 + i));
    }
    __device__ __forceinline__ void consume(const float* st, const float* w0s, uint32_t val, int sub, float4& g, float& gl) const {
        const uint32_t f = payload_slot(val);
        const float z = st[H1 + K];
        gl = z;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        if (s) {
            const float4 sv = *reinterpret_cast<const float4*>(st + H1 + sub * 4);
            acc[0] = z * sv.x; acc[1] = z * sv.y; acc[2] = z * sv.z; acc[3] = z * sv.w;
        }
        const float4* wr = reinterpret_cast<const float4*>(w0s + ((size_t)f * K + sub * 4) * H1);
#pragma unroll
        for (int o4 = 0; o4 < H1 / 4; ++o4) {
            const float4 d = *reinterpret_cast<const float4*>(st + o4 * 4);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const float4 w = wr[kk * (H1 / 4) + o4];
                acc[kk] = fmaf(d.x, w.x, fmaf(d.y, w.y, fmaf(d.z, w.z, fmaf(d.w, w.w, acc[kk]))));
            }
        }
        g = make_float4(acc[0], acc[1], acc[2], acc[3]);
    }
    __device__ __forceinline__ void fetch(uint32_t val, int sub, bool, float4& g, float& gl) const {
        const uint32_t b = payload_sample(val), f = payload_slot(val);
        const float z = __ldg(dz + b);
        gl = z;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        if (s) {
            const float4 sv = __ldg(reinterpret_cast<const float4*>(s + (size_t)b * K) + sub);
            acc[0] = z * sv.x; acc[1] = z * sv.y; acc[2] = z * sv.z; acc[3] = z * sv.w;
        }
        const float4* dh = reinterpret_cast<const float4*>(dh1 + (size_t)b * H1);
        const float4* wr = reinterpret_cast<const float4*>(W0 + ((size_t)f * K + sub * 4) * H1);
#pragma unroll
        for (int o4 = 0; o4 < H1 / 4; ++o4) {
            const float4 d = __ldg(dh + o4);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const float4 w = __ldg(wr + kk * (H1 / 4) + o4);
                acc[kk] = fmaf(d.x, w.x, fmaf(d.y, w.y, fmaf(d.z, w.z, fmaf(d.w, w.w, acc[kk]))));
            }
        }
        g = make_float4(acc[0], acc[1], acc[2], acc[3]);
    }
};
