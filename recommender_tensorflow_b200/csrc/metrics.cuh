// EVAL metrics of the heads, streamed on the device (dfm_metrics_* / dfm_evaluate, DESIGN.md §8.6).
//
// One batch of [n] logits, labels and optional weights becomes additions to a fixed-size metric state in device memory
// (dfm_metric_state, include/deepfm_b200.h) from which the host finishes every metric of both heads.  The logistic head
// follows TF 1.12 metrics_impl._confusion_matrix_at_thresholds / auc / precision / recall and head.py _eval_metric_ops:
//   p     = 1.f / (1.f + expf(-z))                 float32, IEEE division, full-precision expf (the head kernel's sigmoid)
//   th    = float32([0 - 1e-7] + [(i + 1) / 199 for i in range(198)] + [1 + 1e-7])    (TF's 200 thresholds, as constant())
//   bin   = #{t : p > t}  in [0, 200]              (branch-free binary search over the 200 sorted thresholds)
//   pos   = label > 0.5;  class = z > 0            (argmax([0, z]), a tie goes to class 0)
// and the sums Σw, Σw·y, Σw·p64, Σw·loss64 in float64, where p64 and loss64 = max(z, 0) - z y + log1p(exp(-|z|)) (the head
// kernel's sigmoid cross-entropy) are evaluated in double from the float32 logit, as the host's get_binary_metrics does.
// The squared head keeps Σw, Σw·y, Σw·z, Σw·(y - z)^2 only.  An unweighted call uses w = 1.
//
// Determinism: no float atomics.  A CTA owns the tiles b, b + grid, ... (grid depends on n alone), each thread keeps its
// partial sums in registers in a fixed sample order, the CTA reduces them with a fixed shuffle tree and writes ONE
// partial per CTA; metrics_reduce_kernel then sums the partials in CTA order and adds the batch to the state.  A rerun
// is bit-identical whatever the scheduling.
#pragma once
#include <stdint.h>

namespace metrics {

constexpr int BINS = 201;                 // DFM_METRIC_BINS: bins of the 200 thresholds
constexpr int KEYS = 2 * BINS;            // (label class, bin): [0][bin] negatives, [1][bin] positives
constexpr int NI = KEYS + 4;              // int64 fields per batch:   bin counts, tp fp fn correct
constexpr int ND = KEYS + 8;              // float64 fields per batch: bin weights, w_tp w_fp w_fn w_correct, 4 sums
constexpr int TILE = 512;                 // samples per CTA tile
constexpr int THREADS = 256;
constexpr int MAX_BLOCKS = 296;           // 2 CTAs per SM of the B200
constexpr int REDUCE_THREADS = 512;       // >= max(NI, ND)

struct Part {                              // one CTA's share of a batch
    long long i[NI];
    double d[ND];
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// grid = min(ceil(n / TILE), MAX_BLOCKS) CTAs of THREADS threads; part[blockIdx.x] receives the CTA's totals
__global__ void __launch_bounds__(THREADS) metrics_accumulate_kernel(const float* __restrict__ logits, const float* __restrict__ labels,
                                                                     const float* __restrict__ weights, int64_t n, int sq,
                                                                     Part* __restrict__ part) {
    __shared__ float s_th[256];            // thresholds, padded with +inf so that the search needs no bound check
    __shared__ int2 s_kw[TILE];            // per sample of the tile: key (-1: none), weight bits
    __shared__ double s_red[THREADS / 32][8];
    __shared__ long long s_redi[THREADS / 32][4];
    const int t = threadIdx.x;
    for (int j = t; j < 256; j += THREADS) {
        float v;
        if (j == 0) v = __double2float_rn(0.0 - 1e-7);
        else if (j < 199) v = __double2float_rn((double)j / 199.0);
        else if (j == 199) v = __double2float_rn(1.0 + 1e-7);
        else v = __int_as_float(0x7f800000);
        s_th[j] = v;
    }
    double sw = 0.0, swy = 0.0, swp = 0.0, swl = 0.0, wtp = 0.0, wfp = 0.0, wfn = 0.0, wok = 0.0;
    long long ctp = 0, cfp = 0, cfn = 0, cok = 0;
    long long c0 = 0, c1 = 0;              // keys t and t + THREADS of this thread
    double w0 = 0.0, w1 = 0.0;
    const int k0 = t, k1 = t + THREADS;
    const int64_t n_tiles = (n + TILE - 1) / TILE;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        __syncthreads();                   // s_th written / the previous tile's keys consumed
#pragma unroll 1
        for (int r = 0; r < TILE / THREADS; ++r) {
            const int j = r * THREADS + t;
            const int64_t i = tile * TILE + j;
            int key = -1;
            float w = 1.f;
            if (i < n) {
                const float z = logits[i], y = labels[i];
                if (weights) w = weights[i];
                const double wd = w, zd = z, yd = y;
                double pred, loss;
                if (sq) {
                    const double d = yd - zd;
                    pred = zd;
                    loss = d * d;
                } else {
                    const float p = 1.f / (1.f + expf(-z));
                    int c = 0;
#pragma unroll
                    for (int s = 128; s; s >>= 1) c = (p > s_th[c + s - 1]) ? c + s : c;
                    const bool pos = y > 0.5f, cls = z > 0.f;
                    key = (pos ? BINS : 0) + c;
                    ctp += cls && pos; cfp += cls && !pos; cfn += !cls && pos; cok += cls == pos;
                    wtp += (cls && pos) ? wd : 0.0; wfp += (cls && !pos) ? wd : 0.0;
                    wfn += (!cls && pos) ? wd : 0.0; wok += (cls == pos) ? wd : 0.0;
                    pred = 1.0 / (1.0 + exp(-zd));
                    loss = fmax(zd, 0.0) - zd * yd + log1p(exp(-fabs(zd)));
                }
                sw += wd; swy += wd * yd; swp += wd * pred; swl += wd * loss;
            }
            s_kw[j] = make_int2(key, __float_as_int(w));
        }
        __syncthreads();
        if (!sq) {
            // the (class, bin) totals: thread t owns keys t and t + THREADS and scans the tile in sample order
#pragma unroll 4
            for (int j = 0; j < TILE; ++j) {
                const int2 kw = s_kw[j];
                if (kw.x == k0) { ++c0; w0 += (double)__int_as_float(kw.y); }
                if (kw.x == k1) { ++c1; w1 += (double)__int_as_float(kw.y); }
            }
        }
    }
    Part& out = part[blockIdx.x];
    if (k0 < KEYS) { out.i[k0] = c0; out.d[k0] = w0; }
    if (k1 < KEYS) { out.i[k1] = c1; out.d[k1] = w1; }
    double v[8] = {wtp, wfp, wfn, wok, sw, swy, swp, swl};
    long long c[4] = {ctp, cfp, cfn, cok};
    const int lane = t & 31, warp = t >> 5;
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = warp_sum(v[q]);
#pragma unroll
    for (int q = 0; q < 4; ++q) c[q] = warp_sum(c[q]);
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) s_red[warp][q] = v[q];
#pragma unroll
        for (int q = 0; q < 4; ++q) s_redi[warp][q] = c[q];
    }
    __syncthreads();
    if (t < 8) {
        double a = 0.0;
        for (int wi = 0; wi < THREADS / 32; ++wi) a += s_red[wi][t];
        out.d[KEYS + t] = a;
    } else if (t < 12) {
        long long a = 0;
        for (int wi = 0; wi < THREADS / 32; ++wi) a += s_redi[wi][t - 8];
        out.i[KEYS + t - 8] = a;
    }
}

// one CTA: the partials of the batch summed in CTA order, then added to the state (st_i: n followed by the NI int64
// fields, st_d: the ND float64 fields of dfm_metric_state).  Every field of every partial is written (zeros for what
// the squared head does not form).
__global__ void __launch_bounds__(REDUCE_THREADS) metrics_reduce_kernel(const Part* __restrict__ part, int n_parts, int64_t n,
                                                                        long long* __restrict__ st_i, double* __restrict__ st_d) {
    const int t = threadIdx.x;
    if (t == 0) st_i[0] += n;
    if (t < NI) {
        long long a = 0;
        for (int b = 0; b < n_parts; ++b) a += part[b].i[t];
        st_i[1 + t] += a;
    }
    if (t < ND) {
        double a = 0.0;
        for (int b = 0; b < n_parts; ++b) a += part[b].d[t];
        st_d[t] += a;
    }
}

}  // namespace metrics
