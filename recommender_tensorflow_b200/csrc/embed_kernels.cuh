// Input-path, embedding/linear lookup, FM interaction, sparse-gradient reduction and sparse
// optimizer kernels (K1, K2, K5, K6 of SURVEY.md §8a).  Hand-written for sm_100a.
#pragma once
#include "dfm_types.cuh"
#include "farmhash.cuh"
#include "replay.cuh"

__device__ __forceinline__ void add4(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }

// payload of a (row, lookup) sort pair: sample index and value slot of the lookup, packed so that neither a division
// nor the slot count is needed to take it apart (at most 256 value slots per sample, 2^24 samples per batch)
constexpr int PAYLOAD_SLOT_BITS = 8;
__host__ __device__ __forceinline__ uint32_t payload_pack(uint32_t b, uint32_t slot) { return (b << PAYLOAD_SLOT_BITS) | slot; }
__host__ __device__ __forceinline__ uint32_t payload_sample(uint32_t v) { return v >> PAYLOAD_SLOT_BITS; }
__host__ __device__ __forceinline__ uint32_t payload_slot(uint32_t v) { return v & ((1u << PAYLOAD_SLOT_BITS) - 1u); }

// Claim table of one step: 2 bits per slot (slot = global row & mask), 01 = looked up once in the batch, 11 = more than
// once.  transform_kernel marks, fused_rows_kernel (applies the gradient of once-only rows itself) and row_apply_kernel
// (skips them) test; a slot shared by two rows of the batch reads "more than once" for both, which is always safe.
__device__ __forceinline__ void claim_mark(uint32_t* __restrict__ claim, uint32_t mask, uint32_t row) {
    const uint32_t s = row & mask, sh = (s & 15u) * 2u;
    const uint32_t old = atomicOr(claim + (s >> 4), 1u << sh);
    if ((old >> sh) & 1u) atomicOr(claim + (s >> 4), 2u << sh);
}
__device__ __forceinline__ bool claim_once(const uint32_t* __restrict__ claim, uint32_t mask, uint32_t row) {
    const uint32_t s = row & mask;
    return ((__ldg(claim + (s >> 4)) >> ((s & 15u) * 2u)) & 3u) == 1u;
}

// =============================================================================================
// optimizer arithmetic, in the float32 op order of the TF-1.12 kernels (SURVEY.md A.3)
// =============================================================================================
__device__ __forceinline__ float adam_upd(float m, float v, float alpha, float eps) {
    return __fdiv_rn(__fmul_rn(alpha, m), __fadd_rn(__fsqrt_rn(v), eps));
}
// python/training/adam.py::_apply_sparse_shared on one (already de-duplicated) touched element
__device__ __forceinline__ void adam_sparse_apply(float& w, float& m, float& v, float g, const OptDev& o) {
    m = __fadd_rn(__fmul_rn(m, o.b1), __fmul_rn(g, o.omb1));
    v = __fadd_rn(__fmul_rn(v, o.b2), __fmul_rn(__fmul_rn(g, g), o.omb2));
    w = __fsub_rn(w, adam_upd(m, v, o.alpha, o.eps));
}
// core/kernels/training_ops.cc ApplyAdam (dense)
__device__ __forceinline__ void adam_dense_apply(float& w, float& m, float& v, float g, const OptDev& o) {
    m = __fadd_rn(m, __fmul_rn(__fsub_rn(g, m), o.omb1));
    v = __fadd_rn(v, __fmul_rn(__fsub_rn(__fmul_rn(g, g), v), o.omb2));
    w = __fsub_rn(w, __fdiv_rn(__fmul_rn(m, o.alpha), __fadd_rn(__fsqrt_rn(v), o.eps)));
}
// Adagrad / FTRL(lr_power=-0.5, l1=l2=0) / SGD.  s1 = accumulator, s2 = FTRL "linear" slot.
__device__ __forceinline__ void other_apply(float& w, float& s1, float& s2, float g, const OptDev& o) {
    if (o.kind == DFM_OPT_ADAGRAD) {
        s1 = __fadd_rn(s1, __fmul_rn(g, g));
        w = __fsub_rn(w, __fdiv_rn(__fmul_rn(o.lr, g), __fsqrt_rn(s1)));
    } else if (o.kind == DFM_OPT_FTRL) {
        float na = __fadd_rn(s1, __fmul_rn(g, g));
        float sna = __fsqrt_rn(na), sa = __fsqrt_rn(s1);
        float t1 = __fadd_rn(s2, g);
        float t2 = __fmul_rn(__fdiv_rn(__fsub_rn(sna, sa), o.lr), w);
        s2 = __fsub_rn(t1, t2);
        w = __fdiv_rn(-s2, __fdiv_rn(sna, o.lr));
        s1 = na;
    } else if (o.kind == DFM_OPT_RMSPROP) {   // training_ops.cc ApplyRMSProp: s1 = ms, s2 = mom, b2 = rho, b1 = momentum
        s1 = __fadd_rn(s1, __fmul_rn(__fsub_rn(__fmul_rn(g, g), s1), __fsub_rn(1.0f, o.b2)));
        s2 = __fadd_rn(__fmul_rn(s2, o.b1), __fdiv_rn(__fmul_rn(g, o.lr), __fsqrt_rn(__fadd_rn(s1, o.eps))));
        w = __fsub_rn(w, s2);
    } else {  // SGD
        w = __fsub_rn(w, __fmul_rn(o.lr, g));
    }
}
__device__ __forceinline__ void sparse_apply(float& w, float& s1, float& s2, float g, const OptDev& o) {
    if (o.kind == DFM_OPT_ADAM) adam_sparse_apply(w, s1, s2, g, o);
    else other_apply(w, s1, s2, g, o);
}
__device__ __forceinline__ void dense_apply(float& w, float& s1, float& s2, float g, const OptDev& o) {
    if (o.kind == DFM_OPT_ADAM) adam_dense_apply(w, s1, s2, g, o);
    else other_apply(w, s1, s2, g, o);
}

// TF's AdamOptimizer applies `m *= b1; v *= b2; w -= alpha_t m/(sqrt(v)+eps)` to EVERY row at every
// step (non-lazy, SURVEY.md §7 hard part 1).  A row whose last materialised step is `last` is
// brought up to step `upto` by replaying exactly those skipped steps in registers.  alpha[] holds
// the per-step alpha_t history.  Once an update is too small to change w in float32 all later ones
// are too (|update| shrinks by >= 8% per step), so the loop stops early and only m, v keep decaying.
__device__ __forceinline__ void adam_replay(float& w, float& m, float& v, int last, int upto,
                                            const float* __restrict__ alpha, const OptDev& o) {
    if (m == 0.f && v == 0.f) return;
    int tau = last + 1;
    for (; tau <= upto; ++tau) {
        m = __fmul_rn(m, o.b1);
        v = __fmul_rn(v, o.b2);
        float wn = __fsub_rn(w, adam_upd(m, v, __ldg(alpha + tau), o.eps));
        bool same = (wn == w);
        w = wn;
        if (same && o.safe_early) { ++tau; break; }
    }
    int rem = upto - tau + 1;
    if (rem > 0) {
        if (rem <= 256) {
            for (int j = 0; j < rem; ++j) { m = __fmul_rn(m, o.b1); v = __fmul_rn(v, o.b2); }
        } else {
            m = (float)((double)m * pow((double)o.b1, (double)rem));
            v = (float)((double)v * pow((double)o.b2, (double)rem));
        }
    }
}

// Replay of a whole float4 lane slice in ONE loop (shared trip count, 4-way ILP) with MUFU-based
// sqrt / reciprocal: the replayed updates add up to at most ~1e-2 and each carries <= 2^-21 relative
// error, i.e. < 1e-8 absolute on w - far inside the 1e-5 parity bar - while the exact IEEE sequence
// costs ~5x more instructions and made the catch-up compute-bound on Criteo-sized tables.
__device__ __forceinline__ float fast_upd(float m, float v, float alpha, float eps) {
    float sq, rc;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(v));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(sq + eps));
    return alpha * m * rc;
}
__device__ __forceinline__ void adam_replay4(float4& w, float4& m, float4& v, int last, int upto,
                                             const float* __restrict__ alpha, const OptDev& o) {
    int tau = last + 1;
    for (; tau <= upto; ++tau) {
        const float a = __ldg(alpha + tau);
        m.x *= o.b1; m.y *= o.b1; m.z *= o.b1; m.w *= o.b1;
        v.x *= o.b2; v.y *= o.b2; v.z *= o.b2; v.w *= o.b2;
        float4 wn;
        wn.x = w.x - fast_upd(m.x, v.x, a, o.eps); wn.y = w.y - fast_upd(m.y, v.y, a, o.eps);
        wn.z = w.z - fast_upd(m.z, v.z, a, o.eps); wn.w = w.w - fast_upd(m.w, v.w, a, o.eps);
        const bool same = wn.x == w.x && wn.y == w.y && wn.z == w.z && wn.w == w.w;
        w = wn;
        if (same && o.safe_early) { ++tau; break; }
    }
    int rem = upto - tau + 1;
    if (rem > 0) {
        float d1, d2;
        if (rem <= 64) {
            d1 = 1.f; d2 = 1.f;
            for (int j = 0; j < rem; ++j) { d1 *= o.b1; d2 *= o.b2; }
        } else {
            d1 = (float)pow((double)o.b1, (double)rem);
            d2 = (float)pow((double)o.b2, (double)rem);
        }
        m.x *= d1; m.y *= d1; m.z *= d1; m.w *= d1;
        v.x *= d2; v.y *= d2; v.z *= d2; v.w *= d2;
    }
}

__device__ __forceinline__ void adam_replay1(float& w, float& m, float& v, int last, int upto,
                                             const float* __restrict__ alpha, const OptDev& o) {
    if (m == 0.f && v == 0.f) return;
    float4 w4 = make_float4(w, 0.f, 0.f, 0.f), m4 = make_float4(m, 0.f, 0.f, 0.f), v4 = make_float4(v, 1.f, 1.f, 1.f);
    adam_replay4(w4, m4, v4, last, upto, alpha, o);
    w = w4.x; m = m4.x; v = v4.x;
}

// Both optimizer groups of one step as the row kernels see them.  Every kernel that reads a table row (gather, serve)
// or rewrites it (row_update, tiny_update, flush) replays the non-lazy Adam decay of that row IN REGISTERS from the
// stored state (replay.cuh); only the kernels that rewrite the row anyway store the result.  There is no separate
// catch-up pass over the touched rows any more.
struct RowReplay {
    ReplayTab rd, rl;     // embedding / linear group
    int upto;             // rows are brought to this step; < 0: nothing to replay
    int emb_adam, lin_adam;
    int same;             // both groups share hyper-parameters: one coefficient set serves both
};

// w, m, v: this lane's float4 slice of the embedding row and its Adam slots; lr = {lin w, lin m, lin v, last_step}.
// lin_lane: this lane also owns the linear weight.  Afterwards lr.w = upto (callers that store the row store it).
__device__ __forceinline__ void replay_row(float4& w, float4& m, float4& v, float4& lr, bool lin_lane, const RowReplay& rr,
                                           const ReplayStep& rs, const OptDev& od, const OptDev& ol) {
    const int last = __float_as_int(lr.w);
    if (rr.upto < 0 || last >= rr.upto) return;
    bool lin_done = !(rr.lin_adam && lin_lane);
    if (rr.emb_adam) {
        if (rr.rd.closed) {
            const ReplayCoef c = replay_coef(rr.rd, rs, last);
            replay_elem(w.x, m.x, v.x, c, od.eps); replay_elem(w.y, m.y, v.y, c, od.eps);
            replay_elem(w.z, m.z, v.z, c, od.eps); replay_elem(w.w, m.w, v.w, c, od.eps);
            if (!lin_done && rr.same) { replay_elem(lr.x, lr.y, lr.z, c, ol.eps); lin_done = true; }
        } else {
            adam_replay4(w, m, v, last, rr.upto, rr.rd.alpha, od);
        }
    }
    if (!lin_done) {
        if (rr.rl.closed) {
            const ReplayStep sl = (rr.same && rr.rd.closed) ? rs : replay_step_load(rr.rl, rr.upto);
            const ReplayCoef c = replay_coef(rr.rl, sl, last);
            replay_elem(lr.x, lr.y, lr.z, c, ol.eps);
        } else {
            adam_replay1(lr.x, lr.y, lr.z, last, rr.upto, rr.rl.alpha, ol);
        }
    }
    lr.w = __int_as_float(rr.upto);
}

// this lane's slice of an embedding row + the linear weight, as of step rr.upto (read-only: nothing is written back)
__device__ __forceinline__ void load_row_current(const Table& tb, size_t row, int sub, bool has_emb, const RowReplay& rr,
                                                 const ReplayStep& rs, const OptDev& od, const OptDev& ol, float4& w, float& lw) {
    float4 lr = __ldg(tab_lin(tb, row));
    w = has_emb ? __ldg(tab_w(tb, row) + sub) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (rr.upto >= 0 && __float_as_int(lr.w) < rr.upto) {
        float4 m = w, v = w;
        if (rr.emb_adam) { m = __ldg(tab_s1(tb, row) + sub); v = __ldg(tab_s2(tb, row) + sub); }
        replay_row(w, m, v, lr, sub == 0, rr, rs, od, ol);
    }
    lw = lr.x;
}

// =============================================================================================
// K1: feature-column transforms -> ids [B, dc] + sort keys (global row index) + payload
// =============================================================================================
// h % nb by Barrett reduction: q = floor(h * floor(2^64 / nb) / 2^64) is the quotient or one less (h / nb - h rcp / 2^64 < 1),
// so one conditional subtraction makes the remainder exact; the generic 64-bit modulo is a ~150-instruction routine and
// was a third of transform_kernel's instruction stream on the Criteo-shaped batch (26 hashed columns).
__device__ __forceinline__ uint64_t mod_buckets(uint64_t h, const ColDev& c) {
    if (c.nb_rcp == 0) return h % c.nb;
    uint64_t r = h - __umul64hi(h, c.nb_rcp) * c.nb;
    return r >= c.nb ? r - c.nb : r;
}
// Vocabulary lookup through the column's open-addressing table (TF-1.12 index_table_from_tensor / _from_file: a HashTable
// from key to index, unknown keys -> OOV bucket or default_value).  Slot = {key, index}; string keys are their
// Fingerprint64 (the OOV bucket needs it anyway) and a fingerprint match is confirmed by comparing the bytes, so the
// result is exact; int keys are the sign-extended value.  Linear probing from vocab_mix(key); the table is at most half
// full, so a probe ends at an empty slot.
__device__ __forceinline__ int32_t vocab_probe(const BatchPtrs& bp, const ColDev& c, int f, int b,
                                            const uint8_t* __restrict__ voc_bytes, const int32_t* __restrict__ voc_offs) {
    uint64_t key, fp = 0;
    const uint8_t* p = nullptr;
    int len = 0;
    if (c.dtype == DFM_STRING) {
        const int32_t* off = bp.off[f];
        const int s = off[b];
        len = off[b + 1] - s;
        if (len <= 0) return -1;
        p = reinterpret_cast<const uint8_t*>(bp.cat[f]) + s;
        fp = fh::fp64_mem(p, len);
        key = fp & c.fp_mask;
    } else {
        const int32_t v = reinterpret_cast<const int32_t*>(bp.cat[f])[b];
        if (v == -1) return -1;
        key = (uint64_t)(int64_t)v;
    }
    for (uint32_t i = (uint32_t)vocab_mix(key) & c.tab_mask;; i = (i + 1) & c.tab_mask) {
        const longlong2 e = __ldg(c.vtab + i);
        if (e.y < 0) break;
        if ((uint64_t)e.x != key) continue;
        if (c.dtype != DFM_STRING) return (int32_t)e.y;
        const int vs = voc_offs[c.voc_off + (int)e.y], ve = voc_offs[c.voc_off + (int)e.y + 1];
        if (ve - vs != len) continue;
        bool eq = true;
        for (int q = 0; q < len && eq; ++q) eq = voc_bytes[vs + q] == p[q];
        if (eq) return (int32_t)e.y;
    }
    if (c.num_oov > 0) {
        if (c.dtype != DFM_STRING) {        // AsString(key), as the hashed int column does
            uint64_t lo, hi;
            const int n = fh::itoa16((int32_t)(int64_t)key, lo, hi);
            fp = fh::fp64_short(lo, hi, n);
        }
        return c.voc_cnt + (int32_t)(fp % (uint64_t)c.num_oov);
    }
    return c.dflt;
}

// VTAB: the model has vocabulary columns looked up through a hash table (vocab_probe); otherwise every vocabulary
// column is a short string list and is scanned.
template <bool VTAB>
__device__ __forceinline__ int32_t transform_one(const BatchPtrs& bp, const ColDev& c, int f, int b,
                                                 const float* __restrict__ bounds,
                                                 const uint8_t* __restrict__ voc_bytes,
                                                 const int32_t* __restrict__ voc_offs, int* err) {
    switch (c.kind) {
        case DFM_COL_HASH: {
            if (c.dtype == DFM_STRING) {
                const int32_t* off = bp.off[f];
                int s = off[b], e = off[b + 1];
                int len = e - s;
                if (len <= 0) return -1;
                uint64_t h = fh::fp64_mem(reinterpret_cast<const uint8_t*>(bp.cat[f]) + s, len);
                return (int32_t)mod_buckets(h, c);
            } else {
                int32_t v = reinterpret_cast<const int32_t*>(bp.cat[f])[b];
                if (v == -1) return -1;
                uint64_t lo, hi;
                int len = fh::itoa16(v, lo, hi);
                return (int32_t)mod_buckets(fh::fp64_short(lo, hi, len), c);
            }
        }
        case DFM_COL_BUCKETIZED: {
            float x = c.dtype == DFM_FLOAT32 ? reinterpret_cast<const float*>(bp.cat[f])[b]
                                             : (float)reinterpret_cast<const int32_t*>(bp.cat[f])[b];
            int cnt = 0;
            for (int j = 0; j < c.bnd_cnt; ++j) cnt += (bounds[c.bnd_off + j] <= x) ? 1 : 0;
            return cnt;
        }
        case DFM_COL_VOCAB: {
            if (VTAB && c.vtab) return vocab_probe(bp, c, f, b, voc_bytes, voc_offs);
            const int32_t* off = bp.off[f];
            int s = off[b], e = off[b + 1];
            int len = e - s;
            if (len <= 0) return -1;
            const uint8_t* p = reinterpret_cast<const uint8_t*>(bp.cat[f]) + s;
            for (int j = 0; j < c.voc_cnt; ++j) {
                int vs = voc_offs[c.voc_off + j], ve = voc_offs[c.voc_off + j + 1];
                if (ve - vs != len) continue;
                bool eq = true;
                for (int q = 0; q < len; ++q) eq = eq && (voc_bytes[vs + q] == p[q]);
                if (eq) return j;
            }
            if (c.num_oov > 0) return c.voc_cnt + (int32_t)(fh::fp64_mem(p, len) % (uint64_t)c.num_oov);
            return c.dflt;
        }
        default: {  // identity
            int32_t v = reinterpret_cast<const int32_t*>(bp.cat[f])[b];
            if (v == -1) return -1;
            if (v < 0 || (uint64_t)v >= c.nb) {
                if (c.dflt >= 0) return c.dflt;      // default_value
                atomicOr(err, 1); return -1;
            }
            return v;
        }
    }
}

// Crossed column (TF-1.12 sparse_cross_hashed, reached through tf.feature_column.crossed_column): slot j of sample b is
// one combination of constituent value slots, j read as a mixed-radix number over the constituents' widths (first key
// most significant, the order of TF's product iterator).  f(v) per constituent, chained with FingerprintCat64 from the
// hash key (core/kernels/sparse_cross_op.cc HashCrosser):
//   raw string -> Fingerprint64(bytes);  raw int32 -> (uint64)(int64)v;  categorical -> (uint64)(int64)id
// Absent values make the combination absent (-1): padding slots ('' / -1) of a multivalent raw key (a SparseTensor in
// TF), and ids a categorical key drops (empty string, identity -1).  A single-valued raw key is a dense tensor in TF and
// drops nothing.  A vocabulary key without OOV buckets maps an unknown string to the id -1, which TF keeps and crosses.
// Only the CROSS instantiation of transform_kernel contains this code, so models without crossed columns run the
// kernel as it was.  The key loop is not unrolled (transform_one is inlined into it once).
template <bool VTAB>
__device__ __forceinline__ int32_t transform_cross(const BatchPtrs& bp, const ColDev* __restrict__ cols, int f, int b,
                                                   int j, const float* __restrict__ bounds,
                                                   const uint8_t* __restrict__ voc_bytes,
                                                   const int32_t* __restrict__ voc_offs, int* err) {
    const ColDev& c = cols[f];
    uint64_t h = c.hash_key;
    int stride = c.width;
    const int n_keys = c.n_keys;
#pragma unroll 1
    for (int i = 0; i < n_keys; ++i) {
        {
            const int s = c.keys[i];
            const ColDev k = cols[s];
            stride /= k.width;
            const int d = j / stride;
            j -= d * stride;
            const int vi = b * k.width + d;
            uint64_t v;
            if (k.kind == DFM_COL_RAW) {
                if (k.dtype == DFM_STRING) {
                    const int32_t* off = bp.off[s];
                    const int a = off[vi], e = off[vi + 1];
                    if (e <= a && k.width > 1) return -1;
                    v = fh::fp64_mem(reinterpret_cast<const uint8_t*>(bp.cat[s]) + a, e - a);
                } else {
                    const int32_t x = reinterpret_cast<const int32_t*>(bp.cat[s])[vi];
                    if (x == -1 && k.width > 1) return -1;
                    v = (uint64_t)(int64_t)x;
                }
            } else {
                if (k.kind == DFM_COL_VOCAB && (k.dtype == DFM_STRING ? bp.off[s][vi + 1] <= bp.off[s][vi]
                                                                      : reinterpret_cast<const int32_t*>(bp.cat[s])[vi] == -1))
                    return -1;
                const int32_t id = transform_one<VTAB>(bp, k, s, vi, bounds, voc_bytes, voc_offs, err);
                if (id < 0 && k.kind != DFM_COL_VOCAB) return -1;
                v = (uint64_t)(int64_t)id;
            }
            h = fh::fp_cat64(h, v);
        }
    }
    return (int32_t)mod_buckets(h, cols[f]);
}

// One block = TILE consecutive samples x all value slots (a single-valued column has one slot, a multivalent
// column `width`).  Phase 1: work item w -> (slot w / TILE, sample w % TILE), so a warp reads 32 consecutive
// samples of ONE column (coalesced for single-valued columns, uniform column kind) and the columns of a sample are
// transformed in parallel by different warps (a hashed string column costs ~100x an identity column).
// Phase 2 writes ids / keys / payload sample-major: ids [B, n_slots], payload = payload_pack(b, slot).
// CROSS: the model has crossed columns (transform_cross above).  VTAB: it has hash-table vocabularies (vocab_probe).
template <int TILE, bool CROSS = false, bool VTAB = false>
__global__ void __launch_bounds__(256) transform_kernel(BatchPtrs bp, const ColDev* __restrict__ cols,
                                                        const float* __restrict__ bounds,
                                                        const uint8_t* __restrict__ voc_bytes,
                                                        const int32_t* __restrict__ voc_offs, int B, int n_slots,
                                                        const int32_t* __restrict__ slot_col, const int32_t* __restrict__ slot_j,
                                                        const uint32_t* __restrict__ row_off, uint32_t R,
                                                        int32_t* __restrict__ ids, uint32_t* __restrict__ keys,
                                                        uint32_t* __restrict__ vals, int* err,
                                                        const int32_t* __restrict__ key_slot, int n_key_slots,
                                                        uint32_t* __restrict__ claim = nullptr, uint32_t claim_mask = 0) {
    extern __shared__ int32_t sid[];  // [TILE][n_slots]
    const int b0 = blockIdx.x * TILE;
    const int nb = min(TILE, B - b0);
    for (int w = threadIdx.x; w < TILE * n_slots; w += blockDim.x) {
        const int slot = w / TILE, t = w - slot * TILE;
        if (t < nb) {
            const int f = slot_col ? slot_col[slot] : slot;      // null slot tables: every column single-valued
            ColDev c = cols[f];
            const int j = slot_col ? slot_j[slot] : 0;
            const int vi = slot_col ? (b0 + t) * c.width + j : b0 + t;
            sid[t * n_slots + slot] = CROSS && c.kind == DFM_COL_CROSSED
                                          ? transform_cross<VTAB>(bp, cols, f, b0 + t, j, bounds, voc_bytes, voc_offs, err)
                                          : transform_one<VTAB>(bp, c, f, vi, bounds, voc_bytes, voc_offs, err);
        }
    }
    __syncthreads();
    const int nloc = nb * n_slots;
    const int64_t g0 = (int64_t)b0 * n_slots;
    // four items per thread and round: the claim marks are L2 atomics whose old value decides about a second one, and a
    // warp stalls at the first use of a pending result, so the first atomics of a round are all issued before any is tested
    for (int w0 = threadIdx.x; w0 < nloc; w0 += 4 * blockDim.x) {
        uint32_t crow[4], cold[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int w = w0 + u * blockDim.x;
            crow[u] = 0xffffffffu; cold[u] = 0;
            if (w < nloc) {
                int32_t id = sid[w];
                int slot = w % n_slots;
                ids[g0 + w] = id;
                const uint32_t grow = id >= 0 ? row_off[slot_col ? slot_col[slot] : slot] + (uint32_t)id : R;
                if (claim && id >= 0) {
                    const uint32_t s = grow & claim_mask;
                    crow[u] = s;
                    cold[u] = atomicOr(claim + (s >> 4), 1u << ((s & 15u) * 2u));
                }
                if (keys) {
                    // key_slot: only the listed slots go through the sort (tiny-vocabulary columns are reduced densely, see
                    // tiny_reduce_kernel); their pairs are packed [sample][key slot], the payload keeps the full-slot numbering
                    int64_t at = g0 + w;
                    if (key_slot) {
                        const int ks = key_slot[slot];
                        at = ks >= 0 ? (int64_t)(b0 + w / n_slots) * n_key_slots + ks : -1;
                    }
                    if (at >= 0) {
                        keys[at] = grow;
                        vals[at] = payload_pack((uint32_t)(b0 + w / n_slots), (uint32_t)slot);
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t sh = (crow[u] & 15u) * 2u;
            if (crow[u] != 0xffffffffu && ((cold[u] >> sh) & 1u)) atomicOr(claim + (crow[u] >> 4), 2u << sh);
        }
    }
}

static __global__ void fingerprint_kernel(const uint8_t* __restrict__ bytes, const int32_t* __restrict__ offs, int64_t n,
                                   uint64_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = fh::fp64_mem(bytes + offs[i], offs[i + 1] - offs[i]);
}

// =============================================================================================
// segments of the sorted (row, lookup) list
// =============================================================================================
__device__ __forceinline__ void seg_heads(const uint32_t* __restrict__ keys, int64_t i, uint32_t R, bool& rh, bool& ph) {
    uint32_t k = keys[i];
    uint32_t prev = i > 0 ? keys[i - 1] : 0xffffffffu;
    bool valid = k < R;
    rh = valid && (i == 0 || k != prev);
    ph = valid && (rh || (i % PIECE_C) == 0);
}

static __global__ void seg_flag_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t R,
                                unsigned long long* __restrict__ flags, SegCounts* __restrict__ cnt) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool rh, ph;
    seg_heads(keys, i, R, rh, ph);
    flags[i] = ((unsigned long long)(rh ? 1u : 0u) << 32) | (ph ? 1u : 0u);
    uint32_t k = keys[i];
    if (k >= R) {
        if (i == 0 || keys[i - 1] < R) cnt->n_valid = (uint32_t)i;
    } else if (i == n - 1) {
        cnt->n_valid = (uint32_t)n;
    }
}

static __global__ void seg_fill_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t n, uint32_t R,
                                const unsigned long long* __restrict__ scanned,
                                const unsigned long long* __restrict__ total, SegCounts* __restrict__ cnt,
                                uint32_t* __restrict__ row_start, uint32_t* __restrict__ row_piece0,
                                uint32_t* __restrict__ piece_start, uint32_t* __restrict__ urow, uint32_t* __restrict__ uval) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        uint32_t U = (uint32_t)(*total >> 32), P = (uint32_t)(*total & 0xffffffffu);
        uint32_t nv = cnt->n_valid;
        cnt->n_rows = U;
        cnt->n_pieces = P;
        cnt->n_hot = 0;
        row_start[U] = nv;
        row_piece0[U] = P;
        piece_start[P] = nv;
    }
    if (i >= n) return;
    bool rh, ph;
    seg_heads(keys, i, R, rh, ph);
    if (!ph) return;
    unsigned long long s = scanned[i];
    uint32_t ridx = (uint32_t)(s >> 32), pidx = (uint32_t)(s & 0xffffffffu);
    piece_start[pidx] = (uint32_t)i;
    if (rh) {
        row_start[ridx] = (uint32_t)i;
        row_piece0[ridx] = pidx;
        urow[ridx] = keys[i];      // compact (coalesced) copies of the row id and of the first lookup of every
        uval[ridx] = vals[i];      // unique row: they remove one dependent-load level from the row kernels
    }
}

// Two-launch segment builder (flags + scan + fill of the three kernels above were 5 launches):
//   seg_count_kernel  every tile of 2048 sorted pairs counts its row heads / piece heads; the LAST block to finish
//                     turns the per-tile counts into exclusive prefixes (one thread walks 32 tiles at a time) and
//                     closes the lists (totals, number of valid lookups, sentinels)
//   seg_fill_kernel2  every tile re-derives its flags, scans them inside the block and writes row_start / row_piece0 /
//                     piece_start / urow / uval (+ pos_row for the sharded requester)
// A single-launch version with decoupled look-back measured 67 us for 832 tiles (the chain starts cold: every tile
// publishes at the same moment), this one needs no spinning.  The element count may live in device memory (n_dev).
constexpr int SB_ITEMS = 8, SB_TILE = 256 * SB_ITEMS;
static_assert(SB_ITEMS == 8, "seg_tile_flags loads a thread's run as two uint4");

__device__ __forceinline__ void seg_tile_flags(const uint32_t* __restrict__ keys, int64_t i0, int64_t n, uint32_t R, uint32_t (&k)[SB_ITEMS],
                                               uint32_t& rows, uint32_t& pieces, uint32_t& rmask, uint32_t& pmask, uint32_t& vmask) {
    if (i0 + SB_ITEMS <= n) {        // a thread's run is 32 contiguous, 32-byte aligned bytes: two vector loads instead of eight scalar ones
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(keys + i0)), b = __ldg(reinterpret_cast<const uint4*>(keys + i0) + 1);
        k[0] = a.x; k[1] = a.y; k[2] = a.z; k[3] = a.w; k[4] = b.x; k[5] = b.y; k[6] = b.z; k[7] = b.w;
    } else {
#pragma unroll
        for (int j = 0; j < SB_ITEMS; ++j) k[j] = (i0 + j < n) ? keys[i0 + j] : 0xffffffffu;
    }
    uint32_t prev = (i0 > 0 && i0 < n) ? keys[i0 - 1] : 0xffffffffu;
    rows = 0; pieces = 0; rmask = 0; pmask = 0; vmask = 0;
#pragma unroll
    for (int j = 0; j < SB_ITEMS; ++j) {
        const int64_t i = i0 + j;
        const bool valid = i < n && k[j] < R;
        const bool rh = valid && (i == 0 || k[j] != prev);
        const bool ph = valid && (rh || (i % PIECE_C) == 0);
        rows += rh; pieces += ph;
        rmask |= (uint32_t)rh << j; pmask |= (uint32_t)ph << j; vmask |= (uint32_t)valid << j;
        prev = k[j];
    }
}

static __global__ void __launch_bounds__(256) seg_count_kernel(const uint32_t* __restrict__ keys, int64_t n_host, const uint32_t* __restrict__ n_dev,
                                                        uint32_t R, unsigned long long* tile_cnt, unsigned int* __restrict__ ticket,
                                                        SegCounts* __restrict__ cnt, uint32_t* __restrict__ row_start,
                                                        uint32_t* __restrict__ row_piece0, uint32_t* __restrict__ piece_start) {
    __shared__ unsigned long long wsum[8];
    __shared__ uint32_t winv[8];
    __shared__ bool last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n = n_dev ? (int64_t)*reinterpret_cast<const volatile uint32_t*>(n_dev) : n_host;
    const int64_t tiles = (n + SB_TILE - 1) / SB_TILE;
    const int64_t tile = blockIdx.x;
    if (tile < tiles) {
        uint32_t k[SB_ITEMS], rows, pieces, rmask, pmask, vmask;
        seg_tile_flags(keys, tile * SB_TILE + (int64_t)tid * SB_ITEMS, n, R, k, rows, pieces, rmask, pmask, vmask);
        unsigned long long v = ((unsigned long long)rows << 32) | pieces;
        // lookups without a row (keys >= R, sorted last): counted here so that the closing thread needs no binary search
        // over the keys (21 dependent global loads, ~8 of this kernel's 20 us)
        const int64_t i0 = tile * SB_TILE + (int64_t)tid * SB_ITEMS;
        uint32_t inval = (uint32_t)max((int64_t)0, min((int64_t)SB_ITEMS, n - i0)) - __popc(vmask);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) { v += __shfl_xor_sync(0xffffffffu, v, o); inval += __shfl_xor_sync(0xffffffffu, inval, o); }
        if (lane == 0) { wsum[warp] = v; winv[warp] = inval; }
        __syncthreads();
        if (tid == 0) {
            unsigned long long t = 0;
            uint32_t iv = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) { t += wsum[w]; iv += winv[w]; }
            tile_cnt[tile] = t;
            if (iv) atomicAdd(ticket + 1, iv);
        }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last block: exclusive prefix over the tile counts, 8 tiles per thread and 2048 per round (one warp walking 32
    // tiles at a time made 26 dependent L2 round trips for the 832 tiles of a 1.7 M pair list: most of this kernel's time)
    __shared__ unsigned long long ptot[9];
    unsigned long long run = 0;
    for (int64_t c0 = 0; c0 < tiles; c0 += 256 * 8) {
        const int64_t tb = c0 + (int64_t)tid * 8;
        unsigned long long c[8], sum = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { c[j] = tb + j < tiles ? __ldcg(tile_cnt + tb + j) : 0ull; sum += c[j]; }
        unsigned long long inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long x = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += x;
        }
        if (lane == 31) ptot[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long w = lane < 8 ? ptot[lane] : 0ull;
            unsigned long long winc = w;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                const unsigned long long x = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += x;
            }
            if (lane < 8) ptot[lane] = winc - w;
            if (lane == 7) ptot[8] = winc;
        }
        __syncthreads();
        unsigned long long ex = run + ptot[warp] + (inc - sum);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (tb + j < tiles) { tile_cnt[tb + j] = ex; ex += c[j]; }
        run += ptot[8];
        __syncthreads();
    }
    if (tid != 0) return;
    {
        const uint32_t Ur = (uint32_t)(run >> 32), P = (uint32_t)(run & 0xffffffffu);
        const uint32_t nv = (uint32_t)n - __ldcg(ticket + 1);      // the invalid keys (>= R) sort last
        cnt->n_rows = Ur; cnt->n_pieces = P; cnt->n_valid = nv; cnt->n_hot = 0;
        row_start[Ur] = nv; row_piece0[Ur] = P; piece_start[P] = nv;
        ticket[0] = 0; ticket[1] = 0;
    }
}

static __global__ void __launch_bounds__(256) seg_fill_kernel2(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t n_host,
                                                        const uint32_t* __restrict__ n_dev, uint32_t R,
                                                        const unsigned long long* __restrict__ tile_cnt,
                                                        uint32_t* __restrict__ row_start, uint32_t* __restrict__ row_piece0,
                                                        uint32_t* __restrict__ piece_start, uint32_t* __restrict__ urow, uint32_t* __restrict__ uval,
                                                        uint32_t* __restrict__ pos_row /* optional: unique-row index of every sorted position */) {
    __shared__ unsigned long long wtot[33];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n = n_dev ? (int64_t)*reinterpret_cast<const volatile uint32_t*>(n_dev) : n_host;
    const int64_t tile = blockIdx.x;
    if (tile * SB_TILE >= n) return;
    const int64_t i0 = tile * SB_TILE + (int64_t)tid * SB_ITEMS;
    uint32_t k[SB_ITEMS], rows, pieces, rmask, pmask, vmask;
    seg_tile_flags(keys, i0, n, R, k, rows, pieces, rmask, pmask, vmask);
    const unsigned long long mine = ((unsigned long long)rows << 32) | pieces;
    unsigned long long inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const unsigned long long w = lane < 8 ? wtot[lane] : 0ull;
        unsigned long long winc = w;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < 8) wtot[lane] = winc - w;
    }
    __syncthreads();
    // The lists of a tile are contiguous in the output (ranks follow positions), but a thread's 8 entries would go out as
    // 4-byte stores 32 bytes apart (5 lists: 23 % of the stall samples on the LSU queue, 7 % issue-active, 47 us for 1.7 M
    // pairs, profiles/r02br): they are staged in shared memory and written by consecutive threads instead.
    __shared__ uint32_t s_rs[SB_TILE], s_rp[SB_TILE], s_ur[SB_TILE], s_uv[SB_TILE], s_ps[SB_TILE];
    __shared__ unsigned long long s_tot;
    const unsigned long long tile_base = __ldg(tile_cnt + tile);
    const unsigned long long loc = wtot[warp] + (inc - mine);                  // exclusive (rows, pieces) before this thread, inside the tile
    if (tid == 255) s_tot = loc + mine;
    const int64_t t0 = tile * SB_TILE;
    for (int q = tid; q < SB_TILE; q += 256) s_uv[q] = t0 + q < n ? __ldg(vals + t0 + q) : 0u;      // coalesced payloads of the tile
    __syncthreads();
    uint32_t myv[SB_ITEMS];
#pragma unroll
    for (int j = 0; j < SB_ITEMS; ++j) myv[j] = s_uv[tid * SB_ITEMS + j];
    __syncthreads();                                                            // s_uv is rewritten in compacted order below
    uint32_t lr = (uint32_t)(loc >> 32), lp = (uint32_t)(loc & 0xffffffffu);
    const uint32_t r_tile = (uint32_t)(tile_base >> 32), p_tile = (uint32_t)(tile_base & 0xffffffffu);
    uint32_t pr[SB_ITEMS];
#pragma unroll
    for (int j = 0; j < SB_ITEMS; ++j) {
        if ((pmask >> j) & 1u) {
            const uint32_t i = (uint32_t)(i0 + j);
            s_ps[lp] = i;
            if ((rmask >> j) & 1u) {
                s_rs[lr] = i;
                s_rp[lr] = p_tile + lp;
                s_ur[lr] = k[j];
                s_uv[lr] = myv[j];
                ++lr;
            }
            ++lp;
        }
        pr[j] = r_tile + lr - 1;
    }
    if (pos_row) {
        if (vmask == 0xffu) {
            uint4* d = reinterpret_cast<uint4*>(pos_row + i0);
            d[0] = make_uint4(pr[0], pr[1], pr[2], pr[3]);
            d[1] = make_uint4(pr[4], pr[5], pr[6], pr[7]);
        } else {
#pragma unroll
            for (int j = 0; j < SB_ITEMS; ++j)
                if ((vmask >> j) & 1u) pos_row[i0 + j] = pr[j];
        }
    }
    __syncthreads();
    const uint32_t nr = (uint32_t)(s_tot >> 32), np = (uint32_t)(s_tot & 0xffffffffu);
    for (uint32_t q = tid; q < nr; q += 256) {
        row_start[r_tile + q] = s_rs[q];
        row_piece0[r_tile + q] = s_rp[q];
        urow[r_tile + q] = s_ur[q];
        uval[r_tile + q] = s_uv[q];
    }
    for (uint32_t q = tid; q < np; q += 256) piece_start[p_tile + q] = s_ps[q];
}

// Small batches (BASELINE configs[0] / [1]: 128 .. 16 384 pairs): sort + segments in ONE single-CTA launch instead of
// histogram + one launch per digit + count + fill (5-6 dependent launches of a few microseconds each; the step is a
// chain of such launches).  The pairs are sorted in shared memory by a bitonic network over (key << 32 | position) -
// distinct composites, so the order is the stable order of the radix sort and everything downstream is bit-identical -
// and the segment lists are written exactly as seg_count_kernel / seg_fill_kernel2 write them.
constexpr int SS_MAX = 16384, SS_THREADS = 1024;
static __global__ void __launch_bounds__(SS_THREADS) small_segments_kernel(uint32_t* __restrict__ keys, uint32_t* __restrict__ vals, int n, int m /* power of two >= max(n, 64) */,
                                                                    uint32_t R, SegCounts* __restrict__ cnt, uint32_t* __restrict__ row_start,
                                                                    uint32_t* __restrict__ row_piece0, uint32_t* __restrict__ piece_start,
                                                                    uint32_t* __restrict__ urow, uint32_t* __restrict__ uval, uint32_t* __restrict__ pos_row) {
    extern __shared__ __align__(16) unsigned long long ss_comp[];      // [m] composites, then [m] payloads
    uint32_t* sv = reinterpret_cast<uint32_t*>(ss_comp + m);
    __shared__ unsigned long long wtot[33];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < m; i += SS_THREADS) {
        ss_comp[i] = i < n ? (((unsigned long long)keys[i] << 32) | (unsigned)i) : ~0ull;
        sv[i] = i < n ? vals[i] : 0u;
    }
    __syncthreads();
    for (int k = 2; k <= m; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int p = tid; p < (m >> 1); p += SS_THREADS) {
                const int l = 2 * p - (p & (j - 1)), r = l + j;
                const unsigned long long a = ss_comp[l], b = ss_comp[r];
                const bool up = (l & k) == 0;
                if ((a > b) == up) { ss_comp[l] = b; ss_comp[r] = a; }
            }
            __syncthreads();
        }
    }
    // this thread's contiguous run of positions: flags, block-wide exclusive scan of (row heads, piece heads), lists
    const int per = (m + SS_THREADS - 1) / SS_THREADS;
    const int i0 = tid * per;
    uint32_t rows = 0, pieces = 0, valid_cnt = 0;
    for (int j = 0; j < per; ++j) {
        const int i = i0 + j;
        if (i < n) {
            const uint32_t k = (uint32_t)(ss_comp[i] >> 32);
            const uint32_t prev = i > 0 ? (uint32_t)(ss_comp[i - 1] >> 32) : 0xffffffffu;
            const bool valid = k < R, rh = valid && (i == 0 || k != prev), ph = valid && (rh || (i % PIECE_C) == 0);
            rows += rh; pieces += ph; valid_cnt += valid;
        }
    }
    const unsigned long long mine = ((unsigned long long)rows << 32) | pieces;
    unsigned long long inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    uint32_t vsum = valid_cnt;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) vsum += __shfl_xor_sync(0xffffffffu, vsum, o);
    __shared__ uint32_t wvalid[32];
    if (lane == 31) wtot[warp] = inc;
    if (lane == 0) wvalid[warp] = vsum;
    __syncthreads();
    if (warp == 0) {
        const unsigned long long w = wtot[lane];
        unsigned long long winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        wtot[lane] = winc - w;
        if (lane == 31) wtot[32] = winc;
        uint32_t v = wvalid[lane];
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) wvalid[0] = v;
    }
    __syncthreads();
    const unsigned long long run = wtot[warp] + (inc - mine);
    uint32_t ridx = (uint32_t)(run >> 32), pidx = (uint32_t)(run & 0xffffffffu);
    for (int j = 0; j < per; ++j) {
        const int i = i0 + j;
        if (i < n) {
            const unsigned long long c = ss_comp[i];
            const uint32_t k = (uint32_t)(c >> 32), v = sv[(uint32_t)c];
            const uint32_t prev = i > 0 ? (uint32_t)(ss_comp[i - 1] >> 32) : 0xffffffffu;
            const bool valid = k < R, rh = valid && (i == 0 || k != prev), ph = valid && (rh || (i % PIECE_C) == 0);
            keys[i] = k; vals[i] = v;
            if (ph) {
                piece_start[pidx] = (uint32_t)i;
                if (rh) { row_start[ridx] = (uint32_t)i; row_piece0[ridx] = pidx; urow[ridx] = k; uval[ridx] = v; ++ridx; }
                ++pidx;
            }
            if (pos_row && valid) pos_row[i] = ridx - 1;
        }
    }
    if (tid == 0) {
        const unsigned long long tot = wtot[32];
        const uint32_t Ur = (uint32_t)(tot >> 32), P = (uint32_t)(tot & 0xffffffffu), nv = wvalid[0];
        cnt->n_rows = Ur; cnt->n_pieces = P; cnt->n_valid = nv; cnt->n_hot = 0;
        row_start[Ur] = nv; row_piece0[Ur] = P; piece_start[P] = nv;
    }
}

// =============================================================================================
// non-lazy Adam: materialise the deferred decay of EVERY row (dfm_flush: before a checkpoint / dfm_get_tensor)
// =============================================================================================
// table layout: see Table (dfm_types.cuh).  The two optimizers share the step index, so the one last_step
// in the linear float4 serves both the embedding row and the linear weight.
template <int K>
__global__ void __launch_bounds__(256) catchup_all_kernel(Table tb, uint64_t R, RowReplay rr, OptDev od, OptDev ol, bool has_emb) {
    constexpr int LPR = K / 4;
    const int sub = threadIdx.x % LPR;
    const uint64_t gpb = blockDim.x / LPR;
    const ReplayStep rs = replay_step_load(rr.rd.closed ? rr.rd : rr.rl, rr.upto);
    for (uint64_t base = (uint64_t)blockIdx.x * gpb; base < R; base += (uint64_t)gridDim.x * gpb) {   // block-uniform trip count
        const uint64_t row = base + threadIdx.x / LPR;
        float4 lr = make_float4(0.f, 0.f, 0.f, 0.f);
        bool work = false;
        if (row < R) { lr = *tab_lin(tb, row); work = __float_as_int(lr.w) < rr.upto; }
        float4 w = make_float4(0.f, 0.f, 0.f, 0.f), m = w, v = w;
        bool idle = true;
        if (work && has_emb && rr.emb_adam) {
            m = tab_s1(tb, row)[sub]; v = tab_s2(tb, row)[sub];
            // slices that were never touched (m = v = 0) do not move under non-lazy Adam: nothing more to read or write
            idle = m.x == 0.f && m.y == 0.f && m.z == 0.f && m.w == 0.f && v.x == 0.f && v.y == 0.f && v.z == 0.f && v.w == 0.f;
            if (!idle) w = tab_w(tb, row)[sub];
        }
        if (work) replay_row(w, m, v, lr, sub == 0, rr, rs, od, ol);
        if (work && !idle) { tab_w(tb, row)[sub] = w; tab_s1(tb, row)[sub] = m; tab_s2(tb, row)[sub] = v; }
        __syncwarp();  // every lane of a group has read last_step before lane 0 rewrites it
        // last_step is always advanced, also for idle rows
        if (work && sub == 0) *tab_lin(tb, row) = lr;
    }
}

// =============================================================================================
// K2: fused embedding + linear gather, FM second-order term, first-order sum, input_layer write
// =============================================================================================
// One warp per sample; a table row of K floats is read by K/4 lanes as float4, so one warp round
// covers 128/K fields and every h0 store is a fully coalesced 512-byte line.
//   trainers/deep_fm.py:39     linear_model       -> zacc += sum_f w_f[id] + sum_j x_j wn_j + bias
//   trainers/deep_fm.py:52-73  input_layer        -> h0[b, f*K..]
//   trainers/deep_fm.py:79-87  FM                 -> zacc += 0.5 * sum_k((sum_f E)^2 - sum_f E^2)
template <int K, bool BAGS>
__global__ void __launch_bounds__(256) gather_fm_kernel(const int32_t* __restrict__ ids, int B, int dc, int dn, int n_slots,
                                                        const int32_t* __restrict__ field_slot0 /*[dc+1] or null: 1 slot per field*/,
                                                        float* __restrict__ inv_cnt /*[B, dc] or null*/,
                                                        const uint32_t* __restrict__ row_off,
                                                        Table tb, BatchPtrs bp,
                                                        const float* __restrict__ num_emb,
                                                        const float* __restrict__ num_lin,
                                                        const float* __restrict__ bias, int use_linear, int use_mf,
                                                        int need_emb, float* __restrict__ h0, float* __restrict__ s_out,
                                                        float* __restrict__ zacc, const uint32_t* __restrict__ uidx,
                                                        const float* __restrict__ rowbuf, int rowbuf_stride,
                                                        RowReplay rr, OptDev od, OptDev ol) {
    constexpr int LPR = K / 4;       // lanes per row
    constexpr int FPR = 32 / LPR;    // fields per warp round
    const int lane = threadIdx.x & 31;
    const int sub = lane % LPR, grp = lane / LPR;
    const int warps_per_block = blockDim.x >> 5;
    const int d = dc + dn;
    const float b0 = (use_linear && bias) ? bias[0] : 0.f;
    const ReplayStep rs = replay_step_load(rr.rd.closed ? rr.rd : rr.rl, rr.upto);
    for (int b = blockIdx.x * warps_per_block + (threadIdx.x >> 5); b < B; b += gridDim.x * warps_per_block) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
        float lin = 0.f;
        const int32_t* idrow = ids + (int64_t)b * n_slots;
        float4* hrow = reinterpret_cast<float4*>(h0 + (int64_t)b * d * K);
        for (int f0 = 0; f0 < dc; f0 += FPR) {
            int f = f0 + grp;
            if (f < dc) {
                const int s0 = BAGS ? field_slot0[f] : f, s1 = BAGS ? field_slot0[f + 1] : f + 1;
                float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
                float lsum = 0.f;
                int cnt = 0;
                for (int sl = s0; sl < s1; ++sl) {      // one slot for a single-valued column; a multi-hot bag is mean-pooled
                    int32_t id = idrow[sl];
                    if (id >= 0) {
                        ++cnt;
                        if (rowbuf) {   // sharded: rows were fetched from their owners into rowbuf[unique index]
                            const float* rp = rowbuf + (size_t)__ldg(uidx + (int64_t)b * n_slots + sl) * rowbuf_stride;
                            if (need_emb) add4(e, __ldg(reinterpret_cast<const float4*>(rp) + sub));
                            if (use_linear && sub == 0) lsum += __ldg(rp + K);
                        } else {
                            // the row as of the previous step: the deferred non-lazy Adam decay is replayed in registers
                            // (nothing is written back here; the optimizer kernel replays again when it rewrites the row)
                            size_t row = (size_t)row_off[f] + (uint32_t)id;
                            float4 w; float lw;
                            load_row_current(tb, row, sub, need_emb != 0, rr, rs, od, ol, w, lw);
                            if (need_emb) add4(e, w);
                            if (use_linear && sub == 0) lsum += lw;
                        }
                    }
                }
                if (BAGS) {
                    if (cnt > 1) { const float ic = 1.0f / (float)cnt; e.x *= ic; e.y *= ic; e.z *= ic; e.w *= ic; }
                    if (sub == 0) inv_cnt[(int64_t)b * dc + f] = cnt ? 1.0f / (float)cnt : 0.f;
                }
                lin += lsum;
                if (need_emb) {
                    hrow[f * LPR + sub] = e;
                    s.x += e.x; s.y += e.y; s.z += e.z; s.w += e.w;
                    q.x += e.x * e.x; q.y += e.y * e.y; q.z += e.z * e.z; q.w += e.w * e.w;
                }
            }
        }
        for (int j0 = 0; j0 < dn; j0 += FPR) {
            int j = j0 + grp;
            if (j < dn) {
                float x = __ldg(bp.num[j] + b);
                if (need_emb) {
                    float4 ve = __ldg(reinterpret_cast<const float4*>(num_emb + j * K) + sub);
                    float4 e = make_float4(x * ve.x, x * ve.y, x * ve.z, x * ve.w);
                    hrow[(dc + j) * LPR + sub] = e;
                    s.x += e.x; s.y += e.y; s.z += e.z; s.w += e.w;
                    q.x += e.x * e.x; q.y += e.y * e.y; q.z += e.z * e.z; q.w += e.w * e.w;
                }
                if (use_linear && sub == 0) lin += x * __ldg(num_lin + j);
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
        if (need_emb && grp == 0) reinterpret_cast<float4*>(s_out + (int64_t)b * K)[sub] = s;
        if (lane == 0) {
            float z = 0.f;
            if (use_linear) z += lin + b0;
            if (use_mf) z += 0.5f * t;
            zacc[b] = z;
        }
    }
}

// =============================================================================================
// K5/K6: deterministic segmented reduction of the sparse gradients + sparse optimizer apply
// =============================================================================================
// gradient of lookup (b, f): dE[b, f*K..] (already = dz*(s-E) + dh0, written by the tower's last
// backward GEMM epilogue or by de_fm_kernel) and dz[b] for the linear weight.
template <int K, bool BAGS>
struct GradSrc {
    static constexpr bool SUB_E = false;
    __device__ __forceinline__ bool sub_e() const { return false; }
    const float* erow = nullptr; int erow_stride = 0;     // (unused here; see GradSrcFused)
    const float* dE;    // [B, d*K] or nullptr
    const float* dz;    // [B]
    int dc, dK;         // dK = d*K
    const float* flat;  // sharded owner side: gradient rows [n][flat_stride] = {g[K], g_lin, pad}, payload = row of `flat`
    int flat_stride;
    int n_slots;                // lookups per sample
    const int32_t* slot_field;  // BAGS: slot -> field
    const float* inv_cnt;       // BAGS: [B, dc] 1 / (present slots) of every field
    __device__ __forceinline__ void fetch(uint32_t val, int sub, bool want_lin, float4& g, float& gl) const {
        if (flat) {
            const float* rp = flat + (size_t)val * flat_stride;
            g = __ldg(reinterpret_cast<const float4*>(rp) + sub);
            gl = want_lin ? __ldg(rp + K) : 0.f;
            return;
        }
        uint32_t b = payload_sample(val), f = payload_slot(val);
        if (BAGS) f = (uint32_t)__ldg(slot_field + f);
        g = dE ? __ldg(reinterpret_cast<const float4*>(dE + (size_t)b * dK + (size_t)f * K) + sub)
               : make_float4(0.f, 0.f, 0.f, 0.f);
        if (BAGS) {   // mean combiner: every present slot of the bag receives dE / count
            const float ic = __ldg(inv_cnt + (size_t)b * dc + f);
            g.x *= ic; g.y *= ic; g.z *= ic; g.w *= ic;
        }
        gl = want_lin ? __ldg(dz + b) : 0.f;
    }
};

// list the pieces of hot rows (rows with > DIRECT_T lookups); order is irrelevant, every piece sum goes to its own slot
static __global__ void __launch_bounds__(256) hot_pieces_kernel(const uint32_t* __restrict__ row_start, const uint32_t* __restrict__ row_piece0,
                                                         SegCounts* __restrict__ cnt, uint32_t* __restrict__ hot_list) {
    const uint32_t U = cnt->n_rows;
    for (uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; u < U; u += gridDim.x * blockDim.x) {
        if (row_start[u + 1] - row_start[u] <= (uint32_t)DIRECT_T) continue;
        const uint32_t p0 = row_piece0[u], p1 = row_piece0[u + 1];
        uint32_t base = atomicAdd(&cnt->n_hot, p1 - p0);
        for (uint32_t p = p0; p < p1; ++p) hot_list[base + (p - p0)] = p;
    }
}

// level 1: one warp per piece of a hot row.  The 128/K lane groups stride over the piece's entries
// (4 independent loads in flight per group), then a fixed butterfly combines them -> the summation
// order is a function of the sorted order only.
template <int K, typename SRC>
__global__ void __launch_bounds__(256) piece_reduce_kernel(const uint32_t* __restrict__ svals,
                                                           const uint32_t* __restrict__ piece_start,
                                                           const uint32_t* __restrict__ hot_list,
                                                           const SegCounts* __restrict__ cnt, SRC src,
                                                           float* __restrict__ piece_sum /*[slots][K+4]*/) {
    constexpr int LPR = K / 4, G = 32 / LPR;
    const int lane = threadIdx.x & 31, sub = lane % LPR, grp = lane / LPR;
    const uint32_t NH = cnt->n_hot;
    const uint32_t nwarps = gridDim.x * (blockDim.x >> 5);
    const uint32_t warp0 = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (uint32_t hp = warp0; hp < NH; hp += nwarps) {
        const uint32_t pp = __ldg(hot_list + hp);
        const uint32_t beg = __ldg(piece_start + pp), end = __ldg(piece_start + pp + 1);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float accl = 0.f;
        for (uint32_t i = beg + grp; i < end; i += 4 * G) {
            uint32_t v[4];
            float4 g[4];
            float gl[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = (i + u * G < end) ? __ldg(svals + i + u * G) : 0xffffffffu;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                gl[u] = 0.f;
                if (v[u] != 0xffffffffu) src.fetch(v[u], sub, sub == 0, g[u], gl[u]);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) { add4(acc, g[u]); accl += gl[u]; }
        }
#pragma unroll
        for (int o = LPR; o < 32; o <<= 1) {
            acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
            acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
            accl += __shfl_xor_sync(0xffffffffu, accl, o);
        }
        if (grp == 0) {
            float* dst = piece_sum + (size_t)piece_slot(beg) * (K + 4);
            reinterpret_cast<float4*>(dst)[sub] = acc;
            if (sub == 0) dst[K] = accl;
        }
    }
}

// The optimizer step of one unique row, by its lane group (lane `sub` holds elements 4 sub .. 4 sub + 3 of w / s1 / s2;
// lr = {lin w, lin s1, lin s2, last_step} is on every lane): first the non-lazy Adam decay steps the row skipped since
// it was last written (replayed in registers), then this step's gradient g / gl (gl on lane 0).  sub_e: g is still
// sum(dz s + dh0) of the fused step, and dE = g - sum(dz) * E with E = the row as the forward pass saw it (the replayed w).
// The record is stored with last_step = step.
__device__ __forceinline__ void row_step(const Table& tb, size_t row, int sub, float4 w, float4 s1, float4 s2, float4 lr, float4 g,
                                         float gl, bool sub_e, int emb_slots, const OptDev& od, const OptDev& ol, bool has_emb,
                                         bool has_lin, int step, const RowReplay& rr, const ReplayStep& rs) {
    replay_row(w, s1, s2, lr, sub == 0, rr, rs, od, ol);
    if (sub_e) { g.x = fmaf(-gl, w.x, g.x); g.y = fmaf(-gl, w.y, g.y); g.z = fmaf(-gl, w.z, g.z); g.w = fmaf(-gl, w.w, g.w); }
    if (has_emb) {
        sparse_apply(w.x, s1.x, s2.x, g.x, od);
        sparse_apply(w.y, s1.y, s2.y, g.y, od);
        sparse_apply(w.z, s1.z, s2.z, g.z, od);
        sparse_apply(w.w, s1.w, s2.w, g.w, od);
        tab_w(tb, row)[sub] = w;
        if (emb_slots >= 1) tab_s1(tb, row)[sub] = s1;
        if (emb_slots >= 2) tab_s2(tb, row)[sub] = s2;
    }
    if (sub == 0) {
        if (has_lin) sparse_apply(lr.x, lr.y, lr.z, gl, ol);
        lr.w = __int_as_float(step);
        *tab_lin(tb, row) = lr;
    }
}

// dE = dz * (s - E) when there is no DNN tower (otherwise the last backward GEMM epilogue does it);
// accumulate != 0 adds to an existing dE (hidden_units == [] case).
static __global__ void de_fm_kernel(const float* __restrict__ h0, const float* __restrict__ s, const float* __restrict__ dz,
                             int64_t total, int dK, int K, float* __restrict__ dE, int accumulate) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) {
        int64_t b = i / dK;
        int c = (int)(i - b * dK) % K;
        float v = dz[b] * (s[b * K + c] - h0[i]);
        dE[i] = accumulate ? dE[i] + v : v;
    }
}

// =============================================================================================
// row sharding (SURVEY.md 8e): rank r owns global rows {g : g % W == r}, stored at local index g / W
// =============================================================================================
// global-row sort key -> owner-major key  owner * Rl + local  (Rl = ceil(R / W)); empty bags -> W * Rl
static __global__ void shard_rekey_kernel(uint32_t* __restrict__ keys, int64_t n, uint32_t R, uint32_t W, uint32_t Rl) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        uint32_t g = keys[i];
        keys[i] = g < R ? (g % W) * Rl + g / W : W * Rl;
    }
}
// per sorted position: lookup -> unique index; per unique row: local row id for its owner + per-owner counts
static __global__ void __launch_bounds__(256) shard_uniq_kernel(const uint32_t* __restrict__ skeys, const uint32_t* __restrict__ svals, int64_t n,
                                                         uint32_t limit, uint32_t Rl, uint32_t W, int n_slots,
                                                         const uint32_t* __restrict__ pos_row, uint32_t* __restrict__ uidx,
                                                         uint32_t* __restrict__ req_rows, int32_t* __restrict__ counts,
                                                         uint8_t* __restrict__ once_lk = nullptr) {
    // once_lk[lookup] = 1: the lookup's row is looked up exactly once in this rank's batch
    // per-owner counts are aggregated per block in shared memory first: the sorted keys put (almost) every
    // lookup of a block on the same owner, and same-address global atomics serialise in L2
    __shared__ int sc[64];
    if (threadIdx.x < 64) sc[threadIdx.x] = 0;
    __syncthreads();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        uint32_t k = skeys[i];
        if (k >= limit) {
            uidx[(size_t)payload_sample(svals[i]) * n_slots + payload_slot(svals[i])] = 0xffffffffu;
        } else {
            bool rh = (i == 0) || (k != skeys[i - 1]);
            const uint32_t ridx = pos_row[i];
            uidx[(size_t)payload_sample(svals[i]) * n_slots + payload_slot(svals[i])] = ridx;
            if (once_lk) once_lk[(size_t)payload_sample(svals[i]) * n_slots + payload_slot(svals[i])] = (rh && (i + 1 >= n || skeys[i + 1] != k)) ? 1 : 0;
            if (rh) {
                req_rows[ridx] = k % Rl;
                uint32_t o = k / Rl;
                if (W <= 64) atomicAdd(&sc[o], 1); else atomicAdd(&counts[o], 1);
            }
        }
    }
    __syncthreads();
    if (W <= 64 && threadIdx.x < W && sc[threadIdx.x]) atomicAdd(&counts[threadIdx.x], sc[threadIdx.x]);
}
static __global__ void iota_kernel(uint32_t* __restrict__ v, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}
// =============================================================================================
// tiny-vocabulary columns (<= TINY_MAX buckets: the 19 genre flags, gender, age and release-year buckets of the
// ML-100K schema = 22 of its 26 columns, 85 % of the lookups but only 72 table rows).  Sorting their lookups only to
// find out that a row was hit 30 000 times is wasted work: their gradient rows are reduced DENSELY instead — a block
// per 128 samples accumulates per-row sums in shared memory (every warp owns private accumulators and walks its
// samples in index order; warps, then blocks, are combined in fixed order, so the sum is deterministic) — and a
// small kernel applies the optimizer to the rows that were hit.  The sort / segment /
// piece machinery then sees only the large columns.
// =============================================================================================
constexpr int TINY_MAX = 8;               // buckets of a "tiny" column
constexpr int TINY_SPB = 512;             // samples per block (64 per warp)

// Block = (128 consecutive samples) x (one group of 32/LPR adjacent tiny columns), warp = 16 of the samples in index
// order; the lane groups of a warp take the columns of the group side by side (adjacent columns are adjacent in dE and
// in the id row, so the reads coalesce).  Each warp owns private accumulators [row of the column group][K + 4] =
// {g[K], g_lin, count, -, -}; warps are combined in fixed order.
template <int K>
__global__ void __launch_bounds__(256) tiny_reduce_kernel(const int32_t* __restrict__ ids, int B, int n_slots, const int32_t* __restrict__ tslot,
                                                          const int32_t* __restrict__ trow0 /* [n_tiny + 1] */, int n_tiny, int n_trows,
                                                          const float* __restrict__ dE, const float* __restrict__ dz, int dK,
                                                          float* __restrict__ partial) {
    constexpr int LPR = K / 4, G = 32 / LPR, RW = K + 4;
    extern __shared__ __align__(16) float tacc[];     // [8][rows of this column group][RW]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, sub = lane % LPR, grp = lane / LPR;
    const int c0 = blockIdx.y * G, c1 = min(n_tiny, c0 + G);
    const int rbase = __ldg(trow0 + c0), per = (__ldg(trow0 + c1) - rbase) * RW;
    for (int i = threadIdx.x; i < 8 * per; i += 256) tacc[i] = 0.f;
    __syncthreads();
    float* my = tacc + warp * per;
    const int b_begin = blockIdx.x * TINY_SPB + warp * (TINY_SPB / 8);
    const int b_end = min(B, b_begin + TINY_SPB / 8);
    const int c = c0 + grp;
    const bool cok = c < c1;
    const int slot = cok ? __ldg(tslot + c) : 0, r0 = cok ? __ldg(trow0 + c) - rbase : 0;
    constexpr int U = 8;                 // samples in flight per lane group; id, gradient row and dz are independent loads
    for (int b = b_begin; b < b_end; b += U) {
        int id[U];
        float4 x[U];
        float z[U];
#pragma unroll
        for (int q = 0; q < U; ++q) {
            const bool ok = cok && b + q < b_end;
            id[q] = ok ? __ldg(ids + (size_t)(b + q) * n_slots + slot) : -1;
            x[q] = (ok && dE) ? __ldg(reinterpret_cast<const float4*>(dE + (size_t)(b + q) * dK + (size_t)slot * K) + sub) : make_float4(0.f, 0.f, 0.f, 0.f);
            z[q] = (ok && sub == 0) ? __ldg(dz + b + q) : 0.f;
        }
#pragma unroll
        for (int q = 0; q < U; ++q)
            if (id[q] >= 0) {
                float* row = my + (r0 + id[q]) * RW;
                float4* a4 = reinterpret_cast<float4*>(row) + sub;
                float4 v = *a4;
                v.x += x[q].x; v.y += x[q].y; v.z += x[q].z; v.w += x[q].w;
                *a4 = v;
                if (sub == 0) { row[K] += z[q]; row[K + 1] += 1.f; }
            }
    }
    __syncthreads();
    float* out = partial + ((size_t)blockIdx.x * n_trows + rbase) * RW;
    for (int e = threadIdx.x; e < per; e += 256) {
        float sacc = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) sacc += tacc[w * per + e];
        out[e] = sacc;
    }
}

// one WARP per row of a tiny column: the lane groups take the blocks' partial sums round-robin (in block order), a fixed
// butterfly combines the groups, then the sparse optimizer (rows that were not hit stay as they are — the non-lazy
// Adam decay reaches them through the catch-up, like any other idle row)
template <int K>
__global__ void __launch_bounds__(256) tiny_update_kernel(const float* __restrict__ partial, int n_blocks, const uint32_t* __restrict__ trow_grow,
                                                          int n_trows, Table tb, int emb_slots, OptDev od, OptDev ol, bool has_emb, bool has_lin,
                                                          int step, RowReplay rr) {
    constexpr int LPR = K / 4, G = 32 / LPR, RW = K + 4;
    const ReplayStep rs = replay_step_load(rr.rd.closed ? rr.rd : rr.rl, rr.upto);
    const int lane = threadIdx.x & 31, sub = lane % LPR, grp = lane / LPR;
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= n_trows) return;                        // warp-uniform
    const size_t per = (size_t)n_trows * RW;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    float gl = 0.f, cnt = 0.f;
    for (int j0 = grp; j0 < n_blocks; j0 += 8 * G) {      // 8 independent loads in flight, added in block order
        float4 t[8];
        float tl[8], tc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int j = j0 + q * G;
            t[q] = make_float4(0.f, 0.f, 0.f, 0.f); tl[q] = 0.f; tc[q] = 0.f;
            if (j < n_blocks) {
                const float* p = partial + j * per + (size_t)r * RW;
                t[q] = __ldg(reinterpret_cast<const float4*>(p) + sub);
                const float2 lc = __ldg(reinterpret_cast<const float2*>(p + K));
                tl[q] = lc.x; tc[q] = lc.y;
            }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) { g.x += t[q].x; g.y += t[q].y; g.z += t[q].z; g.w += t[q].w; gl += tl[q]; cnt += tc[q]; }
    }
#pragma unroll
    for (int o = LPR; o < 32; o <<= 1) {
        g.x += __shfl_xor_sync(0xffffffffu, g.x, o); g.y += __shfl_xor_sync(0xffffffffu, g.y, o);
        g.z += __shfl_xor_sync(0xffffffffu, g.z, o); g.w += __shfl_xor_sync(0xffffffffu, g.w, o);
        gl += __shfl_xor_sync(0xffffffffu, gl, o); cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if (cnt == 0.f || grp != 0) return;
    const size_t row = trow_grow[r];
    float4 lr = *tab_lin(tb, row);
    float4 w = make_float4(0.f, 0.f, 0.f, 0.f), s1 = w, s2 = w;
    if (has_emb) {
        w = tab_w(tb, row)[sub];
        if (emb_slots >= 1) s1 = tab_s1(tb, row)[sub];
        if (emb_slots >= 2) s2 = tab_s2(tb, row)[sub];
    }
    row_step(tb, row, sub, w, s1, s2, lr, g, gl, false, emb_slots, od, ol, has_emb, has_lin, step, rr, rs);
}

// owner side: reply[i] = {emb w[K], lin w, pad} of local row recv_rows[i]
template <int K>
__global__ void __launch_bounds__(256) shard_serve_kernel(const uint32_t* __restrict__ recv_rows, int64_t n,
                                                          Table tb, bool has_emb, bool has_lin,
                                                          float* __restrict__ reply, int reply_stride,
                                                          RowReplay rr, OptDev od, OptDev ol) {
    constexpr int LPR = K / 4;
    const int sub = threadIdx.x % LPR;
    const int64_t gpb = blockDim.x / LPR;
    const ReplayStep rs = replay_step_load(rr.rd.closed ? rr.rd : rr.rl, rr.upto);
    for (int64_t i = (int64_t)blockIdx.x * gpb + threadIdx.x / LPR; i < n; i += (int64_t)gridDim.x * gpb) {
        size_t row = recv_rows[i];
        float* rp = reply + (size_t)i * reply_stride;
        float4 e; float lw;
        load_row_current(tb, row, sub, has_emb, rr, rs, od, ol, e, lw);     // replayed in registers, not written back
        reinterpret_cast<float4*>(rp)[sub] = e;
        if (sub == 0) rp[K] = has_lin ? lw : 0.f;
    }
}
