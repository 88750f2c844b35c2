// K6, staged: segmented gradient reduction + sparse optimizer for the unique rows of a step, with the table records and
// the first gradient operand of every row brought into shared memory by cp.async (LDGSTS) a few iterations ahead.
//
// Why: ncu on the unstaged kernel at the Criteo shape (1.7 M unique rows of 256 bytes, profiles/r02b) showed 25 % occupancy,
// 32 % issue-active and 1.8 TB/s: every lane group held one row's loads in registers, so an SM had ~14 KB in flight —
// a quarter of what HBM latency needs.  cp.async costs no registers: each warp keeps NST-1 iterations (8 rows each at
// K = 16) in flight, ~90 KB per SM, and the arithmetic of iteration i overlaps the traffic of i+1, i+2.  The dense
// operand of the fused step's gradient source (W0, 40 KB at the Criteo shape) is copied to shared memory once per CTA:
// read through L1 it cost 16 dependent L2-latency loads per row (profiles/r02d: long-scoreboard stalls on LDG).
//
// Work split: a lane group (K/4 lanes) owns one row end to end, a warp owns 32/(K/4) consecutive rows per iteration, and
// every warp runs its own pipeline (no block-wide barriers: a group's data is copied by its own lanes).
// Per row the staging slot holds  [ record: w | {lin w, s1, s2, last_step} | slot1 | slot2 ][ gradient operand ][ meta ].
#pragma once
#include "dfm_types.cuh"
#include "embed_kernels.cuh"

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// staging interface of the plain gradient sources (dE buffer of the unfused step / flat gradient rows of the sharded owner)
template <int K, bool BAGS = false>
struct StageSrcPlain {
    static constexpr bool SUB_E = false;
    static constexpr int STAGE_F = K + 4;           // [g[K] | g_lin, 1 / count (BAGS), pad]
    GradSrc<K, BAGS> s;
    const float* erow = nullptr; int erow_stride = 0;       // (only sources with SUB_E carry the fetched rows)
    __device__ __forceinline__ bool sub_e() const { return false; }
    __device__ __forceinline__ void stage_async(uint32_t val, float* dst, int sub) const {
        constexpr int LPR = K / 4;
        if (s.flat) {
            const float* rp = s.flat + (size_t)val * s.flat_stride;
            cp_async16(dst + sub * 4, rp + sub * 4);
            if (sub == 0) cp_async16(dst + K, rp + K);
        } else {
            const uint32_t b = payload_sample(val);
            uint32_t f = payload_slot(val);
            if (BAGS) f = (uint32_t)__ldg(s.slot_field + f);
            if (s.dE) cp_async16(dst + sub * 4, s.dE + (size_t)b * s.dK + (size_t)f * K + sub * 4);
            if (sub == LPR - 1) cp_async4(dst + K, s.dz + b);
            if (BAGS && sub == 0) cp_async4(dst + K + 1, s.inv_cnt + (size_t)b * s.dc + f);
        }
    }
    int aux_floats() const { return 0; }                              // no per-CTA shared-memory operand
    __device__ __forceinline__ void aux_load(float*, int) const {}
    __device__ __forceinline__ void consume(const float* st, const float*, uint32_t, int sub, float4& g, float& gl) const {
        g = (s.flat || s.dE) ? *reinterpret_cast<const float4*>(st + sub * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (BAGS && !s.flat) {   // mean combiner, as in GradSrc::fetch: every present slot of the bag receives dE / count
            const float ic = st[K + 1];
            g.x *= ic; g.y *= ic; g.z *= ic; g.w *= ic;
        }
        gl = st[K];
    }
    __device__ __forceinline__ void fetch(uint32_t val, int sub, bool want_lin, float4& g, float& gl) const { s.fetch(val, sub, want_lin, g, gl); }
};

// The gradient sum of unique row u (its lookups are beg .. end-1 of the sorted order; act: the row has work here), called
// by every lane of the warp.  Rows with <= DIRECT_T lookups add them in sorted (= sample) order, the first one from the
// staging slot `staged`; hotter rows add their piece sums in order; very hot rows (> COOP_PIECES pieces) are summed by
// the whole warp: its lane groups take the pieces round-robin and a fixed butterfly combines them.  The summation order
// is thus a function of the sorted order only.  gl is complete on lane 0 of the group (on every lane if SRC::SUB_E).
template <int K, typename SRC>
__device__ __forceinline__ void row_grad_sum(const SRC& src, const float* staged, const float* aux, bool act, uint32_t u, uint32_t v0,
                                             uint32_t beg, uint32_t end, const uint32_t* __restrict__ svals,
                                             const uint32_t* __restrict__ row_piece0, const uint32_t* __restrict__ piece_start,
                                             const float* __restrict__ piece_sum, float4& g, float& gl) {
    constexpr int LPR = K / 4, G = 32 / LPR;
    const int lane = threadIdx.x & 31, sub = lane % LPR, grp = lane / LPR;
    g = make_float4(0.f, 0.f, 0.f, 0.f);
    gl = 0.f;
    bool coop = false;
    if (!act) {
    } else if (end - beg <= (uint32_t)DIRECT_T) {
        src.consume(staged, aux, v0, sub, g, gl);             // first lookup of the row: staged a few iterations ahead
        for (uint32_t i = beg + 1; i < end; i += 4) {         // further lookups of the same row (rare with large tables)
            uint32_t v[4];
            float4 t[4];
            float tl[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = (i + q < end) ? __ldg(svals + i + q) : 0xffffffffu;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                t[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                tl[q] = 0.f;
                if (v[q] != 0xffffffffu) src.fetch(v[q], sub, sub == 0, t[q], tl[q]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) { add4(g, t[q]); gl += tl[q]; }
        }
    } else {
        const uint32_t p0 = __ldg(row_piece0 + u), p1 = __ldg(row_piece0 + u + 1);
        if (p1 - p0 > (uint32_t)COOP_PIECES) {
            coop = true;      // summed below by the whole warp
        } else {
            for (uint32_t p = p0; p < p1; p += 4) {
                float4 t[4];
                float tl[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    t[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                    tl[q] = 0.f;
                    if (p + q < p1) {
                        const float* ps = piece_sum + (size_t)piece_slot(__ldg(piece_start + p + q)) * (K + 4);
                        t[q] = __ldg(reinterpret_cast<const float4*>(ps) + sub);
                        if (sub == 0) tl[q] = __ldg(ps + K);
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) { add4(g, t[q]); gl += tl[q]; }
            }
        }
    }
    uint32_t cmask = __ballot_sync(0xffffffffu, coop && sub == 0);
    while (cmask) {
        const int src_lane = __ffs(cmask) - 1;
        cmask &= cmask - 1;
        const uint32_t cu = __shfl_sync(0xffffffffu, u, src_lane);
        const uint32_t p0 = __ldg(row_piece0 + cu), p1 = __ldg(row_piece0 + cu + 1);
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        float al = 0.f;
        for (uint32_t p = p0 + grp; p < p1; p += 4 * G) {
            float4 t[4];
            float tl[4];
            uint32_t ps_slot[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) ps_slot[q] = (p + q * G < p1) ? piece_slot(__ldg(piece_start + p + q * G)) : 0xffffffffu;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                t[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                tl[q] = 0.f;
                if (ps_slot[q] != 0xffffffffu) {
                    const float* ps = piece_sum + (size_t)ps_slot[q] * (K + 4);
                    t[q] = __ldg(reinterpret_cast<const float4*>(ps) + sub);
                    if (sub == 0) tl[q] = __ldg(ps + K);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) { add4(a, t[q]); al += tl[q]; }
        }
#pragma unroll
        for (int o = LPR; o < 32; o <<= 1) {
            a.x += __shfl_xor_sync(0xffffffffu, a.x, o); a.y += __shfl_xor_sync(0xffffffffu, a.y, o);
            a.z += __shfl_xor_sync(0xffffffffu, a.z, o); a.w += __shfl_xor_sync(0xffffffffu, a.w, o);
            al += __shfl_xor_sync(0xffffffffu, al, o);
        }
        if (lane / LPR == src_lane / LPR) { g = a; gl = al; }
    }
    if (SRC::SUB_E) gl = __shfl_sync(0xffffffffu, gl, lane - sub);   // the piece paths keep sum(dz) on lane 0 of the group only
}

template <int K, typename SRC>
struct RowApplyCfg {
    static constexpr int LPR = K / 4, G = 32 / LPR;
    static constexpr int RSMAX = 3 * K + 4;                       // record floats staged (w | lin4 | slot1 | slot2)
    static constexpr int SLOT = RSMAX + SRC::STAGE_F + 4;         // + meta {row, first lookup, begin, end}
    static constexpr int NST = K >= 16 ? 3 : 2;                   // pipeline stages per warp
    static constexpr int SMEM = 8 * NST * G * SLOT * 4;      // + SRC::aux_floats() * 4 (per-CTA operand, e.g. W0 of the fused step)
};

template <int K, typename SRC>
__global__ void __launch_bounds__(256, 2) row_apply_kernel(const uint32_t* __restrict__ urow, const uint32_t* __restrict__ uval,
                                                           const uint32_t* __restrict__ svals, const uint32_t* __restrict__ row_start,
                                                           const uint32_t* __restrict__ row_piece0, const uint32_t* __restrict__ piece_start,
                                                           const SegCounts* __restrict__ cnt, SRC src, const float* __restrict__ piece_sum,
                                                           Table tb, int emb_slots, OptDev od, OptDev ol, bool has_emb, bool has_lin, int step,
                                                           RowReplay rr) {
    using C = RowApplyCfg<K, SRC>;
    constexpr int LPR = C::LPR, G = C::G, RSMAX = C::RSMAX, SLOT = C::SLOT, NST = C::NST;
    constexpr int CPL = (RSMAX / 4 + LPR - 1) / LPR;               // 16-byte record chunks per lane (upper bound)
    extern __shared__ __align__(16) float ra_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = lane % LPR, grp = lane / LPR;
    float* wbase = ra_smem + ((size_t)warp * NST * G + grp) * SLOT;      // this lane group's slot of stage 0
    float* aux = ra_smem + (size_t)8 * NST * G * SLOT;                   // per-CTA operand of the gradient source
    src.aux_load(aux, threadIdx.x);
    __syncthreads();
    const ReplayStep rs = replay_step_load(rr.rd.closed ? rr.rd : rr.rl, rr.upto);
    const uint32_t U = cnt->n_rows;
    const uint32_t nw = gridDim.x * 8, gw = blockIdx.x * 8 + warp;
    const uint32_t n_chunks = (U + G - 1) / G;                     // chunks of G rows; this warp takes chunk gw, gw + nw, ...
    const uint32_t n_it = n_chunks > gw ? (n_chunks - gw - 1) / nw + 1 : 0;
    const int rec_f4 = (has_emb ? (K + 4 + emb_slots * K) : 4) / 4;     // 16-byte chunks of the record that exist
    const uint32_t u_step = nw * G;

    // Software pipeline: iteration j's copies are issued NST-1 iterations before it is computed; its meta
    // {row, first lookup, begin, end} is loaded (plain coalesced loads) one iteration before the copies are issued.
    uint32_t m_row = 0, m_v0 = 0xffffffffu, m_beg = 0, m_end = 0;   // meta of the iteration issued next
    uint32_t u_meta = gw * G + grp;                                // row index the meta registers refer to
    uint32_t it_meta = 0;
    int st_issue = 0, st_use = 0;
#define RA_LOAD_META()                                                                                                   \
    do {                                                                                                                 \
        m_row = 0; m_v0 = 0xffffffffu; m_beg = 0; m_end = 0;                                                             \
        if (it_meta < n_it && u_meta < U) {                                                                              \
            m_row = __ldg(urow + u_meta); m_v0 = __ldg(uval + u_meta);                                                   \
            m_beg = __ldg(row_start + u_meta); m_end = __ldg(row_start + u_meta + 1);                                    \
        }                                                                                                                \
    } while (0)
#define RA_ISSUE()                                                                                                       \
    do {                                                                                                                 \
        float* slot_i = wbase + (size_t)st_issue * G * SLOT;                                                             \
        if (m_end > m_beg) {                                                                                             \
            const float* rec = tb.rec + (size_t)m_row * tb.stride;                                                       \
            _Pragma("unroll") for (int q = 0; q < CPL; ++q) {                                                            \
                const int c = sub + q * LPR;                                                                             \
                if (c < rec_f4) cp_async16(slot_i + c * 4, rec + c * 4);                                                 \
            }                                                                                                            \
            src.stage_async(m_v0, slot_i + RSMAX, sub);                                                                  \
        }                                                                                                                \
        if (sub == 0) *reinterpret_cast<uint4*>(slot_i + RSMAX + SRC::STAGE_F) = make_uint4(m_row, m_v0, m_beg, m_end);  \
        cp_async_commit();                                                                                               \
        st_issue = st_issue + 1 == NST ? 0 : st_issue + 1;                                                               \
        ++it_meta; u_meta += u_step;                                                                                     \
        RA_LOAD_META();                                                                                                  \
    } while (0)
    RA_LOAD_META();
#pragma unroll
    for (int p = 0; p < NST - 1; ++p) RA_ISSUE();

    uint32_t u = gw * G + grp;
    for (uint32_t it = 0; it < n_it; ++it, u += u_step) {         // warp-uniform trip count
        RA_ISSUE();
        cp_async_wait<NST - 1>();
        __syncwarp();
        const float* slot = wbase + (size_t)st_use * G * SLOT;
        st_use = st_use + 1 == NST ? 0 : st_use + 1;
        const uint4 meta = *reinterpret_cast<const uint4*>(slot + RSMAX + SRC::STAGE_F);
        const uint32_t row = meta.x, v0 = meta.y, beg = meta.z, end = meta.w;
        const bool act = end > beg;
        float4 w = make_float4(0.f, 0.f, 0.f, 0.f), s1 = w, s2 = w, lr = w;
        if (act) {
            if (has_emb) {
                w = *reinterpret_cast<const float4*>(slot + sub * 4);
                lr = *reinterpret_cast<const float4*>(slot + K);
                if (emb_slots >= 1) s1 = *reinterpret_cast<const float4*>(slot + K + 4 + sub * 4);
                if (emb_slots >= 2) s2 = *reinterpret_cast<const float4*>(slot + 2 * K + 4 + sub * 4);
            } else {
                lr = *reinterpret_cast<const float4*>(slot);
            }
        }
        float4 g;
        float gl;
        row_grad_sum<K>(src, slot + RSMAX, aux, act, u, v0, beg, end, svals, row_piece0, piece_start, piece_sum, g, gl);
        if (act) row_step(tb, row, sub, w, s1, s2, lr, g, gl, SRC::SUB_E && src.sub_e(), emb_slots, od, ol, has_emb, has_lin, step, rr, rs);
        __syncwarp();      // the slot is overwritten by the copies issued in the next iteration
    }
    cp_async_wait<0>();
#undef RA_LOAD_META
#undef RA_ISSUE
}


// Requester side of the row-sharded step: per-unique-row gradient sums of the local batch (no table access here: the
// rows live on their owners), stored either as local gradient rows gsum[u] = {g[K], g_lin, pad} that the collectives
// send on (rt == nullptr), or straight into the owners' gradient segments over NVLink (rt).  Same warp-level cp.async
// pipeline as row_apply_kernel; what is staged per row is the first lookup's gradient operand and, for the fused
// source, the row E as it was fetched (dE = sum(dz s + dh0) - sum(dz) E).  A warp's G consecutive rows are contiguous
// at the destination unless they straddle two owners, so they leave as one staged, fully coalesced store.
template <int K, typename SRC>
struct RowGsumCfg {
    static constexpr int LPR = K / 4, G = 32 / LPR;
    static constexpr int SLOT = K + SRC::STAGE_F + 4;             // [E row | gradient operand | meta]
    static constexpr int NST = 3;
    static constexpr int OUT = G * (K + 4);                       // per-warp output tile
    static constexpr int SMEM = 8 * (NST * G * SLOT + OUT) * 4;
};

template <int K, typename SRC>
__global__ void __launch_bounds__(256, 2) row_gsum_kernel(const uint32_t* __restrict__ urow, const uint32_t* __restrict__ uval,
                                                          const uint32_t* __restrict__ svals, const uint32_t* __restrict__ row_start,
                                                          const uint32_t* __restrict__ row_piece0, const uint32_t* __restrict__ piece_start,
                                                          const SegCounts* __restrict__ cnt, SRC src, const float* __restrict__ piece_sum,
                                                          const PeerRoute* __restrict__ rt, float* __restrict__ gsum, bool skip_single) {
    // skip_single: rows with exactly one lookup were already stored by fused_rows_kernel (row-buffer mode)
    using C = RowGsumCfg<K, SRC>;
    constexpr int LPR = C::LPR, G = C::G, SLOT = C::SLOT, NST = C::NST, RW = K + 4, RW4 = RW / 4;
    extern __shared__ __align__(16) float ra_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = lane % LPR, grp = lane / LPR;
    float* wbase = ra_smem + ((size_t)warp * NST * G + grp) * SLOT;
    float* otile = ra_smem + (size_t)8 * NST * G * SLOT + (size_t)warp * C::OUT;
    float* aux = ra_smem + (size_t)8 * (NST * G * SLOT + C::OUT);
    src.aux_load(aux, threadIdx.x);
    __syncthreads();
    const bool sub_e = SRC::SUB_E && src.sub_e();
    const uint32_t U = cnt->n_rows;
    const uint32_t nw = gridDim.x * 8, gw = blockIdx.x * 8 + warp;
    const uint32_t n_chunks = (U + G - 1) / G;
    const uint32_t n_it = n_chunks > gw ? (n_chunks - gw - 1) / nw + 1 : 0;
    const uint32_t u_step = nw * G;
    uint32_t m_v0 = 0xffffffffu, m_beg = 0, m_end = 0;
    uint32_t u_meta = gw * G + grp, it_meta = 0;
    int st_issue = 0, st_use = 0;
#define RG_LOAD_META()                                                                                                   \
    do {                                                                                                                 \
        m_v0 = 0xffffffffu; m_beg = 0; m_end = 0;                                                                        \
        if (it_meta < n_it && u_meta < U) { m_v0 = __ldg(uval + u_meta); m_beg = __ldg(row_start + u_meta); m_end = __ldg(row_start + u_meta + 1); } \
        if (skip_single && m_end - m_beg == 1) m_end = m_beg;                                                            \
    } while (0)
#define RG_ISSUE()                                                                                                       \
    do {                                                                                                                 \
        float* slot_i = wbase + (size_t)st_issue * G * SLOT;                                                             \
        if (m_end > m_beg) {                                                                                             \
            if (sub_e) cp_async16(slot_i + sub * 4, src.erow + (size_t)u_meta * src.erow_stride + sub * 4);              \
            src.stage_async(m_v0, slot_i + K, sub);                                                                      \
        }                                                                                                                \
        if (sub == 0) *reinterpret_cast<uint4*>(slot_i + K + SRC::STAGE_F) = make_uint4(0u, m_v0, m_beg, m_end);         \
        cp_async_commit();                                                                                               \
        st_issue = st_issue + 1 == NST ? 0 : st_issue + 1;                                                               \
        ++it_meta; u_meta += u_step;                                                                                     \
        RG_LOAD_META();                                                                                                  \
    } while (0)
    RG_LOAD_META();
#pragma unroll
    for (int p = 0; p < NST - 1; ++p) RG_ISSUE();

    uint32_t u = gw * G + grp;
    for (uint32_t it = 0; it < n_it; ++it, u += u_step) {
        RG_ISSUE();
        cp_async_wait<NST - 1>();
        __syncwarp();
        const float* slot = wbase + (size_t)st_use * G * SLOT;
        st_use = st_use + 1 == NST ? 0 : st_use + 1;
        const uint4 meta = *reinterpret_cast<const uint4*>(slot + K + SRC::STAGE_F);
        const uint32_t v0 = meta.y, beg = meta.z, end = meta.w;
        const bool act = end > beg;
        float4 g;
        float gl;
        row_grad_sum<K>(src, slot + K, aux, act, u, v0, beg, end, svals, row_piece0, piece_start, piece_sum, g, gl);
        if (act && sub_e) {
            const float4 e = *reinterpret_cast<const float4*>(slot + sub * 4);
            g.x = fmaf(-gl, e.x, g.x); g.y = fmaf(-gl, e.y, g.y); g.z = fmaf(-gl, e.z, g.z); g.w = fmaf(-gl, e.w, g.w);
        }
        // the warp's rows -> one contiguous store (rows left out by skip_single are not touched: fused_rows_kernel stored them)
        const unsigned rowmask = __ballot_sync(0xffffffffu, act && sub == 0);
        reinterpret_cast<float4*>(otile + grp * RW)[sub] = g;
        if (sub == 0) *reinterpret_cast<float4*>(otile + grp * RW + K) = make_float4(gl, 0.f, 0.f, 0.f);
        __syncwarp();
        const uint32_t u0 = u - grp;                              // first row of this warp's chunk
        if (u0 < U && rowmask) {
            const uint32_t n_rows = min((uint32_t)G, U - u0);
            const int o0 = rt ? route_find(rt->send_off, rt->W, u0) : 0, o1 = rt ? route_find(rt->send_off, rt->W, u0 + n_rows - 1) : 0;
            if (o0 == o1) {
                float4* dst = reinterpret_cast<float4*>(rt ? rt->peer_grecv[o0] + (size_t)(rt->dst_off[o0] + (u0 - rt->send_off[o0])) * RW
                                                           : gsum + (size_t)u0 * RW);
                for (uint32_t j = lane; j < n_rows * RW4; j += 32)
                    if ((rowmask >> ((j / RW4) * LPR)) & 1u) dst[j] = reinterpret_cast<const float4*>(otile)[j];
            } else {
                for (uint32_t q = 0; q < n_rows; ++q) {
                    if (!((rowmask >> (q * LPR)) & 1u)) continue;
                    const uint32_t uu = u0 + q;
                    const int o = route_find(rt->send_off, rt->W, uu);
                    float4* dst = reinterpret_cast<float4*>(rt->peer_grecv[o] + (size_t)(rt->dst_off[o] + (uu - rt->send_off[o])) * RW);
                    if (lane < RW4) dst[lane] = reinterpret_cast<const float4*>(otile + q * RW)[lane];
                }
            }
        }
        __syncwarp();
    }
    cp_async_wait<0>();
#undef RG_LOAD_META
#undef RG_ISSUE
}
