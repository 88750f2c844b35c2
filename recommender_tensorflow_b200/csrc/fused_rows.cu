// Record-staged train step for small towers at the shapes BASELINE.json names (embedding_size 16, first hidden layer 16):
// ONE persistent kernel per step does gather + FM + tower forward/backward + the sparse optimizer of every table row that
// is looked up exactly once in the batch (with large tables that is almost every row), so such a row's record crosses
// HBM once in each direction per step instead of read (forward) + read + write (optimizer).
//
//   trainers/deep_fm.py:39      linear_model      }
//   trainers/deep_fm.py:52-73   input_layer       }  whole 208-byte table records [w | lin,m,v,last | m[K] | v[K]] are
//   trainers/deep_fm.py:79-87   FM block          }  brought into shared memory by 1-D bulk copies (TMA, cp.async.bulk,
//   trainers/deep_fm.py:93-112  DNN block         }  completion on an mbarrier) issued by a producer warp a tile ahead
//   trainers/deep_fm.py:114-125 head, loss
//   trainers/model_utils.py:57-66 optimizer       the non-lazy Adam decay is replayed in place (replay.cuh), the gradient
//                                                 of a once-only row is applied in place and the record leaves by a bulk
//                                                 store; rows looked up several times in the batch are left untouched
//                                                 and go through the sorted, ordered reduction (row_apply_kernel) afterwards
//
// Which lookups are "once only" is read from a 2-bit-per-slot claim table (L2 resident, filled by transform_kernel with
// one atomicOr per lookup: 01 = seen once, 11 = seen more than once; slot = global row mod table size, so a collision can
// only send a once-only row down the sorted path, never the reverse).  Both consumers of the table (this kernel and
// row_apply_kernel) apply the same test, so every row is updated by exactly one of them.
//
// Tile = 8 samples (the N of mma.m16n8k8), 16 consumer warps: two warps replay / FM-reduce one sample, then the three
// layer-0 products
//      H^T  [16 x 8]   = W0^T [16 x D] . E^T [D x 8]            (k-steps split over the warps, partials combined in order)
//      dW0  [D x 16]  += E^T  [D x 8]  . dh1' [8 x 16]          (warp w owns the fields w, w+16, ..; fp32 register accumulators)
//      dE^T [K x 8]    = W0_f [K x 16] . dh1'^T [16 x 8]        (per field; staged through shared memory so that the optimizer
//                                                                runs row-wise on float4 slices of the record)
// run on the tensor cores as 3xTF32 (a_hi b_hi + a_lo b_hi + a_hi b_lo, large and small terms in separate accumulators,
// every MMA chain at most 5 k-steps long and folded into fp32 registers with round-to-nearest adds).
// The in-kernel Adam step forms m and v in TF's float32 op order; the displacement alpha m / (sqrt(v) + eps) uses the MUFU
// sqrt / reciprocal (relative error <= 2^-21 on a displacement of ~lr, i.e. ~1e-10 on w; the IEEE sequence cost 20 % of the
// kernel's instructions, profiles/r02u).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "fused_rows_args.cuh"
#include "tc_gemm.cuh"

__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(tc::smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(tc::smem_u32(bar)) : "memory");
}
// completion of this thread's earlier cp.async copies counts as one (pre-counted) arrival on the mbarrier
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(tc::smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bar_consumers() { asm volatile("bar.sync 1, %0;" ::"n"(FR_CW * 32) : "memory"); }
constexpr int FR_P3W = 8;                      // warps that run the small upper part of the tower (P3)
__device__ __forceinline__ void bar_p3() { asm volatile("bar.sync 2, %0;" ::"n"(FR_P3W * 32) : "memory"); }

// "slot s may be refilled": one hardware barrier per slot (ids 3 ..), consumers arrive without waiting, the producer
// warps wait in bar.sync and issue nothing meanwhile (an mbarrier try_wait loop, even with nanosleep back-off, was 23 %
// of the kernel's issued instructions in profiles/r02au).  The rounds of one barrier cannot mix: the consumers' arrival
// for tile it + NSLOT needs the producers' copies of that tile, which are issued after their wait for tile it returned.
constexpr int FR_BAR_SLOT = 3;
__device__ __forceinline__ void slot_free_arrive(int s) { asm volatile("bar.arrive %0, %1;" ::"r"(FR_BAR_SLOT + s), "n"(FR_THREADS) : "memory"); }
__device__ __forceinline__ void slot_free_wait(int s) { asm volatile("bar.sync %0, %1;" ::"r"(FR_BAR_SLOT + s), "n"(FR_THREADS) : "memory"); }

// non-blocking: has the phase with this parity completed?  (acquire: the bulk copies it counted are visible afterwards)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(tc::smem_u32(bar)), "r"(parity) : "memory");
    return done != 0;
}
// D = A(16x8, row) * B(8x8, col) + C on tf32 operands held as fp32 bit patterns whose low 13 bits are zero
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2], const float (&c)[4]) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%10, %11, %12, %13};"
                 : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(c[3]));
}
// fp32 -> tf32 hi / lo operands of the 3xTF32 products.  cvt.rna.tf32.f32 is emulated on sm_100a (add 0x1000, infinity test,
// select, mask: 9 instructions per split, 14 % of this kernel's instruction stream in profiles/r02au).  mma.sync reads only
// the upper 19 bits of a tf32 operand, so "bits + 0x1000" IS the round-to-nearest (ties away) operand; the mask is only
// needed where hi is used as a number, i.e. in the subtraction.  Same values as cvt.rna for every finite input below 2^127.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(x) + 0x1000u;
    lo = __float_as_uint(x - __uint_as_float(hi & 0xffffe000u)) + 0x1000u;
}
// sparse optimizer step of one element inside the kernel (see the note on the Adam displacement above)
// FAST: instantiation for Adam everywhere with the closed-form replay - the other optimizers (IEEE divisions / square
// roots) and the step-by-step replay fallback (double-precision pow) are not compiled in at all
template <bool FAST>
__device__ __forceinline__ void apply_elem(float& w, float& s1, float& s2, float g, const OptDev& o) {
    if (FAST || o.kind == DFM_OPT_ADAM) {
        s1 = __fadd_rn(__fmul_rn(s1, o.b1), __fmul_rn(g, o.omb1));
        s2 = __fadd_rn(__fmul_rn(s2, o.b2), __fmul_rn(__fmul_rn(g, g), o.omb2));
        w -= fast_upd(s1, s2, o.alpha, o.eps);
    } else {
        other_apply(w, s1, s2, g, o);
    }
}
template <bool FAST>
__device__ __forceinline__ void fr_replay_row(float4& w, float4& m, float4& v, float4& lr, bool lin_lane, const RowReplay& rr,
                                              const ReplayStep& rs, const OptDev& od, const OptDev& ol) {
    if constexpr (FAST) {      // replay_row's common case: same arithmetic, same order
        const int last = __float_as_int(lr.w);
        if (rr.upto < 0 || last >= rr.upto) return;
        const ReplayCoef c = replay_coef(rr.rd, rs, last);
        replay_elem(w.x, m.x, v.x, c, od.eps); replay_elem(w.y, m.y, v.y, c, od.eps);
        replay_elem(w.z, m.z, v.z, c, od.eps); replay_elem(w.w, m.w, v.w, c, od.eps);
        if (rr.lin_adam && lin_lane) replay_elem(lr.x, lr.y, lr.z, c, ol.eps);
        lr.w = __int_as_float(rr.upto);
    } else {
        replay_row(w, m, v, lr, lin_lane, rr, rs, od, ol);
    }
}
// 3xTF32 product: main += a_hi b_hi;  cross += a_lo b_hi + a_hi b_lo
__device__ __forceinline__ void mma3(float (&cm)[4], float (&cx)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                     const uint32_t (&bh)[2], const uint32_t (&bl)[2]) {
    mma_tf32(cm, ah, bh, cm);
    mma_tf32(cx, al, bh, cx);
    mma_tf32(cx, ah, bl, cx);
}

// RB (row-buffer mode, the row-sharded requester): the rows were fetched from their owners into a row buffer
// [unique row][w[K] | lin, pad] (ES = 0 records of K + 4 floats, nothing to replay), the table lives elsewhere: the
// gradient row of a row looked up once in the local batch is stored straight into its owner's gradient segment (peer
// memory over NVLink, or the local send buffer of the collective path); rows looked up several times are left to
// row_gsum_kernel, which skips the single ones.
template <int K, int H1, int ES, bool RB, bool FAST>
__global__ void __launch_bounds__(FR_THREADS, 1) fused_rows_kernel(FusedRowsArgs A) {
    static_assert(!RB || ES == 0, "row-buffer records carry no optimizer slots");
    static_assert(K == 16 && H1 == 16, "instantiated for embedding_size 16 / first hidden layer 16");
    constexpr int NT = FR_CW * 32;                               // consumer threads
    const FusedArgs& a = A.f;
    const SmallMlpDesc& m = a.m;
    extern __shared__ __align__(16) float smem[];
    const int D = a.D, dc = a.dc, dn = a.dn, d = dc + dn;
    constexpr int RS = K + 4 + ES * K;                           // floats per staged record
    const int SST = A.sst;
    const int nrows = FR_TS * dc;
    // Shared-memory carve-up: the offsets come from the host (fr_layout).  Computed here they are chains of a dozen
    // dependent integer operations on kernel parameters, and the compiler re-derives them inside the tile loop rather
    // than hold fifteen pointers in registers: 15 % of the kernel's instructions in profiles/r02bc were this arithmetic.
    const FrLayout& L = A.lay;
    float* W0s = smem;                                           // [D][FR_W0S]
    float* ups = smem + L.ups;
    float* gup = smem + L.gup;
    float* slots = smem + L.slots;                               // [NSLOT][TS][SST]
    uint32_t* rowix = reinterpret_cast<uint32_t*>(smem + L.rowix);               // [NSLOT][TS*dc] global row (~0: no row)
    uint32_t* once = reinterpret_cast<uint32_t*>(smem + L.once);                 // [NSLOT][TS*dc] 1: this kernel applies the row's gradient
    float* xsb = smem + L.xsb;                                   // [NSLOT][TS][dn]
    float* ysb = smem + L.ysb;                                   // [NSLOT][TS] labels (a global load would sit on P3's critical path)
    float* part = smem + L.part;                                 // [CW][TS][H1] layer-0 partials; later the warps' dE staging
    float* p1 = smem + L.p1;                                     // [CW][2K + 4] FM / linear partials of P1
    float* dh1s = smem + L.dh1s;                                 // [TS][H1]
    float* acts = smem + L.acts;                                 // [TS][act_stride]
    float* dacts = smem + L.dacts;
    float* zs = smem + L.zs;                                     // [TS]
    float* dzs = smem + L.dzs;
    float* red = smem + L.red;
    float* ss = smem + L.ss;                                     // [TS][K]
    float* gnum = smem + L.gnum;                                 // [dn*K | dn] numeric_embeddings / numeric linear gradients of this CTA
    const int n_gnum = dn * K + dn;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
    uint64_t* full = bars;                                       // [NSLOT] records landed

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int train = a.train;
    const int ntiles = (a.B + FR_TS - 1) / FR_TS;
    if (tid == 0) {
        for (int s = 0; s < FR_NSLOT; ++s) tc::mbar_init(&full[s], FR_PW);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < D * H1; i += FR_THREADS) W0s[(i / H1) * FR_W0S + (i % H1)] = a.dw[m.off_W[0] + i];
    for (int i = tid; i < m.up_count; i += FR_THREADS) { ups[i] = a.dw[m.up_begin + i]; gup[i] = 0.f; }
    for (int i = tid; i < n_gnum; i += FR_THREADS) gnum[i] = 0.f;
    __syncthreads();

    // =========================================================================================== producer warps
    // A warp issues its bulk copies one after the other (~90 cycles each, measured: tools/gather_bench.cu - one issuing
    // warp per SM moves 0.66 TB/s chip-wide, 16 warps 4.6 TB/s), so the rows of a tile are split over FR_PW warps.
    if (warp >= FR_CW) {
        constexpr uint32_t rsb = (uint32_t)RS * 4u;
        const int pw = warp - FR_CW;
        const int per = (nrows + FR_PW - 1) / FR_PW;         // rows of a tile per producer warp (<= 32 * FR_NR)
        const int r0 = pw * per, r1 = min(nrows, r0 + per);
        int32_t idn[FR_NR];
        auto load_ids = [&](int tile) {
#pragma unroll
            for (int q = 0; q < FR_NR; ++q) {
                const int r = r0 + lane + 32 * q;
                idn[q] = -1;
                if (tile < ntiles && r < r1) {
                    const int64_t gi = (int64_t)tile * nrows + r;
                    if (gi < (int64_t)a.B * dc) {
                        if (RB) {          // unique-row index of the lookup (~0: no row) + "looked up once" flag in bit 30
                            const uint32_t u = __ldg(a.uidx + gi);
                            idn[q] = u == 0xffffffffu ? -1 : (int32_t)(u | (__ldg(A.once_lk + gi) ? 0x40000000u : 0u));
                        } else {
                            idn[q] = __ldg(a.ids + gi);
                        }
                    }
                }
            }
        };
        load_ids(blockIdx.x);
        int it = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int s = it % FR_NSLOT;
            if (it >= FR_NSLOT) slot_free_wait(s);
            float* slot = slots + (size_t)s * FR_TS * SST;
            uint32_t row[FR_NR], cw[FR_NR];
#pragma unroll
            for (int q = 0; q < FR_NR; ++q) {
                const int r = r0 + lane + 32 * q;
                row[q] = 0xffffffffu; cw[q] = 0;
                if (r < r1 && idn[q] >= 0) row[q] = RB ? ((uint32_t)idn[q] & 0x3fffffffu) : __ldg(a.row_off + r % dc) + (uint32_t)idn[q];
            }
            if (!RB && train && A.claim) {
#pragma unroll
                for (int q = 0; q < FR_NR; ++q)
                    if (row[q] != 0xffffffffu) cw[q] = __ldg(A.claim + ((row[q] & A.claim_mask) >> 4));
            }
            uint32_t nvalid = 0;
#pragma unroll
            for (int q = 0; q < FR_NR; ++q) {
                const int r = r0 + lane + 32 * q;
                if (r < r1) {
                    uint32_t one = 0;
                    if (row[q] != 0xffffffffu) {
                        ++nvalid;
                        if (RB) one = ((uint32_t)idn[q] >> 30) & 1u;
                        else one = ((cw[q] >> (((row[q] & A.claim_mask) & 15u) * 2u)) & 3u) == 1u ? 1u : 0u;
                    } else {
                        const int sl = r / dc, f = r - sl * dc;
                        float* dst = slot + (size_t)sl * SST + f * RS;
                        for (int c = 0; c < RS; c += 4) *reinterpret_cast<float4*>(dst + c) = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    rowix[s * nrows + r] = row[q];
                    once[s * nrows + r] = one;
                }
            }
            for (int q = pw * 32 + lane; q < FR_TS * dn; q += 32 * FR_PW) {
                const int j = q / FR_TS, sl = q - j * FR_TS, b = tile * FR_TS + sl;
                xsb[(s * FR_TS + sl) * dn + j] = b < a.B ? __ldg(a.bp.num[j] + b) : 0.f;
            }
            if (pw == FR_PW - 1 && lane < FR_TS) {
                const int b = tile * FR_TS + lane;
                ysb[s * FR_TS + lane] = (train && b < a.B) ? __ldg(a.labels + b) : 0.f;
            }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) nvalid += __shfl_xor_sync(0xffffffffu, nvalid, o);
            __syncwarp();                                   // this warp's meta data is written before its arrival ...
            if (lane == 0) tc::mbar_expect_tx(&full[s], nvalid * rsb);      // ... which also announces its byte count
            __syncwarp();
#pragma unroll
            for (int q = 0; q < FR_NR; ++q) {
                const int r = r0 + lane + 32 * q;
                if (r < r1 && row[q] != 0xffffffffu) {
                    const int sl = r / dc, f = r - sl * dc;
                    const float* srcp = RB ? a.rowbuf + (size_t)row[q] * a.rowbuf_stride : a.tb.rec + (size_t)row[q] * a.tb.stride;
                    bulk_load(slot + (size_t)sl * SST + f * RS, srcp, rsb, &full[s]);
                }
            }
            load_ids(tile + gridDim.x);                     // in flight while the consumers work
        }
        for (int q = max(it - FR_NSLOT, 0); q < it; ++q) slot_free_wait(q % FR_NSLOT);     // pair the consumers' last arrivals
        return;
    }

    // =========================================================================================== consumer warps
    auto UP = [&](int packed_off) { return ups + (packed_off - m.up_begin); };
    auto GUP = [&](int packed_off) { return gup + (packed_off - m.up_begin); };
    const float* num_emb = a.off_num_emb >= 0 ? a.dw + a.off_num_emb : nullptr;
    const float* num_lin = a.off_num_lin >= 0 ? a.dw + a.off_num_lin : nullptr;
    const float bias0 = (a.use_linear && a.off_bias >= 0) ? a.dw[a.off_bias] : 0.f;
    const ReplayStep rs = replay_step_load(a.rr.rd.closed ? a.rr.rd : a.rr.rl, a.rr.upto);
    const int g = lane >> 2, t = lane & 3;                   // MMA fragment coordinates (also: P1 field group / float4 slice)
    const bool use_mf = a.use_mf != 0, use_lin = a.use_linear != 0;
    const bool inline_apply = train && (RB || A.claim != nullptr);
    float wacc[FR_NF][2][4];                                 // dW0 of this warp's fields: [field][unit tile][fragment]
#pragma unroll
    for (int i = 0; i < FR_NF; ++i) {
#pragma unroll
        for (int n = 0; n < 2; ++n) { wacc[i][n][0] = 0.f; wacc[i][n][1] = 0.f; wacc[i][n][2] = 0.f; wacc[i][n][3] = 0.f; }
    }
    float loss_acc = 0.f, dz_acc = 0.f;
    float* gst = part + (size_t)warp * FR_TS * H1;           // this warp's [8 samples][16] staging of a field's dE (chunk-swizzled)

    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int s = it % FR_NSLOT;
        const int b0 = tile * FR_TS;
        float* slot = slots + (size_t)s * FR_TS * SST;
        const uint32_t* rix = rowix + s * nrows;
        const uint32_t* onc = once + s * nrows;
        const float* xs = xsb + (size_t)s * FR_TS * dn;
        const float* ys = ysb + s * FR_TS;
        tc::mbar_wait(&full[s], (it / FR_NSLOT) & 1);
        // ------------------------------------------------------------------ P1: two warps per sample: replay in place, FM / linear partial sums
        if (!(A.ablate & 64)) {
            const int sl = warp / FR_WPS, half = warp - sl * FR_WPS, sub = t;     // FR_WPS warps share a sample: fields half*8+g, +8*FR_WPS, ..
            float* srow = slot + (size_t)sl * SST;
            float4 sv = make_float4(0.f, 0.f, 0.f, 0.f), qv = sv;
            float lin = 0.f;
#pragma unroll 2
            for (int f = half * 8 + g; f < dc; f += 8 * FR_WPS) {
                if (rix[sl * dc + f] != 0xffffffffu) {
                    float* rec = srow + f * RS;
                    float4 e = *reinterpret_cast<const float4*>(rec + sub * 4);
                    float4 lr = *reinterpret_cast<const float4*>(rec + K);
                    if (a.rr.upto >= 0 && __float_as_int(lr.w) < a.rr.upto && !(A.ablate & 1)) {
                        float4 mm = make_float4(0.f, 0.f, 0.f, 0.f), vv = mm;
                        if (ES >= 1) mm = *reinterpret_cast<const float4*>(rec + K + 4 + sub * 4);
                        if (ES >= 2) vv = *reinterpret_cast<const float4*>(rec + 2 * K + 4 + sub * 4);
                        fr_replay_row<FAST>(e, mm, vv, lr, sub == 0, a.rr, rs, a.od, a.ol);
                        *reinterpret_cast<float4*>(rec + sub * 4) = e;
                        if (ES >= 1) *reinterpret_cast<float4*>(rec + K + 4 + sub * 4) = mm;
                        if (ES >= 2) *reinterpret_cast<float4*>(rec + 2 * K + 4 + sub * 4) = vv;
                        if (sub == 0) *reinterpret_cast<float4*>(rec + K) = lr;
                    }
                    sv.x += e.x; sv.y += e.y; sv.z += e.z; sv.w += e.w;
                    qv.x = fmaf(e.x, e.x, qv.x); qv.y = fmaf(e.y, e.y, qv.y); qv.z = fmaf(e.z, e.z, qv.z); qv.w = fmaf(e.w, e.w, qv.w);
                    if (sub == 0) lin += lr.x;
                }
            }
            for (int j = half * 8 + g; j < dn; j += 8 * FR_WPS) {
                const float x = xs[sl * dn + j];
                float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
                if (num_emb) {
                    const float4 ve = __ldg(reinterpret_cast<const float4*>(num_emb + j * K) + sub);
                    e = make_float4(x * ve.x, x * ve.y, x * ve.z, x * ve.w);
                }
                *reinterpret_cast<float4*>(srow + dc * RS + j * K + sub * 4) = e;
                sv.x += e.x; sv.y += e.y; sv.z += e.z; sv.w += e.w;
                qv.x = fmaf(e.x, e.x, qv.x); qv.y = fmaf(e.y, e.y, qv.y); qv.z = fmaf(e.z, e.z, qv.z); qv.w = fmaf(e.w, e.w, qv.w);
                if (sub == 0 && use_lin && num_lin) lin = fmaf(x, __ldg(num_lin + j), lin);
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {               // fixed butterfly over the field groups
                sv.x += __shfl_xor_sync(0xffffffffu, sv.x, o); sv.y += __shfl_xor_sync(0xffffffffu, sv.y, o);
                sv.z += __shfl_xor_sync(0xffffffffu, sv.z, o); sv.w += __shfl_xor_sync(0xffffffffu, sv.w, o);
                qv.x += __shfl_xor_sync(0xffffffffu, qv.x, o); qv.y += __shfl_xor_sync(0xffffffffu, qv.y, o);
                qv.z += __shfl_xor_sync(0xffffffffu, qv.z, o); qv.w += __shfl_xor_sync(0xffffffffu, qv.w, o);
                lin += __shfl_xor_sync(0xffffffffu, lin, o);
            }
            float* pw = p1 + warp * (2 * K + 4);
            if (g == 0) {
                reinterpret_cast<float4*>(pw)[sub] = sv;
                reinterpret_cast<float4*>(pw + K)[sub] = qv;
                if (sub == 0) pw[2 * K] = lin;
            }
        }
        bar_consumers();
        // ------------------------------------------------------------------ P2: H^T = W0^T E^T, k-steps round-robin over the warps
        {
            float cm[4] = {0.f, 0.f, 0.f, 0.f}, cx[4] = {0.f, 0.f, 0.f, 0.f};
            for (int ks = warp; ks < ((A.ablate & 2) ? 0 : D / 8); ks += FR_CW) {
                const int col0 = ks * 8, f = col0 / K;
                const int off = f < dc ? f * RS + (col0 - f * K) : dc * RS + (col0 - dc * K);
                const float* w0 = W0s + (size_t)(col0 + t) * FR_W0S + g;
                const float* ep = slot + (size_t)g * SST + off + t;
                uint32_t ah[4], al[4], bh[2], bl[2];
                split_tf32(w0[0], ah[0], al[0]);
                split_tf32(w0[8], ah[1], al[1]);
                split_tf32(w0[4 * FR_W0S], ah[2], al[2]);
                split_tf32(w0[4 * FR_W0S + 8], ah[3], al[3]);
                split_tf32(ep[0], bh[0], bl[0]);
                split_tf32(ep[4], bh[1], bl[1]);
                mma3(cm, cx, ah, al, bh, bl);
            }
            float* pw = part + (size_t)warp * FR_TS * H1;    // [sample][unit]
            pw[(2 * t) * H1 + g] = cm[0] + cx[0];
            pw[(2 * t + 1) * H1 + g] = cm[1] + cx[1];
            pw[(2 * t) * H1 + g + 8] = cm[2] + cx[2];
            pw[(2 * t + 1) * H1 + g + 8] = cm[3] + cx[3];
        }
        bar_consumers();
        // ------------------------------------------------------------------ P3 (warps 0..7): rest of the tower, head, loss, backward to dh1'
        const bool p3_fast = m.L == 2 && m.H[1] == 16;       // the reference default tower [16, 16]: a sample lives in one half-warp
        if (p3_fast) {
            if (warp < 4 && !(A.ablate & 4)) {
                // thread = (sample sl, unit o); every cross-thread dependence stays inside a half-warp: no block barriers
                const int sl = tid >> 4, o = tid & 15, b = b0 + sl;
                const unsigned hm = 0xffffffffu;
                float* ar = acts + sl * m.act_stride;
                float* dr = dacts + sl * m.act_stride;
                // field sums of the two half-sample warps -> s (kept for the FM gradient), FM + linear logit
                const float* pa = p1 + (FR_WPS * sl) * (2 * K + 4);
                float sk = pa[o], qk = pa[K + o], lk = pa[2 * K];
#pragma unroll
                for (int w = 1; w < FR_WPS; ++w) { sk += pa[w * (2 * K + 4) + o]; qk += pa[w * (2 * K + 4) + K + o]; lk += pa[w * (2 * K + 4) + 2 * K]; }
                ss[sl * K + o] = sk;
                if (b < a.B && a.s_out) a.s_out[(size_t)b * K + o] = sk;
                float tq = sk * sk - qk;
#pragma unroll
                for (int x = 8; x >= 1; x >>= 1) tq += __shfl_xor_sync(hm, tq, x);
                float zlf = 0.f;
                if (use_lin) zlf += lk + bias0;
                if (use_mf) zlf += 0.5f * tq;
                // layer 0 (partials of P2 in warp order), layer 1, head
                float h1 = UP(m.off_b[0])[o];
#pragma unroll
                for (int w = 0; w < FR_CW; ++w) h1 += part[((size_t)w * FR_TS + sl) * H1 + o];
                h1 = fmaxf(h1, 0.f);
                ar[o] = h1;
                __syncwarp();
                const float* W1 = UP(m.off_W[1]);
                float h2 = UP(m.off_b[1])[o];
#pragma unroll
                for (int j = 0; j < 16; ++j) h2 = fmaf(ar[j], W1[j * 16 + o], h2);
                h2 = fmaxf(h2, 0.f);
                ar[16 + o] = h2;
                const float wo = UP(m.off_Wo)[o];
                // the head sums h2 . Wo in unit order like the general path
                float z = UP(m.off_bo)[0];
                {
                    const float* Wo = UP(m.off_Wo);
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 16; ++j) z = fmaf(ar[16 + j], Wo[j], z);
                }
                z += zlf;
                float gz = 0.f, lterm = 0.f;
                if (b < a.B && train) {
                    const float y = ys[sl];
                    lterm = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
                    gz = (1.f / (1.f + expf(-z)) - y) * a.scale;
                }
                if (o == 0) {
                    if (b < a.B) {
                        a.logits[b] = z;
                        if (a.logits_out) a.logits_out[b] = z;
                        if (train) a.dz_out[b] = gz;
                    }
                    dzs[sl] = gz;
                    red[sl] = lterm;
                }
                if (train) {
                    const float d2 = h2 > 0.f ? gz * wo : 0.f;
                    dr[16 + o] = d2;
                    __syncwarp();
                    float v = 0.f;
#pragma unroll
                    for (int q = 0; q < 16; ++q) v = fmaf(dr[16 + q], W1[o * 16 + q], v);
                    v = h1 > 0.f ? v : 0.f;
                    dr[o] = v;
                    dh1s[tid] = v;
                    if (b < a.B) a.dh1_out[(size_t)b * H1 + o] = v;
                }
            }
        }
        // The tower above layer 0 is small and serial (4 or 8 warps, ~2.8 K cycles per tile); the other consumer warps use
        // that window to replay the deferred Adam of the NEXT tile's records in place, if they have landed.  A replayed
        // record carries last_step = upto, so P1 of that tile skips it: same arithmetic on the same values, only earlier.
        {
            const int p3w = p3_fast ? 4 : FR_P3W;
            const int nt = tile + gridDim.x;
            if (!RB && warp >= p3w && nt < ntiles && a.rr.upto >= 0 && !(A.ablate & 1)) {
                const int s1 = (it + 1) % FR_NSLOT;
                uint32_t ok = lane == 0 ? (mbar_test(&full[s1], ((it + 1) / FR_NSLOT) & 1) ? 1u : 0u) : 0u;
                ok = __shfl_sync(0xffffffffu, ok, 0);
                if (ok) {
                    float* slot1 = slots + (size_t)s1 * FR_TS * SST;
                    const uint32_t* rix1 = rowix + s1 * nrows;
                    for (int r = (warp - p3w) * 8 + g; r < nrows; r += (FR_CW - p3w) * 8) {
                        if (rix1[r] != 0xffffffffu) {
                            const int sl = r / dc, f = r - sl * dc;
                            float* rec = slot1 + (size_t)sl * SST + f * RS;
                            float4 lr = *reinterpret_cast<const float4*>(rec + K);
                            if (__float_as_int(lr.w) < a.rr.upto) {
                                float4 e = *reinterpret_cast<const float4*>(rec + t * 4);
                                float4 mm = make_float4(0.f, 0.f, 0.f, 0.f), vv = mm;
                                if (ES >= 1) mm = *reinterpret_cast<const float4*>(rec + K + 4 + t * 4);
                                if (ES >= 2) vv = *reinterpret_cast<const float4*>(rec + 2 * K + 4 + t * 4);
                                fr_replay_row<FAST>(e, mm, vv, lr, t == 0, a.rr, rs, a.od, a.ol);
                                *reinterpret_cast<float4*>(rec + t * 4) = e;
                                if (ES >= 1) *reinterpret_cast<float4*>(rec + K + 4 + t * 4) = mm;
                                if (ES >= 2) *reinterpret_cast<float4*>(rec + 2 * K + 4 + t * 4) = vv;
                                if (t == 0) *reinterpret_cast<float4*>(rec + K) = lr;
                            }
                        }
                    }
                }
            }
        }
        if (!p3_fast && warp < FR_P3W) {
            constexpr int PT = FR_P3W * 32;
            if (tid < FR_TS * H1) {
                const int sl = tid / H1, o = tid - sl * H1;
                float v = UP(m.off_b[0])[o];
#pragma unroll
                for (int w = 0; w < FR_CW; ++w) v += part[((size_t)w * FR_TS + sl) * H1 + o];
                acts[sl * m.act_stride + o] = fmaxf(v, 0.f);
            } else {
                // field sums of the two half-sample warps -> s (kept for the FM gradient), FM + linear logit
                const int q = tid - FR_TS * H1, sl = q / K, k = q - sl * K;
                const float* pa = p1 + (FR_WPS * sl) * (2 * K + 4);
                float sk = pa[k], qk = pa[K + k], lk = pa[2 * K];
#pragma unroll
                for (int w = 1; w < FR_WPS; ++w) { sk += pa[w * (2 * K + 4) + k]; qk += pa[w * (2 * K + 4) + K + k]; lk += pa[w * (2 * K + 4) + 2 * K]; }
                ss[sl * K + k] = sk;
                if (b0 + sl < a.B && a.s_out) a.s_out[(size_t)(b0 + sl) * K + k] = sk;
                float tq = sk * sk - qk;
#pragma unroll
                for (int o = 8; o >= 1; o >>= 1) tq += __shfl_xor_sync(0xffffffffu, tq, o);
                if (k == 0) {
                    float z = 0.f;
                    if (use_lin) z += lk + bias0;
                    if (use_mf) z += 0.5f * tq;
                    zs[sl] = z;
                }
            }
            bar_p3();
            int aoff = 0;
            for (int l = 1; l < m.L; ++l) {
                const int Hin = m.H[l - 1], Hout = m.H[l];
                const float* W = UP(m.off_W[l]);
                const float* bb = UP(m.off_b[l]);
                for (int idx = tid; idx < FR_TS * Hout; idx += PT) {
                    const int sl = idx / Hout, o = idx - sl * Hout;
                    const float* arow = acts + sl * m.act_stride + aoff;
                    float v = bb[o];
                    for (int j = 0; j < Hin; ++j) v = fmaf(arow[j], W[j * Hout + o], v);
                    acts[sl * m.act_stride + aoff + Hin + o] = fmaxf(v, 0.f);
                }
                aoff += Hin;
                bar_p3();
            }
            const int HL = m.H[m.L - 1];
            const float* Wo = UP(m.off_Wo);
            if (tid < FR_TS) {
                const int sl = tid, b = b0 + sl;
                const float* arow = acts + sl * m.act_stride + aoff;
                float z = UP(m.off_bo)[0];
                for (int j = 0; j < HL; ++j) z = fmaf(arow[j], Wo[j], z);
                z += zs[sl];
                float gz = 0.f, lterm = 0.f;
                if (b < a.B) {
                    a.logits[b] = z;
                    if (a.logits_out) a.logits_out[b] = z;
                    if (train) {
                        const float y = ys[sl];
                        lterm = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
                        gz = (1.f / (1.f + expf(-z)) - y) * a.scale;
                        a.dz_out[b] = gz;
                    }
                }
                dzs[sl] = gz;
                red[sl] = lterm;
            }
            if (train) {
                bar_p3();
                for (int idx = tid; idx < FR_TS * HL; idx += PT) {
                    const int sl = idx / HL, j = idx - sl * HL;
                    dacts[sl * m.act_stride + aoff + j] = acts[sl * m.act_stride + aoff + j] > 0.f ? dzs[sl] * Wo[j] : 0.f;
                }
                bar_p3();
                int ao = aoff;
                for (int l = m.L - 1; l >= 1; --l) {
                    const int Hin = m.H[l - 1], Hout = m.H[l];
                    const float* W = UP(m.off_W[l]);
                    const int in_off = ao - Hin;
                    for (int idx = tid; idx < FR_TS * Hin; idx += PT) {
                        const int sl = idx / Hin, j = idx - sl * Hin;
                        const float* drow = dacts + sl * m.act_stride + ao;
                        float v = 0.f;
                        for (int o = 0; o < Hout; ++o) v = fmaf(drow[o], W[j * Hout + o], v);
                        dacts[sl * m.act_stride + in_off + j] = acts[sl * m.act_stride + in_off + j] > 0.f ? v : 0.f;
                    }
                    ao = in_off;
                    bar_p3();
                }
                if (tid < FR_TS * H1) {
                    const int sl = tid / H1, j = tid - sl * H1;
                    const float v = dacts[sl * m.act_stride + j];
                    dh1s[tid] = v;
                    if (b0 + sl < a.B) a.dh1_out[(size_t)(b0 + sl) * H1 + j] = v;
                } else {
                    // gradients of everything above W0: each output owned by one thread, samples walked in order
                    const int gt = tid - FR_TS * H1, gn = PT - FR_TS * H1;
                    int go = 0;
                    for (int l = 0; l < m.L; ++l) {
                        const int Hl = m.H[l];
                        for (int j = gt; j < Hl; j += gn) {
                            float v = 0.f;
                            for (int r = 0; r < FR_TS; ++r) v += dacts[r * m.act_stride + go + j];
                            GUP(m.off_b[l])[j] += v;
                        }
                        if (l + 1 < m.L) {
                            const int Hn = m.H[l + 1];
                            for (int qx = gt; qx < Hl * Hn; qx += gn) {
                                const int j = qx / Hn, o = qx - j * Hn;
                                float v = 0.f;
                                for (int r = 0; r < FR_TS; ++r) v = fmaf(acts[r * m.act_stride + go + j], dacts[r * m.act_stride + go + Hl + o], v);
                                GUP(m.off_W[l + 1])[qx] += v;
                            }
                        } else {
                            for (int j = gt; j < Hl; j += gn) {
                                float v = 0.f;
                                for (int r = 0; r < FR_TS; ++r) v = fmaf(acts[r * m.act_stride + go + j], dzs[r], v);
                                GUP(m.off_Wo)[j] += v;
                            }
                        }
                        go += Hl;
                    }
                    if (gt == 0) {
                        float x = 0.f, c = 0.f;
                        for (int r = 0; r < FR_TS; ++r) { x += red[r]; c += dzs[r]; }
                        loss_acc += x;
                        dz_acc += c;
                    }
                }
            }
        }
        bar_consumers();                                      // dh1', dz, s of the tile are ready
        if (train && p3_fast && warp >= 4 && warp < 8) {
            // gradients of everything above W0 (fast path): each output owned by one thread, samples walked in order
            const int gt = tid - 128;
#pragma unroll
            for (int q = 0; q < 2; ++q) {                     // dW1[j][o]
                const int qx = gt + 128 * q, j = qx >> 4, o = qx & 15;
                float v = 0.f;
#pragma unroll
                for (int r = 0; r < FR_TS; ++r) v = fmaf(acts[r * m.act_stride + j], dacts[r * m.act_stride + 16 + o], v);
                GUP(m.off_W[1])[qx] += v;
            }
            if (gt < 16) {
                float v = 0.f;
                for (int r = 0; r < FR_TS; ++r) v += dacts[r * m.act_stride + gt];
                GUP(m.off_b[0])[gt] += v;
            } else if (gt < 32) {
                const int j = gt - 16;
                float v = 0.f;
                for (int r = 0; r < FR_TS; ++r) v += dacts[r * m.act_stride + 16 + j];
                GUP(m.off_b[1])[j] += v;
            } else if (gt < 48) {
                const int j = gt - 32;
                float v = 0.f;
                for (int r = 0; r < FR_TS; ++r) v = fmaf(acts[r * m.act_stride + 16 + j], dzs[r], v);
                GUP(m.off_Wo)[j] += v;
            } else if (gt == 48) {
                float x = 0.f, c = 0.f;
                for (int r = 0; r < FR_TS; ++r) { x += red[r]; c += dzs[r]; }
                loss_acc += x;
                dz_acc += c;
            }
        }
        if (train) {
            // -------------------------------------------------------------- P4/P5: warp w owns the fields w, w + 16, ..
            uint32_t bWh[2][2], bWl[2][2];                   // dh1' as B of the dW0 product: [unit tile][k = sample t, t + 4]
            uint32_t bEh[2][2], bEl[2][2];                   // dh1'^T as B of the dE product: [k-step over units][k = unit t, t + 4], n = sample g
#pragma unroll
            for (int n = 0; n < 2; ++n) {
                split_tf32(dh1s[t * H1 + n * 8 + g], bWh[n][0], bWl[n][0]);
                split_tf32(dh1s[(t + 4) * H1 + n * 8 + g], bWh[n][1], bWl[n][1]);
                split_tf32(dh1s[g * H1 + n * 8 + t], bEh[n][0], bEl[n][0]);
                split_tf32(dh1s[g * H1 + n * 8 + t + 4], bEh[n][1], bEl[n][1]);
            }
            const float zero4[4] = {0.f, 0.f, 0.f, 0.f};
            const float dzr = dzs[g];                         // row-wise view of the update: lane = (sample g, float4 slice t)
#pragma unroll
            for (int i = 0; i < FR_NF; ++i) {
                const int f = A.p4f[warp * FR_NF + i];        // dW0 fields of this warp (fixed: register accumulators)
                if (f < d && !(A.ablate & 8)) {               // warp-uniform
                    const int off = f < dc ? f * RS : dc * RS + (f - dc) * K;
                    // dW0[f*K.., :] += E_f^T dh1'
                    {
                        const float* ep = slot + (size_t)t * SST + off + g;
                        uint32_t ah[4], al[4];
                        split_tf32(ep[0], ah[0], al[0]);
                        split_tf32(ep[8], ah[1], al[1]);
                        split_tf32(ep[4 * (size_t)SST], ah[2], al[2]);
                        split_tf32(ep[4 * (size_t)SST + 8], ah[3], al[3]);
#pragma unroll
                        for (int n = 0; n < 2; ++n) {
                            float dm[4], dx[4];
                            mma_tf32(dm, ah, bWh[n], zero4);
                            mma_tf32(dx, al, bWh[n], zero4);
                            mma_tf32(dx, ah, bWl[n], dx);
#pragma unroll
                            for (int q = 0; q < 4; ++q) wacc[i][n][q] += dm[q] + dx[q];
                        }
                    }
                }
            }
            // dE + update tasks are dealt separately from the dW0 fields so that the warps finish together (39 fields over
            // 16 warps as "field f -> warp f mod 16" left the three-field warps 23 % over the mean: fr_balance)
#pragma unroll
            for (int i = 0; i < FR_N5; ++i) {
                const int f = A.p5f[warp * FR_N5 + i];
                if (f < d) {                                  // warp-uniform
                    const int off = f < dc ? f * RS : dc * RS + (f - dc) * K;
                    if (f >= dc || inline_apply) {
                        // dE_f^T = W0_f dh1'^T  (fragment: k = g, g + 8; samples 2t, 2t + 1)
                        float cm[4] = {0.f, 0.f, 0.f, 0.f}, cx[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                        for (int kk = 0; kk < ((A.ablate & 16) ? 0 : 2); ++kk) {
                            const float* w0 = W0s + (size_t)(f * K + g) * FR_W0S + kk * 8 + t;
                            uint32_t ah[4], al[4];
                            split_tf32(w0[0], ah[0], al[0]);
                            split_tf32(w0[8 * FR_W0S], ah[1], al[1]);
                            split_tf32(w0[4], ah[2], al[2]);
                            split_tf32(w0[8 * FR_W0S + 4], ah[3], al[3]);
                            mma3(cm, cx, ah, al, bEh[kk], bEl[kk]);
                        }
                        // fragment -> [sample][k] staging; 16-byte chunk c of sample sl sits at chunk c ^ (sl >> 1)
                        __syncwarp();
                        {
                            const int c0 = ((g >> 2) ^ t) * 4 + (g & 3), c1 = (((g >> 2) + 2) ^ t) * 4 + (g & 3);
                            gst[(2 * t) * K + c0] = cm[0] + cx[0];
                            gst[(2 * t + 1) * K + c0] = cm[1] + cx[1];
                            gst[(2 * t) * K + c1] = cm[2] + cx[2];
                            gst[(2 * t + 1) * K + c1] = cm[3] + cx[3];
                        }
                        __syncwarp();
                        float4 gr = *reinterpret_cast<const float4*>(gst + g * K + ((t ^ (g >> 1)) & 3) * 4);    // lane = (sample g, slice t)
                        if (RB && f < dc) {
                            if (onc[g * dc + f]) {
                                const float* rec = slot + (size_t)g * SST + off;
                                if (use_mf) {
                                    const float4 w = *reinterpret_cast<const float4*>(rec + t * 4);
                                    const float4 sv = *reinterpret_cast<const float4*>(ss + g * K + t * 4);
                                    gr.x = fmaf(dzr, sv.x - w.x, gr.x); gr.y = fmaf(dzr, sv.y - w.y, gr.y);
                                    gr.z = fmaf(dzr, sv.z - w.z, gr.z); gr.w = fmaf(dzr, sv.w - w.w, gr.w);
                                }
                                const uint32_t u = rix[g * dc + f];
                                float* dst;
                                if (A.route) {
                                    const PeerRoute* rt = A.route;
                                    const int o = route_find(rt->send_off, rt->W, u);
                                    dst = rt->peer_grecv[o] + (size_t)(rt->dst_off[o] + (u - rt->send_off[o])) * (K + 4);
                                } else {
                                    dst = A.gsum + (size_t)u * (K + 4);
                                }
                                *reinterpret_cast<float4*>(dst + t * 4) = gr;
                                if (t == 0) *reinterpret_cast<float4*>(dst + K) = make_float4(dzr, 0.f, 0.f, 0.f);
                            }
                        } else if (f < dc) {
                            if (onc[g * dc + f] && !(A.ablate & 32)) {
                                float* rec = slot + (size_t)g * SST + off;
                                float4 w = *reinterpret_cast<const float4*>(rec + t * 4);
                                float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
                                if (ES >= 1) s1 = *reinterpret_cast<const float4*>(rec + K + 4 + t * 4);
                                if (ES >= 2) s2 = *reinterpret_cast<const float4*>(rec + 2 * K + 4 + t * 4);
                                if (use_mf) {
                                    const float4 sv = *reinterpret_cast<const float4*>(ss + g * K + t * 4);
                                    gr.x = fmaf(dzr, sv.x - w.x, gr.x); gr.y = fmaf(dzr, sv.y - w.y, gr.y);
                                    gr.z = fmaf(dzr, sv.z - w.z, gr.z); gr.w = fmaf(dzr, sv.w - w.w, gr.w);
                                }
                                if (!(A.ablate & 256)) {
                                apply_elem<FAST>(w.x, s1.x, s2.x, gr.x, A.od_t); apply_elem<FAST>(w.y, s1.y, s2.y, gr.y, A.od_t);
                                apply_elem<FAST>(w.z, s1.z, s2.z, gr.z, A.od_t); apply_elem<FAST>(w.w, s1.w, s2.w, gr.w, A.od_t);
                                }
                                // the record goes straight back to the table (4 lanes = 64 contiguous bytes per store)
                                float* grec = a.tb.rec + (size_t)rix[g * dc + f] * a.tb.stride;
                                if (A.ablate & 128) grec = gst;
                                *reinterpret_cast<float4*>(grec + t * 4) = w;
                                if (ES >= 1) *reinterpret_cast<float4*>(grec + K + 4 + t * 4) = s1;
                                if (ES >= 2) *reinterpret_cast<float4*>(grec + 2 * K + 4 + t * 4) = s2;
                                if (t == 0) {
                                    float4 lr = *reinterpret_cast<const float4*>(rec + K);
                                    if (use_lin) apply_elem<FAST>(lr.x, lr.y, lr.z, dzr, A.ol_t);
                                    lr.w = __int_as_float(A.step);
                                    *reinterpret_cast<float4*>(grec + K) = lr;
                                }
                            }
                        } else {
                            // numeric field j: d numeric_embeddings[j, k] += sum_b x_bj dE[b, dc + j, k];  d numeric linear[j] += sum_b x_bj dz_b
                            const int j = f - dc;
                            const float x = xs[g * dn + j];
                            if (use_mf) {
                                const float4 sv = *reinterpret_cast<const float4*>(ss + g * K + t * 4);
                                const float4 e = *reinterpret_cast<const float4*>(slot + (size_t)g * SST + off + t * 4);
                                gr.x = fmaf(dzr, sv.x - e.x, gr.x); gr.y = fmaf(dzr, sv.y - e.y, gr.y);
                                gr.z = fmaf(dzr, sv.z - e.z, gr.z); gr.w = fmaf(dzr, sv.w - e.w, gr.w);
                            }
                            float4 u = make_float4(x * gr.x, x * gr.y, x * gr.z, x * gr.w);
                            float ul = x * dzr;
#pragma unroll
                            for (int o = 4; o < 32; o <<= 1) {           // over the samples (fixed butterfly)
                                u.x += __shfl_xor_sync(0xffffffffu, u.x, o); u.y += __shfl_xor_sync(0xffffffffu, u.y, o);
                                u.z += __shfl_xor_sync(0xffffffffu, u.z, o); u.w += __shfl_xor_sync(0xffffffffu, u.w, o);
                                ul += __shfl_xor_sync(0xffffffffu, ul, o);
                            }
                            if (g == 0) {                                // field j belongs to this warp alone: plain read-modify-write
                                float4* gp = reinterpret_cast<float4*>(gnum + j * K + t * 4);
                                float4 v = *gp;
                                v.x += u.x; v.y += u.y; v.z += u.z; v.w += u.w;
                                *gp = v;
                                if (t == 0) gnum[dn * K + j] += ul;
                            }
                        }
                    }
                }
            }
        }
        // this thread is done with the slot (the scratch of the tile is protected by the barrier after the next tile's P1)
        __syncwarp();
        fence_async_smem();                                   // this thread's writes to the slot precede the next bulk copies into it
        slot_free_arrive(s);
    }
    if (train) {
        const int acc_tid = (m.L == 2 && m.H[1] == 16) ? 128 + 48 : FR_TS * H1;   // the thread that accumulated the loss / dz sums
        if (tid == acc_tid) GUP(m.off_bo)[0] = dz_acc;
        bar_consumers();
        for (int i = tid; i < m.up_count; i += NT) a.up_partial[(size_t)blockIdx.x * m.up_count + i] = gup[i];
        for (int i = tid; i < n_gnum; i += NT) A.numg_partial[(size_t)blockIdx.x * n_gnum + i] = gnum[i];
        float* wp = a.w0_partial + (size_t)blockIdx.x * D * H1;
#pragma unroll
        for (int i = 0; i < FR_NF; ++i) {
            const int f = A.p4f[warp * FR_NF + i];
            if (f < d) {
#pragma unroll
                for (int n = 0; n < 2; ++n) {
                    float* p0 = wp + (size_t)(f * K + g) * H1 + n * 8 + 2 * t;
                    *reinterpret_cast<float2*>(p0) = make_float2(wacc[i][n][0], wacc[i][n][1]);
                    *reinterpret_cast<float2*>(p0 + 8 * H1) = make_float2(wacc[i][n][2], wacc[i][n][3]);
                }
            }
        }
        if (tid == acc_tid) { a.head_part[blockIdx.x * 2] = loss_acc; a.head_part[blockIdx.x * 2 + 1] = dz_acc; }
    }
}

// ---- compaction of the pairs that need the sort (3 small launches; order preserving, so the stable sort keeps the
//      lookups of a row in batch order and the ordered reduction stays deterministic)
constexpr int CP_ITEMS = 8, CP_TILE = 256 * CP_ITEMS;
__device__ __forceinline__ int cp_state(const uint32_t* __restrict__ keys, int64_t i, int64_t n, uint32_t R, const uint32_t* __restrict__ claim,
                                        uint32_t mask, uint32_t& key) {        // 0: no row, 1: once only, 2: goes through the sort
    if (i >= n) return 0;
    key = __ldg(keys + i);
    if (key >= R) return 0;
    return claim_once(claim, mask, key) ? 1 : 2;
}
__global__ void __launch_bounds__(256) cp_count_kernel(const uint32_t* __restrict__ keys, int64_t n, uint32_t R, const uint32_t* __restrict__ claim,
                                                       uint32_t mask, uint32_t* __restrict__ blk_cnt /*[2][blocks]*/) {
    int keep = 0, once = 0;
#pragma unroll
    for (int j = 0; j < CP_ITEMS; ++j) {
        uint32_t key;
        const int st = cp_state(keys, (int64_t)blockIdx.x * CP_TILE + j * 256 + threadIdx.x, n, R, claim, mask, key);
        keep += st == 2; once += st == 1;
    }
    __shared__ int sk[8], so[8];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) { keep += __shfl_xor_sync(0xffffffffu, keep, o); once += __shfl_xor_sync(0xffffffffu, once, o); }
    if ((threadIdx.x & 31) == 0) { sk[threadIdx.x >> 5] = keep; so[threadIdx.x >> 5] = once; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int a = 0, b = 0;
        for (int w = 0; w < 8; ++w) { a += sk[w]; b += so[w]; }
        blk_cnt[blockIdx.x] = a; blk_cnt[gridDim.x + blockIdx.x] = b;
    }
}
__global__ void __launch_bounds__(1024) cp_scan_kernel(uint32_t* __restrict__ blk_cnt, int nblk, uint32_t* __restrict__ n_out) {
    __shared__ uint32_t ws[32];
    __shared__ uint32_t carry, once_total;
    if (threadIdx.x == 0) { carry = 0; once_total = 0; }
    __syncthreads();
    for (int base = 0; base < nblk; base += 1024) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < nblk ? blk_cnt[i] : 0u, oc = i < nblk ? blk_cnt[nblk + i] : 0u;
        uint32_t x = v, y = oc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, x, o); if ((threadIdx.x & 31) >= o) x += t; }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) y += __shfl_xor_sync(0xffffffffu, y, o);
        if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
        if ((threadIdx.x & 31) == 0 && y) atomicAdd(&once_total, y);
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t w = ws[threadIdx.x];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, w, o); if (threadIdx.x >= o) w += t; }
            ws[threadIdx.x] = w;
        }
        __syncthreads();
        const uint32_t before = carry + ((threadIdx.x >> 5) ? ws[(threadIdx.x >> 5) - 1] : 0u) + x - v;     // exclusive
        if (i < nblk) blk_cnt[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) { n_out[0] = carry; n_out[1] = once_total; }
}
__global__ void __launch_bounds__(256) cp_scatter_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t n, uint32_t R,
                                                         const uint32_t* __restrict__ claim, uint32_t mask, const uint32_t* __restrict__ blk_off,
                                                         uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
    __shared__ uint32_t wc[CP_ITEMS * 8 + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t key[CP_ITEMS], rank[CP_ITEMS];
    bool keep[CP_ITEMS];
#pragma unroll
    for (int j = 0; j < CP_ITEMS; ++j) {
        keep[j] = cp_state(keys, (int64_t)blockIdx.x * CP_TILE + j * 256 + threadIdx.x, n, R, claim, mask, key[j]) == 2;
        const unsigned b = __ballot_sync(0xffffffffu, keep[j]);
        rank[j] = __popc(b & ((1u << lane) - 1u));
        if (lane == 0) wc[j * 8 + warp] = __popc(b);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int q = 0; q < CP_ITEMS * 8; ++q) { const uint32_t c = wc[q]; wc[q] = run; run += c; }
    }
    __syncthreads();
    const uint32_t base = blk_off[blockIdx.x];
#pragma unroll
    for (int j = 0; j < CP_ITEMS; ++j)
        if (keep[j]) {
            const uint32_t at = base + wc[j * 8 + warp] + rank[j];
            keys_out[at] = key[j];
            vals_out[at] = __ldg(vals + (int64_t)blockIdx.x * CP_TILE + j * 256 + threadIdx.x);
        }
}
cudaError_t fused_rows_compact(const uint32_t* keys_in, const uint32_t* vals_in, int64_t n, uint32_t R, const uint32_t* claim, uint32_t claim_mask,
                               uint32_t* keys_out, uint32_t* vals_out, uint32_t* scratch, uint32_t* n_out, cudaStream_t st, int64_t* launches) {
    const int nblk = (int)std::max<int64_t>((n + CP_TILE - 1) / CP_TILE, 1);
    cp_count_kernel<<<nblk, 256, 0, st>>>(keys_in, n, R, claim, claim_mask, scratch);
    cp_scan_kernel<<<1, 1024, 0, st>>>(scratch, nblk, n_out);
    cp_scatter_kernel<<<nblk, 256, 0, st>>>(keys_in, vals_in, n, R, claim, claim_mask, scratch, keys_out, vals_out);
    if (launches) *launches += 3;
    return cudaGetLastError();
}

bool fused_rows_supported(int K, int H1, int dc, int dn) {
    return K == 16 && H1 == 16 && dc > 0 && FR_TS * dc <= 32 * FR_NR * FR_PW && dc + dn <= FR_CW * FR_NF;
}
// Deals the per-field tasks of P4 / P5 to the consumer warps: longest task first onto the least loaded warp that still has
// a free place (at most FR_NF dW0 fields - register accumulators - and FR_N5 dE tasks per warp).  Costs are warp
// instructions per tile and task, counted on the SASS (DFM_FR_COST="dE+update,dE numeric,dW0" overrides them).
void fr_balance(FusedRowsArgs& A, int dc, int dn, bool cat_tasks) {
    static int cost[3] = {0, 0, 0};
    if (!cost[0]) {
        cost[0] = 150; cost[1] = 100; cost[2] = 45;
        if (const char* e = getenv("DFM_FR_COST")) sscanf(e, "%d,%d,%d", &cost[0], &cost[1], &cost[2]);
    }
    A.ablate = getenv("DFM_FR_ABLATE") ? atoi(getenv("DFM_FR_ABLATE")) : 0;
    const int c_cat = A.rowbuf_mode ? (cost[0] * 2) / 3 : cost[0];
    int load[FR_CW] = {}, n4[FR_CW] = {}, n5[FR_CW] = {};
    memset(A.p4f, 0xff, sizeof(A.p4f));
    memset(A.p5f, 0xff, sizeof(A.p5f));
    auto place = [&](int f, int c, int* cnt, int cap, uint8_t* tab, int per) {
        int best = -1;
        for (int w = 0; w < FR_CW; ++w)
            if (cnt[w] < cap && (best < 0 || load[w] < load[best])) best = w;
        tab[best * per + cnt[best]++] = (uint8_t)f;
        load[best] += c;
    };
    if (cat_tasks)
        for (int f = 0; f < dc; ++f) place(f, c_cat, n5, FR_N5, A.p5f, FR_N5);
    for (int f = dc; f < dc + dn; ++f) place(f, cost[1], n5, FR_N5, A.p5f, FR_N5);
    for (int f = 0; f < dc + dn; ++f) place(f, cost[2], n4, FR_NF, A.p4f, FR_NF);
}
// offsets (in floats from the start of dynamic shared memory) of the kernel's arrays; fused_rows_smem_bytes bounds the total
void fr_layout(FusedRowsArgs& A, const SmallMlpDesc& m, int K, int dc, int dn) {
    FrLayout& L = A.lay;
    const int H1 = m.H[0], nrows = FR_TS * dc, n_gnum = dn * K + dn;
    int o = m.D * FR_W0S;
    L.ups = o; o += m.up_count;
    L.gup = o; o += m.up_count + ((4 - ((2 * m.up_count) & 3)) & 3);
    L.slots = o; o += FR_NSLOT * FR_TS * A.sst;
    L.rowix = o; o += FR_NSLOT * nrows;
    L.once = o; o += FR_NSLOT * nrows;
    L.xsb = o; o += FR_NSLOT * FR_TS * (dn > 0 ? dn : 1);
    L.ysb = o; o += FR_NSLOT * FR_TS;
    o += (4 - (o & 3)) & 3;
    L.part = o; o += FR_CW * FR_TS * H1;
    L.p1 = o; o += FR_CW * (2 * K + 4);
    L.dh1s = o; o += FR_TS * H1;
    L.acts = o; o += FR_TS * m.act_stride;
    L.dacts = o; o += FR_TS * m.act_stride;
    L.zs = o; o += FR_TS;
    L.dzs = o; o += FR_TS;
    L.red = o; o += FR_TS;
    o += (4 - (o & 3)) & 3;
    L.ss = o; o += FR_TS * K;
    L.gnum = o; o += n_gnum;
    o += o & 1;
    L.bars = o;
}
size_t fused_rows_smem_bytes(const SmallMlpDesc& m, int K, int dc, int dn, int rs) {
    size_t f = (size_t)m.D * FR_W0S + 2 * (size_t)m.up_count + 8;
    f += (size_t)FR_NSLOT * FR_TS * fr_sst(dc, dn, K, rs);
    f += (size_t)FR_NSLOT * (2 * FR_TS * dc + FR_TS * (dn > 0 ? dn : 1) + FR_TS + 8);
    f += (size_t)FR_CW * FR_TS * m.H[0] + (size_t)FR_CW * (2 * K + 4) + (size_t)FR_TS * m.H[0] + 2 * (size_t)FR_TS * m.act_stride + 3 * FR_TS +
         (size_t)FR_TS * K + (size_t)(dn * K + dn) + 16;
    return f * 4 + 2 * FR_NSLOT * 8 + 64;
}

int fused_rows_grid(int B, int sm_count, bool side_stream_busy) {
    // The kernel fills an SM (registers, 224 KB of shared memory), so nothing else runs beside it: with the compaction /
    // sort / segment kernels of the repeated lookups on the side stream, a few SMs are left to them (measured on the
    // Criteo-shaped step: none reserved 0.865 ms, 8 reserved 0.819, 16 reserved 0.859).  Every CTA walks ceil(tiles / grid)
    // tiles, so between 4 and 12 reserved SMs the count with the fewest tiles per CTA is taken, the larger reserve on a tie
    // (B = 65 536 on 148 SMs: 4 reserved = 57 tiles per CTA, 8 reserved = 59: step 0.839 -> 0.814 ms).  DFM_FR_RESERVE overrides.
    static const int reserve_env = getenv("DFM_FR_RESERVE") ? atoi(getenv("DFM_FR_RESERVE")) : -1;
    const int tiles = (B + FR_TS - 1) / FR_TS;
    int reserve = 0;
    if (side_stream_busy) {
        reserve = reserve_env;
        if (reserve < 0) {
            int best_per = 1 << 30;
            for (int r = 12; r >= 4; --r) {
                const int g = std::max(1, sm_count - r), per = (tiles + g - 1) / g;
                if (per < best_per) { best_per = per; reserve = r; }
            }
        }
    }
    return std::max(1, std::min(tiles, sm_count - reserve));
}

template <int ES, bool RB>
static cudaError_t fr_attr(int smem_bytes) {
    cudaError_t e = cudaFuncSetAttribute(fused_rows_kernel<16, 16, ES, RB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    return e ? e : cudaFuncSetAttribute(fused_rows_kernel<16, 16, ES, RB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
}
cudaError_t fused_rows_set_attr(int smem_bytes) {
    cudaError_t e = fr_attr<0, false>(smem_bytes);
    if (!e) e = fr_attr<1, false>(smem_bytes);
    if (!e) e = fr_attr<2, false>(smem_bytes);
    if (!e) e = fr_attr<0, true>(smem_bytes);
    return e;
}
template <int ES, bool RB>
static void fr_go(const FusedRowsArgs& A, int grid, size_t smem_bytes, cudaStream_t st) {
    // FAST: every optimizer step the kernel takes is Adam and every replay is the closed form (row-buffer mode does neither)
    const RowReplay& rr = A.f.rr;
    const bool replay_fast = rr.upto < 0 || (rr.emb_adam && rr.rd.closed && (rr.same || !rr.lin_adam));
    const bool apply_fast = RB || !A.f.train || A.claim == nullptr || (A.od_t.kind == DFM_OPT_ADAM && (!A.f.use_linear || A.ol_t.kind == DFM_OPT_ADAM));
    static const bool allow = getenv("DFM_FR_NO_FAST") == nullptr;
    if (allow && replay_fast && apply_fast) fused_rows_kernel<16, 16, ES, RB, true><<<grid, FR_THREADS, smem_bytes, st>>>(A);
    else fused_rows_kernel<16, 16, ES, RB, false><<<grid, FR_THREADS, smem_bytes, st>>>(A);
}
cudaError_t fused_rows_launch(const FusedRowsArgs& A, int grid, size_t smem_bytes, cudaStream_t st) {
    if (A.rowbuf_mode) {
        fr_go<0, true>(A, grid, smem_bytes, st);
        return cudaGetLastError();
    }
    switch (A.emb_slots) {
        case 0: fr_go<0, false>(A, grid, smem_bytes, st); break;
        case 1: fr_go<1, false>(A, grid, smem_bytes, st); break;
        default: fr_go<2, false>(A, grid, smem_bytes, st); break;
    }
    return cudaGetLastError();
}
