// Arguments / launch interface of the record-staged step kernel (fused_rows.cu; the kernel lives in its own translation unit).
#pragma once
#include "fused_small.cuh"

constexpr int FR_TS = 8;                       // samples per tile
#ifndef FR_CW_N
#define FR_CW_N 16
#endif
constexpr int FR_CW = FR_CW_N;                 // consumer warps: 16 (96 registers per thread); -DFR_CW_N=24 (72 registers, 540 bytes of
                                               // spill traffic per thread) measured SLOWER: kernel 0.65 -> 0.75 ms (gpurun_out/r02bb.txt)
constexpr int FR_WPS = FR_CW / 8;              // consumer warps per sample in P1 (FR_TS = 8)
constexpr int FR_PW = 4;                       // producer warps (bulk-copy issue is serial within a warp)
constexpr int FR_THREADS = (FR_CW + FR_PW) * 32;
constexpr int FR_NSLOT = 3;                    // tile slots: loading / computing / draining its stores
constexpr int FR_W0S = 20;                     // floats per W0 row in shared memory (H1 = 16 padded: conflict-free A fragments)
constexpr int FR_NR = 2;                       // rows per producer lane and tile (FR_TS * dc <= 32 * FR_NR * FR_PW)
constexpr int FR_NF = FR_CW == 16 ? 3 : 2;     // dW0 fields per consumer warp (d <= 48)
constexpr int FR_N5 = FR_CW == 16 ? 4 : 3;     // dE / update tasks per consumer warp

struct FrLayout { int ups, gup, slots, rowix, once, xsb, ysb, part, p1, dh1s, acts, dacts, zs, dzs, red, ss, gnum, bars; };

struct FusedRowsArgs {
    FusedArgs f;
    FrLayout lay;            // shared-memory offsets in floats (fr_layout)
    const uint32_t* claim; uint32_t claim_mask;    // 2 bits per slot; nullptr: no in-kernel optimizer (every row goes the sorted way)
    int rs;                  // floats per staged record: K + 4 + emb_slots * K
    int sst;                 // floats per sample in a tile slot (dc records + dn numeric embeddings, = 4 mod 32)
    int emb_slots;
    int step;                // the step being applied
    OptDev od_t, ol_t;       // this step's optimizer constants (alpha_t)
    float* numg_partial;     // [grid][dn * K + dn] gradients of numeric_embeddings / numeric linear weights
    // row-buffer mode (row-sharded requester): records come from f.rowbuf[f.uidx[lookup]], gradient rows of the rows
    // looked up once go to route (peer memory) or, route == nullptr, to gsum[unique row]
    int rowbuf_mode; const uint8_t* once_lk; const PeerRoute* route; float* gsum;
    int ablate;              // DFM_FR_ABLATE (timing experiments only, results are wrong): 1 no replay, 2 no P2, 4 no P3, 8 no P4, 16 no dE product, 32 no update / stores, 64 no P1
    uint8_t p4f[FR_CW * FR_NF], p5f[FR_CW * FR_N5];    // fields of each consumer warp's P4 / P5 tasks (0xff: none), fr_balance
};

__host__ __device__ inline int fr_sst(int dc, int dn, int K, int rs) {
    const int base = dc * rs + dn * K;
    return base + ((4 - base % 32) + 32) % 32;
}
// host interface (fused_rows.cu)
bool fused_rows_supported(int K, int H1, int dc, int dn);                     // shape limits of the instantiated kernel
size_t fused_rows_smem_bytes(const SmallMlpDesc& m, int K, int dc, int dn, int rs, bool weighted);   // weighted: room for staged weights
int fused_rows_grid(int B, int sm_count, bool side_stream_busy);                                     // CTAs (= per-CTA partial sets) of a launch
// Deterministic stream compaction of the step's (row, lookup) pairs: only the lookups whose claim state is "more than
// once" go through the sort / ordered reduction.  n_out[0] = pairs kept, n_out[1] = once-only lookups.  scratch: n / 2048 + 2 words.
cudaError_t fused_rows_compact(const uint32_t* keys_in, const uint32_t* vals_in, int64_t n, uint32_t R, const uint32_t* claim, uint32_t claim_mask,
                               uint32_t* keys_out, uint32_t* vals_out, uint32_t* scratch, uint32_t* n_out, cudaStream_t st, int64_t* launches);
void fr_layout(FusedRowsArgs& A, const SmallMlpDesc& m, int K, int dc, int dn);      // needs A.sst
void fr_balance(FusedRowsArgs& A, int dc, int dn, bool cat_tasks);   // cat_tasks: the kernel applies / forwards the once-only rows' gradients
cudaError_t fused_rows_set_attr(int smem_bytes, bool weighted, bool squared);   // also the WGT / SQ instantiations
cudaError_t fused_rows_launch(const FusedRowsArgs& A, int grid, size_t smem_bytes, cudaStream_t st, bool squared);   // squared: SQ for a train step
