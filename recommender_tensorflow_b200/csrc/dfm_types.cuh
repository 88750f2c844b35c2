// Internal device/host shared types of libdeepfm_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/deepfm_b200.h"

struct ColDev {
    int32_t  kind, dtype;
    uint64_t nb;            // bucket count used for the modulo (hash) / range check (identity)
    uint64_t nb_rcp;        // floor(2^64 / nb) (nb >= 2; 0: use the plain modulo): fingerprint % nb without a 64-bit division
    int32_t  bnd_off, bnd_cnt;
    int32_t  voc_off, voc_cnt, num_oov, width;   // width: value slots per sample (multivalent column), >= 1
    // crossed column: constituents = cols[keys[0..n_keys)] (source columns, hashing order), chain seeded with hash_key
    uint64_t hash_key;
    int32_t  n_keys;
    uint8_t  keys[DFM_MAX_CROSS_KEYS];
    // vocabulary: id of an unknown key (-1 = dropped).  identity: id of a value outside [0, nb), -1 = error
    int32_t  dflt;
    // vocabulary looked up through its hash table (vtab != nullptr): capacity tab_mask + 1 slots, power of two >= 2 V
    uint32_t tab_mask;
    const longlong2* vtab;  // slot = {key (string: fingerprint & fp_mask, int: the int64 value), vocabulary index or -1 = empty}
    uint64_t fp_mask;       // ~0; fewer bits only to test the byte comparison (DFM_VOCAB_FP_BITS)
};

// probe start of a vocabulary hash-table key: fixed 64-bit mixer (splitmix64 finaliser), the same on host and device
__host__ __device__ __forceinline__ uint64_t vocab_mix(uint64_t k) {
    k ^= k >> 30; k *= 0xbf58476d1ce4e5b9ull;
    k ^= k >> 27; k *= 0x94d049bb133111ebull;
    return k ^ (k >> 31);
}

// raw batch as kernel parameter (pointer tables by value: no H2D copy of pointer arrays)
struct BatchPtrs {
    const void*    cat[DFM_MAX_CAT];
    const int32_t* off[DFM_MAX_CAT];
    const float*   num[DFM_MAX_NUM];
    const float*   labels;
};

// optimizer constants as seen by one step (SURVEY.md A.3)
struct OptDev {
    int32_t kind;
    float   lr, b1, b2, eps;
    float   omb1, omb2;     // (1 - beta) evaluated in float32 like TF
    float   alpha;          // Adam: lr * sqrt(1 - b2^t) / (1 - b1^t) for the current step
    int32_t safe_early;     // Adam replay may stop once the update no longer changes w
};

// segment bookkeeping produced by the sort stage
struct SegCounts {
    uint32_t n_rows;     // unique table rows touched by the batch
    uint32_t n_pieces;   // sorted array cut at row changes and multiples of PIECE_C
    uint32_t n_valid;    // lookups that are not empty bags
    uint32_t n_hot;      // pieces that belong to rows with > DIRECT_T lookups
};

constexpr int PIECE_C = 256;      // max entries per piece
constexpr int COOP_PIECES = 8;    // rows with more pieces than this are summed by a whole warp in the update kernel
constexpr int DIRECT_T = 32;      // rows with <= DIRECT_T lookups are summed directly in the update kernel

// piece -> slot in the piece-sum buffer (collision free for pieces of rows with > DIRECT_T lookups)
__host__ __device__ __forceinline__ uint32_t piece_slot(uint32_t head_pos) {
    return (head_pos >> 5) * 2u + ((head_pos % PIECE_C) == 0 ? 0u : 1u);
}

// One record per table row, 64-byte aligned:  [ w[K] | {lin_w, lin_s1, lin_s2, last_step} | s1[K] | s2[K] | pad ]
// (K = 16, Adam: 256 bytes).  The forward reads w and the linear weight from ONE 128-byte line; the catch-up and
// the optimizer touch two adjacent lines (ncu showed 8 sectors fetched per lookup when the embedding record and
// the linear record lived in separate arrays).  Without embeddings (linear-only model) the record is the float4.
struct Table {
    float* rec;
    int stride;             // floats per row
    int lin_off;            // float offset of the {w, s1, s2, last_step} float4
    int s1_off, s2_off;     // float offsets of the embedding optimizer slots
};
__device__ __forceinline__ float4* tab_lin(const Table& t, size_t row) {
    return reinterpret_cast<float4*>(t.rec + row * t.stride + t.lin_off);
}
__device__ __forceinline__ float4* tab_w(const Table& t, size_t row) { return reinterpret_cast<float4*>(t.rec + row * t.stride); }
__device__ __forceinline__ float4* tab_s1(const Table& t, size_t row) { return reinterpret_cast<float4*>(t.rec + row * t.stride + t.s1_off); }
__device__ __forceinline__ float4* tab_s2(const Table& t, size_t row) { return reinterpret_cast<float4*>(t.rec + row * t.stride + t.s2_off); }

// Row-sharded step with the exchanges fused into the kernels over NVLink peer memory (CUDA IPC mappings of
// every rank's receive buffers): routing table of one step, computed on the host from the W x W matrix of
// per-(source, owner) unique-row counts.
constexpr int MAX_PEERS = 16;
struct PeerRoute {
    int32_t  W, me;
    uint32_t send_off[MAX_PEERS + 1];   // my unique-row list is owner-major: rows for owner o = [send_off[o], send_off[o+1])
    uint32_t dst_off[MAX_PEERS];        // start of my segment inside owner o's receive buffers (recv_rows / grecv)
    uint32_t recv_off[MAX_PEERS + 1];   // as owner: entries received from source s = [recv_off[s], recv_off[s+1])
    uint32_t reply_off[MAX_PEERS];      // start, inside source s's row buffer, of the rows I serve for it (= s's send_off[me])
    float*    peer_rowbuf[MAX_PEERS];   // mapped pointers, own buffers at index `me`
    float*    peer_grecv[MAX_PEERS];
    uint32_t* peer_recv_rows[MAX_PEERS];
};
__device__ __forceinline__ int route_find(const uint32_t* off, int W, uint32_t i) {
    int o = 0;
    while (o + 1 < W && i >= off[o + 1]) ++o;
    return o;
}
