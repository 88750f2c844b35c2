// GPU CSV record decoder (SURVEY.md §8f rank 2): replaces tf.data.TextLineDataset(csv) + tf.decode_csv(value, DEFAULTS)
// of the reference's input_fn (trainers/ml_100k.py:44-58) for the columns the model consumes.  The host only moves
// whole records (lines) around; field splitting, RFC-4180 unquoting, int32 parsing, default substitution and the
// label threshold run on the device and leave the batch in the layout dfm_raw_batch expects (int32 and float32 columns,
// Arrow-style string columns, float labels) — no per-field work on the CPU.
//
// Pipeline of one dfm_csv_decode call (byte / integer work, HBM-bound):
//   csv_count_nl      16 bytes per thread: newline count                      -> exclusive scan (prims)
//   csv_line_starts   same bytes: position after every newline                -> line_start[r]
//   csv_parse         thread per record: walk the fields; ints and floats parsed in place, strings measured (pos, length, flags)
//   exclusive scan    per string column: lengths -> Arrow offsets
//   csv_copy_strings  thread per (record, string column): unquote / default -> bytes
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/deepfm_b200.h"
#include "prims.cuh"

namespace {

constexpr int CSV_CHUNK = 16;      // bytes per thread in the newline kernels

struct CsvDev {
    int n_fields;
    const int32_t* kind;           // [n_fields] DFM_CSV_*
    const int32_t* slot;           // [n_fields] index among the int / string outputs
    const int32_t* int_default;    // [n_fields]
    const int32_t* def_off;        // [n_fields + 1] offsets into def_bytes (string defaults)
    const char* def_bytes;
    int label_field, label_min;
    int delim;                     // the field separator as a loaded `char` compares (sign-extended)
    const int32_t* fslot;          // [n_fields] index among the float outputs (float32 fields, int32 fields with as_float), -1
    const uint32_t* float_default; // [n_fields] bits of the value of an empty float32 field
};

__device__ __forceinline__ void csv_fail(unsigned long long* err, uint32_t rec, uint32_t code) {
    atomicMin(err, ((unsigned long long)rec << 8) | code);
}

// ---- float32 fields: strings::safe_strtof of TF 1.12 (the grammar is stated in oracle/strtof.py) -------------------
// Decimal -> float32, correctly rounded (half to even) for any number of digits:
//   1. the first 19 significant digits -> w (uint64), decimal exponent q, sticky = a nonzero digit was dropped;
//   2. Clinger: w <= 2^24, |q| <= 10 and nothing dropped -> one IEEE multiply / divide of two exact floats;
//   3. Eisel-Lemire: w * (64-bit truncated 5^q) in 128 bits; the bits below the rounding bit tell whether the
//      truncations (< 2^69 units of the product) can change the result;
//   4. otherwise csv_float_slow: the digits (120 significant + sticky) against the halfway points as big integers.
constexpr int POW5_MIN = -64, POW5_MAX = 38;   // every q that can reach the float32 range with 1..19 digits
struct Pow5 { unsigned long long m; int e; };   // 5^q = m * 2^e (m in [2^63, 2^64), rounded down)
// Global rather than __constant__: the lanes of a warp index it with their own exponents, and the constant cache
// serialises divergent addresses.
__device__ const Pow5 g_pow5[POW5_MAX - POW5_MIN + 1] = {
    {0xa87fea27a539e9a5ull, -212}, {0xd29fe4b18e88640eull, -210}, {0x83a3eeeef9153e89ull, -207},
    {0xa48ceaaab75a8e2bull, -205}, {0xcdb02555653131b6ull, -203}, {0x808e17555f3ebf11ull, -200},
    {0xa0b19d2ab70e6ed6ull, -198}, {0xc8de047564d20a8bull, -196}, {0xfb158592be068d2eull, -194},
    {0x9ced737bb6c4183dull, -191}, {0xc428d05aa4751e4cull, -189}, {0xf53304714d9265dfull, -187},
    {0x993fe2c6d07b7fabull, -184}, {0xbf8fdb78849a5f96ull, -182}, {0xef73d256a5c0f77cull, -180},
    {0x95a8637627989aadull, -177}, {0xbb127c53b17ec159ull, -175}, {0xe9d71b689dde71afull, -173},
    {0x9226712162ab070dull, -170}, {0xb6b00d69bb55c8d1ull, -168}, {0xe45c10c42a2b3b05ull, -166},
    {0x8eb98a7a9a5b04e3ull, -163}, {0xb267ed1940f1c61cull, -161}, {0xdf01e85f912e37a3ull, -159},
    {0x8b61313bbabce2c6ull, -156}, {0xae397d8aa96c1b77ull, -154}, {0xd9c7dced53c72255ull, -152},
    {0x881cea14545c7575ull, -149}, {0xaa242499697392d2ull, -147}, {0xd4ad2dbfc3d07787ull, -145},
    {0x84ec3c97da624ab4ull, -142}, {0xa6274bbdd0fadd61ull, -140}, {0xcfb11ead453994baull, -138},
    {0x81ceb32c4b43fcf4ull, -135}, {0xa2425ff75e14fc31ull, -133}, {0xcad2f7f5359a3b3eull, -131},
    {0xfd87b5f28300ca0dull, -129}, {0x9e74d1b791e07e48ull, -126}, {0xc612062576589ddaull, -124},
    {0xf79687aed3eec551ull, -122}, {0x9abe14cd44753b52ull, -119}, {0xc16d9a0095928a27ull, -117},
    {0xf1c90080baf72cb1ull, -115}, {0x971da05074da7beeull, -112}, {0xbce5086492111aeaull, -110},
    {0xec1e4a7db69561a5ull, -108}, {0x9392ee8e921d5d07ull, -105}, {0xb877aa3236a4b449ull, -103},
    {0xe69594bec44de15bull, -101}, {0x901d7cf73ab0acd9ull, -98}, {0xb424dc35095cd80full, -96},
    {0xe12e13424bb40e13ull, -94}, {0x8cbccc096f5088cbull, -91}, {0xafebff0bcb24aafeull, -89},
    {0xdbe6fecebdedd5beull, -87}, {0x89705f4136b4a597ull, -84}, {0xabcc77118461cefcull, -82},
    {0xd6bf94d5e57a42bcull, -80}, {0x8637bd05af6c69b5ull, -77}, {0xa7c5ac471b478423ull, -75},
    {0xd1b71758e219652bull, -73}, {0x83126e978d4fdf3bull, -70}, {0xa3d70a3d70a3d70aull, -68},
    {0xccccccccccccccccull, -66}, {0x8000000000000000ull, -63}, {0xa000000000000000ull, -61},
    {0xc800000000000000ull, -59}, {0xfa00000000000000ull, -57}, {0x9c40000000000000ull, -54},
    {0xc350000000000000ull, -52}, {0xf424000000000000ull, -50}, {0x9896800000000000ull, -47},
    {0xbebc200000000000ull, -45}, {0xee6b280000000000ull, -43}, {0x9502f90000000000ull, -40},
    {0xba43b74000000000ull, -38}, {0xe8d4a51000000000ull, -36}, {0x9184e72a00000000ull, -33},
    {0xb5e620f480000000ull, -31}, {0xe35fa931a0000000ull, -29}, {0x8e1bc9bf04000000ull, -26},
    {0xb1a2bc2ec5000000ull, -24}, {0xde0b6b3a76400000ull, -22}, {0x8ac7230489e80000ull, -19},
    {0xad78ebc5ac620000ull, -17}, {0xd8d726b7177a8000ull, -15}, {0x878678326eac9000ull, -12},
    {0xa968163f0a57b400ull, -10}, {0xd3c21bcecceda100ull, -8}, {0x84595161401484a0ull, -5}, {0xa56fa5b99019a5c8ull, -3},
    {0xcecb8f27f4200f3aull, -1}, {0x813f3978f8940984ull, 2}, {0xa18f07d736b90be5ull, 4}, {0xc9f2c9cd04674edeull, 6},
    {0xfc6f7c4045812296ull, 8}, {0x9dc5ada82b70b59dull, 11}, {0xc5371912364ce305ull, 13}, {0xf684df56c3e01bc6ull, 15},
    {0x9a130b963a6c115cull, 18}, {0xc097ce7bc90715b3ull, 20}, {0xf0bdc21abb48db20ull, 22}, {0x96769950b50d88f4ull, 25}
};

__device__ const float g_pow10f[11] = {1e0f, 1e1f, 1e2f, 1e3f, 1e4f, 1e5f, 1e6f, 1e7f, 1e8f, 1e9f, 1e10f};   // exact in float32

__device__ __forceinline__ bool csv_is_space(char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

// Little-endian 32-bit-limb natural number; 20 limbs bound every comparison csv_float_slow makes (< 430 bits).
struct CsvBig {
    static constexpr int L = 20;
    uint32_t d[L];
    int n;
    __device__ void set(uint32_t v) { d[0] = v; n = v ? 1 : 0; }
    __device__ void mul_add(uint32_t m, uint32_t a) {
        unsigned long long c = a;
        for (int i = 0; i < n; ++i) { c += (unsigned long long)d[i] * m; d[i] = (uint32_t)c; c >>= 32; }
        if (c && n < L) d[n++] = (uint32_t)c;
    }
    __device__ void mul_pow5(int e) {
        for (; e >= 13; e -= 13) mul_add(1220703125u, 0);     // 5^13
        uint32_t m = 1;
        for (; e > 0; --e) m *= 5;
        mul_add(m, 0);
    }
    __device__ void shl(int s) {
        if (!n) return;
        const int w = s >> 5, b = s & 31;
        int nn = min(n + w + 1, L);
        for (int i = nn - 1; i >= 0; --i) {
            const int j = i - w;
            const uint32_t hi = (j >= 0 && j < n) ? d[j] : 0, lo = (j - 1 >= 0 && j - 1 < n) ? d[j - 1] : 0;
            d[i] = b ? (hi << b) | (lo >> (32 - b)) : hi;
        }
        while (nn > 0 && !d[nn - 1]) --nn;
        n = nn;
    }
};

__device__ int csv_big_cmp(const CsvBig& a, const CsvBig& b) {
    if (a.n != b.n) return a.n < b.n ? -1 : 1;
    for (int i = a.n - 1; i >= 0; --i)
        if (a.d[i] != b.d[i]) return a.d[i] < b.d[i] ? -1 : 1;
    return 0;
}

// The exact decision.  The value (digits text[m0, m1) of a validated field, '.' included, times 10^ex) lies in
// [c0, c0 + 2 ulp): compare it with the halfway points above c0 (every halfway point has at most 113 significant
// digits, so 120 digits plus the sticky bit decide).
__device__ __noinline__ uint32_t csv_float_slow(const char* __restrict__ text, uint32_t m0, uint32_t m1, long long ex, uint32_t c0) {
    CsvBig D;
    D.set(0);
    int nsig = 0;
    long long k = ex;
    bool dot = false, sticky = false;
    for (uint32_t i = m0; i < m1; ++i) {
        const char c = text[i];
        if (c == '.') { dot = true; continue; }
        const uint32_t dg = (uint32_t)(c - '0');
        if (nsig < 120) {
            if (nsig || dg) { D.mul_add(10, dg); ++nsig; }
            if (dot) --k;
        } else {
            sticky |= dg != 0;
            if (!dot) ++k;
        }
    }
    uint32_t u = c0;
    for (int it = 0; it < 3 && u < 0x7f800000u; ++it) {
        const int ef = (int)(u >> 23), b = max(ef, 1) - 151;
        const uint32_t sig = (u & 0x7fffffu) | (ef ? 0x800000u : 0u);
        CsvBig X = D, Y;                   // X = D * 10^k, Y = (2 sig + 1) * 2^b, scaled to integers
        Y.set(2 * sig + 1);
        if (k >= 0) X.mul_pow5((int)k); else Y.mul_pow5((int)-k);
        if (k >= b) X.shl((int)(k - b)); else Y.shl((int)(b - k));
        int c = csv_big_cmp(X, Y);
        if (c == 0 && sticky) c = 1;
        if (c < 0) return u;
        if (c == 0) return u + (u & 1);
        ++u;
    }
    return u;
}

// w * 10^q (w != 0 the first 19 significant digits, sticky: more nonzero digits follow) -> float32 bits of |value|.
__device__ __forceinline__ uint32_t csv_decimal_to_float(unsigned long long w, int nsig, long long q, bool sticky, const char* __restrict__ text,
                                                        uint32_t m0, uint32_t m1, long long ex) {
    if (q + nsig - 1 > 38) return 0x7f800000u;            // >= 1e39
    if (q + nsig <= -46) return 0u;                       // < 1e-46, below half the smallest subnormal
    if (!sticky && w <= (1ull << 24) && q >= -10 && q <= 10) {
        const float f = (float)w;
        return __float_as_uint(q >= 0 ? __fmul_rn(f, g_pow10f[q]) : __fdiv_rn(f, g_pow10f[-q]));
    }
    const Pow5 p = g_pow5[q - POW5_MIN];
    const int lz = __clzll((long long)w);
    const unsigned __int128 N = (unsigned __int128)(w << lz) * p.m;    // value ~ N * 2^E, N in [2^126, 2^128)
    const int E = p.e + (int)q - lz;
    const int t = (int)(N >> 127) ? 127 : 126;
    const int sh = max(t - 23, -(E + 149));                // bits of N below the float's last place (>= 103)
    // N <= exact < N + 2^69: the 128-bit product drops < 2^64, the dropped digits < 2^68 (w >= 10^18 when sticky)
    const unsigned __int128 one = 1;
    uint32_t c0;
    if (sh >= 130) return 0u;                              // < 2^-150
    if (sh == 129) {
        if (N < ~(unsigned __int128)0 - (one << 70)) return 0u;
        c0 = 0;
    } else {
        const uint32_t keep = sh == 128 ? 0u : (uint32_t)(N >> sh);
        const uint32_t rbit = (uint32_t)(N >> (sh - 1)) & 1u;
        const unsigned __int128 below = (one << (sh - 1)) - 1, F = N & below;
        c0 = min(((uint32_t)(E + sh + 149) << 23) + keep, 0x7f800000u);
        // a carry from the truncations could reach the rounding bit, or the value may sit exactly halfway
        if ((F >> 70) != (below >> 70) && !(rbit && F == 0)) return min(c0 + rbit, 0x7f800000u);
    }
    return csv_float_slow(text, m0, m1, ex, c0);
}

__device__ __forceinline__ bool csv_special(const char* __restrict__ text, uint32_t i, uint32_t end, uint32_t& bits) {
    const uint32_t n = end - i;
    const char* name = (text[i] | 0x20) == 'n' ? "nan" : "infinity";
    if (n != 3 && !(n == 8 && name[0] == 'i')) return false;
    for (uint32_t j = 0; j < n; ++j)
        if ((text[i + j] | 0x20) != name[j]) return false;
    bits |= name[0] == 'n' ? 0x7fc00000u : 0x7f800000u;
    return true;
}

// text[i, end): an unquoted field, not empty -> float32 bits; false if it is not a valid float
__device__ __forceinline__ bool csv_parse_float(const char* __restrict__ text, uint32_t i, uint32_t end, uint32_t& bits) {
    while (i < end && csv_is_space(text[i])) ++i;
    while (end > i && csv_is_space(text[end - 1])) --end;
    if (i == end) return false;
    bits = 0;
    if (text[i] == '-' || text[i] == '+') { bits = text[i] == '-' ? 0x80000000u : 0u; ++i; }
    if (i < end && ((text[i] | 0x20) == 'i' || (text[i] | 0x20) == 'n')) return csv_special(text, i, end, bits);
    const uint32_t m0 = i;
    unsigned long long w = 0;
    int nsig = 0, nd = 0;
    long long q = 0;
    bool dot = false, sticky = false;
    for (; i < end; ++i) {
        const char c = text[i];
        if (c == '.' && !dot) { dot = true; continue; }
        const uint32_t dg = (uint32_t)(c - '0');
        if (dg > 9) break;
        ++nd;
        if (nsig < 19) {
            if (nsig || dg) { w = w * 10 + dg; ++nsig; }
            if (dot) --q;
        } else {
            sticky |= dg != 0;
            if (!dot) ++q;
        }
    }
    const uint32_t m1 = i;
    if (!nd) return false;
    long long ex = 0;
    if (i < end && (text[i] | 0x20) == 'e') {
        ++i;
        const bool eneg = i < end && text[i] == '-';
        if (i < end && (text[i] == '-' || text[i] == '+')) ++i;
        int ned = 0;
        for (; i < end && (uint32_t)(text[i] - '0') <= 9; ++i, ++ned)
            if (ex < 10000000000ll) ex = ex * 10 + (text[i] - '0');    // saturates beyond any field length (< 2^32)
        if (!ned) return false;
        if (eneg) ex = -ex;
    }
    if (i != end) return false;
    if (w) bits |= csv_decimal_to_float(w, nsig, q + ex, sticky, text, m0, m1, ex);
    return true;
}

__global__ void __launch_bounds__(256) csv_count_nl_kernel(const uint4* __restrict__ text16, int64_t n_bytes, uint32_t* __restrict__ counts) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t base = t * CSV_CHUNK;
    if (base >= n_bytes) return;
    uint4 v = text16[t];           // the buffer is padded to a multiple of 16 bytes
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i)
        if (base + i < n_bytes && ((w[i >> 2] >> ((i & 3) * 8)) & 0xffu) == '\n') ++c;
    counts[t] = c;
}

__global__ void __launch_bounds__(256) csv_line_starts_kernel(const uint4* __restrict__ text16, int64_t n_bytes, const uint32_t* __restrict__ offs,
                                                              uint32_t* __restrict__ line_start, uint32_t max_records) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t base = t * CSV_CHUNK;
    if (base >= n_bytes) return;
    if (t == 0) line_start[0] = 0;
    uint4 v = text16[t];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t k = offs[t];
#pragma unroll
    for (int i = 0; i < 16; ++i)
        if (base + i < n_bytes && ((w[i >> 2] >> ((i & 3) * 8)) & 0xffu) == '\n') {
            ++k;
            if (k <= max_records) line_start[k] = (uint32_t)(base + i + 1);
        }
}

// One thread per record.  Field grammar = tf.decode_csv (RFC 4180): a field is either unquoted (no '"' inside) or
// quoted with '""' as the escaped quote; an empty field takes the column default; the record must have exactly
// n_fields fields.  int32 fields: optional blanks, sign, digits, optional blanks.  FLOAT: the schema has float32
// fields or int32 fields that are also written as float32 (schemas without launch the int / string code alone).
template <bool FLOAT>
__global__ void __launch_bounds__(128) csv_parse_kernel(const char* __restrict__ text, const uint32_t* __restrict__ line_start,
                                                        const int32_t* __restrict__ line_idx /* null: record r is line r */, uint32_t n_rec,
                                                        CsvDev cfg, int32_t* const* __restrict__ int_out, uint32_t* const* __restrict__ str_pos,
                                                        uint32_t* const* __restrict__ str_len, uint8_t* const* __restrict__ str_flag,
                                                        float* const* __restrict__ float_out, float* __restrict__ labels,
                                                        unsigned long long* __restrict__ err) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const uint32_t li = line_idx ? (uint32_t)line_idx[r] : r;
    uint32_t p = line_start[li], e = line_start[li + 1];
    if (e > p && text[e - 1] == '\n') --e;
    if (e > p && text[e - 1] == '\r') --e;
    int field = 0;
    while (true) {
        uint32_t s, raw_len, nq = 0;
        if (p < e && text[p] == '"') {
            s = ++p;
            while (true) {
                if (p >= e) { csv_fail(err, r, DFM_CSV_ERR_QUOTE); return; }
                if (text[p] == '"') {
                    if (p + 1 < e && text[p + 1] == '"') { ++nq; p += 2; continue; }
                    break;
                }
                ++p;
            }
            raw_len = p - s;
            ++p;                                   // closing quote
            if (p < e && text[p] != cfg.delim) { csv_fail(err, r, DFM_CSV_ERR_QUOTE); return; }
        } else {
            s = p;
            while (p < e && text[p] != cfg.delim) {
                if (text[p] == '"') { csv_fail(err, r, DFM_CSV_ERR_QUOTE); return; }
                ++p;
            }
            raw_len = p - s;
        }
        if (field >= cfg.n_fields) { csv_fail(err, r, DFM_CSV_ERR_FIELDS); return; }
        const int kind = cfg.kind[field];
        if (kind == DFM_CSV_INT32) {
            int32_t v = cfg.int_default[field];
            if (raw_len) {
                uint32_t i = s, end = s + raw_len;
                while (i < end && text[i] == ' ') ++i;
                bool neg = false;
                if (i < end && (text[i] == '-' || text[i] == '+')) { neg = text[i] == '-'; ++i; }
                long long acc = 0;
                int nd = 0;
                while (i < end && text[i] >= '0' && text[i] <= '9') {
                    acc = acc * 10 + (text[i] - '0');
                    if (acc > 2147483648ll) acc = 2147483649ll;     // saturate: flagged below
                    ++i; ++nd;
                }
                while (i < end && text[i] == ' ') ++i;
                if (neg) acc = -acc;
                if (!nd || i != end || nq || acc > 2147483647ll || acc < -2147483648ll) { csv_fail(err, r, DFM_CSV_ERR_INT); return; }
                v = (int32_t)acc;
            }
            const int sl = cfg.slot[field];
            if (sl >= 0) int_out[sl][r] = v;
            if (field == cfg.label_field) labels[r] = v >= cfg.label_min ? 1.f : 0.f;
            if (FLOAT) {
                const int fs = cfg.fslot[field];
                if (fs >= 0) float_out[fs][r] = __int2float_rn(v);         // tf.to_float
            }
        } else if (FLOAT && kind == DFM_CSV_FLOAT32) {
            uint32_t bits = cfg.float_default[field];
            if (raw_len && (nq || !csv_parse_float(text, s, s + raw_len, bits))) { csv_fail(err, r, DFM_CSV_ERR_FLOAT); return; }
            float_out[cfg.fslot[field]][r] = __uint_as_float(bits);
        } else if (kind == DFM_CSV_STRING) {
            const int sl = cfg.slot[field];
            if (raw_len) {
                str_pos[sl][r] = s;
                str_len[sl][r] = raw_len - nq;
                str_flag[sl][r] = nq ? 1 : 0;
            } else {
                str_pos[sl][r] = 0;
                str_len[sl][r] = (uint32_t)(cfg.def_off[field + 1] - cfg.def_off[field]);
                str_flag[sl][r] = 2;
            }
        }
        ++field;
        if (p >= e) break;
        ++p;                                       // the delimiter; a trailing one leaves one more (empty) field
    }
    if (field != cfg.n_fields) csv_fail(err, r, DFM_CSV_ERR_FIELDS);
}

__global__ void __launch_bounds__(256) csv_copy_strings_kernel(const char* __restrict__ text, uint32_t n_rec, int n_str, CsvDev cfg,
                                                               const int32_t* __restrict__ str_field, const uint32_t* const* __restrict__ str_pos,
                                                               const uint32_t* const* __restrict__ offsets, const uint8_t* const* __restrict__ str_flag,
                                                               char* const* __restrict__ bytes_out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_rec * (uint32_t)n_str) return;
    const uint32_t sl = t / n_rec, r = t % n_rec;          // consecutive threads -> consecutive records of one column
    const uint32_t o0 = offsets[sl][r], len = offsets[sl][r + 1] - o0;
    char* dst = bytes_out[sl] + o0;
    const uint8_t fl = str_flag[sl][r];
    if (fl == 2) {
        const char* d = cfg.def_bytes + cfg.def_off[str_field[sl]];
        for (uint32_t i = 0; i < len; ++i) dst[i] = d[i];
    } else if (fl == 0) {
        const char* src = text + str_pos[sl][r];
        for (uint32_t i = 0; i < len; ++i) dst[i] = src[i];
    } else {
        const char* src = text + str_pos[sl][r];
        for (uint32_t i = 0; i < len; ++i) {
            const char c = *src++;
            if (c == '"') ++src;                               // '""' -> '"'
            dst[i] = c;
        }
    }
}

}  // namespace

struct dfm_csv_reader {
    int device = 0, n_fields = 0, n_int = 0, n_str = 0, n_float = 0, label_field = -1, label_min = 0;
    bool label_raw = false;      // dfm_csv_config.label_raw: labels are the label field's float32 column
    char delim = ',';
    int32_t max_records = 0;
    int64_t max_bytes = 0;
    std::vector<int32_t> kind, slot, fslot, str_field;
    cudaStream_t stream = nullptr;
    // device
    char* text = nullptr;                  // staging for dfm_csv_decode_host (max_bytes, 16-byte padded)
    int32_t *d_kind = nullptr, *d_slot = nullptr, *d_int_default = nullptr, *d_def_off = nullptr, *d_str_field = nullptr;
    char* d_def_bytes = nullptr;
    int32_t* d_fslot = nullptr; uint32_t* d_float_default = nullptr;
    std::vector<float*> float_out;
    float** d_float_out = nullptr;
    uint32_t *counts = nullptr, *line_start = nullptr;
    void* scan_temp = nullptr;
    uint32_t* d_total = nullptr;
    unsigned long long* d_err = nullptr;
    std::vector<int32_t*> int_out;
    std::vector<uint32_t*> str_pos, str_off;
    std::vector<uint8_t*> str_flag;
    std::vector<char*> str_bytes;
    int32_t** d_int_out = nullptr; uint32_t **d_str_pos = nullptr, **d_str_off = nullptr; uint8_t** d_str_flag = nullptr; char** d_str_bytes = nullptr;
    float* labels = nullptr;
    uint32_t* h_total = nullptr; unsigned long long* h_err = nullptr;      // pinned
    int32_t n_records = 0;
    // file-resident mode (dfm_csv_load): the whole text and its line starts stay in HBM, batches are lists of line numbers
    char* file_text = nullptr; uint32_t* file_line_start = nullptr; int64_t file_lines = 0, file_bytes = 0;
    int32_t* d_line_idx = nullptr; int32_t* h_line_idx = nullptr;     // [max_records], pinned staging
    std::string error;
};

static thread_local std::string g_csv_error;

#define CSV_FAIL(r, code, ...)                                   \
    do {                                                         \
        char buf_[256];                                          \
        snprintf(buf_, sizeof buf_, __VA_ARGS__);                \
        if (r) (r)->error = buf_; else g_csv_error = buf_;       \
        return code;                                             \
    } while (0)
#define CSV_CK(r, call)                                                                               \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess) CSV_FAIL(r, DFM_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));    \
    } while (0)

template <typename T>
static cudaError_t csv_alloc(T** p, size_t n) { return cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(n, 1) * sizeof(T)); }

extern "C" const char* dfm_csv_last_error(const dfm_csv_reader* r) { return r ? r->error.c_str() : g_csv_error.c_str(); }

extern "C" void dfm_csv_destroy(dfm_csv_reader* r) {
    if (!r) return;
    cudaSetDevice(r->device);
    if (r->stream) { cudaStreamSynchronize(r->stream); cudaStreamDestroy(r->stream); }
    void* ptrs[] = {r->text, r->d_kind, r->d_slot, r->d_int_default, r->d_def_off, r->d_str_field, r->d_def_bytes, r->counts, r->line_start,
                    r->scan_temp, r->d_total, r->d_err, r->d_int_out, r->d_str_pos, r->d_str_off, r->d_str_flag, r->d_str_bytes, r->labels,
                    r->d_fslot, r->d_float_default, r->d_float_out};
    for (void* p : ptrs) if (p) cudaFree(p);
    for (auto p : r->int_out) cudaFree(p);
    for (auto p : r->float_out) cudaFree(p);
    for (auto p : r->str_pos) cudaFree(p);
    for (auto p : r->str_off) cudaFree(p);
    for (auto p : r->str_flag) cudaFree(p);
    for (auto p : r->str_bytes) cudaFree(p);
    if (r->file_text) cudaFree(r->file_text);
    if (r->file_line_start) cudaFree(r->file_line_start);
    if (r->d_line_idx) cudaFree(r->d_line_idx);
    if (r->h_line_idx) cudaFreeHost(r->h_line_idx);
    if (r->h_total) cudaFreeHost(r->h_total);
    if (r->h_err) cudaFreeHost(r->h_err);
    delete r;
}

extern "C" int dfm_csv_create(const dfm_csv_config* cfg, dfm_csv_reader** out) {
    if (!cfg || !out || cfg->n_fields <= 0 || !cfg->kind || cfg->max_records <= 0 || cfg->max_bytes <= 0)
        CSV_FAIL((dfm_csv_reader*)nullptr, DFM_ERR_INVALID_ARG, "dfm_csv_create: bad configuration");
    if (cfg->max_bytes >= (int64_t)1 << 32) CSV_FAIL((dfm_csv_reader*)nullptr, DFM_ERR_UNSUPPORTED, "dfm_csv_create: max_bytes must be < 4 GiB");
    const int32_t delim = cfg->field_delim ? cfg->field_delim : ',';
    if (delim < 1 || delim > 255 || delim == '"' || delim == '\n' || delim == '\r')
        CSV_FAIL((dfm_csv_reader*)nullptr, DFM_ERR_INVALID_ARG, "dfm_csv_create: field_delim %d must be one byte other than '\"', '\\n' and '\\r'", cfg->field_delim);
    for (int f = 0; f < cfg->n_fields; ++f)
        if (cfg->as_float && cfg->as_float[f] && cfg->kind[f] != DFM_CSV_INT32)
            CSV_FAIL((dfm_csv_reader*)nullptr, DFM_ERR_INVALID_ARG, "dfm_csv_create: as_float is set on field %d, which is not an int32 field", f);
    dfm_csv_reader* r = new dfm_csv_reader();
    r->delim = (char)delim;
    r->device = cfg->device; r->n_fields = cfg->n_fields; r->max_records = cfg->max_records;
    r->max_bytes = (cfg->max_bytes + 15) / 16 * 16;
    r->label_field = cfg->label_field; r->label_min = cfg->label_min;
    r->label_raw = cfg->label_raw != 0 && cfg->label_field >= 0;
    std::vector<int32_t> int_default(cfg->n_fields, 0), def_off(cfg->n_fields + 1, 0);
    std::vector<uint32_t> float_default(cfg->n_fields, 0);
    std::string def_bytes;
    for (int f = 0; f < cfg->n_fields; ++f) {
        const int k = cfg->kind[f];
        r->kind.push_back(k);
        // a raw int32 label is written as float32 like an as_float field: that column is the labels
        const bool int_as_float = (cfg->as_float && cfg->as_float[f]) || (r->label_raw && f == r->label_field);
        r->fslot.push_back(k == DFM_CSV_FLOAT32 || (k == DFM_CSV_INT32 && int_as_float) ? r->n_float++ : -1);
        if (k == DFM_CSV_INT32) {
            r->slot.push_back(r->n_int++);
            if (cfg->int_default) int_default[f] = cfg->int_default[f];
        } else if (k == DFM_CSV_FLOAT32) {
            r->slot.push_back(-1);
            if (cfg->float_default) memcpy(&float_default[f], &cfg->float_default[f], 4);
        } else if (k == DFM_CSV_STRING) {
            r->slot.push_back(r->n_str++);
            r->str_field.push_back(f);
            if (cfg->str_default && cfg->str_default[f]) def_bytes += cfg->str_default[f];
        } else if (k == DFM_CSV_SKIP) {
            r->slot.push_back(-1);
        } else {
            delete r;
            CSV_FAIL((dfm_csv_reader*)nullptr, DFM_ERR_INVALID_ARG, "dfm_csv_create: field %d has unknown kind %d", f, k);
        }
        def_off[f + 1] = (int32_t)def_bytes.size();
    }
    if (r->label_field >= 0 && (r->label_field >= cfg->n_fields ||
                                (r->kind[r->label_field] != DFM_CSV_INT32 && !(r->label_raw && r->kind[r->label_field] == DFM_CSV_FLOAT32)))) {
        delete r;
        CSV_FAIL((dfm_csv_reader*)nullptr, DFM_ERR_INVALID_ARG,
                 "dfm_csv_create: label_field must be an int32 field (or a float32 field with label_raw)");
    }
    *out = r;     // from here on dfm_csv_destroy cleans up
#define CR(call)                                                                                                  \
    do {                                                                                                          \
        cudaError_t e_ = (call);                                                                                  \
        if (e_ != cudaSuccess) { g_csv_error = std::string(#call ": ") + cudaGetErrorString(e_); dfm_csv_destroy(r); *out = nullptr; return DFM_ERR_CUDA; } \
    } while (0)
    CR(cudaSetDevice(r->device));
    CR(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking));
    const size_t nf = cfg->n_fields, mr = (size_t)r->max_records, n_chunks = (size_t)r->max_bytes / CSV_CHUNK;
    CR(csv_alloc(&r->text, (size_t)r->max_bytes));
    CR(csv_alloc(&r->d_kind, nf)); CR(csv_alloc(&r->d_slot, nf)); CR(csv_alloc(&r->d_int_default, nf)); CR(csv_alloc(&r->d_def_off, nf + 1));
    CR(csv_alloc(&r->d_str_field, (size_t)r->n_str)); CR(csv_alloc(&r->d_def_bytes, def_bytes.size()));
    CR(cudaMemcpy(r->d_kind, r->kind.data(), nf * 4, cudaMemcpyHostToDevice));
    CR(cudaMemcpy(r->d_slot, r->slot.data(), nf * 4, cudaMemcpyHostToDevice));
    CR(cudaMemcpy(r->d_int_default, int_default.data(), nf * 4, cudaMemcpyHostToDevice));
    CR(cudaMemcpy(r->d_def_off, def_off.data(), (nf + 1) * 4, cudaMemcpyHostToDevice));
    if (r->n_str) CR(cudaMemcpy(r->d_str_field, r->str_field.data(), (size_t)r->n_str * 4, cudaMemcpyHostToDevice));
    if (!def_bytes.empty()) CR(cudaMemcpy(r->d_def_bytes, def_bytes.data(), def_bytes.size(), cudaMemcpyHostToDevice));
    CR(csv_alloc(&r->counts, n_chunks + 1)); CR(csv_alloc(&r->line_start, mr + 2));
    CR(cudaMalloc(&r->scan_temp, std::max(prims::scan_temp_bytes((int64_t)n_chunks, 4), prims::scan_temp_bytes((int64_t)mr + 1, 4)) + 256));
    CR(csv_alloc(&r->d_total, 1)); CR(csv_alloc(&r->d_err, 1)); CR(csv_alloc(&r->labels, mr));
    CR(cudaMallocHost(&r->h_total, 4)); CR(cudaMallocHost(&r->h_err, 8));
    for (int i = 0; i < r->n_int; ++i) { int32_t* p = nullptr; CR(csv_alloc(&p, mr)); r->int_out.push_back(p); }
    for (int i = 0; i < r->n_str; ++i) {
        uint32_t *a = nullptr, *b = nullptr; uint8_t* c = nullptr; char* d = nullptr;
        CR(csv_alloc(&a, mr)); r->str_pos.push_back(a);
        CR(csv_alloc(&b, mr + 1)); r->str_off.push_back(b);
        CR(csv_alloc(&c, mr)); r->str_flag.push_back(c);
        // unquoting only shrinks a field; a default can be longer than the (empty) field it replaces
        const size_t def_len = (size_t)(def_off[r->str_field[i] + 1] - def_off[r->str_field[i]]);
        CR(csv_alloc(&d, (size_t)r->max_bytes + def_len * mr)); r->str_bytes.push_back(d);
    }
    if (r->n_float) {
        CR(csv_alloc(&r->d_fslot, nf)); CR(csv_alloc(&r->d_float_default, nf)); CR(csv_alloc(&r->d_float_out, (size_t)r->n_float));
        CR(cudaMemcpy(r->d_fslot, r->fslot.data(), nf * 4, cudaMemcpyHostToDevice));
        CR(cudaMemcpy(r->d_float_default, float_default.data(), nf * 4, cudaMemcpyHostToDevice));
        for (int i = 0; i < r->n_float; ++i) { float* p = nullptr; CR(csv_alloc(&p, mr)); r->float_out.push_back(p); }
        CR(cudaMemcpy(r->d_float_out, r->float_out.data(), (size_t)r->n_float * 8, cudaMemcpyHostToDevice));
    }
    CR(csv_alloc(&r->d_int_out, (size_t)r->n_int)); CR(csv_alloc(&r->d_str_pos, (size_t)r->n_str)); CR(csv_alloc(&r->d_str_off, (size_t)r->n_str));
    CR(csv_alloc(&r->d_str_flag, (size_t)r->n_str)); CR(csv_alloc(&r->d_str_bytes, (size_t)r->n_str));
    if (r->n_int) CR(cudaMemcpy(r->d_int_out, r->int_out.data(), (size_t)r->n_int * 8, cudaMemcpyHostToDevice));
    if (r->n_str) {
        CR(cudaMemcpy(r->d_str_pos, r->str_pos.data(), (size_t)r->n_str * 8, cudaMemcpyHostToDevice));
        CR(cudaMemcpy(r->d_str_off, r->str_off.data(), (size_t)r->n_str * 8, cudaMemcpyHostToDevice));
        CR(cudaMemcpy(r->d_str_flag, r->str_flag.data(), (size_t)r->n_str * 8, cudaMemcpyHostToDevice));
        CR(cudaMemcpy(r->d_str_bytes, r->str_bytes.data(), (size_t)r->n_str * 8, cudaMemcpyHostToDevice));
    }
#undef CR
    return DFM_OK;
}

// newline scan of `text_dev` -> line_start[0..n_rec] (device), n_rec on the host (one stream sync)
static int csv_split_lines(dfm_csv_reader* r, const char* text_dev, int64_t n_bytes, uint32_t* counts, void* scan_temp, uint32_t* line_start,
                           int64_t max_lines, int64_t* n_rec_out, cudaStream_t st) {
    const int64_t n_chunks = (n_bytes + CSV_CHUNK - 1) / CSV_CHUNK;
    const uint4* t16 = reinterpret_cast<const uint4*>(text_dev);
    csv_count_nl_kernel<<<(unsigned)((n_chunks + 255) / 256), 256, 0, st>>>(t16, n_bytes, counts);
    prims::exclusive_scan_u32(counts, counts, n_chunks, scan_temp, r->d_total, st, nullptr);
    csv_line_starts_kernel<<<(unsigned)((n_chunks + 255) / 256), 256, 0, st>>>(t16, n_bytes, counts, line_start, (uint32_t)std::min<int64_t>(max_lines + 1, 0xffffffffll));
    CSV_CK(r, cudaMemcpyAsync(r->h_total, r->d_total, 4, cudaMemcpyDeviceToHost, st));
    char last = 0;
    CSV_CK(r, cudaMemcpyAsync(&last, text_dev + n_bytes - 1, 1, cudaMemcpyDeviceToHost, st));
    CSV_CK(r, cudaStreamSynchronize(st));
    int64_t n_rec = *r->h_total;
    if (last != '\n') {                    // final record without a newline
        ++n_rec;
        if (n_rec <= max_lines) {
            const uint32_t end = (uint32_t)n_bytes;
            CSV_CK(r, cudaMemcpyAsync(line_start + n_rec, &end, 4, cudaMemcpyHostToDevice, st));
        }
    }
    *n_rec_out = n_rec;
    return DFM_OK;
}

// fields of n_rec records (record i = line line_idx[i], or line i) -> the reader's output columns; one stream sync
static int csv_parse_records(dfm_csv_reader* r, const char* text_dev, const uint32_t* line_start, const int32_t* line_idx, int64_t n_rec,
                             int32_t* n_records_out, cudaStream_t st) {
    CSV_CK(r, cudaMemsetAsync(r->d_err, 0xff, 8, st));
    // label_raw: the labels are a float column the kernel writes anyway, so it forms no thresholded label
    CsvDev cfg{r->n_fields, r->d_kind, r->d_slot, r->d_int_default, r->d_def_off, r->d_def_bytes, r->label_raw ? -1 : r->label_field, r->label_min, (int)r->delim,
               r->d_fslot, r->d_float_default};
    auto parse = r->n_float ? csv_parse_kernel<true> : csv_parse_kernel<false>;
    parse<<<(unsigned)((n_rec + 127) / 128), 128, 0, st>>>(text_dev, line_start, line_idx, (uint32_t)n_rec, cfg, r->d_int_out, r->d_str_pos, r->d_str_off,
                                                           r->d_str_flag, r->d_float_out, r->labels, r->d_err);
    for (int i = 0; i < r->n_str; ++i)
        prims::exclusive_scan_u32(r->str_off[i], r->str_off[i], n_rec, r->scan_temp, r->str_off[i] + n_rec, st, nullptr);
    if (r->n_str) {
        const int64_t nt = n_rec * r->n_str;
        csv_copy_strings_kernel<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(text_dev, (uint32_t)n_rec, r->n_str, cfg, r->d_str_field, r->d_str_pos, r->d_str_off,
                                                                              r->d_str_flag, r->d_str_bytes);
    }
    CSV_CK(r, cudaMemcpyAsync(r->h_err, r->d_err, 8, cudaMemcpyDeviceToHost, st));
    CSV_CK(r, cudaStreamSynchronize(st));
    CSV_CK(r, cudaGetLastError());
    if (*r->h_err != ~0ull) {
        const unsigned code = (unsigned)(*r->h_err & 0xff);
        const unsigned long long rec = *r->h_err >> 8;
        const char* what = code == DFM_CSV_ERR_FIELDS ? "wrong number of fields" : code == DFM_CSV_ERR_INT ? "field is not a valid int32"
                         : code == DFM_CSV_ERR_FLOAT ? "field is not a valid float" : "quoting error";
        CSV_FAIL(r, DFM_ERR_PARSE, "record %llu: %s", rec, what);
    }
    r->n_records = (int32_t)n_rec;
    if (n_records_out) *n_records_out = (int32_t)n_rec;
    return DFM_OK;
}

static int csv_decode_impl(dfm_csv_reader* r, const char* text_dev, int64_t n_bytes, int32_t* n_records_out, cudaStream_t st) {
    if (n_bytes < 0 || n_bytes > r->max_bytes) CSV_FAIL(r, DFM_ERR_INVALID_ARG, "dfm_csv_decode: %lld bytes exceed max_bytes", (long long)n_bytes);
    if (reinterpret_cast<uintptr_t>(text_dev) & 15) CSV_FAIL(r, DFM_ERR_INVALID_ARG, "dfm_csv_decode: text must be 16-byte aligned (and readable up to the next multiple of 16)");
    r->n_records = 0;
    if (n_records_out) *n_records_out = 0;
    if (n_bytes == 0) return DFM_OK;
    int64_t n_rec = 0;
    int rc = csv_split_lines(r, text_dev, n_bytes, r->counts, r->scan_temp, r->line_start, r->max_records, &n_rec, st);
    if (rc) return rc;
    if (n_rec > r->max_records) CSV_FAIL(r, DFM_ERR_INVALID_ARG, "dfm_csv_decode: %lld records exceed max_records %d", (long long)n_rec, r->max_records);
    return csv_parse_records(r, text_dev, r->line_start, nullptr, n_rec, n_records_out, st);
}

// ---- file-resident mode ------------------------------------------------------------------------------------------
// A training CSV is small next to HBM (ML-100K train.csv: 13 MB), so the whole text is uploaded once and split into
// lines on the device; a batch is then just the list of line numbers the host's shuffle selected (256 KB for 65 536
// records instead of 10 MB of text), and no byte of the file is touched by the CPU again.
extern "C" int dfm_csv_load(dfm_csv_reader* r, const char* text_host, int64_t n_bytes, int64_t* n_lines_out) {
    if (!r || !text_host || n_bytes <= 0) return DFM_ERR_INVALID_ARG;
    if (n_bytes >= (int64_t)1 << 32) CSV_FAIL(r, DFM_ERR_UNSUPPORTED, "dfm_csv_load: files of 4 GiB and more are not supported");
    CSV_CK(r, cudaSetDevice(r->device));
    cudaStream_t st = r->stream;
    if (r->file_text) { cudaFree(r->file_text); r->file_text = nullptr; }
    if (r->file_line_start) { cudaFree(r->file_line_start); r->file_line_start = nullptr; }
    const int64_t padded = (n_bytes + 15) / 16 * 16, n_chunks = padded / CSV_CHUNK;
    CSV_CK(r, csv_alloc(&r->file_text, (size_t)padded));
    CSV_CK(r, cudaMemsetAsync(r->file_text + padded - 16, 0, 16, st));
    CSV_CK(r, cudaMemcpyAsync(r->file_text, text_host, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
    uint32_t* counts = nullptr; void* scan_temp = nullptr; uint32_t* starts = nullptr;
    CSV_CK(r, csv_alloc(&counts, (size_t)n_chunks + 1));
    CSV_CK(r, cudaMalloc(&scan_temp, prims::scan_temp_bytes(n_chunks, 4) + 256));
    // first pass only counts the lines, so that the line-start array has the right size
    const uint4* t16 = reinterpret_cast<const uint4*>(r->file_text);
    csv_count_nl_kernel<<<(unsigned)((n_chunks + 255) / 256), 256, 0, st>>>(t16, n_bytes, counts);
    prims::exclusive_scan_u32(counts, counts, n_chunks, scan_temp, r->d_total, st, nullptr);
    CSV_CK(r, cudaMemcpyAsync(r->h_total, r->d_total, 4, cudaMemcpyDeviceToHost, st));
    CSV_CK(r, cudaStreamSynchronize(st));
    const int64_t cap = (int64_t)*r->h_total + 1;
    CSV_CK(r, csv_alloc(&starts, (size_t)cap + 2));
    int64_t n_lines = 0;
    int rc = csv_split_lines(r, r->file_text, n_bytes, counts, scan_temp, starts, cap, &n_lines, st);
    CSV_CK(r, cudaStreamSynchronize(st));
    cudaFree(counts); cudaFree(scan_temp);
    if (rc) { cudaFree(starts); return rc; }
    r->file_line_start = starts; r->file_lines = n_lines; r->file_bytes = n_bytes;
    if (!r->d_line_idx) {
        CSV_CK(r, csv_alloc(&r->d_line_idx, (size_t)r->max_records));
        CSV_CK(r, cudaMallocHost(&r->h_line_idx, (size_t)r->max_records * 4));
    }
    if (n_lines_out) *n_lines_out = n_lines;
    return DFM_OK;
}

extern "C" int dfm_csv_decode_lines(dfm_csv_reader* r, const int32_t* line_idx_host, int32_t n, void* stream) {
    if (!r || (!line_idx_host && n)) return DFM_ERR_INVALID_ARG;
    if (!r->file_text) CSV_FAIL(r, DFM_ERR_INVALID_ARG, "dfm_csv_decode_lines: call dfm_csv_load first");
    if (n < 0 || n > r->max_records) CSV_FAIL(r, DFM_ERR_INVALID_ARG, "dfm_csv_decode_lines: %d records exceed max_records %d", n, r->max_records);
    CSV_CK(r, cudaSetDevice(r->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : r->stream;
    r->n_records = 0;
    if (n == 0) return DFM_OK;
    for (int32_t i = 0; i < n; ++i) {
        if (line_idx_host[i] < 0 || line_idx_host[i] >= r->file_lines) CSV_FAIL(r, DFM_ERR_INVALID_ARG, "dfm_csv_decode_lines: line %d out of range", line_idx_host[i]);
        r->h_line_idx[i] = line_idx_host[i];
    }
    CSV_CK(r, cudaMemcpyAsync(r->d_line_idx, r->h_line_idx, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    return csv_parse_records(r, r->file_text, r->file_line_start, r->d_line_idx, n, nullptr, st);
}

extern "C" int dfm_csv_decode(dfm_csv_reader* r, const char* text_dev, int64_t n_bytes, int32_t* n_records_out, void* stream) {
    if (!r || (!text_dev && n_bytes)) return DFM_ERR_INVALID_ARG;
    CSV_CK(r, cudaSetDevice(r->device));
    return csv_decode_impl(r, text_dev, n_bytes, n_records_out, stream ? (cudaStream_t)stream : r->stream);
}

extern "C" int dfm_csv_decode_host(dfm_csv_reader* r, const char* text_host, int64_t n_bytes, int32_t* n_records_out, void* stream) {
    if (!r || (!text_host && n_bytes)) return DFM_ERR_INVALID_ARG;
    if (n_bytes < 0 || n_bytes > r->max_bytes) CSV_FAIL(r, DFM_ERR_INVALID_ARG, "dfm_csv_decode_host: %lld bytes exceed max_bytes", (long long)n_bytes);
    CSV_CK(r, cudaSetDevice(r->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : r->stream;
    if (n_bytes) CSV_CK(r, cudaMemcpyAsync(r->text, text_host, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
    return csv_decode_impl(r, r->text, n_bytes, n_records_out, st);
}

extern "C" int32_t dfm_csv_num_records(const dfm_csv_reader* r) { return r ? r->n_records : -1; }
extern "C" const int32_t* dfm_csv_int_column(const dfm_csv_reader* r, int32_t field) {
    if (!r || field < 0 || field >= r->n_fields || r->kind[field] != DFM_CSV_INT32) return nullptr;
    return r->int_out[r->slot[field]];
}
extern "C" const char* dfm_csv_str_bytes(const dfm_csv_reader* r, int32_t field) {
    if (!r || field < 0 || field >= r->n_fields || r->kind[field] != DFM_CSV_STRING) return nullptr;
    return r->str_bytes[r->slot[field]];
}
extern "C" const int32_t* dfm_csv_str_offsets(const dfm_csv_reader* r, int32_t field) {
    if (!r || field < 0 || field >= r->n_fields || r->kind[field] != DFM_CSV_STRING) return nullptr;
    return reinterpret_cast<const int32_t*>(r->str_off[r->slot[field]]);
}
extern "C" const float* dfm_csv_float_column(const dfm_csv_reader* r, int32_t field) {
    if (!r || field < 0 || field >= r->n_fields || r->fslot[field] < 0) return nullptr;
    return r->float_out[r->fslot[field]];
}
extern "C" const float* dfm_csv_labels(const dfm_csv_reader* r) {
    if (!r) return nullptr;
    return r->label_raw ? r->float_out[r->fslot[r->label_field]] : r->labels;
}
