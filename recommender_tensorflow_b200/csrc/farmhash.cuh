// Device-side FarmHash Fingerprint64 (farmhashna::Hash64) — the function behind TF-1.12's
// string_to_hash_bucket_fast, reached by the reference through
// tf.feature_column.categorical_column_with_hash_bucket (trainers/ml_100k.py:19-20,29-30).
// Keys of <= 16 bytes (every key of the BASELINE configs) are hashed entirely from two 64-bit
// registers; longer keys read the byte string from global memory.
#pragma once
#include <stdint.h>

namespace fh {

static constexpr uint64_t k0 = 0xc3a5c85c97cb3127ULL;
static constexpr uint64_t k1 = 0xb492b66fbe98f273ULL;
static constexpr uint64_t k2 = 0x9ae16a3b2f90404fULL;

__device__ __forceinline__ uint64_t rot(uint64_t v, int s) { return (v >> s) | (v << (64 - s)); }  // 0 < s < 64
__device__ __forceinline__ uint64_t smix(uint64_t v) { return v ^ (v >> 47); }

__device__ __forceinline__ uint64_t h16(uint64_t u, uint64_t v, uint64_t mul) {
    uint64_t a = (u ^ v) * mul;
    a ^= (a >> 47);
    uint64_t b = (v ^ a) * mul;
    b ^= (b >> 47);
    return b * mul;
}

// little-endian 64-bit window at byte offset o (0..8) of the 16-byte register pair (lo, hi)
__device__ __forceinline__ uint64_t win64(uint64_t lo, uint64_t hi, int o) {
    if (o == 0) return lo;
    if (o >= 8) return hi;  // o == 8
    return (lo >> (8 * o)) | (hi << (64 - 8 * o));
}
// 32-bit window at byte offset o (0..12)
__device__ __forceinline__ uint64_t win32(uint64_t lo, uint64_t hi, int o) {
    uint64_t v;
    if (o >= 8) v = hi >> (8 * (o - 8));
    else if (o == 0) v = lo;
    else v = (lo >> (8 * o)) | (hi << (64 - 8 * o));
    return v & 0xffffffffULL;
}

// Fingerprint64 of a key of len <= 16 bytes held in (lo = bytes 0..7, hi = bytes 8..15), unused bytes 0
__device__ __forceinline__ uint64_t fp64_short(uint64_t lo, uint64_t hi, int len) {
    if (len >= 8) {
        uint64_t mul = k2 + (uint64_t)len * 2;
        uint64_t a = lo + k2;
        uint64_t b = win64(lo, hi, len - 8);
        uint64_t c = rot(b, 37) * mul + a;
        uint64_t d = (rot(a, 25) + b) * mul;
        return h16(c, d, mul);
    }
    if (len >= 4) {
        uint64_t mul = k2 + (uint64_t)len * 2;
        uint64_t a = lo & 0xffffffffULL;
        return h16((uint64_t)len + (a << 3), win32(lo, hi, len - 4), mul);
    }
    if (len > 0) {
        uint32_t a = (uint32_t)(lo & 0xff);
        uint32_t b = (uint32_t)((lo >> (8 * (len >> 1))) & 0xff);
        uint32_t c = (uint32_t)((lo >> (8 * (len - 1))) & 0xff);
        uint32_t y = a + (b << 8);
        uint32_t z = (uint32_t)len + (c << 2);
        return smix((uint64_t)y * k2 ^ (uint64_t)z * k0) * k2;
    }
    return k2;
}

__device__ __forceinline__ uint64_t ld64(const uint8_t* p) {
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) v |= (uint64_t)p[i] << (8 * i);
    return v;
}

struct Pair { uint64_t first, second; };
__device__ __forceinline__ Pair weak32(const uint8_t* s, uint64_t a, uint64_t b) {
    uint64_t w = ld64(s), x = ld64(s + 8), y = ld64(s + 16), z = ld64(s + 24);
    a += w;
    b = rot(b + a + z, 21);
    uint64_t c = a;
    a += x;
    a += y;
    b += rot(a, 44);
    Pair r; r.first = a + z; r.second = b + c;
    return r;
}

// Fingerprint64 of an arbitrary byte string in global memory
__device__ inline uint64_t fp64_mem(const uint8_t* s, int len) {
    if (len <= 16) {
        uint64_t lo = 0, hi = 0;
        for (int i = 0; i < len; ++i) {
            uint64_t c = s[i];
            if (i < 8) lo |= c << (8 * i); else hi |= c << (8 * (i - 8));
        }
        return fp64_short(lo, hi, len);
    }
    if (len <= 32) {
        uint64_t mul = k2 + (uint64_t)len * 2;
        uint64_t a = ld64(s) * k1;
        uint64_t b = ld64(s + 8);
        uint64_t c = ld64(s + len - 8) * mul;
        uint64_t d = ld64(s + len - 16) * k2;
        return h16(rot(a + b, 43) + rot(c, 30) + d, a + rot(b + k2, 18) + c, mul);
    }
    if (len <= 64) {
        uint64_t mul = k2 + (uint64_t)len * 2;
        uint64_t a = ld64(s) * k2;
        uint64_t b = ld64(s + 8);
        uint64_t c = ld64(s + len - 8) * mul;
        uint64_t d = ld64(s + len - 16) * k2;
        uint64_t y = rot(a + b, 43) + rot(c, 30) + d;
        uint64_t z = h16(y, a + rot(b + k2, 18) + c, mul);
        uint64_t e = ld64(s + 16) * mul;
        uint64_t f = ld64(s + 24);
        uint64_t g = (y + ld64(s + len - 32)) * mul;
        uint64_t h = (z + ld64(s + len - 24)) * mul;
        return h16(rot(e + f, 43) + rot(g, 30) + h, e + rot(f + a, 18) + g, mul);
    }
    uint64_t x = 81;
    uint64_t y = 81 * k1 + 113;
    uint64_t z = smix(y * k2 + 113) * k2;
    Pair v = {0, 0}, w = {0, 0};
    x = x * k2 + ld64(s);
    const uint8_t* end = s + ((len - 1) / 64) * 64;
    const uint8_t* last64 = end + ((len - 1) & 63) - 63;
    do {
        x = rot(x + y + v.first + ld64(s + 8), 37) * k1;
        y = rot(y + v.second + ld64(s + 48), 42) * k1;
        x ^= w.second;
        y += v.first + ld64(s + 40);
        z = rot(z + w.first, 33) * k1;
        v = weak32(s, v.second * k1, x + w.first);
        w = weak32(s + 32, z + w.second, y + ld64(s + 16));
        uint64_t t = z; z = x; x = t;
        s += 64;
    } while (s != end);
    uint64_t mul = k1 + ((z & 0xff) << 1);
    s = last64;
    w.first += (uint64_t)((len - 1) & 63);
    v.first += w.first;
    w.first += v.first;
    x = rot(x + y + v.first + ld64(s + 8), 37) * mul;
    y = rot(y + v.second + ld64(s + 48), 42) * mul;
    x ^= w.second * 9;
    y += v.first * 9 + ld64(s + 40);
    z = rot(z + w.first, 33) * mul;
    v = weak32(s, v.second * mul, x + w.first);
    w = weak32(s + 32, z + w.second, y + ld64(s + 16));
    { uint64_t t = z; z = x; x = t; }
    return h16(h16(v.first, w.first, mul) + smix(y) * k0 + z, h16(v.second, w.second, mul) + x, mul);
}

// AsString(int32) -> decimal ASCII in (lo, hi); returns the length (TF `as_string`, no padding)
__device__ __forceinline__ int itoa16(int32_t v, uint64_t& lo, uint64_t& hi) {
    bool neg = v < 0;
    uint32_t mag = neg ? (0u - (uint32_t)v) : (uint32_t)v;
    uint64_t digits = 0;   // up to 10 digits, least-significant first, 4 bits each
    int nd = 0;
    do { digits |= (uint64_t)(mag % 10u) << (4 * nd); mag /= 10u; ++nd; } while (mag);
    int len = nd + (neg ? 1 : 0);
    lo = 0; hi = 0;
    if (neg) lo = (uint64_t)'-';
    for (int j = 0; j < nd; ++j) {
        uint64_t c = (uint64_t)('0' + ((digits >> (4 * (nd - 1 - j))) & 0xf));
        int pos = j + (neg ? 1 : 0);
        if (pos < 8) lo |= c << (8 * pos); else hi |= c << (8 * (pos - 8));
    }
    return len;
}

// FingerprintCat64 (TF-1.12 core/lib/hash/hash.h): the combiner sparse_cross_hashed chains over the constituents of a
// feature cross, h = FingerprintCat64(h, f(v)) starting from the hash key
__device__ __forceinline__ uint64_t fp_cat64(uint64_t fp1, uint64_t fp2) {
    constexpr uint64_t kMul = 0xc6a4a7935bd1e995ULL;
    uint64_t r = fp1 ^ kMul;
    r ^= smix(fp2 * kMul) * kMul;
    r *= kMul;
    r = smix(r) * kMul;
    return smix(r);
}

}  // namespace fh
