// Device-side MurmurHash3_x64_128 (first 64-bit half, seed 0) over the ASCII bytes of one k-mer
// window: the function the reference calls for every window through
// `mur3::murmurhash3_x64_128(kmer.as_bytes(), 0).0` (core/src/domain/dtos/kmers_map.rs:157-159,
// :414-421).  The hash is NOT a rolling hash: every window is hashed independently.
// Integer-only; no tensor cores apply.  64-bit values live in register pairs; multiplies by the
// murmur constants are spelled out as one IMAD.WIDE + two IMAD, rotates as two funnel shifts.
#pragma once
#include <cstdint>

namespace cls {

constexpr uint64_t kC1 = 0x87c37b91114253d5ULL;
constexpr uint64_t kC2 = 0x4cf5ad432745937fULL;

__device__ __forceinline__ uint64_t pack64(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// x * C (mod 2^64) for a compile-time constant C: IMAD.WIDE for lo * C.lo, then the two cross terms are
// accumulated into the high word by two chained IMADs - three instructions (spelled in PTX: left to itself the
// compiler emits two independent IMADs plus an add, four instructions for the same latency).
template <uint64_t C>
__device__ __forceinline__ uint64_t mulc(uint64_t x) {
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    uint32_t rl, rh;
    asm("{\n\t"
        ".reg .u64 t;\n\t"
        ".reg .u32 th;\n\t"
        "mul.wide.u32 t, %2, %4;\n\t"
        "mov.b64 {%0, th}, t;\n\t"
        "mad.lo.u32 th, %2, %5, th;\n\t"
        "mad.lo.u32 %1, %3, %4, th;\n\t"
        "}"
        : "=r"(rl), "=r"(rh)
        : "r"(lo), "r"(hi), "n"((uint32_t)C), "n"((uint32_t)(C >> 32)));
    return pack64(rl, rh);
}

// rotate left by a compile-time amount
template <int R>
__device__ __forceinline__ uint64_t rotlc(uint64_t x) {
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    if constexpr (R >= 32) { const uint32_t t = lo; lo = hi; hi = t; }
    constexpr int S = R & 31;
    if constexpr (S == 0) return pack64(lo, hi);
    return pack64(__funnelshift_l(hi, lo, S), __funnelshift_l(lo, hi, S));
}

// x * 5 + c
__device__ __forceinline__ uint64_t mul5add(uint64_t x, uint32_t c) {
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    const uint64_t r = (uint64_t)lo * 5u + c;
    return pack64((uint32_t)r, (uint32_t)(r >> 32) + hi * 5u);
}

// k ^ (k >> 33)
__device__ __forceinline__ uint64_t xorshift33(uint64_t k) {
    const uint32_t hi = (uint32_t)(k >> 32);
    return pack64((uint32_t)k ^ (hi >> 1), hi);
}

__device__ __forceinline__ uint64_t fmix64_d(uint64_t k) {
    k = xorshift33(k);
    k = mulc<0xff51afd7ed558ccdULL>(k);
    k = xorshift33(k);
    k = mulc<0xc4ceb9fe1a85ec53ULL>(k);
    return xorshift33(k);
}

// pre-mix of one 8-byte word in the k1 / k2 lane of a block
__device__ __forceinline__ uint64_t premix_k1(uint64_t w) { return mulc<kC2>(rotlc<31>(mulc<kC1>(w))); }
__device__ __forceinline__ uint64_t premix_k2(uint64_t w) { return mulc<kC1>(rotlc<33>(mulc<kC2>(w))); }

__device__ __forceinline__ void mm_block(uint64_t &h1, uint64_t &h2, uint64_t k1, uint64_t k2) {
    h1 ^= premix_k1(k1);
    h1 = mul5add(rotlc<27>(h1) + h2, 0x52dce729u);
    h2 ^= premix_k2(k2);
    h2 = mul5add(rotlc<31>(h2) + h1, 0x38495ab5u);
}

__device__ __forceinline__ uint64_t mm_finish(uint64_t h1, uint64_t h2, uint64_t len) {
    h1 ^= len; h2 ^= len;
    h1 += h2; h2 += h1;
    h1 = fmix64_d(h1); h2 = fmix64_d(h2);
    return h1 + h2;
}

// Runtime-k variant (any k >= 1): byte-wise reads from a shared-memory ASCII string; used for k != 35.
__device__ __forceinline__ uint64_t load_le_smem(const uint8_t *p, int n) {
    uint64_t v = 0;
    for (int i = 0; i < n; ++i) v |= (uint64_t)p[i] << (8 * i);
    return v;
}

__device__ inline uint64_t murmur_window_generic(const uint8_t *s, uint32_t pos, uint32_t k) {
    const uint8_t *d = s + pos;
    uint64_t h1 = 0, h2 = 0;
    const uint32_t nblocks = k / 16;
    for (uint32_t b = 0; b < nblocks; ++b)
        mm_block(h1, h2, load_le_smem(d + 16 * b, 8), load_le_smem(d + 16 * b + 8, 8));
    const uint8_t *tail = d + 16 * nblocks;
    const int t = (int)(k & 15u);
    if (t > 8) h2 ^= premix_k2(load_le_smem(tail + 8, t - 8));
    if (t > 0) h1 ^= premix_k1(load_le_smem(tail, t > 8 ? 8 : t));
    return mm_finish(h1, h2, (uint64_t)k);
}

}  // namespace cls
