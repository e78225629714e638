// BLAKE3-256 for sm_100a (and the host side of the Fiat-Shamir channel): the hash behind
// winter-crypto `Blake3_256<Felt>`, which the reference fixes as Prover::HashFn
// (/root/reference src/training/prover.rs:225, src/aggregation/prover.rs:198).
//
// One thread owns one 16-word state and walks its message block by block; the seven rounds are fully
// unrolled with the message schedule resolved at compile time, so state and message stay in registers.
// Rotations by 16 and 8 are byte permutes (PRMT), by 12 and 7 funnel shifts (SHF).
#pragma once
#include <cstdint>
#include <cstring>
#include "f128.cuh"

namespace zkb {

#define B3_CHUNK_START 1u
#define B3_CHUNK_END 2u
#define B3_PARENT 4u
#define B3_ROOT 8u

#define B3_IV0 0x6A09E667u
#define B3_IV1 0xBB67AE85u
#define B3_IV2 0x3C6EF372u
#define B3_IV3 0xA54FF53Au
#define B3_IV4 0x510E527Fu
#define B3_IV5 0x9B05688Cu
#define B3_IV6 0x1F83D9ABu
#define B3_IV7 0x5BE0CD19u

__host__ __device__ __forceinline__ uint32_t b3_rotr16(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __byte_perm(x, 0, 0x1032);
#else
    return (x >> 16) | (x << 16);
#endif
}
__host__ __device__ __forceinline__ uint32_t b3_rotr8(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __byte_perm(x, 0, 0x0321);
#else
    return (x >> 8) | (x << 24);
#endif
}
__host__ __device__ __forceinline__ uint32_t b3_rotr(uint32_t x, int n) {
#ifdef __CUDA_ARCH__
    return __funnelshift_r(x, x, n);
#else
    return (x >> n) | (x << (32 - n));
#endif
}

// a + b + m.  The xors and rotations of G can only issue on the ALU pipe (8 of its 12 operations with a + b + m as one
// IADD3), which is what binds the leaf-hashing kernel (ALU pipe 94-96 % busy, FMA pipe 22 %).  On the device the three-input
// sums are therefore written as two multiply-adds by a constant-bank 1 that ptxas cannot fold: they issue on the FMA pipe
// (IMAD), leaving 8 ALU + 6 FMA-pipe operations per G instead of 10 + 2.
#ifdef __CUDACC__
__constant__ uint32_t b3_one = 1;
#endif
#if defined(__CUDA_ARCH__) && !defined(ZKB_B3_PLAIN_ADDS)
__device__ __forceinline__ uint32_t b3_add3(uint32_t a, uint32_t b, uint32_t m) {
    uint32_t t, r;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(t) : "r"(a), "r"(b3_one), "r"(b));
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(t), "r"(b3_one), "r"(m));
    return r;
}
#else
__host__ __device__ __forceinline__ uint32_t b3_add3(uint32_t a, uint32_t b, uint32_t m) { return a + b + m; }
#endif

#define B3_G(a, b, c, d, mx, my)      \
    a = b3_add3(a, b, (mx)); d = b3_rotr16(d ^ a); \
    c = c + d;        b = b3_rotr(b ^ c, 12); \
    a = b3_add3(a, b, (my)); d = b3_rotr8(d ^ a);  \
    c = c + d;        b = b3_rotr(b ^ c, 7);

#define B3_ROUND(m0, m1, m2, m3, m4, m5, m6, m7, m8, m9, m10, m11, m12, m13, m14, m15) \
    B3_G(s0, s4, s8, s12, m0, m1) B3_G(s1, s5, s9, s13, m2, m3)                         \
    B3_G(s2, s6, s10, s14, m4, m5) B3_G(s3, s7, s11, s15, m6, m7)                       \
    B3_G(s0, s5, s10, s15, m8, m9) B3_G(s1, s6, s11, s12, m10, m11)                     \
    B3_G(s2, s7, s8, s13, m12, m13) B3_G(s3, s4, s9, s14, m14, m15)

// cv <- first 8 words of compress(cv, m, counter, block_len, flags)
__host__ __device__ __forceinline__ void b3_compress(uint32_t cv[8], const uint32_t m[16], uint32_t counter_lo,
                                                     uint32_t block_len, uint32_t flags) {
    uint32_t s0 = cv[0], s1 = cv[1], s2 = cv[2], s3 = cv[3], s4 = cv[4], s5 = cv[5], s6 = cv[6], s7 = cv[7];
    uint32_t s8 = B3_IV0, s9 = B3_IV1, s10 = B3_IV2, s11 = B3_IV3;
    uint32_t s12 = counter_lo, s13 = 0, s14 = block_len, s15 = flags;
    B3_ROUND(m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], m[8], m[9], m[10], m[11], m[12], m[13], m[14], m[15])
    B3_ROUND(m[2], m[6], m[3], m[10], m[7], m[0], m[4], m[13], m[1], m[11], m[12], m[5], m[9], m[14], m[15], m[8])
    B3_ROUND(m[3], m[4], m[10], m[12], m[13], m[2], m[7], m[14], m[6], m[5], m[9], m[0], m[11], m[15], m[8], m[1])
    B3_ROUND(m[10], m[7], m[12], m[9], m[14], m[3], m[13], m[15], m[4], m[0], m[11], m[2], m[5], m[8], m[1], m[6])
    B3_ROUND(m[12], m[13], m[9], m[11], m[15], m[10], m[14], m[8], m[7], m[2], m[5], m[3], m[0], m[1], m[6], m[4])
    B3_ROUND(m[9], m[14], m[11], m[5], m[8], m[12], m[15], m[1], m[13], m[3], m[0], m[10], m[2], m[6], m[4], m[7])
    B3_ROUND(m[11], m[15], m[5], m[0], m[1], m[9], m[8], m[6], m[14], m[10], m[2], m[12], m[3], m[4], m[7], m[13])
    cv[0] = s0 ^ s8; cv[1] = s1 ^ s9; cv[2] = s2 ^ s10; cv[3] = s3 ^ s11;
    cv[4] = s4 ^ s12; cv[5] = s5 ^ s13; cv[6] = s6 ^ s14; cv[7] = s7 ^ s15;
}

__host__ __device__ __forceinline__ void b3_iv(uint32_t cv[8]) {
    cv[0] = B3_IV0; cv[1] = B3_IV1; cv[2] = B3_IV2; cv[3] = B3_IV3;
    cv[4] = B3_IV4; cv[5] = B3_IV5; cv[6] = B3_IV6; cv[7] = B3_IV7;
}

// parent node of the BLAKE3 tree: out = compress(IV, l || r, 0, 64, PARENT [| ROOT])
__host__ __device__ __forceinline__ void b3_parent(const uint32_t l[8], const uint32_t r[8], bool root, uint32_t out[8]) {
    uint32_t m[16];
#pragma unroll
    for (int i = 0; i < 8; i++) { m[i] = l[i]; m[8 + i] = r[i]; }
    b3_iv(out);
    b3_compress(out, m, 0, 64, B3_PARENT | (root ? B3_ROOT : 0u));
}
// hash(a || b) of two digests: 64 bytes = one ROOT chunk (Blake3_256::merge, the Merkle tree's inner nodes)
__host__ __device__ __forceinline__ void b3_merge(const uint32_t a[8], const uint32_t b[8], uint32_t out[8]) {
    uint32_t m[16];
#pragma unroll
    for (int i = 0; i < 8; i++) { m[i] = a[i]; m[8 + i] = b[i]; }
    b3_iv(out);
    b3_compress(out, m, 0, 64, B3_CHUNK_START | B3_CHUNK_END | B3_ROOT);
}
// hash(seed || v_le64): 40 bytes = one ROOT chunk (Blake3_256::merge_with_int)
__host__ __device__ __forceinline__ void b3_with_int(const uint32_t seed[8], uint64_t v, uint32_t out[8]) {
    uint32_t m[16];
#pragma unroll
    for (int i = 0; i < 8; i++) m[i] = seed[i];
    m[8] = (uint32_t)v; m[9] = (uint32_t)(v >> 32);
#pragma unroll
    for (int i = 10; i < 16; i++) m[i] = 0;
    b3_iv(out);
    b3_compress(out, m, 0, 40, B3_CHUNK_START | B3_CHUNK_END | B3_ROOT);
}

#ifdef __CUDACC__
// BLAKE3 of `count` field elements (16 B each) read from base[j * stride]; this is
// Blake3_256::hash_elements over a matrix row stored with an arbitrary element stride.
// count <= 255 (TraceInfo width limit) => at most 4 chunks, handled with a two-slot CV stack.
// Element e lives at base[(e / bw) * blk_stride + (e % bw) * stride]; bw_magic = ceil(2^16 / bw) makes the division a
// multiply-shift (exact for e, bw <= 256).  One block: bw = 256, bw_magic = 256.
__device__ __forceinline__ void b3_hash_elems(const fe* __restrict__ base, size_t stride, uint32_t count, uint32_t out[8],
                                              uint32_t bw, uint32_t bw_magic, size_t blk_stride) {
    const uint32_t nchunks = count <= 64 ? 1u : (count + 63u) / 64u;
    uint32_t st0[8], st1[8];
    for (uint32_t c = 0; c < nchunks; c++) {
        uint32_t cv[8];
        b3_iv(cv);
        const uint32_t e0 = c * 64u;
        const uint32_t ne = (count - e0) < 64u ? (count - e0) : 64u;  // elements in this chunk
        const uint32_t nblk = ne == 0 ? 1u : (ne + 3u) / 4u;
        for (uint32_t b = 0; b < nblk; b++) {
            uint32_t m[16];
            const uint32_t eb = e0 + 4u * b;
            const uint32_t nb = (e0 + ne - eb) < 4u ? (e0 + ne - eb) : 4u;
#pragma unroll
            for (uint32_t q = 0; q < 4; q++) {
                uint4 v = make_uint4(0, 0, 0, 0);
                if (q < nb) {
                    const uint32_t e = eb + q, blk = (e * bw_magic) >> 16;
                    v = *reinterpret_cast<const uint4*>(base + (size_t)blk * blk_stride + (size_t)(e - blk * bw) * stride);
                }
                m[4 * q] = v.x; m[4 * q + 1] = v.y; m[4 * q + 2] = v.z; m[4 * q + 3] = v.w;
            }
            uint32_t flags = (b == 0 ? B3_CHUNK_START : 0u);
            if (b + 1 == nblk) flags |= B3_CHUNK_END | (nchunks == 1 ? B3_ROOT : 0u);
            b3_compress(cv, m, c, nb * 16u, flags);
        }
        if (nchunks == 1) {
#pragma unroll
            for (int i = 0; i < 8; i++) out[i] = cv[i];
            return;
        }
        if (c == 0) {
#pragma unroll
            for (int i = 0; i < 8; i++) st0[i] = cv[i];
        } else if (c == 1) {
            uint32_t t[8];
            b3_parent(st0, cv, nchunks == 2, t);
#pragma unroll
            for (int i = 0; i < 8; i++) st0[i] = t[i];
        } else if (c == 2) {
            if (nchunks == 3) { b3_parent(st0, cv, true, out); return; }
#pragma unroll
            for (int i = 0; i < 8; i++) st1[i] = cv[i];
        } else {
            uint32_t t[8];
            b3_parent(st1, cv, false, t);
            b3_parent(st0, t, true, out);
            return;
        }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = st0[i];
}
// Chaining value of chunk c (64 elements, the last one shorter) of the same strided element sequence; count > 64, so no chunk
// is the root.  Used where a row's chunks are hashed by different threads (k_hash_lde_rows_split).
__device__ __forceinline__ void b3_chunk_cv_elems(const fe* __restrict__ base, size_t stride, uint32_t count, uint32_t c, uint32_t cv[8],
                                                  uint32_t bw, uint32_t bw_magic, size_t blk_stride) {
    b3_iv(cv);
    const uint32_t e0 = c * 64u;
    const uint32_t ne = (count - e0) < 64u ? (count - e0) : 64u;
    const uint32_t nblk = (ne + 3u) / 4u;
    for (uint32_t b = 0; b < nblk; b++) {
        uint32_t m[16];
        const uint32_t eb = e0 + 4u * b;
        const uint32_t nb = (e0 + ne - eb) < 4u ? (e0 + ne - eb) : 4u;
#pragma unroll
        for (uint32_t q = 0; q < 4; q++) {
            uint4 v = make_uint4(0, 0, 0, 0);
            if (q < nb) {
                const uint32_t e = eb + q, blk = (e * bw_magic) >> 16;
                v = *reinterpret_cast<const uint4*>(base + (size_t)blk * blk_stride + (size_t)(e - blk * bw) * stride);
            }
            m[4 * q] = v.x; m[4 * q + 1] = v.y; m[4 * q + 2] = v.z; m[4 * q + 3] = v.w;
        }
        const uint32_t flags = (b == 0 ? B3_CHUNK_START : 0u) | (b + 1 == nblk ? B3_CHUNK_END : 0u);
        b3_compress(cv, m, c, nb * 16u, flags);
    }
}
#endif

// ---- host-side BLAKE3 for the channel (inputs are tiny: seeds, digests, OOD frames) ----------------
static inline void b3_chunk_cv_host(const uint8_t* in, size_t len, uint64_t chunk, bool root, uint32_t out[8]) {
    uint32_t cv[8];
    b3_iv(cv);
    size_t nblk = len == 0 ? 1 : (len + 63) / 64;
    for (size_t b = 0; b < nblk; b++) {
        uint32_t m[16];
        memset(m, 0, 64);
        size_t bl = (b + 1 < nblk) ? 64 : len - 64 * b;
        memcpy(m, in + 64 * b, bl);
        uint32_t flags = (b == 0 ? B3_CHUNK_START : 0u);
        if (b + 1 == nblk) flags |= B3_CHUNK_END | (root ? B3_ROOT : 0u);
        b3_compress(cv, m, (uint32_t)chunk, (uint32_t)bl, flags);
    }
    memcpy(out, cv, 32);
}
static inline void b3_subtree_host(const uint8_t* in, size_t len, uint64_t c0, size_t nc, bool root, uint32_t out[8]) {
    if (nc == 1) { b3_chunk_cv_host(in, len, c0, false, out); return; }
    size_t left = 1;
    while (left * 2 <= nc - 1) left *= 2;
    uint32_t l[8], r[8];
    b3_subtree_host(in, left * 1024, c0, left, false, l);
    b3_subtree_host(in + left * 1024, len - left * 1024, c0 + left, nc - left, false, r);
    b3_parent(l, r, root, out);
}
static inline void b3_hash_host(const uint8_t* in, size_t len, uint8_t out[32]) {
    uint32_t cv[8];
    size_t nc = len <= 1024 ? 1 : (len + 1023) / 1024;
    if (nc == 1) b3_chunk_cv_host(in, len, 0, true, cv);
    else b3_subtree_host(in, len, 0, nc, true, cv);
    memcpy(out, cv, 32);
}

}  // namespace zkb
