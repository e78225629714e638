// f128 device arithmetic for sm_100a: the STARK base field of the reference
// (winter-math f128::BaseElement, selected at /root/reference src/training/prover.rs:9,
// src/aggregation/prover.rs:12): p = 2^128 - 45*2^40 + 1, canonical little-endian u128.
//
// Elements are four 32-bit limbs in registers (one uint4 / 128-bit access in memory).  A product is
// 16 IMAD.WIDE (even/odd carry chains) folded twice with 2^128 = C (mod p), C = 45*2^40 - 1 = K*2^32 - 1,
// K = 0x2D00: the folds multiply by the 14-bit K only (fe_reduce256).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace zkb {

struct __align__(16) fe {
    uint32_t x[4];
};

#define ZKB_C0 0xFFFFFFFFu
#define ZKB_C1 0x00002CFFu
// p limbs: {0x00000001, 0xFFFFD300, 0xFFFFFFFF, 0xFFFFFFFF}

__device__ __forceinline__ fe fe_zero() { fe r; r.x[0] = r.x[1] = r.x[2] = r.x[3] = 0; return r; }
__device__ __forceinline__ fe fe_one() { fe r; r.x[0] = 1; r.x[1] = r.x[2] = r.x[3] = 0; return r; }
__device__ __forceinline__ fe fe_from_u64(uint64_t v) { fe r; r.x[0] = (uint32_t)v; r.x[1] = (uint32_t)(v >> 32); r.x[2] = r.x[3] = 0; return r; }
__device__ __forceinline__ bool fe_is_zero(const fe& a) { return (a.x[0] | a.x[1] | a.x[2] | a.x[3]) == 0; }
__device__ __forceinline__ bool fe_eq(const fe& a, const fe& b) {
    return ((a.x[0] ^ b.x[0]) | (a.x[1] ^ b.x[1]) | (a.x[2] ^ b.x[2]) | (a.x[3] ^ b.x[3])) == 0;
}

__device__ __forceinline__ fe fe_load(const fe* p) {
    uint4 v = *reinterpret_cast<const uint4*>(p);
    fe r; r.x[0] = v.x; r.x[1] = v.y; r.x[2] = v.z; r.x[3] = v.w; return r;
}
__device__ __forceinline__ fe fe_ldg(const fe* p) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    fe r; r.x[0] = v.x; r.x[1] = v.y; r.x[2] = v.z; r.x[3] = v.w; return r;
}
__device__ __forceinline__ void fe_store(fe* p, const fe& a) {
    *reinterpret_cast<uint4*>(p) = make_uint4(a.x[0], a.x[1], a.x[2], a.x[3]);
}

// r + C with carry-out  <=>  r >= p; select the wrapped value then (canonicalisation step)
__device__ __forceinline__ fe fe_canon(const fe& a, uint32_t carry_in) {
    uint32_t t0, t1, t2, t3, cy;
    asm("add.cc.u32 %0, %5, %9;\n\t"
        "addc.cc.u32 %1, %6, %10;\n\t"
        "addc.cc.u32 %2, %7, 0;\n\t"
        "addc.cc.u32 %3, %8, 0;\n\t"
        "addc.u32 %4, 0, 0;"
        : "=r"(t0), "=r"(t1), "=r"(t2), "=r"(t3), "=r"(cy)
        : "r"(a.x[0]), "r"(a.x[1]), "r"(a.x[2]), "r"(a.x[3]), "r"(ZKB_C0), "r"(ZKB_C1));
    bool sel = (cy | carry_in) != 0;
    fe r;
    r.x[0] = sel ? t0 : a.x[0]; r.x[1] = sel ? t1 : a.x[1]; r.x[2] = sel ? t2 : a.x[2]; r.x[3] = sel ? t3 : a.x[3];
    return r;
}

__device__ __forceinline__ fe fe_add(const fe& a, const fe& b) {
    fe s; uint32_t cy;
    asm("add.cc.u32 %0, %5, %9;\n\t"
        "addc.cc.u32 %1, %6, %10;\n\t"
        "addc.cc.u32 %2, %7, %11;\n\t"
        "addc.cc.u32 %3, %8, %12;\n\t"
        "addc.u32 %4, 0, 0;"
        : "=r"(s.x[0]), "=r"(s.x[1]), "=r"(s.x[2]), "=r"(s.x[3]), "=r"(cy)
        : "r"(a.x[0]), "r"(a.x[1]), "r"(a.x[2]), "r"(a.x[3]), "r"(b.x[0]), "r"(b.x[1]), "r"(b.x[2]), "r"(b.x[3]));
    return fe_canon(s, cy);
}

__device__ __forceinline__ fe fe_sub(const fe& a, const fe& b) {
    fe d; uint32_t bw;
    asm("sub.cc.u32 %0, %5, %9;\n\t"
        "subc.cc.u32 %1, %6, %10;\n\t"
        "subc.cc.u32 %2, %7, %11;\n\t"
        "subc.cc.u32 %3, %8, %12;\n\t"
        "subc.u32 %4, 0, 0;"  // 0 or 0xFFFFFFFF
        : "=r"(d.x[0]), "=r"(d.x[1]), "=r"(d.x[2]), "=r"(d.x[3]), "=r"(bw)
        : "r"(a.x[0]), "r"(a.x[1]), "r"(a.x[2]), "r"(a.x[3]), "r"(b.x[0]), "r"(b.x[1]), "r"(b.x[2]), "r"(b.x[3]));
    // on borrow add p, i.e. subtract C (mod 2^128)
    fe r;
    asm("sub.cc.u32 %0, %4, %8;\n\t"
        "subc.cc.u32 %1, %5, %9;\n\t"
        "subc.cc.u32 %2, %6, 0;\n\t"
        "subc.u32 %3, %7, 0;"
        : "=r"(r.x[0]), "=r"(r.x[1]), "=r"(r.x[2]), "=r"(r.x[3])
        : "r"(d.x[0]), "r"(d.x[1]), "r"(d.x[2]), "r"(d.x[3]), "r"(bw & ZKB_C0), "r"(bw & ZKB_C1));
    return r;
}
__device__ __forceinline__ fe fe_neg(const fe& a) { return fe_sub(fe_zero(), a); }

// 128x128 -> 256-bit product, even/odd accumulation so every mad.lo/mad.hi pair is one IMAD.WIDE
__device__ __forceinline__ void mul_wide(const fe& a, const fe& b, uint32_t r[8]) {
    uint32_t e0, e1, e2, e3, e4, e5, e6, e7, o0, o1, o2, o3, o4, o5, o6;
    const uint32_t a0 = a.x[0], a1 = a.x[1], a2 = a.x[2], a3 = a.x[3];
    const uint32_t b0 = b.x[0], b1 = b.x[1], b2 = b.x[2], b3 = b.x[3];
    asm("{\n\t"
        // row b0
        "mul.lo.u32 %0, %15, %19;\n\t mul.hi.u32 %1, %15, %19;\n\t"
        "mul.lo.u32 %2, %17, %19;\n\t mul.hi.u32 %3, %17, %19;\n\t"
        "mul.lo.u32 %8, %16, %19;\n\t mul.hi.u32 %9, %16, %19;\n\t"
        "mul.lo.u32 %10, %18, %19;\n\t mul.hi.u32 %11, %18, %19;\n\t"
        // row b1: a0,a2 -> odd ; a1,a3 -> even
        "mad.lo.cc.u32 %8, %15, %20, %8;\n\t madc.hi.cc.u32 %9, %15, %20, %9;\n\t"
        "madc.lo.cc.u32 %10, %17, %20, %10;\n\t madc.hi.cc.u32 %11, %17, %20, %11;\n\t"
        "addc.u32 %12, 0, 0;\n\t"
        "mad.lo.cc.u32 %2, %16, %20, %2;\n\t madc.hi.cc.u32 %3, %16, %20, %3;\n\t"
        "madc.lo.cc.u32 %4, %18, %20, 0;\n\t madc.hi.u32 %5, %18, %20, 0;\n\t"
        // row b2: a0,a2 -> even ; a1,a3 -> odd
        "mad.lo.cc.u32 %2, %15, %21, %2;\n\t madc.hi.cc.u32 %3, %15, %21, %3;\n\t"
        "madc.lo.cc.u32 %4, %17, %21, %4;\n\t madc.hi.cc.u32 %5, %17, %21, %5;\n\t"
        "addc.u32 %6, 0, 0;\n\t"
        "mad.lo.cc.u32 %10, %16, %21, %10;\n\t madc.hi.cc.u32 %11, %16, %21, %11;\n\t"
        "madc.lo.cc.u32 %12, %18, %21, %12;\n\t madc.hi.cc.u32 %13, %18, %21, 0;\n\t"
        "addc.u32 %14, 0, 0;\n\t"
        // row b3: a0,a2 -> odd ; a1,a3 -> even
        "mad.lo.cc.u32 %10, %15, %22, %10;\n\t madc.hi.cc.u32 %11, %15, %22, %11;\n\t"
        "madc.lo.cc.u32 %12, %17, %22, %12;\n\t madc.hi.cc.u32 %13, %17, %22, %13;\n\t"
        "addc.u32 %14, %14, 0;\n\t"
        "mad.lo.cc.u32 %4, %16, %22, %4;\n\t madc.hi.cc.u32 %5, %16, %22, %5;\n\t"
        "madc.lo.cc.u32 %6, %18, %22, %6;\n\t madc.hi.u32 %7, %18, %22, 0;\n\t"
        "}"
        : "=&r"(e0), "=&r"(e1), "=&r"(e2), "=&r"(e3), "=&r"(e4), "=&r"(e5), "=&r"(e6), "=&r"(e7),
          "=&r"(o0), "=&r"(o1), "=&r"(o2), "=&r"(o3), "=&r"(o4), "=&r"(o5), "=&r"(o6)
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(b2), "r"(b3));
    // r = even + (odd << 32)
    r[0] = e0;
    asm("add.cc.u32 %0, %7, %14;\n\t"
        "addc.cc.u32 %1, %8, %15;\n\t"
        "addc.cc.u32 %2, %9, %16;\n\t"
        "addc.cc.u32 %3, %10, %17;\n\t"
        "addc.cc.u32 %4, %11, %18;\n\t"
        "addc.cc.u32 %5, %12, %19;\n\t"
        "addc.u32 %6, %13, %20;"
        : "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(e1), "r"(e2), "r"(e3), "r"(e4), "r"(e5), "r"(e6), "r"(e7),
          "r"(o0), "r"(o1), "r"(o2), "r"(o3), "r"(o4), "r"(o5), "r"(o6));
}

// lo(128) + hi(128) * 2^128  ->  canonical element (any 256-bit input).
// 2^128 = K*2^32 - 1 (mod p) with K = 45*2^8 = 0x2D00, so hi*2^128 = ((hi*K) << 32) - hi: every product is an IMAD.WIDE by a
// 14-bit immediate and the 32-bit shift is a limb move.  (Folding with C = {0xFFFFFFFF, 0x2CFF} instead makes ptxas split the
// products by 0xFFFFFFFF into IMAD + quarter-rate IMAD.HI: 98.6 -> 87.3 SASS instructions per butterfly, 203.6 -> 237.2 G
// butterflies/s register-resident on B200, tools/mul_variants.cu variant E, profiles/r2_mul_variants.txt.)
//   U  = lo - hi + ((hi*K) << 32)                 six limbs, two's complement while negative, 0 <= U < 2^175
//   r  = U mod 2^128 + ((top*K) << 32) - top      top = U >> 128 < 2^47;  r < 2^128 + 2^93, so at most one wrap
__device__ __forceinline__ fe fe_reduce256(const uint32_t v[8]) {
    const uint32_t k = 0x2D00u;
    uint32_t d0, d1, d2, d3, d4, d5, o0, o1, o2, o3;
    asm("{\n\t"
        "sub.cc.u32 %0, %10, %14;\n\t subc.cc.u32 %1, %11, %15;\n\t subc.cc.u32 %2, %12, %16;\n\t subc.cc.u32 %3, %13, %17;\n\t"
        "subc.u32 %4, 0, 0;\n\t mov.u32 %5, %4;\n\t"                                   // sign extension of lo - hi
        "mad.lo.cc.u32 %1, %14, %18, %1;\n\t madc.hi.cc.u32 %2, %14, %18, %2;\n\t"     // (d1,d2) += h0 K
        "madc.lo.cc.u32 %3, %16, %18, %3;\n\t madc.hi.cc.u32 %4, %16, %18, %4;\n\t"    // (d3,d4) += h2 K
        "addc.u32 %5, %5, 0;\n\t"
        "mul.lo.u32 %6, %15, %18;\n\t mul.hi.u32 %7, %15, %18;\n\t"                    // (o0,o1) = h1 K
        "mul.lo.u32 %8, %17, %18;\n\t mul.hi.u32 %9, %17, %18;\n\t"                    // (o2,o3) = h3 K
        "add.cc.u32 %2, %2, %6;\n\t addc.cc.u32 %3, %3, %7;\n\t addc.cc.u32 %4, %4, %8;\n\t addc.u32 %5, %5, %9;\n\t"
        "}"
        : "=&r"(d0), "=&r"(d1), "=&r"(d2), "=&r"(d3), "=&r"(d4), "=&r"(d5), "=&r"(o0), "=&r"(o1), "=&r"(o2), "=&r"(o3)
        : "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(k));
    // second fold: W = ((top*K) << 32) - top, three limbs, >= 0
    uint32_t q0, q1, w0, w1, w2, cy;
    fe out;
    asm("{\n\t"
        "mul.lo.u32 %0, %10, %12;\n\t mul.hi.u32 %1, %10, %12;\n\t mad.lo.u32 %1, %11, %12, %1;\n\t"
        "sub.cc.u32 %2, 0, %10;\n\t subc.cc.u32 %3, %0, %11;\n\t subc.u32 %4, %1, 0;\n\t"
        "add.cc.u32 %5, %13, %2;\n\t addc.cc.u32 %6, %14, %3;\n\t addc.cc.u32 %7, %15, %4;\n\t addc.cc.u32 %8, %16, 0;\n\t addc.u32 %9, 0, 0;\n\t"
        "}"
        : "=&r"(q0), "=&r"(q1), "=&r"(w0), "=&r"(w1), "=&r"(w2), "=&r"(out.x[0]), "=&r"(out.x[1]), "=&r"(out.x[2]), "=&r"(out.x[3]), "=&r"(cy)
        : "r"(d4), "r"(d5), "r"(k), "r"(d0), "r"(d1), "r"(d2), "r"(d3));
    // a wrap (cy) and "value >= p" are both fixed by adding C modulo 2^128
    return fe_canon(out, cy);
}

__device__ __forceinline__ fe fe_mul(const fe& a, const fe& b) {
    uint32_t w[8];
    mul_wide(a, b, w);
    return fe_reduce256(w);
}
// ---- multiplication by a twiddle that is known in advance --------------------------------------------------------------------
// A twiddle w is used for many butterflies (every column of a tile, several butterflies of a unit), so it pays to hold it as four
// pre-shifted copies W_i = w * 2^(32 i) mod p: x * w = sum_i x_i * W_i is then four ALIGNED 32 x 128-bit rows (16 IMAD.WIDE) whose
// sum is < 2^162 — the 128-bit first fold of fe_reduce256 disappears and only a 34-bit top is folded.  69 instead of 87 SASS
// instructions per butterfly (tools/mul_variants.cu variant F, profiles/r2_mul_variants.txt).
struct __align__(16) fe4 { fe w[4]; };

// a * 2^32 mod p:  (a << 32) = [0, a0, a1, a2] + a3 * 2^128,  and  a3 * 2^128 = ((a3 * K) << 32) - a3  (K = 0x2D00)
__device__ __forceinline__ fe fe_shl32(const fe& a) {
    const uint32_t k = 0x2D00u;
    uint32_t q0, q1, s1, s2, s3, cy, bw;
    fe r;
    asm("{\n\t"
        "mul.lo.u32 %0, %14, %15;\n\t mul.hi.u32 %1, %14, %15;\n\t"
        "add.cc.u32 %2, %11, %0;\n\t addc.cc.u32 %3, %12, %1;\n\t addc.cc.u32 %4, %13, 0;\n\t addc.u32 %5, 0, 0;\n\t"
        "sub.cc.u32 %6, 0, %14;\n\t subc.cc.u32 %7, %2, 0;\n\t subc.cc.u32 %8, %3, 0;\n\t subc.cc.u32 %9, %4, 0;\n\t subc.u32 %10, 0, 0;\n\t"
        "}"
        : "=&r"(q0), "=&r"(q1), "=&r"(s1), "=&r"(s2), "=&r"(s3), "=&r"(cy), "=&r"(r.x[0]), "=&r"(r.x[1]), "=&r"(r.x[2]), "=&r"(r.x[3]), "=&r"(bw)
        : "r"(a.x[0]), "r"(a.x[1]), "r"(a.x[2]), "r"(a.x[3]), "r"(k));
    return fe_canon(r, cy + bw);   // bw is 0 or 0xFFFFFFFF; the true value is in [0, 2^128 + 2^78): net wrap 0 or 1
}
__device__ __forceinline__ fe4 fe4_from(const fe& w) {
    fe4 t;
    t.w[0] = w; t.w[1] = fe_shl32(w); t.w[2] = fe_shl32(t.w[1]); t.w[3] = fe_shl32(t.w[2]);
    return t;
}
// x * w for w given as its four pre-shifted copies; x may be any 128-bit value, the copies must be canonical
__device__ __forceinline__ fe fe_mul_pre4(const fe& x, const fe4& t) {
    const uint32_t k = 0x2D00u;
    uint32_t e0, e1, e2, e3, e4, o0, o1, o2, o3, o4;
    asm("{\n\t"
        "mul.lo.u32 %0, %10, %14;\n\t mul.hi.u32 %1, %10, %14;\n\t mul.lo.u32 %2, %10, %16;\n\t mul.hi.u32 %3, %10, %16;\n\t"
        "mul.lo.u32 %5, %10, %15;\n\t mul.hi.u32 %6, %10, %15;\n\t mul.lo.u32 %7, %10, %17;\n\t mul.hi.u32 %8, %10, %17;\n\t"
        "mad.lo.cc.u32 %0, %11, %18, %0;\n\t madc.hi.cc.u32 %1, %11, %18, %1;\n\t madc.lo.cc.u32 %2, %11, %20, %2;\n\t madc.hi.cc.u32 %3, %11, %20, %3;\n\t"
        "addc.u32 %4, 0, 0;\n\t"
        "mad.lo.cc.u32 %5, %11, %19, %5;\n\t madc.hi.cc.u32 %6, %11, %19, %6;\n\t madc.lo.cc.u32 %7, %11, %21, %7;\n\t madc.hi.cc.u32 %8, %11, %21, %8;\n\t"
        "addc.u32 %9, 0, 0;\n\t"
        "mad.lo.cc.u32 %0, %12, %22, %0;\n\t madc.hi.cc.u32 %1, %12, %22, %1;\n\t madc.lo.cc.u32 %2, %12, %24, %2;\n\t madc.hi.cc.u32 %3, %12, %24, %3;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        "mad.lo.cc.u32 %5, %12, %23, %5;\n\t madc.hi.cc.u32 %6, %12, %23, %6;\n\t madc.lo.cc.u32 %7, %12, %25, %7;\n\t madc.hi.cc.u32 %8, %12, %25, %8;\n\t"
        "addc.u32 %9, %9, 0;\n\t"
        "mad.lo.cc.u32 %0, %13, %26, %0;\n\t madc.hi.cc.u32 %1, %13, %26, %1;\n\t madc.lo.cc.u32 %2, %13, %28, %2;\n\t madc.hi.cc.u32 %3, %13, %28, %3;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        "mad.lo.cc.u32 %5, %13, %27, %5;\n\t madc.hi.cc.u32 %6, %13, %27, %6;\n\t madc.lo.cc.u32 %7, %13, %29, %7;\n\t madc.hi.cc.u32 %8, %13, %29, %8;\n\t"
        "addc.u32 %9, %9, 0;\n\t"
        "}"
        : "=&r"(e0), "=&r"(e1), "=&r"(e2), "=&r"(e3), "=&r"(e4), "=&r"(o0), "=&r"(o1), "=&r"(o2), "=&r"(o3), "=&r"(o4)
        : "r"(x.x[0]), "r"(x.x[1]), "r"(x.x[2]), "r"(x.x[3]),
          "r"(t.w[0].x[0]), "r"(t.w[0].x[1]), "r"(t.w[0].x[2]), "r"(t.w[0].x[3]), "r"(t.w[1].x[0]), "r"(t.w[1].x[1]), "r"(t.w[1].x[2]), "r"(t.w[1].x[3]),
          "r"(t.w[2].x[0]), "r"(t.w[2].x[1]), "r"(t.w[2].x[2]), "r"(t.w[2].x[3]), "r"(t.w[3].x[0]), "r"(t.w[3].x[1]), "r"(t.w[3].x[2]), "r"(t.w[3].x[3]));
    // r = even + (odd << 32): six limbs, r5:r4 < 2^34
    uint32_t r1, r2, r3, r4, r5;
    asm("add.cc.u32 %0, %5, %9;\n\t addc.cc.u32 %1, %6, %10;\n\t addc.cc.u32 %2, %7, %11;\n\t addc.cc.u32 %3, %8, %12;\n\t addc.u32 %4, %13, 0;"
        : "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5)
        : "r"(e1), "r"(e2), "r"(e3), "r"(e4), "r"(o0), "r"(o1), "r"(o2), "r"(o3), "r"(o4));
    uint32_t q0, q1, w0, w1, w2, cy;
    fe out;
    asm("{\n\t"
        "mul.lo.u32 %0, %10, %12;\n\t mul.hi.u32 %1, %10, %12;\n\t mad.lo.u32 %1, %11, %12, %1;\n\t"
        "sub.cc.u32 %2, 0, %10;\n\t subc.cc.u32 %3, %0, %11;\n\t subc.u32 %4, %1, 0;\n\t"
        "add.cc.u32 %5, %13, %2;\n\t addc.cc.u32 %6, %14, %3;\n\t addc.cc.u32 %7, %15, %4;\n\t addc.cc.u32 %8, %16, 0;\n\t addc.u32 %9, 0, 0;\n\t"
        "}"
        : "=&r"(q0), "=&r"(q1), "=&r"(w0), "=&r"(w1), "=&r"(w2), "=&r"(out.x[0]), "=&r"(out.x[1]), "=&r"(out.x[2]), "=&r"(out.x[3]), "=&r"(cy)
        : "r"(r4), "r"(r5), "r"(k), "r"(e0), "r"(r1), "r"(r2), "r"(r3));
    return fe_canon(out, cy);
}

// 128-bit square -> 256 bits with 10 wide products instead of 16: the six off-diagonal products are summed once, doubled by a
// one-bit funnel shift, and the four squares added on top
__device__ __forceinline__ void sqr_wide(const fe& a, uint32_t r[8]) {
    const uint32_t a0 = a.x[0], a1 = a.x[1], a2 = a.x[2], a3 = a.x[3];
    uint32_t o1, o2, o3, o4, o5, o6, e2, e3, e4, e5;
    asm("{\n\t"
        "mul.lo.u32 %0, %10, %11;\n\t mul.hi.u32 %1, %10, %11;\n\t"      // a0 a1 @1
        "mul.lo.u32 %2, %10, %13;\n\t mul.hi.u32 %3, %10, %13;\n\t"      // a0 a3 @3
        "mul.lo.u32 %4, %12, %13;\n\t mul.hi.u32 %5, %12, %13;\n\t"      // a2 a3 @5
        "mad.lo.cc.u32 %2, %11, %12, %2;\n\t madc.hi.cc.u32 %3, %11, %12, %3;\n\t"  // + a1 a2 @3
        "addc.cc.u32 %4, %4, 0;\n\t addc.u32 %5, %5, 0;\n\t"
        "mul.lo.u32 %6, %10, %12;\n\t mul.hi.u32 %7, %10, %12;\n\t"      // a0 a2 @2
        "mul.lo.u32 %8, %11, %13;\n\t mul.hi.u32 %9, %11, %13;\n\t"      // a1 a3 @4
        "}"
        : "=&r"(o1), "=&r"(o2), "=&r"(o3), "=&r"(o4), "=&r"(o5), "=&r"(o6), "=&r"(e2), "=&r"(e3), "=&r"(e4), "=&r"(e5)
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3));
    // T = odd + even (limbs 1..7), then D = 2T
    uint32_t t2, t3, t4, t5, t6, t7;
    asm("add.cc.u32 %0, %6, %11;\n\t addc.cc.u32 %1, %7, %12;\n\t addc.cc.u32 %2, %8, %13;\n\t addc.cc.u32 %3, %9, %14;\n\t"
        "addc.cc.u32 %4, %10, 0;\n\t addc.u32 %5, 0, 0;"
        : "=r"(t2), "=r"(t3), "=r"(t4), "=r"(t5), "=r"(t6), "=r"(t7)
        : "r"(o2), "r"(o3), "r"(o4), "r"(o5), "r"(o6), "r"(e2), "r"(e3), "r"(e4), "r"(e5));
    const uint32_t d1 = o1 << 1, d2 = __funnelshift_l(o1, t2, 1), d3 = __funnelshift_l(t2, t3, 1), d4 = __funnelshift_l(t3, t4, 1),
                   d5 = __funnelshift_l(t4, t5, 1), d6 = __funnelshift_l(t5, t6, 1), d7 = __funnelshift_l(t6, t7, 1);
    uint32_t s0, s1, s2, s3, s4, s5, s6, s7;
    asm("mul.lo.u32 %0, %8, %8;\n\t mul.hi.u32 %1, %8, %8;\n\t mul.lo.u32 %2, %9, %9;\n\t mul.hi.u32 %3, %9, %9;\n\t"
        "mul.lo.u32 %4, %10, %10;\n\t mul.hi.u32 %5, %10, %10;\n\t mul.lo.u32 %6, %11, %11;\n\t mul.hi.u32 %7, %11, %11;"
        : "=r"(s0), "=r"(s1), "=r"(s2), "=r"(s3), "=r"(s4), "=r"(s5), "=r"(s6), "=r"(s7)
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3));
    r[0] = s0;
    asm("add.cc.u32 %0, %7, %14;\n\t addc.cc.u32 %1, %8, %15;\n\t addc.cc.u32 %2, %9, %16;\n\t addc.cc.u32 %3, %10, %17;\n\t"
        "addc.cc.u32 %4, %11, %18;\n\t addc.cc.u32 %5, %12, %19;\n\t addc.u32 %6, %13, %20;"
        : "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(s1), "r"(s2), "r"(s3), "r"(s4), "r"(s5), "r"(s6), "r"(s7), "r"(d1), "r"(d2), "r"(d3), "r"(d4), "r"(d5), "r"(d6), "r"(d7));
}
__device__ __forceinline__ fe fe_sqr(const fe& a) {
    uint32_t w[8];
    sqr_wide(a, w);
    return fe_reduce256(w);
}

// Lazy sum of products: a 288-bit integer accumulator takes unreduced 256-bit products (up to 2^32 of them) and is reduced once.
// Exact integer arithmetic, so the canonical result equals the sum of the individually reduced products.
struct acc288 { uint32_t v[9]; };
__device__ __forceinline__ void acc288_zero(acc288& a) {
#pragma unroll
    for (int i = 0; i < 9; i++) a.v[i] = 0;
}
__device__ __forceinline__ void acc288_mad(acc288& a, const fe& x, const fe& y) {
    uint32_t w[8];
    mul_wide(x, y, w);
    asm("add.cc.u32 %0, %0, %9;\n\t addc.cc.u32 %1, %1, %10;\n\t addc.cc.u32 %2, %2, %11;\n\t addc.cc.u32 %3, %3, %12;\n\t"
        "addc.cc.u32 %4, %4, %13;\n\t addc.cc.u32 %5, %5, %14;\n\t addc.cc.u32 %6, %6, %15;\n\t addc.cc.u32 %7, %7, %16;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(a.v[0]), "+r"(a.v[1]), "+r"(a.v[2]), "+r"(a.v[3]), "+r"(a.v[4]), "+r"(a.v[5]), "+r"(a.v[6]), "+r"(a.v[7]), "+r"(a.v[8])
        : "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]));
}
__device__ __forceinline__ fe acc288_reduce(const acc288& a) {
    const fe lo = fe_reduce256(a.v);
    // limb 8 carries weight 2^256 = C^2 = 2025*2^80 - 90*2^40 + 1 (mod p, and < 2^92 so the product below is canonical)
    const uint32_t k0 = 0x00000001u, k1 = 0xFFFFA600u, k2 = 0x07E8FFFFu, t = a.v[8];
    fe hi;
    uint32_t m0, m1;
    asm("mul.lo.u32 %0, %6, %7;\n\t mul.hi.u32 %1, %6, %7;\n\t"      // t k0 @0
        "mul.lo.u32 %2, %6, %9;\n\t mul.hi.u32 %3, %6, %9;\n\t"      // t k2 @2
        "mul.lo.u32 %4, %6, %8;\n\t mul.hi.u32 %5, %6, %8;"            // t k1 @1
        : "=r"(hi.x[0]), "=r"(hi.x[1]), "=r"(hi.x[2]), "=r"(hi.x[3]), "=r"(m0), "=r"(m1)
        : "r"(t), "r"(k0), "r"(k1), "r"(k2));
    asm("add.cc.u32 %0, %0, %3;\n\t addc.cc.u32 %1, %1, %4;\n\t addc.u32 %2, %2, 0;"
        : "+r"(hi.x[1]), "+r"(hi.x[2]), "+r"(hi.x[3]) : "r"(m0), "r"(m1));
    return fe_add(lo, hi);
}

// a^e for a 128-bit exponent given as limbs (used for inversion and small fixed powers)
__device__ __forceinline__ fe fe_pow_u64(fe b, uint64_t e) {
    fe r = fe_one();
    while (e) { if (e & 1) r = fe_mul(r, b); b = fe_sqr(b); e >>= 1; }
    return r;
}
// a^(p-2); inv(0) = 0 as in winter-math.  p - 2 = 0xFFFFFFFF_FFFFFFFF_FFFFD2FF_FFFFFFFF: 80 ones, 1101001011111111, 32 ones.
// Addition chain over e_k = a^(2^k - 1): 127 squarings + 12 multiplications (square-and-multiply needs 127 + 121).
__device__ __forceinline__ fe fe_sqr_n(fe x, int k) {
    for (int i = 0; i < k; i++) x = fe_sqr(x);
    return x;
}
// The chain is written once: fe_inv_inline is inlined into its caller (the batch verifier's kernels), fe_inv is the prover's
// out-of-line call.  Calling fe_inv from more kernels would change how the prover's callers are allocated around the call.
__device__ __forceinline__ fe fe_inv_inline(const fe& a) {
    const fe e2 = fe_mul(fe_sqr(a), a);
    const fe e4 = fe_mul(fe_sqr_n(e2, 2), e2);
    const fe e8 = fe_mul(fe_sqr_n(e4, 4), e4);
    const fe e16 = fe_mul(fe_sqr_n(e8, 8), e8);
    const fe e32 = fe_mul(fe_sqr_n(e16, 16), e16);
    const fe e64 = fe_mul(fe_sqr_n(e32, 32), e32);
    fe r = fe_mul(fe_sqr_n(e64, 16), e16);   // bits 127..48
    r = fe_mul(fe_sqr_n(r, 2), e2);          // 11
    r = fe_mul(fe_sqr_n(r, 2), a);           // 01
    r = fe_mul(fe_sqr_n(r, 3), a);           // 001
    r = fe_mul(fe_sqr_n(r, 9), e8);          // 0 11111111
    return fe_mul(fe_sqr_n(r, 32), e32);     // 32 ones
}
__device__ __noinline__ fe fe_inv(const fe& a) { return fe_inv_inline(a); }

}  // namespace zkb
