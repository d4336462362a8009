// BLS12-381 base field Fp on 12 x 32-bit limbs, Montgomery form (R = 2^384), values kept canonical in [0, p).
//
// Replaces arkworks' Fp<MontBackend<FqConfig,6>,6> (the type named at reference src/hasher.rs:1040) for the
// hot path of src/bls.rs:427-458.  12 x u32 little-endian limbs with R = 2^384 are byte-identical to
// arkworks' 6 x u64 limbs, so no conversion is needed at the boundary.
//
// The multiply is an operand-scanning Montgomery product over two carry-save accumulators ("even" and
// "odd" columns) so that every 32x32->64 MAC is a single IMAD.WIDE.U32(.X) whose carry rides the predicate
// chain: 300 IMAD-pipe instructions per product (12*12 product + 12*12 reduction + 12 quotients) and ~70
// ALU-pipe instructions.  Each carry chain is ONE asm statement, so the compiler cannot interleave chains.
//
// Lineage: the even/odd carry-save scheme and the helper shapes (cmad_n, madc_n_rshift, mad_n_redc) follow the public
// mont_t.cuh of supranational/sppark (Apache-2.0), restated for 12 limbs with one asm statement per carry chain; the
// reference itself (arkworks' MontBackend) has no GPU code.
//
// The same source builds for the host (g++, tests/hostemu) with plain-C fallbacks of every asm block, which
// is how the algorithm layer above is debugged without a GPU.  The product library is nvcc-only.
#pragma once
#include <cstdint>
#include <cstddef>
#include "consts.cuh"

#if defined(__CUDACC__)
#define BLS_HD __device__ __forceinline__
#define BLS_NOINLINE __device__ __noinline__
#define BLS_CONST static __device__ __constant__
#else
#define BLS_HD static inline
#define BLS_NOINLINE static __attribute__((noinline))
#define BLS_CONST static const
#endif

#ifdef BLS_ASM_VOLATILE
#define BLS_ASM asm volatile
#else
#define BLS_ASM asm
#endif

namespace bls {

struct alignas(16) fp { uint32_t l[12]; };

// p, little-endian 32-bit limbs (SURVEY A.1)
#define BLS_P0 0xffffaaabu
#define BLS_P1 0xb9feffffu
#define BLS_P2 0xb153ffffu
#define BLS_P3 0x1eabfffeu
#define BLS_P4 0xf6b0f624u
#define BLS_P5 0x6730d2a0u
#define BLS_P6 0xf38512bfu
#define BLS_P7 0x64774b84u
#define BLS_P8 0x434bacd7u
#define BLS_P9 0x4b1ba7b6u
#define BLS_P10 0x397fe69au
#define BLS_P11 0x1a0111eau
#define BLS_M0 0xfffcfffdu      // -p^-1 mod 2^32

BLS_HD uint32_t fp_p_limb(int i) {
    const uint32_t P[12] = {BLS_P0, BLS_P1, BLS_P2, BLS_P3, BLS_P4, BLS_P5, BLS_P6, BLS_P7, BLS_P8, BLS_P9, BLS_P10, BLS_P11};
    return P[i];
}

// ------------------------------------------------------------------------------------------------ add / sub
#if defined(__CUDA_ARCH__)
// r = a + b (384-bit, carry out impossible for a,b < p < 2^381).  Outputs are early-clobber: limb i is written before
// the inputs of limbs > i are read, so an output must never share a register with an input.
BLS_HD void fp_add_raw(fp& r, const fp& a, const fp& b) {
    BLS_ASM("add.cc.u32 %0, %12, %24;\n\taddc.cc.u32 %1, %13, %25;\n\taddc.cc.u32 %2, %14, %26;\n\taddc.cc.u32 %3, %15, %27;\n\t"
        "addc.cc.u32 %4, %16, %28;\n\taddc.cc.u32 %5, %17, %29;\n\taddc.cc.u32 %6, %18, %30;\n\taddc.cc.u32 %7, %19, %31;\n\t"
        "addc.cc.u32 %8, %20, %32;\n\taddc.cc.u32 %9, %21, %33;\n\taddc.cc.u32 %10, %22, %34;\n\taddc.u32 %11, %23, %35;"
        : "=&r"(r.l[0]), "=&r"(r.l[1]), "=&r"(r.l[2]), "=&r"(r.l[3]), "=&r"(r.l[4]), "=&r"(r.l[5]), "=&r"(r.l[6]), "=&r"(r.l[7]), "=&r"(r.l[8]), "=&r"(r.l[9]), "=&r"(r.l[10]), "=&r"(r.l[11])
        : "r"(a.l[0]), "r"(a.l[1]), "r"(a.l[2]), "r"(a.l[3]), "r"(a.l[4]), "r"(a.l[5]), "r"(a.l[6]), "r"(a.l[7]), "r"(a.l[8]), "r"(a.l[9]), "r"(a.l[10]), "r"(a.l[11]),
          "r"(b.l[0]), "r"(b.l[1]), "r"(b.l[2]), "r"(b.l[3]), "r"(b.l[4]), "r"(b.l[5]), "r"(b.l[6]), "r"(b.l[7]), "r"(b.l[8]), "r"(b.l[9]), "r"(b.l[10]), "r"(b.l[11]));
}
// r = a - b (384-bit), returns the borrow as 0 / 0xffffffff
BLS_HD uint32_t fp_sub_raw(fp& r, const fp& a, const fp& b) {
    uint32_t br;
    BLS_ASM("sub.cc.u32 %0, %13, %25;\n\tsubc.cc.u32 %1, %14, %26;\n\tsubc.cc.u32 %2, %15, %27;\n\tsubc.cc.u32 %3, %16, %28;\n\t"
        "subc.cc.u32 %4, %17, %29;\n\tsubc.cc.u32 %5, %18, %30;\n\tsubc.cc.u32 %6, %19, %31;\n\tsubc.cc.u32 %7, %20, %32;\n\t"
        "subc.cc.u32 %8, %21, %33;\n\tsubc.cc.u32 %9, %22, %34;\n\tsubc.cc.u32 %10, %23, %35;\n\tsubc.cc.u32 %11, %24, %36;\n\t"
        "subc.u32 %12, 0, 0;"
        : "=&r"(r.l[0]), "=&r"(r.l[1]), "=&r"(r.l[2]), "=&r"(r.l[3]), "=&r"(r.l[4]), "=&r"(r.l[5]), "=&r"(r.l[6]), "=&r"(r.l[7]), "=&r"(r.l[8]), "=&r"(r.l[9]), "=&r"(r.l[10]), "=&r"(r.l[11]), "=&r"(br)
        : "r"(a.l[0]), "r"(a.l[1]), "r"(a.l[2]), "r"(a.l[3]), "r"(a.l[4]), "r"(a.l[5]), "r"(a.l[6]), "r"(a.l[7]), "r"(a.l[8]), "r"(a.l[9]), "r"(a.l[10]), "r"(a.l[11]),
          "r"(b.l[0]), "r"(b.l[1]), "r"(b.l[2]), "r"(b.l[3]), "r"(b.l[4]), "r"(b.l[5]), "r"(b.l[6]), "r"(b.l[7]), "r"(b.l[8]), "r"(b.l[9]), "r"(b.l[10]), "r"(b.l[11]));
    return br;
}
#else
BLS_HD void fp_add_raw(fp& r, const fp& a, const fp& b) {
    uint64_t c = 0;
    for (int i = 0; i < 12; i++) { c += (uint64_t)a.l[i] + b.l[i]; r.l[i] = (uint32_t)c; c >>= 32; }
}
BLS_HD uint32_t fp_sub_raw(fp& r, const fp& a, const fp& b) {
    uint64_t br = 0;
    for (int i = 0; i < 12; i++) { uint64_t d = (uint64_t)a.l[i] - b.l[i] - br; r.l[i] = (uint32_t)d; br = (d >> 32) & 1; }
    return br ? 0xffffffffu : 0u;
}
#endif

BLS_HD fp fp_modulus() {
    fp m;
#pragma unroll
    for (int i = 0; i < 12; i++) m.l[i] = fp_p_limb(i);
    return m;
}
BLS_HD fp fp_zero() {
    fp r;
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = 0;
    return r;
}
// Montgomery 1 = R mod p
BLS_HD fp fp_one() {
    const uint32_t O[12] = BLS_C_ONE;
    fp r;
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = O[i];
    return r;
}
// R^2 mod p (to-Montgomery multiplier)
BLS_HD fp fp_r2() {
    const uint32_t O[12] = BLS_C_R2;
    fp r;
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = O[i];
    return r;
}
BLS_HD fp fp_select(uint32_t mask, const fp& a, const fp& b) {   // mask ? a : b, mask in {0, ~0}
    fp r;
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = (a.l[i] & mask) | (b.l[i] & ~mask);
    return r;
}
BLS_HD fp fp_csel(bool c, const fp& a, const fp& b) { return fp_select(c ? 0xffffffffu : 0u, a, b); }
BLS_HD bool fp_is_zero(const fp& a) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) o |= a.l[i];
    return o == 0;
}
BLS_HD bool fp_eq(const fp& a, const fp& b) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) o |= a.l[i] ^ b.l[i];
    return o == 0;
}
// reduce a value in [0, 2p) to [0, p)
BLS_HD fp fp_reduce_once(const fp& a) {
    fp t; uint32_t br = fp_sub_raw(t, a, fp_modulus());
    return fp_select(br, a, t);
}
BLS_HD fp fp_add(const fp& a, const fp& b) { fp s; fp_add_raw(s, a, b); return fp_reduce_once(s); }
BLS_HD fp fp_sub(const fp& a, const fp& b) {
    fp d; uint32_t br = fp_sub_raw(d, a, b);
    fp m = fp_modulus();
#pragma unroll
    for (int i = 0; i < 12; i++) m.l[i] &= br;
    fp r; fp_add_raw(r, d, m); return r;
}
BLS_HD fp fp_neg(const fp& a) {
    fp d; fp_sub_raw(d, fp_modulus(), a);
    return fp_select(fp_is_zero(a) ? 0xffffffffu : 0u, a, d);
}
BLS_HD fp fp_dbl(const fp& a) { return fp_add(a, a); }
// a / 2 mod p: (a + (a odd ? p : 0)) >> 1 -- ALU only (the Montgomery image of a/2 is half the image of a)
BLS_HD fp fp_half(const fp& a) {
    uint32_t mask = 0u - (a.l[0] & 1u);
    fp m = fp_modulus();
#pragma unroll
    for (int i = 0; i < 12; i++) m.l[i] &= mask;
    fp t; fp_add_raw(t, a, m);                       // < 2p < 2^382: no carry out
    fp r;
#pragma unroll
    for (int i = 0; i < 11; i++) r.l[i] = (t.l[i] >> 1) | (t.l[i + 1] << 31);
    r.l[11] = t.l[11] >> 1;
    return r;
}
// canonical (non-Montgomery) integer comparison helpers work on canonical limbs
BLS_HD bool fp_raw_geq(const fp& a, const fp& b) { fp t; return fp_sub_raw(t, a, b) == 0; }

// ------------------------------------------------------------------------------------------------ Montgomery product
#if defined(__CUDA_ARCH__)
// acc[0..11] += a[0,2,..,10] * bi along one carry chain; the carry out is added to top
#define BLS_CMAD_BODY                                                                                                   \
    "mad.lo.cc.u32 %0, %13, %19, %0;\n\tmadc.hi.cc.u32 %1, %13, %19, %1;\n\t"                                            \
    "madc.lo.cc.u32 %2, %14, %19, %2;\n\tmadc.hi.cc.u32 %3, %14, %19, %3;\n\t"                                           \
    "madc.lo.cc.u32 %4, %15, %19, %4;\n\tmadc.hi.cc.u32 %5, %15, %19, %5;\n\t"                                           \
    "madc.lo.cc.u32 %6, %16, %19, %6;\n\tmadc.hi.cc.u32 %7, %16, %19, %7;\n\t"                                           \
    "madc.lo.cc.u32 %8, %17, %19, %8;\n\tmadc.hi.cc.u32 %9, %17, %19, %9;\n\t"                                           \
    "madc.lo.cc.u32 %10, %18, %19, %10;\n\tmadc.hi.cc.u32 %11, %18, %19, %11;\n\t"                                       \
    "addc.u32 %12, %12, 0;"
BLS_HD void cmad_n(uint32_t* acc, uint32_t& top, uint32_t a0, uint32_t a2, uint32_t a4, uint32_t a6, uint32_t a8, uint32_t a10, uint32_t bi) {
    BLS_ASM(BLS_CMAD_BODY
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10]), "+r"(acc[11]), "+r"(top)
        : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(a8), "r"(a10), "r"(bi));
}
// e0 += o[1] (carry into the chain); then o[j],o[j+1] = a_j*bi + o[j+2],o[j+3] for the five low pairs and
// o[10],o[11] = a_10*bi + carry: "accumulate the odd columns while shifting the accumulator down two limbs"
BLS_HD void madc_n_rshift(uint32_t& e0, uint32_t* o, uint32_t a1, uint32_t a3, uint32_t a5, uint32_t a7, uint32_t a9, uint32_t a11, uint32_t bi) {
    BLS_ASM("add.cc.u32 %12, %12, %1;\n\t"
        "madc.lo.cc.u32 %0, %13, %19, %2;\n\tmadc.hi.cc.u32 %1, %13, %19, %3;\n\t"
        "madc.lo.cc.u32 %2, %14, %19, %4;\n\tmadc.hi.cc.u32 %3, %14, %19, %5;\n\t"
        "madc.lo.cc.u32 %4, %15, %19, %6;\n\tmadc.hi.cc.u32 %5, %15, %19, %7;\n\t"
        "madc.lo.cc.u32 %6, %16, %19, %8;\n\tmadc.hi.cc.u32 %7, %16, %19, %9;\n\t"
        "madc.lo.cc.u32 %8, %17, %19, %10;\n\tmadc.hi.cc.u32 %9, %17, %19, %11;\n\t"
        "madc.lo.cc.u32 %10, %18, %19, 0;\n\tmadc.hi.u32 %11, %18, %19, 0;"
        : "+r"(o[0]), "+r"(o[1]), "+r"(o[2]), "+r"(o[3]), "+r"(o[4]), "+r"(o[5]), "+r"(o[6]), "+r"(o[7]), "+r"(o[8]), "+r"(o[9]), "+r"(o[10]), "+r"(o[11]), "+r"(e0)
        : "r"(a1), "r"(a3), "r"(a5), "r"(a7), "r"(a9), "r"(a11), "r"(bi));
}
#else
BLS_HD void cmad_n(uint32_t* acc, uint32_t& top, uint32_t a0, uint32_t a2, uint32_t a4, uint32_t a6, uint32_t a8, uint32_t a10, uint32_t bi) {
    const uint32_t a[6] = {a0, a2, a4, a6, a8, a10};
    uint64_t c = 0;
    for (int j = 0; j < 6; j++) {
        unsigned __int128 t = (unsigned __int128)a[j] * bi + (((uint64_t)acc[2 * j + 1] << 32) | acc[2 * j]) + c;
        acc[2 * j] = (uint32_t)t; acc[2 * j + 1] = (uint32_t)(t >> 32); c = (uint64_t)(t >> 64);
    }
    top += (uint32_t)c;
}
BLS_HD void madc_n_rshift(uint32_t& e0, uint32_t* o, uint32_t a1, uint32_t a3, uint32_t a5, uint32_t a7, uint32_t a9, uint32_t a11, uint32_t bi) {
    const uint32_t a[6] = {a1, a3, a5, a7, a9, a11};
    uint64_t s = (uint64_t)e0 + o[1]; e0 = (uint32_t)s; uint64_t c = s >> 32;
    for (int j = 0; j < 6; j++) {
        uint64_t addend = j < 5 ? (((uint64_t)o[2 * j + 3] << 32) | o[2 * j + 2]) : 0;
        unsigned __int128 t = (unsigned __int128)a[j] * bi + addend + c;
        o[2 * j] = (uint32_t)t; o[2 * j + 1] = (uint32_t)(t >> 32); c = (uint64_t)(t >> 64);
    }
}
#endif

// one row of the interleaved product/reduction: even/odd swap roles every call
BLS_HD void mad_n_redc(uint32_t* even, uint32_t* odd, const fp& a, uint32_t bi, bool first) {
    if (first) {
#pragma unroll
        for (int j = 0; j < 12; j += 2) {
            uint64_t te = (uint64_t)a.l[j] * bi, to = (uint64_t)a.l[j + 1] * bi;
            even[j] = (uint32_t)te; even[j + 1] = (uint32_t)(te >> 32);
            odd[j] = (uint32_t)to; odd[j + 1] = (uint32_t)(to >> 32);
        }
    } else {
        madc_n_rshift(even[0], odd, a.l[1], a.l[3], a.l[5], a.l[7], a.l[9], a.l[11], bi);
        cmad_n(even, odd[11], a.l[0], a.l[2], a.l[4], a.l[6], a.l[8], a.l[10], bi);
    }
    uint32_t mi = even[0] * BLS_M0;
    uint32_t drop = 0;
    cmad_n(odd, drop, BLS_P1, BLS_P3, BLS_P5, BLS_P7, BLS_P9, BLS_P11, mi);
    cmad_n(even, odd[11], BLS_P0, BLS_P2, BLS_P4, BLS_P6, BLS_P8, BLS_P10, mi);
}

BLS_HD fp fp_mul_inl(const fp& a, const fp& b) {
    uint32_t even[12], odd[12];
#pragma unroll
    for (int i = 0; i < 12; i += 2) {
        mad_n_redc(even, odd, a, b.l[i], i == 0);
        mad_n_redc(odd, even, a, b.l[i + 1], false);
    }
    // merge: result = even + (odd >> 32); even[0] absorbs odd[1], ...
    fp r, s;
#pragma unroll
    for (int i = 0; i < 11; i++) { r.l[i] = even[i]; s.l[i] = odd[i + 1]; }
    r.l[11] = even[11]; s.l[11] = 0;
    fp t; fp_add_raw(t, r, s);
    return fp_reduce_once(t);
}

// ------------------------------------------------------------------------------------------------ double-width arithmetic
// Unreduced 768-bit products and a separate Montgomery reduction, for lazy reduction in Fp2 (one reduction per output
// coefficient instead of one per product).  Rows are added into a resolved 24-limb accumulator T with two carry chains
// (even / odd columns of the multiplicand); the carry out of a chain that ends at limb k is *counted* in C[k] instead of
// rippling (limbs >= 12 are never read before the final resolve, so deferring the carries is exact).
struct fpw { uint32_t l[24]; };
#if defined(__CUDACC__)
#pragma nv_diag_suppress 550
#endif
#if defined(__CUDA_ARCH__)
BLS_HD uint32_t add12c(uint32_t* r, const uint32_t* a, const uint32_t* b, uint32_t cin) {      // r = a + b + cin, returns carry (0/1)
    uint32_t cout, tmp;
    BLS_ASM("add.cc.u32 %13, %38, 0xffffffff;\n\taddc.cc.u32 %0, %14, %26;\n\taddc.cc.u32 %1, %15, %27;\n\taddc.cc.u32 %2, %16, %28;\n\taddc.cc.u32 %3, %17, %29;\n\t"
        "addc.cc.u32 %4, %18, %30;\n\taddc.cc.u32 %5, %19, %31;\n\taddc.cc.u32 %6, %20, %32;\n\taddc.cc.u32 %7, %21, %33;\n\t"
        "addc.cc.u32 %8, %22, %34;\n\taddc.cc.u32 %9, %23, %35;\n\taddc.cc.u32 %10, %24, %36;\n\taddc.cc.u32 %11, %25, %37;\n\taddc.u32 %12, 0, 0;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7]), "=&r"(r[8]), "=&r"(r[9]), "=&r"(r[10]), "=&r"(r[11]), "=&r"(cout), "=&r"(tmp)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(a[8]), "r"(a[9]), "r"(a[10]), "r"(a[11]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]), "r"(b[8]), "r"(b[9]), "r"(b[10]), "r"(b[11]), "r"(cin));
    return cout;
}
BLS_HD uint32_t sub12b(uint32_t* r, const uint32_t* a, const uint32_t* b, uint32_t bin) {      // r = a - b - bin, returns borrow (0/1)
    uint32_t bout, tmp;
    BLS_ASM("sub.cc.u32 %13, 0, %38;\n\tsubc.cc.u32 %0, %14, %26;\n\tsubc.cc.u32 %1, %15, %27;\n\tsubc.cc.u32 %2, %16, %28;\n\tsubc.cc.u32 %3, %17, %29;\n\t"
        "subc.cc.u32 %4, %18, %30;\n\tsubc.cc.u32 %5, %19, %31;\n\tsubc.cc.u32 %6, %20, %32;\n\tsubc.cc.u32 %7, %21, %33;\n\t"
        "subc.cc.u32 %8, %22, %34;\n\tsubc.cc.u32 %9, %23, %35;\n\tsubc.cc.u32 %10, %24, %36;\n\tsubc.cc.u32 %11, %25, %37;\n\tsubc.u32 %12, 0, 0;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7]), "=&r"(r[8]), "=&r"(r[9]), "=&r"(r[10]), "=&r"(r[11]), "=&r"(bout), "=&r"(tmp)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(a[8]), "r"(a[9]), "r"(a[10]), "r"(a[11]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]), "r"(b[8]), "r"(b[9]), "r"(b[10]), "r"(b[11]), "r"(bin));
    return bout & 1u;
}
#else
BLS_HD uint32_t add12c(uint32_t* r, const uint32_t* a, const uint32_t* b, uint32_t cin) {
    uint64_t c = cin; uint32_t t[12];
    for (int i = 0; i < 12; i++) { c += (uint64_t)a[i] + b[i]; t[i] = (uint32_t)c; c >>= 32; }
    for (int i = 0; i < 12; i++) r[i] = t[i];
    return (uint32_t)c;
}
BLS_HD uint32_t sub12b(uint32_t* r, const uint32_t* a, const uint32_t* b, uint32_t bin) {
    uint64_t br = bin; uint32_t t[12];
    for (int i = 0; i < 12; i++) { uint64_t d = (uint64_t)a[i] - b[i] - br; t[i] = (uint32_t)d; br = (d >> 32) & 1; }
    for (int i = 0; i < 12; i++) r[i] = t[i];
    return (uint32_t)br;
}
#endif
BLS_HD void fpw_add(fpw& r, const fpw& a, const fpw& b) { uint32_t c = add12c(r.l, a.l, b.l, 0); add12c(r.l + 12, a.l + 12, b.l + 12, c); }
BLS_HD void fpw_sub(fpw& r, const fpw& a, const fpw& b) { uint32_t c = sub12b(r.l, a.l, b.l, 0); sub12b(r.l + 12, a.l + 12, b.l + 12, c); }   // mod 2^768

// T = a * b, 768 bits, resolved.  a, b < 2^384 (not necessarily reduced).
BLS_HD void fp_mul_wide(fpw& T, const fp& a, const fp& b) {
    uint32_t C[14];
#pragma unroll
    for (int i = 0; i < 24; i++) T.l[i] = 0;
#pragma unroll
    for (int i = 0; i < 14; i++) C[i] = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        cmad_n(&T.l[i], C[i], a.l[0], a.l[2], a.l[4], a.l[6], a.l[8], a.l[10], b.l[i]);              // carry belongs to limb i+12
        if (i < 11) cmad_n(&T.l[i + 1], C[i + 1], a.l[1], a.l[3], a.l[5], a.l[7], a.l[9], a.l[11], b.l[i]);   // limb i+13
        else {      // last odd row: the top pair lands on limbs 22,23 and the product cannot carry out of limb 23
            uint32_t drop = 0; cmad_n(&T.l[12], drop, a.l[1], a.l[3], a.l[5], a.l[7], a.l[9], a.l[11], b.l[11]);
        }
    }
    // resolve: limb 12+k += C[k] (C[k] counts carries out of the chains that ended at limb 11+k)
    uint32_t hi[12], cc[12];
#pragma unroll
    for (int k = 0; k < 12; k++) { hi[k] = T.l[12 + k]; cc[k] = C[k]; }
    add12c(&T.l[12], hi, cc, 0);
}
// Montgomery reduction of X < p * 2^384 to [0, p)
BLS_HD fp fp_redc_wide(const fpw& Xin) {
    fpw X = Xin; uint32_t C[14];
#pragma unroll
    for (int i = 0; i < 14; i++) C[i] = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        uint32_t m = X.l[i] * BLS_M0;
        cmad_n(&X.l[i], C[i], BLS_P0, BLS_P2, BLS_P4, BLS_P6, BLS_P8, BLS_P10, m);
        if (i < 11) cmad_n(&X.l[i + 1], C[i + 1], BLS_P1, BLS_P3, BLS_P5, BLS_P7, BLS_P9, BLS_P11, m);
        else { uint32_t drop = 0; cmad_n(&X.l[12], drop, BLS_P1, BLS_P3, BLS_P5, BLS_P7, BLS_P9, BLS_P11, m); }   // result < 2p: no carry out of limb 23
    }
    fp hi, cc, t;
#pragma unroll
    for (int k = 0; k < 12; k++) { hi.l[k] = X.l[12 + k]; cc.l[k] = C[k]; }
    fp_add_raw(t, hi, cc);
    return fp_reduce_once(t);
}
// p^2 (768 bits): added to a difference of two products to keep it non-negative (it is 0 mod p)
BLS_HD fpw fpw_p_squared() { const uint32_t Q[24] = BLS_C_P_SQUARED; fpw r;
#pragma unroll
    for (int i = 0; i < 24; i++) r.l[i] = Q[i];
    return r; }

#if defined(__CUDACC__)
BLS_NOINLINE fp fp_mul(fp a, fp b) { return fp_mul_inl(a, b); }
BLS_NOINLINE fp fp_sqr(fp a) { return fp_mul_inl(a, a); }
#else
BLS_NOINLINE fp fp_mul(const fp& a, const fp& b) { return fp_mul_inl(a, b); }
BLS_NOINLINE fp fp_sqr(const fp& a) { return fp_mul_inl(a, a); }
#endif

BLS_HD fp fp_to_mont(const fp& a) { return fp_mul(a, fp_r2()); }
BLS_HD fp fp_from_mont(const fp& a) { fp one = fp_zero(); one.l[0] = 1; return fp_mul(a, one); }

// a^e for a fixed public exponent given as 32-bit LE words; 4-bit fixed window
BLS_HD fp fp_pow(const fp& a, const uint32_t* e, int nwords) {
    fp tab[16];
    tab[0] = fp_one(); tab[1] = a;
    for (int i = 2; i < 16; i++) tab[i] = fp_mul(tab[i - 1], a);
    fp r = fp_one();
    bool started = false;
    for (int w = nwords - 1; w >= 0; w--) {
        uint32_t word = e[w];
        for (int s = 28; s >= 0; s -= 4) {
            uint32_t d = (word >> s) & 15;
            if (started) { r = fp_sqr(r); r = fp_sqr(r); r = fp_sqr(r); r = fp_sqr(r); }
            if (d) { r = started ? fp_mul(r, tab[d]) : tab[d]; started = true; }
        }
    }
    return r;
}

// fixed exponents derived from p (32-bit LE words)
BLS_CONST uint32_t EXP_P_MINUS_2[12] = BLS_C_EXP_PM2;
// (p-3)/4 ; note (p+1)/4 = (p-3)/4 + 1
BLS_CONST uint32_t EXP_P_MINUS_3_DIV_4[12] = BLS_C_EXP_PM3D4;

// c z mod p for a canonical z and a 32-bit c (canonical result, no Montgomery factor): 12 MACs for the product, a 64 x 34-bit
// Barrett estimate of the quotient from the top 63 bits (q or q - 1: T = floor(t / 2^350) < 2^63, mu = floor(2^414 / p), so
// floor(T mu / 2^64) > t/p - 1/2 - 2^-30), 12 MACs for q p and one conditional subtraction.  Used for the small coefficients of the
// R1CS matrices (80 % of the non-unit ones in the verify circuit: 2, 3, 4, 12, 2^k ...): 24 MACs instead of 300.
// t (13 limbs, < 2^413) mod p: the Barrett step described above
BLS_HD fp fp_barrett13(const uint32_t* t) {
    const uint32_t PL[12] = BLS_C_P;
    uint64_t T = ((uint64_t)t[12] << 34) | ((uint64_t)t[11] << 2) | (uint64_t)(t[10] >> 30);
#if defined(__CUDA_ARCH__)
    uint32_t q = (uint32_t)__umul64hi(T, BLS_C_MU414);
#else
    uint32_t q = (uint32_t)(((unsigned __int128)T * BLS_C_MU414) >> 64);
#endif
    fp r; uint64_t mc = 0; int64_t br = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        uint64_t m = (uint64_t)PL[i] * q + mc; mc = m >> 32;
        int64_t d = (int64_t)(uint64_t)t[i] - (int64_t)(uint64_t)(uint32_t)m + br; r.l[i] = (uint32_t)d; br = d >> 32;
    }
    return fp_reduce_once(r);                                 // t - q p < 2p < 2^382: the thirteenth limb cancels
}
BLS_HD fp fp_mul_small(const fp& z, uint32_t c) {
    uint32_t t[13]; uint64_t carry = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) { uint64_t v = (uint64_t)z.l[i] * c + carry; t[i] = (uint32_t)v; carry = v >> 32; }
    t[12] = (uint32_t)carry;
    return fp_barrett13(t);
}
// Lazy sums of small-coefficient terms: X = sum c_i z_i (c_i < 2^32, z_i canonical) is accumulated UNREDUCED in 14 limbs -- 12
// IMAD.WIDE and two carry fix-ups per term instead of a product, a Barrett step and a conditional subtraction each -- and reduced
// once.  Negative coefficients enter as |c| (p - z).  Capacity: at most 2^19 terms between reductions (X < 2^432).
struct fp_lacc { uint32_t l[14]; };
BLS_HD void fp_lacc_zero(fp_lacc& a) {
#pragma unroll
    for (int i = 0; i < 14; i++) a.l[i] = 0;
}
BLS_HD void fp_lacc_mad(fp_lacc& a, const fp& z, uint32_t c) {
    uint32_t cy = 0;
    cmad_n(&a.l[0], cy, z.l[0], z.l[2], z.l[4], z.l[6], z.l[8], z.l[10], c);          // limbs 0..11, carry -> limb 12 (and on into 13)
    uint64_t s = (uint64_t)a.l[12] + cy; a.l[12] = (uint32_t)s; a.l[13] += (uint32_t)(s >> 32);
    cmad_n(&a.l[1], a.l[13], z.l[1], z.l[3], z.l[5], z.l[7], z.l[9], z.l[11], c);     // limbs 1..12, carry -> limb 13
}
BLS_HD fp fp_lacc_reduce(const fp_lacc& a) {                   // X < 2^432 -> [0, p)
    const uint32_t K[12] = BLS_C_K400;
    uint32_t hi = (a.l[12] >> 16) | (a.l[13] << 16);          // X >> 400
    uint32_t t[13]; uint64_t carry = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) { uint64_t v = (uint64_t)K[i] * hi + a.l[i] + carry; t[i] = (uint32_t)v; carry = v >> 32; }
    t[12] = (a.l[12] & 0xffffu) + (uint32_t)carry;            // (X mod 2^400) + hi (2^400 mod p) < 2^400 + 2^413: within fp_barrett13's range
    return fp_barrett13(t);
}

BLS_HD fp fp_inv_fermat(const fp& a) { return fp_pow(a, EXP_P_MINUS_2, 12); }          // 0 -> 0

// ------------------------------------------------------------------------------------------------ inversion by divsteps
// Bernstein-Yang "safegcd" (delta = 1 form): (delta, f, g) -> (1 - delta, g, (g - f) / 2) when delta > 0 and g is odd, else
// (1 + delta, f, (g + (g mod 2) f) / 2).  62 divsteps at a time on the low words give a 2x2 transition matrix (entries < 2^62
// in magnitude), which is then applied to the full-width (f, g) exactly and to the Bezout pair (d, e) modulo p.  The published
// bound for 381-bit inputs is floor((49 * 381 + 57) / 17) = 1,101 divsteps <= 18 batches; random inputs end after 13-14 (the loop
// stops when g = 0, a lane that finishes early idles).  Branch-free inside a batch, ALU-pipe work only: ~35 k simple instructions
// against ~490 Montgomery products (150 k IMAD.WIDE) for a^(p-2).  Values are 7 limbs of 62 bits, the top limb signed.
// The same value as the Fermat form for every input (the inverse is unique; 0 -> 0), checked in tests/devcheck.
struct inv_mat { int64_t u, v, q, r; };
BLS_HD int64_t inv_divsteps62(int64_t eta, uint64_t f, uint64_t g, inv_mat& t) {     // eta = -delta
    uint64_t u = 1, v = 0, q = 0, r = 1;
#pragma unroll 2
    for (int i = 0; i < 62; i++) {
        uint64_t c1 = (uint64_t)(eta >> 63), c2 = 0 - (g & 1);                        // delta > 0; g odd
        uint64_t x = (f ^ c1) - c1, y = (u ^ c1) - c1, z = (v ^ c1) - c1;             // (f, u, v) negated when delta > 0
        g += x & c2; q += y & c2; r += z & c2;
        c1 &= c2;
        eta = (int64_t)(((uint64_t)eta ^ c1) - (c1 + 1));                             // swap: delta -> 1 - delta, else delta + 1
        f += g & c1; u += q & c1; v += r & c1;
        g >>= 1; u <<= 1; v <<= 1;
    }
    t.u = (int64_t)u; t.v = (int64_t)v; t.q = (int64_t)q; t.r = (int64_t)r;          // 2^62 times the transition matrix
    return eta;
}
#define BLS_INV_M62 ((int64_t)0x3fffffffffffffffLL)
BLS_HD void inv_to62(int64_t* o, const uint32_t* l) {
    uint64_t w[6];
#pragma unroll
    for (int i = 0; i < 6; i++) w[i] = (uint64_t)l[2 * i] | ((uint64_t)l[2 * i + 1] << 32);
    o[0] = (int64_t)(w[0] & (uint64_t)BLS_INV_M62);
#pragma unroll
    for (int i = 1; i < 6; i++) o[i] = (int64_t)(((w[i - 1] >> (64 - 2 * i)) | (w[i] << (2 * i))) & (uint64_t)BLS_INV_M62);
    o[6] = (int64_t)(w[5] >> 52);
}
// (f, g) <- t (f, g) / 2^62 (exact)
BLS_HD void inv_update_fg(int64_t* f, int64_t* g, const inv_mat& t) {
    __int128 cf = (__int128)t.u * f[0] + (__int128)t.v * g[0], cg = (__int128)t.q * f[0] + (__int128)t.r * g[0];
    cf >>= 62; cg >>= 62;
#pragma unroll
    for (int i = 1; i < 7; i++) {
        cf += (__int128)t.u * f[i] + (__int128)t.v * g[i]; cg += (__int128)t.q * f[i] + (__int128)t.r * g[i];
        f[i - 1] = (int64_t)cf & BLS_INV_M62; g[i - 1] = (int64_t)cg & BLS_INV_M62; cf >>= 62; cg >>= 62;
    }
    f[6] = (int64_t)cf; g[6] = (int64_t)cg;
}
// (d, e) <- t (d, e) / 2^62 mod p, both kept in (-2p, p): a multiple of p is added that clears the low 62 bits
BLS_HD void inv_update_de(int64_t* d, int64_t* e, const inv_mat& t, const int64_t* m) {
    int64_t sd = d[6] >> 63, se = e[6] >> 63;
    int64_t md = (t.u & sd) + (t.v & se), me = (t.q & sd) + (t.r & se);
    __int128 cd = (__int128)t.u * d[0] + (__int128)t.v * e[0], ce = (__int128)t.q * d[0] + (__int128)t.r * e[0];
    md -= (int64_t)((BLS_C_P_INV62 * (uint64_t)cd + (uint64_t)md) & (uint64_t)BLS_INV_M62);
    me -= (int64_t)((BLS_C_P_INV62 * (uint64_t)ce + (uint64_t)me) & (uint64_t)BLS_INV_M62);
    cd += (__int128)m[0] * md; ce += (__int128)m[0] * me;
    cd >>= 62; ce >>= 62;
#pragma unroll
    for (int i = 1; i < 7; i++) {
        cd += (__int128)t.u * d[i] + (__int128)t.v * e[i] + (__int128)m[i] * md; ce += (__int128)t.q * d[i] + (__int128)t.r * e[i] + (__int128)m[i] * me;
        d[i - 1] = (int64_t)cd & BLS_INV_M62; e[i - 1] = (int64_t)ce & BLS_INV_M62; cd >>= 62; ce >>= 62;
    }
    d[6] = (int64_t)cd; e[6] = (int64_t)ce;
}
// x^-1 mod p of the RAW limbs (no Montgomery factor involved; canonical in, canonical out); 0 -> 0
BLS_NOINLINE fp fp_inv_raw(const fp& x) {
    const uint32_t PL[12] = BLS_C_P;
    int64_t m[7], f[7], g[7], d[7], e[7];
    inv_to62(m, PL); inv_to62(g, x.l);
#pragma unroll
    for (int i = 0; i < 7; i++) { f[i] = m[i]; d[i] = 0; e[i] = 0; }
    e[0] = 1;
    int64_t eta = -1;
#pragma unroll 1
    for (int it = 0; it < 18; it++) {
        if ((g[0] | g[1] | g[2] | g[3] | g[4] | g[5] | g[6]) == 0) break;
        inv_mat t;
        eta = inv_divsteps62(eta, (uint64_t)f[0] | ((uint64_t)f[1] << 62), (uint64_t)g[0] | ((uint64_t)g[1] << 62), t);
        inv_update_de(d, e, t, m); inv_update_fg(f, g, t);
    }
    // f = +-gcd, d = +-x^-1 in (-2p, p): bring into (-p, p), apply the sign of f, bring into [0, p)
    int64_t ca = d[6] >> 63, cn = f[6] >> 63;
#pragma unroll
    for (int i = 0; i < 7; i++) { d[i] += m[i] & ca; d[i] = (d[i] ^ cn) - cn; }
#pragma unroll
    for (int i = 0; i < 6; i++) { d[i + 1] += d[i] >> 62; d[i] &= BLS_INV_M62; }
    ca = d[6] >> 63;
#pragma unroll
    for (int i = 0; i < 7; i++) d[i] += m[i] & ca;
#pragma unroll
    for (int i = 0; i < 6; i++) { d[i + 1] += d[i] >> 62; d[i] &= BLS_INV_M62; }
    uint64_t w[6];
#pragma unroll
    for (int i = 0; i < 6; i++) w[i] = ((uint64_t)d[i] >> (2 * i)) | ((uint64_t)d[i + 1] << (62 - 2 * i));
    fp r;
#pragma unroll
    for (int i = 0; i < 6; i++) { r.l[2 * i] = (uint32_t)w[i]; r.l[2 * i + 1] = (uint32_t)(w[i] >> 32); }
    return r;
}
// Montgomery form in and out: (aR)^-1 R^3 R^-1 = a^-1 R
BLS_HD fp fp_inv(const fp& a) {
    const uint32_t O[12] = BLS_C_R3; fp r3;
#pragma unroll
    for (int i = 0; i < 12; i++) r3.l[i] = O[i];
    return fp_mul(fp_inv_raw(a), r3);
}
// t = a^((p-3)/4).  Then a*t = a^((p+1)/4) is the candidate square root and (a*t)*t = a^((p-1)/2) the Legendre symbol.
BLS_HD fp fp_pow_pm3d4(const fp& a) { return fp_pow(a, EXP_P_MINUS_3_DIV_4, 12); }

// bytes: 48-byte big-endian canonical <-> Montgomery
BLS_HD bool fp_from_be48(fp& out, const uint8_t* b, uint32_t top_mask = 0xffu) {
    fp a;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        const uint8_t* q = b + 44 - 4 * i;
        uint32_t b0 = q[0]; if (i == 11) b0 &= top_mask;
        a.l[i] = (b0 << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
    }
    bool ok = !fp_raw_geq(a, fp_modulus());
    out = fp_to_mont(a);
    return ok;
}
BLS_HD void fp_canon_to_be48(uint8_t* b, const fp& a) {
#pragma unroll
    for (int i = 0; i < 12; i++) {
        uint8_t* q = b + 44 - 4 * i; uint32_t w = a.l[i];
        q[0] = (uint8_t)(w >> 24); q[1] = (uint8_t)(w >> 16); q[2] = (uint8_t)(w >> 8); q[3] = (uint8_t)w;
    }
}
// canonical "is a > (p-1)/2", i.e. a > -a as integers (a != 0): 2a > p
BLS_HD bool fp_canon_is_larger_half(const fp& a) {
    fp d; fp_add_raw(d, a, a);           // 2a < 2^382, no overflow
    fp t; return fp_sub_raw(t, fp_modulus(), d) != 0;     // p - 2a borrows <=> 2a > p
}

}  // namespace bls
