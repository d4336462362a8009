// Fp2 = Fp[u]/(u^2+1) on top of fp.cuh.  Values travel by value in registers (24 limbs); mul/sqr are
// out-of-line so the 300-IMAD Montgomery core exists once in the instruction cache.
// Replaces arkworks Fp2<Fq2Config> as used through reference src/bls.rs:443-455 and restated in-circuit at
// src/hasher.rs:352-548 (Fp2Var arithmetic).
#pragma once
#include "fp.cuh"

namespace bls {

struct fp2 { fp c0, c1; };

BLS_HD fp2 fp2_zero() { fp2 r; r.c0 = fp_zero(); r.c1 = fp_zero(); return r; }
BLS_HD fp2 fp2_one() { fp2 r; r.c0 = fp_one(); r.c1 = fp_zero(); return r; }
BLS_HD fp2 fp2_add(const fp2& a, const fp2& b) { fp2 r; r.c0 = fp_add(a.c0, b.c0); r.c1 = fp_add(a.c1, b.c1); return r; }
BLS_HD fp2 fp2_sub(const fp2& a, const fp2& b) { fp2 r; r.c0 = fp_sub(a.c0, b.c0); r.c1 = fp_sub(a.c1, b.c1); return r; }
BLS_HD fp2 fp2_dbl(const fp2& a) { return fp2_add(a, a); }
BLS_HD fp2 fp2_half(const fp2& a) { fp2 r; r.c0 = fp_half(a.c0); r.c1 = fp_half(a.c1); return r; }
BLS_HD fp2 fp2_neg(const fp2& a) { fp2 r; r.c0 = fp_neg(a.c0); r.c1 = fp_neg(a.c1); return r; }
BLS_HD fp2 fp2_conj(const fp2& a) { fp2 r; r.c0 = a.c0; r.c1 = fp_neg(a.c1); return r; }
BLS_HD fp2 fp2_mul_xi(const fp2& a) { fp2 r; r.c0 = fp_sub(a.c0, a.c1); r.c1 = fp_add(a.c0, a.c1); return r; }   // * (1+u)
BLS_HD fp2 fp2_mul_u(const fp2& a) { fp2 r; r.c0 = fp_neg(a.c1); r.c1 = a.c0; return r; }
BLS_HD bool fp2_is_zero(const fp2& a) { return fp_is_zero(a.c0) & fp_is_zero(a.c1); }
BLS_HD bool fp2_eq(const fp2& a, const fp2& b) { return fp_eq(a.c0, b.c0) & fp_eq(a.c1, b.c1); }
BLS_HD fp2 fp2_csel(bool c, const fp2& a, const fp2& b) { fp2 r; r.c0 = fp_csel(c, a.c0, b.c0); r.c1 = fp_csel(c, a.c1, b.c1); return r; }
// Operands and results by value, three (two) calls to the out-of-line fp_mul: measured faster on B200 than memory-to-memory
// operands, than inlined Montgomery products and than a lazily reduced Karatsuba form (profiles/r01_tuning.md).
BLS_NOINLINE fp2 fp2_mul(fp2 a, fp2 b) {                           // Karatsuba: 3 products
    fp t0 = fp_mul(a.c0, b.c0), t1 = fp_mul(a.c1, b.c1);
    fp t2 = fp_mul(fp_add(a.c0, a.c1), fp_add(b.c0, b.c1));
    fp2 r; r.c0 = fp_sub(t0, t1); r.c1 = fp_sub(t2, fp_add(t0, t1)); return r;
}
BLS_NOINLINE fp2 fp2_sqr(fp2 a) {                                  // 2 products
    fp t = fp_mul(a.c0, a.c1);
    fp2 r; r.c0 = fp_mul(fp_add(a.c0, a.c1), fp_sub(a.c0, a.c1)); r.c1 = fp_add(t, t); return r;
}
BLS_HD fp2 fp2_mul_fp(const fp2& a, const fp& s) { fp2 r; r.c0 = fp_mul(a.c0, s); r.c1 = fp_mul(a.c1, s); return r; }

BLS_HD fp fp2_norm(const fp2& a) { return fp_add(fp_sqr(a.c0), fp_sqr(a.c1)); }
BLS_HD fp2 fp2_inv(const fp2& a) {                            // 0 -> 0
    fp ni = fp_inv(fp2_norm(a));
    fp2 r; r.c0 = fp_mul(a.c0, ni); r.c1 = fp_neg(fp_mul(a.c1, ni)); return r;
}

BLS_HD fp fp_two_inv() { const uint32_t O[12] = BLS_C_TWO_INV; fp r;
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = O[i];
    return r; }

// Square root of a given s with s^2 = N(a) = a0^2 + a1^2 ("complex method", one Fp exponentiation).
// With d = (a0 + s)/2 and t = d^((p-3)/4):  x0 = d t satisfies x0^2 = +-d and 1/x0 = +-t, so
//   d residue     : sqrt(a) = (x0, a1 t / 2)
//   d non-residue : sqrt(a) = (-a1 t / 2, x0)
// Returns any one root; callers fix the sign.  The result is verified by squaring by the callers that need it.
BLS_HD fp2 fp2_sqrt_with_norm_root(const fp2& a, const fp& s) {
    fp half = fp_two_inv();
    fp d = fp_mul(fp_add(a.c0, s), half);
    if (fp_is_zero(d)) d = fp_mul(fp_sub(a.c0, s), half);      // s = -a0 (a1 = 0): use the other root of the norm
    fp t = fp_pow_pm3d4(d);
    fp x0 = fp_mul(d, t);
    fp w = fp_mul(fp_mul(a.c1, t), half);
    bool qr = fp_eq(fp_sqr(x0), d);
    fp2 r; r.c0 = fp_csel(qr, x0, fp_neg(w)); r.c1 = fp_csel(qr, w, x0); return r;
}
// full square root; false when a is a non-residue (out then holds garbage)
BLS_HD bool fp2_sqrt(fp2& out, const fp2& a) {
    fp n = fp2_norm(a);
    fp s = fp_mul(n, fp_pow_pm3d4(n));                         // n^((p+1)/4)
    out = fp2_sqrt_with_norm_root(a, s);
    return fp2_eq(fp2_sqr(out), a);
}

// sgn0 of RFC 9380 (reference src/hasher.rs:520-530) -- needs canonical integers
BLS_HD uint32_t fp2_sgn0(const fp2& a) {
    fp c0 = fp_from_mont(a.c0), c1 = fp_from_mont(a.c1);
    uint32_t s0 = c0.l[0] & 1, z0 = fp_is_zero(c0) ? 1u : 0u, s1 = c1.l[0] & 1;
    return s0 | (z0 & s1);
}
// ZCash "y is lexicographically largest": compare c1 first, then c0 (arkworks Fp2 ordering)
BLS_HD bool fp2_lex_largest(const fp2& y) {
    fp c1 = fp_from_mont(y.c1);
    if (!fp_is_zero(c1)) return fp_canon_is_larger_half(c1);
    return fp_canon_is_larger_half(fp_from_mont(y.c0));
}

}  // namespace bls
