// Fp6 = Fp2[v]/(v^3 - xi), xi = 1+u;  Fp12 = Fp6[w]/(w^2 - v)   (SURVEY A.2; arkworks Fq6Config / Fq12Config).
// Fp6/Fp12 values are too large for registers (72 / 144 limbs), so they live in per-thread local memory and
// every routine here is an out-of-line call on references; only Fp2 operands are staged in registers.
// Replaces the arkworks tower used by Bls12::multi_pairing (reference src/bls.rs:454-457).
#pragma once
#include "fp2.cuh"
#include "wide.cuh"

namespace bls {

struct fp6 { fp2 c0, c1, c2; };
struct fp12 { fp6 c0, c1; };

BLS_CONST fp2 FROB1[6] = BLS_C_FROB1;     // xi^(i(p-1)/6)
BLS_CONST fp FROB2[6] = BLS_C_FROB2;      // xi^(i(p^2-1)/6), in Fp

// Fp6 values live in local memory, so the linear operations on them are out-of-line memory-to-memory routines: inlined they are
// 3.5 KB each and made the Fp12 routines 20 KB+ apiece.
BLS_NOINLINE void fp6_add(fp6& r, const fp6& a, const fp6& b) {
    const fp* x = &a.c0.c0; const fp* y = &b.c0.c0; fp* z = &r.c0.c0;
#pragma unroll 1
    for (int i = 0; i < 6; i++) z[i] = fp_add(x[i], y[i]);
}
BLS_NOINLINE void fp6_sub(fp6& r, const fp6& a, const fp6& b) {
    const fp* x = &a.c0.c0; const fp* y = &b.c0.c0; fp* z = &r.c0.c0;
#pragma unroll 1
    for (int i = 0; i < 6; i++) z[i] = fp_sub(x[i], y[i]);
}
BLS_NOINLINE void fp6_neg(fp6& r, const fp6& a) {
    const fp* x = &a.c0.c0; fp* z = &r.c0.c0;
#pragma unroll 1
    for (int i = 0; i < 6; i++) z[i] = fp_neg(x[i]);
}
BLS_NOINLINE void fp6_mul_v(fp6& r, const fp6& a) { fp2 t = fp2_mul_xi(a.c2); fp2 u = a.c1, w = a.c0; r.c2 = u; r.c1 = w; r.c0 = t; }

// 6 Fp2 products (Karatsuba over the cubic extension): the three diagonal and the three cross products as two 3-iteration loops
// (one copy of each body: a third of the code; the instruction cache behind L0 holds 32 KB and the inlined form is 27 KB)
BLS_NOINLINE void fp6_mul(fp6& r, const fp6& a, const fp6& b) {
    const fp2* A = &a.c0; const fp2* B = &b.c0; fp2 v[3], t[3];
#pragma unroll 1
    for (int i = 0; i < 3; i++) v[i] = fp2_mul(A[i], B[i]);
#pragma unroll 1
    for (int k = 0; k < 3; k++) {                                  // (i, j) = (1, 2), (0, 1), (0, 2)
        int i = k == 0 ? 1 : 0, j = k == 1 ? 1 : 2;
        t[k] = fp2_sub(fp2_sub(fp2_mul(fp2_add(A[i], A[j]), fp2_add(B[i], B[j])), v[i]), v[j]);
    }
    r.c0 = fp2_add(v[0], fp2_mul_xi(t[0]));
    r.c1 = fp2_add(t[1], fp2_mul_xi(v[2]));
    r.c2 = fp2_add(t[2], v[1]);
}
// In the Miller loop the Fp6/Fp12 products are sums of Fp2 products accumulated UNREDUCED (wide.cuh) -- one Montgomery reduction
// per output coefficient, no conditional subtractions between the products, fewer Fp6 temporaries.  The final exponentiation keeps
// the separately reduced Karatsuba forms: measured faster there (profiles/r01_tuning.md).
// Schoolbook over the cubic extension, each output coefficient one 3-term dot product (27 wide products + 6 reductions =
// 4,824 IMAD.WIDE against 5,400 for six separately reduced Karatsuba products)
BLS_NOINLINE void fp6_mul_lz(fp6& r, const fp6& a, const fp6& b) {
    fp2 xb1 = fp2_mul_xi(b.c1), xb2 = fp2_mul_xi(b.c2);
    fp2 t0, t1, t2;
    fp2_dot3(t0, a.c0, b.c0, a.c1, xb2, a.c2, xb1);
    fp2_dot3(t1, a.c0, b.c1, a.c1, b.c0, a.c2, xb2);
    fp2_dot3(t2, a.c0, b.c2, a.c1, b.c1, a.c2, b.c0);
    r.c0 = t0; r.c1 = t1; r.c2 = t2;
}
BLS_NOINLINE void fp6_inv(fp6& r, const fp6& a) {
    fp2 t0 = fp2_sub(fp2_sqr(a.c0), fp2_mul_xi(fp2_mul(a.c1, a.c2)));
    fp2 t1 = fp2_sub(fp2_mul_xi(fp2_sqr(a.c2)), fp2_mul(a.c0, a.c1));
    fp2 t2 = fp2_sub(fp2_sqr(a.c1), fp2_mul(a.c0, a.c2));
    fp2 d = fp2_add(fp2_mul(a.c0, t0), fp2_mul_xi(fp2_add(fp2_mul(a.c2, t1), fp2_mul(a.c1, t2))));
    d = fp2_inv(d);
    r.c0 = fp2_mul(t0, d); r.c1 = fp2_mul(t1, d); r.c2 = fp2_mul(t2, d);
}

BLS_HD void fp12_one(fp12& r) {
    r.c0.c0 = fp2_one(); r.c0.c1 = fp2_zero(); r.c0.c2 = fp2_zero();
    r.c1.c0 = fp2_zero(); r.c1.c1 = fp2_zero(); r.c1.c2 = fp2_zero();
}
BLS_HD bool fp12_is_one(const fp12& a) {
    return fp2_eq(a.c0.c0, fp2_one()) & fp2_is_zero(a.c0.c1) & fp2_is_zero(a.c0.c2) &
           fp2_is_zero(a.c1.c0) & fp2_is_zero(a.c1.c1) & fp2_is_zero(a.c1.c2);
}
BLS_HD void fp12_conj(fp12& r, const fp12& a) { r.c0 = a.c0; fp6_neg(r.c1, a.c1); }

// 3 Fp6 products
BLS_NOINLINE void fp12_mul(fp12& r, const fp12& a, const fp12& b) {
    fp6 t0, t1, t2, s0, s1;
    fp6_mul(t0, a.c0, b.c0); fp6_mul(t1, a.c1, b.c1);
    fp6_add(s0, a.c0, a.c1); fp6_add(s1, b.c0, b.c1);
    fp6_mul(t2, s0, s1);
    fp6_sub(t2, t2, t0); fp6_sub(r.c1, t2, t1);
    fp6_mul_v(t1, t1); fp6_add(r.c0, t0, t1);
}
// complex squaring: 2 Fp6 products
BLS_NOINLINE void fp12_sqr(fp12& r, const fp12& a) {
    fp6 ab, s0, s1, t;
    fp6_mul_lz(ab, a.c0, a.c1);
    fp6_add(s0, a.c0, a.c1);
    fp6_mul_v(t, a.c1); fp6_add(s1, a.c0, t);
    fp6_mul_lz(s0, s0, s1);                   // (a0+a1)(a0+v a1) = a0^2 + v a1^2 + (1+v) a0a1
    fp6_sub(s0, s0, ab); fp6_mul_v(t, ab); fp6_sub(r.c0, s0, t);
    fp6_add(r.c1, ab, ab);
}
// f * (c0 + c1 v + c4 v w): the sparse line element of the M-type twist (arkworks mul_by_014).
// In the basis 1, w, .., w^5 (w^2 = v, w^6 = xi) f = sum g_k w^k with g = (c0.c0, c1.c0, c0.c1, c1.c1, c0.c2, c1.c2) and the
// line is l0 + l2 w^2 + l3 w^3: out_k = g_k l0 + g_{k-2} l2 + g_{k-3} l3, indices mod 6, wrapped terms times xi (folded
// into the line coefficient).  Six 3-term dot products: 9,648 IMAD.WIDE against 11,700, and no Fp6 temporaries.
BLS_NOINLINE void fp12_mul_by_014(fp12& f, const fp2& c0, const fp2& c1, const fp2& c4) {
    fp2 l0 = c0, l2 = c1, l3 = c4, xl2 = fp2_mul_xi(c1), xl3 = fp2_mul_xi(c4);
    fp2 o0, o1, o2, o3, o4, o5;
    fp2_dot3(o0, f.c0.c0, l0, f.c0.c2, xl2, f.c1.c1, xl3);
    fp2_dot3(o1, f.c1.c0, l0, f.c1.c2, xl2, f.c0.c2, xl3);
    fp2_dot3(o2, f.c0.c1, l0, f.c0.c0, l2, f.c1.c2, xl3);
    fp2_dot3(o3, f.c1.c1, l0, f.c1.c0, l2, f.c0.c0, l3);
    fp2_dot3(o4, f.c0.c2, l0, f.c0.c1, l2, f.c1.c0, l3);
    fp2_dot3(o5, f.c1.c2, l0, f.c1.c1, l2, f.c0.c1, l3);
    f.c0.c0 = o0; f.c1.c0 = o1; f.c0.c1 = o2; f.c1.c1 = o3; f.c0.c2 = o4; f.c1.c2 = o5;
}
BLS_NOINLINE void fp12_inv(fp12& r, const fp12& a) {
    fp6 t0, t1;
    fp6_mul(t0, a.c0, a.c0); fp6_mul(t1, a.c1, a.c1); fp6_mul_v(t1, t1); fp6_sub(t0, t0, t1);
    fp6_inv(t0, t0);
    fp6_mul(r.c0, a.c0, t0); fp6_mul(t1, a.c1, t0); fp6_neg(r.c1, t1);
}
// a^p
BLS_NOINLINE void fp12_frob(fp12& r, const fp12& a) {
    r.c0.c0 = fp2_conj(a.c0.c0);
    r.c1.c0 = fp2_mul(fp2_conj(a.c1.c0), FROB1[1]);
    r.c0.c1 = fp2_mul(fp2_conj(a.c0.c1), FROB1[2]);
    r.c1.c1 = fp2_mul(fp2_conj(a.c1.c1), FROB1[3]);
    r.c0.c2 = fp2_mul(fp2_conj(a.c0.c2), FROB1[4]);
    r.c1.c2 = fp2_mul(fp2_conj(a.c1.c2), FROB1[5]);
}
// a^(p^2)
BLS_NOINLINE void fp12_frob2(fp12& r, const fp12& a) {
    r.c0.c0 = a.c0.c0;
    r.c1.c0 = fp2_mul_fp(a.c1.c0, FROB2[1]);
    r.c0.c1 = fp2_mul_fp(a.c0.c1, FROB2[2]);
    r.c1.c1 = fp2_mul_fp(a.c1.c1, FROB2[3]);
    r.c0.c2 = fp2_mul_fp(a.c0.c2, FROB2[4]);
    r.c1.c2 = fp2_mul_fp(a.c1.c2, FROB2[5]);
}
// Granger-Scott squaring for elements of the cyclotomic subgroup (after the easy part): 3 Fp4 squarings.
// Inlined three / six times the routine is 52 KB and nearly half of its stall samples are `no_instruction` (32 KB instruction
// cache behind L0).  So ONE copy of the Fp4 squaring and of the two combinations sits inside a 3-iteration loop over the
// coefficient pairs (20 KB, operands indexed in the thread's local memory where they live anyway): final exponentiation
// 442 -> 423 ms at 2^20.  Out-of-line helpers with operands and results by value measured +5.6 % (argument marshalling), with
// operands by reference +25 % (local-memory round trips).  profiles/r01_tuning.md
BLS_NOINLINE void fp12_cyclo_sqr(fp12& r, const fp12& a) {
    const fp2* A = &a.c0.c0; fp12 out; fp2* R = &out.c0.c0;           // tower order: c0.c0 c0.c1 c0.c2 c1.c0 c1.c1 c1.c2
#pragma unroll 1
    for (int p = 0; p < 3; p++) {
        int ia = p == 0 ? 0 : (p == 1 ? 3 : 1), ib = p == 0 ? 4 : (p == 1 ? 2 : 5), oe = p, oo = p == 0 ? 4 : (p == 1 ? 5 : 3);
        fp2 x = A[ia], y = A[ib];
        fp2 ab = fp2_mul(x, y);
        fp2 s = fp2_mul(fp2_add(x, y), fp2_add(x, fp2_mul_xi(y)));
        fp2 te = fp2_sub(fp2_sub(s, ab), fp2_mul_xi(ab)), to = fp2_dbl(ab);
        if (p == 2) to = fp2_mul_xi(to);
        fp2 z = fp2_sub(te, A[oe]); z = fp2_dbl(z); R[oe] = fp2_add(z, te);
        z = fp2_add(to, A[oo]); z = fp2_dbl(z); R[oo] = fp2_add(z, to);
    }
    r = out;
}

}  // namespace bls
