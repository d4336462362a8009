// Optimal-ate pairing check for e(-g1, sig) * e(pk, H(m)) == 1.
// Replaces Bls12::<P>::multi_pairing + PairingOutput.0.is_one() at reference src/bls.rs:454-457 (arkworks
// ark-ec models::bls12: G2 line coefficients in homogeneous projective coordinates, M-type twist, sparse
// mul_by_014, final exponentiation f^(3(p^12-1)/r) with the x-chain of eprint 2020/875).  SURVEY A.8.
//
// B200-first: the reference materialises 68 line-coefficient triples per G2 point (19.6 KB) before the loop;
// here each line is produced and consumed in the same iteration, so a thread's working set is f (576 B) plus
// two running G2 points (2 x 288 B) and stays L1-resident.  Both pairs share the accumulator f.
#pragma once
#include "tower.cuh"
#include "curve.cuh"

namespace bls {

struct g2_proj { fp2 x, y, z; };          // homogeneous projective running point of the Miller loop

// doubling step: R <- 2R, line coefficients (c0, c1, c2) for mul_by_014(c0, c1*px, c2*py)
BLS_NOINLINE void miller_dbl(g2_proj& r, fp2& c0, fp2& c1, fp2& c2) {
    fp2 a = fp2_half(fp2_mul(r.x, r.y));                    // ark-ec multiplies by 1/2; halving is ALU-only and gives the same element
    fp2 b = fp2_sqr(r.y), c = fp2_sqr(r.z);
    fp2 c3 = fp2_add(fp2_dbl(c), c);
    fp2 e = fp2_mul_xi(fp2_dbl(fp2_dbl(c3)));               // 4(1+u) * 3c
    fp2 f = fp2_add(fp2_dbl(e), e);
    fp2 g = fp2_half(fp2_add(b, f));
    fp2 h = fp2_sub(fp2_sqr(fp2_add(r.y, r.z)), fp2_add(b, c));
    fp2 i = fp2_sub(e, b);
    fp2 j = fp2_sqr(r.x);
    fp2 es = fp2_sqr(e);
    r.x = fp2_mul(a, fp2_sub(b, f));
    r.y = fp2_sub(fp2_sqr(g), fp2_add(fp2_dbl(es), es));
    r.z = fp2_mul(b, h);
    c0 = i; c1 = fp2_add(fp2_dbl(j), j); c2 = fp2_neg(h);
}
// addition step: R <- R + Q (Q affine)
BLS_NOINLINE void miller_add(g2_proj& r, const g2_aff& q, fp2& c0, fp2& c1, fp2& c2) {
    fp2 theta = fp2_sub(r.y, fp2_mul(q.y, r.z));
    fp2 lambda = fp2_sub(r.x, fp2_mul(q.x, r.z));
    fp2 c = fp2_sqr(theta), d = fp2_sqr(lambda);
    fp2 e = fp2_mul(lambda, d), f = fp2_mul(r.z, c), g = fp2_mul(r.x, d);
    fp2 h = fp2_sub(fp2_add(e, f), fp2_dbl(g));
    r.x = fp2_mul(lambda, h);
    r.y = fp2_sub(fp2_mul(theta, fp2_sub(g, h)), fp2_mul(e, r.y));
    r.z = fp2_mul(r.z, e);
    c0 = fp2_sub(fp2_mul(theta, q.x), fp2_mul(lambda, q.y)); c1 = fp2_neg(theta); c2 = lambda;
}
// Subgroup test of a signature on the running point its pair leaves at the end of the Miller loop.  The pair (-g1, sig) runs
// R <- 2R (+ sig) over bits 62..0 of |x| from R = sig: the double-and-add of [|x|] sig.  The test accepts iff Z != 0 and
// (X/Z, Y/Z) = -psi(sig), which is g2_in_subgroup's condition [|x|] sig = -psi(sig).  It is exact for every finite point sig on
// the curve, with nothing tracked beside R, because of the two formulas above (homogeneous projective: affine (X/Z, Y/Z)):
//  * miller_dbl: Z3 = b h = Y^2 (2 Y Z) = 2 Y^3 Z.  With Z != 0 and Y != 0 it is the tangent doubling: every output is homogeneous of
//    degree 4 in (X, Y, Z), and at Z = 1, with b' = 4(1+u) and y^2 = x^3 + b', X3/Z3 = x (y^2 - 9b') / (4y^2) = l^2 - 2x and
//    Y3/Z3 = (y^4 + 18b'y^2 - 27b'^2) / (8y^3) = l (x - X3/Z3) - y for l = 3x^2 / (2y); and Z3 != 0.  Y = 0 (a point of order 2)
//    or Z = 0 gives Z3 = 0.
//  * miller_add: Z3 = Z e = Z l^3 with l = X - q.x Z.  With Z != 0 and l != 0 (R != +-Q) it is the chord addition (degree 4 again; at
//    Z = 1, X3/Z3 = t^2/l^2 - x - q.x and Y3/Z3 = (t/l)(x - X3/Z3) - y for t = Y - q.y) and Z3 != 0.  l = 0 (R = +-Q) or Z = 0 gives Z3 = 0.
// Z = 0 stays 0 whatever X and Y hold, since both formulas multiply Z into Z3.  By induction over the 63 doublings and 5 additions:
// either no step was exceptional and R = [|x|] sig with Z != 0, or one was and Z = 0 at the end.
//  * sig in G2 (prime order r): before a doubling R = [k] sig with 2 <= 2k <= |x|, so Y = 0 would mean [2k] sig = O; before an
//    addition R = [k] sig with k even, 2 <= k < |x|, so R = +-sig would mean [k -+ 1] sig = O with 1 <= k -+ 1 <= |x|.  |x| < r rules
//    all of them out: Z != 0, R = [|x|] sig, and R = -psi(sig) holds in G2.  Accepted, as g2_in_subgroup accepts.
//  * sig not in G2: with no exceptional step the comparison is g2_in_subgroup's on the same point, so the answers agree (rejected);
//    after an exceptional step Z = 0 and the test rejects, which is again g2_in_subgroup's answer, since it accepts G2 points only.
// The Z != 0 test and the comparisons come after all arithmetic and are combined without a branch (DESIGN "ptxas and carry chains").
BLS_NOINLINE bool miller_end_in_subgroup(const g2_proj& r, const g2_aff& sig) {
    g2_jac sj, ps; jac_from_aff(sj, sig); g2_psi(ps, sj);                // Z = 1: psi(sig) affine
    fp2 px = fp2_mul(ps.X, r.z), py = fp2_mul(ps.Y, r.z);
    return !fp2_is_zero(r.z) & fp2_eq(r.x, px) & fp2_eq(fp2_neg(r.y), py);
}
BLS_HD void miller_ell(fp12& f, const fp2& c0, const fp2& c1, const fp2& c2, const g1_aff& p) {
    fp12_mul_by_014(f, c0, fp2_mul_fp(c1, p.x), fp2_mul_fp(c2, p.y));
}
// Shared-accumulator Miller loop over up to two pairs; a pair with use == false is skipped
// (ark-ec drops pairs that contain the identity).
BLS_NOINLINE void miller_loop2(fp12& f, const g1_aff& p0, const g2_aff& q0, bool use0, const g1_aff& p1, const g2_aff& q1, bool use1) {
    g2_proj r0, r1;
    r0.x = q0.x; r0.y = q0.y; r0.z = fp2_one();
    r1.x = q1.x; r1.y = q1.y; r1.z = fp2_one();
    fp12_one(f);
    fp2 c0, c1, c2;
    const uint64_t x = BLS_X_ABS;
    for (int i = 62; i >= 0; i--) {
        if (i != 62) fp12_sqr(f, f);
        if (use0) { miller_dbl(r0, c0, c1, c2); miller_ell(f, c0, c1, c2, p0); }
        if (use1) { miller_dbl(r1, c0, c1, c2); miller_ell(f, c0, c1, c2, p1); }
        if ((x >> i) & 1) {
            if (use0) { miller_add(r0, q0, c0, c1, c2); miller_ell(f, c0, c1, c2, p0); }
            if (use1) { miller_add(r1, q1, c0, c1, c2); miller_ell(f, c0, c1, c2, p1); }
        }
    }
    fp12_conj(f, f);                                        // x < 0
}

// a^x for a in the cyclotomic subgroup (x negative: conjugate at the end): square-and-multiply with Granger-Scott squarings (18 Fp
// products each).  Kept as the reference form of the compressed version below (tests/devcheck op 39 compares them).
BLS_NOINLINE void fp12_exp_by_x_gs(fp12& r, const fp12& a) {
    fp12 acc = a;
    const uint64_t x = BLS_X_ABS;
    for (int i = 62; i >= 0; i--) {
        fp12_cyclo_sqr(acc, acc);
        if ((x >> i) & 1) fp12_mul(acc, acc, a);
    }
    fp12_conj(r, acc);
}
// ---- Karabina's compressed squaring (eprint 2010/542) in the arkworks tower.  With s = v w (s^2 = xi) an element is
//   (g0 + g1 s) + (g2 + g3 s) w + (g4 + g5 s) w^2,   g0 = c0.c0, g1 = c1.c1, g2 = c1.c0, g3 = c0.c2, g4 = c0.c1, g5 = c1.c2
// and the Granger-Scott update of (g2, g3, g4, g5) reads only those four coefficients: a squaring of the COMPRESSED form is two Fp4
// squarings (12 Fp products) instead of three (18).  g1 and g0 come back from the cyclotomic relations
//   g1 = (g5^2 xi + 3 g4^2 - 2 g3) / (4 g2)      [ g2 = 0:  g1 = 2 g4 g5 / g3,  and g1 = 0 when g3 = 0 too (the element 1) ]
//   g0 = (2 g1^2 + g2 g5 - 3 g3 g4) xi + 1
// with ONE inversion for all the elements that are decompressed together.  |x| = 2^63 + 2^62 + 2^60 + 2^57 + 2^48 + 2^16, so
// a^|x| = prod a^(2^i) over those six i: 63 compressed squarings with six snapshots, one simultaneous decompression, five products --
// 756 + ~220 Fp products for the squaring part instead of 1,134.  Same group element, hence the same canonical bytes.
struct fp12c { fp2 g2, g3, g4, g5; };
BLS_HD void fp12_compress(fp12c& c, const fp12& a) { c.g2 = a.c1.c0; c.g3 = a.c0.c2; c.g4 = a.c0.c1; c.g5 = a.c1.c2; }
BLS_NOINLINE void fp12c_sqr(fp12c& r, const fp12c& a) {
    fp12c o;
    {   // (t2, t3) = (g2 + g3 s)^2:  g4' = 3 t2 - 2 g4,  g5' = 3 t3 + 2 g5
        fp2 ab = fp2_mul(a.g2, a.g3);
        fp2 sm = fp2_mul(fp2_add(a.g2, a.g3), fp2_add(a.g2, fp2_mul_xi(a.g3)));
        fp2 te = fp2_sub(fp2_sub(sm, ab), fp2_mul_xi(ab)), to = fp2_dbl(ab);
        fp2 z = fp2_sub(te, a.g4); z = fp2_dbl(z); o.g4 = fp2_add(z, te);
        z = fp2_add(to, a.g5); z = fp2_dbl(z); o.g5 = fp2_add(z, to);
    }
    {   // (t4, t5) = (g4 + g5 s)^2:  g3' = 3 t4 - 2 g3,  g2' = 3 xi t5 + 2 g2
        fp2 ab = fp2_mul(a.g4, a.g5);
        fp2 sm = fp2_mul(fp2_add(a.g4, a.g5), fp2_add(a.g4, fp2_mul_xi(a.g5)));
        fp2 te = fp2_sub(fp2_sub(sm, ab), fp2_mul_xi(ab)), to = fp2_mul_xi(fp2_dbl(ab));
        fp2 z = fp2_sub(te, a.g3); z = fp2_dbl(z); o.g3 = fp2_add(z, te);
        z = fp2_add(to, a.g2); z = fp2_dbl(z); o.g2 = fp2_add(z, to);
    }
    r = o;
}
// numerator and denominator of g1 (see above); the rare g2 = 0 branch is taken per thread
BLS_HD void fp12c_g1_fraction(fp2& num, fp2& den, const fp12c& c) {
    if (!fp2_is_zero(c.g2)) {
        fp2 t = fp2_sqr(c.g4);
        num = fp2_sub(fp2_add(fp2_mul_xi(fp2_sqr(c.g5)), fp2_add(fp2_dbl(t), t)), fp2_dbl(c.g3));
        den = fp2_dbl(fp2_dbl(c.g2));
    } else {
        num = fp2_dbl(fp2_mul(c.g4, c.g5));
        den = fp2_is_zero(c.g3) ? fp2_one() : c.g3;
    }
}
BLS_HD void fp12_decompress_with(fp12& r, const fp12c& c, const fp2& g1) {
    fp2 t = fp2_sub(fp2_add(fp2_dbl(fp2_sqr(g1)), fp2_mul(c.g2, c.g5)), fp2_mul(c.g3, c.g4));
    fp2 u = fp2_mul(c.g3, c.g4); t = fp2_sub(t, fp2_dbl(u));                                  // 2 g1^2 + g2 g5 - 3 g3 g4
    r.c0.c0 = fp2_add(fp2_mul_xi(t), fp2_one()); r.c1.c1 = g1; r.c1.c0 = c.g2; r.c0.c2 = c.g3; r.c0.c1 = c.g4; r.c1.c2 = c.g5;
}
// r = prod of the decompressed c[0..n), n <= 6, one Fp2 inversion (Montgomery's trick over the denominators)
BLS_NOINLINE void fp12_decompress_product(fp12& r, const fp12c* c, int n) {
    fp2 num[6], den[6], pre[6];
    for (int i = 0; i < n; i++) { fp12c_g1_fraction(num[i], den[i], c[i]); pre[i] = i ? fp2_mul(pre[i - 1], den[i]) : den[i]; }
    fp2 inv = fp2_inv(pre[n - 1]);                            // denominators are never zero
    fp12 acc, d;
    for (int i = n - 1; i >= 0; i--) {
        fp2 di = i ? fp2_mul(inv, pre[i - 1]) : inv;          // 1 / den[i]
        if (i) inv = fp2_mul(inv, den[i]);
        fp12_decompress_with(d, c[i], fp2_mul(num[i], di));
        if (i == n - 1) acc = d; else fp12_mul(acc, acc, d);
    }
    r = acc;
}
// the same with the snapshots fetched through `load(i)` when they are needed (twice each) instead of sitting in a local array: the split
// final-exponentiation kernels read them from global memory, which keeps 2.3 KB per thread out of the L1-backed stack
template <class LOAD> BLS_HD void fp12_decompress_product_from(fp12& r, LOAD load, int n) {
    fp2 num[6], den[6], pre[6];
    for (int i = 0; i < n; i++) { fp12c c = load(i); fp12c_g1_fraction(num[i], den[i], c); pre[i] = i ? fp2_mul(pre[i - 1], den[i]) : den[i]; }
    fp2 inv = fp2_inv(pre[n - 1]);
    fp12 acc, d;
    for (int i = n - 1; i >= 0; i--) {
        fp2 di = i ? fp2_mul(inv, pre[i - 1]) : inv;
        if (i) inv = fp2_mul(inv, den[i]);
        fp12c c = load(i);
        fp12_decompress_with(d, c, fp2_mul(num[i], di));
        if (i == n - 1) acc = d; else fp12_mul(acc, acc, d);
    }
    r = acc;
}
BLS_NOINLINE void fp12_exp_by_x(fp12& r, const fp12& a) {
    fp12c c, snap[6]; fp12_compress(c, a);
    const uint64_t x = BLS_X_ABS; int k = 0;
    for (int i = 1; i <= 63; i++) {
        fp12c_sqr(c, c);
        if ((x >> i) & 1) snap[k++] = c;                      // i = 16, 48, 57, 60, 62, 63
    }
    fp12 acc; fp12_decompress_product(acc, snap, 6);
    fp12_conj(r, acc);
}
// f^(3 (p^12 - 1)/r): the exact chain of ark-ec's Bls12::final_exponentiation
BLS_NOINLINE void final_exponentiation(fp12& r, const fp12& f) {
    fp12 t, y0, y1, y2;
    fp12_conj(t, f); fp12_inv(y0, f); fp12_mul(r, t, y0);            // f^(p^6 - 1)
    fp12_frob2(t, r); fp12_mul(r, t, r);                             // ^(p^2 + 1)
    fp12_cyclo_sqr(y0, r);
    fp12_exp_by_x(y1, r);
    fp12_conj(y2, r);
    fp12_mul(y1, y1, y2);
    fp12_exp_by_x(y2, y1);
    fp12_conj(y1, y1);
    fp12_mul(y1, y1, y2);
    fp12_exp_by_x(y2, y1);
    fp12_frob(y1, y1);
    fp12_mul(y1, y1, y2);
    fp12_mul(r, r, y0);
    fp12_exp_by_x(y0, y1);
    fp12_exp_by_x(y2, y0);
    fp12_frob2(y0, y1);
    fp12_conj(y1, y1);
    fp12_mul(y1, y1, y2);
    fp12_mul(y1, y1, y0);
    fp12_mul(r, r, y1);
}

// The same chain for the split stage kernels (k_final_squarings / k_final_step in blsgpu.cu): every exp_by_x is a launch of the 63 compressed
// squarings alone (a 4-coefficient state and one small loop body) that leaves its six snapshots in global memory, followed by a launch that
// decompresses them and does the products up to the next exp_by_x.  y0 = r^2 of the one-launch form is recomputed where it is used.
// STEP 0: easy part (r -> r).  STEP k = 1..5: e = the k-th exp_by_x result (decompressed product of its snapshots, conjugated), then the
// products that follow it in the chain.  The next exp_by_x runs on: r after step 0, y1 after steps 1..3, y2 after step 4.
template <int STEP> BLS_HD void final_exponentiation_step(fp12& r, fp12& y1, fp12& y2, const fp12& e) {
    if (STEP == 0) {
        fp12 t, y0;
        fp12_conj(t, r); fp12_inv(y0, r); fp12_mul(r, t, y0);
        fp12_frob2(t, r); fp12_mul(r, t, r);
    } else if (STEP == 1) {
        fp12_conj(y2, r);
        fp12_mul(y1, e, y2);
    } else if (STEP == 2) {
        fp12_conj(y1, y1);
        fp12_mul(y1, y1, e);
    } else if (STEP == 3) {
        fp12_frob(y1, y1);
        fp12_mul(y1, y1, e);
        fp12 y0; fp12_cyclo_sqr(y0, r); fp12_mul(r, r, y0);
    } else if (STEP == 4) {
        y2 = e;
    } else {
        fp12 y0;
        fp12_frob2(y0, y1);
        fp12_conj(y1, y1);
        fp12_mul(y1, y1, e);
        fp12_mul(y1, y1, y0);
        fp12_mul(r, r, y1);
    }
}

// GT wire format: 12 x 48 bytes little-endian canonical, tower order c0.c0.c0 ... c1.c2.c1 (SURVEY A.7)
BLS_HD void fp_to_le48(uint8_t* b, const fp& m) {
    fp a = fp_from_mont(m);
    for (int i = 0; i < 12; i++) { uint32_t w = a.l[i]; b[4 * i] = (uint8_t)w; b[4 * i + 1] = (uint8_t)(w >> 8); b[4 * i + 2] = (uint8_t)(w >> 16); b[4 * i + 3] = (uint8_t)(w >> 24); }
}
BLS_HD void fp12_to_bytes(uint8_t* out, const fp12& a) {
    const fp2* c[6] = {&a.c0.c0, &a.c0.c1, &a.c0.c2, &a.c1.c0, &a.c1.c1, &a.c1.c2};
    for (int i = 0; i < 6; i++) { fp_to_le48(out + 96 * i, c[i]->c0); fp_to_le48(out + 96 * i + 48, c[i]->c1); }
}

}  // namespace bls
