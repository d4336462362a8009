// G1: y^2 = x^3 + 4 over Fp;  G2: y^2 = x^3 + 4(1+u) over Fp2.  Jacobian coordinates (Z = 0 is the identity),
// complete formulas (every exceptional case handled: adversarial inputs reach these through the decoders),
// ZCash compressed codec, and the endomorphism-based subgroup tests.
// Replaces: PublicKey/Signature TryFrom + check() (reference src/bls.rs:219-223, 316-320, 438, 443),
//           Into<Vec<u8>> (bls.rs:254-260, 351-357), aggregate (bls.rs:183-195, 288-300),
//           PublicKey::from(&sk) / sign's scalar mul (bls.rs:210-216, 420-422).
#pragma once
#include "fp2.cuh"

namespace bls {

// ---- field-generic helpers
BLS_HD fp  f_add(const fp& a, const fp& b) { return fp_add(a, b); }
BLS_HD fp2 f_add(const fp2& a, const fp2& b) { return fp2_add(a, b); }
BLS_HD fp  f_sub(const fp& a, const fp& b) { return fp_sub(a, b); }
BLS_HD fp2 f_sub(const fp2& a, const fp2& b) { return fp2_sub(a, b); }
BLS_HD fp  f_mul(const fp& a, const fp& b) { return fp_mul(a, b); }
BLS_HD fp2 f_mul(const fp2& a, const fp2& b) { return fp2_mul(a, b); }
BLS_HD fp  f_sqr(const fp& a) { return fp_sqr(a); }
BLS_HD fp2 f_sqr(const fp2& a) { return fp2_sqr(a); }
BLS_HD fp  f_neg(const fp& a) { return fp_neg(a); }
BLS_HD fp2 f_neg(const fp2& a) { return fp2_neg(a); }
BLS_HD fp  f_inv(const fp& a) { return fp_inv(a); }
BLS_HD fp2 f_inv(const fp2& a) { return fp2_inv(a); }
BLS_HD bool f_is_zero(const fp& a) { return fp_is_zero(a); }
BLS_HD bool f_is_zero(const fp2& a) { return fp2_is_zero(a); }
BLS_HD bool f_eq(const fp& a, const fp& b) { return fp_eq(a, b); }
BLS_HD bool f_eq(const fp2& a, const fp2& b) { return fp2_eq(a, b); }
BLS_HD void f_set_one(fp& a) { a = fp_one(); }
BLS_HD void f_set_one(fp2& a) { a = fp2_one(); }
BLS_HD void f_set_zero(fp& a) { a = fp_zero(); }
BLS_HD void f_set_zero(fp2& a) { a = fp2_zero(); }

template <class F> struct aff { F x, y; };       // identity is carried separately (flag) by the callers
template <class F> struct jac { F X, Y, Z; };
typedef aff<fp> g1_aff;  typedef jac<fp> g1_jac;
typedef aff<fp2> g2_aff; typedef jac<fp2> g2_jac;

template <class F> BLS_HD void jac_set_identity(jac<F>& r) { f_set_one(r.X); f_set_one(r.Y); f_set_zero(r.Z); }
template <class F> BLS_HD bool jac_is_identity(const jac<F>& p) { return f_is_zero(p.Z); }
template <class F> BLS_HD void jac_from_aff(jac<F>& r, const aff<F>& a) { r.X = a.x; r.Y = a.y; f_set_one(r.Z); }
template <class F> BLS_HD void jac_neg(jac<F>& r, const jac<F>& p) { r.X = p.X; r.Y = f_neg(p.Y); r.Z = p.Z; }

// dbl-2009-l (a = 0): 2M + 5S.  Z3 = 2 Y1 Z1, so the identity and 2-torsion map to the identity.
template <class F> BLS_NOINLINE void jac_dbl(jac<F>& r, const jac<F>& p) {
    F A = f_sqr(p.X), B = f_sqr(p.Y), C = f_sqr(B);
    F D = f_sub(f_sub(f_sqr(f_add(p.X, B)), A), C); D = f_add(D, D);
    F E = f_add(f_add(A, A), A), G = f_sqr(E);
    F Z3 = f_mul(p.Y, p.Z); Z3 = f_add(Z3, Z3);
    F X3 = f_sub(G, f_add(D, D));
    F C8 = f_add(C, C); C8 = f_add(C8, C8); C8 = f_add(C8, C8);
    r.Y = f_sub(f_mul(E, f_sub(D, X3)), C8); r.X = X3; r.Z = Z3;
}
// r = p + q, q affine (never the identity).  madd-2007-bl: 7M + 4S, plus the exceptional cases.
// The exceptional-case test is taken only after all arithmetic (no arithmetic follows the branch): ptxas 12.9 was seen
// to miscompile the carry chains it sank across an `if (H == 0) return` placed in the middle (tests/devcheck op 6).
template <class F> BLS_NOINLINE void jac_add_mixed(jac<F>& r, const jac<F>& p, const aff<F>& q) {
    if (f_is_zero(p.Z)) { jac_from_aff(r, q); return; }
    F Z1Z1 = f_sqr(p.Z), U2 = f_mul(q.x, Z1Z1), S2 = f_mul(f_mul(q.y, p.Z), Z1Z1);
    F H = f_sub(U2, p.X), rr = f_sub(S2, p.Y);
    bool h_zero = f_is_zero(H), r_zero = f_is_zero(rr);
    rr = f_add(rr, rr);
    F HH = f_sqr(H), I = f_add(HH, HH); I = f_add(I, I);
    F J = f_mul(H, I), V = f_mul(p.X, I);
    F X3 = f_sub(f_sub(f_sqr(rr), J), f_add(V, V));
    F YJ = f_mul(p.Y, J);
    F Z3 = f_sub(f_sub(f_sqr(f_add(p.Z, H)), Z1Z1), HH);
    F Y3 = f_sub(f_mul(rr, f_sub(V, X3)), f_add(YJ, YJ));
    if (h_zero) {                                          // p == +-q
        if (r_zero) { jac<F> t; jac_from_aff(t, q); jac_dbl(r, t); } else jac_set_identity(r);
    } else { r.X = X3; r.Y = Y3; r.Z = Z3; }
}
// r = p + q, both Jacobian.  add-2007-bl: 11M + 5S, plus the exceptional cases (tested after the arithmetic, as above).
template <class F> BLS_NOINLINE void jac_add(jac<F>& r, const jac<F>& p, const jac<F>& q) {
    if (f_is_zero(p.Z)) { r = q; return; }
    if (f_is_zero(q.Z)) { r = p; return; }
    F Z1Z1 = f_sqr(p.Z), Z2Z2 = f_sqr(q.Z);
    F U1 = f_mul(p.X, Z2Z2), U2 = f_mul(q.X, Z1Z1);
    F S1 = f_mul(f_mul(p.Y, q.Z), Z2Z2), S2 = f_mul(f_mul(q.Y, p.Z), Z1Z1);
    F H = f_sub(U2, U1), rr = f_sub(S2, S1);
    bool h_zero = f_is_zero(H), r_zero = f_is_zero(rr);
    rr = f_add(rr, rr);
    F I = f_add(H, H); I = f_sqr(I);
    F J = f_mul(H, I), V = f_mul(U1, I);
    F X3 = f_sub(f_sub(f_sqr(rr), J), f_add(V, V));
    F SJ = f_mul(S1, J);
    F Z3 = f_mul(f_sub(f_sub(f_sqr(f_add(p.Z, q.Z)), Z1Z1), Z2Z2), H);
    F Y3 = f_sub(f_mul(rr, f_sub(V, X3)), f_add(SJ, SJ));
    if (h_zero) {
        if (r_zero) { jac<F> t = p; jac_dbl(r, t); } else jac_set_identity(r);
    } else { r.X = X3; r.Y = Y3; r.Z = Z3; }
}
// Jacobian -> affine; returns false for the identity
template <class F> BLS_HD bool jac_to_aff(aff<F>& a, const jac<F>& p) {
    if (f_is_zero(p.Z)) { f_set_zero(a.x); f_set_zero(a.y); return false; }
    F zi = f_inv(p.Z), zi2 = f_sqr(zi);
    a.x = f_mul(p.X, zi2); a.y = f_mul(p.Y, f_mul(zi2, zi));
    return true;
}
// p == q with q affine (non-identity)
template <class F> BLS_HD bool jac_eq_aff(const jac<F>& p, const aff<F>& q) {
    if (f_is_zero(p.Z)) return false;
    F zz = f_sqr(p.Z);
    return f_eq(p.X, f_mul(q.x, zz)) & f_eq(p.Y, f_mul(q.y, f_mul(zz, p.Z)));
}
// [|x|] p for the BLS parameter |x| = 0xd201000000010000 (double-and-add, p affine)
template <class F> BLS_HD void jac_mul_x_abs(jac<F>& r, const aff<F>& p) {
    jac_from_aff(r, p);
    const uint64_t x = BLS_X_ABS;
    for (int i = 62; i >= 0; i--) {
        jac_dbl(r, r);
        if ((x >> i) & 1) jac_add_mixed(r, r, p);
    }
}
template <class F> BLS_HD void jac_mul_x_abs_j(jac<F>& r, const jac<F>& p) {
    const jac<F> base = p;                       // r may alias p
    r = base;
    const uint64_t x = BLS_X_ABS;
    for (int i = 62; i >= 0; i--) {
        jac_dbl(r, r);
        if ((x >> i) & 1) jac_add(r, r, base);
    }
}
// [k] p, k = 256-bit little-endian scalar in 8 words (double-and-add, MSB first)
template <class F> BLS_HD void jac_mul_scalar(jac<F>& r, const aff<F>& p, const uint32_t* k) {
    jac_set_identity(r);
    for (int i = 255; i >= 0; i--) {
        jac_dbl(r, r);
        if ((k[i >> 5] >> (i & 31)) & 1) jac_add_mixed(r, r, p);
    }
}

// ------------------------------------------------------------------------------------------------ constants
BLS_HD fp fp_const(const uint32_t (&w)[12]) { fp r;
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = w[i];
    return r; }
BLS_CONST uint32_t C_BETA[12] = BLS_C_BETA;
BLS_CONST uint32_t C_FOUR[12] = BLS_C_FOUR;
BLS_CONST uint32_t C_G1X[12] = BLS_C_G1X;
BLS_CONST uint32_t C_G1Y[12] = BLS_C_G1Y;
BLS_CONST uint32_t C_G1Y_NEG[12] = BLS_C_G1Y_NEG;
BLS_CONST fp2 C_PSI_X = BLS_C_PSI_X;
BLS_CONST fp2 C_PSI_Y = BLS_C_PSI_Y;
BLS_CONST uint32_t C_PSI2_X[12] = BLS_C_PSI2_X;

BLS_HD fp g1_b() { return fp_const(C_FOUR); }
BLS_HD fp2 g2_b() { fp2 r; r.c0 = fp_const(C_FOUR); r.c1 = r.c0; return r; }

// psi(x, y) = (PSI_X conj(x), PSI_Y conj(y)) on Jacobian coordinates (Z -> conj(Z));  hasher.rs:600-616
BLS_HD void g2_psi(g2_jac& r, const g2_jac& p) {
    r.X = fp2_mul(fp2_conj(p.X), C_PSI_X); r.Y = fp2_mul(fp2_conj(p.Y), C_PSI_Y); r.Z = fp2_conj(p.Z);
}
// psi^2(x, y) = (PSI2_X x, -y)
BLS_HD void g2_psi2(g2_jac& r, const g2_jac& p) {
    r.X = fp2_mul_fp(p.X, fp_const(C_PSI2_X)); r.Y = fp2_neg(p.Y); r.Z = p.Z;
}

// Subgroup tests (functionally equal to [r]P == O; Scott, eprint 2021/1130, the forms ark-bls12-381 uses)
// G1: sigma(P) = (beta x, y) must equal -[x^2]P
BLS_HD bool g1_in_subgroup(const g1_aff& p) {
    g1_jac t; jac_mul_x_abs(t, p);                       // [|x|]P
    g1_jac t2; jac_mul_x_abs_j(t2, t);                   // [x^2]P
    g1_aff s; s.x = fp_mul(p.x, fp_const(C_BETA)); s.y = fp_neg(p.y);     // -sigma(P)
    return jac_eq_aff(t2, s);
}
// G2: psi(P) must equal [x]P = -[|x|]P
BLS_HD bool g2_in_subgroup(const g2_aff& p) {
    g2_jac t; jac_mul_x_abs(t, p);
    g2_jac pj; jac_from_aff(pj, p);
    g2_jac ps; g2_psi(ps, pj);                           // Z = 1 -> affine
    g2_aff s; s.x = ps.X; s.y = fp2_neg(ps.Y);           // -psi(P)
    return jac_eq_aff(t, s);
}

// ------------------------------------------------------------------------------------------------ ZCash compressed codec
// decode status
enum { DEC_OK = 0, DEC_INF = 1, DEC_BAD_FLAGS = 2, DEC_RANGE = 3, DEC_NOT_ON_CURVE = 4, DEC_NOT_IN_SUBGROUP = 5 };

// 48 bytes -> affine G1 (Montgomery).  Identity: returns DEC_INF.  Lenient on the infinity encoding like
// ark-bls12-381 0.4 (SURVEY B7).  Subgroup membership is checked (deserialize_compressed = Validate::Yes).
BLS_HD int g1_decode(g1_aff& out, const uint8_t* b) {
    uint32_t flags = b[0];
    out.x = fp_zero(); out.y = fp_zero();
    if (!(flags & 0x80)) return DEC_BAD_FLAGS;
    if (flags & 0x40) return DEC_INF;
    fp x; if (!fp_from_be48(x, b, 0x1f)) return DEC_RANGE;
    fp y2 = fp_add(fp_mul(fp_sqr(x), x), g1_b());
    fp y = fp_mul(y2, fp_pow_pm3d4(y2));                  // y2^((p+1)/4)
    if (!fp_eq(fp_sqr(y), y2)) return DEC_NOT_ON_CURVE;
    bool larger = fp_canon_is_larger_half(fp_from_mont(y));
    if (larger != ((flags & 0x20) != 0)) y = fp_neg(y);
    out.x = x; out.y = y;
    if (!g1_in_subgroup(out)) return DEC_NOT_IN_SUBGROUP;
    return DEC_OK;
}
BLS_HD void g1_encode(uint8_t* b, const g1_aff& a, bool inf) {
    if (inf) { for (int i = 0; i < 48; i++) b[i] = 0; b[0] = 0xc0; return; }
    fp_canon_to_be48(b, fp_from_mont(a.x));
    b[0] |= 0x80; if (fp_canon_is_larger_half(fp_from_mont(a.y))) b[0] |= 0x20;
}
// 96 bytes (x.c1 || x.c0, big-endian) -> affine G2.  SUBGROUP = false stops after the square root: DEC_OK then means "a point on
// the curve", and the caller owes the membership test (the split Miller loop of blsgpu_verify_batch does it, miller_end_in_subgroup).
template <bool SUBGROUP = true> BLS_HD int g2_decode(g2_aff& out, const uint8_t* b) {
    uint32_t flags = b[0];
    out.x = fp2_zero(); out.y = fp2_zero();
    if (!(flags & 0x80)) return DEC_BAD_FLAGS;
    if (flags & 0x40) return DEC_INF;
    fp2 x; bool ok1 = fp_from_be48(x.c1, b, 0x1f); bool ok0 = fp_from_be48(x.c0, b + 48);
    if (!(ok0 & ok1)) return DEC_RANGE;
    fp2 y2 = fp2_add(fp2_mul(fp2_sqr(x), x), g2_b());
    fp2 y; if (!fp2_sqrt(y, y2)) return DEC_NOT_ON_CURVE;
    if (fp2_lex_largest(y) != ((flags & 0x20) != 0)) y = fp2_neg(y);
    out.x = x; out.y = y;
    if (SUBGROUP && !g2_in_subgroup(out)) return DEC_NOT_IN_SUBGROUP;
    return DEC_OK;
}
BLS_HD void g2_encode(uint8_t* b, const g2_aff& a, bool inf) {
    if (inf) { for (int i = 0; i < 96; i++) b[i] = 0; b[0] = 0xc0; return; }
    fp_canon_to_be48(b, fp_from_mont(a.x.c1)); fp_canon_to_be48(b + 48, fp_from_mont(a.x.c0));
    b[0] |= 0x80; if (fp2_lex_largest(a.y)) b[0] |= 0x20;
}

// ------------------------------------------------------------------------------------------------ ZCash uncompressed codec
// 96 bytes x || y (G1) and 192 bytes x.c1 || x.c0 || y.c1 || y.c0 (G2), big-endian; first byte: bit 7 (compression) must be clear, bit 6 =
// infinity (rest ignored, lenient like the compressed form: SURVEY B7), bit 5 is ignored like ark-bls12-381 0.4's read_g1_uncompressed.
// The other wire format of the upstream bls12-381-tests suite (reference tests/readme.md:4-7); validation = on-curve + subgroup
// (deserialize_uncompressed = Validate::Yes).  Not pinned by a reference fixture (the reference vendors no uncompressed vectors).
BLS_HD int g1_decode_uncompressed(g1_aff& out, const uint8_t* b) {
    uint32_t flags = b[0];
    out.x = fp_zero(); out.y = fp_zero();
    if (flags & 0x80) return DEC_BAD_FLAGS;
    if (flags & 0x40) return DEC_INF;
    fp x, y; bool okx = fp_from_be48(x, b, 0x1f), oky = fp_from_be48(y, b + 48);
    if (!(okx & oky)) return DEC_RANGE;
    if (!fp_eq(fp_sqr(y), fp_add(fp_mul(fp_sqr(x), x), g1_b()))) return DEC_NOT_ON_CURVE;
    out.x = x; out.y = y;
    if (!g1_in_subgroup(out)) return DEC_NOT_IN_SUBGROUP;
    return DEC_OK;
}
BLS_HD void g1_encode_uncompressed(uint8_t* b, const g1_aff& a, bool inf) {
    if (inf) { for (int i = 0; i < 96; i++) b[i] = 0; b[0] = 0x40; return; }
    fp_canon_to_be48(b, fp_from_mont(a.x)); fp_canon_to_be48(b + 48, fp_from_mont(a.y));
}
BLS_HD int g2_decode_uncompressed(g2_aff& out, const uint8_t* b) {
    uint32_t flags = b[0];
    out.x = fp2_zero(); out.y = fp2_zero();
    if (flags & 0x80) return DEC_BAD_FLAGS;
    if (flags & 0x40) return DEC_INF;
    fp2 x, y; bool ok = fp_from_be48(x.c1, b, 0x1f); ok &= fp_from_be48(x.c0, b + 48); ok &= fp_from_be48(y.c1, b + 96); ok &= fp_from_be48(y.c0, b + 144);
    if (!ok) return DEC_RANGE;
    if (!fp2_eq(fp2_sqr(y), fp2_add(fp2_mul(fp2_sqr(x), x), g2_b()))) return DEC_NOT_ON_CURVE;
    out.x = x; out.y = y;
    if (!g2_in_subgroup(out)) return DEC_NOT_IN_SUBGROUP;
    return DEC_OK;
}
BLS_HD void g2_encode_uncompressed(uint8_t* b, const g2_aff& a, bool inf) {
    if (inf) { for (int i = 0; i < 192; i++) b[i] = 0; b[0] = 0x40; return; }
    fp_canon_to_be48(b, fp_from_mont(a.x.c1)); fp_canon_to_be48(b + 48, fp_from_mont(a.x.c0));
    fp_canon_to_be48(b + 96, fp_from_mont(a.y.c1)); fp_canon_to_be48(b + 144, fp_from_mont(a.y.c0));
}

}  // namespace bls
