// Single-operation harness shared by the host-emulation build (tests/hostemu) and the device unit-test library
// (tests/devcheck): run_op applies ONE device-library primitive to raw Montgomery limb images, so every layer of the
// CUDA path can be compared host-vs-device (and against big-int arithmetic) in isolation.  TEST TOOL ONLY.
#pragma once
#include "stages.cuh"
#include "wide.cuh"
namespace bls {
struct op_desc { int n_in, n_out; };
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline op_desc op_shape(int op) {
    switch (op) {
        case 1: return {4, 2};    // fp2_mul
        case 2: return {2, 2};    // fp2_sqr
        case 3: return {4, 2};    // fp2_add
        case 4: return {4, 2};    // fp2_sub
        case 5: return {6, 6};    // jac_dbl<fp2>
        case 6: return {10, 6};   // jac_add_mixed<fp2>(jac, aff)
        case 7: return {12, 6};   // jac_add<fp2>
        case 8: return {12, 6};   // fp6_mul
        case 9: return {24, 12};  // fp12_mul
        case 10: return {12, 12}; // fp12_sqr
        case 11: return {18, 12}; // fp12_mul_by_014(f, c0, c1, c4)
        case 12: return {12, 12}; // fp12_cyclo_sqr
        case 13: return {12, 12}; // fp12_inv
        case 14: return {12, 12}; // fp12_frob
        case 15: return {12, 12}; // fp12_frob2
        case 16: return {2, 3};   // fp2_sqrt -> root, ok flag in out[2].l[0]
        case 17: return {2, 2};   // fp2_inv
        case 18: return {3, 3};   // jac_dbl<fp>
        case 19: return {5, 3};   // jac_add_mixed<fp>
        case 20: return {6, 3};   // jac_add<fp>
        case 21: return {2, 1};   // fp_mul
        case 22: return {1, 1};   // fp_inv
        case 35: return {2, 1};   // fp_mul_small(z, low word of the second input)
        case 37: return {12, 24}; // cyclotomic g = easy part of the input: decompress(compress(g)) beside g (Karabina relations)
        case 38: return {12, 24}; // decompress(compressed squaring of g) beside fp12_cyclo_sqr(g)
        case 39: return {12, 24}; // fp12_exp_by_x (compressed squarings) beside fp12_exp_by_x_gs
        case 40: return {12, 24}; // final exponentiation as the split stage kernels run it (easy part, 5 x (63 compressed squarings | decompression from the snapshots + products)) beside final_exponentiation
        case 41: return {12, 24}; // Miller loop of two pairs as the split stage runs it (8 iterations at a time: scaled line coefficients of each pair, then the accumulator update) beside miller_loop2; inputs (p0.x, p0.y, q0, p1.x, p1.y, q1) need not be curve points
        case 36: return {8, 1};   // lazy 14-limb sum: 8 x (c0 z0 + c1 z1 + c2 z2 + c3 (p - z3)), c_i = low word of inputs 4..7, one reduction (fp_lacc_*)
        case 34: return {1, 2};   // fp_inv (divsteps) beside fp_inv_fermat
        case 23: return {4, 6};   // jac_mul_x_abs<fp2>(aff)
        case 24: return {12, 12}; // final_exponentiation
        case 25: return {4, 3};   // fp2_sqrt_ratio(u, v) -> y, is_sq
        case 26: return {2, 2};   // fp2_mul_xi
        case 27: return {3, 2};   // fp2_mul_fp
        case 28: return {10, 6};  // jac_add_mixed<fp2>, separate output
        case 29: return {2, 1};   // fp_redc_wide(fp_mul_wide(a, b)) == fp_mul
        case 30: return {4, 2};   // lazy-reduction fp2 product (3 wide products, 2 reductions)
        case 31: return {2, 1};   // fp_mul_lz (split wide accumulator + reduction) == fp_mul
        case 32: return {4, 2};   // fp2_dot, n = 1 == fp2_mul
        case 33: return {12, 2};  // fp2_dot, n = 3 == x0 y0 + x1 y1 + x2 y2
        case 42: return {2, 6};   // sswu_map(u) -> xn, xd, y
        case 43: return {6, 6};   // iso3_map(xn, xd, y) -> Jacobian X, Y, Z
        case 44: return {6, 6};   // g2_clear_cofactor(Jacobian P)
        case 45: return {2, 3};   // fp2_sgn0(a), fp2_lex_largest(a), fp_canon_is_larger_half(a.c0), each 0/1 in the low word
        case 46: return {1, 2};   // Fp square root as g1_decode takes it: a * a^((p-3)/4), and y^2 == a in out[1].l[0]
        default: return {0, 0};
    }
}
BLS_HD void ld2(fp2& r, const fp* in) { r.c0 = in[0]; r.c1 = in[1]; }
BLS_HD void st2(fp* out, const fp2& a) { out[0] = a.c0; out[1] = a.c1; }
BLS_HD void ld12(fp12& f, const fp* in) { ld2(f.c0.c0, in); ld2(f.c0.c1, in + 2); ld2(f.c0.c2, in + 4); ld2(f.c1.c0, in + 6); ld2(f.c1.c1, in + 8); ld2(f.c1.c2, in + 10); }
BLS_HD void st12(fp* out, const fp12& f) { st2(out, f.c0.c0); st2(out + 2, f.c0.c1); st2(out + 4, f.c0.c2); st2(out + 6, f.c1.c0); st2(out + 8, f.c1.c1); st2(out + 10, f.c1.c2); }
BLS_HD void run_op(int op, const fp* in, fp* out) {
    fp2 a, b, c, d; fp12 f, g, h; g2_jac P, Q, R; g2_aff A; g1_jac p1, q1, r1; g1_aff a1;
    switch (op) {
        case 1: ld2(a, in); ld2(b, in + 2); st2(out, fp2_mul(a, b)); break;
        case 2: ld2(a, in); st2(out, fp2_sqr(a)); break;
        case 3: ld2(a, in); ld2(b, in + 2); st2(out, fp2_add(a, b)); break;
        case 4: ld2(a, in); ld2(b, in + 2); st2(out, fp2_sub(a, b)); break;
        case 5: ld2(P.X, in); ld2(P.Y, in + 2); ld2(P.Z, in + 4); jac_dbl(P, P); st2(out, P.X); st2(out + 2, P.Y); st2(out + 4, P.Z); break;
        case 6: ld2(P.X, in); ld2(P.Y, in + 2); ld2(P.Z, in + 4); ld2(A.x, in + 6); ld2(A.y, in + 8); jac_add_mixed(P, P, A); st2(out, P.X); st2(out + 2, P.Y); st2(out + 4, P.Z); break;
        case 7: ld2(P.X, in); ld2(P.Y, in + 2); ld2(P.Z, in + 4); ld2(Q.X, in + 6); ld2(Q.Y, in + 8); ld2(Q.Z, in + 10); jac_add(R, P, Q); st2(out, R.X); st2(out + 2, R.Y); st2(out + 4, R.Z); break;
        case 8: { fp6 x, y, z; ld2(x.c0, in); ld2(x.c1, in + 2); ld2(x.c2, in + 4); ld2(y.c0, in + 6); ld2(y.c1, in + 8); ld2(y.c2, in + 10); fp6_mul(z, x, y); st2(out, z.c0); st2(out + 2, z.c1); st2(out + 4, z.c2); break; }
        case 9: ld12(f, in); ld12(g, in + 12); fp12_mul(h, f, g); st12(out, h); break;
        case 10: ld12(f, in); fp12_sqr(f, f); st12(out, f); break;
        case 11: ld12(f, in); ld2(a, in + 12); ld2(b, in + 14); ld2(c, in + 16); fp12_mul_by_014(f, a, b, c); st12(out, f); break;
        case 12: ld12(f, in); fp12_cyclo_sqr(f, f); st12(out, f); break;
        case 13: ld12(f, in); fp12_inv(g, f); st12(out, g); break;
        case 14: ld12(f, in); fp12_frob(g, f); st12(out, g); break;
        case 15: ld12(f, in); fp12_frob2(g, f); st12(out, g); break;
        case 16: { ld2(a, in); bool ok = fp2_sqrt(b, a); st2(out, b); out[2] = fp_zero(); out[2].l[0] = ok ? 1u : 0u; break; }
        case 17: ld2(a, in); st2(out, fp2_inv(a)); break;
        case 18: p1.X = in[0]; p1.Y = in[1]; p1.Z = in[2]; jac_dbl(p1, p1); out[0] = p1.X; out[1] = p1.Y; out[2] = p1.Z; break;
        case 19: p1.X = in[0]; p1.Y = in[1]; p1.Z = in[2]; a1.x = in[3]; a1.y = in[4]; jac_add_mixed(p1, p1, a1); out[0] = p1.X; out[1] = p1.Y; out[2] = p1.Z; break;
        case 20: p1.X = in[0]; p1.Y = in[1]; p1.Z = in[2]; q1.X = in[3]; q1.Y = in[4]; q1.Z = in[5]; jac_add(r1, p1, q1); out[0] = r1.X; out[1] = r1.Y; out[2] = r1.Z; break;
        case 21: out[0] = fp_mul(in[0], in[1]); break;
        case 22: out[0] = fp_inv(in[0]); break;
        case 23: ld2(A.x, in); ld2(A.y, in + 2); jac_mul_x_abs(P, A); st2(out, P.X); st2(out + 2, P.Y); st2(out + 4, P.Z); break;
        case 24: ld12(f, in); final_exponentiation(g, f); st12(out, g); break;
        case 25: { ld2(a, in); ld2(b, in + 2); bool sq = fp2_sqrt_ratio(c, a, b); st2(out, c); out[2] = fp_zero(); out[2].l[0] = sq ? 1u : 0u; break; }
        case 26: ld2(a, in); st2(out, fp2_mul_xi(a)); break;
        case 27: ld2(a, in); st2(out, fp2_mul_fp(a, in[2])); break;
        case 28: ld2(P.X, in); ld2(P.Y, in + 2); ld2(P.Z, in + 4); ld2(A.x, in + 6); ld2(A.y, in + 8); jac_add_mixed(R, P, A); st2(out, R.X); st2(out + 2, R.Y); st2(out + 4, R.Z); break;
        case 29: { fpw T; fp_mul_wide(T, in[0], in[1]); out[0] = fp_redc_wide(T); break; }
        case 30: { fpw T0, T1, T2; fp_mul_wide(T0, in[0], in[2]); fp_mul_wide(T1, in[1], in[3]); fp sa, sb; fp_add_raw(sa, in[0], in[1]); fp_add_raw(sb, in[2], in[3]);
                   fp_mul_wide(T2, sa, sb); fpw_sub(T2, T2, T0); fpw_sub(T2, T2, T1); fpw_sub(T0, T0, T1); fpw_add(T0, T0, fpw_p_squared());
                   out[0] = fp_redc_wide(T0); out[1] = fp_redc_wide(T2); break; }
        case 31: out[0] = fp_mul_lz(in[0], in[1]); break;
        case 32: ld2(a, in); ld2(b, in + 2); fp2_dot1(c, a, b); st2(out, c); break;
        case 33: { fp2 x0, y0, x1, y1, x2, y2; ld2(x0, in); ld2(y0, in + 2); ld2(x1, in + 4); ld2(y1, in + 6); ld2(x2, in + 8); ld2(y2, in + 10); fp2_dot3(c, x0, y0, x1, y1, x2, y2); st2(out, c); break; }
        case 35: out[0] = fp_mul_small(in[0], in[1].l[0]); break;
        case 37: case 38: case 39: {
            ld12(f, in); fp12 t, e; fp12_conj(t, f); fp12_inv(e, f); fp12_mul(e, t, e); fp12_frob2(t, e); fp12_mul(g, t, e);      // g = f^((p^6-1)(p^2+1)): cyclotomic
            if (op == 37) { fp12c cc; fp12_compress(cc, g); fp12_decompress_product(h, &cc, 1); st12(out, h); st12(out + 12, g); }
            else if (op == 38) { fp12c cc; fp12_compress(cc, g); fp12c_sqr(cc, cc); fp12_decompress_product(h, &cc, 1); st12(out, h); fp12_cyclo_sqr(t, g); st12(out + 12, t); }
            else { fp12_exp_by_x(h, g); st12(out, h); fp12_exp_by_x_gs(t, g); st12(out + 12, t); }
            break; }
        case 40: {
            ld12(f, in); fp12 r = f, y1, y2, e; fp12c snap[6];
            auto run = [&](const fp12& a) { fp12c cc; fp12_compress(cc, a); int k = 0; for (int i = 1; i <= 63; i++) { fp12c_sqr(cc, cc); if ((BLS_X_ABS >> i) & 1) snap[k++] = cc; } };   // k_final_squarings
            auto fin = [&](fp12& x) { fp12_decompress_product_from(x, [&](int k) { return snap[k]; }, 6); fp12_conj(x, x); };                                                        // head of k_final_step<1..5>
            final_exponentiation_step<0>(r, y1, y2, e);
            run(r); fin(e); final_exponentiation_step<1>(r, y1, y2, e);
            run(y1); fin(e); final_exponentiation_step<2>(r, y1, y2, e);
            run(y1); fin(e); final_exponentiation_step<3>(r, y1, y2, e);
            run(y1); fin(e); final_exponentiation_step<4>(r, y1, y2, e);
            run(y2); fin(e); final_exponentiation_step<5>(r, y1, y2, e);
            st12(out, r); final_exponentiation(h, f); st12(out + 12, h);
            break; }
        case 41: {
            g1_aff p[2]; g2_aff q[2]; p[0].x = in[0]; p[0].y = in[1]; ld2(q[0].x, in + 2); ld2(q[0].y, in + 4); p[1].x = in[6]; p[1].y = in[7]; ld2(q[1].x, in + 8); ld2(q[1].y, in + 10);
            g2_proj r[2]; fp2 line[11][2][3]; fp2 c0, c1, c2; const uint64_t xx = BLS_X_ABS;
            for (int j = 0; j < 2; j++) { r[j].x = q[j].x; r[j].y = q[j].y; r[j].z = fp2_one(); }
            fp12_one(f);
            for (int hi = 62; hi >= 0; hi -= 8) {
                int lo = hi - 7 < 0 ? 0 : hi - 7;
                for (int j = 0; j < 2; j++) {                                                     // k_miller_lines: one pair per thread
                    int s = 0;
                    for (int it = hi; it >= lo; it--) {
                        miller_dbl(r[j], c0, c1, c2); line[s][j][0] = c0; line[s][j][1] = fp2_mul_fp(c1, p[j].x); line[s][j][2] = fp2_mul_fp(c2, p[j].y); s++;
                        if ((xx >> it) & 1) { miller_add(r[j], q[j], c0, c1, c2); line[s][j][0] = c0; line[s][j][1] = fp2_mul_fp(c1, p[j].x); line[s][j][2] = fp2_mul_fp(c2, p[j].y); s++; }
                    }
                }
                int s = 0;                                                                        // k_miller_accum
                for (int it = hi; it >= lo; it--) {
                    if (it != 62) fp12_sqr(f, f);
                    int steps = 1 + (int)((xx >> it) & 1);
                    for (int a2 = 0; a2 < steps; a2++, s++) for (int j = 0; j < 2; j++) fp12_mul_by_014(f, line[s][j][0], line[s][j][1], line[s][j][2]);
                }
            }
            fp12_conj(f, f); st12(out, f);
            miller_loop2(g, p[0], q[0], true, p[1], q[1], true); st12(out + 12, g);
            break; }
        case 36: { fp_lacc a; fp_lacc_zero(a); fp nz; fp_sub_raw(nz, fp_modulus(), in[3]);
                   for (int k = 0; k < 8; k++) { fp_lacc_mad(a, in[0], in[4].l[0]); fp_lacc_mad(a, in[1], in[5].l[0]); fp_lacc_mad(a, in[2], in[6].l[0]); fp_lacc_mad(a, nz, in[7].l[0]); }
                   out[0] = fp_lacc_reduce(a); break; }
        case 34: out[0] = fp_inv(in[0]); out[1] = fp_inv_fermat(in[0]); break;
        case 42: ld2(a, in); sswu_map(b, c, d, a); st2(out, b); st2(out + 2, c); st2(out + 4, d); break;
        case 43: ld2(a, in); ld2(b, in + 2); ld2(c, in + 4); iso3_map(P, a, b, c); st2(out, P.X); st2(out + 2, P.Y); st2(out + 4, P.Z); break;
        case 44: ld2(P.X, in); ld2(P.Y, in + 2); ld2(P.Z, in + 4); g2_clear_cofactor(Q, P); st2(out, Q.X); st2(out + 2, Q.Y); st2(out + 4, Q.Z); break;
        case 45: ld2(a, in); out[0] = fp_zero(); out[1] = fp_zero(); out[2] = fp_zero();
                 out[0].l[0] = fp2_sgn0(a); out[1].l[0] = fp2_lex_largest(a) ? 1u : 0u; out[2].l[0] = fp_canon_is_larger_half(fp_from_mont(a.c0)) ? 1u : 0u; break;
        case 46: { fp y = fp_mul(in[0], fp_pow_pm3d4(in[0])); out[0] = y; out[1] = fp_zero(); out[1].l[0] = fp_eq(fp_sqr(y), in[0]) ? 1u : 0u; break; }
        default: break;
    }
    (void)d;
}
}  // namespace bls
