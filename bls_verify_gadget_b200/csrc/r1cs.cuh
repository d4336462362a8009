// K8: R1CS satisfaction check  (A z) o (B z) == C z  over Fq (the BLS12-381 base field, the constraint field of
// the reference's circuits: src/constraints.rs:18, src/hasher.rs:32), as three CSR sparse mat-vecs.
// Replaces ark-relations' ConstraintSystem::is_satisfied applied to the system synthesised by
// BlsSignatureVerifyGadget::verify (src/constraints.rs:90-128); unlike arkworks' serial early-exit loop every row
// is reported.  Included at the end of blsgpu.cu (same translation unit: one copy of the Fp core).
//
// Mapping: lane <-> witness, warp <-> R1_ROWS (8) consecutive rows, OR-ed into the 64-row word.  All lanes of a warp walk the same CSR row, so column
// indices and coefficients are warp-uniform broadcast loads and the only divergent traffic is the gather of z,
// which is coalesced by transposing each group of 32 witnesses to  uint4 [col][3][32]  first.
//
// What the real verify circuit (714 k rows, built by bls_verify_gadget_b200/gadget) needed beyond the synthetic one:
//  * 93 % of its columns are boolean variables (SHA-256 bits) and 40 % of its "general" coefficients (powers of two of the
//    bit-packing rows) multiply such a column: the transpose packs a column that is 0/1 in all 32 witnesses into one word
//    (+ a flag); the row kernels read that word instead of gathering 1.5 KB, add +-1 / small coefficients into a 64-bit integer
//    side sum, a larger coefficient as a masked addition of its canonical value (warp-uniform branches), and test a row that
//    touched nothing else as a * b == c on integers;
//  * a few hundred rows carry 300-760 general coefficients (linear combinations that grow through runs of cyclotomic
//    squarings).  Round 1 cut rows longer than R1_LONG into 32-entry segments, one warp each, and combined them afterwards
//    (with the round-1 term code a 760-term row serialised ~10^7 instructions on one warp: 34 ms per group).  With the term paths of
//    round 2 a term costs ~70 warp instructions, and the long rows run one warp per ROW, longest first (k_r1cs_long_rows):
//    no partial sums through global memory, one closing reduction per combination instead of one per segment -- 651 -> 506 us per
//    group for the 21,537 long rows of the verify circuit.
// Coefficients +1 / -1 (the bulk of boolean/uint gadget rows) skip the multiply; coefficients of magnitude below 2^32 (2, 3, 4, 12,
// 2^k ...: 80 % of the remaining ones in the verify circuit) take fp_mul_small (24 MACs); z stays canonical:
// coeff(Montgomery) x z(canonical) -> canonical, no conversion of z needed.
#pragma once
#include <algorithm>
#include <vector>

struct r1cs_sys {
    size_t nrows, ncols, nnz[3];
    uint64_t* rowptr[3]; uint32_t* col[3]; fp* coeff[3]; fp* coeffc[3]; uint8_t* cls[3];
    size_t n_long;
    size_t n_rounds;               // 32-term metadata rounds k_r1cs_long_rows walks: sum over long rows and matrices of ceil(nnz / 32)
    uint32_t* long_sorted;         // [n_long] long rows, longest first (k_r1cs_long_rows takes them in this order: longest-processing-time-first over the warps)
    // rows specialised at load time (see "row classes" below)
    uint4* lut_a; uint2* lut_b;    // [nrows] truth-table rows: (col0 | need_b << 31, col1, col2, table) and (col3, col4); col0 = R1_NOT_LUT for other rows
    uint32_t* gen_rows; size_t n_gen, n_lut;     // short rows that are evaluated term by term (lane = assignment)
    uint32_t* fb_rows; uint32_t* fb_count;       // truth-table rows that met a non-0/1 column in the current group: evaluated generically afterwards
};
enum { R1_GENERAL = 0, R1_PLUS_ONE = 1, R1_MINUS_ONE = 2, R1_SMALL_POS = 3, R1_SMALL_NEG = 4 };      // SMALL: |c| < 2^32 (fp_mul_small), c = +|c| or p - |c|
#define R1_GROUP 32
#ifndef R1_LONG
#define R1_LONG 8          // rows that are not truth-table rows and have more non-zeros than this take the lane-parallel metadata path (k_r1cs_long_rows);
#endif                     // measured on the verify circuit: 16 -> 3.67 ms per 128 assignments, 8 / 4 / 2 -> 3.54 / 3.55 / 3.54
// The row kernels are bound by the latency of the z gather (1.5 KB per non-zero and 32 witnesses, from HBM: a group's
// transposed z is 1 GB), not by registers: more resident warps than the pairing kernels' 8 per SM
#ifndef R1_MINB
#define R1_MINB 6
#endif

// coefficient -> Montgomery image (for general z), canonical copy (for 0/1-valued z) and class byte
__global__ void __launch_bounds__(TPB, BLS_MINB) k_r1cs_prepare(const uint8_t* coeff48, size_t nnz, fp* out, fp* outc, uint8_t* cls) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= nnz) return;
    fp v; const uint8_t* b = coeff48 + 48 * i;
    for (int w = 0; w < 12; w++) v.l[w] = b[4 * w] | ((uint32_t)b[4 * w + 1] << 8) | ((uint32_t)b[4 * w + 2] << 16) | ((uint32_t)b[4 * w + 3] << 24);
    fp one = fp_zero(); one.l[0] = 1;
    fp m1; fp_sub_raw(m1, fp_modulus(), one);
    fp nv; fp_sub_raw(nv, fp_modulus(), v);                      // p - v
    uint32_t hi = 0, nhi = 0;
    for (int w = 1; w < 12; w++) { hi |= v.l[w]; nhi |= nv.l[w]; }
    cls[i] = fp_eq(v, one) ? R1_PLUS_ONE : fp_eq(v, m1) ? R1_MINUS_ONE : !hi ? R1_SMALL_POS : !nhi ? R1_SMALL_NEG : R1_GENERAL;
    out[i] = fp_to_mont(v); outc[i] = v;
}
// z[w][col] (48-byte LE canonical) for witnesses w0 .. w0+g-1  ->  zt[(col*3 + c)*32 + lane];
// zbool[col] = (bits of the 32 witnesses, 1) when the column is 0/1-valued in every witness of the group, else (0, 0): such a column
// (bits, bytes and words of the SHA-256 / decomposition gadgets: most non-zeros of the circuit) is then read as ONE broadcast 8-byte
// load instead of a 1.5 KB gather, and its +-1 / small coefficients accumulate in a 64-bit integer beside the field accumulator
// Tiled through shared memory: a CTA takes R1_TT consecutive columns of the 32 assignments.  Phase 1 reads, per assignment, the
// R1_TT * 48 contiguous bytes of its row (coalesced 16-byte loads; the direct form -- each lane fetching 48 bytes from rows 34 MB
// apart -- ran at half of the HBM rate); phase 2 hands each column to a warp, lane = assignment, which writes the three 512-byte
// rows of the transposed copy (the tile's output is one contiguous R1_TT * 1.5 KB block) and the packed 0/1 view.  The row
// stride of the tile is padded by one 16-byte slot so that the 32 lanes of phase 2 fall into distinct bank groups.
#define R1_TT 16
__global__ void __launch_bounds__(256) k_r1cs_transpose(const u32x4* z, size_t ncols, size_t w0, size_t g, u32x4* zt, uint2* zbool) {
    __shared__ u32x4 tile[32][R1_TT * 3 + 1];
    size_t col0 = blockIdx.x * (size_t)R1_TT; int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    size_t ncol_here = ncols - col0 < R1_TT ? ncols - col0 : R1_TT;
    u32x4 zero; zero.x = zero.y = zero.z = zero.w = 0;
#pragma unroll
    for (int k = 0; k < (32 * R1_TT * 3) / 256; k++) {
        int i = threadIdx.x + 256 * k, w = i / (R1_TT * 3), j = i % (R1_TT * 3);
        bool live = (size_t)w < g && (size_t)j < ncol_here * 3;
        tile[w][j] = live ? __ldcs(&z[((w0 + w) * ncols + col0) * 3 + j]) : zero;      // read once: evict-first, so the transposed copy of the non-0/1 columns stays in L2
    }
    __syncthreads();
#pragma unroll
    for (int h = 0; h < R1_TT / 8; h++) {
        int cl = warp + 8 * h; size_t col = col0 + cl;
        if ((size_t)cl >= ncol_here) break;
        u32x4 a = tile[lane][3 * cl], b = tile[lane][3 * cl + 1], c = tile[lane][3 * cl + 2];
        bool small = a.x < 2 && !(a.y | a.z | a.w | b.x | b.y | b.z | b.w | c.x | c.y | c.z | c.w);
        bool all = __all_sync(0xffffffffu, small);
        // a 0/1 column is only ever read through its packed word (every reader tests zbool[col].y first): its 1.5 KB of the transposed
        // copy are not written -- 93 % of the verify circuit's columns, so the transpose writes 0.08 GB per group instead of 1.09 GB
        if (!all) { zt[(col * 3) * 32 + lane] = a; zt[(col * 3 + 1) * 32 + lane] = b; zt[(col * 3 + 2) * 32 + lane] = c; }
        uint32_t pack = __ballot_sync(0xffffffffu, a.x & 1u);        // the column's 32 values as one word when they are all 0 / 1
        if (lane == 0) zbool[col] = make_uint2(all ? pack : 0u, all ? 1u : 0u);
    }
}
__device__ __forceinline__ fp r1cs_load_z(const u32x4* zt, uint32_t col, int lane) {
    u32x4 a = zt[((size_t)col * 3) * 32 + lane], b = zt[((size_t)col * 3 + 1) * 32 + lane], c = zt[((size_t)col * 3 + 2) * 32 + lane];
    fp v; v.l[0] = a.x; v.l[1] = a.y; v.l[2] = a.z; v.l[3] = a.w; v.l[4] = b.x; v.l[5] = b.y; v.l[6] = b.z; v.l[7] = b.w; v.l[8] = c.x; v.l[9] = c.y; v.l[10] = c.z; v.l[11] = c.w;
    return v;
}
// One non-zero: class c, column cj with its packed 0/1 view zb, |coefficient| low word cf (small classes).  Every branch is
// warp-uniform (class per non-zero, zbool per column).  Terms on 0/1 columns with coefficient +-1 or |c| < 2^32 go to the integer
// side sum (|term| < 2^32: no overflow below 2^31 terms); `touched` records whether the field accumulator was used at all.
// Terms on field-valued columns with coefficient +-1 or |c| < 2^32 go to the LAZY 14-limb sum `la` (fp_lacc_*: 12 IMAD.WIDE per term, one
// Barrett reduction per range instead of one per term; a negative coefficient enters as |c| (p - z)).
__device__ __forceinline__ void r1cs_term(const r1cs_sys& s, int m, uint64_t k, uint32_t cj, uint32_t c, uint2 zb, uint32_t cf, const u32x4* zt, int lane,
                                          fp& acc, int64_t& side, bool& touched, fp_lacc& la, bool& la_used, const fp* zpre = nullptr, wacc* wg = nullptr, int* wn = nullptr) {
    if (zb.y) {
        uint32_t bit = (zb.x >> lane) & 1u;
        if (c == R1_PLUS_ONE) side += bit;
        else if (c == R1_MINUS_ONE) side -= bit;
        else if (c == R1_SMALL_POS) side += (int64_t)((uint64_t)bit * cf);
        else if (c == R1_SMALL_NEG) side -= (int64_t)((uint64_t)bit * (BLS_P0 - cf));                  // |c| = p - c: the low words suffice
        else { acc = fp_add(acc, fp_select(0u - bit, s.coeffc[m][k], fp_zero())); touched = true; }   // general coefficient: masked addition
        return;
    }
    touched = true;
    fp zv = zpre ? *zpre : r1cs_load_z(zt, cj, lane);
    if (c == R1_GENERAL) {
        if (!wg) { acc = fp_add(acc, fp_mul(s.coeff[m][k], zv)); return; }
        // lazy form (witness replay): coefficient (Montgomery, < p) x value (canonical, < p) accumulated unreduced, one Montgomery reduction per
        // 8 products (sum < 8 p^2 < 9.8 p^2, the bound of wredc) -- 144 IMAD.WIDE per term instead of a 300-MAC product and a modular addition
        wmac(*wg, s.coeff[m][k], zv);
        if (++*wn == 8) { acc = fp_add(acc, wredc(*wg)); wacc_zero(*wg); *wn = 0; }
        return;
    }
    la_used = true;
    if (c == R1_PLUS_ONE) fp_lacc_mad(la, zv, 1u);
    else if (c == R1_SMALL_POS) fp_lacc_mad(la, zv, cf);
    else { fp nz; fp_sub_raw(nz, fp_modulus(), zv); fp_lacc_mad(la, nz, c == R1_MINUS_ONE ? 1u : BLS_P0 - cf); }      // z = 0 enters as |c| p = 0 (mod p)
}
// sum over the non-zeros [lo, hi) of one matrix: field part returned, integer part in side_out
__device__ __forceinline__ fp r1cs_range_dot(const r1cs_sys& s, int m, uint64_t lo, uint64_t hi, const u32x4* zt, const uint2* zbool, int lane, int64_t& side_out, bool& touched) {
    const uint32_t* col = s.col[m]; const uint8_t* cls = s.cls[m];
    fp acc = fp_zero(); int64_t side = 0; touched = false;
    fp_lacc la; fp_lacc_zero(la); bool la_used = false;
    uint32_t cj_n = 0; uint8_t c_n = 0; uint2 zb_n = make_uint2(0u, 0u);
    if (lo < hi) { cj_n = col[lo]; c_n = cls[lo]; zb_n = zbool[cj_n]; }
    for (uint64_t k = lo; k < hi; k++) {
        uint32_t cj = cj_n; uint8_t c = c_n; uint2 zb = zb_n;
        if (k + 1 < hi) { cj_n = col[k + 1]; c_n = cls[k + 1]; zb_n = zbool[cj_n]; }      // the next term's metadata travels while this term's gather does
        uint32_t cf = (c == R1_SMALL_POS || c == R1_SMALL_NEG) ? s.coeffc[m][k].l[0] : 0u;
        r1cs_term(s, m, k, cj, c, zb, cf, zt, lane, acc, side, touched, la, la_used);
    }
    if (la_used) acc = fp_add(acc, fp_lacc_reduce(la));          // warp-uniform (classes and packed views are)
    side_out = side; return acc;
}
// The same sum with the terms' metadata fetched LANE-PARALLEL: lane t loads column, class, packed view and small coefficient of term
// lo + t (two dependent rounds of independent loads for up to 32 terms), then the terms are evaluated from register broadcasts.  The
// term-by-term walk above chains column -> packed view (-> gather) per term: fine for the 7-term short rows, but a long row (long-scoreboard
// stalls were 36 % of the samples of the round-1 segment kernel) and the latency-bound witness replay pay that latency once per term.  All 32 lanes must call it together.
// metadata of up to 32 consecutive non-zeros, one per lane
struct r1cs_meta { uint32_t col, c, cf, n; uint2 zb; uint64_t base; };
__device__ __forceinline__ void r1cs_meta_fetch(r1cs_meta& t, const r1cs_sys& s, int m, uint64_t lo, uint64_t hi, int lane) {       // round 1: column, class, small coefficient
    t.base = lo; t.n = hi - lo < 32 ? (uint32_t)(hi - lo) : 32u; t.col = 0; t.c = R1_PLUS_ONE; t.cf = 0; t.zb = make_uint2(0u, 1u);
    if ((uint32_t)lane < t.n) {
        t.col = s.col[m][lo + lane]; t.c = s.cls[m][lo + lane];
        if (t.c == R1_SMALL_POS || t.c == R1_SMALL_NEG) t.cf = s.coeffc[m][lo + lane].l[0];
    }
}
__device__ __forceinline__ void r1cs_meta_views(r1cs_meta& t, const uint2* zbool, int lane) { if ((uint32_t)lane < t.n) t.zb = zbool[t.col]; }      // round 2: packed 0/1 views
struct r1cs_accum { fp acc; int64_t side; bool touched; fp_lacc la; bool la_used; };
__device__ __forceinline__ void r1cs_accum_zero(r1cs_accum& a) { a.acc = fp_zero(); a.side = 0; a.touched = false; fp_lacc_zero(a.la); a.la_used = false; }
// PF terms at a time: the gathers of all PF (for field-valued columns) are issued before the first term is evaluated.  PF = 1 in the
// satisfaction kernels (they run at 80 registers and are throughput-bound: pairs measured 13 % slower, profiles/r02_tuning.md); PF = 8 in
// the witness replay, which is bound by the chain of gathers inside one task and has registers to spare.
template <int PF> __device__ __forceinline__ void r1cs_meta_eval(const r1cs_meta& t, const r1cs_sys& s, int m, const u32x4* zt, int lane, r1cs_accum& a, wacc* wg = nullptr, int* wn = nullptr) {
    for (uint32_t k0 = 0; k0 < t.n; k0 += PF) {
        uint32_t cj[PF], c[PF], cf[PF]; uint2 zb[PF]; fp zv[PF];
#pragma unroll
        for (int j = 0; j < PF; j++) {
            uint32_t k = k0 + j < t.n ? k0 + j : t.n - 1;
            cj[j] = __shfl_sync(0xffffffffu, t.col, k); c[j] = __shfl_sync(0xffffffffu, t.c, k); cf[j] = __shfl_sync(0xffffffffu, t.cf, k);
            zb[j] = make_uint2(__shfl_sync(0xffffffffu, t.zb.x, k), __shfl_sync(0xffffffffu, t.zb.y, k));
            if (PF > 1 && k0 + j < t.n && !zb[j].y) zv[j] = r1cs_load_z(zt, cj[j], lane);
        }
#pragma unroll
        for (int j = 0; j < PF; j++)
            if (k0 + j < t.n) r1cs_term(s, m, t.base + k0 + j, cj[j], c[j], zb[j], cf[j], zt, lane, a.acc, a.side, a.touched, a.la, a.la_used, PF > 1 ? &zv[j] : nullptr, wg, wn);
    }
}
__device__ __forceinline__ fp r1cs_accum_close(r1cs_accum& a, int64_t& side_out, bool& touched) {
    if (a.la_used) a.acc = fp_add(a.acc, fp_lacc_reduce(a.la));            // warp-uniform (classes and packed views are)
    side_out = a.side; touched = a.touched; return a.acc;
}
__device__ __forceinline__ fp r1cs_range_dot_wide(const r1cs_sys& s, int m, uint64_t lo, uint64_t hi, const u32x4* zt, const uint2* zbool, int lane, int64_t& side_out, bool& touched) {
    r1cs_accum a; r1cs_accum_zero(a);                            // at most 2^18 terms between reductions of the lazy sum: no combination is that long
    for (uint64_t base = lo; base < hi; base += 32) {
        r1cs_meta t; r1cs_meta_fetch(t, s, m, base, hi, lane); r1cs_meta_views(t, zbool, lane); r1cs_meta_eval<1>(t, s, m, zt, lane, a);
    }
    return r1cs_accum_close(a, side_out, touched);
}
// field part + integer part as one canonical element
__device__ __forceinline__ fp r1cs_finalize(const fp& acc, int64_t side, bool touched) {
    uint64_t mag = side < 0 ? (uint64_t)(-side) : (uint64_t)side;
    fp t = fp_zero(); t.l[0] = (uint32_t)mag; t.l[1] = (uint32_t)(mag >> 32);
    uint32_t neg = side < 0 ? 0xffffffffu : 0u;
    if (!touched) { fp n; fp_sub_raw(n, fp_modulus(), t); return fp_select(neg, n, t); }      // side != 0 when neg, so p - |side| < p
    if (__all_sync(0xffffffffu, side == 0)) return acc;
    fp up = fp_add(acc, t), dn = fp_sub(acc, t);
    return fp_select(neg, dn, up);
}
// a b == c (all canonical).  In the boolean / uint32 gadget rows (95 % of the verify circuit) a and b are small integers
// (bits, 35-bit word sums): when one fits 64 bits and the other 32 bits in every lane the product is a 96-bit integer
// below p and is compared directly -- two Montgomery products per row saved.  The test is warp-uniform.
__device__ __forceinline__ bool r1cs_product_ok(const fp& a, const fp& b, const fp& c) {
    uint32_t ah = a.l[2] | a.l[3] | a.l[4] | a.l[5] | a.l[6] | a.l[7] | a.l[8] | a.l[9] | a.l[10] | a.l[11];
    uint32_t bh = b.l[2] | b.l[3] | b.l[4] | b.l[5] | b.l[6] | b.l[7] | b.l[8] | b.l[9] | b.l[10] | b.l[11];
    bool small = (ah | bh) == 0 && (a.l[1] == 0 || b.l[1] == 0);
    if (__all_sync(0xffffffffu, small)) {
        uint64_t x = ((uint64_t)a.l[1] << 32) | a.l[0], y = ((uint64_t)b.l[1] << 32) | b.l[0];
        uint64_t lo = x * y, hi = __umul64hi(x, y);               // < 2^96
        uint32_t ch = c.l[3] | c.l[4] | c.l[5] | c.l[6] | c.l[7] | c.l[8] | c.l[9] | c.l[10] | c.l[11];
        return ch == 0 && c.l[0] == (uint32_t)lo && c.l[1] == (uint32_t)(lo >> 32) && c.l[2] == (uint32_t)hi && (hi >> 32) == 0;
    }
    fp ab = fp_mul(fp_to_mont(a), b);                             // (aR)(b)/R = ab, canonical
    return fp_eq(ab, c);
}

// ---------------------------------------------------------------------------------------------------------------- row classes
// blsgpu_r1cs_load sorts the rows into three classes (VERDICT r1 item 3: "specialise rows at load time instead of interpreting them"):
//  * truth-table rows: at most R1_LUT_NNZ non-zeros on at most 5 distinct columns (column 0, the constant, counts).  When all of
//    those columns are 0/1 in a group of 32 assignments -- booleanity rows a (1 - a) = 0, AND rows a b = c, XOR rows
//    2a b = a + b - c, the SHA-256 ch / maj forms: 661,550 of the verify circuit's 714,250 rows -- satisfaction is a Boolean
//    function of <= 5 bits.  Its 32-entry table is computed once at load time with exact field arithmetic (k_r1cs_lut_build);
//    k_r1cs_lut then evaluates it BIT-SLICED with lane = row on the packed 32-assignment words: no field arithmetic, no CSR walk,
//    ~40 logic instructions per row and 32 assignments.  A row that meets a column which is not 0/1 in this group is appended to a
//    fallback list and evaluated generically, so the result is exact for every input.
//  * long rows (more than R1_LONG non-zeros): one warp per row, longest first (k_r1cs_long_rows).
//  * the rest ("generic" short rows, mostly the field rows of the pairing part): one warp per row, lane = assignment.
#define R1_NOT_LUT 0xffffffffu
#define R1_NO_COL 0xffffffffu
#ifndef R1_LUT_NNZ
#define R1_LUT_NNZ 16
#endif
// table[idx] = "the row holds when column c_j has the value bit j of idx"; absent columns never match, so the table does not depend on their bits
__global__ void __launch_bounds__(TPB, BLS_MINB) k_r1cs_lut_build(r1cs_sys s, const uint32_t* rows, size_t n) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    uint32_t row = rows[i];
    uint4 A = s.lut_a[row]; uint2 B = s.lut_b[row];
    uint32_t c[5] = {A.x & 0x7fffffffu, A.y, A.z, B.x, B.y};
    uint32_t table = 0;
    for (uint32_t idx = 0; idx < 32; idx++) {
        fp v[3];
        for (int m = 0; m < 3; m++) {
            fp acc = fp_zero();
            for (uint64_t k = s.rowptr[m][row]; k < s.rowptr[m][row + 1]; k++) {
                uint32_t cj = s.col[m][k], bit = 0;
                for (int j = 0; j < 5; j++) if (c[j] == cj) bit = (idx >> j) & 1u;
                if (bit) acc = fp_add(acc, s.coeff[m][k]);                       // Montgomery images: (aR)(bR)/R = abR is compared with cR
            }
            v[m] = acc;
        }
        if (fp_eq(fp_mul(v[0], v[1]), v[2])) table |= 1u << idx;
    }
    A.w = table; s.lut_a[row] = A;
}
// bitwise (x ? b : a)
__device__ __forceinline__ uint32_t r1cs_sel(uint32_t x, uint32_t a, uint32_t b) { return (x & b) | (~x & a); }
__device__ __forceinline__ uint32_t r1cs_tbit(uint32_t T, int i) { return 0u - ((T >> i) & 1u); }
// the 3-input / 5-input truth table T applied to 32 assignments at once (bit w of x_j = value of column j in assignment w)
__device__ __forceinline__ uint32_t r1cs_lut3(uint32_t T, uint32_t x0, uint32_t x1, uint32_t x2) {
    uint32_t m0 = r1cs_sel(x0, r1cs_tbit(T, 0), r1cs_tbit(T, 1)), m1 = r1cs_sel(x0, r1cs_tbit(T, 2), r1cs_tbit(T, 3));
    uint32_t m2 = r1cs_sel(x0, r1cs_tbit(T, 4), r1cs_tbit(T, 5)), m3 = r1cs_sel(x0, r1cs_tbit(T, 6), r1cs_tbit(T, 7));
    return r1cs_sel(x2, r1cs_sel(x1, m0, m1), r1cs_sel(x1, m2, m3));
}
__device__ __forceinline__ uint32_t r1cs_lut5(uint32_t T, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t x4) {
    uint32_t q0 = r1cs_lut3(T, x0, x1, x2), q1 = r1cs_lut3(T >> 8, x0, x1, x2), q2 = r1cs_lut3(T >> 16, x0, x1, x2), q3 = r1cs_lut3(T >> 24, x0, x1, x2);
    return r1cs_sel(x4, r1cs_sel(x3, q0, q1), r1cs_sel(x3, q2, q3));
}
// lane = row (32 consecutive rows per warp), the 32 assignments of the group in the bits of each word.  Writes -- plain stores, no
// atomics -- the 32-bit half word of every assignment for these rows: this kernel runs first in a group and thereby also
// initialises the output (rows of the other classes contribute 0 here and are OR-ed in by the later kernels).
__global__ void __launch_bounds__(256) k_r1cs_lut(r1cs_sys s, const uint2* zbool, size_t w0, size_t g, size_t words, uint32_t* sat32) {
    size_t row = blockIdx.x * (size_t)256 + threadIdx.x; int lane = threadIdx.x & 31;
    uint32_t R = 0;
    if (row < s.nrows) {
        uint4 A = s.lut_a[row];
        if (A.x != R1_NOT_LUT) {
            uint2 z0 = zbool[A.x & 0x7fffffffu], z1 = make_uint2(0u, 1u), z2 = z1, z3 = z1, z4 = z1;
            if (A.y != R1_NO_COL) z1 = zbool[A.y];
            if (A.z != R1_NO_COL) z2 = zbool[A.z];
            if (A.x >> 31) { uint2 B = s.lut_b[row]; z3 = zbool[B.x]; if (B.y != R1_NO_COL) z4 = zbool[B.y]; }
            if (z0.y & z1.y & z2.y & z3.y & z4.y) R = (A.x >> 31) ? r1cs_lut5(A.w, z0.x, z1.x, z2.x, z3.x, z4.x) : r1cs_lut3(A.w, z0.x, z1.x, z2.x);
            else s.fb_rows[atomicAdd(s.fb_count, 1u)] = (uint32_t)row;
        }
    }
    uint32_t mine = 0;                                      // 32 x 32 bit transpose: lane w ends up with the 32 rows of assignment w
#pragma unroll
    for (int w = 0; w < 32; w++) { uint32_t m = __ballot_sync(0xffffffffu, (R >> w) & 1u); if (lane == w) mine = m; }
    size_t half = row >> 5;                                 // warp-uniform
    if ((size_t)lane < g && half < 2 * words) sat32[(w0 + lane) * 2 * words + half] = mine;
}
// one warp per listed row, lane = assignment: the generic evaluation of the generic short rows and, behind them in the same index
// space, of the truth-table rows that fell back in this group (their count is on the device)
#ifndef R1_MINB_ROWS
#define R1_MINB_ROWS R1_MINB
#endif
__global__ void __launch_bounds__(TPB, R1_MINB_ROWS) k_r1cs_rows_list(r1cs_sys s, const u32x4* zt, const uint2* zbool, size_t w0, size_t g, size_t words, uint64_t* sat_bits) {
    size_t warp = blockIdx.x * (size_t)(TPB / 32) + (threadIdx.x >> 5), nwarps = gridDim.x * (size_t)(TPB / 32); int lane = threadIdx.x & 31;
    size_t n = s.n_gen + (size_t)*s.fb_count;
    for (size_t i = warp; i < n; i += nwarps) {
        size_t row = i < s.n_gen ? s.gen_rows[i] : s.fb_rows[i - s.n_gen];
        int64_t sa, sb, sc; bool ta, tb, tc;
        fp a = r1cs_range_dot(s, 0, s.rowptr[0][row], s.rowptr[0][row + 1], zt, zbool, lane, sa, ta);
        fp b = r1cs_range_dot(s, 1, s.rowptr[1][row], s.rowptr[1][row + 1], zt, zbool, lane, sb, tb);
        fp c = r1cs_range_dot(s, 2, s.rowptr[2][row], s.rowptr[2][row + 1], zt, zbool, lane, sc, tc);
        bool ok;
        if (!(ta | tb | tc)) ok = (__int128)sa * (__int128)sb == (__int128)sc;      // only 0/1 columns with small coefficients: |a b - c| < 2^80 < p, so equality mod p is equality
        else ok = r1cs_product_ok(r1cs_finalize(a, sa, ta), r1cs_finalize(b, sb, tb), r1cs_finalize(c, sc, tc));
        if ((size_t)lane < g && ok) atomicOr((unsigned long long*)&sat_bits[(w0 + lane) * words + (row >> 6)], 1ull << (row & 63));
    }
}
// one warp per long row, longest rows first: the three combinations through the lane-parallel metadata path, product test, bit.  Replaced
// round 1's segment + combine pair: no partial sums through global memory (301 MB per launch), one closing reduction per combination
// instead of one per 32-term segment (5.4 segments per long row on the verify circuit).
#ifndef R1_MINB_LONG
#define R1_MINB_LONG R1_MINB
#endif
__global__ void __launch_bounds__(TPB, R1_MINB_LONG) k_r1cs_long_rows(r1cs_sys s, const u32x4* zt, const uint2* zbool, size_t w0, size_t g, size_t words, uint64_t* sat_bits) {
    size_t li = blockIdx.x * (size_t)(TPB / 32) + (threadIdx.x >> 5); int lane = threadIdx.x & 31;
    if (li >= s.n_long) return;
    size_t row = s.long_sorted[li];
    int64_t sa, sb, sc; bool ta, tb, tc;
    fp a = r1cs_range_dot_wide(s, 0, s.rowptr[0][row], s.rowptr[0][row + 1], zt, zbool, lane, sa, ta); a = r1cs_finalize(a, sa, ta);
    fp b = r1cs_range_dot_wide(s, 1, s.rowptr[1][row], s.rowptr[1][row + 1], zt, zbool, lane, sb, tb); b = r1cs_finalize(b, sb, tb);
    fp c = r1cs_range_dot_wide(s, 2, s.rowptr[2][row], s.rowptr[2][row + 1], zt, zbool, lane, sc, tc); c = r1cs_finalize(c, sc, tc);
    bool ok = r1cs_product_ok(a, b, c);
    if ((size_t)lane < g && ok) atomicOr((unsigned long long*)&sat_bits[(w0 + lane) * words + (row >> 6)], 1ull << (row & 63));
}
// one warp per assignment: AND over its bit words (coalesced), lane 0 writes the flag
__global__ void __launch_bounds__(256) k_r1cs_all(const uint64_t* sat_bits, size_t nwit, size_t words, size_t nrows, uint8_t* all_sat) {
    size_t w = blockIdx.x * (size_t)8 + (threadIdx.x >> 5); int lane = threadIdx.x & 31; if (w >= nwit) return;
    bool all = true;
    for (size_t i = lane; i < words; i += 32) {
        uint64_t want = (i + 1 == words && (nrows & 63)) ? ((1ull << (nrows & 63)) - 1) : ~0ull;
        all &= sat_bits[w * words + i] == want;
    }
    all = __all_sync(0xffffffffu, all);
    if (lane == 0) all_sat[w] = all ? 1 : 0;
}

struct dev_tmp { void* p = nullptr; ~dev_tmp() { if (p) cudaFree(p); } };        // scratch device buffer released on every return path
template <class T> static int r1cs_upload(blsgpu_ctx* ctx, T** dst, const std::vector<T>& v) {
    size_t n = v.size() ? v.size() : 1;
    CU(cudaMalloc(dst, n * sizeof(T)));
    if (v.size()) CU(cudaMemcpyAsync(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}
static void r1cs_release(r1cs_sys* s) {
    for (int m = 0; m < 3; m++) { cudaFree(s->rowptr[m]); cudaFree(s->col[m]); cudaFree(s->coeff[m]); cudaFree(s->coeffc[m]); cudaFree(s->cls[m]); }
    cudaFree(s->long_sorted);
    cudaFree(s->lut_a); cudaFree(s->lut_b); cudaFree(s->gen_rows); cudaFree(s->fb_rows); cudaFree(s->fb_count);
    delete s;
}
// builds *s (zero-initialised by the caller, who releases it when this fails): uploads, coefficient classes, row classes, truth tables
static int r1cs_build(blsgpu_ctx* ctx, r1cs_sys* s, const uint64_t* const rowptr[3], const uint32_t* const col[3], const uint8_t* const coeff48[3], size_t nrows, size_t ncols) {
    s->nrows = nrows; s->ncols = ncols;
    bool dev = ctx->ptr_mode == BLSGPU_DEVICE;
    cudaMemcpyKind kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    std::vector<uint64_t> hrp[3]; std::vector<uint32_t> hcol_buf[3]; const uint32_t* hcol[3];      // host copies: the row classes are decided here
    for (int m = 0; m < 3; m++) {
        if (!rowptr[m]) return fail(ctx, BLSGPU_ERR_ARG, "null row pointer array");
        hrp[m].resize(nrows + 1);
        if (dev) { CU(cudaMemcpyAsync(hrp[m].data(), rowptr[m], 8 * (nrows + 1), cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream)); }
        else memcpy(hrp[m].data(), rowptr[m], 8 * (nrows + 1));
        if (hrp[m][0] != 0) return fail(ctx, BLSGPU_ERR_ARG, "rowptr[%d][0] must be 0", m);
        for (size_t r = 0; r < nrows; r++) if (hrp[m][r + 1] < hrp[m][r]) return fail(ctx, BLSGPU_ERR_ARG, "rowptr[%d] is not monotone at row %zu", m, r);
        size_t nnz = s->nnz[m] = hrp[m][nrows], na = nnz ? nnz : 1;
        if (nnz && (!col[m] || !coeff48[m])) return fail(ctx, BLSGPU_ERR_ARG, "null column / coefficient array");
        if (dev) { hcol_buf[m].resize(na); if (nnz) { CU(cudaMemcpyAsync(hcol_buf[m].data(), col[m], 4 * nnz, cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream)); } hcol[m] = hcol_buf[m].data(); }
        else hcol[m] = col[m];
        for (size_t k = 0; k < nnz; k++) if (hcol[m][k] >= ncols) return fail(ctx, BLSGPU_ERR_ARG, "matrix %d: column index %u of non-zero %zu is out of range (ncols = %zu)", m, hcol[m][k], k, ncols);
        CU(cudaMalloc(&s->rowptr[m], 8 * (nrows + 1))); CU(cudaMalloc(&s->col[m], 4 * na)); CU(cudaMalloc(&s->coeff[m], 48 * na)); CU(cudaMalloc(&s->coeffc[m], 48 * na)); CU(cudaMalloc(&s->cls[m], na));
        CU(cudaMemcpyAsync(s->rowptr[m], rowptr[m], 8 * (nrows + 1), kind, ctx->stream));
        if (nnz) {
            CU(cudaMemcpyAsync(s->col[m], col[m], 4 * nnz, kind, ctx->stream));
            dev_tmp raw; CU(cudaMalloc(&raw.p, 48 * nnz));
            CU(cudaMemcpyAsync(raw.p, coeff48[m], 48 * nnz, kind, ctx->stream));
            LAUNCH(k_r1cs_prepare, nblk(nnz), TPB, (const uint8_t*)raw.p, nnz, s->coeff[m], s->coeffc[m], s->cls[m]);
            CU(cudaStreamSynchronize(ctx->stream));
        }
    }
    // row classes: truth-table rows, long rows, generic short rows
    std::vector<uint32_t> long_row, gen_rows, lut_rows; size_t n_rounds = 0;
    std::vector<uint4> lut_a(nrows); std::vector<uint2> lut_b(nrows);
    for (size_t r = 0; r < nrows; r++) {
        lut_a[r] = make_uint4(R1_NOT_LUT, R1_NO_COL, R1_NO_COL, 0u); lut_b[r] = make_uint2(R1_NO_COL, R1_NO_COL);
        size_t len = 0; for (int m = 0; m < 3; m++) len += hrp[m][r + 1] - hrp[m][r];
        // truth-table shape first (at most R1_LUT_NNZ non-zeros over at most five columns), then long / generic by length
        uint32_t c[5]; int d = 0; bool fits = len <= R1_LUT_NNZ && ncols < 0x7fffffffu;
        for (int m = 0; m < 3 && fits; m++)
            for (uint64_t k = hrp[m][r]; k < hrp[m][r + 1] && fits; k++) {
                uint32_t cj = hcol[m][k]; int j = 0; while (j < d && c[j] != cj) j++;
                if (j == d) { if (d == 5) fits = false; else c[d++] = cj; }
            }
        if (fits && d > 0) {
            lut_a[r] = make_uint4(c[0] | (d > 3 ? 0x80000000u : 0u), d > 1 ? c[1] : R1_NO_COL, d > 2 ? c[2] : R1_NO_COL, 0u);
            lut_b[r] = make_uint2(d > 3 ? c[3] : R1_NO_COL, d > 4 ? c[4] : R1_NO_COL);
            lut_rows.push_back((uint32_t)r);
        } else if (len > R1_LONG) {
            long_row.push_back((uint32_t)r);
            for (int m = 0; m < 3; m++) n_rounds += (hrp[m][r + 1] - hrp[m][r] + 31) / 32;
        } else gen_rows.push_back((uint32_t)r);
    }
    s->n_long = long_row.size(); s->n_rounds = n_rounds; s->n_gen = gen_rows.size(); s->n_lut = lut_rows.size();
    {   auto len_of = [&](uint32_t r) { size_t l = 0; for (int m = 0; m < 3; m++) l += hrp[m][r + 1] - hrp[m][r]; return l; };
        std::stable_sort(long_row.begin(), long_row.end(), [&](uint32_t x, uint32_t y) { return len_of(x) > len_of(y); });
        if (int rc = r1cs_upload(ctx, &s->long_sorted, long_row)) return rc; }
    if (int rc = r1cs_upload(ctx, &s->lut_a, lut_a)) return rc;
    if (int rc = r1cs_upload(ctx, &s->lut_b, lut_b)) return rc;
    if (int rc = r1cs_upload(ctx, &s->gen_rows, gen_rows)) return rc;
    CU(cudaMalloc(&s->fb_rows, 4 * (lut_rows.size() ? lut_rows.size() : 1))); CU(cudaMalloc(&s->fb_count, 4));
    if (!lut_rows.empty()) {
        dev_tmp list; CU(cudaMalloc(&list.p, 4 * lut_rows.size()));
        CU(cudaMemcpyAsync(list.p, lut_rows.data(), 4 * lut_rows.size(), cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(k_r1cs_lut_build, nblk(lut_rows.size()), TPB, *s, (const uint32_t*)list.p, lut_rows.size());
        CU(cudaStreamSynchronize(ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" {
int blsgpu_r1cs_load(blsgpu_ctx* ctx, const uint64_t* const rowptr[3], const uint32_t* const col[3], const uint8_t* const coeff48[3], size_t nrows, size_t ncols, int* handle) {
    ENTER(); if (!rowptr || !col || !coeff48 || !handle || !nrows || !ncols) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    int h = -1; for (int i = 0; i < 16; i++) if (!ctx->r1cs[i]) { h = i; break; }
    if (h < 0) return fail(ctx, BLSGPU_ERR_ARG, "too many R1CS systems loaded");
    r1cs_sys* s = new (std::nothrow) r1cs_sys(); if (!s) return fail(ctx, BLSGPU_ERR_ALLOC, "out of host memory");
    memset(s, 0, sizeof *s);
    if (int rc = r1cs_build(ctx, s, rowptr, col, coeff48, nrows, ncols)) { cudaStreamSynchronize(ctx->stream); r1cs_release(s); return rc; }      // nothing half-built stays behind
    ctx->r1cs[h] = s; *handle = h; return 0;
}
int blsgpu_r1cs_free(blsgpu_ctx* ctx, int handle) {
    if (!ctx || handle < 0 || handle >= 16 || !ctx->r1cs[handle]) return BLSGPU_ERR_ARG;
    dev_guard guard_; cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream);
    r1cs_release(ctx->r1cs[handle]); ctx->r1cs[handle] = nullptr; return 0;
}
// ---- on-disk exchange format (VERDICT r1 item 7; written by rust/examples/export_r1cs.rs from arkworks' cs.to_matrices() after
// src/constraints.rs:335-367, and by bls_verify_gadget_b200/gadget.py from the in-repo builder).  All little-endian:
//   "BLSR1CS1" | u32 version = 1 | u32 field_bytes = 48 | u64 nrows | u64 ncols | u64 ninstance | u64 nnz[3] | u64 nwit          (72 bytes)
//   for A, B, C:  rowptr u64[nrows + 1] | col u32[nnz] (zero-padded to a multiple of 8 bytes) | coeff [nnz][48] canonical
//   nwit assignments of ncols x 48 bytes canonical (z = [1, instance.., witness..])
struct r1cs_file_hdr { char magic[8]; uint32_t version, field_bytes; uint64_t nrows, ncols, ninstance, nnz[3], nwit; };
struct file_closer { FILE* f; ~file_closer() { if (f) fclose(f); } };
static int r1cs_file_open(blsgpu_ctx* ctx, const char* path, file_closer& fc, r1cs_file_hdr& h, uint64_t& z_offset) {
    fc.f = fopen(path, "rb"); if (!fc.f) return fail(ctx, BLSGPU_ERR_ARG, "cannot open %s", path);
    if (fread(&h, sizeof h, 1, fc.f) != 1 || memcmp(h.magic, "BLSR1CS1", 8) != 0) return fail(ctx, BLSGPU_ERR_ARG, "%s is not a BLSR1CS1 file", path);
    if (h.version != 1 || h.field_bytes != 48 || !h.nrows || !h.ncols || h.ncols >= 0x7fffffffu) return fail(ctx, BLSGPU_ERR_ARG, "%s: unsupported header (version %u, field bytes %u)", path, h.version, h.field_bytes);
    z_offset = sizeof h;
    for (int m = 0; m < 3; m++) z_offset += 8 * (h.nrows + 1) + ((4 * h.nnz[m] + 7) & ~(uint64_t)7) + 48 * h.nnz[m];
    return 0;
}
extern "C" {
// shape4 (nullable) = {nrows, ncols, ninstance, nwit}
int blsgpu_r1cs_load_file(blsgpu_ctx* ctx, const char* path, int* handle, uint64_t* shape4) {
    ENTER(); if (!path || !handle) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    file_closer fc{nullptr}; r1cs_file_hdr h; uint64_t zoff;
    if (int rc = r1cs_file_open(ctx, path, fc, h, zoff)) return rc;
    std::vector<uint64_t> rp[3]; std::vector<uint32_t> cl[3]; std::vector<uint8_t> cf[3];
    for (int m = 0; m < 3; m++) {
        size_t nnz = h.nnz[m], colb = (4 * nnz + 7) & ~(size_t)7;
        rp[m].resize(h.nrows + 1); cl[m].resize(colb / 4 + 1); cf[m].resize(48 * nnz + 1);
        if (fread(rp[m].data(), 8, h.nrows + 1, fc.f) != h.nrows + 1 || (colb && fread(cl[m].data(), 1, colb, fc.f) != colb) || (nnz && fread(cf[m].data(), 48, nnz, fc.f) != nnz))
            return fail(ctx, BLSGPU_ERR_ARG, "%s: truncated matrix %d", path, m);
        if (rp[m][h.nrows] != nnz) return fail(ctx, BLSGPU_ERR_ARG, "%s: rowptr of matrix %d ends at %llu, header says %llu non-zeros", path, m, (unsigned long long)rp[m][h.nrows], (unsigned long long)nnz);
    }
    const uint64_t* rpp[3] = {rp[0].data(), rp[1].data(), rp[2].data()}; const uint32_t* clp[3] = {cl[0].data(), cl[1].data(), cl[2].data()}; const uint8_t* cfp[3] = {cf[0].data(), cf[1].data(), cf[2].data()};
    int saved = ctx->ptr_mode; ctx->ptr_mode = BLSGPU_HOST;
    int rc = blsgpu_r1cs_load(ctx, rpp, clp, cfp, (size_t)h.nrows, (size_t)h.ncols, handle);
    ctx->ptr_mode = saved;
    if (!rc && shape4) { shape4[0] = h.nrows; shape4[1] = h.ncols; shape4[2] = h.ninstance; shape4[3] = h.nwit; }
    return rc;
}
// checks assignments [first, first + count) stored in the file against the loaded system `handle` (which must have the file's shape);
// sat_bits (count x ceil(nrows/64) words) and all_sat (count bytes, nullable) are HOST pointers
int blsgpu_r1cs_check_file(blsgpu_ctx* ctx, int handle, const char* path, size_t first, size_t count, uint64_t* sat_bits, uint8_t* all_sat) {
    ENTER(); if (!path || !sat_bits || handle < 0 || handle >= 16 || !ctx->r1cs[handle]) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    file_closer fc{nullptr}; r1cs_file_hdr h; uint64_t zoff;
    if (int rc = r1cs_file_open(ctx, path, fc, h, zoff)) return rc;
    const r1cs_sys* s = ctx->r1cs[handle];
    if (h.nrows != s->nrows || h.ncols != s->ncols) return fail(ctx, BLSGPU_ERR_ARG, "%s holds a %llu x %llu system, the handle a %zu x %zu one", path, (unsigned long long)h.nrows, (unsigned long long)h.ncols, s->nrows, s->ncols);
    if (first + count > h.nwit) return fail(ctx, BLSGPU_ERR_ARG, "%s holds %llu assignments", path, (unsigned long long)h.nwit);
    size_t words = (s->nrows + 63) / 64, zb = (size_t)h.ncols * 48;
    std::vector<uint8_t> z; int saved = ctx->ptr_mode, rc = 0;
    for (size_t w = 0; w < count && !rc; w += R1_GROUP) {               // one group of 32 assignments at a time: bounded host memory
        size_t g = count - w < R1_GROUP ? count - w : R1_GROUP; z.resize(g * zb);
        if (fseek(fc.f, (long)(zoff + (first + w) * zb), SEEK_SET) != 0 || fread(z.data(), zb, g, fc.f) != g) return fail(ctx, BLSGPU_ERR_ARG, "%s: truncated assignments", path);
        ctx->ptr_mode = BLSGPU_HOST;
        rc = blsgpu_r1cs_check(ctx, handle, z.data(), g, sat_bits + w * words, all_sat ? all_sat + w : nullptr);
        ctx->ptr_mode = saved;
    }
    return rc;
}
}
// rows per class of a loaded system: counts[0] truth-table rows, [1] generic short rows, [2] long rows, [3] 32-term metadata rounds
// k_r1cs_long_rows walks (sum over long rows and matrices of ceil(nnz / 32))
int blsgpu_r1cs_row_classes(blsgpu_ctx* ctx, int handle, uint64_t counts[4]) {
    if (!ctx || handle < 0 || handle >= 16 || !ctx->r1cs[handle] || !counts) return BLSGPU_ERR_ARG;
    const r1cs_sys* s = ctx->r1cs[handle]; counts[0] = s->n_lut; counts[1] = s->n_gen; counts[2] = s->n_long; counts[3] = s->n_rounds; return 0;
}
}
// one group of <= 32 assignments given in the transposed layout (zt, zbool): truth-table rows first (plain stores: this initialises
// the group's slice of the output), then the rows that fell back, the generic short rows, and the long rows
#ifndef R1_FB_BLOCKS
#define R1_FB_BLOCKS 888          // 148 SMs x 6 resident CTAs: one grid-stride pass over both lists
#endif
static int r1cs_check_group(blsgpu_ctx* ctx, const r1cs_sys& s, const u32x4* zt, const uint2* zbool, size_t w0, size_t g, size_t words, uint64_t* dbits) {
    CU(cudaMemsetAsync(s.fb_count, 0, 4, ctx->stream));
    LAUNCH(k_r1cs_lut, nblk(words * 64, 256), 256, s, zbool, w0, g, words, (uint32_t*)dbits);
    if (s.n_lut || s.n_gen) LAUNCH(k_r1cs_rows_list, R1_FB_BLOCKS, TPB, s, zt, zbool, w0, g, words, dbits);
    if (s.n_long) LAUNCH(k_r1cs_long_rows, nblk(s.n_long, TPB / 32), TPB, s, zt, zbool, w0, g, words, dbits);
    return 0;
}
extern "C" {
int blsgpu_r1cs_check(blsgpu_ctx* ctx, int handle, const uint8_t* z48, size_t nwit, uint64_t* sat_bits, uint8_t* all_sat) {
    ENTER(); if (handle < 0 || handle >= 16 || !ctx->r1cs[handle] || !z48 || !sat_bits) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    if (!nwit) return 0;
    r1cs_sys s = *ctx->r1cs[handle];
    size_t words = (s.nrows + 63) / 64;
    bool host = ctx->ptr_mode == BLSGPU_HOST;
    // host mode stages one group of 32 witnesses at a time (32 * ncols * 48 bytes) so the workspace stays bounded
    size_t zgroup = (size_t)R1_GROUP * s.ncols * 48;
    if (int rc = ws_reserve(ctx, (host ? al(zgroup) : 0) + al(zgroup) + al(8 * s.ncols) + (host ? al(8 * words * nwit) + al(nwit) : 0) + 8192)) return rc;
    u32x4* zstage = host ? ws_take<u32x4>(ctx, zgroup / 16) : nullptr;
    u32x4* zt = ws_take<u32x4>(ctx, zgroup / 16);
    uint2* zbool = ws_take<uint2>(ctx, s.ncols);
    uint64_t* dbits = host ? ws_take<uint64_t>(ctx, words * nwit) : sat_bits;
    uint8_t* dall = all_sat ? (host ? ws_take<uint8_t>(ctx, nwit) : all_sat) : nullptr;
    for (size_t w0 = 0; w0 < nwit; w0 += R1_GROUP) {
        size_t g = nwit - w0 < R1_GROUP ? nwit - w0 : R1_GROUP;
        const u32x4* zsrc; size_t wbase;
        if (host) { CU(cudaMemcpyAsync(zstage, z48 + w0 * s.ncols * 48, g * s.ncols * 48, cudaMemcpyHostToDevice, ctx->stream)); zsrc = zstage; wbase = 0; }
        else { zsrc = (const u32x4*)z48; wbase = w0; }
        LAUNCH(k_r1cs_transpose, nblk(s.ncols, R1_TT), 256, zsrc, s.ncols, wbase, g, zt, zbool);
        if (int rc = r1cs_check_group(ctx, s, zt, zbool, w0, g, words, dbits)) return rc;
    }
    if (dall) LAUNCH(k_r1cs_all, nblk(nwit, 8), 256, (const uint64_t*)dbits, nwit, words, s.nrows, dall);
    if (host) {
        CU(cudaMemcpyAsync(sat_bits, dbits, 8 * words * nwit, cudaMemcpyDeviceToHost, ctx->stream));
        if (all_sat) CU(cudaMemcpyAsync(all_sat, dall, nwit, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return finish_call(ctx);
}
}
