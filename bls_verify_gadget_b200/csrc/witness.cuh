// GPU witness generation for the verify circuit (SURVEY 8(f)-1): replays the witness program recorded by the host-side
// builder (bls_verify_gadget_b200/gadget: one rule per variable, in allocation order) for 32 assignments per warp and
// writes them straight into the layout the satisfaction kernels gather from -- so (pk, msg, sig) bytes go in and the
// per-constraint bits come out without the 34 MB-per-assignment host synthesis and PCIe transfer.
//
// The reference has no counterpart (its witnesses come from running the gadget code under ark-relations'
// ConstraintSystem in "prove" mode, src/constraints.rs:335-370); the values are checked bit for bit against the host
// builder's assignment, which is pinned by the reference's own expectations (tests/test_gadget_circuit.py).
//
// Mapping: lane <-> assignment, warp <-> group of 32, rules strictly in order (a rule reads variables written by earlier
// rules of the same lane: program order makes them visible).  Every branch is warp-uniform (rule kind, coefficient class).
// Included after r1cs.cuh in blsgpu.cu.
#pragma once
#include <cooperative_groups.h>

#ifndef WIT_PF
#define WIT_PF 1          // gathers issued together per batch of terms in the replay (r1cs_meta_eval<PF>): 4 / 8 / 16 measured 1.3x / 1.8x / 4x SLOWER (spills), profiles/r02_tuning.md
#endif
enum { WR_MULADD = 0, WR_INV = 1, WR_NEQ = 2, WR_NEQMULT = 3, WR_BIT = 4, WR_FP2INV = 5, WR_FP12INV = 6, WR_INPUT = 7 };
struct wit_rule { uint8_t kind, pad; uint16_t aux; uint32_t a, b, d; };
// rule in level order with its term ranges resolved (one dependent load less per combination); for WR_FP12INV a_lo is the
// id of the first of twelve consecutive combinations
struct wit_xrule { uint8_t kind, pad; uint16_t aux; uint32_t var; uint32_t a_lo, a_hi, b_lo, b_hi, d_lo, d_hi; };
// light rule: WL_LUT a[0..4] = columns (WL_NO_COL pads), a[5] = 32-entry truth table; WL_SUM / WL_BIT a[0], a[1] = term range in lt_col / lt_coef,
// a[2] = integer slot of the result (WL_SUM, integer-valued); WL_INPUT aux = input slot; flags: 1 = WL_SUM with a 0/1 result, 2 = also export the
// integer as a field element (it is a circuit variable or a field rule reads it)
enum { WL_LUT = 0, WL_SUM = 1, WL_BIT = 2, WL_INPUT = 3, WL_ONE = 4 };
#define WL_NO_COL 0xffffffffu
#define WL_INT 0x80000000u          // lt_col entries with this bit address an integer slot instead of a 0/1 column
struct wit_lrule { uint8_t kind, flags; uint16_t aux; uint32_t var; uint32_t a[6]; };
struct wit_prog {
    size_t nvars, nout, nlc, nterms, nlevels;          // nvars: columns of the program (circuit variables, then scratch values); nout: circuit variables
    wit_rule* rules; uint64_t* lc_ptr; uint32_t* col; fp* coeff; fp* coeffc; uint8_t* cls;
    wit_xrule* xrules; uint64_t* level_ptr;          // dependency levels: rules of one level are independent
    // "light" part (blsgpu_witness_load): rules whose operands and result are 0/1 values or small integers -- the SHA-256 / bit-decomposition
    // gadgets: 715 k of the verify program's 1.04 M rules on 10.4 k of its dependency levels -- run in k_witness_light, one CTA per group of
    // 32 assignments with __syncthreads between levels; the remaining (field) rules keep the level-synchronous kernels above, on 4.3 k levels
    struct wit_lrule* lrules; uint32_t* llevel_ptr; uint32_t* lt_col; long long* lt_coef; size_t n_light, n_llevels, n_islots, n_lterms;
    size_t msg_len, ninputs, nkeys;                  // input slots of the recorded circuit: nkeys = 0: verify (6 + 8 msg_len); nkeys = n: aggregate_verify (3n + 4 + 8 msg_len)
};
#define WIT_POINT_INPUTS 6      // input slots 0..5: pk.x, pk.y, sig x.c0, x.c1, y.c0, y.c1; slot 6 + 8 i + b = bit b of message byte i (any message length)

__device__ __forceinline__ void wit_store(u32x4* zt, size_t col, int lane, const fp& v) {
    u32x4 a, b, c;
    a.x = v.l[0]; a.y = v.l[1]; a.z = v.l[2]; a.w = v.l[3]; b.x = v.l[4]; b.y = v.l[5]; b.z = v.l[6]; b.w = v.l[7]; c.x = v.l[8]; c.y = v.l[9]; c.z = v.l[10]; c.w = v.l[11];
    zt[(col * 3) * 32 + lane] = a; zt[(col * 3 + 1) * 32 + lane] = b; zt[(col * 3 + 2) * 32 + lane] = c;
}
// value of the combination with terms [lo, hi) on this lane's assignment, canonical.  zb (nullable) = the group's packed 0/1 view: a
// column that an earlier level found to be 0/1 in all 32 assignments is read as ONE broadcast 8-byte load instead of a 1.5 KB gather and
// its +-1 / small coefficients go to a 64-bit integer side sum -- the same term rule as the satisfaction kernels (r1cs_term), which is
// what 93 % of the verify circuit's columns and most of the witness program's 4.0 M terms are.
__device__ __forceinline__ fp wit_lc_range(const wit_prog& p, uint64_t lo, uint64_t hi, const u32x4* zt, const uint2* zb, int lane) {
    fp acc = fp_zero();
    if (zb) {
        r1cs_sys view; view.coeff[0] = p.coeff; view.coeffc[0] = p.coeffc; view.col[0] = p.col; view.cls[0] = p.cls;
        int64_t side = 0; bool touched = false;
        r1cs_accum ac; r1cs_accum_zero(ac);                    // metadata of up to 32 terms fetched in one round: the replay is latency-bound
        wacc wg; int wn = 0; wacc_zero(wg);                    // general coefficients on field values: lazy 768-bit sum (r1cs_term)
        for (uint64_t base = lo; base < hi; base += 32) { r1cs_meta t; r1cs_meta_fetch(t, view, 0, base, hi, lane); r1cs_meta_views(t, zb, lane); r1cs_meta_eval<WIT_PF>(t, view, 0, zt, lane, ac, &wg, &wn); }
        if (wn) ac.acc = fp_add(ac.acc, wredc(wg));
        acc = r1cs_accum_close(ac, side, touched);
        return r1cs_finalize(acc, side, touched);
    }
    for (uint64_t k = lo, e = hi; k < e; k++) {
        uint32_t cj = p.col[k]; uint8_t c = p.cls[k];
        fp zv = r1cs_load_z(zt, cj, lane);
        if (c == R1_PLUS_ONE) acc = fp_add(acc, zv);
        else if (c == R1_MINUS_ONE) acc = fp_sub(acc, zv);
        else {
            bool small = zv.l[0] < 2 && !(zv.l[1] | zv.l[2] | zv.l[3] | zv.l[4] | zv.l[5] | zv.l[6] | zv.l[7] | zv.l[8] | zv.l[9] | zv.l[10] | zv.l[11]);
            if (__all_sync(0xffffffffu, small)) acc = fp_add(acc, fp_select(0u - zv.l[0], p.coeffc[k], fp_zero()));       // coefficient times a 0/1 value
            else if (c == R1_SMALL_POS) acc = fp_add(acc, fp_mul_small(zv, p.coeffc[k].l[0]));
            else if (c == R1_SMALL_NEG) acc = fp_sub(acc, fp_mul_small(zv, BLS_P0 - p.coeffc[k].l[0]));
            else acc = fp_add(acc, fp_mul(p.coeff[k], zv));
        }
    }
    return acc;
}
// The three combinations of a product rule (a b + d) with their metadata rounds OVERLAPPED: the replay is bound by the chain of dependent
// loads inside one task (rule -> columns -> packed views -> values), so the column / class / coefficient loads of all three ranges are
// issued together, then the packed views of all three, and only then are the terms evaluated.  Ranges longer than 32 terms finish
// through the chunked loop.
__device__ __forceinline__ void wit_lc3(const wit_prog& p, const wit_xrule& r, const u32x4* zt, const uint2* zb, int lane, fp& a, fp& b, fp& d) {
    r1cs_sys view; view.coeff[0] = p.coeff; view.coeffc[0] = p.coeffc; view.col[0] = p.col; view.cls[0] = p.cls;
    r1cs_meta ta, tb, td;
    r1cs_meta_fetch(ta, view, 0, r.a_lo, r.a_hi, lane); r1cs_meta_fetch(tb, view, 0, r.b_lo, r.b_hi, lane); r1cs_meta_fetch(td, view, 0, r.d_lo, r.d_hi, lane);
    r1cs_meta_views(ta, zb, lane); r1cs_meta_views(tb, zb, lane); r1cs_meta_views(td, zb, lane);
    const r1cs_meta* ts[3] = {&ta, &tb, &td}; const uint32_t his[3] = {r.a_hi, r.b_hi, r.d_hi}; fp* outs[3] = {&a, &b, &d};
#pragma unroll
    for (int k = 0; k < 3; k++) {
        r1cs_accum acc; r1cs_accum_zero(acc);
        wacc wg; int wn = 0; wacc_zero(wg);
        r1cs_meta_eval<WIT_PF>(*ts[k], view, 0, zt, lane, acc, &wg, &wn);
        for (uint64_t base = ts[k]->base + 32; base < his[k]; base += 32) { r1cs_meta t; r1cs_meta_fetch(t, view, 0, base, his[k], lane); r1cs_meta_views(t, zb, lane); r1cs_meta_eval<WIT_PF>(t, view, 0, zt, lane, acc, &wg, &wn); }
        if (wn) acc.acc = fp_add(acc.acc, wredc(wg));
        int64_t side; bool touched; fp v = r1cs_accum_close(acc, side, touched);
        *outs[k] = r1cs_finalize(v, side, touched);
    }
}
__device__ __forceinline__ fp wit_lc(const wit_prog& p, uint32_t id, const u32x4* zt, const uint2* zb, int lane) {
    if (!id) return fp_zero();
    return wit_lc_range(p, p.lc_ptr[id - 1], p.lc_ptr[id], zt, zb, lane);
}
__device__ __forceinline__ fp wit_inv_canon(const fp& a) { return fp_inv_raw(a); }                 // canonical in and out: the divsteps inverse needs no Montgomery factor
// a b for canonical a, b: small-integer shortcut as in r1cs_product_ok
__device__ __forceinline__ fp wit_mul_canon(const fp& a, const fp& b) {
    uint32_t ah = a.l[2] | a.l[3] | a.l[4] | a.l[5] | a.l[6] | a.l[7] | a.l[8] | a.l[9] | a.l[10] | a.l[11];
    uint32_t bh = b.l[2] | b.l[3] | b.l[4] | b.l[5] | b.l[6] | b.l[7] | b.l[8] | b.l[9] | b.l[10] | b.l[11];
    bool small = (ah | bh) == 0 && (a.l[1] == 0 || b.l[1] == 0);
    if (__all_sync(0xffffffffu, small)) {
        uint64_t x = ((uint64_t)a.l[1] << 32) | a.l[0], y = ((uint64_t)b.l[1] << 32) | b.l[0];
        uint64_t lo = x * y, hi = __umul64hi(x, y);
        fp r = fp_zero(); r.l[0] = (uint32_t)lo; r.l[1] = (uint32_t)(lo >> 32); r.l[2] = (uint32_t)hi; r.l[3] = (uint32_t)(hi >> 32);
        return r;                                                     // < 2^96 < p
    }
    return fp_mul(fp_to_mont(a), b);
}
// inputs: fp [6 + 8 msg_len][nwit_padded] canonical (slot-major, so a warp reads 32 consecutive elements)
__global__ void __launch_bounds__(32) k_witness_gen(wit_prog p, const fp* inputs, size_t nwit_padded, u32x4* zt_all) {
    size_t group = blockIdx.x; int lane = threadIdx.x;
    u32x4* zt = zt_all + group * p.nvars * 96;                        // 3 chunks x 32 lanes per variable
    size_t w = group * 32 + lane;
    fp one = fp_zero(); one.l[0] = 1;
    wit_store(zt, 0, lane, one);
    for (size_t v = 1; v < p.nvars; v++) {
        wit_rule r = p.rules[v];
        fp out;
        switch (r.kind) {
            case WR_MULADD: {
                fp d = wit_lc(p, r.d, zt, nullptr, lane);
                if (r.a) { fp a = wit_lc(p, r.a, zt, nullptr, lane), b = wit_lc(p, r.b, zt, nullptr, lane); out = fp_add(wit_mul_canon(a, b), d); }
                else out = d;
                break;
            }
            case WR_INV: out = wit_inv_canon(wit_lc(p, r.a, zt, nullptr, lane)); break;
            case WR_NEQ: { fp a = wit_lc(p, r.a, zt, nullptr, lane); out = fp_zero(); out.l[0] = fp_is_zero(a) ? 0u : 1u; break; }
            case WR_NEQMULT: { fp a = wit_lc(p, r.a, zt, nullptr, lane); out = fp_is_zero(a) ? one : wit_inv_canon(a); break; }
            case WR_BIT: { fp a = wit_lc(p, r.a, zt, nullptr, lane); out = fp_zero(); out.l[0] = (a.l[r.aux >> 5] >> (r.aux & 31)) & 1u; break; }
            case WR_FP2INV: {
                fp2 x; x.c0 = fp_to_mont(wit_lc(p, r.a, zt, nullptr, lane)); x.c1 = fp_to_mont(wit_lc(p, r.b, zt, nullptr, lane));
                fp2 iv = fp2_inv(x); out = fp_from_mont(r.aux ? iv.c1 : iv.c0); break;
            }
            case WR_FP12INV: {
                fp12 x, iv; fp* xf = &x.c0.c0.c0;
                for (int k = 0; k < 12; k++) xf[k] = fp_to_mont(wit_lc(p, r.a + k, zt, nullptr, lane));
                fp12_inv(iv, x); out = fp_from_mont((&iv.c0.c0.c0)[r.aux]); break;
            }
            default: out = inputs[(size_t)r.aux * nwit_padded + w]; break;                 // WR_INPUT
        }
        wit_store(zt, v, lane, out);
    }
}
// Level-synchronous form: one warp per (rule of the current level, group of 32 assignments); a grid-wide barrier between
// levels (cooperative launch).  The verify circuit has 8,816 levels of ~80 rules: with 16 groups a level is ~1,300 independent
// warp tasks, against ONE warp per group walking 707,809 rules in sequence in k_witness_gen (7.3 s, latency bound).
#ifndef WIT_TPB
#define WIT_TPB 128
#endif
#ifndef WIT_BPS
#define WIT_BPS 2
#endif
#ifdef WIT_TRACE
// tuning builds only (profiles/tools/wit_trace.py): the global timer at the start of every level, written by warp 0
__device__ unsigned long long g_wit_trace[32768];
extern "C" int blsgpu_debug_wit_trace(unsigned long long* out, size_t n) { return cudaMemcpyFromSymbol(out, g_wit_trace, 8 * (n < 32768 ? n : 32768)) == cudaSuccess ? 0 : -1; }
#endif
__global__ void __launch_bounds__(WIT_TPB, WIT_BPS) k_witness_levels(wit_prog p, const fp* inputs, size_t nwit_padded, u32x4* zt_all, size_t groups, uint2* zbool_all) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    size_t warp = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * (size_t)blockDim.x) >> 5; int lane = threadIdx.x & 31;
    fp one = fp_zero(); one.l[0] = 1;
    uint64_t lo = p.level_ptr[0], hi = p.level_ptr[1];
    wit_xrule rn; bool pre = warp < (hi - lo) * groups;              // this warp's first rule of the next level is fetched before the barrier (static data)
    if (pre) rn = p.xrules[lo + warp / groups];
    for (size_t level = 0; level < p.nlevels; level++) {
        uint64_t n = hi - lo, hi_next = level + 2 <= p.nlevels ? p.level_ptr[level + 2] : hi;
#ifdef WIT_TRACE
        if (warp == 0 && lane == 0 && level < 32768) { unsigned long long tm; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tm)); g_wit_trace[level] = tm; }
#endif
        for (size_t t = warp; t < n * groups; t += nwarps) {
            wit_xrule r = (t == warp && pre) ? rn : p.xrules[lo + t / groups]; size_t group = t % groups;
            u32x4* zt = zt_all + group * p.nvars * 96; const uint2* zb = zbool_all ? zbool_all + group * p.nvars : nullptr;
            fp out;
            switch (r.kind) {
                case WR_MULADD: {
                    if (zb) { fp a, b, d; wit_lc3(p, r, zt, zb, lane, a, b, d); out = r.a_hi > r.a_lo ? fp_add(wit_mul_canon(a, b), d) : d; break; }
                    fp d = wit_lc_range(p, r.d_lo, r.d_hi, zt, zb, lane);
                    if (r.a_hi > r.a_lo) { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane), b = wit_lc_range(p, r.b_lo, r.b_hi, zt, zb, lane); out = fp_add(wit_mul_canon(a, b), d); }
                    else out = d;
                    break;
                }
                case WR_INV: out = wit_inv_canon(wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane)); break;
                case WR_NEQ: { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane); out = fp_zero(); out.l[0] = fp_is_zero(a) ? 0u : 1u; break; }
                case WR_NEQMULT: { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane); out = fp_is_zero(a) ? one : wit_inv_canon(a); break; }
                case WR_BIT: { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane); out = fp_zero(); out.l[0] = (a.l[r.aux >> 5] >> (r.aux & 31)) & 1u; break; }
                case WR_FP2INV: {
                    fp2 x; x.c0 = fp_to_mont(wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane)); x.c1 = fp_to_mont(wit_lc_range(p, r.b_lo, r.b_hi, zt, zb, lane));
                    fp2 iv = fp2_inv(x); out = fp_from_mont(r.aux ? iv.c1 : iv.c0); break;
                }
                case WR_FP12INV: {
                    fp12 x, iv; fp* xf = &x.c0.c0.c0;
                    for (int k = 0; k < 12; k++) xf[k] = fp_to_mont(wit_lc(p, r.a_lo + k, zt, zb, lane));
                    fp12_inv(iv, x); out = fp_from_mont((&iv.c0.c0.c0)[r.aux]); break;
                }
                default: out = r.aux == 0xffff ? one : inputs[(size_t)r.aux * nwit_padded + group * 32 + lane]; break;       // WR_INPUT; 0xffff: the constant ONE (variable 0)
            }
            if (!zbool_all) wit_store(zt, r.var, lane, out);
            else {                                  // the packed 0/1 view the satisfaction kernels read (r1cs.cuh: k_r1cs_transpose writes the same)
                bool small = out.l[0] < 2 && !(out.l[1] | out.l[2] | out.l[3] | out.l[4] | out.l[5] | out.l[6] | out.l[7] | out.l[8] | out.l[9] | out.l[10] | out.l[11]);
                bool all = __all_sync(0xffffffffu, small); uint32_t pack = __ballot_sync(0xffffffffu, out.l[0] & 1u);
                if (!all) wit_store(zt, r.var, lane, out);           // a 0/1 column lives in its packed word only (every reader tests the flag first)
                if (lane == 0) zbool_all[group * p.nvars + r.var] = make_uint2(all ? pack : 0u, all ? 1u : 0u);
            }
        }
        pre = level + 1 < p.nlevels && warp < (hi_next - hi) * groups;
        if (pre) rn = p.xrules[hi + warp / groups];
        grid.sync();
        lo = hi; hi = hi_next;
    }
}
// Cluster form of the level-synchronous replay: one thread-block CLUSTER (WIT_CL CTAs on WIT_CL SMs, 8 x 256 threads = 64 warps) owns
// one group of 32 assignments, one warp per rule of the current level, and the barrier between levels is the hardware cluster barrier
// (~0.2 us) instead of a grid-wide barrier over every resident CTA (several us, 14.7 k times per launch).  Groups run independently
// side by side (18 clusters fill the 148 SMs; further groups queue behind them), so a launch costs (levels x level latency) per WAVE
// of 18 groups.  The next level's rule record -- static data -- is fetched BEFORE the barrier, so that after it only the loads
// that depend on the previous level's values remain on the critical path.
#ifndef WIT_CL
#define WIT_CL 8
#endif
#define WIT_CL_TPB 256
__device__ __forceinline__ void wit_eval_rule(const wit_prog& p, const wit_xrule& r, const fp* inputs, size_t nwit_padded, size_t group, u32x4* zt, uint2* zbw, int lane) {
    const uint2* zb = zbw;
    fp one = fp_zero(); one.l[0] = 1;
    fp out;
    switch (r.kind) {
        case WR_MULADD: {
            if (zb) { fp a, b, d; wit_lc3(p, r, zt, zb, lane, a, b, d); out = r.a_hi > r.a_lo ? fp_add(wit_mul_canon(a, b), d) : d; break; }
            fp d = wit_lc_range(p, r.d_lo, r.d_hi, zt, zb, lane);
            if (r.a_hi > r.a_lo) { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane), b = wit_lc_range(p, r.b_lo, r.b_hi, zt, zb, lane); out = fp_add(wit_mul_canon(a, b), d); }
            else out = d;
            break;
        }
        case WR_INV: out = wit_inv_canon(wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane)); break;
        case WR_NEQ: { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane); out = fp_zero(); out.l[0] = fp_is_zero(a) ? 0u : 1u; break; }
        case WR_NEQMULT: { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane); out = fp_is_zero(a) ? one : wit_inv_canon(a); break; }
        case WR_BIT: { fp a = wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane); out = fp_zero(); out.l[0] = (a.l[r.aux >> 5] >> (r.aux & 31)) & 1u; break; }
        case WR_FP2INV: {
            fp2 x; x.c0 = fp_to_mont(wit_lc_range(p, r.a_lo, r.a_hi, zt, zb, lane)); x.c1 = fp_to_mont(wit_lc_range(p, r.b_lo, r.b_hi, zt, zb, lane));
            fp2 iv = fp2_inv(x); out = fp_from_mont(r.aux ? iv.c1 : iv.c0); break;
        }
        case WR_FP12INV: {
            fp12 x, iv; fp* xf = &x.c0.c0.c0;
            for (int k = 0; k < 12; k++) xf[k] = fp_to_mont(wit_lc(p, r.a_lo + k, zt, zb, lane));
            fp12_inv(iv, x); out = fp_from_mont((&iv.c0.c0.c0)[r.aux]); break;
        }
        default: out = r.aux == 0xffff ? one : inputs[(size_t)r.aux * nwit_padded + group * 32 + lane]; break;       // WR_INPUT; 0xffff: the constant ONE (variable 0)
    }
    if (!zbw) { wit_store(zt, r.var, lane, out); return; }
    bool small = out.l[0] < 2 && !(out.l[1] | out.l[2] | out.l[3] | out.l[4] | out.l[5] | out.l[6] | out.l[7] | out.l[8] | out.l[9] | out.l[10] | out.l[11]);
    bool all = __all_sync(0xffffffffu, small); uint32_t pack = __ballot_sync(0xffffffffu, out.l[0] & 1u);
    if (!all) wit_store(zt, r.var, lane, out);                // a 0/1 column lives in its packed word only (every reader tests the flag first)
    if (lane == 0) zbw[r.var] = make_uint2(all ? pack : 0u, all ? 1u : 0u);
}
__global__ void __launch_bounds__(WIT_CL_TPB, 1) k_witness_cluster(wit_prog p, const fp* inputs, size_t nwit_padded, u32x4* zt_all, size_t groups, uint2* zbool_all) {
    cooperative_groups::cluster_group cluster = cooperative_groups::this_cluster();
    const unsigned CW = WIT_CL * (WIT_CL_TPB / 32);                                             // warps of the cluster
    size_t group = blockIdx.x / WIT_CL; unsigned cw = cluster.block_rank() * (WIT_CL_TPB / 32) + (threadIdx.x >> 5); int lane = threadIdx.x & 31;
    u32x4* zt = zt_all + group * p.nvars * 96; uint2* zbw = zbool_all ? zbool_all + group * p.nvars : nullptr;
    uint64_t lo = p.level_ptr[0], hi = p.level_ptr[1];
    wit_xrule rn; bool pre = lo + cw < hi;
    if (pre) rn = p.xrules[lo + cw];
    for (size_t level = 0; level < p.nlevels; level++) {
        uint64_t hi_next = level + 2 <= p.nlevels ? p.level_ptr[level + 2] : hi;
        for (uint64_t t = lo + cw; t < hi; t += CW) {
            wit_xrule r = (t == lo + cw && pre) ? rn : p.xrules[t];
            wit_eval_rule(p, r, inputs, nwit_padded, group, zt, zbw, lane);
        }
        pre = level + 1 < p.nlevels && hi + cw < hi_next;
        if (pre) rn = p.xrules[hi + cw];                      // static data: travels while the cluster gathers at the barrier
        cluster.sync();
        lo = hi; hi = hi_next;
    }
}
// ---- the light part: 0/1 and small-integer rules, one CTA per group of 32 assignments.  A truth-table rule is evaluated by ONE THREAD for all
// 32 assignments (bit-sliced on the packed words, like k_r1cs_lut); sums and bit extractions take a warp (lane = assignment, 64-bit integers).
// The barrier between levels is __syncthreads: ~0.1 us instead of the grid barrier, and the per-level latency is one dependent load of packed
// words that this SM wrote itself.  Values: zbool[var] = (packed word, 1); integers in sint[slot][32].
#define WIT_LIGHT_TPB 1024
__global__ void __launch_bounds__(WIT_LIGHT_TPB, 1) k_witness_light(wit_prog p, const fp* inputs, size_t nwit_padded, u32x4* zt_all, uint2* zbool_all, long long* sint_all) {
    size_t group = blockIdx.x; int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint2* zb = zbool_all + group * p.nvars; long long* sint = sint_all + group * p.n_islots * 32; u32x4* zt = zt_all + group * p.nvars * 96;
    // this thread's first truth-table rule and this warp's first sum / bit rule of the NEXT level are fetched before the barrier (static data)
    uint32_t lut_lo = p.llevel_ptr[0], w_lo = p.llevel_ptr[1], nxt = p.llevel_ptr[2];
    wit_lrule rt, rw; bool pre_t = lut_lo + tid < w_lo, pre_w = w_lo + warp < nxt;
    if (pre_t) rt = p.lrules[lut_lo + tid];
    if (pre_w) rw = p.lrules[w_lo + warp];
    for (size_t L = 0; L < p.n_llevels; L++) {
        for (uint32_t i = lut_lo + tid; i < w_lo; i += WIT_LIGHT_TPB) {
            wit_lrule r = (pre_t && i == lut_lo + tid) ? rt : p.lrules[i];
            uint32_t x0 = zb[r.a[0]].x, x1 = r.a[1] != WL_NO_COL ? zb[r.a[1]].x : 0u, x2 = r.a[2] != WL_NO_COL ? zb[r.a[2]].x : 0u;
            uint32_t out;
            if (r.a[3] != WL_NO_COL) { uint32_t x3 = zb[r.a[3]].x, x4 = r.a[4] != WL_NO_COL ? zb[r.a[4]].x : 0u; out = r1cs_lut5(r.a[5], x0, x1, x2, x3, x4); }
            else out = r1cs_lut3(r.a[5], x0, x1, x2);
            zb[r.var] = make_uint2(out, 1u);
        }
        for (uint32_t i = w_lo + warp; i < nxt; i += WIT_LIGHT_TPB / 32) {
            wit_lrule r = (pre_w && i == w_lo + warp) ? rw : p.lrules[i];
            if (r.kind == WL_ONE) { if (lane == 0) zb[r.var] = make_uint2(0xffffffffu, 1u); continue; }
            if (r.kind == WL_INPUT) {
                uint32_t bit = inputs[(size_t)r.aux * nwit_padded + group * 32 + lane].l[0] & 1u;
                uint32_t pack = __ballot_sync(0xffffffffu, bit); if (lane == 0) zb[r.var] = make_uint2(pack, 1u); continue;
            }
            long long sum = 0;
            for (uint32_t t0 = r.a[0]; t0 < r.a[1]; t0 += 32) {                 // the terms' metadata lane-parallel, then broadcasts
                uint32_t n = r.a[1] - t0 < 32 ? r.a[1] - t0 : 32u, myc = 0; long long myk = 0;
                if ((uint32_t)lane < n) { myc = p.lt_col[t0 + lane]; myk = p.lt_coef[t0 + lane]; }
                uint32_t myw = ((uint32_t)lane < n && !(myc & WL_INT)) ? zb[myc].x : 0u;
                for (uint32_t t = 0; t < n; t++) {
                    uint32_t c = __shfl_sync(0xffffffffu, myc, t); long long k = __shfl_sync(0xffffffffu, myk, t); uint32_t wd = __shfl_sync(0xffffffffu, myw, t);
                    long long v = (c & WL_INT) ? sint[(size_t)(c & ~WL_INT) * 32 + lane] : (long long)((wd >> lane) & 1u);
                    sum += k * v;
                }
            }
            if (r.kind == WL_BIT || (r.flags & 1)) {
                uint32_t bit = r.kind == WL_BIT ? (uint32_t)((unsigned long long)sum >> (r.aux & 63)) & 1u : (uint32_t)sum & 1u;
                uint32_t pack = __ballot_sync(0xffffffffu, bit); if (lane == 0) zb[r.var] = make_uint2(pack, 1u);
            } else {
                sint[(size_t)r.a[2] * 32 + lane] = sum;
                if (r.flags & 2) {                            // the value as a canonical field element beside the integer
                    unsigned long long mag = sum < 0 ? (unsigned long long)(-sum) : (unsigned long long)sum;
                    fp v = fp_zero(); v.l[0] = (uint32_t)mag; v.l[1] = (uint32_t)(mag >> 32);
                    if (sum < 0) { fp n; fp_sub_raw(n, fp_modulus(), v); v = n; }
                    wit_store(zt, r.var, lane, v); if (lane == 0) zb[r.var] = make_uint2(0u, 0u);
                }
            }
        }
        lut_lo = nxt; pre_t = pre_w = false;
        if (L + 1 < p.n_llevels) {
            w_lo = p.llevel_ptr[2 * L + 3]; nxt = p.llevel_ptr[2 * L + 4];
            pre_t = lut_lo + tid < w_lo; pre_w = w_lo + warp < nxt;
            if (pre_t) rt = p.lrules[lut_lo + tid];
            if (pre_w) rw = p.lrules[w_lo + warp];
        }
        __syncthreads();
    }
}
// input slots from the decoded points and the message bytes; items whose key or signature does not decode get all-zero inputs
__global__ void __launch_bounds__(TPB, BLS_MINB) k_witness_inputs(const u32x4* pk_soa, const uint8_t* code_pk, const u32x4* sig_soa, const uint8_t* code_sig, const uint8_t* msg, size_t msg_len,
                                                                  size_t nwit, size_t nwit_padded, fp* inputs, uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= nwit_padded) return;
    bool live = i < nwit; uint8_t st = ST_OK;
    if (live) { if (code_pk[i] != DEC_OK) st = ST_BAD_PK; else if (code_sig[i] != DEC_OK) st = ST_BAD_SIG; }      // the circuit inverts z of both points: the identity has no assignment
    bool ok = live && st == ST_OK;
    fp zero = fp_zero();
    for (size_t k = 0; k < 8 * msg_len; k++) { fp b = zero; if (ok) b.l[0] = (msg[msg_len * i + (k >> 3)] >> (k & 7)) & 1u; inputs[(size_t)(WIT_POINT_INPUTS + k) * nwit_padded + i] = b; }
    g1_aff pk; g2_aff sg;
    if (ok) { soa_load_g1(pk, pk_soa, nwit, i); soa_load_g2(sg, sig_soa, nwit, i); }
    inputs[(size_t)0 * nwit_padded + i] = ok ? fp_from_mont(pk.x) : zero; inputs[(size_t)1 * nwit_padded + i] = ok ? fp_from_mont(pk.y) : zero;
    inputs[(size_t)2 * nwit_padded + i] = ok ? fp_from_mont(sg.x.c0) : zero; inputs[(size_t)3 * nwit_padded + i] = ok ? fp_from_mont(sg.x.c1) : zero;
    inputs[(size_t)4 * nwit_padded + i] = ok ? fp_from_mont(sg.y.c0) : zero; inputs[(size_t)5 * nwit_padded + i] = ok ? fp_from_mont(sg.y.c1) : zero;
    if (live && status) status[i] = st;
}
// the same for the aggregate_verify circuit: n keys (decoded into key_soa, item i key k at i * n + k), one bitmap byte per key, message, signature
__global__ void __launch_bounds__(TPB, BLS_MINB) k_witness_inputs_agg(const u32x4* key_soa, const uint8_t* code_key, size_t n, const uint8_t* bitmap, const u32x4* sig_soa, const uint8_t* code_sig,
                                                                      const uint8_t* msg, size_t msg_len, size_t nwit, size_t nwit_padded, fp* inputs, uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= nwit_padded) return;
    bool live = i < nwit; uint8_t st = ST_OK;
    if (live) { for (size_t k = 0; k < n; k++) if (code_key[i * n + k] != DEC_OK) { st = ST_BAD_PK; break; } if (st == ST_OK && code_sig[i] != DEC_OK) st = ST_BAD_SIG; }
    bool ok = live && st == ST_OK;
    fp zero = fp_zero();
    for (size_t k = 0; k < n; k++) {
        g1_aff pk; if (ok) soa_load_g1(pk, key_soa, nwit * n, i * n + k);
        inputs[(2 * k) * nwit_padded + i] = ok ? fp_from_mont(pk.x) : zero; inputs[(2 * k + 1) * nwit_padded + i] = ok ? fp_from_mont(pk.y) : zero;
        fp b = zero; if (ok) b.l[0] = bitmap[i * n + k] ? 1u : 0u; inputs[(2 * n + k) * nwit_padded + i] = b;
    }
    g2_aff sg; if (ok) soa_load_g2(sg, sig_soa, nwit, i);
    inputs[(3 * n + 0) * nwit_padded + i] = ok ? fp_from_mont(sg.x.c0) : zero; inputs[(3 * n + 1) * nwit_padded + i] = ok ? fp_from_mont(sg.x.c1) : zero;
    inputs[(3 * n + 2) * nwit_padded + i] = ok ? fp_from_mont(sg.y.c0) : zero; inputs[(3 * n + 3) * nwit_padded + i] = ok ? fp_from_mont(sg.y.c1) : zero;
    for (size_t k = 0; k < 8 * msg_len; k++) { fp b = zero; if (ok) b.l[0] = (msg[msg_len * i + (k >> 3)] >> (k & 7)) & 1u; inputs[(3 * n + 4 + k) * nwit_padded + i] = b; }
    if (live && status) status[i] = st;
}
// transposed group -> z[w][col] (48-byte LE canonical), the layout of blsgpu_r1cs_check
__global__ void __launch_bounds__(256) k_witness_untranspose(const u32x4* zt_all, const uint2* zbool_all, size_t ncols, size_t nout, size_t nwit, u32x4* z) {
    size_t col = blockIdx.x * (size_t)8 + (threadIdx.x >> 5); int lane = threadIdx.x & 31; size_t group = blockIdx.y;
    size_t w = group * 32 + lane;
    if (col >= nout || w >= nwit) return;
    const u32x4* zt = zt_all + group * ncols * 96;
    u32x4* dst = z + (w * nout + col) * 3;
    if (zbool_all) {                                          // a 0/1 column exists only as its packed word
        uint2 f = zbool_all[group * ncols + col];
        if (f.y) { u32x4 v; v.x = (f.x >> lane) & 1u; v.y = v.z = v.w = 0; u32x4 zero; zero.x = zero.y = zero.z = zero.w = 0; dst[0] = v; dst[1] = zero; dst[2] = zero; return; }
    }
    dst[0] = zt[(col * 3) * 32 + lane]; dst[1] = zt[(col * 3 + 1) * 32 + lane]; dst[2] = zt[(col * 3 + 2) * 32 + lane];
}

static void wit_release(wit_prog* p) {
    cudaFree(p->rules); cudaFree(p->lc_ptr); cudaFree(p->col); cudaFree(p->coeff); cudaFree(p->coeffc); cudaFree(p->cls);
    cudaFree(p->xrules); cudaFree(p->level_ptr); cudaFree(p->lrules); cudaFree(p->llevel_ptr); cudaFree(p->lt_col); cudaFree(p->lt_coef);
    delete p;
}

extern "C" {
// Splits the level-ordered program into its light part (wit_lrule records by light level) and its heavy part (wit_xrule records re-levelled with
// every light column at level 0).  Walks the rules in the given level order, so operands are classified before their users.
struct wit_split { std::vector<wit_lrule> lrules; std::vector<uint32_t> llevel_ptr, lt_col; std::vector<long long> lt_coef; size_t n_islots = 0;
                   std::vector<wit_xrule> xrules; std::vector<uint64_t> hlevel_ptr; };
static bool wit_small_coef(const uint8_t* c48, long long& out) {            // canonical 48-byte LE -> signed integer when |c| < 2^48
    static const uint8_t PB[48] = {0xab, 0xaa, 0xff, 0xff, 0xff, 0xff, 0xfe, 0xb9, 0xff, 0xff, 0x53, 0xb1, 0xfe, 0xff, 0xab, 0x1e, 0x24, 0xf6, 0xb0, 0xf6, 0xa0, 0xd2, 0x30, 0x67,
                                   0xbf, 0x12, 0x85, 0xf3, 0x84, 0x4b, 0x77, 0x64, 0xd7, 0xac, 0x4b, 0x43, 0xb6, 0xa7, 0x1b, 0x4b, 0x9a, 0xe6, 0x7f, 0x39, 0xea, 0x11, 0x01, 0x1a};
    bool hi = false; for (int i = 6; i < 48; i++) hi |= c48[i] != 0;
    if (!hi) { long long v = 0; for (int i = 5; i >= 0; i--) v = (v << 8) | c48[i]; out = v; return true; }
    for (int i = 8; i < 48; i++) if (c48[i] != PB[i]) return false;          // p - c < 2^48 needs the upper bytes of p (a borrow can reach bytes 6, 7 only)
    unsigned long long lo = 0, pl = 0; for (int i = 7; i >= 0; i--) { lo = (lo << 8) | c48[i]; pl = (pl << 8) | PB[i]; }
    if (lo > pl) return false;
    unsigned long long d = pl - lo; if (d >= (1ull << 48)) return false;
    out = -(long long)d; return true;
}
static void wit_split_program(wit_split& S, const wit_rule* hr, const uint64_t* lc_ptr, const uint32_t* lc_col, const uint8_t* lc_coef48, size_t ncols, size_t nout,
                              const uint32_t* order, size_t nkeys, size_t ninputs) {
    enum : uint8_t { HEAVY = 0, LB = 1, LI = 2 };
    std::vector<uint8_t> state(ncols, HEAVY); std::vector<uint32_t> llev(ncols, 0), hlev(ncols, 0), islot(ncols, 0); std::vector<long long> vmin(ncols, 0), vmax(ncols, 0);
    std::vector<uint8_t> is_small; std::vector<long long> coef;              // decoded lazily per term
    auto lo_of = [&](uint32_t id) { return id ? lc_ptr[id - 1] : (uint64_t)0; }; auto hi_of = [&](uint32_t id) { return id ? lc_ptr[id] : (uint64_t)0; };
    size_t nterms = lc_ptr ? 0 : 0; (void)nterms;
    auto bool_input = [&](uint16_t slot) { return nkeys ? ((slot >= 2 * nkeys && slot < 3 * nkeys) || slot >= 3 * nkeys + 4) : slot >= WIT_POINT_INPUTS; };
    struct lrec { wit_lrule r; uint32_t level; }; std::vector<lrec> light; std::vector<uint32_t> heavy_vars;
    const __int128 LIM = (__int128)1 << 62;
    for (size_t oi = 0; oi < ncols; oi++) {
        uint32_t v = order[oi]; const wit_rule& r = hr[v];
        wit_lrule lr; memset(&lr, 0, sizeof lr); lr.var = v; lr.aux = r.aux; for (int k = 0; k < 6; k++) lr.a[k] = WL_NO_COL;
        bool is_light = false; uint32_t level = 0;
        if (r.kind == WR_INPUT) {
            if (r.aux == 0xffff) { lr.kind = WL_ONE; state[v] = LB; is_light = true; }
            else if ((size_t)r.aux < ninputs && bool_input(r.aux)) { lr.kind = WL_INPUT; state[v] = LB; is_light = true; }
        } else if (r.kind == WR_MULADD || r.kind == WR_BIT) {
            // gather the terms; every column must be light and every coefficient a small integer
            uint32_t ids[3] = {r.a, r.kind == WR_BIT ? 0u : r.b, r.kind == WR_BIT ? 0u : r.d}; bool ok = true; uint32_t mx = 0;
            struct term { uint32_t col; long long k; int which; }; std::vector<term> ts;
            for (int q = 0; q < 3 && ok; q++) for (uint64_t t = lo_of(ids[q]); t < hi_of(ids[q]); t++) {
                uint32_t c = lc_col[t]; long long k;
                if (state[c] == HEAVY || !wit_small_coef(lc_coef48 + 48 * t, k)) { ok = false; break; }
                ts.push_back({c, k, q}); if (llev[c] > mx) mx = llev[c];
            }
            if (ok) {
                level = mx + 1;
                if (r.kind == WR_MULADD && !r.a && r.b) ok = false;                   // (never recorded: a rule without a first factor has no second one)
                if (!ok) { }
                else if (r.kind == WR_MULADD && r.a) {                            // product rule: a truth table over <= 5 distinct 0/1 columns
                    uint32_t cs[5]; int d = 0; bool fits = true;
                    for (auto& t : ts) { if (state[t.col] != LB) { fits = false; break; } if (t.col == 0) continue;      // column 0 is the constant 1 (the replay writes it), not a table input
                                         int j = 0; while (j < d && cs[j] != t.col) j++; if (j == d) { if (d == 5) { fits = false; break; } cs[d++] = t.col; } }
                    if (fits && d == 0) { cs[d++] = 0; }                                              // a product of constants: a one-input table on column 0
                    if (fits) {
                        uint32_t table = 0; bool boolean = true;
                        for (uint32_t idx = 0; idx < 32 && boolean; idx++) {
                            __int128 s[3] = {0, 0, 0};
                            for (auto& t : ts) { if (t.col == 0) { s[t.which] += t.k; continue; } int j = 0; while (cs[j] != t.col) j++; if ((idx >> j) & 1) s[t.which] += t.k; }
                            __int128 val = s[0] * s[1] + s[2];
                            if (val == 1) table |= 1u << idx; else if (val != 0) boolean = false;
                        }
                        if (boolean) { lr.kind = WL_LUT; for (int j = 0; j < d; j++) lr.a[j] = cs[j]; lr.a[5] = table; state[v] = LB; is_light = true; }
                    }
                } else {                                                           // a sum (MULADD with d only) or a bit of a sum
                    __int128 mn = 0, mxv = 0;
                    for (auto& t : ts) { __int128 a = t.col == 0 ? 1 : state[t.col] == LB ? 0 : vmin[t.col], b = state[t.col] == LB ? 1 : vmax[t.col]; __int128 x = a * t.k, y = b * t.k; mn += x < y ? x : y; mxv += x < y ? y : x; }
                    bool range_ok = mn > -LIM && mxv < LIM && ts.size() < (1u << 20);
                    if (range_ok && (r.kind == WR_MULADD || (mn >= 0 && r.aux < 63))) {
                        lr.kind = r.kind == WR_BIT ? WL_BIT : WL_SUM; lr.a[0] = (uint32_t)S.lt_col.size();
                        for (auto& t : ts) { S.lt_col.push_back(state[t.col] == LI ? (WL_INT | islot[t.col]) : t.col); S.lt_coef.push_back(t.k); }
                        lr.a[1] = (uint32_t)S.lt_col.size(); is_light = true;
                        if (r.kind == WR_BIT || (mn >= 0 && mxv <= 1)) { state[v] = LB; if (r.kind == WR_MULADD) lr.flags |= 1; }
                        else { state[v] = LI; vmin[v] = (long long)mn; vmax[v] = (long long)mxv; islot[v] = (uint32_t)S.n_islots; lr.a[2] = (uint32_t)S.n_islots++; if (v < nout) lr.flags |= 2; }
                    }
                }
            }
        }
        if (is_light) { llev[v] = level; light.push_back({lr, level}); }
        else heavy_vars.push_back(v);
    }
    // heavy rules: levels among themselves (light columns sit at level 0), integers they read are exported as field elements
    std::vector<uint8_t> export_int(ncols, 0); uint32_t hmax = 0;
    auto scan = [&](uint32_t id, uint32_t& m) { for (uint64_t t = lo_of(id); t < hi_of(id); t++) { uint32_t c = lc_col[t]; if (state[c] == LI) export_int[c] = 1; if (state[c] == HEAVY && hlev[c] > m) m = hlev[c]; } };
    for (uint32_t v : heavy_vars) {
        const wit_rule& r = hr[v]; uint32_t m = 0;
        if (r.kind == WR_INPUT) { hlev[v] = 0; continue; }
        if (r.kind == WR_FP12INV) { for (uint32_t k = 0; k < 12; k++) scan(r.a + k, m); } else { scan(r.a, m); scan(r.b, m); scan(r.d, m); }
        hlev[v] = m + 1; if (hlev[v] > hmax) hmax = hlev[v];
    }
    for (auto& l : light) if (l.r.kind == WL_SUM && !(l.r.flags & 1) && export_int[l.r.var]) l.r.flags |= 2;
    // light records by level, truth-table rules first inside a level
    uint32_t lmax = 0; for (auto& l : light) if (l.level > lmax) lmax = l.level;
    size_t nl = light.empty() ? 0 : (size_t)lmax + 1;
    std::vector<uint32_t> cnt(2 * nl + 1, 0);
    for (auto& l : light) cnt[2 * l.level + (l.r.kind == WL_LUT ? 0 : 1) + 1]++;
    for (size_t i = 0; i < 2 * nl; i++) cnt[i + 1] += cnt[i];
    S.llevel_ptr = cnt; S.lrules.resize(light.size());
    { std::vector<uint32_t> pos(cnt.begin(), cnt.end() - 1); for (auto& l : light) S.lrules[pos[2 * l.level + (l.r.kind == WL_LUT ? 0 : 1)]++] = l.r; }
    size_t nh = (size_t)hmax + 1; std::vector<uint64_t> hc(nh + 1, 0);
    for (uint32_t v : heavy_vars) hc[hlev[v] + 1]++;
    for (size_t i = 0; i < nh; i++) hc[i + 1] += hc[i];
    S.hlevel_ptr = hc; S.xrules.resize(heavy_vars.size());
    { std::vector<uint64_t> pos(hc.begin(), hc.end() - 1);
      for (uint32_t v : heavy_vars) {
          const wit_rule& r = hr[v]; wit_xrule& x = S.xrules[pos[hlev[v]]++];
          x.kind = r.kind; x.pad = 0; x.aux = r.aux; x.var = v;
          if (r.kind == WR_FP12INV) { x.a_lo = r.a; x.a_hi = r.a + 12; x.b_lo = x.b_hi = x.d_lo = x.d_hi = 0; }
          else { x.a_lo = (uint32_t)lo_of(r.a); x.a_hi = (uint32_t)hi_of(r.a); x.b_lo = (uint32_t)lo_of(r.b); x.b_hi = (uint32_t)hi_of(r.b); x.d_lo = (uint32_t)lo_of(r.d); x.d_hi = (uint32_t)hi_of(r.d); }
      } }
}
static int witness_load_impl(blsgpu_ctx* ctx, const uint8_t* rules16, const uint64_t* lc_ptr, const uint32_t* lc_col, const uint8_t* lc_coef48, size_t nvars, size_t nout, size_t nlc, size_t nterms,
                             const uint32_t* order, const uint64_t* level_ptr, size_t nlevels, size_t nkeys, int* handle) {
    if (!rules16 || !lc_ptr || !lc_col || !lc_coef48 || !handle || !nvars || !nout || nout > nvars) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    if (ctx->ptr_mode != BLSGPU_HOST) return fail(ctx, BLSGPU_ERR_ARG, "blsgpu_witness_load takes host pointers (the level-ordered rule tables are built on the host)");
    int h = -1; for (int i = 0; i < 4; i++) if (!ctx->wit[i]) { h = i; break; }
    if (h < 0) return fail(ctx, BLSGPU_ERR_ARG, "too many witness programs loaded");
    wit_prog* p = new (std::nothrow) wit_prog(); if (!p) return fail(ctx, BLSGPU_ERR_ALLOC, "out of host memory");
    memset(p, 0, sizeof *p); p->nvars = nvars; p->nout = nout; p->nlc = nlc; p->nterms = nterms;
    struct guard_t { wit_prog* p; ~guard_t() { if (p) wit_release(p); } } undo{p};          // a failed load leaves nothing behind
    const wit_rule* hr = reinterpret_cast<const wit_rule*>(rules16);
    {   // input slots: verify circuit 0..5 the points, 6 + 8 i + b the message bits; aggregate_verify circuit [0, 2n) keys, [2n, 3n) bitmap bits, [3n, 3n + 4) signature, message bits
        size_t top = 0;
        for (size_t k = 0; k < nvars; k++) if (hr[k].kind == WR_INPUT && hr[k].aux != 0xffff && (size_t)hr[k].aux + 1 > top) top = (size_t)hr[k].aux + 1;
        size_t fixed = nkeys ? 3 * nkeys + 4 : WIT_POINT_INPUTS;
        if (top < fixed || (top - fixed) % 8) return fail(ctx, BLSGPU_ERR_ARG, "witness program: %zu input slots is not %zu + 8 x message bytes%s", top, fixed, nkeys ? "" : " (an aggregate_verify program is loaded with blsgpu_witness_load_aggregate)");
        p->ninputs = top; p->nkeys = nkeys; p->msg_len = (top - fixed) / 8;
    }
    size_t nt = nterms ? nterms : 1;
    CU(cudaMalloc(&p->rules, 16 * nvars)); CU(cudaMalloc(&p->lc_ptr, 8 * (nlc + 1))); CU(cudaMalloc(&p->col, 4 * nt));
    CU(cudaMalloc(&p->coeff, 48 * nt)); CU(cudaMalloc(&p->coeffc, 48 * nt)); CU(cudaMalloc(&p->cls, nt));
    CU(cudaMemcpyAsync(p->rules, rules16, 16 * nvars, cudaMemcpyHostToDevice, ctx->stream)); CU(cudaMemcpyAsync(p->lc_ptr, lc_ptr, 8 * (nlc + 1), cudaMemcpyHostToDevice, ctx->stream));
    if (nterms) {
        CU(cudaMemcpyAsync(p->col, lc_col, 4 * nterms, cudaMemcpyHostToDevice, ctx->stream));
        dev_tmp raw; CU(cudaMalloc(&raw.p, 48 * nterms));
        CU(cudaMemcpyAsync(raw.p, lc_coef48, 48 * nterms, cudaMemcpyHostToDevice, ctx->stream));
        LAUNCH(k_r1cs_prepare, nblk(nterms), TPB, (const uint8_t*)raw.p, nterms, p->coeff, p->coeffc, p->cls);
        CU(cudaStreamSynchronize(ctx->stream));
    }
    if (order && level_ptr && nlevels) {                   // level-synchronous replay: light part + heavy part
        wit_split S; wit_split_program(S, hr, lc_ptr, lc_col, lc_coef48, nvars, nout, order, nkeys, p->ninputs);
        p->nlevels = S.hlevel_ptr.size() - 1; p->n_light = S.lrules.size(); p->n_llevels = S.llevel_ptr.size() / 2; p->n_islots = S.n_islots; p->n_lterms = S.lt_col.size();
        size_t nx = S.xrules.size() ? S.xrules.size() : 1, nlr = S.lrules.size() ? S.lrules.size() : 1, nlt = S.lt_col.size() ? S.lt_col.size() : 1;
        CU(cudaMalloc(&p->xrules, sizeof(wit_xrule) * nx)); CU(cudaMalloc(&p->level_ptr, 8 * S.hlevel_ptr.size()));
        CU(cudaMalloc(&p->lrules, sizeof(wit_lrule) * nlr)); CU(cudaMalloc(&p->llevel_ptr, 4 * (S.llevel_ptr.size() ? S.llevel_ptr.size() : 1)));
        CU(cudaMalloc(&p->lt_col, 4 * nlt)); CU(cudaMalloc(&p->lt_coef, 8 * nlt));
        if (S.xrules.size()) CU(cudaMemcpyAsync(p->xrules, S.xrules.data(), sizeof(wit_xrule) * S.xrules.size(), cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(p->level_ptr, S.hlevel_ptr.data(), 8 * S.hlevel_ptr.size(), cudaMemcpyHostToDevice, ctx->stream));
        if (S.lrules.size()) CU(cudaMemcpyAsync(p->lrules, S.lrules.data(), sizeof(wit_lrule) * S.lrules.size(), cudaMemcpyHostToDevice, ctx->stream));
        if (S.llevel_ptr.size()) CU(cudaMemcpyAsync(p->llevel_ptr, S.llevel_ptr.data(), 4 * S.llevel_ptr.size(), cudaMemcpyHostToDevice, ctx->stream));
        if (S.lt_col.size()) { CU(cudaMemcpyAsync(p->lt_col, S.lt_col.data(), 4 * S.lt_col.size(), cudaMemcpyHostToDevice, ctx->stream)); CU(cudaMemcpyAsync(p->lt_coef, S.lt_coef.data(), 8 * S.lt_coef.size(), cudaMemcpyHostToDevice, ctx->stream)); }
        CU(cudaStreamSynchronize(ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    undo.p = nullptr; ctx->wit[h] = p; *handle = h; return 0;
}
int blsgpu_witness_load(blsgpu_ctx* ctx, const uint8_t* rules16, const uint64_t* lc_ptr, const uint32_t* lc_col, const uint8_t* lc_coef48, size_t nvars, size_t nout, size_t nlc, size_t nterms,
                        const uint32_t* order, const uint64_t* level_ptr, size_t nlevels, int* handle) {
    ENTER(); return witness_load_impl(ctx, rules16, lc_ptr, lc_col, lc_coef48, nvars, nout, nlc, nterms, order, level_ptr, nlevels, 0, handle);
}
// the same for a program of the aggregate_verify circuit (src/constraints.rs:153-191) with nkeys public keys (blsgadget_aggregate_verify_program): its input
// slots are [0, 2n) key coordinates, [2n, 3n) bitmap bits, [3n, 3n + 4) the signature, then 8 bits per message byte
int blsgpu_witness_load_aggregate(blsgpu_ctx* ctx, const uint8_t* rules16, const uint64_t* lc_ptr, const uint32_t* lc_col, const uint8_t* lc_coef48, size_t nvars, size_t nout, size_t nlc, size_t nterms,
                                  const uint32_t* order, const uint64_t* level_ptr, size_t nlevels, size_t nkeys, int* handle) {
    ENTER(); if (!nkeys) return fail(ctx, BLSGPU_ERR_ARG, "nkeys must be positive"); return witness_load_impl(ctx, rules16, lc_ptr, lc_col, lc_coef48, nvars, nout, nlc, nterms, order, level_ptr, nlevels, nkeys, handle);
}
// bytes per message of the circuit the loaded program was recorded for (blsgpu_witness_gen / _check take nwit x that many message bytes)
long blsgpu_witness_msg_len(blsgpu_ctx* ctx, int handle) { return (!ctx || handle < 0 || handle >= 4 || !ctx->wit[handle]) ? -1 : (long)ctx->wit[handle]->msg_len; }
// rule counts of a loaded program: counts[0] light rules, [1] light levels, [2] heavy (field) levels, [3] integer slots
int blsgpu_witness_shape(blsgpu_ctx* ctx, int handle, uint64_t counts[4]) {
    if (!ctx || handle < 0 || handle >= 4 || !ctx->wit[handle] || !counts) return BLSGPU_ERR_ARG;
    const wit_prog* p = ctx->wit[handle]; counts[0] = p->n_light; counts[1] = p->n_llevels; counts[2] = p->nlevels; counts[3] = p->n_islots; return 0;
}
int blsgpu_witness_free(blsgpu_ctx* ctx, int handle) {
    if (!ctx || handle < 0 || handle >= 4 || !ctx->wit[handle]) return BLSGPU_ERR_ARG;
    dev_guard guard_; cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream);
    wit_release(ctx->wit[handle]); ctx->wit[handle] = nullptr; return 0;
}
}
// decode, input slots and the level-synchronous replay for nwit triples: leaves the assignments in the transposed group layout
// (group stride nvars * 96 u32x4) in the workspace; `extra` bytes of workspace are reserved for the caller's own buffers, which it
// takes AFTER this returns.  want_zbool: also the packed 0/1 view per (group, variable).
// bitmap == NULL: verify program (pk48 = nwit keys); else aggregate program (pk48 = nwit x p.nkeys keys, bitmap = nwit x p.nkeys bytes)
static int witness_run(blsgpu_ctx* ctx, const wit_prog& p, const uint8_t* pk48, const uint8_t* bitmap, const uint8_t* msg, const uint8_t* sig96, size_t nwit, uint8_t* status, size_t extra,
                       bool want_zbool, u32x4** zt_out, uint2** zbool_out, uint8_t** dstatus_out) {
    if ((bitmap != nullptr) != (p.nkeys != 0)) return fail(ctx, BLSGPU_ERR_ARG, p.nkeys ? "this is an aggregate_verify program: use the _aggregate entry points" : "this is a verify program: use blsgpu_witness_gen / _check");
    size_t groups = (nwit + 31) / 32, np = groups * 32, ninputs = p.ninputs, nk = p.nkeys ? p.nkeys : 1, nkeys_total = nwit * nk;
    if (int rc = ws_reserve(ctx, al(48 * nkeys_total) + al(nkeys_total) + al(96 * nwit) + al(p.msg_len * nwit + 1) + al(96 * nkeys_total) + al(192 * nwit) + 2 * al(np) + al(nkeys_total + np) + al(48 * ninputs * np) + al(groups * p.nvars * 1536) +
                                 (want_zbool ? al(groups * p.nvars * 8) : 0) + al(groups * (p.n_islots + 1) * 256) + extra + 65536)) return rc;
    const uint8_t *dpk, *dsig, *dmsg, *dbm = nullptr;
    if (int rc = stage_in(ctx, dpk, pk48, 48 * nkeys_total)) return rc;
    if (bitmap) { if (int rc = stage_in(ctx, dbm, bitmap, nkeys_total)) return rc; }
    if (int rc = stage_in(ctx, dsig, sig96, 96 * nwit)) return rc;
    if (int rc = stage_in(ctx, dmsg, msg, p.msg_len * nwit ? p.msg_len * nwit : 1)) return rc;
    u32x4* pk_soa = ws_take<u32x4>(ctx, 6 * nkeys_total); u32x4* sig_soa = ws_take<u32x4>(ctx, 12 * nwit);
    uint8_t* code_pk = ws_take<uint8_t>(ctx, nkeys_total + np); uint8_t* code_sig = ws_take<uint8_t>(ctx, np);
    uint8_t* dstatus = status ? stage_out(ctx, status, nwit) : nullptr;
    fp* inputs = ws_take<fp>(ctx, ninputs * np);
    u32x4* zt_all = ws_take<u32x4>(ctx, groups * p.nvars * 96);
    uint2* zbool_all = want_zbool ? ws_take<uint2>(ctx, groups * p.nvars) : nullptr;
    long long* sint_all = ws_take<long long>(ctx, groups * (p.n_islots + 1) * 32);
    LAUNCH(k_decode_g1, nblk(nkeys_total), TPB, dpk, nkeys_total, pk_soa, code_pk);
    LAUNCH(k_decode_g2<true>, nblk(nwit), TPB, dsig, nwit, sig_soa, code_sig);
    if (bitmap) LAUNCH(k_witness_inputs_agg, nblk(np), TPB, (const u32x4*)pk_soa, (const uint8_t*)code_pk, p.nkeys, dbm, (const u32x4*)sig_soa, (const uint8_t*)code_sig, dmsg, p.msg_len, nwit, np, inputs, dstatus);
    else LAUNCH(k_witness_inputs, nblk(np), TPB, (const u32x4*)pk_soa, (const uint8_t*)code_pk, (const u32x4*)sig_soa, (const uint8_t*)code_sig, dmsg, p.msg_len, nwit, np, inputs, dstatus);
    if (p.xrules && !want_zbool) return fail(ctx, BLSGPU_ERR_ARG, "the level-synchronous replay works on the packed 0/1 view");
    if (p.xrules && p.n_light) LAUNCH(k_witness_light, (unsigned)groups, WIT_LIGHT_TPB, p, (const fp*)inputs, np, zt_all, zbool_all, sint_all);      // 0/1 and small-integer rules first
    if (p.xrules && ctx->wit_cluster) {                    // level-synchronous per group, hardware cluster barrier between levels
        cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3((unsigned)(groups * WIT_CL)); cfg.blockDim = dim3(WIT_CL_TPB); cfg.stream = ctx->stream;
        cudaLaunchAttribute at[1]; at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = WIT_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        wit_prog pc = p; const fp* in_c = inputs;
        CU(cudaLaunchKernelEx(&cfg, k_witness_cluster, pc, in_c, np, zt_all, groups, zbool_all)); ctx->launches++;
    } else if (p.xrules) {                                 // level-synchronous over the whole grid, cooperative launch: every block must be resident
        int per_sm = 0, sms = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_witness_levels, WIT_TPB, 0)); if (per_sm > WIT_BPS) per_sm = WIT_BPS; CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
        if (per_sm < 1) return fail(ctx, BLSGPU_ERR_CUDA, "k_witness_levels does not fit on an SM");
        wit_prog pc = p; const fp* in_c = inputs; void* args[] = {(void*)&pc, (void*)&in_c, (void*)&np, (void*)&zt_all, (void*)&groups, (void*)&zbool_all};
        CU(cudaLaunchCooperativeKernel((void*)k_witness_levels, dim3((unsigned)(per_sm * sms)), dim3(WIT_TPB), args, 0, ctx->stream)); ctx->launches++;
    } else {
        if (p.nvars != p.nout || want_zbool) return fail(ctx, BLSGPU_ERR_ARG, "the sequential replay needs a program without scratch columns (load it with its level order)");
        LAUNCH(k_witness_gen, (unsigned)groups, 32, p, (const fp*)inputs, np, zt_all);
    }
    *zt_out = zt_all; if (zbool_out) *zbool_out = zbool_all; *dstatus_out = dstatus;
    return 0;
}
extern "C" {
// assignments of the verify circuit for nwit (pk48, msg, sig96) triples: z48 = nwit * nout * 48 bytes (the layout of
// blsgpu_r1cs_check), status[i] = 0, or 2 / 3 when the key / signature does not decode to a non-identity point (its assignment
// is then all zeros except z[0] = 1 and the constants).  Pointers follow the context's pointer mode.
static int witness_gen_core(blsgpu_ctx* ctx, int handle, const uint8_t* pk48, const uint8_t* bitmap, const uint8_t* msg, const uint8_t* sig96, size_t nwit, uint8_t* z48, uint8_t* status) {
    if (handle < 0 || handle >= 4 || !ctx->wit[handle] || !pk48 || !msg || !sig96 || !z48) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    if (!nwit) return 0;
    wit_prog p = *ctx->wit[handle];
    size_t groups = (nwit + 31) / 32;
    bool host = ctx->ptr_mode == BLSGPU_HOST;
    size_t zbytes = nwit * p.nout * 48;
    u32x4* zt_all; uint2* zbool_all = nullptr; uint8_t* dstatus;
    if (int rc = witness_run(ctx, p, pk48, bitmap, msg, sig96, nwit, status, host ? al(zbytes) : 0, p.xrules != nullptr, &zt_all, &zbool_all, &dstatus)) return rc;
    uint8_t* dz = host ? ws_take<uint8_t>(ctx, zbytes) : z48;
    { dim3 grid(nblk(p.nout, 8), (unsigned)groups); k_witness_untranspose<<<grid, 256, 0, ctx->stream>>>((const u32x4*)zt_all, (const uint2*)zbool_all, p.nvars, p.nout, nwit, (u32x4*)dz); ctx->launches++; CU(cudaGetLastError()); }
    if (host) CU(cudaMemcpyAsync(z48, dz, zbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (status) { if (int rc = finish_out(ctx, status, dstatus, nwit)) return rc; }
    return finish_call(ctx);
}
// Generation and satisfaction check in one call: the assignments never leave the transposed group layout (no 48-byte row-major
// copy, no second transpose; 34 MB per assignment stay out of the caller's memory).  sat_bits / all_sat as blsgpu_r1cs_check,
// status as blsgpu_witness_gen; the R1CS system must be the one the program was recorded with (same column count).
static int witness_check_core(blsgpu_ctx* ctx, int wit_handle, int r1cs_handle, const uint8_t* pk48, const uint8_t* bitmap, const uint8_t* msg, const uint8_t* sig96, size_t nwit,
                              uint64_t* sat_bits, uint8_t* all_sat, uint8_t* status) {
    if (wit_handle < 0 || wit_handle >= 4 || !ctx->wit[wit_handle] || r1cs_handle < 0 || r1cs_handle >= 16 || !ctx->r1cs[r1cs_handle] || !pk48 || !msg || !sig96 || !sat_bits)
        return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    if (!nwit) return 0;
    wit_prog p = *ctx->wit[wit_handle]; r1cs_sys s = *ctx->r1cs[r1cs_handle];
    if (p.nout != s.ncols) return fail(ctx, BLSGPU_ERR_ARG, "witness program and R1CS system have different column counts");
    if (!p.xrules) return fail(ctx, BLSGPU_ERR_ARG, "blsgpu_witness_check needs a program loaded with its level order");
    size_t groups = (nwit + 31) / 32, words = (s.nrows + 63) / 64, part_bytes = R1_LONG_ROWS ? 64 : (s.n_seg ? s.n_seg : 1) * 32 * 48;
    bool host = ctx->ptr_mode == BLSGPU_HOST;
    u32x4* zt_all; uint2* zbool_all; uint8_t* dstatus;
    if (int rc = witness_run(ctx, p, pk48, bitmap, msg, sig96, nwit, status, al(part_bytes) + (host ? al(8 * words * nwit) + al(nwit) : 0), true, &zt_all, &zbool_all, &dstatus)) return rc;
    u32x4* part = ws_take<u32x4>(ctx, part_bytes / 16);
    uint64_t* dbits = host ? ws_take<uint64_t>(ctx, words * nwit) : sat_bits;
    uint8_t* dall = all_sat ? (host ? ws_take<uint8_t>(ctx, nwit) : all_sat) : nullptr;
    CU(cudaMemsetAsync(dbits, 0, 8 * words * nwit, ctx->stream));
    for (size_t gi = 0; gi < groups; gi++) {
        size_t w0 = gi * 32, g = nwit - w0 < 32 ? nwit - w0 : 32;
        if (int rc = r1cs_check_group(ctx, s, zt_all + gi * p.nvars * 96, zbool_all + gi * p.nvars, part, w0, g, words, dbits)) return rc;
    }
    if (dall) LAUNCH(k_r1cs_all, nblk(nwit, 8), 256, (const uint64_t*)dbits, nwit, words, s.nrows, dall);
    if (host) {
        CU(cudaMemcpyAsync(sat_bits, dbits, 8 * words * nwit, cudaMemcpyDeviceToHost, ctx->stream));
        if (all_sat) CU(cudaMemcpyAsync(all_sat, dall, nwit, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (status) { if (int rc = finish_out(ctx, status, dstatus, nwit)) return rc; }
    return finish_call(ctx);
}
int blsgpu_witness_gen(blsgpu_ctx* ctx, int handle, const uint8_t* pk48, const uint8_t* msg, const uint8_t* sig96, size_t nwit, uint8_t* z48, uint8_t* status) {
    ENTER(); return witness_gen_core(ctx, handle, pk48, nullptr, msg, sig96, nwit, z48, status);
}
int blsgpu_witness_check(blsgpu_ctx* ctx, int wit_handle, int r1cs_handle, const uint8_t* pk48, const uint8_t* msg, const uint8_t* sig96, size_t nwit,
                         uint64_t* sat_bits, uint8_t* all_sat, uint8_t* status) {
    ENTER(); return witness_check_core(ctx, wit_handle, r1cs_handle, pk48, nullptr, msg, sig96, nwit, sat_bits, all_sat, status);
}
// the aggregate_verify circuit (src/constraints.rs:153-191; program from blsgadget_aggregate_verify_program, loaded with blsgpu_witness_load_aggregate):
// pks48 = nwit x nkeys compressed keys, bitmap = nwit x nkeys bytes (0 / non-zero: the participation bits), msg = nwit x L bytes, sig96 = nwit
// aggregate signatures.  status: 2 when any of an item's keys does not decode to a non-identity point (masked-out keys are witnesses too), 3 for the signature.
int blsgpu_witness_gen_aggregate(blsgpu_ctx* ctx, int handle, const uint8_t* pks48, const uint8_t* bitmap, const uint8_t* msg, const uint8_t* sig96, size_t nwit, uint8_t* z48, uint8_t* status) {
    ENTER(); if (!bitmap) return fail(ctx, BLSGPU_ERR_ARG, "null bitmap"); return witness_gen_core(ctx, handle, pks48, bitmap, msg, sig96, nwit, z48, status);
}
int blsgpu_witness_check_aggregate(blsgpu_ctx* ctx, int wit_handle, int r1cs_handle, const uint8_t* pks48, const uint8_t* bitmap, const uint8_t* msg, const uint8_t* sig96, size_t nwit,
                                   uint64_t* sat_bits, uint8_t* all_sat, uint8_t* status) {
    ENTER(); if (!bitmap) return fail(ctx, BLSGPU_ERR_ARG, "null bitmap"); return witness_check_core(ctx, wit_handle, r1cs_handle, pks48, bitmap, msg, sig96, nwit, sat_bits, all_sat, status);
}
}
