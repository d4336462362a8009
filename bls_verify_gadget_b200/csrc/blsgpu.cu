// libblsgpu: kernels + C ABI (include/blsgpu.h) of the B200-native BLS12-381 verify path.
// sm_100a only; no CPU fallback -- every entry point needs a CUDA device.
//
// Kernel inventory (one item per thread, 128-thread CTAs, grid = ceil(n/128) >> 148 SMs):
//   k_decode_g1 / k_decode_g2   K1  compressed bytes -> affine Montgomery limb-SoA + decode code | k_decode_g2<false>: no subgroup test (verify_batch, split form)
//   k_hash_to_g2                K2  message -> H(m) affine limb-SoA            | split form (default): k_hash_field -> k_hash_map (2n threads) -> k_hash_clear
//   k_miller                    K4  (pk, H(m), sig) -> Fp12 Miller value limb-SoA | split form: 8 x (k_miller_lines (2n threads) -> k_miller_accum);
//                                   in verify_batch the last pair of launches also tests sig in G2 on the running point [|x|] sig -> ST_BAD_SIG
//   k_final_exp                 K5  Fp12 -> GT, is_one -> status                   | split form: k_final_step<0>, 5 x (k_final_squarings -> k_final_step<k>)
//   k_miller_accum_coop, k_final_hard_coop   six lanes per item: passes of at most VERIFY_COOP_BELOW items (latency), blsgpu_set_coop
//   k_gt_reduce                 K5' strided product of GT values (per-batch accumulator)
//   k_status_bitmap                 status -> packed ok bitmap
//   k_segsum_g1 / k_segsum_g2   K3  warp-per-segment aggregation, tree reduction in shared memory
//   k_scalar_mul_g1 / _g2       K6  [sk]G1, [sk]H(m)
//   k_encode_g1 / k_encode_g2   K7  affine limb-SoA -> compressed bytes
//   k_fp_mul_raw, k_imad_peak   K0  parity hook and integer-multiply roofline microbenchmark
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <cstdarg>
#include <new>
#include <vector>
#include "stages.cuh"
#include "coop.cuh"
#include "../../include/blsgpu.h"

using namespace bls;

#ifndef BLS_TPB
#define BLS_TPB 128
#endif
#define TPB BLS_TPB
#define VERIFY_CHUNK_DEFAULT ((size_t)1 << 20)
#ifndef VERIFY_COOP_BELOW
#define VERIFY_COOP_BELOW 4096     // blsgpu_set_coop(ctx, 2): passes of at most this many items take the six-lane final exponentiation
#endif
#ifndef BLS_MINB
#define BLS_MINB 2      // resident 128-thread CTAs per SM the heavy kernels are compiled for (register cap = 65536 / (128 * BLS_MINB))
#endif
static inline unsigned nblk(size_t n, unsigned tpb = TPB) { return (unsigned)((n + tpb - 1) / tpb); }

// resident CTAs per SM of single kernels (register cap 65536 / (TPB * MINB)); BLS_MINB is the default for all stage kernels.  Measured at 2^20
// (profiles/r02_tuning.md): the two decoders gain 4 % / 2 % at 4 CTAs (128 registers), the compressed-squaring run 1 % at 3; k_hash_to_g2 loses 6 % at 3,
// its split forms k_hash_field / k_hash_map gain 1 % of the stage at 4 / 3.  k_decode_g2<false> (no subgroup test) takes 35.7 ms at 4 and 35.4 ms
// at 3 (152 registers, no spills), the step the same within its run-to-run spread (profiles/r03_sig_subgroup.md): both forms stay at 4.
#ifndef BLS_MINB_DG1
#define BLS_MINB_DG1 4
#endif
#ifndef BLS_MINB_DG2
#define BLS_MINB_DG2 4
#endif
#ifndef BLS_MINB_HASH
#define BLS_MINB_HASH BLS_MINB
#endif
#ifndef BLS_MINB_SQR
#define BLS_MINB_SQR 3
#endif
#ifndef BLS_MINB_HFIELD
#define BLS_MINB_HFIELD 4
#endif
#ifndef BLS_MINB_HMAP
#define BLS_MINB_HMAP 3
#endif
#ifndef BLS_MINB_LINES
#define BLS_MINB_LINES BLS_MINB
#endif
#ifndef BLS_MINB_HCLEAR
#define BLS_MINB_HCLEAR BLS_MINB
#endif
#ifndef BLS_MINB_ACCUM
#define BLS_MINB_ACCUM BLS_MINB
#endif
#ifndef MILLER_LINE_ITERS
#define MILLER_LINE_ITERS 8        // iterations per k_miller_lines / k_miller_accum pair
#define MILLER_LINE_STEPS 11       // most doubling + addition steps in 8 iterations (62..55 holds the additions of bits 62, 60, 57)
#endif

// Phase skew: the IMAD.WIDE pipe issues one warp instruction per 4 cycles per SM sub-partition and a single warp inside
// fp_mul saturates it; two warps that start together stay in lockstep (both in their IMAD phase, then both in their ALU
// phase), leaving each pipe idle half of the time.  Delaying every second warp of a sub-partition by about one phase at
// kernel entry moves the pair to the stable anti-phase schedule.  BLS_SKEW = delay in cycles (0 = off).
#ifndef BLS_F_IN_SMEM
#define BLS_F_IN_SMEM 0
#endif
#ifndef BLS_SKEW
#define BLS_SKEW 0
#endif
__device__ __forceinline__ void phase_skew() {
#if BLS_SKEW > 0
    if ((threadIdx.x >> 5) & 4) { long long t0 = clock64(); while (clock64() - t0 < BLS_SKEW) { } }
#endif
}
// ================================================================================================ kernels
__global__ void __launch_bounds__(TPB, BLS_MINB) k_fp_mul_raw(const fp* a, const fp* b, fp* out, size_t n, int reps) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    fp x = a[i], y = b[i];
    fp r = fp_mul(x, y);
    for (int k = 1; k < reps; k++) r = fp_mul(r, y);
    out[i] = r;
}
// independent IMAD.WIDE.U32 chains (mode 0) or mad.lo.cc/madc.hi.cc carry chains (mode 1); 16 MACs per inner step
__global__ void __launch_bounds__(256) k_imad_peak(uint32_t* sink, int iters, int mode) {
    uint32_t a = threadIdx.x * 2654435761u + 12345u, b = blockIdx.x * 40503u + 977u;
    if (mode == 0) {
        unsigned long long acc[16];
#pragma unroll
        for (int j = 0; j < 16; j++) acc[j] = (unsigned long long)j * 0x9e3779b97f4a7c15ull + a;
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int j = 0; j < 16; j++)      // the multiplicand changes every iteration (low half of another accumulator): nothing to strength-reduce
                asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[j]) : "r"((uint32_t)acc[(j + 5) & 15]), "r"(b));
        }
        unsigned long long s = 0;
#pragma unroll
        for (int j = 0; j < 16; j++) s ^= acc[j];
        if (s == 0x1234567ull) sink[0] = (uint32_t)s;
    } else {
        uint32_t e[16], o[16];
#pragma unroll
        for (int j = 0; j < 16; j++) { e[j] = a + j; o[j] = b + j; }
        for (int it = 0; it < iters; it++) {
            asm volatile(
                "mad.lo.cc.u32 %0, %16, %24, %0;\n\tmadc.hi.cc.u32 %1, %16, %24, %1;\n\tmadc.lo.cc.u32 %2, %17, %24, %2;\n\tmadc.hi.cc.u32 %3, %17, %24, %3;\n\t"
                "madc.lo.cc.u32 %4, %18, %24, %4;\n\tmadc.hi.cc.u32 %5, %18, %24, %5;\n\tmadc.lo.cc.u32 %6, %19, %24, %6;\n\tmadc.hi.cc.u32 %7, %19, %24, %7;\n\t"
                "madc.lo.cc.u32 %8, %20, %24, %8;\n\tmadc.hi.cc.u32 %9, %20, %24, %9;\n\tmadc.lo.cc.u32 %10, %21, %24, %10;\n\tmadc.hi.cc.u32 %11, %21, %24, %11;\n\t"
                "madc.lo.cc.u32 %12, %22, %24, %12;\n\tmadc.hi.cc.u32 %13, %22, %24, %13;\n\tmadc.lo.cc.u32 %14, %23, %24, %14;\n\tmadc.hi.u32 %15, %23, %24, %15;"
                : "+r"(e[0]), "+r"(e[1]), "+r"(e[2]), "+r"(e[3]), "+r"(e[4]), "+r"(e[5]), "+r"(e[6]), "+r"(e[7]), "+r"(e[8]), "+r"(e[9]), "+r"(e[10]), "+r"(e[11]), "+r"(e[12]), "+r"(e[13]), "+r"(e[14]), "+r"(e[15])
                : "r"(a), "r"(a + 1), "r"(a + 2), "r"(a + 3), "r"(a + 4), "r"(a + 5), "r"(a + 6), "r"(a + 7), "r"(o[3]));
            asm volatile(
                "mad.lo.cc.u32 %0, %16, %24, %0;\n\tmadc.hi.cc.u32 %1, %16, %24, %1;\n\tmadc.lo.cc.u32 %2, %17, %24, %2;\n\tmadc.hi.cc.u32 %3, %17, %24, %3;\n\t"
                "madc.lo.cc.u32 %4, %18, %24, %4;\n\tmadc.hi.cc.u32 %5, %18, %24, %5;\n\tmadc.lo.cc.u32 %6, %19, %24, %6;\n\tmadc.hi.cc.u32 %7, %19, %24, %7;\n\t"
                "madc.lo.cc.u32 %8, %20, %24, %8;\n\tmadc.hi.cc.u32 %9, %20, %24, %9;\n\tmadc.lo.cc.u32 %10, %21, %24, %10;\n\tmadc.hi.cc.u32 %11, %21, %24, %11;\n\t"
                "madc.lo.cc.u32 %12, %22, %24, %12;\n\tmadc.hi.cc.u32 %13, %22, %24, %13;\n\tmadc.lo.cc.u32 %14, %23, %24, %14;\n\tmadc.hi.u32 %15, %23, %24, %15;"
                : "+r"(o[0]), "+r"(o[1]), "+r"(o[2]), "+r"(o[3]), "+r"(o[4]), "+r"(o[5]), "+r"(o[6]), "+r"(o[7]), "+r"(o[8]), "+r"(o[9]), "+r"(o[10]), "+r"(o[11]), "+r"(o[12]), "+r"(o[13]), "+r"(o[14]), "+r"(o[15])
                : "r"(b), "r"(b + 1), "r"(b + 2), "r"(b + 3), "r"(b + 4), "r"(b + 5), "r"(b + 6), "r"(b + 7), "r"(e[5]));
        }
        uint32_t s = 0;
#pragma unroll
        for (int j = 0; j < 16; j++) s ^= e[j] ^ o[j];
        if (s == 0x12345u) sink[0] = s;
    }
}

__global__ void __launch_bounds__(TPB, BLS_MINB_DG1) k_decode_g1(const uint8_t* in48, size_t n, u32x4* soa, uint8_t* code) {
    phase_skew();
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g1_aff p; int rc = g1_decode(p, in48 + 48 * i);
    if (soa) soa_store_g1(soa, n, i, p);
    code[i] = (uint8_t)rc;
}
// SUBGROUP = false: on-curve decode only, for blsgpu_verify_batch's split path, whose Miller loop tests membership (k_miller_lines)
template <bool SUBGROUP> __global__ void __launch_bounds__(TPB, BLS_MINB_DG2) k_decode_g2(const uint8_t* in96, size_t n, u32x4* soa, uint8_t* code) {
    phase_skew();
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g2_aff p; int rc = g2_decode<SUBGROUP>(p, in96 + 96 * i);
    if (soa) soa_store_g2(soa, n, i, p);
    code[i] = (uint8_t)rc;
}
// status/flags from the two decode codes (bls.rs:434-447), then H(m) for the items still alive
__global__ void __launch_bounds__(TPB, BLS_MINB_HASH) k_hash_to_g2(const uint8_t* msg, const uint32_t* off, size_t n, const uint8_t* code_pk, const uint8_t* code_sig,
                                                    u32x4* hm_soa, uint8_t* flags, uint8_t* status) {
    phase_skew();
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    uint8_t st = ST_OK, fl = 0;
    if (code_pk) {
        if (code_pk[i] != DEC_OK) st = ST_BAD_PK;
        else if (code_sig[i] != DEC_OK && code_sig[i] != DEC_INF) st = ST_BAD_SIG;
        else if (code_sig[i] == DEC_INF) fl = FL_SIG_INF;
    }
    if (st == ST_OK) {
        const uint8_t* m; uint32_t len;
        if (off) { m = msg + off[i]; len = off[i + 1] - off[i]; } else { m = msg + 32 * i; len = 32; }
        g2_aff hm; uint8_t f2; stage_hash(hm, f2, m, len);
        soa_store_g2(hm_soa, n, i, hm); fl |= f2;
    }
    flags[i] = fl; if (status) status[i] = st;
}
// ---- hash-to-G2 of the verify path in three launches: SHA-256 / hash_to_field (small state), the two SSWU + isogeny maps with
// one field element per thread (2n threads), then the addition, cofactor clearing and the affine conversion.  Same status / flags rule as above.
__global__ void __launch_bounds__(TPB, BLS_MINB_HFIELD) k_hash_field(const uint8_t* msg, const uint32_t* off, size_t n, const uint8_t* code_pk, const uint8_t* code_sig,
                                                               u32x4* u_soa, uint8_t* flags, uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    uint8_t st = ST_OK, fl = 0;
    if (code_pk) {
        if (code_pk[i] != DEC_OK) st = ST_BAD_PK;
        else if (code_sig[i] != DEC_OK && code_sig[i] != DEC_INF) st = ST_BAD_SIG;
        else if (code_sig[i] == DEC_INF) fl = FL_SIG_INF;
    }
    if (st == ST_OK) {
        const uint8_t* m; uint32_t len;
        if (off) { m = msg + off[i]; len = off[i + 1] - off[i]; } else { m = msg + 32 * i; len = 32; }
        fp2 u0, u1; hash_to_field(u0, u1, m, len);
        soa_store_fp2(u_soa, n, i, 0, u0); soa_store_fp2(u_soa, n, i, 1, u1);
    }
    flags[i] = fl; if (status) status[i] = st;
}
// small passes hash every message while the two decoders run on other streams (verify_core, `forked`): the status / flags rule afterwards
__global__ void k_status_merge(const uint8_t* code_pk, const uint8_t* code_sig, size_t n, uint8_t* flags, uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    uint8_t st = ST_OK, fl = 0;
    if (code_pk[i] != DEC_OK) st = ST_BAD_PK;
    else if (code_sig[i] != DEC_OK && code_sig[i] != DEC_INF) st = ST_BAD_SIG;
    else if (code_sig[i] == DEC_INF) fl = FL_SIG_INF;
    flags[i] = (uint8_t)((flags[i] & FL_HM_INF) | fl); status[i] = st;
}
__global__ void __launch_bounds__(TPB, BLS_MINB_HMAP) k_hash_map(const u32x4* u_soa, const uint8_t* status, size_t n, u32x4* q_soa) {
    size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (t >= 2 * n) return;
    int j = t >= n; size_t i = t - (j ? n : 0);
    if (status && status[i] != ST_OK) return;
    fp2 u = soa_load_fp2(u_soa, n, i, j), xn, xd, y; g2_jac q;
    sswu_map(xn, xd, y, u); iso3_map(q, xn, xd, y);
    soa_store_fp2(q_soa, n, i, 3 * j, q.X); soa_store_fp2(q_soa, n, i, 3 * j + 1, q.Y); soa_store_fp2(q_soa, n, i, 3 * j + 2, q.Z);
}
__global__ void __launch_bounds__(TPB, BLS_MINB_HCLEAR) k_hash_clear(const u32x4* q_soa, const uint8_t* status, size_t n, u32x4* hm_soa, uint8_t* flags) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status && status[i] != ST_OK) return;
    g2_jac q0, q1, h; g2_aff hm;
    q0.X = soa_load_fp2(q_soa, n, i, 0); q0.Y = soa_load_fp2(q_soa, n, i, 1); q0.Z = soa_load_fp2(q_soa, n, i, 2);
    q1.X = soa_load_fp2(q_soa, n, i, 3); q1.Y = soa_load_fp2(q_soa, n, i, 4); q1.Z = soa_load_fp2(q_soa, n, i, 5);
    jac_add(q0, q0, q1); g2_clear_cofactor(h, q0);
    if (!jac_to_aff(hm, h)) flags[i] |= FL_HM_INF;
    soa_store_g2(hm_soa, n, i, hm);
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_miller(const u32x4* pk_soa, const u32x4* hm_soa, const u32x4* sig_soa, const uint8_t* flags,
                                                const uint8_t* status, size_t n, u32x4* f_soa) {
    phase_skew();
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status[i] != ST_OK) return;
    g1_aff pk; g2_aff hm, sig;
    soa_load_g1(pk, pk_soa, n, i); soa_load_g2(hm, hm_soa, n, i); soa_load_g2(sig, sig_soa, n, i);
#if BLS_F_IN_SMEM
    extern __shared__ uint4 f_smem[];                       // accumulator f in shared memory, 592-byte stride (conflict-free 128-bit accesses)
    fp12& f = *reinterpret_cast<fp12*>(f_smem + threadIdx.x * 37);
#else
    fp12 f;
#endif
    stage_miller(f, pk, hm, sig, flags[i]);
    soa_store_fp12(f_soa, n, i, f);
}
// ---- split forms of the long stages (blsgpu_set_split, default on): the same arithmetic as a sequence of short, specialised launches with the
// per-item state in global memory between them.  Two effects, both measured (profiles/r02_tuning.md): (1) a kernel that holds only the point
// arithmetic, or only the accumulator update, or only the compressed squarings has a smaller working set and less code than the one-launch
// stage kernel and runs faster (Miller 585 -> 505 ms, final exponentiation 389 -> 352 ms at 2^20); (2) a CTA of k_miller runs ~21 ms and one of
// k_final_exp ~14 ms, so a batch of a few waves (one GPU's shard of an 8-GPU job) loses a tenth of its time to the partly filled last wave of
// each: short launches make the tail short and give the other lane's kernels gaps to fill (+8 % at 2^17 items).
// Miller loop: the point arithmetic and the accumulation are separate kernels.  k_miller_lines runs the
// doubling / addition steps of ONE pair per thread (2n threads: small state, small code) for a range of iterations and leaves the line
// coefficients, already scaled by the G1 coordinates, in global memory; k_miller_accum squares f and multiplies the lines in (fp12_sqr and
// mul_by_014 only).  Line buffer: step s, pair j, coefficient k at rows ((2 s + j) * 3 + k) * 6 .. of an n-column limb-SoA matrix.
// sig_sub (nullable): the last launch (i_lo = 0) stores the signature's subgroup test there (1 = in G2) for every item with status ST_OK
// and a finite signature -- pair 0 ends on [|x|] sig (miller_end_in_subgroup) -- and the last k_miller_accum(_coop) folds it into the
// status.  Not status[] itself: the pair-1 thread of the same item reads that in this launch.
__global__ void __launch_bounds__(TPB, BLS_MINB_LINES) k_miller_lines(const u32x4* pk_soa, const u32x4* hm_soa, const u32x4* sig_soa, const uint8_t* flags, const uint8_t* status,
                                                                size_t n, u32x4* t_soa, u32x4* lines, int i_hi, int i_lo, uint8_t* sig_sub) {
    size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (t >= 2 * n) return;
    int j = t >= n; size_t i = t - (j ? n : 0);
    if (status[i] != ST_OK) return;
    if (flags[i] & (j ? FL_HM_INF : FL_SIG_INF)) return;
    g1_aff p; g2_aff q; g2_proj r;
    if (j) { soa_load_g1(p, pk_soa, n, i); soa_load_g2(q, hm_soa, n, i); } else { p.x = fp_const(C_G1X); p.y = fp_const(C_G1Y_NEG); soa_load_g2(q, sig_soa, n, i); }
    if (i_hi == 62) { r.x = q.x; r.y = q.y; r.z = fp2_one(); }
    else { r.x = soa_load_fp2(t_soa, n, i, 3 * j); r.y = soa_load_fp2(t_soa, n, i, 3 * j + 1); r.z = soa_load_fp2(t_soa, n, i, 3 * j + 2); }
    const uint64_t x = BLS_X_ABS; int s = 0; fp2 c0, c1, c2;
    for (int it = i_hi; it >= i_lo; it--) {
        miller_dbl(r, c0, c1, c2);
        { u32x4* L = lines + (size_t)(2 * s + j) * 18 * n; soa_store_fp2(L, n, i, 0, c0); soa_store_fp2(L, n, i, 1, fp2_mul_fp(c1, p.x)); soa_store_fp2(L, n, i, 2, fp2_mul_fp(c2, p.y)); s++; }
        if ((x >> it) & 1) {
            miller_add(r, q, c0, c1, c2);
            u32x4* L = lines + (size_t)(2 * s + j) * 18 * n; soa_store_fp2(L, n, i, 0, c0); soa_store_fp2(L, n, i, 1, fp2_mul_fp(c1, p.x)); soa_store_fp2(L, n, i, 2, fp2_mul_fp(c2, p.y)); s++;
        }
    }
    if (i_lo != 0) { soa_store_fp2(t_soa, n, i, 3 * j, r.x); soa_store_fp2(t_soa, n, i, 3 * j + 1, r.y); soa_store_fp2(t_soa, n, i, 3 * j + 2, r.z); }
    else if (j == 0 && sig_sub) sig_sub[i] = miller_end_in_subgroup(r, q) ? 1 : 0;
}
// sig_sub (nullable, see k_miller_lines): in the last launch an item whose signature failed the subgroup test gets ST_BAD_SIG instead of its f.
// Only items with status ST_OK get here, so ST_BAD_PK keeps precedence as in k_hash_field / k_status_merge.
__global__ void __launch_bounds__(TPB, BLS_MINB_ACCUM) k_miller_accum(const uint8_t* flags, uint8_t* status, size_t n, u32x4* f_soa, const u32x4* lines, int i_hi, int i_lo,
                                                                const uint8_t* sig_sub) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status[i] != ST_OK) return;
    uint8_t fl = flags[i]; bool use0 = !(fl & FL_SIG_INF), use1 = !(fl & FL_HM_INF);
    fp12 f; if (i_hi == 62) fp12_one(f); else soa_load_fp12(f, f_soa, n, i);
    const uint64_t x = BLS_X_ABS; int s = 0;
    for (int it = i_hi; it >= i_lo; it--) {
        if (it != 62) fp12_sqr(f, f);
        int steps = 1 + (int)((x >> it) & 1);
        for (int a = 0; a < steps; a++, s++) {
            if (use0) { const u32x4* L = lines + (size_t)(2 * s) * 18 * n; fp12_mul_by_014(f, soa_load_fp2(L, n, i, 0), soa_load_fp2(L, n, i, 1), soa_load_fp2(L, n, i, 2)); }
            if (use1) { const u32x4* L = lines + (size_t)(2 * s + 1) * 18 * n; fp12_mul_by_014(f, soa_load_fp2(L, n, i, 0), soa_load_fp2(L, n, i, 1), soa_load_fp2(L, n, i, 2)); }
        }
    }
    if (i_lo == 0) fp12_conj(f, f);
    if (i_lo == 0 && sig_sub && use0 && !sig_sub[i]) { status[i] = ST_BAD_SIG; return; }
    soa_store_fp12(f_soa, n, i, f);
}
// the 63 compressed squarings of one exp_by_x: in = an Fp12 array (cyclotomic elements), out = six snapshots of four Fp2 (24 x 6 uint4 rows per item)
__global__ void __launch_bounds__(TPB, BLS_MINB_SQR) k_final_squarings(const u32x4* in_soa, u32x4* snap_soa, const uint8_t* status, size_t n) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status[i] != ST_OK) return;
    fp12c c;                                                  // tower positions of g2, g3, g4, g5: c1.c0 = 3, c0.c2 = 2, c0.c1 = 1, c1.c2 = 5
    c.g2 = soa_load_fp2(in_soa, n, i, 3); c.g3 = soa_load_fp2(in_soa, n, i, 2); c.g4 = soa_load_fp2(in_soa, n, i, 1); c.g5 = soa_load_fp2(in_soa, n, i, 5);
    const uint64_t x = BLS_X_ABS; int k = 0;
    for (int j = 1; j <= 63; j++) {
        fp12c_sqr(c, c);
        if ((x >> j) & 1) {
            soa_store_fp2(snap_soa, n, i, 4 * k, c.g2); soa_store_fp2(snap_soa, n, i, 4 * k + 1, c.g3); soa_store_fp2(snap_soa, n, i, 4 * k + 2, c.g4); soa_store_fp2(snap_soa, n, i, 4 * k + 3, c.g5);
            k++;
        }
    }
}
template <int STEP> __global__ void __launch_bounds__(TPB, BLS_MINB) k_final_step(u32x4* f_soa, u32x4* y1_soa, u32x4* y2_soa, const u32x4* snap_soa, const uint8_t* status_in, uint8_t* status_out, size_t n) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status_in[i] != ST_OK) { if (STEP == 5) status_out[i] = status_in[i]; return; }
    fp12 r, y1, y2, e;
    if (STEP >= 1) {                                            // the exp_by_x result first: nothing else is live while the six snapshots are decompressed
        fp12_decompress_product_from(e, [&](int k) { fp12c c; c.g2 = soa_load_fp2(snap_soa, n, i, 4 * k); c.g3 = soa_load_fp2(snap_soa, n, i, 4 * k + 1);
                                                     c.g4 = soa_load_fp2(snap_soa, n, i, 4 * k + 2); c.g5 = soa_load_fp2(snap_soa, n, i, 4 * k + 3); return c; }, 6);
        fp12_conj(e, e);
    }
    if (STEP == 0 || STEP == 1 || STEP == 3 || STEP == 5) soa_load_fp12(r, f_soa, n, i);
    if (STEP == 2 || STEP == 3 || STEP == 5) soa_load_fp12(y1, y1_soa, n, i);
    final_exponentiation_step<STEP>(r, y1, y2, e);
    if (STEP == 0 || STEP == 3 || STEP == 5) soa_store_fp12(f_soa, n, i, r);
    if (STEP >= 1 && STEP <= 3) soa_store_fp12(y1_soa, n, i, y1);
    if (STEP == 4) soa_store_fp12(y2_soa, n, i, y2);
    if (STEP == 5) status_out[i] = fp12_is_one(r) ? ST_OK : ST_FALSE;
}
// generic product of pairings for the GT parity hook: npairs in {1,2}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_miller_pairs(const u32x4* g1_soa, const u32x4* g2_soa, const uint8_t* c1, const uint8_t* c2, size_t npairs, size_t nprod,
                                                      u32x4* f_soa, uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= nprod) return;
    size_t tot = npairs * nprod;
    g1_aff p[2]; g2_aff q[2]; bool use[2] = {false, false}; uint8_t st = ST_OK;
    for (size_t k = 0; k < npairs; k++) {
        size_t j = i * npairs + k;
        soa_load_g1(p[k], g1_soa, tot, j); soa_load_g2(q[k], g2_soa, tot, j);
        if (c1[j] > DEC_INF) st = ST_BAD_PK; else if (c2[j] > DEC_INF && st == ST_OK) st = ST_BAD_SIG;
        use[k] = c1[j] == DEC_OK && c2[j] == DEC_OK;
    }
    if (npairs < 2) { p[1] = p[0]; q[1] = q[0]; }
    status[i] = st;
    if (st != ST_OK) return;
    fp12 f; miller_loop2(f, p[0], q[0], use[0], p[1], q[1], use[1]);
    soa_store_fp12(f_soa, nprod, i, f);
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_final_exp(u32x4* f_soa, const uint8_t* status_in, uint8_t* status_out, size_t n) {
    phase_skew();
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status_in[i] != ST_OK) { status_out[i] = status_in[i]; return; }
    fp12 f, gt; soa_load_fp12(f, f_soa, n, i);
    status_out[i] = stage_final(gt, f);
    soa_store_fp12(f_soa, n, i, gt);
}
// K5 split for the cooperative path: easy part f^((p^6-1)(p^2+1)) per thread (one inversion), hard part six lanes per item
__global__ void __launch_bounds__(TPB, BLS_MINB) k_final_easy(u32x4* f_soa, const uint8_t* status, size_t n) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status[i] != ST_OK) return;
    fp12 f, t, r; soa_load_fp12(f, f_soa, n, i);
    fp12_conj(t, f); fp12_inv(r, f); fp12_mul(r, t, r);
    fp12_frob2(t, r); fp12_mul(r, t, r);
    soa_store_fp12(f_soa, n, i, r);
}
__global__ void __launch_bounds__(128, 2) k_final_hard_coop(u32x4* f_soa, const uint8_t* status_in, uint8_t* status_out, size_t n) {
    __shared__ coop_smem sm[4];                            // 41.5 KB per CTA
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane / 6;
    coop_lane c = coop_init(&sm[warp]);
    size_t item = (blockIdx.x * (size_t)4 + warp) * 5 + g;
    bool in_range = g < 5 && item < n;
    uint8_t st = in_range ? status_in[item] : (uint8_t)ST_BAD_PK;
    bool active = in_range && st == ST_OK;
    fp2 r = c.k == 0 ? fp2_one() : fp2_zero();
    if (active) r = soa_load_fp2(f_soa, n, item, COOP_TOWER_POS[c.k]);
    r = coop_final_exp_hard(c, r);
    bool mine = c.k == 0 ? fp2_eq(r, fp2_one()) : fp2_is_zero(r);
    unsigned ball = __ballot_sync(0xffffffffu, mine);
    if (active) soa_store_fp2(f_soa, n, item, COOP_TOWER_POS[c.k], r);
    if (in_range && c.k == 0) status_out[item] = active ? ((((ball >> (6 * g)) & 63u) == 63u) ? (uint8_t)ST_OK : (uint8_t)ST_FALSE) : st;
}
// The accumulator update of the split Miller loop with six lanes per item (small passes, blsgpu_set_coop): lane k holds the w^k coefficient of f,
// a line l0 + l1 v + l2 v w sits in lanes 0, 2, 3 (w^0, w^2, w^3) of an otherwise zero operand, a pair that is switched off multiplies by one.
// Three to five generic six-lane products per iteration instead of one squaring and two sparse products in one thread: more work, a third of the chain.
// sig_sub: as in k_miller_accum.  Lane 0 writes the status after the last coop_mul, whose __syncwarp orders it after every lane's read.
__global__ void __launch_bounds__(128, 2) k_miller_accum_coop(const uint8_t* flags, uint8_t* status, size_t n, u32x4* f_soa, const u32x4* lines, int i_hi, int i_lo,
                                                            const uint8_t* sig_sub) {
    __shared__ coop_smem sm[4];
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane / 6;
    coop_lane c = coop_init(&sm[warp]);
    size_t item = (blockIdx.x * (size_t)4 + warp) * 5 + g;
    bool active = g < 5 && item < n && status[item] == ST_OK;
    uint8_t fl = active ? flags[item] : (uint8_t)(FL_SIG_INF | FL_HM_INF);
    bool use[2] = {!(fl & FL_SIG_INF), !(fl & FL_HM_INF)};
    fp2 unit = c.k == 0 ? fp2_one() : fp2_zero();
    fp2 f = (active && i_hi != 62) ? soa_load_fp2(f_soa, n, item, COOP_TOWER_POS[c.k]) : unit;
    int slot = c.k == 0 ? 0 : c.k == 2 ? 1 : c.k == 3 ? 2 : -1;           // which line coefficient this lane carries
    const uint64_t x = BLS_X_ABS; int s = 0;
    for (int it = i_hi; it >= i_lo; it--) {
        if (it != 62) f = coop_mul(c, f, f);
        int steps = 1 + (int)((x >> it) & 1);
        for (int a = 0; a < steps; a++, s++)
            for (int j = 0; j < 2; j++) {
                const u32x4* L = lines + (size_t)(2 * s + j) * 18 * n;
                fp2 b = !use[j] ? unit : slot >= 0 ? soa_load_fp2(L, n, item, slot) : fp2_zero();
                f = coop_mul(c, f, b);
            }
    }
    if (i_lo == 0) f = coop_conj(c, f);
    if (active && i_lo == 0 && sig_sub && use[0] && !sig_sub[item]) { if (c.k == 0) status[item] = ST_BAD_SIG; return; }
    if (active) soa_store_fp2(f_soa, n, item, COOP_TOWER_POS[c.k], f);
}
// out[t] = prod_{i = t, t+T, ...} in[i] over items with status <= ST_FALSE (status == NULL: all items)
__global__ void __launch_bounds__(TPB, BLS_MINB) k_gt_reduce(const u32x4* in_soa, const uint8_t* status, size_t n, u32x4* out_soa, size_t T) {
    size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (t >= T) return;
    fp12 acc, x; fp12_one(acc);
    for (size_t i = t; i < n; i += T) {
        if (status && status[i] > ST_FALSE) continue;
        soa_load_fp12(x, in_soa, n, i); fp12_mul(acc, acc, x);
    }
    soa_store_fp12(out_soa, T, t, acc);
}
__global__ void k_gt_mul_into(u32x4* acc_soa, const u32x4* x_soa) {      // single thread: acc *= x
    if (threadIdx.x || blockIdx.x) return;
    fp12 a, x; soa_load_fp12(a, acc_soa, 1, 0); soa_load_fp12(x, x_soa, 1, 0); fp12_mul(a, a, x); soa_store_fp12(acc_soa, 1, 0, a);
}
__global__ void k_gt_set_one(u32x4* acc_soa) { if (threadIdx.x || blockIdx.x) return; fp12 a; fp12_one(a); soa_store_fp12(acc_soa, 1, 0, a); }
__global__ void __launch_bounds__(TPB, BLS_MINB) k_gt_to_bytes(const u32x4* soa, size_t n, uint8_t* out576, const uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    if (status && status[i] != ST_OK) { for (int k = 0; k < 576; k++) out576[576 * i + k] = 0; return; }
    fp12 a; soa_load_fp12(a, soa, n, i); fp12_to_bytes(out576 + 576 * i, a);
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_gt_from_bytes(const uint8_t* in576, size_t n, u32x4* soa) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    fp12 a; fp2* c[6] = {&a.c0.c0, &a.c0.c1, &a.c0.c2, &a.c1.c0, &a.c1.c1, &a.c1.c2};
    const uint8_t* b = in576 + 576 * i;
    for (int k = 0; k < 12; k++) {
        fp v;
        for (int w = 0; w < 12; w++) { const uint8_t* q = b + 48 * k + 4 * w; v.l[w] = q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24); }
        v = fp_to_mont(v);
        if (k & 1) c[k >> 1]->c1 = v; else c[k >> 1]->c0 = v;
    }
    soa_store_fp12(soa, n, i, a);
}
__global__ void k_status_bitmap(const uint8_t* status, size_t n, uint32_t* bitmap32) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    bool ok = i < n && status[i] == ST_OK;
    unsigned m = __ballot_sync(0xffffffffu, ok);
    if ((threadIdx.x & 31) == 0 && i < ((n + 31) / 32) * 32) bitmap32[i >> 5] = m;
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_encode_g1(const u32x4* soa, const uint8_t* inf, size_t n, uint8_t* out48) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g1_aff p; soa_load_g1(p, soa, n, i); g1_encode(out48 + 48 * i, p, inf && inf[i]);
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_encode_g2(const u32x4* soa, const uint8_t* flags, uint8_t mask, size_t n, uint8_t* out96) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g2_aff p; soa_load_g2(p, soa, n, i); g2_encode(out96 + 96 * i, p, flags && (flags[i] & mask));
}
// canonical Fr check: sk < r, little-endian 32 bytes -> 8 words
__device__ __forceinline__ bool load_scalar(uint32_t* k, const uint8_t* sk) {
    const uint32_t R[8] = BLS_C_R_ORDER;
    for (int w = 0; w < 8; w++) k[w] = sk[4 * w] | ((uint32_t)sk[4 * w + 1] << 8) | ((uint32_t)sk[4 * w + 2] << 16) | ((uint32_t)sk[4 * w + 3] << 24);
    for (int w = 7; w >= 0; w--) { if (k[w] != R[w]) return k[w] < R[w]; }
    return false;
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_scalar_mul_g1(const uint8_t* sk32, size_t n, uint8_t* pk48, uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    uint32_t k[8]; bool canon = load_scalar(k, sk32 + 32 * i);
    if (status) status[i] = canon ? ST_OK : ST_BAD_SK;
    g1_aff g; g.x = fp_const(C_G1X); g.y = fp_const(C_G1Y);
    g1_jac r; jac_mul_scalar(r, g, k);
    g1_aff a; bool ok = jac_to_aff(a, r); g1_encode(pk48 + 48 * i, a, !ok || !canon);
}
// sig = [sk] H(m): H(m) comes from k_hash_to_g2's limb-SoA output
__global__ void __launch_bounds__(TPB, BLS_MINB) k_scalar_mul_g2(const uint8_t* sk32, const u32x4* hm_soa, const uint8_t* flags, size_t n, uint8_t* sig96, uint8_t* status) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    uint32_t k[8]; bool canon = load_scalar(k, sk32 + 32 * i);
    uint32_t nz = 0; for (int w = 0; w < 8; w++) nz |= k[w];
    if (!canon || !nz) { status[i] = ST_BAD_SK; for (int b = 0; b < 96; b++) sig96[96 * i + b] = 0; return; }   // bls.rs:417-419
    status[i] = ST_OK;
    g2_aff hm; soa_load_g2(hm, hm_soa, n, i);
    g2_jac r;
    if (flags[i] & FL_HM_INF) jac_set_identity(r); else jac_mul_scalar(r, hm, k);
    g2_aff a; bool ok = jac_to_aff(a, r); g2_encode(sig96 + 96 * i, a, !ok);
}

// K3: segmented aggregation.  L lanes cooperate on one segment (32/L segments per warp; L is picked so that a lane folds
// >= ~64 points): each lane folds a strided slice with mixed additions, the L partial sums are combined by a shared-memory
// tree of full Jacobian additions, and the Jacobian result goes to HBM.  The to-affine inversion (one 380-bit
// exponentiation per segment) runs in a second, thread-per-segment kernel so that it is not serialised on one lane per warp.
template <class F> struct segsum_traits;
template <> struct segsum_traits<fp>  { enum { K = 2 }; static __device__ __forceinline__ void load(aff<fp>& p, const u32x4* s, size_t n, size_t i) { soa_load_g1(p, s, n, i); }
                                        static __device__ __forceinline__ void store(u32x4* s, size_t n, size_t i, const aff<fp>& p) { soa_store_g1(s, n, i, p); }
                                        static __device__ __forceinline__ void storej(u32x4* s, size_t n, size_t i, const jac<fp>& p) { soa_store_fp(s, n, i, 0, p.X); soa_store_fp(s, n, i, 1, p.Y); soa_store_fp(s, n, i, 2, p.Z); }
                                        static __device__ __forceinline__ void loadj(jac<fp>& p, const u32x4* s, size_t n, size_t i) { p.X = soa_load_fp(s, n, i, 0); p.Y = soa_load_fp(s, n, i, 1); p.Z = soa_load_fp(s, n, i, 2); } };
template <> struct segsum_traits<fp2> { enum { K = 4 }; static __device__ __forceinline__ void load(aff<fp2>& p, const u32x4* s, size_t n, size_t i) { soa_load_g2(p, s, n, i); }
                                        static __device__ __forceinline__ void store(u32x4* s, size_t n, size_t i, const aff<fp2>& p) { soa_store_g2(s, n, i, p); }
                                        static __device__ __forceinline__ void storej(u32x4* s, size_t n, size_t i, const jac<fp2>& p) { soa_store_fp2(s, n, i, 0, p.X); soa_store_fp2(s, n, i, 1, p.Y); soa_store_fp2(s, n, i, 2, p.Z); }
                                        static __device__ __forceinline__ void loadj(jac<fp2>& p, const u32x4* s, size_t n, size_t i) { p.X = soa_load_fp2(s, n, i, 0); p.Y = soa_load_fp2(s, n, i, 1); p.Z = soa_load_fp2(s, n, i, 2); } };
#define SEG_WARPS 4
template <class F> __global__ void __launch_bounds__(32 * SEG_WARPS) k_segsum(const u32x4* pts_soa, const uint8_t* code, size_t npts, const uint32_t* seg_off, size_t seg_stride,
                                                                            const uint64_t* bitmap, size_t nseg, u32x4* out_jac, uint8_t* status, uint8_t bad_code,
                                                                            const uint32_t* idx /* nullable: member i of the flat list is point idx[i] of the resident pool */, int L) {
    __shared__ jac<F> sm[SEG_WARPS][32];
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, sub = lane / L, sl = lane % L, per_warp = 32 / L;
    size_t s = (blockIdx.x * (size_t)SEG_WARPS + warp) * per_warp + sub;
    bool active = s < nseg;
    size_t lo = 0, hi = 0;
    if (active) { if (seg_off) { lo = seg_off[s]; hi = seg_off[s + 1]; } else { lo = s * seg_stride; hi = lo + seg_stride; } }
    jac<F> acc; jac_set_identity(acc);
    unsigned bad = 0, cnt = 0;
    for (size_t i = lo + sl; i < hi; i += L) {
        if (bitmap && !((bitmap[i >> 6] >> (i & 63)) & 1)) continue;
        cnt++;
        size_t pi = idx ? (size_t)idx[i] : i;
        if (pi >= npts) { bad = 1; continue; }
        uint8_t c = code[pi];
        if (c > DEC_INF) { bad = 1; continue; }
        if (c == DEC_INF) continue;
        aff<F> p; segsum_traits<F>::load(p, pts_soa, npts, pi);
        jac_add_mixed(acc, acc, p);
    }
    sm[warp][lane] = acc;
    __syncwarp();
    for (int w = L >> 1; w >= 1; w >>= 1) {
        if (sl < w) { jac<F> o = sm[warp][lane + w]; jac_add(acc, acc, o); sm[warp][lane] = acc; }
        __syncwarp();
        bad |= __shfl_down_sync(0xffffffffu, bad, w); cnt += __shfl_down_sync(0xffffffffu, cnt, w);     // stays inside the L-lane group for sl < w
    }
    if (active && sl == 0) {
        segsum_traits<F>::storej(out_jac, nseg, s, acc);
        status[s] = bad ? bad_code : (cnt == 0 ? ST_EMPTY : ST_OK);
    }
}
template <class F> __global__ void __launch_bounds__(TPB, BLS_MINB) k_jac_to_aff(const u32x4* jac_soa, size_t n, u32x4* aff_soa, uint8_t* inf) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    jac<F> p; segsum_traits<F>::loadj(p, jac_soa, n, i);
    aff<F> a; bool ok = jac_to_aff(a, p);
    segsum_traits<F>::store(aff_soa, n, i, a); inf[i] = ok ? 0 : 1;
}
// lanes per segment: the largest power of two <= 32 that still leaves ~64 points per lane (at least 1)
static int seg_lanes(size_t avg_len) { int L = 32; while (L > 1 && avg_len / L < 64) L >>= 1; return L; }
// fast_aggregate_verify glue: status/flags from the aggregation outcome and the signature decode code
__global__ void k_fav_status(const uint8_t* agg_status, const uint8_t* agg_inf, const uint8_t* code_sig, size_t n, uint8_t* code_pk_out) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    // empty committee => None => identity key => InvalidPublicKey (tests.rs:312-316); identity aggregate => bls.rs:434
    code_pk_out[i] = (agg_status[i] != ST_OK || agg_inf[i]) ? DEC_BAD_FLAGS : DEC_OK;
}

// ---- random-linear-combination batch check (SURVEY 8(f)-3): prod_i e(r_i pk_i, H(m_i)) * e(-g1, sum_i r_i sig_i) == 1
// r_i: 64 non-zero bits of SHA-256(seed16 || le64(global index))
__device__ __forceinline__ uint64_t rlc_scalar(const uint8_t* seed16, uint64_t idx) {
    sha256_ctx c; sha256_init(c);
    for (int i = 0; i < 16; i++) sha256_put(c, seed16[i]);
    for (int i = 0; i < 8; i++) sha256_put(c, (uint32_t)(idx >> (8 * i)) & 0xffu);
    uint32_t d[8]; sha256_final(c, d);
    uint64_t r = ((uint64_t)d[0] << 32) | d[1];
    return r ? r : 1;
}
template <class F> __device__ __forceinline__ void jac_mul_u64(jac<F>& r, const aff<F>& p, uint64_t k) {
    jac_set_identity(r);
    for (int i = 63; i >= 0; i--) { jac_dbl(r, r); if ((k >> i) & 1) jac_add_mixed(r, r, p); }
}
// pk <- [r] pk (affine, in place); rsig <- [r] sig (Jacobian); pair 0 of the Miller loop is switched off for the item
__global__ void __launch_bounds__(TPB, BLS_MINB) k_rlc_scale(u32x4* pk_soa, const u32x4* sig_soa, uint8_t* flags, const uint8_t* status, size_t n, size_t idx0,
                                                              const uint8_t* seed16, u32x4* rsig_jac) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g2_jac rs; jac_set_identity(rs);
    if (status[i] == ST_OK) {
        uint64_t r = rlc_scalar(seed16, idx0 + i);
        g1_aff pk; soa_load_g1(pk, pk_soa, n, i);
        g1_jac rp; jac_mul_u64(rp, pk, r);
        g1_aff a; jac_to_aff(a, rp); soa_store_g1(pk_soa, n, i, a);          // pk has prime order r > 2^64: [r]pk is never the identity
        if (!(flags[i] & FL_SIG_INF)) { g2_aff sg; soa_load_g2(sg, sig_soa, n, i); jac_mul_u64(rs, sg, r); }
        flags[i] |= FL_SIG_INF;
    }
    segsum_traits<fp2>::storej(rsig_jac, n, i, rs);
}
// out[t] = sum_{i = t, t+T, ...} in[i] (Jacobian G2)
__global__ void __launch_bounds__(TPB, BLS_MINB) k_g2_jac_reduce(const u32x4* in_jac, size_t n, u32x4* out_jac, size_t T) {
    size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (t >= T) return;
    g2_jac acc, x; jac_set_identity(acc);
    for (size_t i = t; i < n; i += T) { segsum_traits<fp2>::loadj(x, in_jac, n, i); jac_add(acc, acc, x); }
    segsum_traits<fp2>::storej(out_jac, T, t, acc);
}
__global__ void k_g2_jac_add_into(u32x4* acc_jac, const u32x4* x_jac) {
    if (threadIdx.x || blockIdx.x) return;
    g2_jac a, x; segsum_traits<fp2>::loadj(a, acc_jac, 1, 0); segsum_traits<fp2>::loadj(x, x_jac, 1, 0); jac_add(a, a, x); segsum_traits<fp2>::storej(acc_jac, 1, 0, a);
}
__global__ void k_g2_jac_set_identity(u32x4* acc_jac) { if (threadIdx.x || blockIdx.x) return; g2_jac a; jac_set_identity(a); segsum_traits<fp2>::storej(acc_jac, 1, 0, a); }
// bad[0] |= any status other than OK
__global__ void k_any_bad(const uint8_t* status, size_t n, uint32_t* bad) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    bool b = i < n && status[i] != ST_OK;
    if (__any_sync(0xffffffffu, b) && (threadIdx.x & 31) == 0) atomicOr(bad, 1u);
}
// single thread: F * miller(-g1, S), final exponentiation, is_one
__global__ void __launch_bounds__(32, 1) k_rlc_finish(const u32x4* f_acc, const u32x4* s_jac, const uint32_t* bad, uint8_t* all_ok) {
    if (threadIdx.x || blockIdx.x) return;
    fp12 F, f2, gt; soa_load_fp12(F, f_acc, 1, 0);
    g2_jac S; segsum_traits<fp2>::loadj(S, s_jac, 1, 0);
    g2_aff sa; bool have = jac_to_aff(sa, S);
    g1_aff ng; ng.x = fp_const(C_G1X); ng.y = fp_const(C_G1Y_NEG);
    miller_loop2(f2, ng, sa, have, ng, sa, false);
    fp12_mul(F, F, f2);
    final_exponentiation(gt, F);
    all_ok[0] = (fp12_is_one(gt) && !bad[0]) ? 1 : 0;
}

// ---- per-piece forms for the bisecting batch check: the batch is cut into pieces of L items; products / sums are kept per piece
// out[p * T + t] = prod_{i = t, t + T, ... < len_p} in[p * L + i]   (len_p = min(L, n - p L); status filter as k_gt_reduce)
__global__ void __launch_bounds__(TPB, BLS_MINB) k_gt_reduce_seg(const u32x4* in_soa, const uint8_t* status, size_t n, size_t L, u32x4* out_soa, size_t T, size_t P) {
    size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x, p = blockIdx.y; if (t >= T) return;
    size_t lo = p * L, hi = lo + L < n ? lo + L : n;
    fp12 acc, x; fp12_one(acc);
    for (size_t i = lo + t; i < hi; i += T) {
        if (status && status[i] > ST_FALSE) continue;
        soa_load_fp12(x, in_soa, n, i); fp12_mul(acc, acc, x);
    }
    soa_store_fp12(out_soa, P * T, p * T + t, acc);
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_g2_jac_reduce_seg(const u32x4* in_jac, size_t n, size_t L, u32x4* out_jac, size_t T, size_t P) {
    size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x, p = blockIdx.y; if (t >= T) return;
    size_t lo = p * L, hi = lo + L < n ? lo + L : n;
    g2_jac acc, x; jac_set_identity(acc);
    for (size_t i = lo + t; i < hi; i += T) { segsum_traits<fp2>::loadj(x, in_jac, n, i); jac_add(acc, acc, x); }
    segsum_traits<fp2>::storej(out_jac, P * T, p * T + t, acc);
}
// one block per piece (thread 0 works): ok[p] = [ F_p * miller(-g1, S_p) ]^((p^12-1)/r) == 1  -- the pieces' finishes run side by side,
// so locating the failing pieces costs one single-thread latency (~20 ms) whatever their number
__global__ void __launch_bounds__(32, 1) k_rlc_finish_seg(const u32x4* f_piece, const u32x4* s_piece, size_t P, uint8_t* ok) {
    size_t p = blockIdx.x; if (threadIdx.x || p >= P) return;
    fp12 F, f2, gt; soa_load_fp12(F, f_piece, P, p);
    g2_jac S; segsum_traits<fp2>::loadj(S, s_piece, P, p);
    g2_aff sa; bool have = jac_to_aff(sa, S);
    g1_aff ng; ng.x = fp_const(C_G1X); ng.y = fp_const(C_G1Y_NEG);
    miller_loop2(f2, ng, sa, have, ng, sa, false);
    fp12_mul(F, F, f2);
    final_exponentiation(gt, F);
    ok[p] = fp12_is_one(gt) ? 1 : 0;
}

// ---- uncompressed <-> compressed point encodings (K7'): status = BLSGPU_DE_* of the INPUT; an undecodable input gives an all-zero output
__global__ void __launch_bounds__(TPB, BLS_MINB) k_g1_recode(const uint8_t* in, size_t n, uint8_t* out, uint8_t* code, int to_uncompressed) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g1_aff p; int rc = to_uncompressed ? g1_decode(p, in + 48 * i) : g1_decode_uncompressed(p, in + 96 * i);
    uint8_t* o = out + (to_uncompressed ? 96 : 48) * i;
    if (rc > DEC_INF) { for (int k = 0; k < (to_uncompressed ? 96 : 48); k++) o[k] = 0; }
    else if (to_uncompressed) g1_encode_uncompressed(o, p, rc == DEC_INF); else g1_encode(o, p, rc == DEC_INF);
    if (code) code[i] = (uint8_t)rc;
}
__global__ void __launch_bounds__(TPB, BLS_MINB) k_g2_recode(const uint8_t* in, size_t n, uint8_t* out, uint8_t* code, int to_uncompressed) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g2_aff p; int rc = to_uncompressed ? g2_decode(p, in + 96 * i) : g2_decode_uncompressed(p, in + 192 * i);
    uint8_t* o = out + (to_uncompressed ? 192 : 96) * i;
    if (rc > DEC_INF) { for (int k = 0; k < (to_uncompressed ? 192 : 96); k++) o[k] = 0; }
    else if (to_uncompressed) g2_encode_uncompressed(o, p, rc == DEC_INF); else g2_encode(o, p, rc == DEC_INF);
    if (code) code[i] = (uint8_t)rc;
}
// ---- aggregate_verify (distinct messages): per-signature glue.  sig_status / sig_flags for the (-g1, sig) Miller loops:
__global__ void k_aggv_sig_status(const uint8_t* code_sig, size_t nsig, uint8_t* st, uint8_t* flags) {
    size_t s = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (s >= nsig) return;
    st[s] = (code_sig[s] == DEC_OK || code_sig[s] == DEC_INF) ? ST_OK : ST_BAD_SIG;
    flags[s] = FL_HM_INF | (code_sig[s] == DEC_INF ? FL_SIG_INF : 0);            // the (pk, H(m)) slot of k_miller is switched off
}
// F_s = f_sig[s] * prod_{j in pairs of s} f_pair[j]; status: a bad key wins over a bad signature (the order of src/bls.rs:434-447), no pairs = ST_EMPTY
__global__ void __launch_bounds__(TPB, BLS_MINB) k_aggv_combine(const u32x4* f_pair, const uint8_t* pair_status, size_t npairs, const uint32_t* pair_off,
                                                                 u32x4* f_sig, const uint8_t* sig_status, size_t nsig, uint8_t* status) {
    size_t s = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (s >= nsig) return;
    uint32_t lo = pair_off[s], hi = pair_off[s + 1];
    uint8_t st = sig_status[s];
    for (uint32_t j = lo; j < hi; j++) if (pair_status[j] != ST_OK) { st = ST_BAD_PK; break; }
    if (st == ST_OK && lo == hi) st = ST_EMPTY;
    status[s] = st;
    if (st != ST_OK) return;
    fp12 acc, x; soa_load_fp12(acc, f_sig, nsig, s);
    for (uint32_t j = lo; j < hi; j++) { soa_load_fp12(x, f_pair, npairs, j); fp12_mul(acc, acc, x); }
    soa_store_fp12(f_sig, nsig, s, acc);
}

// ================================================================================================ context
struct blsgpu_ctx {
    int device; cudaStream_t own_stream, stream; int ptr_mode; char err[512];
    uint8_t* ws; size_t ws_bytes, ws_used; unsigned long long launches;
    struct r1cs_sys* r1cs[16]; struct wit_prog* wit[4];
    uint8_t* rlc_acc;                   // accumulators of blsgpu_verify_batch_rlc that live across passes (allocated on first use)
    struct { u32x4* soa; uint8_t* code; size_t n; } pool[16];   // resident decoded validator pools
    int coop;                           // hard part of the final exponentiation with six lanes per item (coop.cuh): 0 = never, 1 = always, 2 (default) = for passes of at most VERIFY_COOP_BELOW items
    int wit_cluster;                    // 1 = witness replay with one thread-block cluster per group of 32 assignments; 0 (default) = grid-wide level barrier
    int lanes; cudaStream_t lane_stream[4]; cudaEvent_t lane_done[4], fork;   // concurrent sub-ranges of a verify pass
    int split;                          // 1 (default) = hash-to-G2, Miller loop and final exponentiation as sequences of short specialised launches, 0 = one launch each
    size_t chunk;                       // items per internal pass of verify_batch (bounds the workspace); multiple of 64
    int prof; cudaEvent_t ev[8];        // stage boundaries of the last verify_batch chunk: g1 | g2 | hash | miller | final | epilogue
};
// every entry point runs on the context's device and leaves the caller's current device as it found it
struct dev_guard { int prev; dev_guard() : prev(-1) { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } } ~dev_guard() { if (prev >= 0) cudaSetDevice(prev); } };
#define STAGE_MARK(k) do { if (ctx->prof) CU(cudaEventRecord(ctx->ev[k], ctx->stream)); } while (0)
static int fail(blsgpu_ctx* c, int code, const char* fmt, ...) {
    if (c) { va_list ap; va_start(ap, fmt); vsnprintf(c->err, sizeof c->err, fmt, ap); va_end(ap); }
    return code;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(ctx, BLSGPU_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
#define LAUNCH(kern, grid, block, ...) do { kern<<<(grid), (block), 0, ctx->stream>>>(__VA_ARGS__); ctx->launches++; CU(cudaGetLastError()); } while (0)

static int ws_reserve(blsgpu_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->ws_bytes) { ctx->ws_used = 0; return 0; }
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->ws) { cudaFree(ctx->ws); ctx->ws = nullptr; ctx->ws_bytes = 0; }
    size_t want = bytes + (bytes >> 3);
    if (cudaMalloc(&ctx->ws, want) != cudaSuccess) { cudaGetLastError(); return fail(ctx, BLSGPU_ERR_ALLOC, "cudaMalloc of %zu workspace bytes failed", want); }
    ctx->ws_bytes = want; ctx->ws_used = 0; return 0;
}
template <class T> static T* ws_take(blsgpu_ctx* ctx, size_t count) {
    size_t off = (ctx->ws_used + 255) & ~(size_t)255; ctx->ws_used = off + count * sizeof(T);
    return reinterpret_cast<T*>(ctx->ws + off);
}
static inline size_t al(size_t b) { return (b + 255) & ~(size_t)255; }
// input staging: host mode copies to the workspace, device mode uses the pointer as is
template <class T> static int stage_in(blsgpu_ctx* ctx, const T*& dev, const T* user, size_t count) {
    if (!user) { dev = nullptr; return 0; }
    if (ctx->ptr_mode == BLSGPU_DEVICE) { dev = user; return 0; }
    T* d = ws_take<T>(ctx, count ? count : 1);
    if (count) CU(cudaMemcpyAsync(d, user, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    dev = d; return 0;
}
template <class T> static T* stage_out(blsgpu_ctx* ctx, T* user, size_t count) {
    if (!user) return nullptr;
    return ctx->ptr_mode == BLSGPU_DEVICE ? user : ws_take<T>(ctx, count ? count : 1);
}
template <class T> static int finish_out(blsgpu_ctx* ctx, T* user, const T* dev, size_t count) {
    if (!user || ctx->ptr_mode == BLSGPU_DEVICE || !count) return 0;
    CU(cudaMemcpyAsync(user, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    return 0;
}
static int finish_call(blsgpu_ctx* ctx) {
    if (ctx->ptr_mode == BLSGPU_HOST) CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}
static size_t msg_bytes_total(blsgpu_ctx* ctx, const uint32_t* off, size_t n, int& rc) {
    rc = 0;
    if (!off) return 32 * n;
    if (ctx->ptr_mode == BLSGPU_HOST) return off[n];
    uint32_t last = 0;
    if (cudaMemcpyAsync(&last, off + n, 4, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = BLSGPU_ERR_CUDA;
    return last;
}

// GT product of n values (limb-SoA, filtered by status) into a single value at dst (limb-SoA, n = 1)
static int gt_product(blsgpu_ctx* ctx, const u32x4* in_soa, const uint8_t* status, size_t n, u32x4* tmp_a, u32x4* tmp_b, u32x4* dst) {
    const u32x4* cur = in_soa; size_t cnt = n; const uint8_t* st = status; u32x4* bufs[2] = {tmp_a, tmp_b}; int which = 0;
    while (true) {
        size_t T = (cnt + 7) / 8;                       // radix-8 tree: every pass multiplies 8 values per thread
        u32x4* out = T == 1 ? dst : bufs[which];
        LAUNCH(k_gt_reduce, nblk(T), TPB, cur, st, cnt, out, T);
        if (T == 1) break;
        cur = out; cnt = T; st = nullptr; which ^= 1;
    }
    return 0;
}

extern "C" {

int blsgpu_create(blsgpu_ctx** out, int device) {
    if (!out) return BLSGPU_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return BLSGPU_ERR_CUDA; }
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) return BLSGPU_ERR_CUDA; }
    if (device >= ndev) return BLSGPU_ERR_ARG;
    dev_guard guard_;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return BLSGPU_ERR_CUDA;
    if (prop.major != 10) return BLSGPU_ERR_CUDA;                         // sm_100a cubin only: no other device can run it
    if (cudaSetDevice(device) != cudaSuccess) return BLSGPU_ERR_CUDA;
    blsgpu_ctx* c = new (std::nothrow) blsgpu_ctx(); if (!c) return BLSGPU_ERR_ALLOC;
    memset(c, 0, sizeof *c); c->device = device; c->ptr_mode = BLSGPU_HOST; c->chunk = VERIFY_CHUNK_DEFAULT; c->lanes = 2; c->wit_cluster = 0; c->split = 1; c->coop = 2;
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return BLSGPU_ERR_CUDA; }
    c->stream = c->own_stream;
    *out = c; return 0;
}
void blsgpu_destroy(blsgpu_ctx* ctx) {
    if (!ctx) return;
    dev_guard guard_; cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 16; i++) if (ctx->r1cs[i]) blsgpu_r1cs_free(ctx, i);
    for (int i = 0; i < 4; i++) if (ctx->wit[i]) blsgpu_witness_free(ctx, i);
    for (int i = 0; i < 16; i++) if (ctx->pool[i].soa) { cudaFree(ctx->pool[i].soa); cudaFree(ctx->pool[i].code); }
    if (ctx->ws) cudaFree(ctx->ws);
    if (ctx->rlc_acc) cudaFree(ctx->rlc_acc);
    if (ctx->ev[0]) for (int i = 0; i < 8; i++) cudaEventDestroy(ctx->ev[i]);
    if (ctx->lane_stream[0]) { for (int l = 0; l < 4; l++) { cudaStreamDestroy(ctx->lane_stream[l]); cudaEventDestroy(ctx->lane_done[l]); } cudaEventDestroy(ctx->fork); }
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}
const char* blsgpu_last_error(blsgpu_ctx* ctx) { return ctx ? ctx->err : "no context (no usable sm_100 CUDA device, or bad device ordinal)"; }
int blsgpu_set_stream(blsgpu_ctx* ctx, void* s, int use_own) { if (!ctx) return BLSGPU_ERR_ARG; ctx->stream = use_own ? ctx->own_stream : (cudaStream_t)s; return 0; }
int blsgpu_set_pointer_mode(blsgpu_ctx* ctx, int mode) { if (!ctx || (mode != BLSGPU_HOST && mode != BLSGPU_DEVICE)) return BLSGPU_ERR_ARG; ctx->ptr_mode = mode; return 0; }
int blsgpu_synchronize(blsgpu_ctx* ctx) { if (!ctx) return BLSGPU_ERR_ARG; dev_guard guard_; CU(cudaSetDevice(ctx->device)); CU(cudaStreamSynchronize(ctx->stream)); return 0; }
uint64_t blsgpu_launch_count(blsgpu_ctx* ctx) { return ctx ? ctx->launches : 0; }
int blsgpu_set_coop(blsgpu_ctx* ctx, int on) { if (!ctx || on < 0 || on > 2) return BLSGPU_ERR_ARG; ctx->coop = on; return 0; }
int blsgpu_set_witness_mode(blsgpu_ctx* ctx, int cluster) { if (!ctx) return BLSGPU_ERR_ARG; ctx->wit_cluster = cluster ? 1 : 0; return 0; }
int blsgpu_set_split(blsgpu_ctx* ctx, int on) { if (!ctx) return BLSGPU_ERR_ARG; ctx->split = on ? 1 : 0; return 0; }
int blsgpu_set_lanes(blsgpu_ctx* ctx, int lanes) { if (!ctx || lanes < 1 || lanes > 4) return BLSGPU_ERR_ARG; ctx->lanes = lanes; return 0; }
int blsgpu_set_chunk(blsgpu_ctx* ctx, size_t items) { if (!ctx || items < 64 || (items & 63)) return BLSGPU_ERR_ARG; ctx->chunk = items; return 0; }
int blsgpu_set_profiling(blsgpu_ctx* ctx, int on) {
    if (!ctx) return BLSGPU_ERR_ARG;
    dev_guard guard_; CU(cudaSetDevice(ctx->device));
    if (on && !ctx->ev[0]) for (int i = 0; i < 8; i++) CU(cudaEventCreate(&ctx->ev[i]));
    ctx->prof = on ? 1 : 0; return 0;
}
int blsgpu_stage_times(blsgpu_ctx* ctx, float* ms6) {
    if (!ctx || !ms6 || !ctx->ev[0]) return BLSGPU_ERR_ARG;
    dev_guard guard_; CU(cudaSetDevice(ctx->device)); CU(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 6; i++) CU(cudaEventElapsedTime(&ms6[i], ctx->ev[i], ctx->ev[i + 1]));
    return 0;
}

#define ENTER() if (!ctx) return BLSGPU_ERR_ARG; dev_guard guard_; CU(cudaSetDevice(ctx->device))

int blsgpu_fp_mul_raw(blsgpu_ctx* ctx, const uint8_t* a48, const uint8_t* b48, size_t n, uint8_t* out48, int reps) {
    ENTER(); if (!a48 || !b48 || !out48) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!n) return 0;
    if (int rc = ws_reserve(ctx, 3 * al(48 * n) + 4096)) return rc;
    const uint8_t *da, *db; if (int rc = stage_in(ctx, da, a48, 48 * n)) return rc; if (int rc = stage_in(ctx, db, b48, 48 * n)) return rc;
    uint8_t* dout = stage_out(ctx, out48, 48 * n);
    LAUNCH(k_fp_mul_raw, nblk(n), TPB, (const fp*)da, (const fp*)db, (fp*)dout, n, reps < 1 ? 1 : reps);
    if (int rc = finish_out(ctx, out48, dout, 48 * n)) return rc;
    return finish_call(ctx);
}
int blsgpu_imad_peak(blsgpu_ctx* ctx, int mode, double* mac32_per_sec, double* ms_out) {
    ENTER(); if (!mac32_per_sec) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (int rc = ws_reserve(ctx, 4096)) return rc;
    uint32_t* sink = ws_take<uint32_t>(ctx, 16);
    int sms = 0; CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
    const int iters = 8192, blocks = sms * 8, threads = 256;
    cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    double best = 1e30;
    if (mode == 2) {
        // the Montgomery multiplier itself, 8 warps per sub-partition, 2000 dependent products per thread: the rate the
        // IMAD.WIDE pipe sustains on the real instruction mix (300 MAC32 per product)
        size_t n = (size_t)sms * 128 * 8; const int reps = 2000;
        if (int rc = ws_reserve(ctx, 3 * al(48 * n) + 4096)) return rc;
        fp* a = ws_take<fp>(ctx, n); fp* b = ws_take<fp>(ctx, n); fp* o = ws_take<fp>(ctx, n);
        CU(cudaMemsetAsync(a, 0x5a, 48 * n, ctx->stream)); CU(cudaMemsetAsync(b, 0x13, 48 * n, ctx->stream));
        for (int rep = 0; rep < 4; rep++) {
            CU(cudaEventRecord(e0, ctx->stream));
            LAUNCH(k_fp_mul_raw, nblk(n), TPB, (const fp*)a, (const fp*)b, o, n, reps);
            CU(cudaEventRecord(e1, ctx->stream)); CU(cudaEventSynchronize(e1));
            float ms = 0; CU(cudaEventElapsedTime(&ms, e0, e1));
            if (rep && ms < best) best = ms;
        }
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        *mac32_per_sec = (double)n * reps * 300.0 / (best * 1e-3); if (ms_out) *ms_out = best;
        return 0;
    }
    for (int rep = 0; rep < 6; rep++) {
        CU(cudaEventRecord(e0, ctx->stream));
        LAUNCH(k_imad_peak, blocks, threads, sink, iters, mode);
        CU(cudaEventRecord(e1, ctx->stream)); CU(cudaEventSynchronize(e1));
        float ms = 0; CU(cudaEventElapsedTime(&ms, e0, e1));
        if (rep && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    double macs = (double)blocks * threads * (double)iters * 16.0;
    *mac32_per_sec = macs / (best * 1e-3); if (ms_out) *ms_out = best;
    return 0;
}

int blsgpu_deserialize_g1(blsgpu_ctx* ctx, const uint8_t* in48, size_t n, uint8_t* status) {
    ENTER(); if (!in48 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!n) return 0;
    if (int rc = ws_reserve(ctx, al(48 * n) + al(n) + 4096)) return rc;
    const uint8_t* din; if (int rc = stage_in(ctx, din, in48, 48 * n)) return rc;
    uint8_t* dst = stage_out(ctx, status, n);
    LAUNCH(k_decode_g1, nblk(n), TPB, din, n, (u32x4*)nullptr, dst);
    if (int rc = finish_out(ctx, status, dst, n)) return rc;
    return finish_call(ctx);
}
int blsgpu_deserialize_g2(blsgpu_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* status) {
    ENTER(); if (!in96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!n) return 0;
    if (int rc = ws_reserve(ctx, al(96 * n) + al(n) + 4096)) return rc;
    const uint8_t* din; if (int rc = stage_in(ctx, din, in96, 96 * n)) return rc;
    uint8_t* dst = stage_out(ctx, status, n);
    LAUNCH(k_decode_g2<true>, nblk(n), TPB, din, n, (u32x4*)nullptr, dst);
    if (int rc = finish_out(ctx, status, dst, n)) return rc;
    return finish_call(ctx);
}

static int hash_stage(blsgpu_ctx* ctx, const uint8_t* dmsg, const uint32_t* doff, size_t n, const uint8_t* code_pk, const uint8_t* code_sig, u32x4* hm_soa, u32x4* scratch36,
                      uint8_t* flags, uint8_t* dstatus);
int blsgpu_hash_to_g2_batch(blsgpu_ctx* ctx, const uint8_t* msg, const uint32_t* msg_off, size_t n, uint8_t* out96) {
    ENTER(); if (!msg || !out96) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!n) return 0;
    int rc; size_t mb = msg_bytes_total(ctx, msg_off, n, rc); if (rc) return fail(ctx, rc, "reading msg_off failed");
    if ((rc = ws_reserve(ctx, al(mb + 1) + al(4 * (n + 1)) + al(192 * n) + al(96 * n) + al(n) + (ctx->split ? al(576 * n) : 0) + 8192))) return rc;
    const uint8_t* dmsg; const uint32_t* doff;
    if ((rc = stage_in(ctx, dmsg, msg, mb ? mb : 1))) return rc; if ((rc = stage_in(ctx, doff, msg_off, n + 1))) return rc;
    u32x4* hm = ws_take<u32x4>(ctx, 12 * n); uint8_t* flags = ws_take<uint8_t>(ctx, n);
    uint8_t* dout = stage_out(ctx, out96, 96 * n);
    u32x4* scratch = ctx->split ? ws_take<u32x4>(ctx, 36 * n) : nullptr;
    if ((rc = hash_stage(ctx, dmsg, doff, n, nullptr, nullptr, hm, scratch, flags, nullptr))) return rc;
    LAUNCH(k_encode_g2, nblk(n), TPB, hm, flags, (uint8_t)FL_HM_INF, n, dout);
    if ((rc = finish_out(ctx, out96, dout, 96 * n))) return rc;
    return finish_call(ctx);
}

// hash-to-G2 stage of the verify paths: status / flags from the decode codes, H(m) into hm_soa.  scratch36 = 36 n rows that are not live yet
// (the Miller accumulator array): the split form keeps the two mapped points there, and u0, u1 in the 12 rows of hm_soa.
static int hash_stage(blsgpu_ctx* ctx, const uint8_t* dmsg, const uint32_t* doff, size_t n, const uint8_t* code_pk, const uint8_t* code_sig, u32x4* hm_soa, u32x4* scratch36,
                      uint8_t* flags, uint8_t* dstatus) {
    if (ctx->split) {
        LAUNCH(k_hash_field, nblk(n), TPB, dmsg, doff, n, code_pk, code_sig, hm_soa, flags, dstatus);
        LAUNCH(k_hash_map, nblk(2 * n), TPB, (const u32x4*)hm_soa, (const uint8_t*)dstatus, n, scratch36);
        LAUNCH(k_hash_clear, nblk(n), TPB, (const u32x4*)scratch36, (const uint8_t*)dstatus, n, hm_soa, flags);
    } else LAUNCH(k_hash_to_g2, nblk(n), TPB, dmsg, doff, n, code_pk, code_sig, hm_soa, flags, dstatus);
    return 0;
}
// Miller loop in its split form: iterations 62..0 eight at a time, lines of both pairs (a pair switched off in flags costs nothing), then the accumulator update.
// sig_sub (n bytes, nullable): the signatures were decoded without the subgroup test, and the loop does it (k_miller_lines); failures become ST_BAD_SIG
static int miller_stage_split(blsgpu_ctx* ctx, const u32x4* pk_soa, const u32x4* hm_soa, const u32x4* sig_soa, const uint8_t* flags, uint8_t* dstatus, size_t n,
                              u32x4* f_soa, u32x4* t_soa /* 36 n rows */, u32x4* lines /* MILLER_LINE_STEPS * 36 n rows */, uint8_t* sig_sub, bool coop = false) {
    for (int hi = 62; hi >= 0; hi -= MILLER_LINE_ITERS) {
        int lo = hi - MILLER_LINE_ITERS + 1 < 0 ? 0 : hi - MILLER_LINE_ITERS + 1;
        LAUNCH(k_miller_lines, nblk(2 * n), TPB, pk_soa, hm_soa, sig_soa, flags, (const uint8_t*)dstatus, n, t_soa, lines, hi, lo, sig_sub);
        if (coop) LAUNCH(k_miller_accum_coop, nblk(n, 20), 128, flags, dstatus, n, f_soa, (const u32x4*)lines, hi, lo, (const uint8_t*)sig_sub);
        else LAUNCH(k_miller_accum, nblk(n), TPB, flags, dstatus, n, f_soa, (const u32x4*)lines, hi, lo, (const uint8_t*)sig_sub);
    }
    return 0;
}
// core of verify once pk (limb-SoA + code) is known: decode sig, hash, Miller, final exp, epilogue.
// sig_sub_in_miller: with the split stage kernels, the signature's subgroup test runs on the Miller loop's running point (k_miller_lines) instead of
// in the decoder, which saves the decoder's [|x|] sig ladder (the loop computes the same point); the outcome is the same ST_BAD_SIG.
static int verify_core(blsgpu_ctx* ctx, const u32x4* pk_soa, const uint8_t* code_pk, const uint8_t* dmsg, const uint32_t* doff, const uint8_t* dsig, size_t n,
                       uint8_t* dstatus, uint32_t* dbitmap, u32x4* gt_acc /* limb-SoA n=1, multiplied into; nullable */, bool forked = false, bool sig_sub_in_miller = false) {
    u32x4* sig_soa = ws_take<u32x4>(ctx, 12 * n); u32x4* hm_soa = ws_take<u32x4>(ctx, 12 * n); u32x4* f_soa = ws_take<u32x4>(ctx, 36 * n);
    uint8_t* code_sig = ws_take<uint8_t>(ctx, n); uint8_t* flags = ws_take<uint8_t>(ctx, n);
    uint8_t* sig_sub = sig_sub_in_miller && ctx->split ? ws_take<uint8_t>(ctx, n) : nullptr;
    auto decode_sig = sig_sub ? k_decode_g2<false> : k_decode_g2<true>;
    if (forked) {
        // Small pass (the caller recorded ctx->fork before it enqueued the key decoder on ctx->stream): the signature decoder and the hash run on
        // the two lane streams beside it -- three independent serial chains instead of one after the other -- and the status rule follows the join.
        cudaStream_t main_stream = ctx->stream; int rc = 0;
        ctx->stream = ctx->lane_stream[0]; cudaStreamWaitEvent(ctx->stream, ctx->fork, 0);
        decode_sig<<<nblk(n), TPB, 0, ctx->stream>>>(dsig, n, sig_soa, code_sig); ctx->launches++; cudaEventRecord(ctx->lane_done[0], ctx->stream);
        ctx->stream = ctx->lane_stream[1]; cudaStreamWaitEvent(ctx->stream, ctx->fork, 0);
        rc = hash_stage(ctx, dmsg, doff, n, nullptr, nullptr, hm_soa, f_soa, flags, nullptr); cudaEventRecord(ctx->lane_done[1], ctx->stream);
        ctx->stream = main_stream;
        CU(cudaStreamWaitEvent(main_stream, ctx->lane_done[0], 0)); CU(cudaStreamWaitEvent(main_stream, ctx->lane_done[1], 0));
        if (rc) return rc;
        CU(cudaGetLastError());
        LAUNCH(k_status_merge, nblk(n, 256), 256, code_pk, (const uint8_t*)code_sig, n, flags, dstatus);
    } else {
    STAGE_MARK(1);
    LAUNCH(decode_sig, nblk(n), TPB, dsig, n, sig_soa, code_sig);
    STAGE_MARK(2);
    if (int rc = hash_stage(ctx, dmsg, doff, n, code_pk, code_sig, hm_soa, f_soa, flags, dstatus)) return rc;
    }
    STAGE_MARK(3);
    // Small passes are latency-bound (one item per thread: a lone warp walks the whole Miller loop and final exponentiation): below
    // VERIFY_COOP_BELOW items the hard part of the final exponentiation runs with six lanes per item (coop.cuh), which shortens its chain.
    bool coop = ctx->coop == 1 || (ctx->coop == 2 && n <= VERIFY_COOP_BELOW);
    u32x4 *y1_soa = nullptr, *y2_soa = nullptr, *snap_soa = nullptr;
    if (ctx->split) {
        // iterations 62..0 eight at a time: lines of both pairs, then the accumulator update
        u32x4* t_soa = ws_take<u32x4>(ctx, 36 * n); y1_soa = t_soa; y2_soa = ws_take<u32x4>(ctx, 36 * n);      // the running points are dead once the loop ends
        u32x4* lines = ws_take<u32x4>(ctx, (size_t)MILLER_LINE_STEPS * 2 * 18 * n);
        if (int rc = miller_stage_split(ctx, pk_soa, hm_soa, sig_soa, flags, dstatus, n, f_soa, t_soa, lines, sig_sub, coop)) return rc;
        snap_soa = lines;                                      // 144 rows of the 396-row line buffer, which is dead once the loop ends
    } else {
#if BLS_F_IN_SMEM
    { static bool attr_set = false; if (!attr_set) { cudaFuncSetAttribute(k_miller, cudaFuncAttributeMaxDynamicSharedMemorySize, TPB * 592); attr_set = true; }
      k_miller<<<nblk(n), TPB, TPB * 592, ctx->stream>>>(pk_soa, (const u32x4*)hm_soa, (const u32x4*)sig_soa, (const uint8_t*)flags, (const uint8_t*)dstatus, n, f_soa); ctx->launches++; CU(cudaGetLastError()); }
#else
    LAUNCH(k_miller, nblk(n), TPB, pk_soa, (const u32x4*)hm_soa, (const u32x4*)sig_soa, (const uint8_t*)flags, (const uint8_t*)dstatus, n, f_soa);
#endif
    }
    STAGE_MARK(4);
    if (coop) {
        LAUNCH(k_final_easy, nblk(n), TPB, f_soa, (const uint8_t*)dstatus, n);
        LAUNCH(k_final_hard_coop, nblk(n, 20), 128, f_soa, (const uint8_t*)dstatus, dstatus, n);
    } else if (ctx->split) {
        const uint8_t* cst = dstatus;
        LAUNCH(k_final_step<0>, nblk(n), TPB, f_soa, y1_soa, y2_soa, (const u32x4*)snap_soa, cst, dstatus, n);
        LAUNCH(k_final_squarings, nblk(n), TPB, (const u32x4*)f_soa, snap_soa, cst, n);
        LAUNCH(k_final_step<1>, nblk(n), TPB, f_soa, y1_soa, y2_soa, (const u32x4*)snap_soa, cst, dstatus, n);
        LAUNCH(k_final_squarings, nblk(n), TPB, (const u32x4*)y1_soa, snap_soa, cst, n);
        LAUNCH(k_final_step<2>, nblk(n), TPB, f_soa, y1_soa, y2_soa, (const u32x4*)snap_soa, cst, dstatus, n);
        LAUNCH(k_final_squarings, nblk(n), TPB, (const u32x4*)y1_soa, snap_soa, cst, n);
        LAUNCH(k_final_step<3>, nblk(n), TPB, f_soa, y1_soa, y2_soa, (const u32x4*)snap_soa, cst, dstatus, n);
        LAUNCH(k_final_squarings, nblk(n), TPB, (const u32x4*)y1_soa, snap_soa, cst, n);
        LAUNCH(k_final_step<4>, nblk(n), TPB, f_soa, y1_soa, y2_soa, (const u32x4*)snap_soa, cst, dstatus, n);
        LAUNCH(k_final_squarings, nblk(n), TPB, (const u32x4*)y2_soa, snap_soa, cst, n);
        LAUNCH(k_final_step<5>, nblk(n), TPB, f_soa, y1_soa, y2_soa, (const u32x4*)snap_soa, cst, dstatus, n);
    } else LAUNCH(k_final_exp, nblk(n), TPB, f_soa, (const uint8_t*)dstatus, dstatus, n);
    STAGE_MARK(5);
    if (dbitmap) LAUNCH(k_status_bitmap, nblk(((n + 31) / 32) * 32, 256), 256, (const uint8_t*)dstatus, n, dbitmap);
    if (gt_acc) {
        u32x4* ta = ws_take<u32x4>(ctx, 36 * ((n + 7) / 8)); u32x4* tb = ws_take<u32x4>(ctx, 36 * ((n + 63) / 64)); u32x4* one = ws_take<u32x4>(ctx, 36);
        if (int rc = gt_product(ctx, f_soa, dstatus, n, ta, tb, one)) return rc;
        LAUNCH(k_gt_mul_into, 1, 32, gt_acc, (const u32x4*)one);
    }
    STAGE_MARK(6);
    return 0;
}
static size_t verify_ws_bytes(size_t n, size_t mb) {
    return 2 * al(576 * n) + al((size_t)MILLER_LINE_STEPS * 2 * 288 * n) /* state of the split stage kernels: running points / y1, y2, line buffer / snapshots */ + al(48 * n) + al(96 * n) + al(mb + 1) + al(4 * (n + 1)) + al(n) * 7 + al(96 * n) + 2 * al(192 * n) + al(576 * n) + al(8 * ((n + 63) / 64)) +
           al(576 * ((n + 7) / 8)) + al(576 * ((n + 63) / 64)) + 3 * al(576) + 65536;
}
static int ensure_lanes(blsgpu_ctx* ctx);
// One contiguous sub-range [base, base+m) of a verify batch, enqueued entirely on ctx->stream (the caller may have pointed
// it at a lane stream): staging, the five stage kernels, epilogue, outputs, and the range's GT partial (limb-SoA, n = 1).
static int verify_range(blsgpu_ctx* ctx, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off, const uint8_t* sig96, size_t base, size_t m,
                        uint8_t* status, uint64_t* ok_bitmap, u32x4* gt_acc, size_t mb0, size_t mb) {
    int rc = 0;
    const uint8_t *dpk, *dsig, *dmsg; const uint32_t* doff;
    if ((rc = stage_in(ctx, dpk, pk48 + 48 * base, 48 * m))) return rc;
    if ((rc = stage_in(ctx, dsig, sig96 + 96 * base, 96 * m))) return rc;
    if (ctx->ptr_mode == BLSGPU_HOST) {
        // offsets in a host range are rebased by the kernel through (msg - mb0): stage the range's bytes only
        if ((rc = stage_in(ctx, dmsg, msg + mb0, mb ? mb : 1))) return rc;
        dmsg -= msg_off ? mb0 : 0;
    } else dmsg = msg_off ? msg : msg + mb0;
    if ((rc = stage_in(ctx, doff, msg_off ? msg_off + base : nullptr, m + 1))) return rc;
    uint8_t* dstatus = stage_out(ctx, status + base, m);
    uint32_t* dbitmap = (uint32_t*)stage_out(ctx, ok_bitmap ? ok_bitmap + base / 64 : nullptr, (m + 63) / 64);
    u32x4* pk_soa = ws_take<u32x4>(ctx, 6 * m); uint8_t* code_pk = ws_take<uint8_t>(ctx, m);
    if (gt_acc) LAUNCH(k_gt_set_one, 1, 32, gt_acc);
    if (dbitmap) CU(cudaMemsetAsync(dbitmap, 0, 8 * ((m + 63) / 64), ctx->stream));
    STAGE_MARK(0);
    // a small pass on the context's own stream (not a lane of a larger pass, not a profiled pass): decoders and hash side by side
    bool forked = ctx->coop == 2 && m <= VERIFY_COOP_BELOW && !ctx->prof && ctx->split && ctx->stream != ctx->lane_stream[0] && ctx->stream != ctx->lane_stream[1];
    if (forked) { if ((rc = ensure_lanes(ctx))) return rc; forked = ctx->stream != ctx->lane_stream[0] && ctx->stream != ctx->lane_stream[1]; }
    if (forked) CU(cudaEventRecord(ctx->fork, ctx->stream));
    LAUNCH(k_decode_g1, nblk(m), TPB, dpk, m, pk_soa, code_pk);
    if ((rc = verify_core(ctx, pk_soa, code_pk, dmsg, doff, dsig, m, dstatus, dbitmap, gt_acc, forked, true))) return rc;
    if ((rc = finish_out(ctx, status + base, dstatus, m))) return rc;
    if (ok_bitmap && (rc = finish_out(ctx, ok_bitmap + base / 64, (uint64_t*)dbitmap, (m + 63) / 64))) return rc;
    return 0;
}
#define MAX_LANES 4
static int ensure_lanes(blsgpu_ctx* ctx) {
    if (ctx->lane_stream[0]) return 0;
    for (int l = 0; l < MAX_LANES; l++) { CU(cudaStreamCreateWithFlags(&ctx->lane_stream[l], cudaStreamNonBlocking)); CU(cudaEventCreateWithFlags(&ctx->lane_done[l], cudaEventDisableTiming)); }
    CU(cudaEventCreateWithFlags(&ctx->fork, cudaEventDisableTiming));
    return 0;
}

int blsgpu_verify_batch(blsgpu_ctx* ctx, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off, const uint8_t* sig96, size_t n,
                        uint8_t* status, uint64_t* ok_bitmap, uint8_t* gt_acc_le576) {
    ENTER(); if (!pk48 || !msg || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    int rc = 0;
    // Passes of <= ctx->chunk items bound the workspace (8.7 KB per item: ~9 GB at 2^20, of which 6.3 KB is the line buffer of the split Miller loop).  Inside a pass the items are split into `lanes`
    // contiguous sub-ranges enqueued on separate streams: the stage kernels of different sub-ranges are independent, so the
    // tail wave of one kernel overlaps the next sub-range's kernels (and, in host mode, its H2D copies) instead of idling SMs.
    // All range boundaries are multiples of 64 so bitmap words never straddle ranges.
    uint8_t gt_host[576];
    const uint32_t* off_host = ctx->ptr_mode == BLSGPU_HOST ? msg_off : nullptr;
    size_t total_mb = 0;
    if (msg_off && !off_host) { total_mb = msg_bytes_total(ctx, msg_off, n, rc); if (rc) return fail(ctx, rc, "reading msg_off failed"); }
    for (size_t base = 0; base < n; base += ctx->chunk) {
        size_t m = n - base < ctx->chunk ? n - base : ctx->chunk;
        int lanes = ctx->lanes; if (lanes > MAX_LANES) lanes = MAX_LANES;
        while (lanes > 1 && m / lanes < 8192) lanes--;                     // keep every lane above ~0.2 waves of CTAs
        size_t per = ((m + lanes - 1) / lanes + 63) & ~(size_t)63;
        size_t ws = 65536;
        for (int l = 0; l < lanes; l++) {
            size_t lo = base + l * per, hi = lo + per < base + m ? lo + per : base + m; if (lo >= hi) break;
            size_t mb = msg_off ? (off_host ? off_host[hi] - off_host[lo] : total_mb) : 32 * (hi - lo);
            ws += verify_ws_bytes(hi - lo, ctx->ptr_mode == BLSGPU_HOST ? mb : 0) + 4096;
        }
        if ((rc = ws_reserve(ctx, ws))) return rc;
        u32x4* gt_lane[MAX_LANES] = {nullptr, nullptr, nullptr, nullptr};
        cudaStream_t main_stream = ctx->stream;
        if (lanes > 1) { if ((rc = ensure_lanes(ctx))) return rc; CU(cudaEventRecord(ctx->fork, main_stream)); }
        int used = 0;
        for (int l = 0; l < lanes; l++) {
            size_t lo = base + l * per, hi = lo + per < base + m ? lo + per : base + m; if (lo >= hi) break;
            size_t mb0 = msg_off ? (off_host ? off_host[lo] : 0) : 32 * lo;
            size_t mb = msg_off ? (off_host ? off_host[hi] - off_host[lo] : 0) : 32 * (hi - lo);
            if (gt_acc_le576) gt_lane[l] = ws_take<u32x4>(ctx, 36);
            if (lanes > 1) { ctx->stream = ctx->lane_stream[l]; cudaStreamWaitEvent(ctx->stream, ctx->fork, 0); }
            rc = verify_range(ctx, pk48, msg, msg_off, sig96, lo, hi - lo, status, ok_bitmap, gt_lane[l], mb0, mb);
            if (lanes > 1) { if (!rc) cudaEventRecord(ctx->lane_done[l], ctx->stream); ctx->stream = main_stream; }
            if (rc) return rc;
            used = l + 1;
        }
        if (lanes > 1) for (int l = 0; l < used; l++) CU(cudaStreamWaitEvent(main_stream, ctx->lane_done[l], 0));
        if (gt_acc_le576) {
            for (int l = 1; l < used; l++) LAUNCH(k_gt_mul_into, 1, 32, gt_lane[0], (const u32x4*)gt_lane[l]);
            uint8_t* dgt = ws_take<uint8_t>(ctx, 576);
            LAUNCH(k_gt_to_bytes, 1, TPB, (const u32x4*)gt_lane[0], (size_t)1, dgt, (const uint8_t*)nullptr);
            if (n <= ctx->chunk) {
                CU(cudaMemcpyAsync(gt_acc_le576, dgt, 576, ctx->ptr_mode == BLSGPU_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
            } else {
                // several passes: fold the pass partials one by one (synchronises; only taken for n > chunk)
                uint8_t part[2][576];
                CU(cudaMemcpyAsync(part[1], dgt, 576, cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream));
                if (base == 0) memcpy(gt_host, part[1], 576);
                else {
                    memcpy(part[0], gt_host, 576);
                    int saved = ctx->ptr_mode; ctx->ptr_mode = BLSGPU_HOST;
                    rc = blsgpu_gt_fold(ctx, &part[0][0], 2, gt_host); ctx->ptr_mode = saved; if (rc) return rc;
                }
                if (base + m >= n) {
                    if (ctx->ptr_mode == BLSGPU_DEVICE) { CU(cudaMemcpyAsync(gt_acc_le576, gt_host, 576, cudaMemcpyHostToDevice, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream)); }
                    else memcpy(gt_acc_le576, gt_host, 576);
                }
            }
        }
        if (ctx->ptr_mode == BLSGPU_HOST || n > ctx->chunk) CU(cudaStreamSynchronize(ctx->stream));
    }
    return 0;
}

// Random-linear-combination batch check: see include/blsgpu.h.  Single stream, passes of <= ctx->chunk items.
int blsgpu_verify_batch_rlc(blsgpu_ctx* ctx, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off, const uint8_t* sig96, size_t n,
                            const uint8_t seed16[16], uint8_t* status, uint8_t* all_ok) {
    ENTER(); if (!pk48 || !msg || !sig96 || !seed16 || !all_ok) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    int rc = 0;
    const uint32_t* off_host = ctx->ptr_mode == BLSGPU_HOST ? msg_off : nullptr;
    size_t total_mb = 0;
    if (msg_off && !off_host) { total_mb = msg_bytes_total(ctx, msg_off, n, rc); if (rc) return fail(ctx, rc, "reading msg_off failed"); }
    // accumulators that live across passes are separate allocations (the workspace is re-carved per pass)
    if (!ctx->rlc_acc) CU(cudaMalloc(&ctx->rlc_acc, 2048));
    u32x4* f_acc = reinterpret_cast<u32x4*>(ctx->rlc_acc); u32x4* s_acc = f_acc + 36; uint32_t* bad = reinterpret_cast<uint32_t*>(ctx->rlc_acc + 1024);
    uint8_t* dseed = ctx->rlc_acc + 1040; uint8_t* dok = ctx->rlc_acc + 1056;
    auto release = [&]() {};
    cudaMemcpyKind in_kind = ctx->ptr_mode == BLSGPU_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CU(cudaMemcpyAsync(dseed, seed16, 16, in_kind, ctx->stream)); CU(cudaMemsetAsync(bad, 0, 4, ctx->stream));
    LAUNCH(k_gt_set_one, 1, 32, f_acc); LAUNCH(k_g2_jac_set_identity, 1, 32, s_acc);
    for (size_t base = 0; base < n && !rc; base += ctx->chunk) {
        size_t m = n - base < ctx->chunk ? n - base : ctx->chunk;
        size_t mb0 = msg_off ? (off_host ? off_host[base] : 0) : 32 * base;
        size_t mb = msg_off ? (off_host ? off_host[base + m] - off_host[base] : total_mb) : 32 * m;
        if ((rc = ws_reserve(ctx, verify_ws_bytes(m, ctx->ptr_mode == BLSGPU_HOST ? mb : 0) + al(288 * m) + al(288 * ((m + 7) / 8)) + al(288 * ((m + 63) / 64)) + al(288) + 65536))) break;
        const uint8_t *dpk, *dsig, *dmsg; const uint32_t* doff;
        if ((rc = stage_in(ctx, dpk, pk48 + 48 * base, 48 * m))) break;
        if ((rc = stage_in(ctx, dsig, sig96 + 96 * base, 96 * m))) break;
        if (ctx->ptr_mode == BLSGPU_HOST) { if ((rc = stage_in(ctx, dmsg, msg + mb0, mb ? mb : 1))) break; dmsg -= msg_off ? mb0 : 0; }
        else dmsg = msg_off ? msg : msg + mb0;
        if ((rc = stage_in(ctx, doff, msg_off ? msg_off + base : nullptr, m + 1))) break;
        uint8_t* dstatus = status ? stage_out(ctx, status + base, m) : ws_take<uint8_t>(ctx, m);
        u32x4* pk_soa = ws_take<u32x4>(ctx, 6 * m); uint8_t* code_pk = ws_take<uint8_t>(ctx, m);
        u32x4* sig_soa = ws_take<u32x4>(ctx, 12 * m); u32x4* hm_soa = ws_take<u32x4>(ctx, 12 * m); u32x4* f_soa = ws_take<u32x4>(ctx, 36 * m);
        uint8_t* code_sig = ws_take<uint8_t>(ctx, m); uint8_t* flags = ws_take<uint8_t>(ctx, m);
        u32x4* rs = ws_take<u32x4>(ctx, 18 * m); u32x4* ja = ws_take<u32x4>(ctx, 18 * ((m + 7) / 8)); u32x4* jb = ws_take<u32x4>(ctx, 18 * ((m + 63) / 64)); u32x4* jone = ws_take<u32x4>(ctx, 18);
        u32x4* ta = ws_take<u32x4>(ctx, 36 * ((m + 7) / 8)); u32x4* tb = ws_take<u32x4>(ctx, 36 * ((m + 63) / 64)); u32x4* one = ws_take<u32x4>(ctx, 36);
        LAUNCH(k_decode_g1, nblk(m), TPB, dpk, m, pk_soa, code_pk);
        LAUNCH(k_decode_g2<true>, nblk(m), TPB, dsig, m, sig_soa, code_sig);
        if ((rc = hash_stage(ctx, dmsg, doff, m, code_pk, code_sig, hm_soa, f_soa, flags, dstatus))) break;
        LAUNCH(k_any_bad, nblk(((m + 31) / 32) * 32, 256), 256, (const uint8_t*)dstatus, m, bad);
        LAUNCH(k_rlc_scale, nblk(m), TPB, pk_soa, (const u32x4*)sig_soa, flags, (const uint8_t*)dstatus, m, base, (const uint8_t*)dseed, rs);
        {   // sum of the scaled signatures (radix-8 tree, like the GT product)
            const u32x4* cur = rs; size_t cnt = m; u32x4* bufs[2] = {ja, jb}; int which = 0;
            while (true) {
                size_t T = (cnt + 7) / 8; u32x4* out = T == 1 ? jone : bufs[which];
                LAUNCH(k_g2_jac_reduce, nblk(T), TPB, cur, cnt, out, T);
                if (T == 1) break;
                cur = out; cnt = T; which ^= 1;
            }
            LAUNCH(k_g2_jac_add_into, 1, 32, s_acc, (const u32x4*)jone);
        }
        if (ctx->split) {                                        // verify_ws_bytes counts the running-point array and the line buffer
            u32x4* t_soa = ws_take<u32x4>(ctx, 36 * m); u32x4* lines = ws_take<u32x4>(ctx, (size_t)MILLER_LINE_STEPS * 2 * 18 * m);
            if ((rc = miller_stage_split(ctx, pk_soa, hm_soa, sig_soa, flags, dstatus, m, f_soa, t_soa, lines, nullptr))) break;
        } else LAUNCH(k_miller, nblk(m), TPB, (const u32x4*)pk_soa, (const u32x4*)hm_soa, (const u32x4*)sig_soa, (const uint8_t*)flags, (const uint8_t*)dstatus, m, f_soa);
        if ((rc = gt_product(ctx, f_soa, dstatus, m, ta, tb, one))) break;
        LAUNCH(k_gt_mul_into, 1, 32, f_acc, (const u32x4*)one);
        if (status && (rc = finish_out(ctx, status + base, dstatus, m))) break;
        if (ctx->ptr_mode == BLSGPU_HOST || n > ctx->chunk) { cudaError_t e = cudaStreamSynchronize(ctx->stream); if (e != cudaSuccess) { rc = fail(ctx, BLSGPU_ERR_CUDA, "sync failed: %s", cudaGetErrorString(e)); break; } }
    }
    if (!rc) {
        k_rlc_finish<<<1, 32, 0, ctx->stream>>>(f_acc, s_acc, bad, dok); ctx->launches++;
        cudaError_t e = cudaMemcpyAsync(all_ok, dok, 1, ctx->ptr_mode == BLSGPU_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess && ctx->ptr_mode == BLSGPU_HOST) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, BLSGPU_ERR_CUDA, "rlc finish failed: %s", cudaGetErrorString(e));
    }
    release();
    return rc;
}

// Batch check that returns the EXACT per-item outcome (SURVEY 8(f)-3: "fall back to per-item checks to recover the exact bitmap when
// the batch fails").  One random-linear-combination equation per PIECE of RLC_PIECE items, all pieces finished side by side; a piece
// whose equation fails is re-run through the per-item path (blsgpu_verify_batch) inside this call.  status[i] and ok_bitmap equal
// blsgpu_verify_batch's except with probability <= 2^-64 per failing piece over the seed; fallback_items (nullable, host) = items re-run.
#define RLC_PIECE 4096
int blsgpu_verify_batch_rlc_bisect(blsgpu_ctx* ctx, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off, const uint8_t* sig96, size_t n,
                                   const uint8_t seed16[16], uint8_t* status, uint64_t* ok_bitmap, uint64_t* fallback_items) {
    ENTER(); if (!pk48 || !msg || !sig96 || !seed16 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (fallback_items) *fallback_items = 0;
    if (!n) return 0;
    int rc = 0; bool host = ctx->ptr_mode == BLSGPU_HOST;
    const uint32_t* off_host = host ? msg_off : nullptr;
    size_t total_mb = 0;
    if (msg_off && !off_host) { total_mb = msg_bytes_total(ctx, msg_off, n, rc); if (rc) return fail(ctx, rc, "reading msg_off failed"); }
    if (!ctx->rlc_acc) CU(cudaMalloc(&ctx->rlc_acc, 2048));
    uint8_t* dseed = ctx->rlc_acc + 1040;
    CU(cudaMemcpyAsync(dseed, seed16, 16, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
    const size_t L = RLC_PIECE;
    std::vector<uint8_t> piece_ok((n + L - 1) / L, 1);
    size_t chunk = ctx->chunk >= L ? ctx->chunk / L * L : L;                 // pieces never straddle passes
    for (size_t base = 0; base < n; base += chunk) {
        size_t m = n - base < chunk ? n - base : chunk, P = (m + L - 1) / L, T0 = (L + 7) / 8;
        size_t mb0 = msg_off ? (off_host ? off_host[base] : 0) : 32 * base;
        size_t mb = msg_off ? (off_host ? off_host[base + m] - off_host[base] : total_mb) : 32 * m;
        if ((rc = ws_reserve(ctx, verify_ws_bytes(m, host ? mb : 0) + al(288 * m) + 2 * al(288 * P * T0) + 2 * al(576 * P * T0) + al(P) + 65536))) return rc;
        const uint8_t *dpk, *dsig, *dmsg; const uint32_t* doff;
        if ((rc = stage_in(ctx, dpk, pk48 + 48 * base, 48 * m))) return rc;
        if ((rc = stage_in(ctx, dsig, sig96 + 96 * base, 96 * m))) return rc;
        if (host) { if ((rc = stage_in(ctx, dmsg, msg + mb0, mb ? mb : 1))) return rc; dmsg -= msg_off ? mb0 : 0; }
        else dmsg = msg_off ? msg : msg + mb0;
        if ((rc = stage_in(ctx, doff, msg_off ? msg_off + base : nullptr, m + 1))) return rc;
        uint8_t* dstatus = stage_out(ctx, status + base, m);
        u32x4* pk_soa = ws_take<u32x4>(ctx, 6 * m); uint8_t* code_pk = ws_take<uint8_t>(ctx, m);
        u32x4* sig_soa = ws_take<u32x4>(ctx, 12 * m); u32x4* hm_soa = ws_take<u32x4>(ctx, 12 * m); u32x4* f_soa = ws_take<u32x4>(ctx, 36 * m);
        uint8_t* code_sig = ws_take<uint8_t>(ctx, m); uint8_t* flags = ws_take<uint8_t>(ctx, m);
        u32x4* rs = ws_take<u32x4>(ctx, 18 * m); u32x4* ja = ws_take<u32x4>(ctx, 18 * P * T0); u32x4* jb = ws_take<u32x4>(ctx, 18 * P * T0);
        u32x4* ta = ws_take<u32x4>(ctx, 36 * P * T0); u32x4* tb = ws_take<u32x4>(ctx, 36 * P * T0); uint8_t* dok = ws_take<uint8_t>(ctx, P);
        LAUNCH(k_decode_g1, nblk(m), TPB, dpk, m, pk_soa, code_pk);
        LAUNCH(k_decode_g2<true>, nblk(m), TPB, dsig, m, sig_soa, code_sig);
        if ((rc = hash_stage(ctx, dmsg, doff, m, code_pk, code_sig, hm_soa, f_soa, flags, dstatus))) return rc;
        LAUNCH(k_rlc_scale, nblk(m), TPB, pk_soa, (const u32x4*)sig_soa, flags, (const uint8_t*)dstatus, m, base, (const uint8_t*)dseed, rs);
        const u32x4* s_piece; const u32x4* f_piece;
        {   // per-piece sums of the scaled signatures: radix-8 trees, all pieces in one launch per level
            const u32x4* cur = rs; size_t cnt_n = m, len = L; u32x4* bufs[2] = {ja, jb}; int which = 0;
            while (true) {
                size_t T = (len + 7) / 8; u32x4* out = bufs[which];
                k_g2_jac_reduce_seg<<<dim3(nblk(T), (unsigned)P), TPB, 0, ctx->stream>>>(cur, cnt_n, len, out, T, P); ctx->launches++; CU(cudaGetLastError());
                cur = out; cnt_n = P * T; len = T; which ^= 1;
                if (T == 1) break;
            }
            s_piece = cur;
        }
        if (ctx->split) {
            u32x4* t_soa = ws_take<u32x4>(ctx, 36 * m); u32x4* lines = ws_take<u32x4>(ctx, (size_t)MILLER_LINE_STEPS * 2 * 18 * m);
            if ((rc = miller_stage_split(ctx, pk_soa, hm_soa, sig_soa, flags, dstatus, m, f_soa, t_soa, lines, nullptr))) return rc;
        } else LAUNCH(k_miller, nblk(m), TPB, (const u32x4*)pk_soa, (const u32x4*)hm_soa, (const u32x4*)sig_soa, (const uint8_t*)flags, (const uint8_t*)dstatus, m, f_soa);
        {
            const u32x4* cur = f_soa; const uint8_t* st = dstatus; size_t cnt_n = m, len = L; u32x4* bufs[2] = {ta, tb}; int which = 0;
            while (true) {
                size_t T = (len + 7) / 8; u32x4* out = bufs[which];
                k_gt_reduce_seg<<<dim3(nblk(T), (unsigned)P), TPB, 0, ctx->stream>>>(cur, st, cnt_n, len, out, T, P); ctx->launches++; CU(cudaGetLastError());
                cur = out; st = nullptr; cnt_n = P * T; len = T; which ^= 1;
                if (T == 1) break;
            }
            f_piece = cur;
        }
        LAUNCH(k_rlc_finish_seg, (unsigned)P, 32, f_piece, s_piece, P, dok);
        if ((rc = finish_out(ctx, status + base, dstatus, m))) return rc;
        CU(cudaMemcpyAsync(piece_ok.data() + base / L, dok, P, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    // failing pieces: the per-item path on exactly those items (adjacent failing pieces are merged into one call)
    uint64_t rerun = 0;
    for (size_t p = 0; p < piece_ok.size(); ) {
        if (piece_ok[p]) { p++; continue; }
        size_t q = p; while (q < piece_ok.size() && !piece_ok[q]) q++;
        size_t lo = p * L, hi = q * L < n ? q * L : n;
        const uint8_t* m_ptr; const uint32_t* o_ptr;
        std::vector<uint32_t> rebased;
        if (!msg_off) { m_ptr = msg + 32 * lo; o_ptr = nullptr; }
        else if (host) { rebased.resize(hi - lo + 1); for (size_t i = 0; i <= hi - lo; i++) rebased[i] = msg_off[lo + i] - msg_off[lo]; m_ptr = msg + msg_off[lo]; o_ptr = rebased.data(); }
        else { m_ptr = msg; o_ptr = msg_off + lo; }                       // device offsets are absolute into msg
        if ((rc = blsgpu_verify_batch(ctx, pk48 + 48 * lo, m_ptr, o_ptr, sig96 + 96 * lo, hi - lo, status + lo, nullptr, nullptr))) return rc;
        if (!host) CU(cudaStreamSynchronize(ctx->stream));
        rerun += hi - lo; p = q;
    }
    if (fallback_items) *fallback_items = rerun;
    if (ok_bitmap) {
        if (host) { size_t words = (n + 63) / 64; for (size_t w = 0; w < words; w++) ok_bitmap[w] = 0; for (size_t i = 0; i < n; i++) if (status[i] == ST_OK) ok_bitmap[i >> 6] |= 1ull << (i & 63); }
        else { CU(cudaMemsetAsync(ok_bitmap, 0, 8 * ((n + 63) / 64), ctx->stream)); LAUNCH(k_status_bitmap, nblk(((n + 31) / 32) * 32, 256), 256, (const uint8_t*)status, n, (uint32_t*)ok_bitmap); }
    }
    return finish_call(ctx);
}

int blsgpu_gt_fold(blsgpu_ctx* ctx, const uint8_t* parts, size_t nparts, uint8_t* out) {
    ENTER(); if (!parts || !out || !nparts) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    if (int rc = ws_reserve(ctx, al(576 * nparts) * 2 + al(576 * ((nparts + 7) / 8)) + al(576 * ((nparts + 63) / 64)) + 2 * al(576) + 8192)) return rc;
    const uint8_t* din; if (int rc = stage_in(ctx, din, parts, 576 * nparts)) return rc;
    u32x4* soa = ws_take<u32x4>(ctx, 36 * nparts); u32x4* ta = ws_take<u32x4>(ctx, 36 * ((nparts + 7) / 8)); u32x4* tb = ws_take<u32x4>(ctx, 36 * ((nparts + 63) / 64)); u32x4* one = ws_take<u32x4>(ctx, 36);
    uint8_t* dout = stage_out(ctx, out, 576);
    LAUNCH(k_gt_from_bytes, nblk(nparts), TPB, din, nparts, soa);
    if (int rc = gt_product(ctx, soa, nullptr, nparts, ta, tb, one)) return rc;
    LAUNCH(k_gt_to_bytes, 1, TPB, (const u32x4*)one, (size_t)1, dout, (const uint8_t*)nullptr);
    if (int rc = finish_out(ctx, out, dout, 576)) return rc;
    return finish_call(ctx);
}

int blsgpu_pairing_gt(blsgpu_ctx* ctx, const uint8_t* g1_48, const uint8_t* g2_96, size_t npairs, size_t nprod, uint8_t* gt, uint8_t* status) {
    ENTER(); if (!g1_48 || !g2_96 || !gt || npairs < 1 || npairs > 2) return fail(ctx, BLSGPU_ERR_ARG, "bad argument (npairs must be 1 or 2)");
    if (!nprod) return 0;
    size_t tot = npairs * nprod;
    if (int rc = ws_reserve(ctx, al(48 * tot) + al(96 * tot) + al(96 * tot) + al(192 * tot) + 3 * al(tot) + al(576 * nprod) * 2 + 2 * al(nprod) + 8192)) return rc;
    const uint8_t *d1, *d2; if (int rc = stage_in(ctx, d1, g1_48, 48 * tot)) return rc; if (int rc = stage_in(ctx, d2, g2_96, 96 * tot)) return rc;
    u32x4* s1 = ws_take<u32x4>(ctx, 6 * tot); u32x4* s2 = ws_take<u32x4>(ctx, 12 * tot); uint8_t* c1 = ws_take<uint8_t>(ctx, tot); uint8_t* c2 = ws_take<uint8_t>(ctx, tot);
    u32x4* f = ws_take<u32x4>(ctx, 36 * nprod);
    uint8_t* dst = status && ctx->ptr_mode == BLSGPU_DEVICE ? status : ws_take<uint8_t>(ctx, nprod);
    uint8_t* dgt = stage_out(ctx, gt, 576 * nprod);
    LAUNCH(k_decode_g1, nblk(tot), TPB, d1, tot, s1, c1);
    LAUNCH(k_decode_g2<true>, nblk(tot), TPB, d2, tot, s2, c2);
    LAUNCH(k_miller_pairs, nblk(nprod), TPB, (const u32x4*)s1, (const u32x4*)s2, (const uint8_t*)c1, (const uint8_t*)c2, npairs, nprod, f, dst);
    uint8_t* scratch = ws_take<uint8_t>(ctx, nprod);       // is_one outcome, not reported by this hook
    LAUNCH(k_final_exp, nblk(nprod), TPB, f, (const uint8_t*)dst, scratch, nprod);
    LAUNCH(k_gt_to_bytes, nblk(nprod), TPB, (const u32x4*)f, nprod, dgt, (const uint8_t*)dst);
    if (int rc = finish_out(ctx, gt, dgt, 576 * nprod)) return rc;
    if (status) if (int rc = finish_out(ctx, status, dst, nprod)) return rc;
    return finish_call(ctx);
}

int blsgpu_sk_to_pk_batch(blsgpu_ctx* ctx, const uint8_t* sk32, size_t n, uint8_t* pk48, uint8_t* status) {
    ENTER(); if (!sk32 || !pk48) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!n) return 0;
    if (int rc = ws_reserve(ctx, al(32 * n) + al(48 * n) + al(n) + 4096)) return rc;
    const uint8_t* dsk; if (int rc = stage_in(ctx, dsk, sk32, 32 * n)) return rc;
    uint8_t* dpk = stage_out(ctx, pk48, 48 * n); uint8_t* dst = stage_out(ctx, status, n);
    LAUNCH(k_scalar_mul_g1, nblk(n), TPB, dsk, n, dpk, dst);
    if (int rc = finish_out(ctx, pk48, dpk, 48 * n)) return rc;
    if (int rc = finish_out(ctx, status, dst, n)) return rc;
    return finish_call(ctx);
}
int blsgpu_sign_batch(blsgpu_ctx* ctx, const uint8_t* sk32, const uint8_t* msg, const uint32_t* msg_off, size_t n, uint8_t* sig96, uint8_t* status) {
    ENTER(); if (!sk32 || !msg || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!n) return 0;
    int rc; size_t mb = msg_bytes_total(ctx, msg_off, n, rc); if (rc) return fail(ctx, rc, "reading msg_off failed");
    if ((rc = ws_reserve(ctx, al(32 * n) + al(mb + 1) + al(4 * (n + 1)) + al(192 * n) + al(96 * n) + 2 * al(n) + 8192))) return rc;
    const uint8_t *dsk, *dmsg; const uint32_t* doff;
    if ((rc = stage_in(ctx, dsk, sk32, 32 * n))) return rc; if ((rc = stage_in(ctx, dmsg, msg, mb ? mb : 1))) return rc; if ((rc = stage_in(ctx, doff, msg_off, n + 1))) return rc;
    u32x4* hm = ws_take<u32x4>(ctx, 12 * n); uint8_t* flags = ws_take<uint8_t>(ctx, n);
    uint8_t* dsig = stage_out(ctx, sig96, 96 * n); uint8_t* dst = stage_out(ctx, status, n);
    LAUNCH(k_hash_to_g2, nblk(n), TPB, dmsg, doff, n, (const uint8_t*)nullptr, (const uint8_t*)nullptr, hm, flags, (uint8_t*)nullptr);
    LAUNCH(k_scalar_mul_g2, nblk(n), TPB, dsk, (const u32x4*)hm, (const uint8_t*)flags, n, dsig, dst);
    if ((rc = finish_out(ctx, sig96, dsig, 96 * n))) return rc; if ((rc = finish_out(ctx, status, dst, n))) return rc;
    return finish_call(ctx);
}

static int seg_total(blsgpu_ctx* ctx, const uint32_t* seg_off, size_t nseg, size_t& npts) {
    if (ctx->ptr_mode == BLSGPU_HOST) { npts = seg_off[nseg]; return 0; }
    uint32_t last = 0; CU(cudaMemcpyAsync(&last, seg_off + nseg, 4, cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream)); npts = last; return 0;
}
int blsgpu_g1_aggregate(blsgpu_ctx* ctx, const uint8_t* pts48, const uint32_t* seg_off, size_t nseg, uint8_t* out48, uint8_t* status) {
    ENTER(); if (!seg_off || !out48 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!nseg) return 0;
    size_t npts; if (int rc = seg_total(ctx, seg_off, nseg, npts)) return rc;
    if (npts && !pts48) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (int rc = ws_reserve(ctx, al(48 * npts + 16) + al(4 * (nseg + 1)) + al(96 * npts + 16) + al(npts + 1) + al(96 * nseg) + al(144 * nseg) + al(48 * nseg) + 3 * al(nseg) + 8192)) return rc;
    const uint8_t* din; const uint32_t* dseg;
    if (int rc = stage_in(ctx, din, pts48, 48 * npts)) return rc; if (int rc = stage_in(ctx, dseg, seg_off, nseg + 1)) return rc;
    u32x4* soa = ws_take<u32x4>(ctx, 6 * npts + 1); uint8_t* code = ws_take<uint8_t>(ctx, npts + 1);
    u32x4* osoa = ws_take<u32x4>(ctx, 6 * nseg); uint8_t* oinf = ws_take<uint8_t>(ctx, nseg);
    uint8_t* dout = stage_out(ctx, out48, 48 * nseg); uint8_t* dst = stage_out(ctx, status, nseg);
    if (npts) LAUNCH(k_decode_g1, nblk(npts), TPB, din, npts, soa, code);
    { int L = seg_lanes(npts / nseg); u32x4* ojac = ws_take<u32x4>(ctx, 9 * nseg);
      LAUNCH(k_segsum<fp>, nblk(nseg, SEG_WARPS * (32 / L)), 32 * SEG_WARPS, (const u32x4*)soa, (const uint8_t*)code, npts, dseg, (size_t)0, (const uint64_t*)nullptr, nseg, ojac, dst, (uint8_t)ST_BAD_PK, (const uint32_t*)nullptr, L);
      LAUNCH(k_jac_to_aff<fp>, nblk(nseg), TPB, (const u32x4*)ojac, nseg, osoa, oinf); }
    LAUNCH(k_encode_g1, nblk(nseg), TPB, (const u32x4*)osoa, (const uint8_t*)oinf, nseg, dout);
    if (int rc = finish_out(ctx, out48, dout, 48 * nseg)) return rc; if (int rc = finish_out(ctx, status, dst, nseg)) return rc;
    return finish_call(ctx);
}
int blsgpu_g2_aggregate(blsgpu_ctx* ctx, const uint8_t* pts96, const uint32_t* seg_off, size_t nseg, uint8_t* out96, uint8_t* status) {
    ENTER(); if (!seg_off || !out96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!nseg) return 0;
    size_t npts; if (int rc = seg_total(ctx, seg_off, nseg, npts)) return rc;
    if (npts && !pts96) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (int rc = ws_reserve(ctx, al(96 * npts + 16) + al(4 * (nseg + 1)) + al(192 * npts + 16) + al(npts + 1) + al(192 * nseg) + al(288 * nseg) + al(96 * nseg) + 3 * al(nseg) + 8192)) return rc;
    const uint8_t* din; const uint32_t* dseg;
    if (int rc = stage_in(ctx, din, pts96, 96 * npts)) return rc; if (int rc = stage_in(ctx, dseg, seg_off, nseg + 1)) return rc;
    u32x4* soa = ws_take<u32x4>(ctx, 12 * npts + 1); uint8_t* code = ws_take<uint8_t>(ctx, npts + 1);
    u32x4* osoa = ws_take<u32x4>(ctx, 12 * nseg); uint8_t* oinf = ws_take<uint8_t>(ctx, nseg);
    uint8_t* dout = stage_out(ctx, out96, 96 * nseg); uint8_t* dst = stage_out(ctx, status, nseg);
    if (npts) LAUNCH(k_decode_g2<true>, nblk(npts), TPB, din, npts, soa, code);
    { int L = seg_lanes(npts / nseg); u32x4* ojac = ws_take<u32x4>(ctx, 18 * nseg);
      LAUNCH(k_segsum<fp2>, nblk(nseg, SEG_WARPS * (32 / L)), 32 * SEG_WARPS, (const u32x4*)soa, (const uint8_t*)code, npts, dseg, (size_t)0, (const uint64_t*)nullptr, nseg, ojac, dst, (uint8_t)ST_BAD_SIG, (const uint32_t*)nullptr, L);
      LAUNCH(k_jac_to_aff<fp2>, nblk(nseg), TPB, (const u32x4*)ojac, nseg, osoa, oinf); }
    LAUNCH(k_encode_g2, nblk(nseg), TPB, (const u32x4*)osoa, (const uint8_t*)oinf, (uint8_t)1, nseg, dout);
    if (int rc = finish_out(ctx, out96, dout, 96 * nseg)) return rc; if (int rc = finish_out(ctx, status, dst, nseg)) return rc;
    return finish_call(ctx);
}

int blsgpu_fast_aggregate_verify_batch(blsgpu_ctx* ctx, const uint8_t* pks48, const uint64_t* bitmap, size_t k, const uint8_t* msg32, const uint8_t* sig96, size_t ncomm,
                                       uint8_t* status, uint8_t* agg_pk48_out) {
    ENTER(); if (!msg32 || !sig96 || !status || (k && !pks48)) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!ncomm) return 0;
    int rc; size_t npts = ncomm * k;
    size_t need = al(48 * npts + 16) + al(8 * ((npts + 63) / 64 + 1)) + al(96 * npts + 16) + al(npts + 1) + al(96 * ncomm) * 2 + al(144 * ncomm) + al(48 * ncomm) + 4 * al(ncomm) + verify_ws_bytes(ncomm, 32 * ncomm);
    if ((rc = ws_reserve(ctx, need))) return rc;
    const uint8_t *dpks, *dmsg, *dsig; const uint64_t* dbm;
    if ((rc = stage_in(ctx, dpks, pks48, 48 * npts))) return rc; if ((rc = stage_in(ctx, dbm, bitmap, (npts + 63) / 64))) return rc;
    if ((rc = stage_in(ctx, dmsg, msg32, 32 * ncomm))) return rc; if ((rc = stage_in(ctx, dsig, sig96, 96 * ncomm))) return rc;
    u32x4* soa = ws_take<u32x4>(ctx, 6 * npts + 1); uint8_t* code = ws_take<uint8_t>(ctx, npts + 1);
    u32x4* agg_soa = ws_take<u32x4>(ctx, 6 * ncomm); uint8_t* agg_inf = ws_take<uint8_t>(ctx, ncomm); uint8_t* agg_st = ws_take<uint8_t>(ctx, ncomm); uint8_t* code_pk = ws_take<uint8_t>(ctx, ncomm);
    uint8_t* dstatus = stage_out(ctx, status, ncomm); uint8_t* dagg = stage_out(ctx, agg_pk48_out, 48 * ncomm);
    if (npts) LAUNCH(k_decode_g1, nblk(npts), TPB, dpks, npts, soa, code);
    { int L = seg_lanes(k); u32x4* ojac = ws_take<u32x4>(ctx, 9 * ncomm);
      LAUNCH(k_segsum<fp>, nblk(ncomm, SEG_WARPS * (32 / L)), 32 * SEG_WARPS, (const u32x4*)soa, (const uint8_t*)code, npts, (const uint32_t*)nullptr, k, dbm, ncomm, ojac, agg_st, (uint8_t)ST_BAD_PK, (const uint32_t*)nullptr, L);
      LAUNCH(k_jac_to_aff<fp>, nblk(ncomm), TPB, (const u32x4*)ojac, ncomm, agg_soa, agg_inf); }
    if (dagg) LAUNCH(k_encode_g1, nblk(ncomm), TPB, (const u32x4*)agg_soa, (const uint8_t*)agg_inf, ncomm, dagg);
    LAUNCH(k_fav_status, nblk(ncomm), TPB, (const uint8_t*)agg_st, (const uint8_t*)agg_inf, (const uint8_t*)nullptr, ncomm, code_pk);
    // the aggregate of subgroup points is in the subgroup: the check() of bls.rs:438 on it cannot fail, so it is not re-run
    if ((rc = verify_core(ctx, agg_soa, code_pk, dmsg, nullptr, dsig, ncomm, dstatus, nullptr, nullptr))) return rc;
    if ((rc = finish_out(ctx, status, dstatus, ncomm))) return rc; if ((rc = finish_out(ctx, agg_pk48_out, dagg, 48 * ncomm))) return rc;
    return finish_call(ctx);
}

// ---- Eth2 AggregateVerify (distinct messages; the category reference tests/readme.md:4-7 names and does not vendor):
// signature s covers the pairs [pair_off[s], pair_off[s+1]): true iff  e(-g1, sig_s) * prod_j e(pk_j, H(m_j)) == 1  with every key
// KeyValidate-d (decodes, not the identity, in the subgroup) and the signature in the subgroup.  Every pair's Miller loop is an
// independent item (full parallelism over npairs + nsig loops, the single-pair form of k_miller); the Miller values of a signature are
// multiplied and ONE final exponentiation per signature decides.  status[s]: 0 / 1, 2 = a key failed, 3 = the signature failed, 4 = no pairs.
int blsgpu_aggregate_verify_batch(blsgpu_ctx* ctx, const uint8_t* pks48, const uint8_t* msg, const uint32_t* msg_off, const uint32_t* pair_off,
                                  const uint8_t* sig96, size_t nsig, uint8_t* status) {
    ENTER(); if (!pair_off || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!nsig) return 0;
    int rc; size_t npairs; if ((rc = seg_total(ctx, pair_off, nsig, npairs))) return rc;
    if (npairs && (!pks48 || !msg)) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    size_t mb = msg_bytes_total(ctx, msg_off, npairs, rc); if (rc) return fail(ctx, rc, "reading msg_off failed");
    size_t np1 = npairs ? npairs : 1;
    if ((rc = ws_reserve(ctx, al(48 * np1) + al(mb + 1) + al(4 * (np1 + 1)) + al(4 * (nsig + 1)) + al(96 * nsig) + al(96 * np1) + 2 * al(192 * np1) + al(576 * np1) + 5 * al(np1) +
                              al(96 * nsig) + 2 * al(192 * nsig) + al(576 * nsig) + 4 * al(nsig) + 65536))) return rc;
    const uint8_t *dpk, *dmsg, *dsig; const uint32_t *doff, *dpair;
    if ((rc = stage_in(ctx, dpk, pks48, 48 * npairs))) return rc; if ((rc = stage_in(ctx, dmsg, msg, mb ? mb : 1))) return rc;
    if ((rc = stage_in(ctx, doff, msg_off, npairs + 1))) return rc; if ((rc = stage_in(ctx, dpair, pair_off, nsig + 1))) return rc;
    if ((rc = stage_in(ctx, dsig, sig96, 96 * nsig))) return rc;
    u32x4* pk_soa = ws_take<u32x4>(ctx, 6 * np1); u32x4* hm_soa = ws_take<u32x4>(ctx, 12 * np1); u32x4* zero_g2 = ws_take<u32x4>(ctx, 12 * np1); u32x4* f_pair = ws_take<u32x4>(ctx, 36 * np1);
    uint8_t* code_pk = ws_take<uint8_t>(ctx, np1); uint8_t* code_inf = ws_take<uint8_t>(ctx, np1); uint8_t* pflags = ws_take<uint8_t>(ctx, np1); uint8_t* pstatus = ws_take<uint8_t>(ctx, np1);
    u32x4* sig_soa = ws_take<u32x4>(ctx, 12 * nsig); u32x4* zero_g1 = ws_take<u32x4>(ctx, 6 * nsig); u32x4* zero_hm = ws_take<u32x4>(ctx, 12 * nsig); u32x4* f_sig = ws_take<u32x4>(ctx, 36 * nsig);
    uint8_t* code_sig = ws_take<uint8_t>(ctx, nsig); uint8_t* sflags = ws_take<uint8_t>(ctx, nsig); uint8_t* sstatus = ws_take<uint8_t>(ctx, nsig);
    uint8_t* dstatus = stage_out(ctx, status, nsig);
    if (npairs) {
        LAUNCH(k_decode_g1, nblk(npairs), TPB, dpk, npairs, pk_soa, code_pk);
        CU(cudaMemsetAsync(code_inf, DEC_INF, npairs, ctx->stream));          // "signature = identity" for every pair item: k_hash_to_g2 then switches the (-g1, sig) slot off
        CU(cudaMemsetAsync(zero_g2, 0, 192 * npairs, ctx->stream));
        LAUNCH(k_hash_to_g2, nblk(npairs), TPB, dmsg, doff, npairs, (const uint8_t*)code_pk, (const uint8_t*)code_inf, hm_soa, pflags, pstatus);
        LAUNCH(k_miller, nblk(npairs), TPB, (const u32x4*)pk_soa, (const u32x4*)hm_soa, (const u32x4*)zero_g2, (const uint8_t*)pflags, (const uint8_t*)pstatus, npairs, f_pair);
    }
    LAUNCH(k_decode_g2<true>, nblk(nsig), TPB, dsig, nsig, sig_soa, code_sig);
    LAUNCH(k_aggv_sig_status, nblk(nsig), TPB, (const uint8_t*)code_sig, nsig, sstatus, sflags);
    CU(cudaMemsetAsync(zero_g1, 0, 96 * nsig, ctx->stream)); CU(cudaMemsetAsync(zero_hm, 0, 192 * nsig, ctx->stream));
    LAUNCH(k_miller, nblk(nsig), TPB, (const u32x4*)zero_g1, (const u32x4*)zero_hm, (const u32x4*)sig_soa, (const uint8_t*)sflags, (const uint8_t*)sstatus, nsig, f_sig);
    LAUNCH(k_aggv_combine, nblk(nsig), TPB, (const u32x4*)f_pair, (const uint8_t*)pstatus, npairs, dpair, f_sig, (const uint8_t*)sstatus, nsig, dstatus);
    LAUNCH(k_final_exp, nblk(nsig), TPB, f_sig, (const uint8_t*)dstatus, dstatus, nsig);
    if ((rc = finish_out(ctx, status, dstatus, nsig))) return rc;
    return finish_call(ctx);
}

// ---- the uncompressed wire format: compressed <-> uncompressed with full validation of the input (status: BLSGPU_DE_* per item)
static int recode(blsgpu_ctx* ctx, const uint8_t* in, size_t n, uint8_t* out, uint8_t* status, size_t in_sz, size_t out_sz, bool g2, int to_unc) {
    if (!in || !out) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    if (!n) return 0;
    if (int rc = ws_reserve(ctx, al(in_sz * n) + al(out_sz * n) + al(n) + 8192)) return rc;
    const uint8_t* din; if (int rc = stage_in(ctx, din, in, in_sz * n)) return rc;
    uint8_t* dout = stage_out(ctx, out, out_sz * n); uint8_t* dst = stage_out(ctx, status, n);
    if (g2) LAUNCH(k_g2_recode, nblk(n), TPB, din, n, dout, dst, to_unc); else LAUNCH(k_g1_recode, nblk(n), TPB, din, n, dout, dst, to_unc);
    if (int rc = finish_out(ctx, out, dout, out_sz * n)) return rc;
    if (int rc = finish_out(ctx, status, dst, n)) return rc;
    return finish_call(ctx);
}
int blsgpu_g1_uncompress(blsgpu_ctx* ctx, const uint8_t* in48, size_t n, uint8_t* out96, uint8_t* status) { ENTER(); return recode(ctx, in48, n, out96, status, 48, 96, false, 1); }
int blsgpu_g1_compress(blsgpu_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* out48, uint8_t* status) { ENTER(); return recode(ctx, in96, n, out48, status, 96, 48, false, 0); }
int blsgpu_g2_uncompress(blsgpu_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* out192, uint8_t* status) { ENTER(); return recode(ctx, in96, n, out192, status, 96, 192, true, 1); }
int blsgpu_g2_compress(blsgpu_ctx* ctx, const uint8_t* in192, size_t n, uint8_t* out96, uint8_t* status) { ENTER(); return recode(ctx, in192, n, out96, status, 192, 96, true, 0); }

// ---- resident validator pool (cfg 3a): keys are decoded and subgroup-checked once and stay in HBM as affine limb-SoA
int blsgpu_pool_create(blsgpu_ctx* ctx, const uint8_t* pks48, size_t n, int* handle, uint8_t* status) {
    ENTER(); if (!pks48 || !handle || !n) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    int h = -1; for (int i = 0; i < 16; i++) if (!ctx->pool[i].soa) { h = i; break; }
    if (h < 0) return fail(ctx, BLSGPU_ERR_ARG, "too many pools");
    if (int rc = ws_reserve(ctx, al(48 * n) + al(n) + 8192)) return rc;
    const uint8_t* din; if (int rc = stage_in(ctx, din, pks48, 48 * n)) return rc;
    u32x4* soa; uint8_t* code;
    if (cudaMalloc(&soa, 96 * n) != cudaSuccess || cudaMalloc(&code, n) != cudaSuccess) { cudaGetLastError(); return fail(ctx, BLSGPU_ERR_ALLOC, "pool allocation failed"); }
    LAUNCH(k_decode_g1, nblk(n), TPB, din, n, soa, code);
    if (status) { if (ctx->ptr_mode == BLSGPU_DEVICE) CU(cudaMemcpyAsync(status, code, n, cudaMemcpyDeviceToDevice, ctx->stream)); else CU(cudaMemcpyAsync(status, code, n, cudaMemcpyDeviceToHost, ctx->stream)); }
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->pool[h].soa = soa; ctx->pool[h].code = code; ctx->pool[h].n = n; *handle = h; return 0;
}
int blsgpu_pool_free(blsgpu_ctx* ctx, int handle) {
    if (!ctx || handle < 0 || handle >= 16 || !ctx->pool[handle].soa) return BLSGPU_ERR_ARG;
    dev_guard guard_; cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->pool[handle].soa); cudaFree(ctx->pool[handle].code); ctx->pool[handle].soa = nullptr; ctx->pool[handle].code = nullptr; ctx->pool[handle].n = 0; return 0;
}
int blsgpu_pool_fast_aggregate_verify(blsgpu_ctx* ctx, int handle, const uint32_t* idx, const uint64_t* bitmap, size_t k, const uint8_t* msg32, const uint8_t* sig96, size_t ncomm,
                                      uint8_t* status, uint8_t* agg_pk48_out) {
    ENTER(); if (handle < 0 || handle >= 16 || !ctx->pool[handle].soa || !idx || !msg32 || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    if (!ncomm) return 0;
    int rc; size_t nm = ncomm * k;
    if ((rc = ws_reserve(ctx, al(4 * nm + 16) + al(8 * ((nm + 63) / 64 + 1)) + al(96 * ncomm) * 2 + al(144 * ncomm) + al(48 * ncomm) + 4 * al(ncomm) + verify_ws_bytes(ncomm, 32 * ncomm)))) return rc;
    const uint32_t* didx; const uint8_t *dmsg, *dsig; const uint64_t* dbm;
    if ((rc = stage_in(ctx, didx, idx, nm))) return rc; if ((rc = stage_in(ctx, dbm, bitmap, (nm + 63) / 64))) return rc;
    if ((rc = stage_in(ctx, dmsg, msg32, 32 * ncomm))) return rc; if ((rc = stage_in(ctx, dsig, sig96, 96 * ncomm))) return rc;
    u32x4* agg_soa = ws_take<u32x4>(ctx, 6 * ncomm); uint8_t* agg_inf = ws_take<uint8_t>(ctx, ncomm); uint8_t* agg_st = ws_take<uint8_t>(ctx, ncomm); uint8_t* code_pk = ws_take<uint8_t>(ctx, ncomm);
    uint8_t* dstatus = stage_out(ctx, status, ncomm); uint8_t* dagg = stage_out(ctx, agg_pk48_out, 48 * ncomm);
    { int L = seg_lanes(k); u32x4* ojac = ws_take<u32x4>(ctx, 9 * ncomm);
      LAUNCH(k_segsum<fp>, nblk(ncomm, SEG_WARPS * (32 / L)), 32 * SEG_WARPS, (const u32x4*)ctx->pool[handle].soa, (const uint8_t*)ctx->pool[handle].code, ctx->pool[handle].n, (const uint32_t*)nullptr, k, dbm, ncomm,
             ojac, agg_st, (uint8_t)ST_BAD_PK, didx, L);
      LAUNCH(k_jac_to_aff<fp>, nblk(ncomm), TPB, (const u32x4*)ojac, ncomm, agg_soa, agg_inf); }
    if (dagg) LAUNCH(k_encode_g1, nblk(ncomm), TPB, (const u32x4*)agg_soa, (const uint8_t*)agg_inf, ncomm, dagg);
    LAUNCH(k_fav_status, nblk(ncomm), TPB, (const uint8_t*)agg_st, (const uint8_t*)agg_inf, (const uint8_t*)nullptr, ncomm, code_pk);
    if ((rc = verify_core(ctx, agg_soa, code_pk, dmsg, nullptr, dsig, ncomm, dstatus, nullptr, nullptr))) return rc;
    if ((rc = finish_out(ctx, status, dstatus, ncomm))) return rc; if ((rc = finish_out(ctx, agg_pk48_out, dagg, 48 * ncomm))) return rc;
    return finish_call(ctx);
}

}  // extern "C"

#include "r1cs.cuh"
#include "witness.cuh"
#include "multi.cuh"
