// Signature sets (include/blsgpu.h: blsgpu_verify_signature_sets, blsgpu_pool_verify_signature_sets): set s = the keys
// [key_off[s], key_off[s+1]) of a flat list (compressed bytes or resident-pool indices, an optional participation bitmap over the flat list),
// one message of any length, one signature.  Included from blsgpu.cu after the verify paths it reuses.
//
// Front of a pass: k_decode_g1 over the pass's keys (not for a pool), k_segsum over the sets (Jacobian sums + status), then either
//   per set:  k_jac_to_aff -> k_fav_status -> verify_core (the signature's subgroup test on the Miller loop's running point), or
//   RLC:      k_decode_g2<true> -> k_sets_rlc_prep -> hash_stage -> rlc_pieces (Miller loop with pair 0 off, per-piece trees, k_rlc_finish_seg);
// a piece whose equation fails is re-run per set.  The signatures of the RLC form are subgroup-checked in the decoder: no per-set Miller loop
// runs on them there, so the running point that the per-set form tests does not exist.

// a pass closes at the first piece boundary at which it holds this many keys or more (decoded: 96 B per key, with staging ~1.6 GB at 2^24)
#define SETS_PASS_KEYS ((size_t)1 << 24)

// RLC form, one thread per set: the status rule of k_fav_status on the sum (a bad or unselected-only set and an identity aggregate give
// code_pk = DEC_BAD_FLAGS), then for a live set pk_soa = [r_s] aggregate (affine), rsig = [r_s] sig, and code_sig = DEC_INF, which makes
// hash_stage set FL_SIG_INF: pair 0 of the set's Miller loop is switched off, its signature is in the per-piece sum instead.  The aggregate is
// made affine first and the ladder runs on mixed additions: one inversion more than a ladder on the Jacobian sum with full additions, and
// measured the faster of the two by a small margin (profiles/sets_r01.md).
__global__ void __launch_bounds__(TPB, BLS_MINB) k_sets_rlc_prep(const u32x4* agg_jac, const uint8_t* agg_st, const u32x4* sig_soa, uint8_t* code_sig, size_t n, size_t idx0,
                                                                  const uint8_t* seed16, u32x4* pk_soa, uint8_t* code_pk, u32x4* rsig_jac) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; if (i >= n) return;
    g1_jac a; segsum_traits<fp>::loadj(a, agg_jac, n, i);
    bool pk_ok = agg_st[i] == ST_OK && !jac_is_identity(a);
    uint8_t cs = code_sig[i];
    g2_jac rs; jac_set_identity(rs);
    code_pk[i] = pk_ok ? (uint8_t)DEC_OK : (uint8_t)DEC_BAD_FLAGS;
    if (pk_ok && cs <= DEC_INF) {
        g1_aff base; jac_to_aff(base, a);
        rlc_scale_item(pk_soa, sig_soa, n, i, base, cs == DEC_INF, seed16, idx0 + i, rs);
        code_sig[i] = DEC_INF;
    }
    segsum_traits<fp2>::storej(rsig_jac, n, i, rs);
}

struct sets_in {
    const uint8_t* pks48; int pool; const uint32_t* idx;        // pool < 0: compressed keys pks48; else indices idx into ctx->pool[pool]
    const uint32_t* key_off; const uint64_t* bitmap; const uint8_t* msg; const uint32_t* msg_off; const uint8_t* sig96;
};

static size_t sets_ws_bytes(size_t m, size_t nk, size_t mb, bool pool, bool rlc) {
    size_t P = (m + RLC_PIECE - 1) / RLC_PIECE, T0 = (RLC_PIECE + 7) / 8;
    return (pool ? al(4 * nk + 16) : al(48 * nk + 16) + al(96 * nk + 16) + al(nk + 1)) + al(8 * ((nk + 63) / 64 + 2)) + al(4 * (m + 1)) + al(144 * m) + al(96 * m) + 4 * al(m) +
           verify_ws_bytes(m, mb) + (rlc ? al(288 * m) + 2 * al(288 * P * T0) + 2 * al(576 * P * T0) + al(P) : 0) + 65536;
}

// One pass: sets [s0, s0 + m), keys [k0, k1) of the flat list (offsets, bitmap bits and pool indices stay absolute), message bytes [mb0, mb0 + mb)
// (host mode).  dseed == NULL: per-set outcome into status.  Otherwise the RLC form: status 0 / 2 / 3 and one ok flag per piece into piece_ok (host).
static int sets_pass(blsgpu_ctx* ctx, const sets_in& in, size_t s0, size_t m, size_t k0, size_t k1, size_t mb0, size_t mb, const uint8_t* dseed,
                     uint8_t* status, uint8_t* piece_ok) {
    int rc = 0; bool host = ctx->ptr_mode == BLSGPU_HOST, pool = in.pool >= 0, rlc = dseed != nullptr; size_t nk = k1 - k0;
    if ((rc = ws_reserve(ctx, sets_ws_bytes(m, nk, host ? mb : 0, pool, rlc)))) return rc;
    const uint32_t* dkoff; if ((rc = stage_in(ctx, dkoff, in.key_off + s0, m + 1))) return rc;
    const uint64_t* dbm = nullptr;
    if (in.bitmap) {
        if (host) { size_t w0 = k0 / 64; if ((rc = stage_in(ctx, dbm, in.bitmap + w0, (k1 + 63) / 64 - w0))) return rc; dbm -= w0; }
        else dbm = in.bitmap;
    }
    const u32x4* pts; const uint8_t* code; size_t npts, pt_base = 0; const uint32_t* didx = nullptr;
    if (pool) {
        pts = ctx->pool[in.pool].soa; code = ctx->pool[in.pool].code; npts = ctx->pool[in.pool].n;
        if (host) { if ((rc = stage_in(ctx, didx, in.idx + k0, nk))) return rc; didx -= k0; } else didx = in.idx;
    } else {
        const uint8_t* dpks; if ((rc = stage_in(ctx, dpks, in.pks48 + 48 * k0, 48 * nk))) return rc;
        u32x4* soa = ws_take<u32x4>(ctx, 6 * nk + 1); uint8_t* c = ws_take<uint8_t>(ctx, nk + 1);
        if (nk) LAUNCH(k_decode_g1, nblk(nk), TPB, dpks, nk, soa, c);
        pts = soa; code = c; npts = nk; pt_base = k0;
    }
    const uint8_t *dsig, *dmsg; const uint32_t* doff;
    if ((rc = stage_in(ctx, dsig, in.sig96 + 96 * s0, 96 * m))) return rc;
    if (host) { if ((rc = stage_in(ctx, dmsg, in.msg + mb0, mb ? mb : 1))) return rc; dmsg -= in.msg_off ? mb0 : 0; }      // offsets stay absolute
    else dmsg = in.msg_off ? in.msg : in.msg + mb0;
    if ((rc = stage_in(ctx, doff, in.msg_off ? in.msg_off + s0 : nullptr, m + 1))) return rc;
    uint8_t* dstatus = stage_out(ctx, status + s0, m);
    u32x4* ojac = ws_take<u32x4>(ctx, 9 * m); uint8_t* agg_st = ws_take<uint8_t>(ctx, m); uint8_t* code_pk = ws_take<uint8_t>(ctx, m);
    int L = seg_lanes(nk / m);
    LAUNCH(k_segsum<fp>, nblk(m, SEG_WARPS * (32 / L)), 32 * SEG_WARPS, pts, code, npts, dkoff, (size_t)0, dbm, m, ojac, agg_st, (uint8_t)ST_BAD_PK, didx, L, pt_base);
    if (!rlc) {
        u32x4* agg_soa = ws_take<u32x4>(ctx, 6 * m); uint8_t* agg_inf = ws_take<uint8_t>(ctx, m);
        LAUNCH(k_jac_to_aff<fp>, nblk(m), TPB, (const u32x4*)ojac, m, agg_soa, agg_inf);
        LAUNCH(k_fav_status, nblk(m), TPB, (const uint8_t*)agg_st, (const uint8_t*)agg_inf, (const uint8_t*)nullptr, m, code_pk);
        if ((rc = verify_core(ctx, agg_soa, code_pk, dmsg, doff, dsig, m, dstatus, nullptr, nullptr, false, true))) return rc;
        if ((rc = finish_out(ctx, status + s0, dstatus, m))) return rc;
        if (host) CU(cudaStreamSynchronize(ctx->stream));
        return 0;
    }
    size_t P = (m + RLC_PIECE - 1) / RLC_PIECE, T0 = (RLC_PIECE + 7) / 8;
    u32x4* pk_soa = ws_take<u32x4>(ctx, 6 * m); u32x4* sig_soa = ws_take<u32x4>(ctx, 12 * m); u32x4* hm_soa = ws_take<u32x4>(ctx, 12 * m); u32x4* f_soa = ws_take<u32x4>(ctx, 36 * m);
    uint8_t* code_sig = ws_take<uint8_t>(ctx, m); uint8_t* flags = ws_take<uint8_t>(ctx, m);
    u32x4* rs = ws_take<u32x4>(ctx, 18 * m); u32x4* ja = ws_take<u32x4>(ctx, 18 * P * T0); u32x4* jb = ws_take<u32x4>(ctx, 18 * P * T0);
    u32x4* ta = ws_take<u32x4>(ctx, 36 * P * T0); u32x4* tb = ws_take<u32x4>(ctx, 36 * P * T0); uint8_t* dok = ws_take<uint8_t>(ctx, P);
    LAUNCH(k_decode_g2<true>, nblk(m), TPB, dsig, m, sig_soa, code_sig);
    LAUNCH(k_sets_rlc_prep, nblk(m), TPB, (const u32x4*)ojac, (const uint8_t*)agg_st, (const u32x4*)sig_soa, code_sig, m, s0, dseed, pk_soa, code_pk, rs);
    if ((rc = hash_stage(ctx, dmsg, doff, m, code_pk, code_sig, hm_soa, f_soa, flags, dstatus))) return rc;
    if ((rc = rlc_pieces(ctx, rs, pk_soa, hm_soa, sig_soa, flags, dstatus, m, f_soa, ja, jb, ta, tb, dok))) return rc;
    if ((rc = finish_out(ctx, status + s0, dstatus, m))) return rc;
    CU(cudaMemcpyAsync(piece_ok + s0 / RLC_PIECE, dok, P, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int verify_sets(blsgpu_ctx* ctx, const sets_in& in, size_t nsets, const uint8_t* seed16, uint8_t* status, uint64_t* ok_bitmap, uint64_t* fallback_sets) {
    if (fallback_sets) *fallback_sets = 0;
    if (!nsets) return 0;
    int rc = 0; bool host = ctx->ptr_mode == BLSGPU_HOST;
    // passes are planned on the host: read key_off there once in device mode
    std::vector<uint32_t> koff_copy;
    const uint32_t* koff = in.key_off;
    if (!host) {
        koff_copy.resize(nsets + 1);
        CU(cudaMemcpyAsync(koff_copy.data(), in.key_off, 4 * (nsets + 1), cudaMemcpyDeviceToHost, ctx->stream)); CU(cudaStreamSynchronize(ctx->stream));
        koff = koff_copy.data();
    }
    for (size_t s = 0; s < nsets; s++) if (koff[s + 1] < koff[s]) return fail(ctx, BLSGPU_ERR_ARG, "key_off decreases at set %zu", s);
    if (koff[nsets] && !in.pks48 && in.pool < 0) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    const size_t L = RLC_PIECE, chunk = ctx->chunk >= L ? ctx->chunk / L * L : L;
    // sets [a, b) (a on a piece boundary) in passes of whole pieces: at most `chunk` sets, closed once SETS_PASS_KEYS keys are reached
    auto run = [&](size_t a, size_t b, const uint8_t* dseed, uint8_t* piece_ok) -> int {
        for (size_t s0 = a; s0 < b; ) {
            size_t s1 = s0;
            do { s1 = s1 + L < b ? s1 + L : b; } while (s1 < b && s1 - s0 + L <= chunk && koff[s1] - koff[s0] < SETS_PASS_KEYS);
            size_t mb0 = in.msg_off ? (host ? in.msg_off[s0] : 0) : 32 * s0, mb = in.msg_off ? (host ? in.msg_off[s1] - in.msg_off[s0] : 0) : 32 * (s1 - s0);
            if (int r = sets_pass(ctx, in, s0, s1 - s0, koff[s0], koff[s1], mb0, mb, dseed, status, piece_ok)) return r;
            s0 = s1;
        }
        return 0;
    };
    uint64_t rerun = 0;
    if (!seed16) { if ((rc = run(0, nsets, nullptr, nullptr))) return rc; }
    else {
        if (!ctx->rlc_acc) CU(cudaMalloc(&ctx->rlc_acc, 2048));
        uint8_t* dseed = ctx->rlc_acc + 1040;
        CU(cudaMemcpyAsync(dseed, seed16, 16, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
        std::vector<uint8_t> piece_ok((nsets + L - 1) / L, 1);
        if ((rc = run(0, nsets, dseed, piece_ok.data()))) return rc;
        // failing pieces: the per-set form on exactly those sets (adjacent failing pieces in one run)
        for (size_t p = 0; p < piece_ok.size(); ) {
            if (piece_ok[p]) { p++; continue; }
            size_t q = p; while (q < piece_ok.size() && !piece_ok[q]) q++;
            size_t lo = p * L, hi = q * L < nsets ? q * L : nsets;
            if ((rc = run(lo, hi, nullptr, nullptr))) return rc;
            rerun += hi - lo; p = q;
        }
    }
    if (fallback_sets) *fallback_sets = rerun;
    if (ok_bitmap) {
        if (host) { size_t words = (nsets + 63) / 64; for (size_t w = 0; w < words; w++) ok_bitmap[w] = 0; for (size_t i = 0; i < nsets; i++) if (status[i] == ST_OK) ok_bitmap[i >> 6] |= 1ull << (i & 63); }
        else { CU(cudaMemsetAsync(ok_bitmap, 0, 8 * ((nsets + 63) / 64), ctx->stream)); LAUNCH(k_status_bitmap, nblk(((nsets + 31) / 32) * 32, 256), 256, (const uint8_t*)status, nsets, (uint32_t*)ok_bitmap); }
    }
    return finish_call(ctx);
}

extern "C" {
int blsgpu_verify_signature_sets(blsgpu_ctx* ctx, const uint8_t* pks48, const uint32_t* key_off, const uint64_t* bitmap, const uint8_t* msg, const uint32_t* msg_off,
                                 const uint8_t* sig96, size_t nsets, const uint8_t* seed16, uint8_t* status, uint64_t* ok_bitmap, uint64_t* fallback_sets) {
    ENTER(); if (!key_off || !msg || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    sets_in in = {pks48, -1, nullptr, key_off, bitmap, msg, msg_off, sig96};
    return verify_sets(ctx, in, nsets, seed16, status, ok_bitmap, fallback_sets);
}
int blsgpu_pool_verify_signature_sets(blsgpu_ctx* ctx, int handle, const uint32_t* idx, const uint32_t* key_off, const uint64_t* bitmap, const uint8_t* msg,
                                      const uint32_t* msg_off, const uint8_t* sig96, size_t nsets, const uint8_t* seed16, uint8_t* status, uint64_t* ok_bitmap,
                                      uint64_t* fallback_sets) {
    ENTER(); if (handle < 0 || handle >= 16 || !ctx->pool[handle].soa || !idx || !key_off || !msg || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    sets_in in = {nullptr, handle, idx, key_off, bitmap, msg, msg_off, sig96};
    return verify_sets(ctx, in, nsets, seed16, status, ok_bitmap, fallback_sets);
}
}  // extern "C"
