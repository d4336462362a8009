// Signature sets (include/blsgpu.h: blsgpu_verify_signature_sets, blsgpu_pool_verify_signature_sets): set s = the keys
// [key_off[s], key_off[s+1]) of a flat list (compressed bytes or resident-pool indices, an optional participation bitmap over the flat list),
// one message of any length, one signature.  Included from blsgpu.cu after the verify paths it reuses.
//
// Front of a pass: k_decode_g1 over the pass's keys (not for a pool), stage_items for the messages and signatures, k_segsum over the sets
// (Jacobian sums + status), then either
//   per set:  k_jac_to_aff -> k_fav_status -> verify_core (the signature's subgroup test on the Miller loop's running point), or
//   RLC:      rlc_carve -> k_decode_g2<true> -> k_sets_rlc_prep -> hash_stage -> rlc_pieces (Miller loop with pair 0 off, per-piece trees) -> k_rlc_finish_seg;
// rerun_failing_pieces re-runs a piece whose equation fails per set.  The signatures of the RLC form are subgroup-checked in the decoder: no per-set Miller loop
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
    const uint32_t* key_off; const uint64_t* bitmap;
    batch_in sets;                                              // message and signature of each set (no pk48)
};

static size_t sets_ws_bytes(const blsgpu_ctx* ctx, size_t m, size_t nk, size_t mb, bool pool, bool rlc) {
    return (pool ? al(4 * nk + 16) : al(48 * nk + 16) + al(96 * nk + 16) + al(nk + 1)) + al(8 * ((nk + 63) / 64 + 2)) + al(4 * (m + 1)) + al(144 * m) + al(96 * m) + 4 * al(m) +
           (rlc ? stage_ws_bytes(m, mb) + rlc_ws_bytes(ctx, m, RLC_PIECE) : verify_ws_bytes(m, mb)) + 65536;
}

// One pass: sets [s0, s0 + m), keys [k0, k1) of the flat list (offsets, bitmap bits and pool indices stay absolute).
// dseed == NULL: per-set outcome into status.  Otherwise the RLC form: status 0 / 2 / 3 and one ok flag per piece into piece_ok (host).
static int sets_pass(blsgpu_ctx* ctx, const sets_in& in, size_t s0, size_t m, size_t k0, size_t k1, const uint8_t* dseed, uint8_t* status, uint8_t* piece_ok) {
    int rc = 0; bool host = ctx->ptr_mode == BLSGPU_HOST, pool = in.pool >= 0, rlc = dseed != nullptr; size_t nk = k1 - k0;
    if ((rc = ws_reserve(ctx, sets_ws_bytes(ctx, m, nk, pass_msg_bytes(ctx, in.sets, s0, s0 + m), pool, rlc)))) return rc;
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
    batch_dev d; if ((rc = stage_items(ctx, in.sets, s0, s0 + m, d))) return rc;
    uint8_t* dstatus = stage_out(ctx, status + s0, m);
    u32x4* ojac = ws_take<u32x4>(ctx, 9 * m); uint8_t* agg_st = ws_take<uint8_t>(ctx, m);
    int L = seg_lanes(nk / m);
    LAUNCH(k_segsum<fp>, nblk(m, SEG_WARPS * (32 / L)), 32 * SEG_WARPS, pts, code, npts, dkoff, (size_t)0, dbm, m, ojac, agg_st, (uint8_t)ST_BAD_PK, didx, L, pt_base);
    if (!rlc) {
        u32x4* agg_soa = ws_take<u32x4>(ctx, 6 * m); uint8_t* agg_inf = ws_take<uint8_t>(ctx, m); uint8_t* code_pk = ws_take<uint8_t>(ctx, m);
        LAUNCH(k_jac_to_aff<fp>, nblk(m), TPB, (const u32x4*)ojac, m, agg_soa, agg_inf);
        LAUNCH(k_fav_status, nblk(m), TPB, (const uint8_t*)agg_st, (const uint8_t*)agg_inf, (const uint8_t*)nullptr, m, code_pk);
        if ((rc = verify_core(ctx, agg_soa, code_pk, d.msg, d.msg_off, d.sig96, m, dstatus, nullptr, nullptr, false, true))) return rc;
        if ((rc = finish_out(ctx, status + s0, dstatus, m))) return rc;
        if (host) CU(cudaStreamSynchronize(ctx->stream));
        return 0;
    }
    size_t P = (m + RLC_PIECE - 1) / RLC_PIECE;
    rlc_bufs b = rlc_carve(ctx, m, RLC_PIECE); const u32x4 *f, *s;
    LAUNCH(k_decode_g2<true>, nblk(m), TPB, d.sig96, m, b.sig_soa, b.code_sig);
    LAUNCH(k_sets_rlc_prep, nblk(m), TPB, (const u32x4*)ojac, (const uint8_t*)agg_st, (const u32x4*)b.sig_soa, b.code_sig, m, s0, dseed, b.pk_soa, b.code_pk, b.rs);
    if ((rc = hash_stage(ctx, d.msg, d.msg_off, m, b.code_pk, b.code_sig, b.hm_soa, b.f_soa, b.flags, dstatus))) return rc;
    if ((rc = rlc_pieces(ctx, b, dstatus, m, RLC_PIECE, f, s))) return rc;
    LAUNCH(k_rlc_finish_seg, (unsigned)P, 32, f, s, P, (const uint32_t*)nullptr, b.ok);
    if ((rc = finish_out(ctx, status + s0, dstatus, m))) return rc;
    CU(cudaMemcpyAsync(piece_ok + s0 / RLC_PIECE, b.ok, P, cudaMemcpyDeviceToHost, ctx->stream));
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
    const size_t L = RLC_PIECE, chunk = piece_chunk(ctx);
    // sets [a, b) (a on a piece boundary) in passes of whole pieces: at most `chunk` sets, closed once SETS_PASS_KEYS keys are reached
    auto run = [&](size_t a, size_t b, const uint8_t* dseed, uint8_t* piece_ok) -> int {
        for (size_t s0 = a; s0 < b; ) {
            size_t s1 = s0;
            do { s1 = s1 + L < b ? s1 + L : b; } while (s1 < b && s1 - s0 + L <= chunk && koff[s1] - koff[s0] < SETS_PASS_KEYS);
            if (int r = sets_pass(ctx, in, s0, s1 - s0, koff[s0], koff[s1], dseed, status, piece_ok)) return r;
            s0 = s1;
        }
        return 0;
    };
    uint64_t rerun = 0;
    if (!seed16) { if ((rc = run(0, nsets, nullptr, nullptr))) return rc; }
    else {
        uint8_t* dseed; if ((rc = rlc_seed(ctx, seed16, dseed))) return rc;
        std::vector<uint8_t> piece_ok((nsets + L - 1) / L, 1);
        if ((rc = run(0, nsets, dseed, piece_ok.data()))) return rc;
        if ((rc = rerun_failing_pieces(piece_ok, nsets, L, rerun, [&](size_t lo, size_t hi) { return run(lo, hi, nullptr, nullptr); }))) return rc;
    }
    if (fallback_sets) *fallback_sets = rerun;
    if ((rc = bitmap_from_status(ctx, status, nsets, ok_bitmap))) return rc;
    return finish_call(ctx);
}

extern "C" {
int blsgpu_verify_signature_sets(blsgpu_ctx* ctx, const uint8_t* pks48, const uint32_t* key_off, const uint64_t* bitmap, const uint8_t* msg, const uint32_t* msg_off,
                                 const uint8_t* sig96, size_t nsets, const uint8_t* seed16, uint8_t* status, uint64_t* ok_bitmap, uint64_t* fallback_sets) {
    ENTER(); if (!key_off || !msg || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "null pointer");
    sets_in in = {pks48, -1, nullptr, key_off, bitmap, {nullptr, msg, msg_off, sig96}};
    return verify_sets(ctx, in, nsets, seed16, status, ok_bitmap, fallback_sets);
}
int blsgpu_pool_verify_signature_sets(blsgpu_ctx* ctx, int handle, const uint32_t* idx, const uint32_t* key_off, const uint64_t* bitmap, const uint8_t* msg,
                                      const uint32_t* msg_off, const uint8_t* sig96, size_t nsets, const uint8_t* seed16, uint8_t* status, uint64_t* ok_bitmap,
                                      uint64_t* fallback_sets) {
    ENTER(); if (handle < 0 || handle >= 16 || !ctx->pool[handle].soa || !idx || !key_off || !msg || !sig96 || !status) return fail(ctx, BLSGPU_ERR_ARG, "bad argument");
    sets_in in = {nullptr, handle, idx, key_off, bitmap, {nullptr, msg, msg_off, sig96}};
    return verify_sets(ctx, in, nsets, seed16, status, ok_bitmap, fallback_sets);
}
}  // extern "C"
