"""Signature sets (blsgpu_verify_signature_sets / blsgpu_pool_verify_signature_sets): set s = keys [key_off[s], key_off[s+1]) of a flat list,
one message of any length, one signature; per-set pairing checks, or per-piece random linear combinations with the exact outcome.

The per-set reference is ora_verify_sets below: a plain loop over the CPU oracle's own calls -- aggregate the selected keys (each deserialised
with the subgroup check; an empty selection is None), then verify the aggregate against the set's message and signature (an identity
aggregate is InvalidPublicKey, src/bls.rs:434)."""
import numpy as np
import pytest
from conftest import hx

R_ORDER = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001

@pytest.fixture(scope="module")
def C():
    from oracle import cwrap
    return cwrap

def bits_to_words(sel):
    sel = np.asarray(sel, bool); w = np.zeros(max((sel.size + 63) // 64, 1), np.uint64)
    for j in np.nonzero(sel)[0]: w[j // 64] |= np.uint64(1) << np.uint64(j % 64)
    return w[:(sel.size + 63) // 64]

def ora_verify_sets(C, pks48, key_off, msgs, sig96, bitmap=None, threads=None):
    """status per set: 0 / 1, 2 = a selected key fails / nothing selected / identity aggregate, 3 = the signature fails"""
    threads = threads or C.hw_threads()
    pk = np.frombuffer(bytes(pks48), np.uint8).reshape(-1, 48); ko = np.asarray(key_off, np.int64); n = ko.size - 1
    sel = np.ones(pk.shape[0], bool)
    if bitmap is not None: sel = ((np.asarray(bitmap, np.uint64)[np.arange(pk.shape[0]) // 64] >> (np.arange(pk.shape[0]) % 64).astype(np.uint64)) & np.uint64(1)).astype(bool)
    cs = np.concatenate([[0], np.cumsum(sel)]).astype(np.uint32)
    agg, ast = C.g1_aggregate(pk[sel].reshape(-1), cs[ko], threads=threads)
    st = C.verify(agg, list(msgs), sig96, threads=threads)
    st[ast != 0] = 2
    return st

def fixture_sets(eth):
    """the 11 fast_aggregate_verify fixtures, one set each, then every verify fixture as a one-key set -> (pks, key_off, msgs, sigs, verdicts)"""
    pks, ko, msgs, sigs, want = [], [0], [], [], []
    for c in eth["fast_aggregate_verify"]:
        i = c["input"]; pks += [hx(p) for p in i["pubkeys"]]; ko.append(len(pks)); msgs.append(hx(i["message"])); sigs.append(hx(i["signature"])); want.append(c["output"])
    for c in eth["verify"]:
        i = c["input"]; pk, sg = hx(i["pubkey"]), hx(i["signature"])
        if len(pk) != 48 or len(sg) != 96: continue
        pks.append(pk); ko.append(len(pks)); msgs.append(hx(i["message"])); sigs.append(sg); want.append(c["output"])
    return b"".join(pks), np.array(ko, np.uint32), msgs, b"".join(sigs), np.array(want)

# ------------------------------------------------------------------------------------------ CPU: the per-set reference
def test_ora_verify_sets_fixtures(C, eth):
    pks, ko, msgs, sigs, want = fixture_sets(eth)
    assert len(want) >= 11 + 20
    st = ora_verify_sets(C, pks, ko, msgs, sigs)
    assert np.array_equal(st == 0, want)

def test_ora_verify_sets_equals_fast_aggregate_verify(C):
    """uniform sets (k keys, 32-byte messages): status for status what the oracle's fast_aggregate_verify reports, with and without a bitmap"""
    rng = np.random.default_rng(41); nc, k = 24, 5
    sk = [int(x) for x in rng.integers(1, 1 << 62, size=nc * k)]
    pk = C.sk_to_pk(b"".join(s.to_bytes(32, "little") for s in sk)).reshape(nc * k, 48).copy()
    msg = rng.integers(0, 256, size=(nc, 32), dtype=np.uint8)
    agg_sk = b"".join((sum(sk[c * k:(c + 1) * k]) % R_ORDER).to_bytes(32, "little") for c in range(nc))
    sig, _ = C.sign(agg_sk, [m.tobytes() for m in msg]); sig = sig.reshape(nc, 96).copy()
    pk[k * 1 + 2, 7] ^= 0x55; pk[k * 2 + 1] = 0; pk[k * 2 + 1, 0] = 0xc0; sig[3, 90:] = 0xff; msg[4, 0] ^= 1; sig[5] = sig[6]
    pk[k * 7 + 1] = pk[k * 7]; pk[k * 7 + 1, 0] ^= 0x20                                                       # K, -K in one committee
    ko = np.arange(nc + 1, dtype=np.uint32) * k; msgs = [m.tobytes() for m in msg]
    for bm in (None, bits_to_words(rng.random(nc * k) < 0.6)):
        want = C.fast_aggregate_verify(pk.reshape(-1), k, msg.reshape(-1), sig.reshape(-1), bitmap=bm)
        st = ora_verify_sets(C, pk.reshape(-1), ko, msgs, sig.reshape(-1), bitmap=bm)
        assert np.array_equal(st, want)
        assert len(set(st.tolist())) >= 3

# ------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctx():
    from bls_verify_gadget_b200 import Context
    c = Context(0); yield c; c.close()

SEED = bytes(range(16))

def both_modes(ctx, *args, **kw):
    """per-set and RLC results of one call; RLC must equal per-set (statuses and bitmap)"""
    st, bm, rerun = ctx.verify_signature_sets(*args, **kw)
    assert rerun == 0
    st2, bm2, _ = ctx.verify_signature_sets(*args, seed16=SEED, **kw)
    assert np.array_equal(st2, st) and np.array_equal(bm2, bm)
    return st

def make_sets(ctx, sizes, msg_lens, rng, pool=4096):
    """valid sets over a key pool: keys (copies in the flat list), sk of every flat member, messages, signature = [sum of sks] H(m)"""
    from bls_verify_gadget_b200 import synth
    sk_b = synth.fast_secret_keys(pool, seed=int(rng.integers(1 << 30))); pool_pk, st = ctx.sk_to_pk(sk_b); assert not st.any()
    pool_pk = pool_pk.reshape(pool, 48); sk = [int.from_bytes(sk_b[32 * i:32 * i + 32].tobytes(), "little") for i in range(pool)]
    idx = rng.integers(0, pool, size=int(sum(sizes))).astype(np.uint32)
    ko = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint32)
    msgs = [rng.bytes(int(l)) for l in msg_lens]
    return pool_pk, sk, idx, ko, msgs

def sign_sets(ctx, sk_sums, msgs):
    sig, st = ctx.sign(b"".join((s % R_ORDER).to_bytes(32, "little") for s in sk_sums), msgs)
    return sig.reshape(len(msgs), 96).copy(), st

@pytest.mark.gpu
def test_fixture_sets_both_entry_points_and_modes(ctx, eth):
    pks, ko, msgs, sigs, want = fixture_sets(eth)
    st = both_modes(ctx, pks, ko, msgs, sigs)
    assert np.array_equal(st == 0, want)
    pk = np.frombuffer(pks, np.uint8).reshape(-1, 48)
    h, pst = ctx.pool_create(pk.reshape(-1))
    try:
        for seed in (None, SEED):
            s2, _, _ = ctx.pool_verify_signature_sets(h, np.arange(pk.shape[0]), ko, msgs, sigs, seed16=seed)
            assert np.array_equal(s2, st)
    finally: ctx.pool_free(h)

@pytest.mark.gpu
def test_ragged_sets_differential_against_the_oracle(ctx, C, pyv):
    """~3,000 sets of 0..1000 keys with messages of 0..250 bytes, a participation bitmap, and every corruption kind repeated"""
    rng = np.random.default_rng(2026); n = 3000
    sizes = rng.choice([0, 1, 2, 3, 17, 64, 128, 512, 1000], size=n); lens = rng.integers(0, 251, size=n)
    kinds = ["bad_key", "subgroup_key", "identity_member", "cancel", "empty", "unselected", "bad_sig", "sig_subgroup", "identity_sig", "wrong_msg", "other_sig"]
    plan = {}
    for j, s in enumerate(range(5, n, 13)):
        plan[s] = kinds[j % len(kinds)]; sizes[s] = 0 if plan[s] == "empty" else max(sizes[s], 2)
    pool_pk, sk, idx, ko, msgs = make_sets(ctx, sizes, lens, rng)
    flat = pool_pk[idx].copy(); fsk = [sk[i] for i in idx]
    sel = rng.random(flat.shape[0]) < 0.85
    ident48 = np.zeros(48, np.uint8); ident48[0] = 0xc0; ident96 = np.zeros(96, np.uint8); ident96[0] = 0xc0
    g1_bad = np.frombuffer(hx(pyv["g1_not_in_subgroup"]), np.uint8); g2_bad = np.frombuffer(hx(pyv["g2_not_in_subgroup"]), np.uint8)
    for s, kind in plan.items():
        lo, hi = int(ko[s]), int(ko[s + 1])
        if kind == "empty" or hi == lo: continue
        sel[lo] = True
        if kind == "bad_key": flat[lo, 5] ^= 0x55; flat[lo, 0] = 0x80 | (flat[lo, 0] & 0x1f); flat[lo, 47] ^= 0x0f
        elif kind == "subgroup_key": flat[lo] = g1_bad
        elif kind == "identity_member": flat[lo] = ident48; fsk[lo] = 0
        elif kind == "cancel": sel[lo:hi] = False; sel[lo] = True
        elif kind == "unselected": sel[lo:hi] = False
    for s, kind in plan.items():                                                      # P and -P as the only selected members
        lo, hi = int(ko[s]), int(ko[s + 1])
        if kind == "cancel" and hi - lo >= 2: flat[lo + 1] = flat[lo]; flat[lo + 1, 0] ^= 0x20; fsk[lo + 1] = R_ORDER - fsk[lo]; sel[lo + 1] = True
    sums = [sum(fsk[i] for i in range(int(ko[s]), int(ko[s + 1])) if sel[i]) for s in range(n)]
    sig, _ = sign_sets(ctx, [x if x % R_ORDER else 1 for x in sums], msgs)
    msgs = list(msgs)
    for s, kind in plan.items():
        if kind == "bad_sig": sig[s, 92:] = 0xff
        elif kind == "sig_subgroup": sig[s] = g2_bad
        elif kind == "identity_sig": sig[s] = ident96
        elif kind == "wrong_msg": msgs[s] = msgs[s] + b"!"
        elif kind == "other_sig": sig[s] = sig[(s + 1) % n]
    bm = bits_to_words(sel)
    want = ora_verify_sets(C, flat.reshape(-1), ko, msgs, sig.reshape(-1), bitmap=bm)
    st = both_modes(ctx, flat.reshape(-1), ko, msgs, sig.reshape(-1), bitmap=bm)
    assert np.array_equal(st, want)
    assert {0, 1, 2, 3} <= set(st.tolist()) and (st == 0).sum() > n // 2
    for s, kind in plan.items():                                                      # each corruption reaches the outcome it is about
        if kind in ("bad_key", "subgroup_key", "empty", "unselected", "cancel"): assert st[s] == 2, (s, kind)
        if kind in ("bad_sig", "sig_subgroup") and st[s] != 2: assert st[s] == 3, (s, kind)
        if kind in ("wrong_msg", "other_sig") and st[s] not in (2, 3): assert st[s] == 1, (s, kind)

@pytest.mark.gpu
def test_uniform_sets_equal_fast_aggregate_verify(ctx):
    """uniform sets give byte-identical status to blsgpu_fast_aggregate_verify_batch, pool sets to blsgpu_pool_fast_aggregate_verify"""
    from bls_verify_gadget_b200 import synth
    nc, k = 300, 64
    pks, msg, sig, pool_pk, idx = synth.committees(ctx, nc, k=k, pool=2048)
    pks = pks.reshape(nc * k, 48).copy(); msg = msg.reshape(nc, 32).copy(); sig = sig.reshape(nc, 96).copy()
    msg[3, 0] ^= 1; sig[7, 95] ^= 1; pks[11 * k + 3, 9] ^= 0x33; sig[13] = sig[14]; sig[20] = 0; sig[20, 0] = 0xc0
    ko = np.arange(nc + 1, dtype=np.uint32) * k
    h, _ = ctx.pool_create(pool_pk.reshape(-1))
    try:
        for bm in (None, bits_to_words(np.random.default_rng(8).random(nc * k) < 0.66)):
            want = ctx.fast_aggregate_verify(pks.reshape(-1), k, msg.reshape(-1), sig.reshape(-1), bitmap=bm)
            st = both_modes(ctx, pks.reshape(-1), ko, msg.reshape(-1), sig.reshape(-1), bitmap=bm, fixed32=True)
            assert np.array_equal(st, want)
            pwant = ctx.pool_fast_aggregate_verify(h, idx.reshape(-1), k, msg.reshape(-1), sig.reshape(-1), bitmap=bm)
            for seed in (None, SEED):
                pst, _, _ = ctx.pool_verify_signature_sets(h, idx.reshape(-1), ko, msg.reshape(-1), sig.reshape(-1), seed16=seed, bitmap=bm, fixed32=True)
                assert np.array_equal(pst, pwant)
            if bm is None: assert (st == 0).sum() >= nc - 8 and st[3] == 1 and st[11] == 2
    finally: ctx.pool_free(h)

@pytest.mark.gpu
def test_rlc_fallback_is_exact(ctx, pyv):
    """3 x 4,096 + 777 sets of 1..8 keys: only pieces whose equation fails are re-run; decode failures need no re-run; the same across
    several passes and with the one-launch stage kernels"""
    rng = np.random.default_rng(4096); n = 3 * 4096 + 777
    sizes = rng.integers(1, 9, size=n)
    pool_pk, sk, idx, ko, _ = make_sets(ctx, sizes, [0] * n, rng)
    msg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    flat = pool_pk[idx].copy()
    sig, st = sign_sets(ctx, [sum(sk[i] for i in idx[int(ko[s]):int(ko[s + 1])]) for s in range(n)], [m.tobytes() for m in msg]); assert not st.any()
    run = lambda f, m, s, seed: ctx.verify_signature_sets(f.reshape(-1), ko, m.reshape(-1), s.reshape(-1), seed16=seed, fixed32=True)
    st, bm, rerun = run(flat, msg, sig, SEED)
    assert not st.any() and rerun == 0 and int(np.unpackbits(bm.view(np.uint8)).sum()) == n
    f2, s2 = flat.copy(), sig.copy()
    f2[int(ko[100]), 3] ^= 0x41; f2[int(ko[12300])] = np.frombuffer(hx(pyv["g1_not_in_subgroup"]), np.uint8); s2[5000, 92:] = 0xff
    st, bm, rerun = run(f2, msg, s2, SEED)
    assert rerun == 0 and sorted(np.nonzero(st)[0].tolist()) == [100, 5000, 12300] and st[5000] == 3 and st[12300] == 2
    m3, s3 = msg.copy(), s2.copy()
    m3[4096 + 10, 0] ^= 1; s3[3 * 4096 + 500] = s3[3 * 4096 + 501]
    want, wbm, r0 = run(f2, m3, s3, None)
    assert r0 == 0 and sorted(np.nonzero(want)[0].tolist()) == [100, 4106, 5000, 12300, 12788]
    st, bm, rerun = run(f2, m3, s3, SEED)
    assert np.array_equal(st, want) and np.array_equal(bm, wbm) and rerun == 4096 + 777
    ctx.set_chunk(4096)
    try: st2, bm2, rerun2 = run(f2, m3, s3, b"another seed 16b")
    finally: ctx.set_chunk(1 << 20)
    assert np.array_equal(st2, want) and np.array_equal(bm2, wbm) and rerun2 == rerun
    ctx.set_split(0)
    try: st3, bm3, rerun3 = run(f2, m3, s3, SEED); st4, _, _ = run(f2, m3, s3, None)
    finally: ctx.set_split(1)
    assert np.array_equal(st3, want) and np.array_equal(bm3, wbm) and rerun3 == rerun and np.array_equal(st4, want)

@pytest.mark.gpu
def test_rlc_weights_are_random(ctx):
    """two sets over one message with their signatures swapped: with equal weights the batch equation would hold; both must report 1"""
    rng = np.random.default_rng(55)
    pool_pk, sk, idx, ko, _ = make_sets(ctx, [3, 5], [32, 32], rng, pool=64)
    m = rng.bytes(32)
    sig, st = sign_sets(ctx, [sum(sk[i] for i in idx[:3]), sum(sk[i] for i in idx[3:])], [m, m]); assert not st.any()
    flat = pool_pk[idx].reshape(-1)
    st, _, rerun = ctx.verify_signature_sets(flat, ko, [m, m], sig.reshape(-1), seed16=SEED)
    assert st.tolist() == [0, 0] and rerun == 0
    st, _, rerun = ctx.verify_signature_sets(flat, ko, [m, m], sig[::-1].reshape(-1), seed16=SEED)
    assert st.tolist() == [1, 1] and rerun == 2

@pytest.mark.gpu
def test_pool_sets_equal_compressed_key_sets(ctx):
    rng = np.random.default_rng(303); n = 400
    sizes = rng.choice([0, 1, 4, 33, 200], size=n); lens = rng.integers(0, 100, size=n)
    pool_pk, sk, idx, ko, msgs = make_sets(ctx, sizes, lens, rng, pool=1024)
    sig, _ = sign_sets(ctx, [max(sum(sk[i] for i in idx[int(ko[s]):int(ko[s + 1])]), 1) for s in range(n)], msgs)
    bad_pool = pool_pk.copy(); bad_pool[17, 4] ^= 0x5a; bad_pool[17, 0] = 0x80 | (bad_pool[17, 0] & 0x1f); bad_pool[17, 47] ^= 0x3c
    h, pst = ctx.pool_create(bad_pool.reshape(-1))
    try:
        assert pst[17] > 1
        ix = idx.copy(); s_oob = int(np.nonzero(sizes > 1)[0][0]); ix[int(ko[s_oob]) + 1] = 1024 + 5        # out-of-range index
        s_bad = [s for s in range(n) if 17 in ix[int(ko[s]):int(ko[s + 1])].tolist() and s != s_oob]
        if not s_bad: s_bad = [int(np.nonzero(sizes > 0)[0][-1])]; ix[int(ko[s_bad[0]])] = 17
        sel = rng.random(ix.size) < 0.9; sel[int(ko[s_oob]) + 1] = True
        for s in s_bad: sel[int(ko[s]):int(ko[s + 1])] |= ix[int(ko[s]):int(ko[s + 1])] == 17
        bm = bits_to_words(sel)
        ref_keys = np.concatenate([bad_pool, np.zeros((8, 48), np.uint8)])                                  # index 1029 -> an all-zero (undecodable) key
        for b in (None, bm):
            want, _, _ = ctx.verify_signature_sets(ref_keys[np.minimum(ix, 1024 + 7)].reshape(-1), ko, msgs, sig.reshape(-1), bitmap=b)
            for seed in (None, SEED):
                st, _, _ = ctx.pool_verify_signature_sets(h, ix, ko, msgs, sig.reshape(-1), seed16=seed, bitmap=b)
                assert np.array_equal(st, want)
            assert st[s_oob] == 2 and all(st[s] == 2 for s in s_bad) and (b is not None or (st == 0).sum() > n // 2)    # the signatures cover every key
    finally: ctx.pool_free(h)

@pytest.mark.gpu
def test_device_pointer_mode_and_null_pointers(ctx):
    import torch
    from bls_verify_gadget_b200 import _lib, BlsGpuError
    rng = np.random.default_rng(77); n = 700
    sizes = rng.choice([0, 1, 2, 9, 70], size=n); lens = rng.integers(0, 80, size=n)
    pool_pk, sk, idx, ko, msgs = make_sets(ctx, sizes, lens, rng, pool=512)
    sig, _ = sign_sets(ctx, [max(sum(sk[i] for i in idx[int(ko[s]):int(ko[s + 1])]), 1) for s in range(n)], msgs)
    sig[9] = sig[10]; msgs[30] = msgs[30] + b"x"
    flat = pool_pk[idx].reshape(-1); sel = rng.random(idx.size) < 0.8; bm = bits_to_words(sel)
    h, _ = ctx.pool_create(pool_pk.reshape(-1))
    try:
        host = {seed: ctx.verify_signature_sets(flat, ko, msgs, sig.reshape(-1), seed16=seed, bitmap=bm) for seed in (None, SEED)}
        phost = ctx.pool_verify_signature_sets(h, idx, ko, msgs, sig.reshape(-1), bitmap=bm)
        mflat, moff = _lib.pack_msgs(msgs)
        d = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in
             dict(pk=flat, ko=ko.view(np.int32), bm=bm.view(np.int64), msg=mflat, off=moff.view(np.int32), sig=sig.reshape(-1), idx=idx.view(np.int32), seed=np.frombuffer(SEED, np.uint8)).items()}
        dst = torch.empty(n, dtype=torch.uint8, device="cuda"); dok = torch.empty((n + 63) // 64, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize(); ctx.set_pointer_mode(True)
        try:
            for seed in (None, SEED):
                rerun = ctx.verify_signature_sets_ptr(d["pk"].data_ptr(), d["ko"].data_ptr(), d["bm"].data_ptr(), d["msg"].data_ptr(), d["off"].data_ptr(), d["sig"].data_ptr(), n,
                                                      d["seed"].data_ptr() if seed else None, dst.data_ptr(), dok.data_ptr())
                ctx.synchronize()
                assert np.array_equal(dst.cpu().numpy(), host[seed][0]) and np.array_equal(dok.cpu().numpy().view(np.uint64), host[seed][1]) and rerun == host[seed][2]
            ctx.pool_verify_signature_sets_ptr(h, d["idx"].data_ptr(), d["ko"].data_ptr(), d["bm"].data_ptr(), d["msg"].data_ptr(), d["off"].data_ptr(), d["sig"].data_ptr(), n,
                                               None, dst.data_ptr()); ctx.synchronize()
            assert np.array_equal(dst.cpu().numpy(), phost[0])
        finally: ctx.set_pointer_mode(False)
        st = np.empty(n, np.uint8)
        for args in ((flat, None, None, mflat, moff, sig.reshape(-1)), (flat, ko, None, None, moff, sig.reshape(-1)), (flat, ko, None, mflat, moff, None)):
            with pytest.raises(BlsGpuError, match="rc=-1"): ctx.verify_signature_sets_ptr(*args, n, None, st)
        with pytest.raises(BlsGpuError, match="rc=-1"): ctx.verify_signature_sets_ptr(flat, ko, None, mflat, moff, sig.reshape(-1), n, None, None)
        with pytest.raises(BlsGpuError, match="rc=-1"): ctx.pool_verify_signature_sets_ptr(h, None, ko, None, mflat, moff, sig.reshape(-1), n, None, st)
        with pytest.raises(BlsGpuError, match="rc=-1"): ctx.pool_verify_signature_sets_ptr(h + 1, idx, ko, None, mflat, moff, sig.reshape(-1), n, None, st)
        assert ctx.verify_signature_sets_ptr(flat, ko, None, mflat, moff, sig.reshape(-1), 0, None, st) == 0      # nsets == 0
    finally: ctx.pool_free(h)
