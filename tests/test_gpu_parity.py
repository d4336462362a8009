"""Parity tests proper: the CUDA path through the C ABI (libblsgpu.so via ctypes) against the CPU oracle on the same
seeded inputs, against the reference's fixtures (tests/golden/eth_vectors.json = /root/reference/tests/test_cases/**
and the inline KATs), and through size-independent properties at larger sizes.  Bit-exact everywhere (integer work).
The harness mirrors /root/reference/tests/tests.rs."""
import hashlib
import numpy as np
import pytest
from conftest import hx

pytestmark = pytest.mark.gpu

@pytest.fixture(scope="module")
def ctx():
    from bls_verify_gadget_b200 import Context
    c = Context(0); yield c; c.close()

@pytest.fixture(scope="module")
def C():
    from oracle import cwrap
    return cwrap

P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
DE_MAP = {0: 0, 1: 0, 2: 1, 3: 2, 4: 3, 5: 4}      # GPU BLSGPU_DE_* -> oracle DE_* (infinity decodes fine in the oracle)

# ------------------------------------------------------------------------------------------ K0: Fp Montgomery product
def test_fp_mul_million(ctx, C):
    rng = np.random.default_rng(1)
    edge = [0, 1, P - 1, P - 2, (1 << 384) % P, 1 << 380, (1 << 381) - 1 - 0, 2, (P - 1) // 2, 0xffffffff, 1 << 32, (1 << 352) - 1, (1 << 384) % P - 1]
    edge = [e % P for e in edge]
    ea = b"".join(x.to_bytes(48, "little") for x in edge for _ in edge); eb = b"".join(y.to_bytes(48, "little") for _ in edge for y in edge)
    n = 1 << 20
    a = rng.integers(0, 256, size=(n, 48), dtype=np.uint8); b = rng.integers(0, 256, size=(n, 48), dtype=np.uint8)
    a[:, 47] &= 0x0f; b[:, 47] &= 0x0f                                    # < 2^380 < p
    a[::7, 40:47] = 0xff; b[::5, 0:20] = 0xff; a[::11, :] = np.frombuffer((P - 1).to_bytes(48, "little"), dtype=np.uint8)
    A = np.concatenate([np.frombuffer(ea, dtype=np.uint8), a.reshape(-1)]); B = np.concatenate([np.frombuffer(eb, dtype=np.uint8), b.reshape(-1)])
    got = ctx.fp_mul_raw(A, B)
    assert np.array_equal(got, C.fp_mul_raw(A, B))
    # chained: r = a*b*b*b (reps=3) == oracle applied three times
    sub = slice(0, 48 * 4096)
    r = C.fp_mul_raw(C.fp_mul_raw(C.fp_mul_raw(A[sub], B[sub]), B[sub]), B[sub])
    assert np.array_equal(ctx.fp_mul_raw(A[sub], B[sub], reps=3), r)

# ------------------------------------------------------------------------------------------ K1: decode / validate
@pytest.mark.parametrize("kind,key,size", [("deserialization_G1", "pubkey", 48), ("deserialization_G2", "signature", 96)])
def test_deser_fixtures(ctx, eth, kind, key, size):                       # tests.rs:337-364
    fn = ctx.deserialize_g1 if size == 48 else ctx.deserialize_g2
    for c in eth[kind]:
        s = c["input"][key]
        ok = len(s) % 2 == 0 and len(s) >= 2 * size and fn(bytes.fromhex(s)[:size])[0] <= 1
        assert ok == c["output"], c["name"]

def _mutated_points(valid, size, rng, n):
    """valid encodings with random mutations: flag flips, random x, x >= p, sign flips"""
    out = np.tile(np.frombuffer(valid, dtype=np.uint8).reshape(-1, size), (n // (len(valid) // size) + 1, 1))[:n].copy()
    for i in range(n):
        m = i % 8
        if m == 1: out[i, 0] ^= 0x20                                      # other sign: still valid
        elif m == 2: out[i, 0] ^= 0x80                                    # compression flag cleared
        elif m == 3: out[i, 0] |= 0x40                                    # infinity flag with garbage
        elif m == 4: out[i, 1:] = rng.integers(0, 256, size=size - 1, dtype=np.uint8); out[i, 0] = 0x80 | (out[i, 0] & 0x0f)   # random x
        elif m == 5: out[i, :48] = 0xff; out[i, 0] = 0x9f                 # x (or x.c1) >= p
        elif m == 6: out[i, size - 1] ^= 1                                # neighbouring x
        elif m == 7 and size == 96: out[i, 48:] = np.frombuffer(P.to_bytes(48, "big"), dtype=np.uint8)   # x.c0 == p
    return out.reshape(-1)

def test_deser_differential(ctx, C, pyv):
    rng = np.random.default_rng(5)
    pks = b"".join(hx(v["pk"]) for v in pyv["sign_items"]) + hx(pyv["g1_not_in_subgroup"])
    sigs = b"".join(hx(v["sig"]) for v in pyv["sign_items"]) + hx(pyv["g2_not_in_subgroup"])
    a = _mutated_points(pks, 48, rng, 1024); b = _mutated_points(sigs, 96, rng, 512)
    g1 = ctx.deserialize_g1(a); g2 = ctx.deserialize_g2(b)
    assert [DE_MAP[x] for x in g1] == list(C.deser_g1(a)) and [DE_MAP[x] for x in g2] == list(C.deser_g2(b))
    assert len(set(g1)) >= 5 and len(set(g2)) >= 5                        # every outcome class was exercised
    assert ctx.deserialize_g1(hx(pyv["g1_not_in_subgroup"]))[0] == 5 and ctx.deserialize_g2(hx(pyv["g2_not_in_subgroup"]))[0] == 5

def test_cofactor_torsion_points_rejected(ctx, C):
    """points of the cofactor subgroups must fail the endomorphism membership tests exactly like [r]P != O"""
    from oracle import pyref as R
    rng = np.random.default_rng(9); pts1 = []; pts2 = []
    h1 = 0x396c8c005555e1568c00aaab0000aaab
    x = 3
    while len(pts1) < 24:
        x += 1
        try: Pt = R.deser_g1(bytes([0x80]) + x.to_bytes(47, "big"), subgroup=False)
        except R.DeserErr: continue
        for k in (R.r, R.r * 3, R.r * (h1 // 3), R.r * (h1 // 11), R.r * (h1 // 10177)):      # kill the r-part, land in cofactor subgroups
            Q = R.g1mul(k, Pt)
            if Q is not None: pts1.append(R.ser_g1(Q))
    x = 1
    while len(pts2) < 8:
        x += 1
        try: Qt = R.deser_g2(bytes([0x80]) + bytes(47) + x.to_bytes(48, "big"), subgroup=False)
        except R.DeserErr: continue
        Q = R.smul(R.r, Qt)
        if Q is not None: pts2.append(R.ser_g2(Q))
    a = b"".join(pts1); b = b"".join(pts2)
    assert set(ctx.deserialize_g1(a)) == {5} and set(C.deser_g1(a)) == {4}
    assert set(ctx.deserialize_g2(b)) == {5} and set(C.deser_g2(b)) == {4}

# ------------------------------------------------------------------------------------------ K2: hash-to-G2
def test_hash_to_g2_kats(ctx, eth, pyv):                                  # bls.rs:643-652
    assert ctx.hash_to_g2([bytes(32)]).tobytes().hex() == eth["inline_kats"]["hash_to_g2_zero32"]
    msgs = [hx(v["msg"]) for v in pyv["hash_to_g2"]]
    assert ctx.hash_to_g2(msgs).tobytes().hex() == "".join(v["out"] for v in pyv["hash_to_g2"])

def test_hash_to_g2_differential(ctx, C):
    rng = np.random.default_rng(11)
    lens = [0, 1, 31, 32, 33, 54, 55, 56, 63, 64, 65, 118, 119, 120, 128, 250, 300] + list(rng.integers(0, 200, size=239))
    msgs = [rng.bytes(int(l)) for l in lens]                              # ragged, incl. empty and SHA padding boundaries
    assert np.array_equal(ctx.hash_to_g2(msgs), C.hash_to_g2(msgs, threads=8))

# ------------------------------------------------------------------------------------------ K6/K7: sk -> pk, sign, encode
def test_sign_fixtures(ctx, eth):                                         # tests.rs:203-237
    for c in eth["sign"]:
        sk = hx(c["input"]["privkey"])[::-1]
        sig, st = ctx.sign(sk, [hx(c["input"]["message"])])
        if c["output"] is None: assert st[0] == 5, c["name"]
        else: assert st[0] == 0 and sig.tobytes() == hx(c["output"]), c["name"]

def test_sk_to_pk_and_sign_differential(ctx, C, eth):
    from bls_verify_gadget_b200 import synth
    n = 64; sk = synth.secret_keys(n); msg = synth.messages(n)
    sk[32 * 5:32 * 6] = 0                                                 # zero key -> InvalidSecretKey on sign
    sk[32 * 6:32 * 7] = 0xff                                              # non-canonical
    pk, st = ctx.sk_to_pk(sk); opk = C.sk_to_pk(sk)
    good = np.ones(n, bool); good[6] = False
    assert st[6] == 5 and np.array_equal(pk.reshape(n, 48)[good], opk.reshape(n, 48)[good])
    msgs = [msg[32 * i:32 * i + 32].tobytes() for i in range(n)]
    sig, st = ctx.sign(sk, msgs); osig, ost = C.sign(sk, msgs, threads=8)
    assert list(st) == list(ost) and np.array_equal(sig, osig)
    k = eth["inline_kats"]                                                # bls.rs:620-641 aggregate KAT
    pks, _ = ctx.sk_to_pk(b"".join(hx(s) for s in k["aggregate_sks_le_hex"]))
    agg, st = ctx.g1_aggregate(pks, [0, 4])
    assert st[0] == 0 and agg.tobytes().hex() == k["aggregate_pk"]

# ------------------------------------------------------------------------------------------ K3: aggregation
def test_aggregate_fixtures(ctx, eth):                                    # tests.rs:271-294
    for c in eth["aggregate"]:
        out, st = ctx.g2_aggregate(b"".join(hx(s) for s in c["input"]), [0, len(c["input"])])
        if c["output"] is None: assert st[0] == 4, c["name"]
        else: assert st[0] == 0 and out.tobytes() == hx(c["output"]), c["name"]

def test_g1_segmented_aggregate_differential(ctx, C):
    from bls_verify_gadget_b200 import synth
    n = 700; pk, _ = ctx.sk_to_pk(synth.secret_keys(n)); pk = pk.reshape(n, 48).copy()
    seg = [0, 1, 1, 3, 12, 22, 40, 41, 553, 700]                          # ragged, an empty segment, one of 512 (one lane per segment)
    pk[4] = pk[3]                                                         # segment [3, 12) opens with K, K: the running sum equals the added point, the doubling branch of the addition
    pk[13] = pk[12]; pk[13, 0] ^= 0x20                                    # segment [12, 22) opens with P, -P: the running sum cancels to the identity
    pk[30] = 0; pk[30, 0] = 0xc0                                          # identity member
    out, st = ctx.g1_aggregate(pk.reshape(-1), seg); oout, ost = C.g1_aggregate(pk.reshape(-1), seg, threads=8)
    assert list(st) == list(ost) == [0, 4, 0, 0, 0, 0, 0, 0, 0]
    ok = st == 0
    assert np.array_equal(out.reshape(-1, 48)[ok], oout.reshape(-1, 48)[ok])
    pk[600, 5] ^= 0x55                                                    # a member that no longer decodes
    out, st = ctx.g1_aggregate(pk.reshape(-1), seg); oout, ost = C.g1_aggregate(pk.reshape(-1), seg, threads=8)
    assert list(st) == list(ost) and st[-1] == 2

def test_fast_aggregate_verify_fixtures(ctx, eth):                        # tests.rs:297-334
    for c in eth["fast_aggregate_verify"]:
        i = c["input"]; pks = b"".join(hx(s) for s in i["pubkeys"])
        st = ctx.fast_aggregate_verify(pks, len(i["pubkeys"]), hx(i["message"]), hx(i["signature"]))[0]
        assert (st == 0) == c["output"], c["name"]

def test_committees_differential(ctx, C):
    from bls_verify_gadget_b200 import synth
    nc, k = 6, 64
    pks, msg, sig, _, _ = synth.committees(ctx, nc, k=k, pool=256)
    sig = sig.copy(); msg = msg.copy()
    msg[32 * 1] ^= 1                                                      # committee 1: wrong message
    sig[96 * 2 + 95] ^= 1                                                 # committee 2: undecodable / wrong signature
    st, agg = ctx.fast_aggregate_verify(pks, k, msg, sig, want_agg=True)
    ost, oagg = C.fast_aggregate_verify(pks, k, msg, sig, want_agg=True, threads=8)
    assert list(st) == list(ost) and st[0] == 0 and st[1] == 1 and np.array_equal(agg, oagg)
    # participation bitmap (gadget semantics, constraints.rs:181-182): 2/3 of the bits; signature no longer matches
    rng = np.random.default_rng(3); bits = rng.random(nc * k) < 0.66
    bm = np.zeros((nc * k + 63) // 64, dtype=np.uint64)
    for j in np.nonzero(bits)[0]: bm[j // 64] |= np.uint64(1) << np.uint64(j % 64)
    st, agg = ctx.fast_aggregate_verify(pks, k, msg, sig, bitmap=bm, want_agg=True)
    ost, oagg = C.fast_aggregate_verify(pks, k, msg, sig, bitmap=bm, want_agg=True, threads=8)
    assert list(st) == list(ost) and np.array_equal(agg, oagg)

# ------------------------------------------------------------------------------------------ K4/K5: pairing, verify
def test_gt_bytes(ctx, C, pyv):                                           # SURVEY A.9 anchor (parity-unpinned vs arkworks)
    from oracle import pyref as R
    gt, st = ctx.pairing_gt(R.ser_g1(R.G1), R.ser_g2(R.G2), 1)
    assert st[0] == 0 and hashlib.sha256(gt[0].tobytes()).hexdigest() == pyv["gt_anchor"]["sha256"]
    tp = pyv["gt_two_pair"]
    gt, st = ctx.pairing_gt(b"".join(hx(s) for s in tp["g1"]), b"".join(hx(s) for s in tp["g2"]), 2)
    assert gt[0].tobytes().hex() == tp["bytes"]
    # a pair with the identity is dropped: e(O, g2) * e(g1, g2) == e(g1, g2)
    gt2, _ = ctx.pairing_gt(bytes([0xc0]) + bytes(47) + R.ser_g1(R.G1), R.ser_g2(R.G2) * 2, 2)
    assert hashlib.sha256(gt2[0].tobytes()).hexdigest() == pyv["gt_anchor"]["sha256"]
    assert ctx.gt_fold(np.concatenate([gt2[0], gt2[0]])).tobytes() == C.gt_mul(gt2[0], gt2[0]).tobytes()

def test_verify_fixtures(ctx, eth):                                       # tests.rs:240-268
    pk = b"".join(hx(c["input"]["pubkey"]) for c in eth["verify"]); sig = b"".join(hx(c["input"]["signature"]) for c in eth["verify"])
    msgs = [hx(c["input"]["message"]) for c in eth["verify"]]
    st = ctx.verify(pk, msgs, sig)                                        # one batch (a small pass: six-lane final exponentiation by default)
    for c, s in zip(eth["verify"], st): assert (s == 0) == c["output"], c["name"]
    ctx.set_coop(0)                                                       # the same through the thread-per-item final-exponentiation kernels of the large passes
    try: st0 = ctx.verify(pk, msgs, sig)
    finally: ctx.set_coop(2)
    assert np.array_equal(st0, st)
    for c in eth["verify"]:                                               # and one by one (n = 1 calls must work)
        i = c["input"]; assert (ctx.verify(hx(i["pubkey"]), [hx(i["message"])], hx(i["signature"]))[0] == 0) == c["output"]

def test_verify_differential_with_corruptions(ctx, C):
    from bls_verify_gadget_b200 import synth
    n = 320
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=8, fast=False)
    msgs = [msg[32 * i:32 * i + 32].tobytes() for i in range(n)]
    st, bm, gt = ctx.verify(pk, msgs, sig, want_bitmap=True, want_gt=True)
    ost, ogt = C.verify(pk, msgs, sig, want_gt=True, threads=8)
    assert list(st) == list(ost) == list(exp) and set(st) == {0, 1, 2, 3}
    assert gt.tobytes() == ogt.tobytes()
    bits = [(int(bm[i // 64]) >> (i % 64)) & 1 for i in range(n)]
    assert bits == [int(s == 0) for s in st]
    # fixed-32 fast path and ragged path agree
    assert np.array_equal(ctx.verify(pk, msg, sig, fixed32=True), st)
    ctx.set_coop(0)                                                       # thread-per-item final exponentiation (what passes above 4,096 items run)
    try: st0, gt0 = ctx.verify(pk, msgs, sig, want_gt=True)
    finally: ctx.set_coop(2)
    assert np.array_equal(st0, st) and gt0.tobytes() == gt.tobytes()

def test_verify_ragged_messages_and_identity_signature(ctx, C):
    from bls_verify_gadget_b200 import synth
    rng = np.random.default_rng(21); n = 40
    sk = synth.secret_keys(n); msgs = [rng.bytes(int(l)) for l in rng.integers(0, 150, size=n)]; msgs[0] = b""
    pk, _ = ctx.sk_to_pk(sk); sig, _ = ctx.sign(sk, msgs)
    sig = sig.copy(); sig[96 * 3:96 * 4] = 0; sig[96 * 3] = 0xc0          # identity signature: accepted by check(), verifies false (SURVEY B2)
    st = ctx.verify(pk, msgs, sig); ost = C.verify(pk, msgs, sig, threads=8)
    assert list(st) == list(ost) and st[3] == 1 and (np.delete(st, 3) == 0).all()

def test_verify_large_batch_properties(ctx):
    """2^16 triples (the 2^20 run is bench.py's): statuses equal the by-construction expectation, the bitmap is the
    status vector, and the GT accumulator is invariant under a permutation of the batch (product is commutative)."""
    from bls_verify_gadget_b200 import synth
    n = 1 << 16
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=64)
    st, bm, gt = ctx.verify(pk, msg, sig, want_bitmap=True, want_gt=True, fixed32=True)
    assert np.array_equal(st, exp)
    assert np.array_equal(np.unpackbits(bm.view(np.uint8), bitorder="little")[:n], (st == 0).astype(np.uint8))
    for lanes in (1, 4):                                                  # serial kernels vs four concurrent sub-range streams
        ctx.set_lanes(lanes)
        st_l, bm_l, gt_l = ctx.verify(pk, msg, sig, want_bitmap=True, want_gt=True, fixed32=True)
        assert np.array_equal(st_l, st) and np.array_equal(bm_l, bm) and gt_l.tobytes() == gt.tobytes()
    ctx.set_lanes(2)
    perm = np.random.default_rng(2).permutation(n)
    st2, gt2 = ctx.verify(pk.reshape(n, 48)[perm].reshape(-1), msg.reshape(n, 32)[perm].reshape(-1), sig.reshape(n, 96)[perm].reshape(-1), want_gt=True, fixed32=True)
    assert np.array_equal(st2, exp[perm]) and gt2.tobytes() == gt.tobytes()
    # two-way split == what two ranks would produce; fold of the partials == whole-batch accumulator
    h = n // 2
    parts = [ctx.verify(pk[:48 * h], msg[:32 * h], sig[:96 * h], want_gt=True, fixed32=True)[1], ctx.verify(pk[48 * h:], msg[32 * h:], sig[96 * h:], want_gt=True, fixed32=True)[1]]
    assert ctx.gt_fold(np.concatenate(parts)).tobytes() == gt.tobytes()

# ------------------------------------------------------------------------------------------ K8: R1CS check
def _plant(mats, nfree, nrows, ncols, rng, nwit, break_rows):
    zs = []
    for w in range(nwit):
        z = [1] + [int.from_bytes(rng.bytes(47), "little") for _ in range(nfree - 1)] + [0] * nrows
        for i in range(nrows):
            d = []
            for m in range(2):
                rp, col, cf = mats[m]
                d.append(sum(int.from_bytes(cf[48 * k:48 * k + 48].tobytes(), "little") * z[col[k]] for k in range(int(rp[i]), int(rp[i + 1]))) % P)
            z[nfree + i] = d[0] * d[1] % P
        for r in break_rows.get(w, []): z[nfree + r] = (z[nfree + r] + 1) % P
        zs.append(b"".join(v.to_bytes(48, "little") for v in z))
    return b"".join(zs)

def test_r1cs_differential(ctx, C):
    from bls_verify_gadget_b200 import synth
    rng = np.random.default_rng(17); nrows, ncols, nwit = 200, 260, 37
    mats, nfree = synth.r1cs_system(nrows, ncols)
    broken = {3: [0, 63, 64, 199], 36: [100]}
    z = _plant(mats, nfree, nrows, ncols, rng, nwit, broken)
    h = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], nrows, ncols)
    bits, allsat = ctx.r1cs_check(h, z, nwit, nrows)
    obits, oall = C.r1cs_check([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], nrows, ncols, z, nwit, threads=8)
    ctx.r1cs_free(h)
    assert np.array_equal(bits, obits) and list(allsat) == list(oall)
    assert allsat.sum() == nwit - 2 and allsat[3] == 0 and allsat[36] == 0
    unsat = lambda w: [i for i in range(nrows) if not (int(bits[w, i // 64]) >> (i % 64)) & 1]
    assert unsat(3) == [0, 63, 64, 199] and unsat(36) == [100]

def test_r1cs_coefficient_classes_and_packed_columns(ctx, C):
    """Crafted system for the kernel's special cases: coefficients on both sides of every class boundary (0, +-1, 2, 2^32 - 1 | 2^32,
    p - (2^32 - 1) | p - 2^32, random), columns that are 0/1 in one group of 32 assignments but not in the next, rows of 1..120
    non-zeros (short rows, the integer-only path, 32-entry segments of long rows), satisfied and unsatisfied rows, a ragged second
    group -- every per-constraint bit must equal the oracle's."""
    rng = np.random.default_rng(23); nwit = 45; nbool = 24; nfld = 40; nrows = 300
    special = [0, 1, 2, 3, 12, (1 << 32) - 1, 1 << 32, (1 << 32) + 1, P - 1, P - 2, P - ((1 << 32) - 1), P - (1 << 32), P - (1 << 32) - 1, 1 << 200, (P - 1) // 2]
    def coeff(): return special[int(rng.integers(0, len(special)))] if rng.random() < 0.8 else int.from_bytes(rng.bytes(48), "little") % P
    ncols = 1 + nbool + nfld + nrows                      # constant, 0/1 columns, field columns, one product column per row
    rows = []
    for r in range(nrows):
        mats = []
        for m in range(2):
            n = int(rng.choice([1, 2, 3, 5, 9, 17, 40, 120], p=[.2, .2, .15, .15, .1, .1, .05, .05]))
            only_bool = rng.random() < 0.5                # rows that touch only 0/1 columns take the integer-only test
            cols = rng.choice(np.arange(0, 1 + nbool) if only_bool else np.arange(0, 1 + nbool + nfld), size=min(n, (1 + nbool) if only_bool else 1 + nbool + nfld), replace=False)
            mats.append([(int(c), coeff() if not only_bool or rng.random() < 0.3 else int(rng.choice([1, P - 1, 2, 5, P - 3, (1 << 32) - 1]))) for c in sorted(cols)])
        if r < 20: mats = [[(1 + (3 * r) % nbool, 1)], [(1 + (5 * r + 1) % nbool, 1)]]      # AND gates: all three combinations stay on 0/1 columns
        mats.append([(1 + nbool + nfld + r, 1)])          # C row: the product column
        rows.append(mats)
    z = np.zeros((nwit, ncols), dtype=object); z[:, 0] = 1
    z[:, 1:1 + nbool] = rng.integers(0, 2, size=(nwit, nbool))
    z[35, 5] = 7; z[40, 9] = P - 1                          # columns 5 and 9 stop being 0/1 in the second group only
    edge = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, 1 << 380, (1 << 64) - 1]
    for w in range(nwit):
        for c in range(1 + nbool, 1 + nbool + nfld): z[w, c] = edge[int(rng.integers(0, len(edge)))] if rng.random() < 0.3 else int.from_bytes(rng.bytes(48), "little") % P
    z[:, 30] = rng.integers(0, 2, size=nwit)              # a "field" column that happens to be 0/1 everywhere
    for r, (A, B, Cc) in enumerate(rows):
        for w in range(nwit):
            a = sum(cf * z[w, c] for c, cf in A) % P; b = sum(cf * z[w, c] for c, cf in B) % P
            z[w, 1 + nbool + nfld + r] = a * b % P
    bad = [(3, 0), (3, 299), (17, 64), (40, 128), (44, 7)]
    for w, r in bad: z[w, 1 + nbool + nfld + r] = (z[w, 1 + nbool + nfld + r] + 1) % P
    def csr(m):
        rp = [0]; cl = []; cf = []
        for row in rows:
            for c, v in row[m]: cl.append(c); cf.append(v.to_bytes(48, "little"))
            rp.append(len(cl))
        return np.array(rp, np.uint64), np.array(cl, np.uint32), np.frombuffer(b"".join(cf), np.uint8)
    mats = [csr(m) for m in range(3)]
    zb = np.frombuffer(b"".join(int(v).to_bytes(48, "little") for v in z.reshape(-1)), np.uint8)
    h = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], nrows, ncols)
    bits, allsat = ctx.r1cs_check(h, zb, nwit, nrows); ctx.r1cs_free(h)
    obits, oall = C.r1cs_check([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], nrows, ncols, zb, nwit, threads=4)
    assert np.array_equal(bits, obits) and list(allsat) == list(oall)
    unsat = {(w, r) for w in range(nwit) for r in range(nrows) if not (int(bits[w, r // 64]) >> (r % 64)) & 1}
    assert unsat == set(bad)

def test_r1cs_row_classes(ctx, C):
    """One test per row class of blsgpu_r1cs_load (truth-table rows evaluated bit-sliced, their generic fallback, generic short rows,
    long rows): the Boolean gate forms of ark-r1cs-std -- booleanity a(1-a)=0, AND a b = c, XOR 2a b = a + b - c, OR (1-a)(1-b) = 1-c,
    NOT through the constant column, a conditional select on five columns, a constant row -- with every input combination present in
    the 70 assignments, deliberately wrong outputs, and columns that stop being 0/1 in the second / third group only."""
    rng = np.random.default_rng(41); nwit = 70; nb = 12
    ONE = 0; cols = {"b": list(range(1, 1 + nb))}; nextc = [1 + nb]; rows = []; outs = []
    def newcol(): nextc[0] += 1; return nextc[0] - 1
    M = P - 1
    for i in range(nb): rows.append(([(cols["b"][i], 1)], [(ONE, 1), (cols["b"][i], M)], []))                      # booleanity
    for i in range(10):
        a, b = cols["b"][i], cols["b"][(i + 3) % nb]
        c = newcol(); rows.append(([(a, 1)], [(b, 1)], [(c, 1)])); outs.append((c, "and", (a, b)))                   # AND
        c = newcol(); rows.append(([(a, 2)], [(b, 1)], [(a, 1), (b, 1), (c, M)])); outs.append((c, "xor", (a, b)))    # XOR
        c = newcol(); rows.append(([(ONE, 1), (a, M)], [(ONE, 1), (b, M)], [(ONE, 1), (c, M)])); outs.append((c, "or", (a, b)))   # OR
        s, d = cols["b"][(i + 5) % nb], newcol()                                                                      # select: s (a - b) = d - b on five columns with the constant
        rows.append(([(s, 1)], [(a, 1), (b, M)], [(d, 1), (b, M), (ONE, 0)])); outs.append((d, "sel", (s, a, b)))
    rows.append(([(ONE, 3)], [(ONE, 5)], [(ONE, 15)]))                                                                # constant row (satisfied), one column
    rows.append(([(ONE, 3)], [(ONE, 5)], [(ONE, 16)]))                                                                # constant row (never satisfied)
    fa, fb = newcol(), newcol(); fc = newcol(); rows.append(([(fa, 1)], [(fb, 1)], [(fc, 1)]))                        # a field product on three columns: truth-table shape, always falls back
    wide = [newcol() for _ in range(6)]; wc = newcol(); rows.append(([(c, 1 + k) for k, c in enumerate(wide)], [(ONE, 1)], [(wc, 1)]))      # 8 distinct columns, 8 non-zeros: generic short row
    lcols = [newcol() for _ in range(40)]; lc = newcol()                                                              # 42 non-zeros: a long row (bit-packing shape with a few odd coefficients)
    lcoef = [(1 << (k + 20)) if k % 7 else (P - 3 - k if k % 2 else (0x1234567 << 200) + k) for k in range(40)]
    rows.append(([(c, lcoef[k]) for k, c in enumerate(lcols)], [(ONE, 1)], [(lc, 1)]))
    ncols = nextc[0]; nrows = len(rows)
    z = np.zeros((nwit, ncols), dtype=object); z[:, 0] = 1; z[:, 1:1 + nb] = rng.integers(0, 2, size=(nwit, nb))
    fn = {"and": lambda a, b: a & b, "xor": lambda a, b: a ^ b, "or": lambda a, b: a | b, "sel": lambda s, a, b: a if s else b}
    for w in range(nwit):
        for c, k, ins in outs: z[w, c] = fn[k](*[int(z[w, i]) for i in ins])
        z[w, fa] = int.from_bytes(rng.bytes(48), "little") % P; z[w, fb] = int.from_bytes(rng.bytes(48), "little") % P; z[w, fc] = z[w, fa] * z[w, fb] % P
        for c in wide: z[w, c] = int(rng.integers(0, 2)) if w < 32 else int.from_bytes(rng.bytes(48), "little") % P
        z[w, wc] = sum((1 + k) * z[w, c] for k, c in enumerate(wide)) % P
        for k, c in enumerate(lcols): z[w, c] = int(rng.integers(0, 2)) if (w < 32 or k % 3) else int.from_bytes(rng.bytes(48), "little") % P
        z[w, lc] = (sum(lcoef[k] * z[w, c] for k, c in enumerate(lcols)) + (1 if w in (7, 50) else 0)) % P             # two assignments break the long row
    flips = [(2, outs[0][0]), (31, outs[5][0]), (33, outs[9][0]), (64, outs[39][0]), (69, outs[17][0])]              # wrong gate outputs (still 0/1)
    for w, c in flips: z[w, c] ^= 1
    z[40, cols["b"][2]] = 2; z[66, outs[3][0]] = P - 1; z[5, fc] = (z[5, fc] + 1) % P                                 # non-0/1 values: second and third group only
    def csr(m):
        rp = [0]; cl = []; cf = []
        for row in rows:
            for c, v in row[m]: cl.append(c); cf.append(int(v).to_bytes(48, "little"))
            rp.append(len(cl))
        return np.array(rp, np.uint64), np.array(cl, np.uint32), np.frombuffer(b"".join(cf) + b"\0", np.uint8)[:48 * len(cl)]
    mats = [csr(m) for m in range(3)]
    zb = np.frombuffer(b"".join(int(v).to_bytes(48, "little") for v in z.reshape(-1)), np.uint8)
    h = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], nrows, ncols)
    cls = ctx.r1cs_row_classes(h)
    assert cls == {"truth_table": nrows - 2, "generic": 1, "long": 1, "segments": 4}
    bits, allsat = ctx.r1cs_check(h, zb, nwit, nrows); ctx.r1cs_free(h)
    obits, oall = C.r1cs_check([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], nrows, ncols, zb, nwit, threads=4)
    assert np.array_equal(bits, obits) and list(allsat) == list(oall)
    sat = lambda w, r: (int(bits[w, r // 64]) >> (r % 64)) & 1
    # independent expectation: the planted flips break exactly the rows whose gate they belong to, in their assignment only
    for w in range(nwit):
        for r, (A, B, Cc) in enumerate(rows):
            ev = lambda lc: sum(cf * int(z[w, c]) for c, cf in lc) % P
            assert sat(w, r) == int(ev(A) * ev(B) % P == ev(Cc)), (w, r)
    assert not allsat.any()                                                                                         # the unsatisfiable constant row

def test_r1cs_load_rejects_bad_systems(ctx):
    """a column index out of range or a non-monotone row pointer is an argument error and leaves no half-built system behind (all 16 handles stay usable)"""
    from bls_verify_gadget_b200._lib import BlsGpuError
    one = (1).to_bytes(48, "little")
    rp = np.array([0, 1, 2], np.uint64); cf = np.frombuffer(one * 2, np.uint8)
    for _ in range(20):
        with pytest.raises(BlsGpuError): ctx.r1cs_load([rp] * 3, [np.array([0, 7], np.uint32)] * 3, [cf] * 3, 2, 3)
    with pytest.raises(BlsGpuError): ctx.r1cs_load([np.array([0, 2, 1], np.uint64)] * 3, [np.array([0, 1], np.uint32)] * 3, [cf] * 3, 2, 3)
    hs = [ctx.r1cs_load([rp] * 3, [np.array([0, 1], np.uint32)] * 3, [cf] * 3, 2, 3) for _ in range(16)]
    assert sorted(hs) == list(range(16))
    for h in hs: ctx.r1cs_free(h)

def test_r1cs_verify_circuit_on_gpu(ctx, C):
    """K8 on the REAL system: the matrices and assignments of BlsSignatureVerifyGadget::verify (constraints.rs:90-128) built
    by the host-side builder (714 k rows).  Assignments of a valid and an invalid signature are both satisfying (the gadget
    returns a Boolean), a perturbed one is not; every per-constraint bit must equal the oracle's."""
    from bls_verify_gadget_b200 import gadget as G
    pk = bytes.fromhex("a491d1b0ecd9bb917989f0e74f0dea0422eac4a873e5e2644f368dffb9a6e20fd6e10c1b77654d067c0618f6e5a7f79a")
    sig = bytes.fromhex("882730e5d03f6b42c3abc26d3372625034e1d871b65a8a6b900a56dae22da98abbe1b68f85e49fe7652a55ec3d0591c2"
                        "0767677e33e5cbb1207315c41a9ac03be39c2e7668edc043d6cb1d9fd93033caa8a1c5b0e84bedaeb6c64972503a43eb")
    c = G.verify_circuit(pk, bytes.fromhex("56" * 32), sig); assert c.result is True         # constraints.rs:326-332
    z, res = G.verify_witnesses([(pk, bytes.fromhex("56" * 32), sig), (pk, bytes.fromhex("78" * 32), sig)], threads=2)
    assert list(res) == [True, False]
    bad = z[0].reshape(c.ncols, 48).copy(); bad[c.ncols // 2, 0] ^= 1; bad[c.ncols - 5, 3] ^= 0x40
    zz = np.concatenate([z[0], z[1], bad.reshape(-1)])
    mats = c.matrices()
    h = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c.nrows, c.ncols)
    bits, allsat = ctx.r1cs_check(h, zz, 3, c.nrows)
    ctx.r1cs_free(h)
    obits, oall = C.r1cs_check([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c.nrows, c.ncols, zz, 3, threads=C.hw_threads())
    assert np.array_equal(bits, obits) and list(allsat) == list(oall) == [1, 1, 0]

def test_r1cs_aggregate_verify_circuit_on_gpu(ctx, C):
    """K8 on the aggregate_verify system (constraints.rs:153-191: 512 masked keys + participant count, 739,876 rows): both of the
    reference's cases (bitmap {0,1}: true; all set: false) are satisfying assignments of the SAME matrices; GPU bits = oracle bits."""
    from bls_verify_gadget_b200 import gadget as G
    pk1 = bytes.fromhex("a491d1b0ecd9bb917989f0e74f0dea0422eac4a873e5e2644f368dffb9a6e20fd6e10c1b77654d067c0618f6e5a7f79a")
    pk2 = bytes.fromhex("b301803f8b5ac4a1133581fc676dfedc60d891dd5fa99028805e5ea5b08d3491af75d0707adab3b70c6a6a580217bf81")
    sig = bytes.fromhex("912c3615f69575407db9392eb21fee18fff797eeb2fbe1816366ca2a08ae574d8824dbfafb4c9eaa1cf61b63c6f9b69911f269b664c42947dd1b53ef1081926c"
                        "1e82bb2a465f927124b08391a5249036146d6f3f1e17ff5f162f779746d830d1")
    msg = bytes.fromhex("56" * 32)
    c1 = G.aggregate_verify_circuit(pk1 + pk2 * 511, [1, 1] + [0] * 510, msg, sig); c2 = G.aggregate_verify_circuit(pk1 + pk2 * 511, [1] * 512, msg, sig)
    assert (c1.result, c1.count, c2.result, c2.count) == (True, 2, False, 512) and (c1.nrows, c1.ncols) == (c2.nrows, c2.ncols)
    z1 = c1.assignment(); z2 = c2.assignment(); bad = z1.reshape(c1.ncols, 48).copy(); bad[c1.ncols // 2, 0] ^= 1  # (a masked-out key coordinate would be unconstrained: the circuit multiplies it by its bit)
    zz = np.concatenate([z1, z2, bad.reshape(-1)]); mats = c1.matrices()
    h = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c1.nrows, c1.ncols)
    bits, allsat = ctx.r1cs_check(h, zz, 3, c1.nrows); ctx.r1cs_free(h)
    obits, oall = C.r1cs_check([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c1.nrows, c1.ncols, zz, 3, threads=C.hw_threads())
    assert np.array_equal(bits, obits) and list(allsat) == list(oall) == [1, 1, 0]

def test_gpu_witness_generation_matches_host_builder(ctx, C):
    """blsgpu_witness_gen (SURVEY 8(f)-1) replays the builder's witness program on the GPU: the assignments must equal the host
    synthesis byte for byte for valid and invalid signatures and distinct keys, satisfy every row of the verify circuit, and
    undecodable inputs must be flagged."""
    from bls_verify_gadget_b200 import gadget as G, synth
    n = 37                                                                                    # two groups, the second ragged
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=5, fast=False)                # wrong msg / swaps / tampered sig / identity pk
    triples = [(pk[48 * i:48 * i + 48].tobytes(), msg[32 * i:32 * i + 32].tobytes(), sig[96 * i:96 * i + 96].tobytes()) for i in range(n)]
    prog = G.verify_program(*triples[0]); nvars = prog["nvars"]
    h = ctx.witness_load(prog)                                                                # level-synchronous replay (cooperative launch)
    z, st = ctx.witness_gen(h, pk, msg, sig, nvars)
    assert prog["ncols"] > nvars and prog["level_ptr"].size - 1 > 1000                        # scratch columns exist; thousands of dependency levels
    assert list(st) == [0 if e in (0, 1) else e for e in exp]                                 # 2: identity key, 3: undecodable signature
    good = [i for i in range(n) if exp[i] in (0, 1)]
    zh, res = G.verify_witnesses([triples[i] for i in good], ncols=nvars)
    assert list(res) == [exp[i] == 0 for i in good]
    for k, i in enumerate(good): assert np.array_equal(z[i], zh[k]), f"assignment {i} differs from the host synthesis"
    c = G.verify_circuit(*triples[good[0]]); mats = c.matrices(); assert c.ncols == nvars
    hh = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c.nrows, c.ncols)
    bits, allsat = ctx.r1cs_check(hh, z.reshape(-1), n, c.nrows)
    assert list(allsat) == [1 if e in (0, 1) else 0 for e in exp]                             # flagged items carry no assignment
    fbits, fall, fst = ctx.witness_check(h, hh, pk, msg, sig, c.nrows)                        # fused: generation + check without the row-major copy
    assert np.array_equal(fbits, bits) and np.array_equal(fall, allsat) and np.array_equal(fst, st)
    ctx.r1cs_free(hh); ctx.witness_free(h)

@pytest.mark.parametrize("mlen", [0, 31, 33, 250])
def test_gpu_witness_generation_any_message_length(ctx, C, mlen):
    """The gadget takes &[UInt8] of any length (constraints.rs:90-95) and the reference tests 0..250-byte messages (hasher.rs:1005-1026):
    a witness program recorded for messages of `mlen` bytes (its own circuit: the number of SHA-256 blocks depends on the length) replays
    to the host synthesis byte for byte for a valid triple, a wrong message and a swapped signature, and satisfies its own system."""
    from bls_verify_gadget_b200 import gadget as G, synth
    rng = np.random.default_rng(100 + mlen); n = 3
    sk = synth.secret_keys(n); msgs = [rng.bytes(mlen) for _ in range(n)]
    pk, _ = ctx.sk_to_pk(sk); sig, st = ctx.sign(sk, msgs); assert not st.any()
    S = sig.reshape(n, 96).copy(); S[[1, 2]] = S[[2, 1]]                                      # items 1 and 2: someone else's signature (valid points)
    triples = [(pk[48 * i:48 * i + 48].tobytes(), msgs[i], S[i].tobytes()) for i in range(n)]
    want = C.verify(pk, msgs, S.reshape(-1)); assert list(want) == [0, 1, 1]
    prog = G.verify_program(*triples[0]); nvars = prog["nvars"]; assert prog["msg_len"] == mlen
    h = ctx.witness_load(prog); assert ctx.witness_msg_len(h) == mlen
    z, gst = ctx.witness_gen(h, pk, b"".join(msgs), S.reshape(-1), nvars); assert not gst.any()
    zh, res = G.verify_witnesses(triples, ncols=nvars)
    assert list(res) == [s == 0 for s in want] and np.array_equal(z, zh)
    c = G.verify_circuit(*triples[0]); mats = c.matrices(); assert c.ncols == nvars
    hh = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c.nrows, c.ncols)
    fbits, fall, fst = ctx.witness_check(h, hh, pk, b"".join(msgs), S.reshape(-1), c.nrows); assert list(fall) == [1, 1, 1] and not fst.any()
    ctx.r1cs_free(hh); ctx.witness_free(h)

def test_gpu_witness_generation_aggregate_circuit(ctx, C):
    """The witness program of the aggregate_verify circuit (constraints.rs:153-191: keys masked by a witness bitmap, summed with the complete
    addition, participant count by UInt32::addmany, then verify on the aggregate) replayed on the GPU: assignments equal the host synthesis
    byte for byte for different bitmaps / keys / messages (valid aggregate, wrong bitmap, wrong message), every row of the circuit's own
    system holds, and an item with an undecodable key is flagged.  8 keys keep the host side quick; the reference's 512-key instance differs
    only in the loop count (test_r1cs_aggregate_verify_circuit_on_gpu checks that system)."""
    from bls_verify_gadget_b200 import gadget as G, synth
    nk = 8; n = 4; rng = np.random.default_rng(8)
    sk = synth.secret_keys(nk * n); pk, _ = ctx.sk_to_pk(sk); PKS = pk.reshape(n, nk, 48).copy()
    msgs = [rng.bytes(32) for _ in range(n)]; bitmaps = np.array([[1, 1, 0, 1, 0, 0, 1, 0], [1] * 8, [0, 1, 0, 0, 0, 0, 0, 0], [1, 0, 1, 0, 1, 0, 1, 0]], np.uint8)
    R = synth.R_ORDER; sigs = []
    for i in range(n):                                                                      # aggregate signature of the selected keys: (sum of their sks) * H(m)
        s = sum(int.from_bytes(sk[32 * (i * nk + k):32 * (i * nk + k) + 32].tobytes(), "little") for k in range(nk) if bitmaps[i, k]) % R
        sg, st = ctx.sign(np.frombuffer(s.to_bytes(32, "little"), np.uint8), [msgs[i]]); assert not st.any(); sigs.append(sg)
    SIG = np.concatenate(sigs).reshape(n, 96).copy()
    bm_used = bitmaps.copy(); bm_used[2] = [1, 1, 0, 0, 0, 0, 0, 0]                           # item 2: a bitmap that does not match its signature -> false
    M = list(msgs); M[3] = bytes([M[3][0] ^ 1]) + M[3][1:]                                    # item 3: wrong message -> false
    prog = G.aggregate_verify_program(PKS[0].reshape(-1), bm_used[0], M[0], SIG[0]); nvars = prog["nvars"]; assert prog["nkeys"] == nk
    h = ctx.witness_load(prog)
    z, st = ctx.witness_gen_aggregate(h, PKS.reshape(-1), bm_used, b"".join(M), SIG.reshape(-1), nvars, nk); assert not st.any()
    want = [True, True, False, False]
    c0 = None
    for i in range(n):
        c = G.aggregate_verify_circuit(PKS[i].reshape(-1), bm_used[i], M[i], SIG[i])
        assert c.result == want[i] and c.count == int(bm_used[i].sum()) and c.ncols == nvars
        assert np.array_equal(z[i], c.assignment()), f"assignment {i} differs from the host synthesis"
        if i == 0: c0 = c
        else: c.free()
    mats = c0.matrices(); hh = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c0.nrows, c0.ncols)
    bits, allsat = ctx.r1cs_check(hh, z.reshape(-1), n, c0.nrows); assert list(allsat) == [1] * n
    bad = PKS.copy(); bad[1, 5, 47] ^= 1                                                      # an undecodable key, even a masked-out one, leaves no assignment
    fb, fa, fs = ctx.witness_check_aggregate(h, hh, bad.reshape(-1), bm_used, b"".join(M), SIG.reshape(-1), c0.nrows, nk)
    assert list(fs) == [0, 2, 0, 0] and list(fa) == [1, 0, 1, 1] and np.array_equal(fb[[0, 2, 3]], bits[[0, 2, 3]])
    from bls_verify_gadget_b200._lib import BlsGpuError
    with pytest.raises(BlsGpuError): ctx.witness_gen(h, pk[:48 * n], b"".join(M), SIG.reshape(-1), nvars)      # an aggregate program through the verify entry point
    ctx.r1cs_free(hh); ctx.witness_free(h); c0.free()

def test_rlc_batch_check_agrees_with_per_item_verify(ctx):
    """blsgpu_verify_batch_rlc (one pairing-product equation per batch, SURVEY 8(f)-3): true exactly when every item of the
    batch verifies, for every corruption kind, several seeds, ragged messages, and across internal passes."""
    from bls_verify_gadget_b200 import synth
    n = 200
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=10 ** 9, fast=False)          # all valid
    msgs = [msg[32 * i:32 * i + 32].tobytes() for i in range(n)]
    assert not ctx.verify(pk, msgs, sig).any()
    for seed in (bytes(16), bytes(range(16)), b"\xff" * 16):
        ok, st = ctx.verify_rlc(pk, msgs, sig, seed); assert ok and not st.any()
    ctx.set_chunk(64)
    try: ok, st = ctx.verify_rlc(pk, msgs, sig, bytes(range(16))); assert ok and not st.any()      # 4 passes: accumulators carried across
    finally: ctx.set_chunk(1 << 20)
    P, S = pk.reshape(n, 48), sig.reshape(n, 96)
    def check(p, m, s, want_status=None):
        ok, st = ctx.verify_rlc(p.reshape(-1), m, s.reshape(-1), b"seed-seed-seed-16"[:16])
        full = ctx.verify(p.reshape(-1), m, s.reshape(-1))
        assert ok == (not full.any()) and not ok
        if want_status is not None: assert st[want_status[0]] == want_status[1]
    m2 = list(msgs); m2[17] = m2[17][:-1] + bytes([m2[17][-1] ^ 1]); check(P, m2, S)                    # wrong message
    p2 = P.copy(); p2[[3, 4]] = p2[[4, 3]]; check(p2, msgs, S)                                             # swapped keys: both items false, products do not cancel
    s2 = S.copy(); s2[[100, 101]] = s2[[101, 100]]; check(P, msgs, s2)                                     # swapped signatures (valid subgroup points)
    s3 = S.copy(); s3[7, 92:] = 0xff; check(P, msgs, s3, (7, 3))                                           # undecodable signature
    p3 = P.copy(); p3[0] = 0; p3[0, 0] = 0xc0; check(p3, msgs, S, (0, 2))                                  # identity public key
    # ragged messages through the offsets path
    rng = np.random.default_rng(9); rag = [rng.bytes(int(l)) for l in rng.integers(0, 90, size=24)]
    sk = synth.secret_keys(24); rpk, _ = ctx.sk_to_pk(sk); rsig, _ = ctx.sign(sk, rag)
    ok, st = ctx.verify_rlc(rpk, rag, rsig, bytes(16)); assert ok
    ok, st = ctx.verify_rlc(rpk, rag[1:] + rag[:1], rsig, bytes(16)); assert not ok

def test_rlc_bisect_returns_the_exact_per_item_outcome(ctx):
    """blsgpu_verify_batch_rlc_bisect (SURVEY 8(f)-3, "fall back to per-item checks to recover the exact bitmap"): status bytes and
    ok-bitmap equal blsgpu_verify_batch's for clean batches, for bad items confined to some pieces of 4,096 (only those are re-run),
    for every corruption kind, ragged messages, a ragged last piece, and across internal passes."""
    from bls_verify_gadget_b200 import synth
    n = 3 * 4096 + 777
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=10 ** 9)                                    # all valid
    seed = bytes(range(16))
    st, bm, rerun = ctx.verify_rlc_bisect(pk, msg, sig, seed, fixed32=True)
    assert not st.any() and rerun == 0 and int(np.unpackbits(bm.view(np.uint8)).sum()) == n
    P, M, S = pk.reshape(n, 48).copy(), msg.reshape(n, 32).copy(), sig.reshape(n, 96).copy()
    M[4096 + 5, 0] ^= 1                                                                                      # wrong message          (piece 1)
    S[[4096 + 900, 4096 + 901]] = S[[4096 + 901, 4096 + 900]]                                                # swapped signatures     (piece 1)
    S[3 * 4096 + 10, 92:] = 0xff                                                                             # undecodable signature  (piece 3): decode status, no re-run needed
    P[7] = 0; P[7, 0] = 0xc0                                                                                 # identity public key    (piece 0): decode status
    P[[3 * 4096 + 700, 3 * 4096 + 701]] = P[[3 * 4096 + 701, 3 * 4096 + 700]]                                # swapped keys           (piece 3, the ragged one)
    want, wbm = ctx.verify(P.reshape(-1), M.reshape(-1), S.reshape(-1), want_bitmap=True, fixed32=True)
    assert sorted(np.nonzero(want)[0].tolist()) == [7, 4101, 4996, 4997, 12298, 12988, 12989]
    st, bm, rerun = ctx.verify_rlc_bisect(P.reshape(-1), M.reshape(-1), S.reshape(-1), seed, fixed32=True)
    assert np.array_equal(st, want) and np.array_equal(bm, wbm) and rerun == 4096 + 777                      # pieces 1 and 3 only
    ctx.set_chunk(4096)
    try: st2, bm2, rerun2 = ctx.verify_rlc_bisect(P.reshape(-1), M.reshape(-1), S.reshape(-1), b"another seed 16b", fixed32=True)
    finally: ctx.set_chunk(1 << 20)
    assert np.array_equal(st2, want) and np.array_equal(bm2, wbm) and rerun2 == rerun
    # ragged messages; a batch smaller than one piece falls back as a whole
    rng = np.random.default_rng(19); rag = [rng.bytes(int(l)) for l in rng.integers(0, 70, size=150)]
    sk = synth.secret_keys(150); rpk, _ = ctx.sk_to_pk(sk); rsig, _ = ctx.sign(sk, rag)
    st, bm, rerun = ctx.verify_rlc_bisect(rpk, rag, rsig, seed); assert not st.any() and rerun == 0
    rag2 = list(rag); rag2[77] = rag2[77] + b"x"
    st, bm, rerun = ctx.verify_rlc_bisect(rpk, rag2, rsig, seed); w2, wb2 = ctx.verify(rpk, rag2, rsig, want_bitmap=True)
    assert np.array_equal(st, w2) and np.array_equal(bm, wb2) and rerun == 150 and sorted(np.nonzero(st)[0].tolist()) == [77]

def test_aggregate_verify_distinct_messages(ctx, C, eth):
    """Eth2 AggregateVerify (SURVEY 8(f)-4; the upstream category reference tests/readme.md:4-7 names): GPU = oracle for valid
    aggregates of 1..9 (key, message) pairs with ragged messages, a tampered aggregate, a wrong message, a swapped key, an identity key,
    an undecodable key, an undecodable / identity signature, no pairs -- and a bad key wins over a bad signature (src/bls.rs:434-447 order)."""
    from bls_verify_gadget_b200 import synth
    rng = np.random.default_rng(77); R = synth.R_ORDER
    sizes = [1, 2, 3, 9, 4, 1, 5, 2, 3, 0, 2, 6]; npairs = sum(sizes)
    sk = synth.secret_keys(npairs); msgs = [rng.bytes(int(l)) for l in rng.integers(0, 80, size=npairs)]
    pk, _ = ctx.sk_to_pk(sk); sigs, st = ctx.sign(sk, msgs); assert not st.any()
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint32)
    seg = off.copy(); agg, ast = ctx.g2_aggregate(sigs, seg)                               # Signature::aggregate per group (bls.rs:288-300)
    assert list(ast) == [4 if s == 0 else 0 for s in sizes]
    P = pk.reshape(npairs, 48).copy(); A = agg.reshape(len(sizes), 96).copy(); M = list(msgs)
    A[9] = 0; A[9, 0] = 0xc0                                                               # group 9 has no pairs: identity signature
    want = [0] * len(sizes); want[9] = 4
    A[1] = A[2]; want[1] = 1                                                               # someone else's (valid) aggregate
    j = int(off[4]) + 2; M[j] = M[j] + b"!"; want[4] = 1                                   # wrong message
    j = int(off[6]); P[[j, j + 1]] = P[[j + 1, j]]; want[6] = 1                            # swapped keys inside a group
    j = int(off[7]) + 1; P[j] = 0; P[j, 0] = 0xc0; want[7] = 2                             # identity key
    j = int(off[8]); P[j, 47] ^= 1; want[8] = 2                                            # undecodable key (w.h.p. not on the curve / not in the subgroup)
    A[10, 95] ^= 1; want[10] = 3                                                           # undecodable signature
    j = int(off[11]) + 3; P[j] = 0; P[j, 0] = 0xc0; A[11, 95] ^= 1; want[11] = 2           # bad key AND bad signature: the key is reported
    got = ctx.aggregate_verify(P.reshape(-1), M, off, A.reshape(-1))
    ora = C.aggregate_verify(P.reshape(-1), M, off, A.reshape(-1), threads=8)
    assert list(got) == list(ora) == want
    # the reference's fast_aggregate_verify fixtures (tests.rs:297-334) seen as AggregateVerify with k copies of the message: by bilinearity
    # the same verdict -- the one pin this path has on the reference's golden vectors
    for c in eth["fast_aggregate_verify"]:
        i = c["input"]; keys = [hx(s) for s in i["pubkeys"]]; sgn = hx(i["signature"])
        if any(len(k) != 48 for k in keys) or len(sgn) != 96: continue
        st = ctx.aggregate_verify(b"".join(keys), [hx(i["message"])] * len(keys), np.array([0, len(keys)], np.uint32), sgn)
        assert (st[0] == 0) == c["output"], c["name"]
    # one pair = BLS::verify; an identity signature over real pairs is false, not an error (SURVEY B2)
    one = ctx.aggregate_verify(pk[:48], msgs[:1], np.array([0, 1], np.uint32), sigs[:96]); assert list(one) == [0] == list(ctx.verify(pk[:48], msgs[:1], sigs[:96]))
    ident = np.zeros(96, np.uint8); ident[0] = 0xc0
    assert list(ctx.aggregate_verify(pk[:96], msgs[:2], np.array([0, 2], np.uint32), ident)) == [1] == list(C.aggregate_verify(pk[:96], msgs[:2], np.array([0, 2], np.uint32), ident))

def test_uncompressed_point_encodings(ctx, C, eth):
    """compressed <-> uncompressed ZCash encodings (SURVEY 8(f)-4): GPU = oracle byte for byte in both directions on generated points, the
    identity, every deserialisation fixture of the reference (their decode verdict carries over), and crafted bad uncompressed inputs
    (compression flag set, x >= p, off the curve, on the curve but outside the subgroup)."""
    from bls_verify_gadget_b200 import synth
    n = 40; sk = synth.secret_keys(n); pk, _ = ctx.sk_to_pk(sk); sg, _ = ctx.sign(sk, [bytes([i]) * (i % 5) for i in range(n)])
    pk = np.concatenate([pk, np.frombuffer(bytes([0xc0]) + bytes(47), np.uint8)]); sg = np.concatenate([sg, np.frombuffer(bytes([0xc0]) + bytes(95), np.uint8)])
    u1, s1 = ctx.g1_uncompress(pk); o1, os1 = C.g1_recode(pk, True); assert np.array_equal(u1, o1) and list(s1[:n]) == [0] * n and s1[n] == 1 and not os1.any()
    u2, s2 = ctx.g2_uncompress(sg); o2, os2 = C.g2_recode(sg, True); assert np.array_equal(u2, o2) and list(s2[:n]) == [0] * n and s2[n] == 1
    c1, t1 = ctx.g1_compress(u1); c2, t2 = ctx.g2_compress(u2); assert np.array_equal(c1, pk) and np.array_equal(c2, sg) and list(t1) == list(s1) and list(t2) == list(s2)
    assert np.array_equal(C.g1_recode(u1, False)[0], pk) and np.array_equal(C.g2_recode(u2, False)[0], sg)
    for kind, key, size, unc in (("deserialization_G1", "pubkey", 48, ctx.g1_uncompress), ("deserialization_G2", "signature", 96, ctx.g2_uncompress)):
        for case in eth[kind]:
            s = case["input"][key]
            if len(s) != 2 * size: continue
            out, st = unc(np.frombuffer(bytes.fromhex(s), np.uint8)); assert (st[0] <= 1) == case["output"], case["name"]
    P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
    good = bytes(u1[:96]); bad = [bytes([good[0] | 0x80]) + good[1:], P.to_bytes(48, "big") + good[48:], good[:95] + bytes([good[95] ^ 1])]
    x = 4                                                                                  # a curve point outside the subgroup: smallest x >= 4 with x^3 + 4 a square
    while pow((x ** 3 + 4) % P, (P - 1) // 2, P) != 1: x += 1
    y = pow((x ** 3 + 4) % P, (P + 1) // 4, P); bad.append(x.to_bytes(48, "big") + y.to_bytes(48, "big"))
    b = np.frombuffer(b"".join(bad), np.uint8); out, st = ctx.g1_compress(b); oo, ost = C.g1_recode(b, False)
    assert list(st) == [2, 3, 4, 5] and [int(v) for v in ost] == [1, 2, 3, 4] and not out.any() and not oo.any()

# ------------------------------------------------------------------------------------------ the reference-shaped API (src/bls.rs)
def test_bls_api_like_reference_tests(ctx, eth):
    from bls_verify_gadget_b200 import BLS, PrivateKey, PublicKey, Signature, BLSError, hash_to_g2
    from bls_verify_gadget_b200.bls import SerializationError
    k = eth["inline_kats"]; params = BLS.setup()
    sk = PrivateKey.try_from(k["sk_le_hex"]); assert sk.to_hex() == k["sk_le_hex"]                       # bls.rs:569-586
    assert PublicKey.try_from(k["pubkey_roundtrip"], ctx).to_hex() == k["pubkey_roundtrip"]              # bls.rs:588-597
    pks = [PublicKey.from_private(PrivateKey.try_from(s), ctx) for s in k["aggregate_sks_le_hex"]]
    assert PublicKey.aggregate(pks, ctx).to_hex() == k["aggregate_pk"] and PublicKey.aggregate([], ctx) is None   # bls.rs:620-641
    assert hash_to_g2(bytes(32), ctx).to_hex() == k["hash_to_g2_zero32"]                                 # bls.rs:643-652
    with pytest.raises(BLSError): BLS.sign(params, PrivateKey(), b"x", ctx=ctx)                          # zero key, bls.rs:417-419
    for c in eth["verify"]:                                                                              # tests.rs:240-268
        i = c["input"]
        try: pk = PublicKey.try_from(i["pubkey"], ctx)
        except SerializationError: pk = PublicKey()
        try: sig = Signature.try_from(i["signature"], ctx)
        except SerializationError: sig = Signature()
        try: res = BLS.verify(params, pk, hx(i["message"]), sig, ctx=ctx)
        except BLSError: res = False
        assert res == c["output"], c["name"]
    rng = np.random.default_rng(4)
    pk, sk = BLS.keygen(params, rng, ctx=ctx); sig = BLS.sign(params, sk, b"hello", ctx=ctx)
    assert BLS.verify(params, pk, b"hello", sig, ctx=ctx) and not BLS.verify(params, pk, b"hellp", sig, ctx=ctx)
    with pytest.raises(BLSError) as e: BLS.verify(params, PublicKey(), b"hello", sig, ctx=ctx)
    assert e.value.kind == "InvalidPublicKey"
    # tests.rs:297-334 through the mirror, and the same fixtures as AggregateVerify over k copies of the message
    for c in eth["fast_aggregate_verify"]:
        i = c["input"]
        try: keys = [PublicKey.try_from(s, ctx) for s in i["pubkeys"]]
        except SerializationError: keys = None
        try: sg = Signature.try_from(i["signature"], ctx)
        except SerializationError: sg = Signature()
        res = keys is not None and BLS.fast_aggregate_verify(params, keys, hx(i["message"]), sg, ctx=ctx)
        assert res == c["output"], c["name"]
        if keys: assert BLS.aggregate_verify(params, keys, [hx(i["message"])] * len(keys), sg, ctx=ctx) == c["output"], c["name"]
    # uncompressed encodings round-trip through the value types
    assert PublicKey.try_from_uncompressed(pk.to_uncompressed(ctx), ctx) == pk and Signature.try_from_uncompressed(sig.to_uncompressed(ctx), ctx) == sig
    with pytest.raises(SerializationError): PublicKey.try_from_uncompressed(bytes([0x80]) + pk.to_uncompressed(ctx)[1:], ctx)

# ------------------------------------------------------------------------------------------ per-primitive device check
def test_device_primitives_match_host_emulation():
    """every primitive of the device library (tests/devcheck/ops.h), device vs host build of the same source: guards against
    compiler-level miscompilation of the carry chains (one was found in round 1: DESIGN.md, 'ptxas and carry chains')."""
    import sys, os
    from conftest import ROOT
    sys.path.insert(0, os.path.join(ROOT, "tests", "devcheck"))
    import run_devcheck
    for seed in (1, 2): assert run_devcheck.check(n=512, seed=seed) == []
    assert run_devcheck.check(n=512, seed=3, edge=True) == []       # 0, 1, p-1, (p+-1)/2 ...: the bounds of the lazy-reduction accumulators

# ------------------------------------------------------------------------------------------ boundary behaviour of the ABI
def test_empty_batch_and_multi_chunk_paths(ctx, C):
    """n = 0 is a no-op; a batch larger than the internal chunk (set to 64 here) takes the multi-pass path: statuses, bitmap
    words and the folded GT accumulator must equal the single-pass results, with ragged messages and in both pointer modes."""
    import torch
    from bls_verify_gadget_b200 import synth
    assert ctx.verify(b"", [], b"").size == 0 and ctx.hash_to_g2([]).size == 0
    rng = np.random.default_rng(33); n = 200
    sk = synth.secret_keys(n); msgs = [rng.bytes(int(l)) for l in rng.integers(0, 90, size=n)]
    pk, _ = ctx.sk_to_pk(sk); sig, _ = ctx.sign(sk, msgs)
    sig = sig.reshape(n, 96).copy(); sig[[3, 64, 130, 199]] = sig[[4, 65, 131, 0]]; sig = sig.reshape(-1)
    st0, bm0, gt0 = ctx.verify(pk, msgs, sig, want_bitmap=True, want_gt=True)
    ctx.set_chunk(64)
    try:
        st1, bm1, gt1 = ctx.verify(pk, msgs, sig, want_bitmap=True, want_gt=True)
        assert np.array_equal(st0, st1) and np.array_equal(bm0, bm1) and gt0.tobytes() == gt1.tobytes() and (st0 != 0).sum() == 4
        # device-pointer mode, fixed 32-byte messages, multi-chunk
        m32 = synth.messages(n); sig32, _ = ctx.sign(sk, m32, fixed32=True)
        ref = ctx.verify(pk, m32, sig32, fixed32=True)
        dev = torch.device("cuda", 0)
        d = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (pk, m32, sig32)]
        dst = torch.zeros(n, dtype=torch.uint8, device=dev); dbm = torch.zeros((n + 63) // 64, dtype=torch.int64, device=dev); dgt = torch.zeros(576, dtype=torch.uint8, device=dev)
        ctx.set_pointer_mode(True)
        ctx.verify_ptr(d[0].data_ptr(), d[1].data_ptr(), None, d[2].data_ptr(), n, dst.data_ptr(), dbm.data_ptr(), dgt.data_ptr()); ctx.synchronize()
        ctx.set_pointer_mode(False)
        assert np.array_equal(dst.cpu().numpy(), ref) and not ref.any()
        assert dgt.cpu().numpy().tobytes() == C.pairing_gt(b"", b"").tobytes()          # all valid: accumulator is one
        assert int(np.unpackbits(dbm.cpu().numpy().view(np.uint8), bitorder="little").sum()) == n
    finally:
        ctx.set_pointer_mode(False); ctx.set_chunk(1 << 20)

def test_resident_pool_committees(ctx, C):
    """cfg 3a: committees as indices into a pool decoded once == the same committees given as compressed keys == the oracle"""
    from bls_verify_gadget_b200 import synth
    nc, k, pool = 8, 96, 512
    pks, msg, sig, pool_pk, idx = synth.committees(ctx, nc, k=k, pool=pool)
    pool_pk = pool_pk.copy(); pool_pk[7, 20] ^= 0x40                            # one undecodable key in the pool
    pks = pool_pk[idx.reshape(-1)].reshape(-1).copy()
    h, codes = ctx.pool_create(pool_pk.reshape(-1)); assert codes[7] > 1 and (np.delete(codes, 7) == 0).all()
    rng = np.random.default_rng(8); bits = rng.random(nc * k) < 0.7
    bm = np.zeros((nc * k + 63) // 64, dtype=np.uint64)
    for j in np.nonzero(bits)[0]: bm[j // 64] |= np.uint64(1) << np.uint64(j % 64)
    for bitmap in (None, bm):
        st, agg = ctx.pool_fast_aggregate_verify(h, idx, k, msg, sig, bitmap=bitmap, want_agg=True)
        st2, agg2 = ctx.fast_aggregate_verify(pks, k, msg, sig, bitmap=bitmap, want_agg=True)
        ost, oagg = C.fast_aggregate_verify(pks, k, msg, sig, bitmap=bitmap, want_agg=True, threads=8)
        assert list(st) == list(st2) == list(ost)
        ok = st <= 1
        assert np.array_equal(agg.reshape(nc, 48)[ok], oagg.reshape(nc, 48)[ok]) and np.array_equal(agg2.reshape(nc, 48)[ok], oagg.reshape(nc, 48)[ok])
    uses7 = [(idx[c] == 7).any() for c in range(nc)]
    st = ctx.pool_fast_aggregate_verify(h, idx, k, msg, sig)
    assert all((s == 2) == u for s, u in zip(st, uses7)) and (st[~np.array(uses7)] == 0).all()
    ctx.pool_free(h)

def test_cooperative_final_exponentiation_matches(ctx, C):
    """six-lanes-per-item hard part (csrc/coop.cuh) == one-thread-per-item final exponentiation == oracle: statuses and GT bytes"""
    from bls_verify_gadget_b200 import synth
    n = 333                                                               # not a multiple of 5 (items per warp) nor 20 (items per CTA)
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=6, fast=False)
    msgs = [msg[32 * i:32 * i + 32].tobytes() for i in range(n)]
    ctx.set_coop(0); st0, gt0 = ctx.verify(pk, msgs, sig, want_gt=True)                     # n = 333 would take the six-lane form by default
    ctx.set_coop(True)
    try: st1, gt1 = ctx.verify(pk, msgs, sig, want_gt=True)
    finally: ctx.set_coop(2)
    ost, ogt = C.verify(pk, msgs, sig, want_gt=True, threads=8)
    assert list(st0) == list(st1) == list(ost) == list(exp) and gt0.tobytes() == gt1.tobytes() == ogt.tobytes()


def test_split_stage_kernels_match_one_launch_form(ctx, C):
    """blsgpu_set_split: the default sequence of short launches (hash_to_field | SSWU + isogeny | cofactor clearing; 8 x (line coefficients |
    accumulator update); easy part + 5 x (compressed squarings | decompression + products)) against the one-launch stage kernels and the
    oracle: statuses, ok-bitmap and GT bytes, on a batch with every corruption kind, the identity signature (its pair is skipped), ragged
    messages, and through the committee path that shares the verify core."""
    from bls_verify_gadget_b200 import synth
    n = 1500                                                              # not a multiple of the CTA size; 2n threads in the per-pair kernels
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=5, fast=False)
    sig = sig.copy(); sig[96 * 7:96 * 8] = 0; sig[96 * 7] = 0xc0          # item 7: identity signature -> decodes, verifies false
    msgs = [msg[32 * i:32 * i + 32].tobytes()[: 1 + (i * 7) % 32] for i in range(n)]      # ragged lengths 1..32
    sk = synth.secret_keys(n); pk2, st = ctx.sk_to_pk(sk); sig2, st = ctx.sign(sk, msgs)
    sig2 = sig2.copy(); sig2[96 * 7:96 * 8] = sig[96 * 7:96 * 8]; sig2[96 * 11 + 5] ^= 0x40
    out = {}
    for mode, coop in ((1, 0), (0, 0), (1, 2)):              # (1, 0): the short launches incl. k_final_squarings / k_final_step; (0, 0): one launch per stage; (1, 2): the defaults (six-lane final exponentiation at this size)
        ctx.set_split(mode); ctx.set_coop(coop)
        try:
            out[(mode, coop)] = (ctx.verify(pk, msg, sig, want_bitmap=True, want_gt=True, fixed32=True), ctx.verify(pk2, msgs, sig2, want_bitmap=True, want_gt=True))
        finally: ctx.set_split(1); ctx.set_coop(2)
    for other in ((0, 0), (1, 2)):
        for a, b in zip(out[(1, 0)], out[other]):
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2].tobytes() == b[2].tobytes()
    out = {1: out[(1, 0)]}
    exp = np.array(exp); exp[7] = 1
    assert list(out[1][0][0]) == list(exp)
    ost, ogt = C.verify(pk2, msgs, sig2, want_gt=True, threads=8)
    assert list(out[1][1][0]) == list(ost) and out[1][1][2].tobytes() == ogt.tobytes() and ost[7] == 1 and ost[11] != 0 and int(np.count_nonzero(ost)) == 2


def test_multi_gpu_abi_matches_single_gpu(ctx):
    """blsgpu_create_multi / blsgpu_multi_verify_batch (every visible device, NCCL all-gather + fold inside the library): status bytes,
    ok-bitmap and GT accumulator must equal the single-GPU call's for a batch with every corruption kind, on every device's copy;
    also a batch so small that some shards are empty, and ragged messages."""
    from bls_verify_gadget_b200 import synth
    from bls_verify_gadget_b200._lib import MultiContext
    n = 3000
    pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=16, fast=False)
    st1, bm1, gt1 = ctx.verify(pk, msg, sig, want_bitmap=True, want_gt=True, fixed32=True)
    assert list(st1) == list(exp)
    mc = MultiContext()
    assert mc.ndev >= 1 and mc.nccl_version >= 20000
    st, bm, gt = mc.verify(pk, msg, sig, fixed32=True)
    assert np.array_equal(st, st1) and np.array_equal(bm, bm1) and gt.tobytes() == gt1.tobytes()
    for i in range(mc.ndev):
        b, g = mc.peek(i, n); assert np.array_equal(b, bm1) and g.tobytes() == gt1.tobytes()
    msgs = [msg[32 * i:32 * i + 32].tobytes()[:1 + i % 32] for i in range(70)]
    a = ctx.verify(pk[:48 * 70], msgs, sig[:96 * 70], want_bitmap=True, want_gt=True); b = mc.verify(pk[:48 * 70], msgs, sig[:96 * 70])
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    a = ctx.verify(pk[:48 * 2], msg[:64], sig[:96 * 2], want_bitmap=True, want_gt=True, fixed32=True); b = mc.verify(pk[:48 * 2], msg[:64], sig[:96 * 2], fixed32=True)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    mc.close()
