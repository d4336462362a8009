"""The group law at its exceptional inputs, on the host build and on the device, and the multi-lane segment sums of every
aggregation entry point.

Part A feeds the curve additions of csrc/curve.cuh (tests/devcheck/ops.h ops 5-7, 18-20, 23, 28) on-curve points where the
formulas need their exceptional branches -- P + P, P + (-P), the identity on either side -- in Jacobian form with chosen Z.
Each output is normalised to affine (Jacobian limbs are not unique) and compared with the big-integer reference oracle/pyref.py:
the host build on the CPU, the device build on the GPU, which must also equal the host build limb for limb.

Part B drives k_segsum (csrc/blsgpu.cu) through g1_aggregate, g2_aggregate, fast_aggregate_verify and the resident-pool path at
segment lengths that select every lane count L = 1 .. 32, with segments crafted to take each exceptional branch in the lane folds
and in the shared-memory tree.  segsum_model restates the kernel's schedule on scalars and shows, without a GPU, that every crafted
segment takes the branch it claims; the GPU tests compare statuses and aggregate bytes with the C oracle and with the model's sums."""
import ctypes, os, sys
import numpy as np
import pytest
from conftest import ROOT
from oracle import pyref as PR

P = PR.p
R = PR.r
RMONT = 1 << 384
RMONT_INV = pow(RMONT, -1, P)

# ============================================================================================== A: one addition at a time
def _img(v): return (v % P) * RMONT % P                      # Montgomery image, the form the limbs hold
def _enc(vals): return np.frombuffer(b"".join(_img(v).to_bytes(48, "little") for v in vals), np.uint8).copy()
def _dec(out):
    limbs = [int.from_bytes(out[48 * i:48 * i + 48].tobytes(), "little") for i in range(out.size // 48)]
    assert all(x < P for x in limbs), "output limbs are not canonical"
    return [x * RMONT_INV % P for x in limbs]

# G1 in Jacobian form with a chosen Z; the identity is any (X, Y, 0)
def _j1(pt, z): return [pt[0] * z * z % P, pt[1] * z * z * z % P, z] if pt is not None else [z * z % P, z * z * z % P, 0]
def _aff1(X, Y, Z):
    if Z == 0: return None
    zi = pow(Z, -1, P); return (X * zi * zi % P, Y * zi * zi * zi % P)
def _j2(pt, z):
    z2 = PR.sqr(z); z3 = PR.mul(z2, z)
    if pt is None: return [*z2, *z3, 0, 0]
    return [*PR.mul(pt[0], z2), *PR.mul(pt[1], z3), *z]
def _aff2(v):
    X, Y, Z = (v[0], v[1]), (v[2], v[3]), (v[4], v[5])
    if Z == PR.ZERO: return None
    zi = PR.inv(Z); zi2 = PR.sqr(zi); return (PR.mul(X, zi2), PR.mul(Y, PR.mul(zi2, zi)))

def _edge_cases():
    """{op: [(name, input values, expected affine point or None)]} for ops 18-20 (G1) and 5-7, 23, 28 (G2)"""
    rng = np.random.default_rng(2024)
    rnd = lambda: int.from_bytes(rng.bytes(48), "little") % P
    cases = {op: [] for op in (18, 19, 20, 5, 6, 7, 28, 23)}
    # ---- G1: y^2 = x^3 + 4
    A, B = PR.g1mul(3, PR.G1), PR.g1mul(5, PR.G1); nA = PR.g1neg(A)
    A2, AB = PR.g1add(A, A), PR.g1add(A, B)
    zs = [1, rnd(), P - 1]
    for i, z1 in enumerate(zs):
        for j, z2 in enumerate(zs):
            tag = "same Z" if i == j else "different Z"
            cases[20] += [(f"P+P {tag}", _j1(A, z1) + _j1(A, z2), A2), (f"P+(-P) {tag}", _j1(A, z1) + _j1(nA, z2), None),
                          (f"P+Q {tag}", _j1(A, z1) + _j1(B, z2), AB)]
        cases[20] += [("O+P", _j1(None, z1) + _j1(A, zs[1]), A), ("P+O", _j1(A, z1) + _j1(None, zs[1]), A), ("O+O", _j1(None, z1) + _j1(None, zs[2]), None),
                      ("O(1,1,0)+P", [1, 1, 0] + _j1(A, z1), A), ("P+O(1,1,0)", _j1(A, z1) + [1, 1, 0], A)]
        cases[19] += [("acc=q", _j1(A, z1) + list(A), A2), ("acc=-q", _j1(nA, z1) + list(A), None), ("acc=O", _j1(None, z1) + list(A), A),
                      ("acc=O(1,1,0)", [1, 1, 0] + list(A), A), ("generic", _j1(B, z1) + list(A), AB)]
        cases[18] += [("2P", _j1(A, z1), A2), ("2O", _j1(None, z1), None)]
    cases[18].append(("2O(1,1,0)", [1, 1, 0], None))
    # ---- G2: y^2 = x^3 + 4(1 + u)
    A, B = PR.smul(3, PR.G2), PR.smul(7, PR.G2); nA = PR.pneg(A)
    A2, AB = PR.padd(A, A), PR.padd(A, B)
    one2 = [1, 0, 1, 0, 0, 0]
    zs = [(1, 0), (rnd(), rnd()), (P - 1, 0), (rnd(), 0), (0, rnd())]          # Z = 1, random, -1, Z with c1 = 0, Z with c0 = 0
    for i, z1 in enumerate(zs):
        for j, z2 in enumerate(zs[:3]):
            tag = "same Z" if i == j else "different Z"
            cases[7] += [(f"P+P {tag}", _j2(A, z1) + _j2(A, z2), A2), (f"P+(-P) {tag}", _j2(A, z1) + _j2(nA, z2), None),
                         (f"P+Q {tag}", _j2(A, z1) + _j2(B, z2), AB)]
        cases[7] += [("O+P", _j2(None, z1) + _j2(A, zs[1]), A), ("P+O", _j2(A, z1) + _j2(None, zs[1]), A), ("O+O", _j2(None, z1) + _j2(None, zs[2]), None),
                     ("O(1,1,0)+P", one2 + _j2(A, z1), A), ("P+O(1,1,0)", _j2(A, z1) + one2, A)]
        qa = [*A[0], *A[1]]
        for op in (6, 28):
            cases[op] += [("acc=q", _j2(A, z1) + qa, A2), ("acc=-q", _j2(nA, z1) + qa, None), ("acc=O", _j2(None, z1) + qa, A),
                          ("acc=O(1,1,0)", one2 + qa, A), ("generic", _j2(B, z1) + qa, AB)]
        cases[5] += [("2P", _j2(A, z1), A2), ("2O", _j2(None, z1), None)]
    cases[5].append(("2O(1,1,0)", one2, None))
    for k in (1, 2, 3, 11):                                                    # [|x|] Q on G2 points (the decoder's subgroup ladder)
        Q = PR.smul(k, PR.G2); cases[23].append((f"[|x|][{k}]G2", [*Q[0], *Q[1]], PR.smul(PR.X, Q)))
    return cases

@pytest.fixture(scope="module")
def edge_cases(): return _edge_cases()

@pytest.fixture(scope="module")
def E():
    from hostemu import emu
    emu.build(); return emu

def _check_against_pyref(op, cases, out):
    n_out = 3 if op in (18, 19, 20) else 6
    vals = _dec(out)
    bad = []
    for c, (name, _, want) in enumerate(cases):
        v = vals[n_out * c:n_out * (c + 1)]
        got = _aff1(*v) if n_out == 3 else _aff2(v)
        if got != want: bad.append(name)
    return bad

def test_host_additions_at_exceptional_inputs_match_pyref(E, edge_cases):
    """host build of csrc/curve.cuh: every exceptional input of every addition / doubling op gives the reference's affine point"""
    for op, cases in edge_cases.items():
        out = E.run_op(op, np.concatenate([_enc(v) for _, v, _ in cases]))
        assert _check_against_pyref(op, cases, out) == [], f"op {op}"

@pytest.mark.gpu
def test_device_additions_at_exceptional_inputs_match_pyref_and_host(E, edge_cases):
    """the same inputs through the device build (one kernel per op, tests/devcheck): the reference's affine points, and the host
    build's limbs exactly"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "devcheck"))
    import run_devcheck
    D = run_devcheck.dev_lib()
    for op, cases in edge_cases.items():
        x = np.concatenate([_enc(v) for _, v, _ in cases]); n_in, n_out = E.op_shape(op)
        got = np.zeros(48 * n_out * len(cases), np.uint8)
        rc = D.dev_run_op(int(op), x.ctypes.data_as(ctypes.c_void_p), got.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(len(cases)))
        assert rc == 0, f"op {op}: rc={rc}"
        assert _check_against_pyref(op, cases, got) == [], f"op {op}"
        want = E.run_op(op, x)
        diff = [cases[c][0] for c in range(len(cases)) if not np.array_equal(got[48 * n_out * c:48 * n_out * (c + 1)], want[48 * n_out * c:48 * n_out * (c + 1)])]
        assert diff == [], f"op {op}: device limbs differ from the host build"

# ============================================================================================== B: k_segsum
ST_OK, ST_BAD_PK, ST_BAD_SIG, ST_EMPTY = 0, 2, 3, 4

def seg_lanes(avg_len):
    """csrc/blsgpu.cu seg_lanes: the largest power of two <= 32 that leaves >= 64 points per lane"""
    L = 32
    while L > 1 and avg_len // L < 64: L >>= 1
    return L

def segsum_model(scal, mask, L):
    """k_segsum (csrc/blsgpu.cu:459-514) for one segment, on scalars: member j is [scal[j]] B for a fixed generator B (0 = an
    identity encoding, None = a member that does not decode or an index outside the pool); mask[j] False = bit j of the
    participation bitmap is clear.  Mirrors the kernel's schedule: lane sl folds members sl, sl + L, ... with jac_add_mixed, then
    the tree adds lane sl + w into lane sl for w = L/2, ..., 1 with jac_add, OR-ing `bad` and adding `cnt` alongside.  In a
    prime-order group a Jacobian value is the identity (Z = 0) exactly when its scalar is 0, so the branch each addition takes
    follows from the scalars.  Returns (sum, bad, cnt, events, lanes whose fold saw a bad member)."""
    k = len(scal); acc = [0] * L; bad = [0] * L; cnt = [0] * L; used = [False] * L; ev = set()
    for sl in range(L):
        for j in range(sl, k, L):
            if mask is not None and not mask[j]: continue
            cnt[sl] += 1
            s = scal[j]
            if s is None: bad[sl] = 1; continue
            if s == 0: continue
            a = acc[sl]; used[sl] = True
            if a == 0: ev.add("mixed_onto_identity")                        # if (f_is_zero(p.Z)) -> q
            elif a == s: ev.add("mixed_double")                             # h_zero, r_zero
            elif (a + s) % R == 0: ev.add("mixed_cancel")                   # h_zero, !r_zero
            acc[sl] = (a + s) % R
        if not used[sl]: ev.add("empty_lane")
    bad_lanes = {sl for sl in range(L) if bad[sl]}
    w = L >> 1
    while w >= 1:
        for sl in range(w):
            a, o = acc[sl], acc[sl + w]
            if a == 0: ev.add(("tree_left_identity", w))
            elif o == 0: ev.add(("tree_right_identity", w))
            elif a == o: ev.add(("tree_double", w))
            elif (a + o) % R == 0: ev.add(("tree_cancel", w))
            acc[sl] = (a + o) % R; bad[sl] |= bad[sl + w]; cnt[sl] += cnt[sl + w]
        w >>= 1
    return acc[0], bad[0], cnt[0], ev, bad_lanes

# Members are indices into a table of points with known scalars: T[i] = [sk_i] B and T[M + i] = -T[i] for i < M (the negation flips
# the sign bit of the compressed encoding), then an identity encoding and an undecodable one.  OOR is an index past the end of the
# table: the resident-pool path rejects it, the byte paths see the undecodable entry instead.
M = 4096
IDENT, BAD = 2 * M, 2 * M + 1
NTAB = 2 * M + 2
OOR = NTAB + 1000

def _neg(i): return i + M if i < M else i - M

_SCAL = []
def table_scalars():
    """sk_i of synth.secret_keys(M), then their negations, 0 for the identity, None for the undecodable entry"""
    if not _SCAL:
        from bls_verify_gadget_b200 import synth
        b = synth.secret_keys(M); sk = [int.from_bytes(b[32 * i:32 * i + 32].tobytes(), "little") for i in range(M)]
        _SCAL.extend(sk + [(R - s) % R for s in sk] + [0, None])
    return _SCAL

def _last_in_lane(k, L, lane):
    return max(j for j in range(k) if j % L == lane)

# The crafted segments.  Every one starts from k distinct random keys.
#   generic             distinct keys (the control)
#   repeat              one key k times: the second member of every lane doubles (mixed), equal lane sums double in the tree
#   lane_cancel         lane 0 opens with K, -K: the running sum cancels, the third member lands on the identity
#   tree_cancel_top     lane L/2 holds the negations of lane 0's members: the first tree level cancels
#   tree_cancel_bottom  odd lanes negate the even lane before them: the last level (w = 1) cancels; L = 1: inside the lane
#   all_cancel          the second half negates the first: every lane, and the segment, sums to the identity
#   ident_lane          every member of the last lane is an identity encoding: an empty lane enters the tree
#   masked_lane         every member of the last lane is masked by the bitmap: an empty lane enters the tree (no bitmap: generic)
#   bad_last_lane       one undecodable member, in the last lane only: the bad flag has to survive every tree level
#   oor_last_lane       as bad_last_lane with an index outside the resident pool (the byte paths see an undecodable key)
#   small_set           a validator set of 48 keys, members drawn with replacement (sync committees of a small network)
def build_segment(name, k, L, rng):
    """(members, mask) of one crafted segment of length k for lane count L; mask None = no bitmap"""
    m = [int(x) for x in rng.choice(M, size=k, replace=False)]
    mask = None
    if name == "repeat": m = [m[0]] * k
    elif name == "lane_cancel": m[L] = _neg(m[0])
    elif name == "tree_cancel_top":
        w = L >> 1
        if w:
            for j in range(w, k, L): m[j] = _neg(m[j - w])
    elif name == "tree_cancel_bottom":
        for j in range(1, k, 2): m[j] = _neg(m[j - 1])
    elif name == "all_cancel":
        h = k // 2; m[h:2 * h] = [_neg(x) for x in m[:h]]
    elif name == "ident_lane":
        for j in range(L - 1, k, L): m[j] = IDENT
    elif name == "masked_lane": mask = [j % L != L - 1 for j in range(k)]
    elif name == "bad_last_lane": m[_last_in_lane(k, L, L - 1)] = BAD
    elif name == "oor_last_lane": m[_last_in_lane(k, L, L - 1)] = OOR
    elif name == "small_set":
        keys = rng.choice(M, size=48, replace=False); m = [int(keys[i]) for i in rng.integers(0, 48, size=k)]
    else: assert name == "generic"
    return m, mask

def claims(name, L):
    """(events the segment must take, whether its sum must be the identity, lanes that must see the bad member) for a segment
    of length >= 64 L"""
    tree = L >= 2
    lv = [L >> s for s in range(1, L.bit_length())]                             # the tree levels w = L/2, ..., 1
    if name == "repeat": return {"mixed_onto_identity", "mixed_double"} | {("tree_double", w) for w in lv}, False, set()
    if name == "lane_cancel": return {"mixed_cancel", "mixed_onto_identity"}, False, set()
    if name == "tree_cancel_top":                                                # L = 2: the first level is the last, the segment cancels
        return ({("tree_cancel", L >> 1)} | ({("tree_left_identity", L >> 2)} if L >= 4 else set())) if tree else set(), L == 2, set()
    if name == "tree_cancel_bottom": return {("tree_cancel", 1)} if tree else {"mixed_cancel"}, True, set()
    if name == "all_cancel": return {"mixed_cancel"} | {("tree_left_identity", w) for w in lv}, True, set()
    if name == "ident_lane": return {"empty_lane"} | ({("tree_right_identity", L >> 1)} if tree else set()), not tree, set()
    if name == "masked_lane": return {"empty_lane"} | ({("tree_right_identity", L >> 1)} if tree else set()), False, set()
    if name in ("bad_last_lane", "oor_last_lane"): return set(), False, {L - 1}
    return set(), False, set()

LENGTHS = (64, 128, 256, 512, 1024, 2048)

def committee_layout(k, names, seed):
    """committees of k members for the patterns `names`: (L, [(name, members, mask)])"""
    L = seg_lanes(k); rng = np.random.default_rng(seed)
    return L, [(n, *build_segment(n, k, L, rng)) for n in names]

FAV_NAMES = ("generic", "repeat", "lane_cancel", "tree_cancel_top", "tree_cancel_bottom", "all_cancel", "ident_lane", "masked_lane",
             "bad_last_lane", "oor_last_lane", "small_set")
G2_NAMES = ("generic", "repeat", "lane_cancel", "tree_cancel_top", "tree_cancel_bottom", "all_cancel", "ident_lane", "bad_last_lane")

# ragged g1_aggregate / g2_aggregate calls: a few long segments set L (from the average length), the short ones -- one member,
# none, fewer members than lanes -- leave lanes empty; the 17-member repeat doubles in the tree's first level
RAGGED_G1 = ((4096, "repeat"), (4096, "tree_cancel_top"), (4096, "all_cancel"), (4096, "bad_last_lane"), (1, "generic"), (0, "generic"),
             (17, "repeat"), (31, "bad_last_lane"), (4096, "ident_lane"))
RAGGED_G2 = ((2048, "repeat"), (2048, "tree_cancel_bottom"), (2048, "lane_cancel"), (2048, "bad_last_lane"), (1, "generic"), (0, "generic"),
             (9, "repeat"), (15, "bad_last_lane"))

def ragged_layout(spec, seed):
    L = seg_lanes(sum(k for k, _ in spec) // len(spec)); rng = np.random.default_rng(seed); segs = []
    for k, name in spec:
        if k == 0: segs.append((name, [], None))
        elif k < 2 * L:                                                      # too short for the lane patterns: keep its shape only
            m = [int(x) for x in rng.choice(M, size=k, replace=False)]
            if name == "repeat": m = [m[0]] * k
            if name == "bad_last_lane": m[-1] = BAD
            segs.append((name, m, None))
        else: segs.append((name, *build_segment(name, k, L, rng)))
    return L, segs

def _model(members, mask, L, use_mask=True):
    sc = table_scalars()
    return segsum_model([sc[i] if i < NTAB else None for i in members], mask if use_mask else None, L)

def test_seg_lanes_matches_the_kernel_thresholds():
    assert [seg_lanes(n) for n in (0, 1, 64, 127, 128, 255, 256, 511, 512, 1023, 1024, 2047, 2048, 1 << 20)] == [1, 1, 1, 1, 2, 2, 4, 4, 8, 8, 16, 16, 32, 32]
    assert [seg_lanes(k) for k in LENGTHS] == [1, 2, 4, 8, 16, 32]
    assert ragged_layout(RAGGED_G1, 0)[0] == 32 and ragged_layout(RAGGED_G2, 0)[0] == 16

@pytest.mark.parametrize("k", LENGTHS)
def test_crafted_committees_take_their_claimed_branches(k):
    """the schedule model: every crafted committee takes the branches it is built for, at every L, with and without its bitmap,
    and the model's tree sums equal the plain sum of the members"""
    sc = table_scalars()
    L, segs = committee_layout(k, FAV_NAMES, seed=k)
    for name, m, mask in segs:
        for use_mask in (False, True):
            if use_mask and mask is None: continue
            s, bad, cnt, ev, bad_lanes = _model(m, mask, L, use_mask)
            want_ev, want_identity, want_bad = claims(name if use_mask or name != "masked_lane" else "generic", L)
            assert want_ev <= ev, (name, L, use_mask, want_ev - ev)
            assert bad_lanes == want_bad, (name, L)
            live = [j for j in range(k) if not (use_mask and not mask[j])]
            if not bad:
                assert s == sum(sc[m[j]] for j in live) % R and cnt == len(live)
                assert (s == 0) == (want_identity or (use_mask and L == 1)), (name, L)
    # the small validator set repeats keys: some lane of some committee opens with the same key twice
    L, segs = committee_layout(512, ("small_set",) * 4, seed=48)
    assert any("mixed_double" in _model(m, None, L)[3] for _, m, _ in segs)

def test_ragged_layouts_take_their_claimed_branches():
    for spec, seed in ((RAGGED_G1, 1), (RAGGED_G2, 2)):
        L, segs = ragged_layout(spec, seed)
        for (k, name), (_, m, mask) in zip(spec, segs):
            s, bad, cnt, ev, bad_lanes = _model(m, mask, L)
            if k >= 2 * L:
                want_ev, want_identity, want_bad = claims(name, L)
                assert want_ev <= ev and bad_lanes == want_bad and (bad or (s == 0) == want_identity), (name, k)
            elif name == "repeat": assert ("tree_double", L >> 1) in ev and "empty_lane" in ev, k
            elif name == "bad_last_lane": assert bad_lanes == {(k - 1) % L} and (k - 1) % L > 0
            elif k == 0: assert cnt == 0

def test_oracle_identity_and_doubling_agree_with_pyref():
    """the reference behaviour the GPU tests rely on: K + K and K + (-K) through the C oracle equal pyref's affine group law; an
    identity aggregate encodes as 0xc0 00..; fast_aggregate_verify reports an identity aggregate key as InvalidPublicKey (status 2,
    src/bls.rs:434), also when the signature is the identity"""
    from oracle import cwrap as C
    from bls_verify_gadget_b200 import synth
    sk = synth.secret_keys(2); pk = C.sk_to_pk(sk).reshape(2, 48)
    K = pk[0].copy(); nK = K.copy(); nK[0] ^= 0x20
    A = PR.deser_g1(K.tobytes(), subgroup=False); B = PR.deser_g1(pk[1].tobytes(), subgroup=False)
    assert PR.deser_g1(nK.tobytes(), subgroup=False) == PR.g1neg(A)
    ident48 = bytes([0xc0]) + bytes(47); ident96 = bytes([0xc0]) + bytes(95)
    out, st = C.g1_aggregate(np.concatenate([K, K, K, nK, pk[1], K, nK]), [0, 2, 4, 7])
    assert list(st) == [0, 0, 0]
    assert out[:48].tobytes() == PR.ser_g1(PR.g1add(A, A)) and out[48:96].tobytes() == ident48 and out[96:].tobytes() == PR.ser_g1(B)
    msg = bytes(32); sig = C.sign(sk[:32], [msg])[0]
    S = PR.deser_g2(sig.tobytes(), subgroup=False); nsig = sig.copy(); nsig[0] ^= 0x20
    out, st = C.g2_aggregate(np.concatenate([sig, sig, sig, nsig]), [0, 2, 4])
    assert list(st) == [0, 0] and out[:96].tobytes() == PR.ser_g2(PR.padd(S, S)) and out[96:].tobytes() == ident96
    st, agg = C.fast_aggregate_verify(np.concatenate([K, nK]), 2, msg, np.frombuffer(ident96, np.uint8), want_agg=True)
    assert st[0] == ST_BAD_PK and agg.tobytes() == ident48
    st = C.fast_aggregate_verify(np.concatenate([K, nK]), 2, msg, sig)
    assert st[0] == ST_BAD_PK

# ---------------------------------------------------------------------------------------------- B on the GPU
@pytest.fixture(scope="module")
def ctx():
    from bls_verify_gadget_b200 import Context
    c = Context(0); yield c; c.close()

@pytest.fixture(scope="module")
def C():
    from oracle import cwrap
    return cwrap

MSG_G2 = b"group law edges: the message every G2 table point signs"

@pytest.fixture(scope="module")
def tables(ctx):
    """compressed G1 and G2 tables: [sk_i] G1 and [sk_i] H(MSG_G2), their negations, the identity, an undecodable entry"""
    from bls_verify_gadget_b200 import synth
    sk = synth.secret_keys(M)
    pk, st = ctx.sk_to_pk(sk); assert not st.any()
    sg, st = ctx.sign(sk, [MSG_G2] * M); assert not st.any()
    out = []
    for pts, size in ((pk, 48), (sg, 96)):
        t = np.zeros((NTAB, size), np.uint8); t[:M] = pts.reshape(M, size); t[M:2 * M] = t[:M]; t[M:2 * M, 0] ^= 0x20
        t[IDENT, 0] = 0xc0
        t[BAD] = t[0]; t[BAD, 0] &= 0x7f                                     # compression flag cleared: does not decode
        out.append(t)
    return out

def _g1_bytes(C, s): return bytes([0xc0]) + bytes(47) if s == 0 else C.sk_to_pk(np.frombuffer(s.to_bytes(32, "little"), np.uint8)).tobytes()
def _g2_bytes(C, s): return bytes([0xc0]) + bytes(95) if s == 0 else C.sign(np.frombuffer(s.to_bytes(32, "little"), np.uint8), [MSG_G2])[0].tobytes()

def _rows(table, members): return table[[i if i < NTAB else BAD for i in members]]

def _check_aggregate(ctx, C, table, L, segs, g2):
    """g1_aggregate / g2_aggregate of the segments: statuses and bytes equal the oracle's and the model's sums"""
    size = 96 if g2 else 48
    pts = np.concatenate([_rows(table, m) for _, m, _ in segs if m] or [np.zeros((0, size), np.uint8)]).reshape(-1)
    off = np.concatenate([[0], np.cumsum([len(m) for _, m, _ in segs])]).astype(np.uint32)
    assert seg_lanes(int(off[-1]) // len(segs)) == L
    got, gst = (ctx.g2_aggregate if g2 else ctx.g1_aggregate)(pts, off)
    want, wst = (C.g2_aggregate if g2 else C.g1_aggregate)(pts, off, threads=C.hw_threads())
    bad_code = ST_BAD_SIG if g2 else ST_BAD_PK
    for c, (name, m, _) in enumerate(segs):
        s, bad, cnt, _, _ = _model(m, None, L)
        st = bad_code if bad else (ST_EMPTY if cnt == 0 else ST_OK)
        assert gst[c] == wst[c] == st, (name, len(m), L, gst[c], wst[c], st)
        if st == ST_OK:
            g, w = got[size * c:size * (c + 1)].tobytes(), want[size * c:size * (c + 1)].tobytes()
            assert g == w == (_g2_bytes if g2 else _g1_bytes)(C, s), (name, len(m), L)

@pytest.mark.gpu
@pytest.mark.parametrize("k", LENGTHS)
def test_g1_g2_aggregate_every_lane_count(ctx, C, tables, k):
    """one g1_aggregate and one g2_aggregate call per segment length, the crafted segments side by side (8 to 11 segments: the last
    warp / CTA is partly filled at every L)"""
    L, segs = committee_layout(k, FAV_NAMES, seed=k)
    _check_aggregate(ctx, C, tables[0], L, segs, g2=False)
    L, segs = committee_layout(k, G2_NAMES, seed=1000 + k)
    _check_aggregate(ctx, C, tables[1], L, segs, g2=True)

@pytest.mark.gpu
def test_g1_g2_aggregate_ragged(ctx, C, tables):
    for spec, seed, g2 in ((RAGGED_G1, 1, False), (RAGGED_G2, 2, True)):
        L, segs = ragged_layout(spec, seed)
        _check_aggregate(ctx, C, tables[int(g2)], L, segs, g2)

def _bitmap(segs, k):
    bits = np.concatenate([np.array(mask if mask is not None else [True] * k, bool) for _, _, mask in segs])
    bm = np.zeros((bits.size + 63) // 64, np.uint64)
    for j in np.nonzero(bits)[0]: bm[j // 64] |= np.uint64(1) << np.uint64(j % 64)
    return bm

@pytest.mark.gpu
@pytest.mark.parametrize("k", LENGTHS)
def test_fast_aggregate_verify_and_pool_every_lane_count(ctx, C, tables, k):
    """fast_aggregate_verify (bytes) and pool_fast_aggregate_verify (indices into a resident pool holding the same table) on the
    crafted committees, without and with a participation bitmap: statuses and aggregate keys equal the oracle's, the signatures are
    [sum of the members' keys] H(m) (the identity where that sum is 0), and the pool path agrees with the byte path"""
    T = tables[0]
    L, segs = committee_layout(k, FAV_NAMES, seed=k)
    nc = len(segs); idx = np.array([m for _, m, _ in segs], np.uint32)
    pks = _rows(T, idx.reshape(-1).tolist()).reshape(-1)
    msg = np.frombuffer(b"".join(bytes([k % 251, c]) * 16 for c in range(nc)), np.uint8).copy()
    h, codes = ctx.pool_create(T.reshape(-1))
    assert codes[IDENT] == 1 and codes[BAD] > 1 and not codes[:2 * M].any()
    try:
        for use_mask in (False, True):
            bm = _bitmap(segs, k) if use_mask else None
            sums, want_st = [], []
            for name, m, mask in segs:
                s, bad, cnt, _, _ = _model(m, mask, L, use_mask)
                sums.append(s); want_st.append(ST_BAD_PK if (bad or cnt == 0 or s == 0) else ST_OK)
            sig = np.zeros((nc, 96), np.uint8); sig[:, 0] = 0xc0
            live = [c for c in range(nc) if sums[c]]
            sk = np.frombuffer(b"".join(sums[c].to_bytes(32, "little") for c in live), np.uint8)
            s_live, st = ctx.sign(sk, msg.reshape(nc, 32)[live].reshape(-1), fixed32=True); assert not st.any()
            sig[live] = s_live.reshape(-1, 96)
            st, agg = ctx.fast_aggregate_verify(pks, k, msg, sig, bitmap=bm, want_agg=True)
            pst, pagg = ctx.pool_fast_aggregate_verify(h, idx, k, msg, sig, bitmap=bm, want_agg=True)
            ost, oagg = C.fast_aggregate_verify(pks, k, msg, sig, bitmap=bm, want_agg=True, threads=C.hw_threads())
            names = [n for n, _, _ in segs]
            assert list(st) == list(pst) == list(ost) == want_st, (L, use_mask, names)
            for c, (name, m, mask) in enumerate(segs):
                s, bad, cnt, _, _ = _model(m, mask, L, use_mask)
                if bad or cnt == 0: continue
                a, pa, oa = (x[48 * c:48 * (c + 1)].tobytes() for x in (agg, pagg, oagg))
                assert a == pa == oa == _g1_bytes(C, s), (name, L, use_mask)
    finally:
        ctx.pool_free(h)
