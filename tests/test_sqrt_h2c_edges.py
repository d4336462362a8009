"""The square roots, the sign rules and the hash-to-curve maps at the inputs that take their data-dependent branches, on the host
build and on the device, against the big-integer reference oracle/pyref.py.

Random inputs never reach these branches: the `d = 0` fallback of fp2_sqrt_with_norm_root (a.c1 = 0 with a.c0 a non-residue of
Fp), sgn0's tie-break (c0 = 0), lex_largest's fall-back to c0 (c1 = 0), SSWU's exceptional case (u = 0 is the only u with
u^2 = -1/Z or 0), the isogeny's kernel (x = -k1/2 is a double root of K2 and a root of K4), and the exceptional additions that
points of small order drive g2_clear_cofactor through.  Part A feeds the single-primitive ops of tests/devcheck/ops.h (16, 25,
42-46) those inputs as Montgomery images; the device build must give the reference's values and the host build's limbs exactly.
Part B builds G2 encodings whose y^2 lies in Fp or in i Fp -- untrusted bytes that reach the fallback through g2_decode -- and runs
them through the decoders, g2_uncompress and the verify batch in each of its modes."""
import ctypes, os, sys
import numpy as np
import pytest
from conftest import ROOT
from oracle import pyref as PR
from test_group_law_edges import _enc, _j2
from test_sig_subgroup_in_miller import curve_points, torsion_points

P = PR.p
RMONT_INV = pow(1 << 384, -1, P)
HALF = (P - 1) // 2

def _legendre(a): return pow(a % P, HALF, P)                # 0, 1, or p - 1
def _rows(out, n_out):
    """raw limb integers of each output item; every field element the library writes is canonical"""
    limbs = [int.from_bytes(out[48 * i:48 * i + 48].tobytes(), "little") for i in range(out.size // 48)]
    assert all(x < P for x in limbs), "output limbs are not canonical"
    return [limbs[n_out * c:n_out * (c + 1)] for c in range(len(limbs) // n_out)]
def _v(x): return x * RMONT_INV % P                         # Montgomery image -> value
def _f2(row, i): return (_v(row[i]), _v(row[i + 1]))
def _flag(x):
    assert x in (0, 1), x
    return x

def _jac_aff(row):
    """affine point of a Jacobian output (X, Y, Z), None for the identity, or "bad identity" when Z = 0 but (X, Y) is not of the form
    (l^2, l^3) with l != 0 -- the identity as jac_set_identity and the doubling formula write it; (0, 0, 0) is no projective point"""
    X, Y, Z = _f2(row, 0), _f2(row, 2), _f2(row, 4)
    if Z == PR.ZERO:
        return None if X != PR.ZERO and PR.mul(PR.sqr(X), X) == PR.sqr(Y) else "bad identity"
    zi = PR.inv(Z); zi2 = PR.sqr(zi)
    return PR.mul(X, zi2), PR.mul(Y, PR.mul(zi2, zi))

# ============================================================================================== A: the primitives
def _fp_edges(rng):
    """(residues, non-residues) of Fp: fixed small values and random ones"""
    rnd = lambda: int.from_bytes(rng.bytes(48), "little") % P
    res, non = [], []
    for a in [1, 2, 3, 4, 5, P - 1, P - 2, HALF, HALF + 1] + [rnd() for _ in range(40)]:
        (res if _legendre(a) == 1 else non).append(a)
    return res, non

def _cases():
    """{op: [(name, input values)]}; op 42 is followed by op 43 on its own output"""
    rng = np.random.default_rng(9380)
    rnd = lambda: int.from_bytes(rng.bytes(48), "little") % P
    res, non = _fp_edges(rng)
    assert len(res) >= 8 and len(non) >= 8 and 2 in non and P - 1 in non
    fixed = [1, 2, 3, 4, 5, P - 1, P - 2, HALF, HALF + 1]
    c = {}
    # ---- fp2_sqrt: a.c1 = 0 takes d = 0 when a.c0 is a non-residue (the norm's root is then -a.c0)
    sq = [("(0, 0)", (0, 0))] + [(f"({a}, 0)", (a, 0)) for a in fixed]
    sq += [("(residue, 0)", (a, 0)) for a in res[-4:]] + [("(non-residue, 0)", (a, 0)) for a in non[-4:]]
    sq += [(f"(0, {a})", (0, a)) for a in (1, 2, P - 1, rnd(), rnd())]
    nn = []
    while len(nn) < 4:                                                         # norm a non-residue: a is not a square
        a = (rnd(), rnd())
        if _legendre(a[0] ** 2 + a[1] ** 2) == P - 1: nn.append(("norm non-residue", a))
    sq += nn + [("random", (rnd(), rnd())) for _ in range(6)] + [("square", PR.sqr((rnd(), rnd()))) for _ in range(4)]
    sq += [("square of (x, 0)", PR.sqr((a, 0))) for a in non[-2:]] + [("square of (0, x)", PR.sqr((0, a))) for a in res[-2:]]
    c[16] = [(n, list(a)) for n, a in sq]
    # ---- fp2_sqrt_ratio(u, v): u = 0; u, v in Fp; u, v in i Fp; v = +-1; square and non-square ratios
    sr = [("u=0 v=1", (0, 0), (1, 0)), ("u=0 v=random", (0, 0), (rnd(), rnd()))]
    sr += [("u, v in Fp", (rnd(), 0), (rnd(), 0)) for _ in range(4)] + [("u, v in Fp, u/v non-residue", (a, 0), (1, 0)) for a in non[-2:]]
    sr += [("u, v in Fp, u/v = -1", (P - 1, 0), (1, 0)), ("u, v in Fp, u/v = 2", (4, 0), (2, 0))]
    sr += [("u, v in i Fp", (0, rnd()), (0, rnd())) for _ in range(4)] + [("u in Fp, v in i Fp", (rnd(), 0), (0, rnd())) for _ in range(2)]
    sr += [("v=1", (rnd(), rnd()), (1, 0)) for _ in range(2)] + [("v=-1", (rnd(), rnd()), (P - 1, 0)) for _ in range(2)]
    for _ in range(4):
        w, v = (rnd(), rnd()), (rnd(), rnd())
        sr += [("square ratio", PR.mul(PR.sqr(w), v), v), ("non-square ratio", PR.mul(PR.mul(PR.Z_SSWU, PR.sqr(w)), v), v)]
    c[25] = [(n, [*u, *v]) for n, u, v in sr]
    # ---- sswu_map: u = 0 is SSWU's exceptional case; c0 = 0 makes sgn0(u) the tie-break on c1
    odd = lambda: rnd() | 1
    even = lambda: rnd() & ~1
    us = [("u=0", (0, 0)), ("u=1", (1, 0)), ("u=-1", (P - 1, 0)), ("u=(0, 1)", (0, 1)), ("u=(0, p-1)", (0, P - 1))]
    us += [(f"u=(0, {b})", (0, b)) for b in (3, 5, odd(), odd())] + [(f"u=(0, {b})", (0, b)) for b in (2, 4, even(), even())]
    us += [("u=(odd, 0)", (a, 0)) for a in (3, odd())] + [("u=(even, 0)", (a, 0)) for a in (2, even())]
    us += [("random u", (rnd(), rnd())) for _ in range(8)]
    c[42] = [(n, list(u)) for n, u in us]
    # ---- iso3_map on the kernel: XD = xd (xn^2 + k1 xn xd + k0 xd^2) has the double root x0 = -k1/2, and K4(x0) = 0 as well.  The map
    # is a rational function of (x, y), so y need not make a curve point.
    x0 = PR.mul(PR.neg(PR.K2[1]), (pow(2, -1, P), 0))
    assert PR.horner(PR.K2, x0) == PR.ZERO and PR.horner(PR.K4, x0) == PR.ZERO
    iso = []
    for xd in ((1, 0), (rnd(), rnd()), (0, rnd())):
        for name, x in (("x0", x0), ("x0+1", PR.add(x0, (1, 0))), ("x0+i", PR.add(x0, (0, 1))), ("x0-1", PR.sub(x0, (1, 0)))):
            iso.append((f"{name}, xd={'1' if xd == (1, 0) else 'random'}", [*PR.mul(x, xd), *xd, rnd(), rnd()]))
    c[43] = iso
    # ---- sign predicates
    sg = [(f"(0, {b})", (0, b)) for b in (1, 2, 3, 4, P - 1, P - 2, HALF, HALF + 1, odd(), even())]
    sg += [(f"({a}, 0)", (a, 0)) for a in (0, 1, HALF, HALF + 1, P - 1)]
    sg += [("c1 = (p-1)/2", (rnd(), HALF)), ("c1 = (p+1)/2", (rnd(), HALF + 1)), ("c0 = (p+1)/2", (HALF + 1, rnd()))]
    sg += [("random", (rnd(), rnd())) for _ in range(8)]
    c[45] = [(n, list(a)) for n, a in sg]
    # ---- Fp square root of g1_decode: p = 3 mod 4, so p - 1 is a non-residue
    c[46] = [(str(a), [a]) for a in (0, 1, 4, P - 1, 2, 3)] + [("residue", [a]) for a in res[-4:]] + [("non-residue", [a]) for a in non[-4:]]
    return c

def _clear_cofactor_cases():
    """[(name, point)] for g2_clear_cofactor: G2 points, hashed points before clearing, generic points of E2(Fp2), cofactor-torsion
    points of large and small order, and G2 points plus torsion.  The expectation [h_eff] P is the slow part: keep the set small."""
    pts = [(f"[{k}]G2", PR.smul(k, PR.G2)) for k in (1, 2, 5)]
    pts += [(f"uncleared H({m!r})", PR.map_to_g2_uncleared(m)) for m in (b"", b"clear the cofactor")]
    pts += [(f"Q{i}", q) for i, q in enumerate(curve_points(2))]
    tors = torsion_points()
    pts += tors + [("[7]G2+" + n, PR.padd(PR.smul(7, PR.G2), t)) for n, t in tors if n.startswith(("order13", "order23", "r*Q0"))]
    return pts

@pytest.fixture(scope="module")
def cases():
    c = _cases()
    rng = np.random.default_rng(44)
    cc = []
    for name, pt in _clear_cofactor_cases():
        want = PR.smul(PR.HEFF, pt)
        for z in ((1, 0), (int.from_bytes(rng.bytes(48), "little") % P, int.from_bytes(rng.bytes(48), "little") % P)):
            cc.append((f"{name} Z={'1' if z == (1, 0) else 'random'}", _j2(pt, z), want))
    return c, cc

@pytest.fixture(scope="module")
def E():
    from hostemu import emu
    emu.build(); return emu

def _run(run, op, cases):
    return run(op, np.concatenate([_enc(v) for _, v in cases]))

def _check_primitives(run, cases):
    """every group of inputs through `run(op, input bytes) -> output bytes`; returns the names of the cases that disagree with pyref"""
    c, cc = cases
    bad = []
    for (name, a), row in zip(c[16], _rows(_run(run, 16, c[16]), 3)):
        a = tuple(a); root = _f2(row, 0); ok = _flag(row[2])
        if ok != (PR.sqrt(a) is not None) or (ok and PR.sqr(root) != a): bad.append(("fp2_sqrt", name, a))
    for (name, uv), row in zip(c[25], _rows(_run(run, 25, c[25]), 3)):
        u, v = tuple(uv[:2]), tuple(uv[2:]); y = _f2(row, 0); sq = _flag(row[2])
        q = PR.mul(u, PR.inv(v)); want_sq = PR.is_square(q)
        if sq != want_sq or PR.sqr(y) != (q if want_sq else PR.mul(PR.Z_SSWU, q)): bad.append(("fp2_sqrt_ratio", name, u, v))
    m = _run(run, 42, c[42])
    for (name, u), row, iso_row in zip(c[42], _rows(m, 6), _rows(run(43, m), 6)):
        u = tuple(u); xn, xd, y = _f2(row, 0), _f2(row, 2), _f2(row, 4); wx, wy = PR.sswu(u)
        if xd == PR.ZERO or PR.mul(xn, PR.inv(xd)) != wx or y != wy: bad.append(("sswu_map", name, u))
        if _jac_aff(iso_row) != PR.iso((wx, wy)): bad.append(("iso3_map(sswu_map)", name, u))
    for (name, v), row in zip(c[43], _rows(_run(run, 43, c[43]), 6)):
        xn, xd, y = tuple(v[0:2]), tuple(v[2:4]), tuple(v[4:6])
        want = PR.iso((PR.mul(xn, PR.inv(xd)), y))
        if name.startswith("x0,") != (want is None) or _jac_aff(row) != want: bad.append(("iso3_map", name))
    for (name, v, want), row in zip(cc, _rows(_run(run, 44, [(n, v) for n, v, _ in cc]), 6)):
        if _jac_aff(row) != want: bad.append(("g2_clear_cofactor", name))
    for (name, a), row in zip(c[45], _rows(_run(run, 45, c[45]), 3)):
        a = tuple(a)
        if [_flag(x) for x in row] != [PR.sgn0(a), int(PR.lex_largest(a)), int(a[0] > HALF)]: bad.append(("sign predicates", name, a, row))
    for (name, (a,)), row in zip(c[46], _rows(_run(run, 46, c[46]), 2)):
        y = _v(row[0]); ok = _flag(row[1])
        if ok != (_legendre(a) != P - 1) or (ok and y * y % P != a): bad.append(("fp root", name, a))
    return bad

def test_case_lists_reach_the_branches(cases):
    """the inputs take the branches they are chosen for, by the reference's arithmetic"""
    c, cc = cases
    # the d = 0 arm: a.c1 = 0 and a.c0 a non-residue, where the norm's root a.c0^((p+1)/2) is -a.c0
    assert sum(1 for _, a in c[16] if a[1] == 0 and a[0] and _legendre(a[0]) == P - 1) >= 8
    assert {PR.sqrt(tuple(a)) is None for _, a in c[16]} == {True, False}
    assert {PR.is_square(PR.mul(tuple(v[:2]), PR.inv(tuple(v[2:])))) for _, v in c[25]} == {True, False}
    # SSWU: tv2 = Z^2 u^4 + Z u^2 vanishes at u = 0 only among these (u^2 = -1/Z has no root in Fp2)
    zu2 = lambda u: PR.mul(PR.Z_SSWU, PR.sqr(tuple(u)))
    assert [n for n, u in c[42] if PR.add(PR.sqr(zu2(u)), zu2(u)) == PR.ZERO] == ["u=0"]
    assert PR.sqrt(PR.neg(PR.inv(PR.Z_SSWU))) is None
    assert sum(1 for _, u in c[42] if u[0] == 0 and u[1] & 1) >= 3 and sum(1 for _, u in c[42] if u[0] == 0 and u[1] and not u[1] & 1) >= 3
    assert sum(1 for _, a in c[45] if a[0] == 0 and a[1] & 1) >= 3 and sum(1 for _, a in c[45] if a[1] == 0 and a[0] > HALF) >= 2
    assert sum(1 for _, (a,) in c[46] if _legendre(a) == P - 1) >= 4
    # the small-order points end on the identity or pass through it in the ladder
    assert any(w is None for _, _, w in cc) and any(w is not None for _, _, w in cc)

def test_host_sqrt_sign_and_h2c_edges_match_pyref(E, cases):
    """host build: each primitive at its exceptional inputs gives the reference's value"""
    assert _check_primitives(E.run_op, cases) == []

@pytest.mark.gpu
def test_device_sqrt_sign_and_h2c_edges_match_pyref_and_host(E, cases):
    """the same inputs through the device build (one kernel per op): the reference's values, and the host build's limbs exactly"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "devcheck"))
    import run_devcheck
    D = run_devcheck.dev_lib()
    def run(op, x):
        n_in, n_out = E.op_shape(op); n = x.size // (48 * n_in)
        got = np.zeros(48 * n_out * n, np.uint8)
        rc = D.dev_run_op(int(op), x.ctypes.data_as(ctypes.c_void_p), got.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n))
        assert rc == 0, f"op {op}: rc={rc}"
        want = E.run_op(op, x)
        diff = [i for i in range(n) if not np.array_equal(got[48 * n_out * i:48 * n_out * (i + 1)], want[48 * n_out * i:48 * n_out * (i + 1)])]
        assert diff == [], f"op {op}: device limbs differ from the host build at items {diff[:8]}"
        return got
    assert _check_primitives(run, cases) == []

# ============================================================================================== B: the decoders
# x = a + b i with y^2 = x^3 + 4(1 + i):  Re(x^3) = a^3 - 3 a b^2,  Im(x^3) = 3 a^2 b - b^3.
#   Im(y^2) = 0:  a^2 = (b^3 - 4) / (3 b).  y^2 = c in Fp: y = sqrt(c) in Fp when c is a residue, y in i Fp (fp2_sqrt's d = 0 arm)
#                 when it is not.  Either way x decodes to a point of E2 -- every element of Fp is a square in Fp2.
#   Re(y^2) = 0:  b^2 = (a^3 + 4) / (3 a)
def _enc_x(x, largest):
    b = bytearray(x[1].to_bytes(48, "big") + x[0].to_bytes(48, "big")); b[0] |= 0xa0 if largest else 0x80
    return bytes(b)

def decoder_xs():
    """[(name, x)] of the decoder inputs"""
    rng = np.random.default_rng(2002)
    rnd = lambda: int.from_bytes(rng.bytes(48), "little") % P
    xs, kinds, t = [], {True: 0, False: 0}, 1
    while min(kinds.values()) < 5:
        t += 1
        a2 = (t ** 3 - 4) * pow(3 * t, -1, P) % P
        if _legendre(a2) != 1: continue
        a = pow(a2, (P + 1) // 4, P); y2 = PR.add(PR.mul(PR.sqr((a, t)), (a, t)), PR.B2); assert y2[1] == 0
        qr = _legendre(y2[0]) == 1
        if kinds[qr] < 5: kinds[qr] += 1; xs.append((f"y^2 in Fp, {'residue' if qr else 'non-residue'}, b={t}", (a, t)))
    n, t = 0, 1
    while n < 4:
        t += 1
        b2 = (t ** 3 + 4) * pow(3 * t, -1, P) % P
        if _legendre(b2) != 1: continue
        b = pow(b2, (P + 1) // 4, P); y2 = PR.add(PR.mul(PR.sqr((t, b)), (t, b)), PR.B2); assert y2[0] == 0
        n += 1; xs.append((f"y^2 in i Fp, a={t}", (t, b)))
    xs += [("x=0", (0, 0))] + [("x.c0=0", (0, b)) for b in (1, 2, rnd(), rnd())] + [("x.c1=0", (a, 0)) for a in (1, 2, rnd(), rnd())]
    return xs

def decoder_encodings():
    """[(name, 96 bytes)]: every x of decoder_xs with both sign flags"""
    return [(f"{n}, {'largest' if s else 'smallest'}", _enc_x(x, s)) for n, x in decoder_xs() for s in (False, True)]

DE_MAP = {0: 0, 1: 0, 2: 1, 3: 2, 4: 3, 5: 4}       # BLSGPU_DE_* -> the C oracle's DE_* (infinity decodes fine in the oracle)

def pyref_status(enc):
    """BLSGPU_DE_* status of pyref.deser_g2"""
    try: return 1 if PR.deser_g2(enc) is None else 0
    except PR.DeserErr as e: return {"not on curve": 4, "subgroup": 5}[str(e)]

@pytest.fixture(scope="module")
def encodings():
    encs = decoder_encodings()
    return encs, [pyref_status(e) for _, e in encs]

def test_decoder_encodings_take_the_fallback(encodings):
    """every y^2-in-Fp encoding is on the curve and outside G2; those with a non-residue y^2 take fp2_sqrt's d = 0 arm"""
    encs, want = encodings
    fam = [w for (n, _), w in zip(encs, want) if n.startswith("y^2 in")]
    assert len(fam) >= 26 and set(fam) == {5}
    assert sum(1 for n, _ in encs if "non-residue" in n) >= 8 and sum(1 for n, _ in encs if ", residue" in n) >= 8
    assert {4, 5} <= set(want)

def test_host_decoder_edges_match_oracles(E, encodings):
    """host build of g2_decode: the statuses of pyref and of the C oracle"""
    from oracle import cwrap as C
    encs, want = encodings
    b = b"".join(e for _, e in encs)
    got = list(E.deser_g2(b))
    assert got == want, [(n, g, w) for (n, _), g, w in zip(encs, got, want) if g != w]
    assert [DE_MAP[x] for x in want] == list(C.deser_g2(b))

@pytest.fixture(scope="module")
def ctx():
    from bls_verify_gadget_b200 import Context
    c = Context(0); yield c; c.close()

@pytest.mark.gpu
def test_decoder_edges_through_the_c_abi(ctx, E, encodings):
    """deserialize_g2 and g2_uncompress give pyref's / the C oracle's / the host build's status (and an all-zero output); a verify
    batch that mixes the encodings as signatures with valid triples reports InvalidSignature (3) for them and 0 for the rest, like the
    C oracle, with equal statuses, ok-bitmap and GT accumulator in the split form without the cooperative kernels, in the one-launch
    form (whose decoder tests membership) and under the defaults (the split path's decoder stops at the curve equation, and the
    Miller loop's end-point test has to reject these points)"""
    from oracle import cwrap as C
    from bls_verify_gadget_b200 import synth
    encs, want = encodings
    b = b"".join(e for _, e in encs); ns = len(encs)
    st = list(ctx.deserialize_g2(b))
    assert st == want == list(E.deser_g2(b)), [(n, s, w) for (n, _), s, w in zip(encs, st, want) if s != w]
    assert [DE_MAP[x] for x in st] == list(C.deser_g2(b))
    out, ust = ctx.g2_uncompress(b)
    assert list(ust) == want and not out.any()
    # the batch: valid triples with the encodings planted as signatures, spread over the batch
    n = 3 * ns
    sk = synth.secret_keys(n); msg = synth.messages(n)
    pk, s = ctx.sk_to_pk(sk); assert not s.any()
    sig, s = ctx.sign(sk, msg, fixed32=True); assert not s.any()
    sig = sig.reshape(n, 96).copy()
    pos = np.random.default_rng(7).permutation(n)[:ns]
    for i, (_, e) in zip(pos, encs): sig[i] = np.frombuffer(e, np.uint8)
    sig = sig.reshape(-1)
    msgs = [msg[32 * i:32 * i + 32].tobytes() for i in range(n)]
    ost, ogt = C.verify(pk, msgs, sig, want_gt=True, threads=C.hw_threads())
    exp = np.zeros(n, np.uint8); exp[pos] = 3
    assert np.array_equal(ost, exp)
    res = {"defaults": ctx.verify(pk, msg, sig, want_bitmap=True, want_gt=True, fixed32=True)}
    for name, split, coop in (("split, coop off", 1, 0), ("one launch", 0, 2)):
        ctx.set_split(split); ctx.set_coop(coop)
        try: res[name] = ctx.verify(pk, msg, sig, want_bitmap=True, want_gt=True, fixed32=True)
        finally: ctx.set_split(1); ctx.set_coop(2)
    for name, (st, bm, gt) in res.items():
        assert np.array_equal(st, ost), (name, np.nonzero(st != ost)[0][:8])
        assert np.array_equal(bm, res["defaults"][1]), name
        assert gt.tobytes() == ogt.tobytes(), name
    bits = np.unpackbits(res["defaults"][1].view(np.uint8), bitorder="little")[:n]
    assert np.array_equal(bits, (ost == 0).astype(np.uint8))
