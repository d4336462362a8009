"""blsgpu_verify_batch with the split stage kernels decodes signatures without the subgroup test and tests membership on the Miller
loop's running point instead: pair (-g1, sig) ends on [|x|] sig, which must equal -psi(sig) (csrc/pairing.cuh miller_end_in_subgroup).
Checked here on points in G2 and outside it -- cofactor-torsion points of large and of small order, G2 points plus torsion -- where an
order-13 point drives the running point through an exceptional addition (R = -sig) and the test must still reject it:
(1) the steps of that pair and the end-point test built for the host (tests/sig_subgroup/end_point_check.cu) against g2_in_subgroup and
[r]Q = O; (2) the same source built for sm_100a, against the host build;
(3) whole verify passes, small (six-lane accumulator, decoders and hash side by side) and large (two lanes), against the one-launch form
(which keeps the decoder's test) and the oracle: statuses, ok-bitmap and GT accumulator bytes."""
import ctypes, os, subprocess
import numpy as np
import pytest
from oracle import pyref as R

H2 = 0x5d543a95414e7f1091d50792876a202cd91de4547085abaa68a205b2e5a7ddfa628f1cb4d9e82ef21537e293a6691ae1616ec6e786f0c70cf1c38e31c7238e5  # #E'(Fp2) = H2 r
MONT = 1 << 384

def curve_points(k):
    """k points of E'(Fp2) with x in Fp (x = 2, 3, ...): their order is a multiple of r times a factor of H2"""
    out, x = [], 1
    while len(out) < k:
        x += 1
        try: out.append(R.deser_g2(bytes([0x80]) + bytes(47) + x.to_bytes(48, "big"), subgroup=False))
        except R.DeserErr: pass
    return out

def torsion_points():
    """(name, point) of the cofactor subgroups: the points test_cofactor_torsion_points_rejected uses ([r] Q, large order) and points of
    small order.  The 13-part of E'(Fp2) is Z/13 x Z/13, so [r H2 / 13^2] Q has order 13; with order 13 the loop's addition after
    R = [12] sig meets R = -sig (an exceptional case: Z becomes 0 and stays 0)."""
    qs = curve_points(3)
    pts = [("r*Q%d" % i, R.smul(R.r, q)) for i, q in enumerate(qs)]
    for order, div in ((13, 169), (23, 529), (2713, 2713), (11953, 11953), (262069, 262069)):
        pts += [("order%d_Q%d" % (order, i), R.smul(R.r * H2 // div, q)) for i, q in enumerate(qs[:2])]
    return [(n, p) for n, p in pts if p is not None]

def mont(v): return (v * MONT % R.p).to_bytes(48, "little")

def end_point_input(points):
    """affine Montgomery limbs x.c0, x.c1, y.c0, y.c1 per point"""
    return np.frombuffer(b"".join(mont(q[0][0]) + mont(q[0][1]) + mont(q[1][0]) + mont(q[1][1]) for q in points), np.uint8).copy()

def build_end_point_check(out_dir, device):
    """tests/sig_subgroup/end_point_check.cu for the host (g++) or for sm_100a (nvcc), into out_dir"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = os.path.join(root, "tests", "sig_subgroup", "end_point_check.cu"); inc = os.path.join(root, "bls_verify_gadget_b200", "csrc")
    so = os.path.join(str(out_dir), "end_point_check_%s.so" % ("dev" if device else "host"))
    if device: cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-I", inc, "-o", so, src]
    else: cmd = ["g++", "-x", "c++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", inc, "-o", so, src]
    subprocess.check_call(cmd)
    return ctypes.CDLL(so)

def run_end_point_check(lib, device, points):
    """-> (end-point test, end point's Z is 0, g2_in_subgroup) per point"""
    x = end_point_input(points); n = len(points); out = np.zeros(3 * n, np.uint32)
    fn = lib.dev_end_point_check if device else lib.host_end_point_check
    assert fn(x.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n), out.ctypes.data_as(ctypes.c_void_p)) == 0
    out = out.reshape(n, 3)
    return out[:, 0], out[:, 1], out[:, 2]

def end_point_cases():
    inside = [("[%d]G2" % k, R.smul(k, R.G2)) for k in (1, 2, 3, R.X, R.r - 1)] + [("H(m)", R.hash_to_g2(b"subgroup test on the Miller loop"))]
    tors = torsion_points()
    outside = tors + [("Q%d" % i, q) for i, q in enumerate(curve_points(3))]
    outside += [("[7]G2+" + n, R.padd(R.smul(7, R.G2), t)) for n, t in tors if n.startswith(("order13", "order23", "r*Q0"))]
    return inside, outside

def test_host_end_point_subgroup_test_matches_g2_in_subgroup(tmp_path):
    """host build: miller_end_in_subgroup on the signature pair's end point == g2_in_subgroup == ([r] Q == O), for points in G2 and
    outside it; the order-13 points end with Z = 0 (the exceptional case is taken and rejected), no other point does"""
    lib = build_end_point_check(tmp_path, device=False)
    inside, outside = end_point_cases()
    cases = inside + outside
    test, z0, sub = run_end_point_check(lib, False, [q for _, q in cases])
    for k, (name, q) in enumerate(cases):
        member = R.smul(R.r, q) is None
        assert member == (k < len(inside)), name
        if name.startswith("order"): assert R.smul(int(name[5:name.index("_")]), q) is None, name
        assert test[k] == sub[k] == int(member), (name, test[k], sub[k])
        assert z0[k] == int(name.startswith("order13")), (name, z0[k])
    assert sum(1 for n, _ in cases if n.startswith("order13")) >= 2

# ------------------------------------------------------------------------------------------ on the GPU
@pytest.fixture(scope="module")
def ctx():
    from bls_verify_gadget_b200 import Context
    c = Context(0); yield c; c.close()

@pytest.mark.gpu
def test_end_point_subgroup_test_device_equals_host(tmp_path):
    """the same source compiled for sm_100a gives the host build's results on the same points"""
    inside, outside = end_point_cases()
    pts = [q for _, q in inside + outside]
    dev = run_end_point_check(build_end_point_check(tmp_path, device=True), True, pts)
    host = run_end_point_check(build_end_point_check(tmp_path, device=False), False, pts)
    for d, h in zip(dev, host): assert np.array_equal(d, h)
    assert list(dev[0]) == [1] * len(inside) + [0] * len(outside)

def special_batch(ctx, n, every, seed):
    """n triples of the bench recipe (every corruption kind) with signatures outside G2 planted across the batch: torsion points, a valid
    signature plus torsion, such signatures beside an infinite or undecodable key, and the infinity signature"""
    from bls_verify_gadget_b200 import synth
    pk, msg, sig, _ = synth.verify_batch_inputs(ctx, n, every=every)
    pk = pk.reshape(n, 48).copy(); sig = sig.reshape(n, 96).copy()
    rng = np.random.default_rng(seed)
    pos = iter(rng.permutation([i for i in range(n) if i % every != every - 1])[:64].tolist())
    tors = torsion_points()
    for _, t in tors: sig[next(pos)] = np.frombuffer(R.ser_g2(t), np.uint8)
    for name, t in tors:
        if name.startswith(("order13", "order23", "r*Q")):
            i = next(pos); sig[i] = np.frombuffer(R.ser_g2(R.padd(R.deser_g2(sig[i].tobytes()), t)), np.uint8)
    for k, (_, t) in enumerate(tors[:4]):
        i = next(pos); sig[i] = np.frombuffer(R.ser_g2(t), np.uint8)
        if k % 2: pk[i] = 0; pk[i, 0] = 0xc0                                # identity key
        else: pk[i, 44:] = 0xff                                             # not on the curve (w.h.p.)
    for _ in range(2): i = next(pos); sig[i] = 0; sig[i, 0] = 0xc0          # infinity signature: decodes, its pair is skipped
    sig[n - 1] = np.frombuffer(R.ser_g2(tors[-1][1]), np.uint8)            # last item of the last lane
    return pk.reshape(-1), msg, sig.reshape(-1)

@pytest.mark.gpu
@pytest.mark.parametrize("n", [2000, 16500])
def test_verify_batch_rejects_non_subgroup_signatures_like_decoder(ctx, n):
    """2,000 items: one pass of <= 4,096 items (six-lane accumulator and final exponentiation, decoders and hash side by side; also the
    thread-per-item accumulator with coop off, and the six-lane one on the context's stream); 16,500 items: two lanes of > 8,192.
    Statuses, ok-bitmap and GT accumulator equal the one-launch form's (whose decoder tests membership) and the oracle's."""
    from oracle import cwrap as C
    pk, msg, sig = special_batch(ctx, n, every=9, seed=n)
    msgs = [msg[32 * i:32 * i + 32].tobytes() for i in range(n)]
    ost, ogt = C.verify(pk, msgs, sig, want_gt=True, threads=C.hw_threads())
    assert (ost == 3).sum() >= 20 and (ost == 2).sum() >= 4 and (ost == 1).sum() >= 2
    modes = [(0, 0), (1, 2)] + ([(1, 0), (1, 1)] if n <= 4096 else [])
    out = {}
    ctx.set_lanes(2)
    for split, coop in modes:
        ctx.set_split(split); ctx.set_coop(coop)
        try: out[(split, coop)] = ctx.verify(pk, msg, sig, want_bitmap=True, want_gt=True, fixed32=True)
        finally: ctx.set_split(1); ctx.set_coop(2)
    for mode, (st, bm, gt) in out.items():
        assert np.array_equal(st, ost), (mode, np.nonzero(st != ost)[0][:8])
        assert gt.tobytes() == ogt.tobytes(), mode
        assert np.array_equal(bm, out[(0, 0)][1]), mode
    bits = np.unpackbits(out[(1, 2)][1].view(np.uint8), bitorder="little")[:n]
    assert np.array_equal(bits, (ost == 0).astype(np.uint8))
