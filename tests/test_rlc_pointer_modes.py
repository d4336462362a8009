"""blsgpu_verify_batch_rlc and blsgpu_verify_batch_rlc_bisect with device pointers: fixed 32-byte messages (msg_off NULL) and ragged
messages whose device offsets are absolute into msg, over 3 pieces of 4,096 and a ragged fourth, with bad items in pieces 1 and 3.
Status, ok-bitmap, items re-run and all_ok must equal the host-pointer call and blsgpu_verify_batch, at the default chunk, with passes of
one piece (bisect) or 64 items (rlc), and with the one-launch stage kernels."""
import ctypes
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N = 3 * 4096 + 777
SEED = np.frombuffer(bytes(range(16)), np.uint8).copy()
BAD = [7, 4101, 4996, 4997, 12298, 12988, 12989]

@pytest.fixture(scope="module")
def ctx():
    from bls_verify_gadget_b200 import Context
    c = Context(0); yield c; c.close()

@pytest.fixture(scope="module")
def batches(ctx):
    """name -> (clean batch, batch with bad items), each (pk48, msg, msg_off or None, sig96) as host arrays"""
    from bls_verify_gadget_b200 import synth
    from bls_verify_gadget_b200._lib import pack_msgs
    sk = synth.fast_secret_keys(N); pk, st = ctx.sk_to_pk(sk); assert not st.any()
    rng = np.random.default_rng(41)
    m32 = synth.fast_random_bytes(32 * N, 0x6d7367)
    rag = [rng.bytes(int(l)) for l in rng.integers(1, 90, size=N)]
    out = {}
    for name, msgs, fixed in (("fixed32", m32, True), ("ragged", rag, False)):
        sig, st = ctx.sign(sk, msgs, fixed32=fixed); assert not st.any()
        flat, off = (m32.copy(), None) if fixed else pack_msgs(rag)
        clean = (pk.copy(), flat, off, sig.copy())
        P, M, S = pk.reshape(N, 48).copy(), flat.copy(), sig.reshape(N, 96).copy()
        M[off[4096 + 5] if off is not None else 32 * (4096 + 5)] ^= 1                   # wrong message          (piece 1)
        S[[4096 + 900, 4096 + 901]] = S[[4096 + 901, 4096 + 900]]                        # swapped signatures     (piece 1)
        S[3 * 4096 + 10, 92:] = 0xff                                                     # undecodable signature  (piece 3)
        P[7] = 0; P[7, 0] = 0xc0                                                         # identity public key    (piece 0): decode status only
        P[[3 * 4096 + 700, 3 * 4096 + 701]] = P[[3 * 4096 + 701, 3 * 4096 + 700]]        # swapped keys           (piece 3)
        out[name] = (clean, (P.reshape(-1), M, off, S.reshape(-1)))
    return out

def _checks(ctx, batch, device, rlc_chunk, bisect_chunk):
    """-> (all_ok, status) of blsgpu_verify_batch_rlc and (status, ok_bitmap, items re-run) of blsgpu_verify_batch_rlc_bisect"""
    import torch
    from bls_verify_gadget_b200 import _lib
    pk, msg, off, sig = batch
    words = (N + 63) // 64
    bufs = [pk, msg, off, sig, SEED, np.zeros(N, np.uint8), np.zeros(1, np.uint8), np.zeros(N, np.uint8), np.zeros(words, np.uint64)]
    if device:
        dev = [None if a is None else torch.from_numpy(np.ascontiguousarray(a).view(np.uint8)).to("cuda:0") for a in bufs]
        args = [None if t is None else t.data_ptr() for t in dev]
    else: args = bufs
    dpk, dmsg, doff, dsig, dseed, rst, rok, bst, bbm = args
    rerun = ctypes.c_uint64(0); p = _lib._p
    ctx.set_pointer_mode(device)
    try:
        ctx.set_chunk(rlc_chunk)
        ctx.verify_rlc_ptr(dpk, dmsg, doff, dsig, N, dseed, rst, rok)
        ctx.set_chunk(bisect_chunk)
        ctx._ck(_lib.lib().blsgpu_verify_batch_rlc_bisect(ctx._h, p(dpk), p(dmsg), p(doff), p(dsig), ctypes.c_size_t(N), p(dseed), p(bst), p(bbm),
                                                          ctypes.byref(rerun)))
        ctx.synchronize()
    finally:
        ctx.set_pointer_mode(False); ctx.set_chunk(1 << 20)
    if device: bufs = bufs[:5] + [t.cpu().numpy().view(a.dtype) for t, a in zip(dev[5:], bufs[5:])]
    return bool(bufs[6][0]), bufs[5], bufs[7], bufs[8], int(rerun.value)

@pytest.mark.parametrize("kind", ["fixed32", "ragged"])
def test_rlc_checks_with_device_pointers_match_host_pointers_and_per_item_verify(ctx, batches, kind):
    clean, bad = batches[kind]
    wst, wbm = np.zeros(N, np.uint8), np.zeros((N + 63) // 64, np.uint64)
    ctx.verify_ptr(*bad, N, wst, wbm)
    assert np.nonzero(wst)[0].tolist() == BAD
    decode = np.where((wst == 2) | (wst == 3), wst, 0)                                    # the rlc form reports decode outcomes only
    all_bits = np.full((N + 63) // 64, ~np.uint64(0)); all_bits[-1] = (np.uint64(1) << np.uint64(N % 64)) - np.uint64(1)
    for split, rlc_chunk, bisect_chunk in ((1, 1 << 20, 1 << 20), (1, 64, 4096), (0, 1 << 20, 1 << 20)):
        ctx.set_split(split)
        try:
            for device in (False, True):
                ok, rst, bst, bbm, rerun = _checks(ctx, clean, device, rlc_chunk, bisect_chunk)
                assert ok and not rst.any() and not bst.any() and np.array_equal(bbm, all_bits) and rerun == 0, (split, rlc_chunk, device)
                ok, rst, bst, bbm, rerun = _checks(ctx, bad, device, rlc_chunk, bisect_chunk)
                assert not ok and np.array_equal(rst, decode), (split, rlc_chunk, device)
                assert np.array_equal(bst, wst) and np.array_equal(bbm, wbm) and rerun == 4096 + 777, (split, bisect_chunk, device)
        finally: ctx.set_split(1)
