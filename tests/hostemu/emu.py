"""ctypes loader for the host-emulation build of the CUDA path's device functions (test tool only)."""
import ctypes, os, subprocess
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__)); ROOT = os.path.dirname(os.path.dirname(HERE))
SO = os.path.join(ROOT, "tests", "_hostemu", "libhostemu.so")
SRC = [os.path.join(HERE, "hostemu.cpp"), os.path.join(ROOT, "tests", "devcheck", "ops.h")] + [os.path.join(ROOT, "bls_verify_gadget_b200", "csrc", f) for f in
      ("fp.cuh", "fp2.cuh", "tower.cuh", "curve.cuh", "h2c.cuh", "pairing.cuh", "stages.cuh", "consts.cuh", "wide.cuh")]
def build():
    """rebuilt when a source is newer than the library; in a read-only tree a stale library is rebuilt in a temporary directory"""
    if not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in SRC):
        so = SO
        try: os.makedirs(os.path.dirname(SO), exist_ok=True)
        except OSError: pass
        if not os.access(os.path.dirname(SO), os.W_OK):
            import tempfile; so = os.path.join(tempfile.mkdtemp(prefix="blsgpu-hostemu-"), "libhostemu.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "bls_verify_gadget_b200", "csrc"), "-o", so, SRC[0]])
        return so
    return SO
_lib = None
def lib():
    global _lib
    if _lib is None: _lib = ctypes.CDLL(build())
    return _lib
def _u8(a):
    if isinstance(a, np.ndarray): return np.ascontiguousarray(a, dtype=np.uint8).reshape(-1)
    return np.frombuffer(bytes(a) + b"\0", dtype=np.uint8)[:len(a)].copy()
def _p(a): return None if a is None else (a if a.size else np.zeros(1, a.dtype)).ctypes.data_as(ctypes.c_void_p)
_sz = ctypes.c_size_t
def _pack(msgs):
    off = np.zeros(len(msgs) + 1, dtype=np.uint32); off[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    return np.frombuffer(b"".join(msgs) + b"\0", dtype=np.uint8).copy(), off
def fp_mul_raw(a, b):
    a = _u8(a); b = _u8(b); n = a.size // 48; o = np.empty(48 * n, np.uint8); lib().emu_fp_mul_raw(_p(a), _p(b), _p(o), _sz(n)); return o
def deser_g1(x): x = _u8(x); n = x.size // 48; st = np.empty(n, np.uint8); lib().emu_deser_g1(_p(x), _sz(n), _p(st)); return st
def deser_g2(x): x = _u8(x); n = x.size // 96; st = np.empty(n, np.uint8); lib().emu_deser_g2(_p(x), _sz(n), _p(st)); return st
def recode_g1(x): x = _u8(x); n = x.size // 48; o = np.empty(48 * n, np.uint8); lib().emu_recode_g1(_p(x), _sz(n), _p(o)); return o
def recode_g2(x): x = _u8(x); n = x.size // 96; o = np.empty(96 * n, np.uint8); lib().emu_recode_g2(_p(x), _sz(n), _p(o)); return o
def hash_to_g2(msgs, cleared=True):
    f, off = _pack(msgs); o = np.empty(96 * len(msgs), np.uint8); lib().emu_hash_to_g2(_p(f), _p(off), _sz(len(msgs)), _p(o), int(cleared)); return o
def verify(pk, msgs, sig, want_gt=False):
    pk = _u8(pk); sig = _u8(sig); f, off = _pack(msgs); n = len(msgs); st = np.empty(n, np.uint8); gt = np.empty(576 * n, np.uint8) if want_gt else None
    lib().emu_verify(_p(pk), _p(f), _p(off), _p(sig), _sz(n), _p(st), _p(gt)); return (st, gt) if want_gt else st
def sk_to_pk(sk): sk = _u8(sk); n = sk.size // 32; o = np.empty(48 * n, np.uint8); lib().emu_sk_to_pk(_p(sk), _sz(n), _p(o)); return o
def sign(sk, msgs):
    sk = _u8(sk); f, off = _pack(msgs); o = np.empty(96 * len(msgs), np.uint8); lib().emu_sign(_p(sk), _p(f), _p(off), _sz(len(msgs)), _p(o)); return o
def g1_sum(pts): x = _u8(pts); o = np.empty(48, np.uint8); lib().emu_g1_sum(_p(x), _sz(x.size // 48), _p(o)); return o
def g2_sum(pts): x = _u8(pts); o = np.empty(96, np.uint8); lib().emu_g2_sum(_p(x), _sz(x.size // 96), _p(o)); return o
def pairing_gt(g1, g2): a = _u8(g1); b = _u8(g2); o = np.empty(576, np.uint8); lib().emu_pairing_gt(_p(a), _p(b), _sz(a.size // 48), _p(o)); return o

def op_shape(op):
    import ctypes as c
    a = c.c_int(); b = c.c_int(); lib().emu_op_shape(int(op), c.byref(a), c.byref(b)); return a.value, b.value
def run_op(op, inp):
    n_in, n_out = op_shape(op); x = _u8(inp); n = x.size // (48 * n_in); o = np.zeros(48 * n_out * n, np.uint8)
    assert lib().emu_run_op(int(op), _p(x), _p(o), _sz(n)) == 0; return o
