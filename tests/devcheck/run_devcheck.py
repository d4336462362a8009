"""Host-emulation vs device comparison of every primitive in tests/devcheck/ops.h on random field elements."""
import ctypes, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from hostemu import emu
P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
SO = os.path.join(ROOT, "tests", "_hostemu", "libdevcheck.so")
def build():
    """nvcc build of devcheck.cu, redone when the CONTENT of any source differs from the stamp beside the library (mtimes do not
    survive the copy to the GPU box); __graft_entry__.build() calls this so that the library travels prebuilt.  When the prebuilt copy
    is stale and its directory cannot be written (a read-only tree), the library is built in a temporary directory instead.
    The digest covers every header of csrc/, not only the ones devcheck.cu names: ops.h reaches h2c.cuh through stages.cuh"""
    import hashlib, subprocess, tempfile
    csrc = os.path.join(ROOT, "bls_verify_gadget_b200", "csrc")
    src = [os.path.join(ROOT, "tests", "devcheck", f) for f in ("devcheck.cu", "ops.h")] + [os.path.join(csrc, f) for f in sorted(os.listdir(csrc)) if f.endswith(".cuh")]
    h = hashlib.sha256()
    for f in src: h.update(open(f, "rb").read())
    digest = h.hexdigest()
    so = SO
    try: os.makedirs(os.path.dirname(SO), exist_ok=True)
    except OSError: pass
    if not os.access(os.path.dirname(SO), os.W_OK) and not _fresh(SO, digest):
        so = os.path.join(tempfile.gettempdir(), "blsgpu-devcheck-" + digest[:16], "libdevcheck.so"); os.makedirs(os.path.dirname(so), exist_ok=True)
    if not _fresh(so, digest):
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-I", csrc, "-o", so, src[0]])
        open(so + ".stamp", "w").write(digest + "\n")
    return so
def _fresh(so, digest):
    stamp = so + ".stamp"
    return os.path.exists(so) and os.path.exists(stamp) and open(stamp).read().strip() == digest
def dev_lib():
    return ctypes.CDLL(os.environ.get("DEVCHECK_SO") or build())
def rand_fp(rng, n):
    a = rng.integers(0, 256, size=(n, 48), dtype=np.uint8); a[:, 47] &= 0x0f      # < 2^380 < p: a valid Montgomery image
    return a
def edge_fp(rng, n):
    """canonical field elements biased to the extremes the lazy-reduction bounds depend on: 0, 1, p-1, p-2, 2^380.., random"""
    specials = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, (1 << 380) - 1, 1 << 380, P - (1 << 32), 0xffffffff, (1 << 352) - 1]
    out = np.zeros((n, 48), np.uint8)
    pick = rng.integers(0, 2 * len(specials), size=n)
    for i in range(n):
        v = specials[pick[i]] if pick[i] < len(specials) else int.from_bytes(rng.bytes(48), "little") % P
        out[i] = np.frombuffer(v.to_bytes(48, "little"), np.uint8)
    return out
EDGE_OPS = (1, 2, 3, 4, 8, 9, 10, 11, 12, 21, 22, 26, 27, 29, 30, 31, 32, 33, 34, 35, 36, 45, 46)      # pure field arithmetic: any canonical input is valid
def check(ops=range(1, 47), n=256, seed=1, edge=False):
    D = dev_lib(); rng = np.random.default_rng(seed); bad = []
    for op in ops:
        n_in, n_out = emu.op_shape(op)
        if not n_in: continue
        if edge and op not in EDGE_OPS: continue
        x = (edge_fp(rng, n * n_in) if edge else rand_fp(rng, n * n_in)).reshape(-1)
        if op in (16,):          # make half of the inputs squares
            pass
        want = emu.run_op(op, x)
        got = np.zeros(48 * n_out * n, np.uint8)
        rc = D.dev_run_op(int(op), x.ctypes.data_as(ctypes.c_void_p), got.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n))
        ok = rc == 0 and np.array_equal(got, want)
        nbad = int((got.reshape(n, -1) != want.reshape(n, -1)).any(axis=1).sum())
        print(f"op {op:2d} in={n_in:2d} out={n_out:2d} rc={rc} {'ok' if ok else 'MISMATCH items=' + str(nbad)}")
        if not ok:
            bad.append(op); g = got.reshape(n, n_out, 48); w = want.reshape(n, n_out, 48)
            print('   mismatching output fps (item 0):', [k for k in range(n_out) if not np.array_equal(g[0, k], w[0, k])], ' items:', np.nonzero((g != w).any(axis=(1, 2)))[0][:8])
    return bad
if __name__ == "__main__":
    bad = check() + check(edge=True, seed=7); print("bad ops:", bad); sys.exit(1 if bad else 0)
