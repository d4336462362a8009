"""ctypes binding of libblsgpu.so (the C ABI of include/blsgpu.h).  There is NO CPU fallback: loading fails loudly
when the library is not built, and Context() fails loudly when no sm_100 CUDA device is usable."""
import ctypes, os, subprocess
import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
SO_PATH = os.environ.get("BLSGPU_SO") or os.path.join(_PKG, "libblsgpu.so")      # BLSGPU_SO: tuning builds (profiles/), never a fallback
import glob
_SOURCES = [os.path.join(_PKG, "csrc", "blsgpu.cu")] + sorted(glob.glob(os.path.join(_PKG, "csrc", "*.cuh"))) + sorted(glob.glob(os.path.join(_ROOT, "include", "*.h")))      # every header the one translation unit includes
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread", "-ldl"]

class BlsGpuError(RuntimeError): pass

def build(force=False, verbose=False, extra_flags=(), out=None):
    """nvcc cross-compiles for sm_100a without a GPU; the .so is kept in-tree so it travels to the GPU box."""
    stale = not os.path.exists(SO_PATH) or any(os.path.getmtime(s) > os.path.getmtime(SO_PATH) for s in _SOURCES)
    if force or stale:
        cmd = ["nvcc"] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + ["-o", out or SO_PATH, _SOURCES[0]]
        subprocess.check_call(cmd)
    return out or SO_PATH

_lib = None
def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise BlsGpuError(f"{SO_PATH} is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); there is no CPU fallback")
        L = ctypes.CDLL(SO_PATH)
        L.blsgpu_last_error.restype = ctypes.c_char_p
        L.blsgpu_launch_count.restype = ctypes.c_uint64
        L.blsgpu_multi_last_error.restype = ctypes.c_char_p
        L.blsgpu_multi_ctx.restype = ctypes.c_void_p
        L.blsgpu_witness_msg_len.restype = ctypes.c_long
        _lib = L
    return _lib

EXPORTS = ["blsgpu_create", "blsgpu_destroy", "blsgpu_last_error", "blsgpu_set_stream", "blsgpu_set_pointer_mode", "blsgpu_synchronize",
           "blsgpu_launch_count", "blsgpu_set_profiling", "blsgpu_stage_times", "blsgpu_set_chunk", "blsgpu_set_lanes", "blsgpu_set_split", "blsgpu_set_coop", "blsgpu_verify_batch", "blsgpu_verify_batch_rlc", "blsgpu_verify_batch_rlc_bisect", "blsgpu_fast_aggregate_verify_batch", "blsgpu_aggregate_verify_batch", "blsgpu_g1_uncompress", "blsgpu_g1_compress", "blsgpu_g2_uncompress", "blsgpu_g2_compress", "blsgpu_pool_create", "blsgpu_pool_free", "blsgpu_pool_fast_aggregate_verify", "blsgpu_verify_signature_sets", "blsgpu_pool_verify_signature_sets", "blsgpu_hash_to_g2_batch", "blsgpu_g1_aggregate",
           "blsgpu_g2_aggregate", "blsgpu_deserialize_g1", "blsgpu_deserialize_g2", "blsgpu_sk_to_pk_batch", "blsgpu_sign_batch", "blsgpu_pairing_gt",
           "blsgpu_gt_fold", "blsgpu_fp_mul_raw", "blsgpu_imad_peak", "blsgpu_r1cs_load", "blsgpu_r1cs_check", "blsgpu_r1cs_free", "blsgpu_r1cs_row_classes", "blsgpu_r1cs_load_file", "blsgpu_r1cs_check_file", "blsgpu_witness_load", "blsgpu_witness_gen", "blsgpu_witness_check", "blsgpu_witness_free", "blsgpu_witness_msg_len", "blsgpu_witness_load_aggregate", "blsgpu_witness_shape", "blsgpu_witness_gen_aggregate", "blsgpu_witness_check_aggregate",
           "blsgpu_create_multi", "blsgpu_destroy_multi", "blsgpu_multi_last_error", "blsgpu_multi_ndev", "blsgpu_multi_nccl_version", "blsgpu_multi_ctx", "blsgpu_multi_verify_batch", "blsgpu_multi_peek"]

_sz = ctypes.c_size_t; _vp = ctypes.c_void_p
def _u8(a):
    if isinstance(a, np.ndarray): return np.ascontiguousarray(a, dtype=np.uint8).reshape(-1)
    b = bytes(a); return np.frombuffer(b + b"\0", dtype=np.uint8)[:len(b)].copy()
def _p(a):
    if a is None: return None
    if isinstance(a, int): return _vp(a)                      # raw device pointer
    if a.size == 0: a = np.zeros(1, dtype=a.dtype)
    return a.ctypes.data_as(_vp)
def _need(name, a, nbytes):
    """the C side trusts the sizes it is given: a short host buffer would be read past its end, so the wrappers check"""
    if a is not None and a.size * a.itemsize != nbytes: raise ValueError(f"{name}: expected {nbytes} bytes, got {a.size * a.itemsize}")
def pack_msgs(msgs):
    off = np.zeros(len(msgs) + 1, dtype=np.uint32)
    if len(msgs): off[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    return np.frombuffer(b"".join(msgs) + b"\0", dtype=np.uint8).copy(), off

class Context:
    """One per GPU per process.  Host-pointer mode by default (numpy in, numpy out); `device_mode()` switches the
    raw-pointer methods (suffix _ptr) to device pointers for callers that keep data resident in HBM (bench.py)."""
    def __init__(self, device=-1):
        self._h = _vp()
        rc = lib().blsgpu_create(ctypes.byref(self._h), int(device))
        if rc != 0:
            self._h = None
            raise BlsGpuError(f"blsgpu_create failed (rc={rc}): no usable sm_100 CUDA device -- this library has no CPU fallback")
    def close(self):
        if getattr(self, "_h", None): lib().blsgpu_destroy(self._h); self._h = None
    def __del__(self):
        try: self.close()
        except Exception: pass
    def _ck(self, rc):
        if rc != 0: raise BlsGpuError(f"rc={rc}: {lib().blsgpu_last_error(self._h).decode()}")
    def set_stream(self, cuda_stream, use_own=False): self._ck(lib().blsgpu_set_stream(self._h, _vp(cuda_stream) if cuda_stream else None, 1 if use_own else 0))
    def set_pointer_mode(self, device): self._ck(lib().blsgpu_set_pointer_mode(self._h, 1 if device else 0))
    def synchronize(self): self._ck(lib().blsgpu_synchronize(self._h))
    def launch_count(self): return int(lib().blsgpu_launch_count(self._h))
    def set_coop(self, mode): self._ck(lib().blsgpu_set_coop(self._h, int(mode)))      # 0 never, 1 always, 2 (library default) small passes only
    def set_lanes(self, lanes): self._ck(lib().blsgpu_set_lanes(self._h, int(lanes)))
    def set_split(self, mode): self._ck(lib().blsgpu_set_split(self._h, int(mode)))
    def set_chunk(self, items): self._ck(lib().blsgpu_set_chunk(self._h, _sz(items)))
    def set_profiling(self, on=True): self._ck(lib().blsgpu_set_profiling(self._h, 1 if on else 0))
    def stage_times(self):
        ms = (ctypes.c_float * 6)(); self._ck(lib().blsgpu_stage_times(self._h, ms))
        return dict(zip(("decode_g1", "decode_g2", "hash_to_g2", "miller", "final_exp", "epilogue"), [float(x) for x in ms]))
    # ---- raw pointer entry points (host numpy arrays or device pointers as ints, matching the pointer mode)
    def verify_ptr(self, pk, msg, off, sig, n, status, bitmap=None, gt=None):
        self._ck(lib().blsgpu_verify_batch(self._h, _p(pk), _p(msg), _p(off), _p(sig), _sz(n), _p(status), _p(bitmap), _p(gt)))
    def verify_rlc_ptr(self, pk, msg, off, sig, n, seed16, status, all_ok):
        self._ck(lib().blsgpu_verify_batch_rlc(self._h, _p(pk), _p(msg), _p(off), _p(sig), _sz(n), _p(seed16), _p(status), _p(all_ok)))
    def verify_rlc(self, pk48, msgs, sig96, seed16, fixed32=False):
        """random-linear-combination batch check (host mode): returns (all_ok bool, per-item decode status)"""
        pk = _u8(pk48); sg = _u8(sig96); n = sg.size // 96
        if fixed32: flat, off = _u8(msgs), None
        else: flat, off = pack_msgs(msgs)
        _need("sig96", sg, 96 * n); _need("pk48", pk, 48 * n)
        if fixed32: _need("msgs", flat, 32 * n)
        elif len(msgs) != n: raise ValueError(f"{len(msgs)} messages for {n} signatures")
        st = np.empty(max(n, 1), np.uint8); ok = np.zeros(1, np.uint8); seed = _u8(seed16); _need("seed16", seed, 16)
        self.verify_rlc_ptr(pk, flat, off, sg, n, seed, st, ok)
        return bool(ok[0]), st[:n]
    def verify_rlc_bisect(self, pk48, msgs, sig96, seed16, fixed32=False):
        """batch check with exact per-item outcome (host mode): -> (status uint8[n], ok_bitmap uint64[ceil(n/64)], items re-run per item)"""
        pk = _u8(pk48); sg = _u8(sig96); n = sg.size // 96
        if fixed32: flat, off = _u8(msgs), None
        else: flat, off = pack_msgs(msgs)
        _need("sig96", sg, 96 * n); _need("pk48", pk, 48 * n)
        if fixed32: _need("msgs", flat, 32 * n)
        elif len(msgs) != n: raise ValueError(f"{len(msgs)} messages for {n} signatures")
        st = np.empty(max(n, 1), np.uint8); bm = np.zeros(max((n + 63) // 64, 1), np.uint64); seed = _u8(seed16); _need("seed16", seed, 16); rerun = ctypes.c_uint64(0)
        self._ck(lib().blsgpu_verify_batch_rlc_bisect(self._h, _p(pk), _p(flat), _p(off), _p(sg), _sz(n), _p(seed), _p(st), _p(bm), ctypes.byref(rerun)))
        return st[:n], bm[:(n + 63) // 64], int(rerun.value)
    def hash_to_g2_ptr(self, msg, off, n, out): self._ck(lib().blsgpu_hash_to_g2_batch(self._h, _p(msg), _p(off), _sz(n), _p(out)))
    def fast_aggregate_verify_ptr(self, pks, bitmap, k, msg, sig, ncomm, status, agg=None):
        self._ck(lib().blsgpu_fast_aggregate_verify_batch(self._h, _p(pks), _p(bitmap), _sz(k), _p(msg), _p(sig), _sz(ncomm), _p(status), _p(agg)))
    # ---- numpy convenience layer (host mode)
    def verify(self, pk48, msgs, sig96, want_bitmap=False, want_gt=False, fixed32=False):
        pk = _u8(pk48); sg = _u8(sig96); n = sg.size // 96
        if fixed32: flat, off = _u8(msgs), None
        else: flat, off = pack_msgs(msgs)
        _need("sig96", sg, 96 * n); _need("pk48", pk, 48 * n)
        if fixed32: _need("msgs", flat, 32 * n)
        elif len(msgs) != n: raise ValueError(f"{len(msgs)} messages for {n} signatures")
        st = np.empty(n, np.uint8); bm = np.zeros((n + 63) // 64, np.uint64) if want_bitmap else None; gt = np.empty(576, np.uint8) if want_gt else None
        self.verify_ptr(pk, flat, off, sg, n, st, bm, gt)
        out = (st,) + ((bm,) if want_bitmap else ()) + ((gt,) if want_gt else ())
        return out[0] if len(out) == 1 else out
    def fast_aggregate_verify(self, pks48, k, msg32, sig96, bitmap=None, want_agg=False):
        pk = _u8(pks48); m = _u8(msg32); sg = _u8(sig96); nc = sg.size // 96
        st = np.empty(nc, np.uint8); agg = np.empty(48 * nc, np.uint8) if want_agg else None
        bm = np.ascontiguousarray(bitmap, dtype=np.uint64) if bitmap is not None else None
        _need("sig96", sg, 96 * nc); _need("msg32", m, 32 * nc); _need("pks48", pk, 48 * nc * k); _need("bitmap", bm, 8 * ((nc * k + 63) // 64))
        self.fast_aggregate_verify_ptr(pk, bm, k, m, sg, nc, st, agg)
        return (st, agg) if want_agg else st
    def aggregate_verify(self, pks48, msgs, pair_off, sig96):
        """Eth2 AggregateVerify (distinct messages): signature s covers pairs [pair_off[s], pair_off[s+1]) of (pks48[j], msgs[j]) -> status per signature"""
        pk = _u8(pks48); sg = _u8(sig96); ns = sg.size // 96; po = np.ascontiguousarray(pair_off, dtype=np.uint32)
        if po.size != ns + 1 or (ns and (po[0] != 0 or np.any(np.diff(po.astype(np.int64)) < 0))): raise ValueError("pair_off must hold nsig + 1 non-decreasing offsets starting at 0")
        npairs = int(po[-1]) if po.size else 0
        if len(msgs) != npairs: raise ValueError(f"{len(msgs)} messages for {npairs} pairs")
        _need("pks48", pk, 48 * npairs); _need("sig96", sg, 96 * ns)
        flat, off = pack_msgs(msgs); st = np.empty(max(ns, 1), np.uint8)
        self._ck(lib().blsgpu_aggregate_verify_batch(self._h, _p(pk), _p(flat), _p(off), _p(po), _p(sg), _sz(ns), _p(st))); return st[:ns]
    def _recode(self, fn, data, in_sz, out_sz):
        a = _u8(data); n = a.size // in_sz; _need("input", a, in_sz * n); out = np.empty(max(out_sz * n, 1), np.uint8); st = np.empty(max(n, 1), np.uint8)
        self._ck(fn(self._h, _p(a), _sz(n), _p(out), _p(st))); return out[:out_sz * n], st[:n]
    def g1_uncompress(self, in48): return self._recode(lib().blsgpu_g1_uncompress, in48, 48, 96)
    def g1_compress(self, in96): return self._recode(lib().blsgpu_g1_compress, in96, 96, 48)
    def g2_uncompress(self, in96): return self._recode(lib().blsgpu_g2_uncompress, in96, 96, 192)
    def g2_compress(self, in192): return self._recode(lib().blsgpu_g2_compress, in192, 192, 96)
    def pool_create(self, pks48):
        a = _u8(pks48); n = a.size // 48; st = np.empty(n, np.uint8); h = ctypes.c_int(-1)
        self._ck(lib().blsgpu_pool_create(self._h, _p(a), _sz(n), ctypes.byref(h), _p(st))); return h.value, st
    def pool_free(self, handle): lib().blsgpu_pool_free(self._h, int(handle))
    def pool_fast_aggregate_verify_ptr(self, handle, idx, bitmap, k, msg, sig, ncomm, status, agg=None):
        self._ck(lib().blsgpu_pool_fast_aggregate_verify(self._h, int(handle), _p(idx), _p(bitmap), _sz(k), _p(msg), _p(sig), _sz(ncomm), _p(status), _p(agg)))
    def pool_fast_aggregate_verify(self, handle, idx, k, msg32, sig96, bitmap=None, want_agg=False):
        ix = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1); m = _u8(msg32); sg = _u8(sig96); nc = sg.size // 96
        st = np.empty(nc, np.uint8); agg = np.empty(48 * nc, np.uint8) if want_agg else None
        bm = np.ascontiguousarray(bitmap, dtype=np.uint64) if bitmap is not None else None
        _need("sig96", sg, 96 * nc); _need("msg32", m, 32 * nc); _need("idx", ix, 4 * nc * k); _need("bitmap", bm, 8 * ((nc * k + 63) // 64))
        self.pool_fast_aggregate_verify_ptr(handle, ix, bm, k, m, sg, nc, st, agg)
        return (st, agg) if want_agg else st
    # ---- signature sets: set s = keys [key_off[s], key_off[s+1]) of the flat list, one message, one signature
    def verify_signature_sets_ptr(self, pks, key_off, bitmap, msg, msg_off, sig, nsets, seed16, status, ok_bitmap=None):
        """-> number of sets re-run per set (raw pointers: numpy arrays in host mode, ints in device mode)"""
        rerun = ctypes.c_uint64(0)
        self._ck(lib().blsgpu_verify_signature_sets(self._h, _p(pks), _p(key_off), _p(bitmap), _p(msg), _p(msg_off), _p(sig), _sz(nsets), _p(seed16), _p(status), _p(ok_bitmap), ctypes.byref(rerun)))
        return int(rerun.value)
    def pool_verify_signature_sets_ptr(self, handle, idx, key_off, bitmap, msg, msg_off, sig, nsets, seed16, status, ok_bitmap=None):
        rerun = ctypes.c_uint64(0)
        self._ck(lib().blsgpu_pool_verify_signature_sets(self._h, int(handle), _p(idx), _p(key_off), _p(bitmap), _p(msg), _p(msg_off), _p(sig), _sz(nsets), _p(seed16), _p(status), _p(ok_bitmap), ctypes.byref(rerun)))
        return int(rerun.value)
    @staticmethod
    def _sets_args(key_off, msgs, sig96, seed16, bitmap, fixed32):
        ko = np.ascontiguousarray(key_off, dtype=np.uint32).reshape(-1); sg = _u8(sig96); n = sg.size // 96
        _need("sig96", sg, 96 * n)
        if ko.size != n + 1 or ko[0] != 0 or np.any(np.diff(ko.astype(np.int64)) < 0): raise ValueError("key_off must hold nsets + 1 non-decreasing offsets starting at 0")
        if fixed32: flat, off = _u8(msgs), None; _need("msgs", flat, 32 * n)
        else:
            if len(msgs) != n: raise ValueError(f"{len(msgs)} messages for {n} signatures")
            flat, off = pack_msgs(msgs)
        nk = int(ko[-1]); bm = np.ascontiguousarray(bitmap, dtype=np.uint64) if bitmap is not None else None; _need("bitmap", bm, 8 * ((nk + 63) // 64))
        seed = None
        if seed16 is not None: seed = _u8(seed16); _need("seed16", seed, 16)
        return ko, flat, off, sg, n, nk, bm, seed
    def verify_signature_sets(self, pks48, key_off, msgs, sig96, seed16=None, bitmap=None, fixed32=False):
        """set s = keys pks48[key_off[s]:key_off[s+1]] (48 bytes each), message msgs[s] (or 32 bytes each with fixed32), signature s.
        seed16 None: one pairing check per set; else per-piece random linear combinations with the exact outcome.
        -> (status uint8[nsets], ok_bitmap uint64[ceil(nsets/64)], sets re-run per set)"""
        ko, flat, off, sg, n, nk, bm, seed = self._sets_args(key_off, msgs, sig96, seed16, bitmap, fixed32)
        pk = _u8(pks48); _need("pks48", pk, 48 * nk)
        st = np.empty(max(n, 1), np.uint8); ok = np.zeros(max((n + 63) // 64, 1), np.uint64)
        rerun = self.verify_signature_sets_ptr(pk, ko, bm, flat, off, sg, n, seed, st, ok)
        return st[:n], ok[:(n + 63) // 64], rerun
    def pool_verify_signature_sets(self, handle, idx, key_off, msgs, sig96, seed16=None, bitmap=None, fixed32=False):
        """verify_signature_sets with the keys as indices into a resident pool (pool_create)"""
        ko, flat, off, sg, n, nk, bm, seed = self._sets_args(key_off, msgs, sig96, seed16, bitmap, fixed32)
        ix = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1); _need("idx", ix, 4 * nk)
        st = np.empty(max(n, 1), np.uint8); ok = np.zeros(max((n + 63) // 64, 1), np.uint64)
        rerun = self.pool_verify_signature_sets_ptr(handle, ix, ko, bm, flat, off, sg, n, seed, st, ok)
        return st[:n], ok[:(n + 63) // 64], rerun
    def hash_to_g2(self, msgs):
        flat, off = pack_msgs(msgs); out = np.empty(96 * len(msgs), np.uint8); self.hash_to_g2_ptr(flat, off, len(msgs), out); return out
    def g1_aggregate(self, pts48, seg_off):
        a = _u8(pts48); seg = np.ascontiguousarray(seg_off, dtype=np.uint32); ns = seg.size - 1
        out = np.empty(48 * ns, np.uint8); st = np.empty(ns, np.uint8)
        if ns < 0 or (ns > 0 and (np.any(np.diff(seg.astype(np.int64)) < 0) or seg[0] != 0)): raise ValueError("seg_off must start at 0 and be non-decreasing")
        _need("pts48", a, 48 * int(seg[-1]) if ns >= 0 and seg.size else 0)
        self._ck(lib().blsgpu_g1_aggregate(self._h, _p(a), _p(seg), _sz(ns), _p(out), _p(st))); return out, st
    def g2_aggregate(self, pts96, seg_off):
        a = _u8(pts96); seg = np.ascontiguousarray(seg_off, dtype=np.uint32); ns = seg.size - 1
        out = np.empty(96 * ns, np.uint8); st = np.empty(ns, np.uint8)
        if ns < 0 or (ns > 0 and (np.any(np.diff(seg.astype(np.int64)) < 0) or seg[0] != 0)): raise ValueError("seg_off must start at 0 and be non-decreasing")
        _need("pts96", a, 96 * int(seg[-1]) if ns >= 0 and seg.size else 0)
        self._ck(lib().blsgpu_g2_aggregate(self._h, _p(a), _p(seg), _sz(ns), _p(out), _p(st))); return out, st
    def deserialize_g1(self, in48):
        a = _u8(in48); n = a.size // 48; st = np.empty(n, np.uint8); self._ck(lib().blsgpu_deserialize_g1(self._h, _p(a), _sz(n), _p(st))); return st
    def deserialize_g2(self, in96):
        a = _u8(in96); n = a.size // 96; st = np.empty(n, np.uint8); self._ck(lib().blsgpu_deserialize_g2(self._h, _p(a), _sz(n), _p(st))); return st
    def sk_to_pk(self, sk_le):
        sk = _u8(sk_le); n = sk.size // 32; out = np.empty(48 * n, np.uint8); st = np.empty(n, np.uint8)
        self._ck(lib().blsgpu_sk_to_pk_batch(self._h, _p(sk), _sz(n), _p(out), _p(st))); return out, st
    def sign(self, sk_le, msgs, fixed32=False):
        sk = _u8(sk_le); n = sk.size // 32
        if fixed32: flat, off = _u8(msgs), None
        else: flat, off = pack_msgs(msgs)
        _need("sk32", sk, 32 * n)
        if fixed32: _need("msgs", flat, 32 * n)
        elif len(msgs) != n: raise ValueError(f"{len(msgs)} messages for {n} secret keys")
        out = np.empty(96 * n, np.uint8); st = np.empty(n, np.uint8)
        self._ck(lib().blsgpu_sign_batch(self._h, _p(sk), _p(flat), _p(off), _sz(n), _p(out), _p(st))); return out, st
    def pairing_gt(self, g1_48, g2_96, npairs):
        a = _u8(g1_48); b = _u8(g2_96); nprod = a.size // 48 // npairs; _need("g1_48", a, 48 * npairs * nprod); _need("g2_96", b, 96 * npairs * nprod); out = np.empty(576 * nprod, np.uint8); st = np.empty(nprod, np.uint8)
        self._ck(lib().blsgpu_pairing_gt(self._h, _p(a), _p(b), _sz(npairs), _sz(nprod), _p(out), _p(st))); return out.reshape(nprod, 576), st
    def gt_fold(self, parts):
        a = _u8(parts); out = np.empty(576, np.uint8); self._ck(lib().blsgpu_gt_fold(self._h, _p(a), _sz(a.size // 576), _p(out))); return out
    def fp_mul_raw(self, a, b, reps=1):
        a = _u8(a); b = _u8(b); n = a.size // 48; out = np.empty(48 * n, np.uint8)
        self._ck(lib().blsgpu_fp_mul_raw(self._h, _p(a), _p(b), _sz(n), _p(out), int(reps))); return out
    def imad_peak(self, mode=0):
        v = ctypes.c_double(); ms = ctypes.c_double(); self._ck(lib().blsgpu_imad_peak(self._h, int(mode), ctypes.byref(v), ctypes.byref(ms))); return v.value, ms.value
    def r1cs_load(self, rowptr, col, coeff48, nrows, ncols):
        rp = [np.ascontiguousarray(x, dtype=np.uint64) for x in rowptr]; cl = [np.ascontiguousarray(x, dtype=np.uint32) for x in col]
        cf = [np.ascontiguousarray(x, dtype=np.uint8) for x in coeff48]; P3 = _vp * 3; h = ctypes.c_int(-1)
        for m in range(3):
            if rp[m].size != nrows + 1: raise ValueError(f"rowptr[{m}] must hold nrows + 1 entries")
            nnz = int(rp[m][-1])
            if cl[m].size < nnz or cf[m].size < 48 * nnz: raise ValueError(f"matrix {m}: rowptr announces {nnz} non-zeros, col / coeff48 hold fewer")
        self._ck(lib().blsgpu_r1cs_load(self._h, P3(*[_p(x) for x in rp]), P3(*[_p(x) for x in cl]), P3(*[_p(x) for x in cf]), _sz(nrows), _sz(ncols), ctypes.byref(h)))
        return h.value
    def r1cs_check(self, handle, z48, nwit, nrows):
        z = _u8(z48); words = (nrows + 63) // 64; bits = np.zeros(nwit * words, np.uint64); allsat = np.zeros(nwit, np.uint8)
        if nwit and z.size % (48 * nwit): raise ValueError("z48 must hold nwit * ncols * 48 bytes")
        self._ck(lib().blsgpu_r1cs_check(self._h, int(handle), _p(z), _sz(nwit), _p(bits), _p(allsat))); return bits.reshape(nwit, words), allsat
    def r1cs_check_ptr(self, handle, z, nwit, bits, allsat): self._ck(lib().blsgpu_r1cs_check(self._h, int(handle), _p(z), _sz(nwit), _p(bits), _p(allsat)))
    def r1cs_free(self, handle): lib().blsgpu_r1cs_free(self._h, int(handle))
    def r1cs_load_file(self, path):
        """-> (handle, dict(nrows, ncols, ninstance, nwit)) from a BLSR1CS1 file (gadget.write_r1cs_file / rust/examples/export_r1cs.rs)"""
        h = ctypes.c_int(-1); shape = (ctypes.c_uint64 * 4)()
        self._ck(lib().blsgpu_r1cs_load_file(self._h, os.fsencode(path), ctypes.byref(h), shape))
        return h.value, dict(zip(("nrows", "ncols", "ninstance", "nwit"), [int(x) for x in shape]))
    def r1cs_check_file(self, handle, path, first, count, nrows):
        words = (nrows + 63) // 64; bits = np.zeros(max(count, 1) * words, np.uint64); allsat = np.zeros(max(count, 1), np.uint8)
        self._ck(lib().blsgpu_r1cs_check_file(self._h, int(handle), os.fsencode(path), _sz(first), _sz(count), _p(bits), _p(allsat)))
        return bits[:count * words].reshape(count, words), allsat[:count]
    def r1cs_row_classes(self, handle):
        c = (ctypes.c_uint64 * 4)(); self._ck(lib().blsgpu_r1cs_row_classes(self._h, int(handle), c))
        return dict(zip(("truth_table", "generic", "long", "segments"), [int(x) for x in c]))
    # ---- GPU witness generation (program from bls_verify_gadget_b200.gadget.verify_program)
    def witness_load(self, program):
        """program: the dict of gadget.verify_program (with its level order: the replay runs level by level)"""
        r = np.ascontiguousarray(program["rules16"], dtype=np.uint8); lp = np.ascontiguousarray(program["lc_ptr"], dtype=np.uint64)
        lc = np.ascontiguousarray(program["lc_col"], dtype=np.uint32); cf = np.ascontiguousarray(program["lc_coef48"], dtype=np.uint8)
        od = np.ascontiguousarray(program["order"], dtype=np.uint32); lv = np.ascontiguousarray(program["level_ptr"], dtype=np.uint64)
        h = ctypes.c_int(-1); nkeys = int(program.get("nkeys", 0))
        args = (self._h, _p(r), _p(lp), _p(lc), _p(cf), _sz(r.size // 16), _sz(program["nvars"]), _sz(lp.size - 1), _sz(lc.size), _p(od), _p(lv), _sz(lv.size - 1))
        if nkeys: self._ck(lib().blsgpu_witness_load_aggregate(*args, _sz(nkeys), ctypes.byref(h)))      # an aggregate_verify program (gadget.aggregate_verify_program)
        else: self._ck(lib().blsgpu_witness_load(*args, ctypes.byref(h)))
        return h.value
    def witness_shape(self, handle):
        c = (ctypes.c_uint64 * 4)(); self._ck(lib().blsgpu_witness_shape(self._h, int(handle), c))
        return dict(zip(("light_rules", "light_levels", "field_levels", "integer_slots"), [int(x) for x in c]))
    def witness_msg_len(self, handle):
        L = int(lib().blsgpu_witness_msg_len(self._h, int(handle)))
        if L < 0: raise BlsGpuError("bad witness program handle")
        return L
    def witness_gen(self, handle, pk48, msg, sig96, nvars):
        """msg: n x L bytes, L = witness_msg_len(handle) (the message length the program was recorded with)"""
        pk = _u8(pk48); m = _u8(msg); sg = _u8(sig96); n = sg.size // 96
        _need("sig96", sg, 96 * n); _need("pk48", pk, 48 * n); _need("msg", m, self.witness_msg_len(handle) * n)
        z = np.empty(n * nvars * 48, np.uint8); st = np.empty(n, np.uint8)
        self._ck(lib().blsgpu_witness_gen(self._h, int(handle), _p(pk), _p(m), _p(sg), _sz(n), _p(z), _p(st))); return z.reshape(n, nvars * 48), st
    def witness_gen_ptr(self, handle, pk, msg, sig, n, z, status=None): self._ck(lib().blsgpu_witness_gen(self._h, int(handle), _p(pk), _p(msg), _p(sig), _sz(n), _p(z), _p(status)))
    def witness_check(self, wit_handle, r1cs_handle, pk, msgs32, sig, nrows):
        """host buffers: generation + satisfaction check in one call -> (bits uint64[n, words], all_sat uint8[n], status uint8[n])"""
        pk = _u8(pk); sg = _u8(sig); m = _u8(msgs32); n = pk.size // 48; words = (nrows + 63) // 64
        _need("pk", pk, 48 * n); _need("sig", sg, 96 * n); _need("msgs", m, self.witness_msg_len(wit_handle) * n)
        bits = np.zeros((n, words), np.uint64); allsat = np.zeros(n, np.uint8); st = np.empty(n, np.uint8)
        self._ck(lib().blsgpu_witness_check(self._h, int(wit_handle), int(r1cs_handle), _p(pk), _p(m), _p(sg), _sz(n), _p(bits), _p(allsat), _p(st))); return bits, allsat, st
    def witness_check_ptr(self, wit_handle, r1cs_handle, pk, msg, sig, n, bits, allsat=None, status=None):
        self._ck(lib().blsgpu_witness_check(self._h, int(wit_handle), int(r1cs_handle), _p(pk), _p(msg), _p(sig), _sz(n), _p(bits), _p(allsat), _p(status)))
    def witness_gen_aggregate(self, handle, pks48, bitmap, msg, sig96, nvars, nkeys):
        """aggregate_verify circuit: pks48 n x nkeys x 48, bitmap n x nkeys bytes, msg n x L, sig96 n x 96 -> (z [n, nvars * 48], status [n])"""
        pk = _u8(pks48); bm = np.ascontiguousarray(bitmap, dtype=np.uint8).reshape(-1); m = _u8(msg); sg = _u8(sig96); n = sg.size // 96
        _need("sig96", sg, 96 * n); _need("pks48", pk, 48 * n * nkeys); _need("bitmap", bm, n * nkeys); _need("msg", m, self.witness_msg_len(handle) * n)
        z = np.empty(n * nvars * 48, np.uint8); st = np.empty(n, np.uint8)
        self._ck(lib().blsgpu_witness_gen_aggregate(self._h, int(handle), _p(pk), _p(bm), _p(m), _p(sg), _sz(n), _p(z), _p(st))); return z.reshape(n, nvars * 48), st
    def witness_check_aggregate(self, wit_handle, r1cs_handle, pks48, bitmap, msg, sig96, nrows, nkeys):
        pk = _u8(pks48); bm = np.ascontiguousarray(bitmap, dtype=np.uint8).reshape(-1); m = _u8(msg); sg = _u8(sig96); n = sg.size // 96; words = (nrows + 63) // 64
        _need("sig96", sg, 96 * n); _need("pks48", pk, 48 * n * nkeys); _need("bitmap", bm, n * nkeys); _need("msg", m, self.witness_msg_len(wit_handle) * n)
        bits = np.zeros((n, words), np.uint64); allsat = np.zeros(n, np.uint8); st = np.empty(n, np.uint8)
        self._ck(lib().blsgpu_witness_check_aggregate(self._h, int(wit_handle), int(r1cs_handle), _p(pk), _p(bm), _p(m), _p(sg), _sz(n), _p(bits), _p(allsat), _p(st))); return bits, allsat, st
    def witness_free(self, handle): lib().blsgpu_witness_free(self._h, int(handle))


class MultiContext:
    """Every GPU of the box behind one handle (blsgpu_create_multi): the batch is sharded contiguously across the devices, the
    ok-bitmap shards and the GT partials are all-gathered with NCCL inside the library and folded on every device.  Host buffers in,
    host buffers out -- the single-process counterpart of bench.py's torchrun path."""
    def __init__(self, devices=None):
        self._h = _vp()
        dev = (ctypes.c_int * len(devices))(*devices) if devices else None
        rc = lib().blsgpu_create_multi(ctypes.byref(self._h), dev, len(devices) if devices else 0)
        if rc != 0:
            self._h = None
            raise BlsGpuError(f"blsgpu_create_multi failed (rc={rc}): no usable sm_100 CUDA device, bad device list, or NCCL not loadable -- there is no CPU fallback")
    @property
    def ndev(self): return int(lib().blsgpu_multi_ndev(self._h))
    @property
    def nccl_version(self): return int(lib().blsgpu_multi_nccl_version(self._h))
    def close(self):
        if getattr(self, "_h", None): lib().blsgpu_destroy_multi(self._h); self._h = None
    def __del__(self):
        try: self.close()
        except Exception: pass
    def _ck(self, rc):
        if rc != 0: raise BlsGpuError(f"rc={rc}: {lib().blsgpu_multi_last_error(self._h).decode()}")
    def verify_ptr(self, pk, msg, off, sig, n, status, bitmap=None, gt=None):
        self._ck(lib().blsgpu_multi_verify_batch(self._h, _p(pk), _p(msg), _p(off), _p(sig), _sz(n), _p(status), _p(bitmap), _p(gt)))
    def verify(self, pk48, msgs, sig96, fixed32=False):
        """-> (status uint8[n], ok_bitmap uint64[ceil(n/64)], gt uint8[576])"""
        pk = _u8(pk48); sg = _u8(sig96); n = sg.size // 96
        if fixed32: flat, off = _u8(msgs), None
        else: flat, off = pack_msgs(msgs)
        _need("sig96", sg, 96 * n); _need("pk48", pk, 48 * n)
        if fixed32: _need("msgs", flat, 32 * n)
        elif len(msgs) != n: raise ValueError(f"{len(msgs)} messages for {n} signatures")
        st = np.empty(max(n, 1), np.uint8); bm = np.zeros(max((n + 63) // 64, 1), np.uint64); gt = np.zeros(576, np.uint8)
        self.verify_ptr(pk, flat, off, sg, n, st, bm, gt)
        return st[:n], bm[:(n + 63) // 64], gt
    def peek(self, i, n):
        bm = np.zeros(max((n + 63) // 64, 1), np.uint64); gt = np.zeros(576, np.uint8)
        self._ck(lib().blsgpu_multi_peek(self._h, int(i), _sz(n), _p(bm), _p(gt))); return bm[:(n + 63) // 64], gt
