#!/usr/bin/env python3
"""bench_sets.py -- signature sets (blsgpu_verify_signature_sets / blsgpu_pool_verify_signature_sets) on one GPU; one JSON line per workload.

  (a) sync-committee shape: 2^14 sets of 512 resident-pool indices (pool of 2^16 keys), all-ones bitmap and a 2/3 bitmap (signatures over the
      selected keys): blsgpu_pool_fast_aggregate_verify against pool sets per set and pool sets in RLC mode.
  (b) attestation-aggregate shape: 2^15 sets of 16..512 compressed keys (sizes drawn from a seed), 32-byte messages: per set against RLC.
  (c) 2^20 one-key sets in RLC mode against blsgpu_verify_batch_rlc_bisect on the same triples.
Inputs are resident in HBM (device pointer mode); a step is one call, timed with CUDA events around `--steps` calls after `--warmup` calls.
Statuses of the compared calls must be identical (checked before timing).  The card's name and power limit are read in the same run.

  python bench_sets.py [--steps K] [--warmup W] [--workloads abc] [--profile]
"""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.abspath(__file__)); sys.path.insert(0, ROOT)
import numpy as np

R_ORDER = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
SEED = bytes(range(16))

def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else None

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3); ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="abc"); ap.add_argument("--profile", action="store_true", help="per-kernel times of one call of each form (torch.profiler, separate from the timed loop)")
    args = ap.parse_args()
    import torch
    from bls_verify_gadget_b200 import Context, synth, _lib
    dev = torch.device("cuda", 0); torch.cuda.set_device(dev)
    ctx = Context(0); stream = torch.cuda.current_stream(dev); ctx.set_stream(stream.cuda_stream)
    gpu = card(); lib_name = os.path.basename(_lib.SO_PATH)
    D = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)
    dseed = D(np.frombuffer(SEED, np.uint8))

    def timed(fn, n_units):
        for _ in range(args.warmup): fn()
        torch.cuda.synchronize(dev)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps): fn()
        e1.record(stream); torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / args.steps
        return {"ms_per_call": ms, "per_sec": n_units / (ms * 1e-3)}

    def kernels(fn):
        from torch.profiler import profile, ProfilerActivity
        fn(); torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            fn(); torch.cuda.synchronize(dev)
        tot = {}
        for e in p.events():
            if e.device_type.name == "CUDA": tot[e.name.split("(")[0].split("<")[0]] = tot.get(e.name.split("(")[0].split("<")[0], 0.0) + e.device_time_total / 1e3
        return dict(sorted(((k, round(v, 2)) for k, v in tot.items()), key=lambda kv: -kv[1])[:14])

    def emit(d):
        d.update({"gpu": gpu, "library": lib_name, "steps": args.steps, "warmup": args.warmup})
        print(json.dumps(d), flush=True)

    ctx.set_pointer_mode(False)
    if "a" in args.workloads:
        nsets, k, pool = 1 << 14, 512, 1 << 16
        sk = synth.fast_secret_keys(pool); pool_pk, st = ctx.sk_to_pk(sk); assert not st.any()
        ski = [int.from_bytes(sk[32 * i:32 * i + 32].tobytes(), "little") for i in range(pool)]
        rng = np.random.default_rng(0x5c)
        idx = rng.integers(0, pool, size=(nsets, k)).astype(np.uint32); msg = synth.fast_random_bytes(32 * nsets, 0x5d)
        h, _ = ctx.pool_create(pool_pk)
        ko = (np.arange(nsets + 1, dtype=np.uint64) * k).astype(np.uint32)
        for name, frac in (("all", 1.0), ("two_thirds", 2 / 3)):
            sel = np.ones((nsets, k), bool) if frac == 1.0 else rng.random((nsets, k)) < frac
            sums = [sum(ski[i] for i in idx[c][sel[c]]) % R_ORDER for c in range(nsets)]
            sig, st = ctx.sign(b"".join(s.to_bytes(32, "little") for s in sums), msg, fixed32=True); assert not st.any()
            bm = np.packbits(sel.reshape(-1), bitorder="little").view(np.uint64)
            d_idx, d_bm, d_msg, d_sig, d_ko = D(idx), D(bm), D(msg), D(sig), D(ko)
            outs = {m: torch.empty(nsets, dtype=torch.uint8, device=dev) for m in ("fav", "sets", "rlc")}
            ctx.set_pointer_mode(True)
            calls = {"fav": lambda: ctx.pool_fast_aggregate_verify_ptr(h, d_idx.data_ptr(), d_bm.data_ptr(), k, d_msg.data_ptr(), d_sig.data_ptr(), nsets, outs["fav"].data_ptr()),
                     "sets": lambda: ctx.pool_verify_signature_sets_ptr(h, d_idx.data_ptr(), d_ko.data_ptr(), d_bm.data_ptr(), d_msg.data_ptr(), None, d_sig.data_ptr(), nsets, None, outs["sets"].data_ptr()),
                     "rlc": lambda: ctx.pool_verify_signature_sets_ptr(h, d_idx.data_ptr(), d_ko.data_ptr(), d_bm.data_ptr(), d_msg.data_ptr(), None, d_sig.data_ptr(), nsets, dseed.data_ptr(), outs["rlc"].data_ptr())}
            for f in calls.values(): f()
            torch.cuda.synchronize(dev)
            ref = outs["fav"].cpu().numpy()
            assert not ref.any() and all(np.array_equal(o.cpu().numpy(), ref) for o in outs.values()), "statuses differ"
            res = {m: timed(f, nsets) for m, f in calls.items()}
            line = {"workload": f"a_sync_committee_{name}", "sets": nsets, "keys_per_set": k, "pool": pool, "selected_frac": float(sel.mean()), "unit": "sets/s", "results": res,
                    "rlc_over_per_set": res["rlc"]["per_sec"] / res["sets"]["per_sec"], "per_set_over_fav": res["sets"]["per_sec"] / res["fav"]["per_sec"]}
            if args.profile: line["kernel_ms"] = {m: kernels(f) for m, f in calls.items()}
            ctx.set_pointer_mode(False); emit(line)
        ctx.pool_free(h)
    if "b" in args.workloads:
        nsets, pool = 1 << 15, 1 << 16
        sk = synth.fast_secret_keys(pool, seed=0x6b); pool_pk, st = ctx.sk_to_pk(sk); assert not st.any()
        ski = [int.from_bytes(sk[32 * i:32 * i + 32].tobytes(), "little") for i in range(pool)]
        rng = np.random.default_rng(0x6c); sizes = rng.integers(16, 513, size=nsets)
        ko = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint32); idx = rng.integers(0, pool, size=int(ko[-1]))
        keys = pool_pk.reshape(pool, 48)[idx]; msg = synth.fast_random_bytes(32 * nsets, 0x6d)
        sums = [sum(ski[i] for i in idx[ko[s]:ko[s + 1]]) % R_ORDER for s in range(nsets)]
        sig, st = ctx.sign(b"".join(s.to_bytes(32, "little") for s in sums), msg, fixed32=True); assert not st.any()
        d_pk, d_ko, d_msg, d_sig = D(keys), D(ko), D(msg), D(sig)
        outs = {m: torch.empty(nsets, dtype=torch.uint8, device=dev) for m in ("sets", "rlc")}
        ctx.set_pointer_mode(True)
        calls = {"sets": lambda: ctx.verify_signature_sets_ptr(d_pk.data_ptr(), d_ko.data_ptr(), None, d_msg.data_ptr(), None, d_sig.data_ptr(), nsets, None, outs["sets"].data_ptr()),
                 "rlc": lambda: ctx.verify_signature_sets_ptr(d_pk.data_ptr(), d_ko.data_ptr(), None, d_msg.data_ptr(), None, d_sig.data_ptr(), nsets, dseed.data_ptr(), outs["rlc"].data_ptr())}
        for f in calls.values(): f()
        torch.cuda.synchronize(dev)
        ref = outs["sets"].cpu().numpy(); assert not ref.any() and np.array_equal(outs["rlc"].cpu().numpy(), ref), "statuses differ"
        res = {m: timed(f, nsets) for m, f in calls.items()}
        line = {"workload": "b_attestation_aggregates", "sets": nsets, "keys": int(ko[-1]), "keys_per_set": "16..512 uniform (seeded)", "unit": "sets/s", "results": res,
                "rlc_over_per_set": res["rlc"]["per_sec"] / res["sets"]["per_sec"]}
        if args.profile: line["kernel_ms"] = {m: kernels(f) for m, f in calls.items()}
        ctx.set_pointer_mode(False); emit(line)
        del d_pk
    if "c" in args.workloads:
        n = 1 << 20
        pk, msg, sig, _ = synth.verify_batch_inputs(ctx, n, every=10 ** 9)
        ko = np.arange(n + 1, dtype=np.uint32)
        d_pk, d_ko, d_msg, d_sig = D(pk), D(ko), D(msg), D(sig)
        outs = {m: torch.empty(n, dtype=torch.uint8, device=dev) for m in ("sets_rlc", "bisect")}
        ctx.set_pointer_mode(True)
        lib = _lib.lib(); import ctypes
        calls = {"sets_rlc": lambda: ctx.verify_signature_sets_ptr(d_pk.data_ptr(), d_ko.data_ptr(), None, d_msg.data_ptr(), None, d_sig.data_ptr(), n, dseed.data_ptr(), outs["sets_rlc"].data_ptr()),
                 "bisect": lambda: ctx._ck(lib.blsgpu_verify_batch_rlc_bisect(ctx._h, ctypes.c_void_p(d_pk.data_ptr()), ctypes.c_void_p(d_msg.data_ptr()), None, ctypes.c_void_p(d_sig.data_ptr()),
                                                                             ctypes.c_size_t(n), ctypes.c_void_p(dseed.data_ptr()), ctypes.c_void_p(outs["bisect"].data_ptr()), None, None))}
        for f in calls.values(): f()
        torch.cuda.synchronize(dev)
        ref = outs["bisect"].cpu().numpy(); assert not ref.any() and np.array_equal(outs["sets_rlc"].cpu().numpy(), ref), "statuses differ"
        res = {m: timed(f, n) for m, f in calls.items()}
        line = {"workload": "c_one_key_sets_vs_rlc_bisect", "sets": n, "unit": "sets/s", "results": res, "sets_over_bisect": res["sets_rlc"]["per_sec"] / res["bisect"]["per_sec"]}
        if args.profile: line["kernel_ms"] = {m: kernels(f) for m, f in calls.items()}
        ctx.set_pointer_mode(False); emit(line)
    ctx.close()

if __name__ == "__main__":
    main()
