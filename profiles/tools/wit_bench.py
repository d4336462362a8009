import sys, os, time, numpy as np, torch
sys.path.insert(0, os.getcwd())
from bls_verify_gadget_b200 import Context, synth, gadget as G
dev = torch.device("cuda", 0); ctx = Context(0); stream = torch.cuda.current_stream(dev); ctx.set_stream(stream.cuda_stream)
n = int(sys.argv[1]) if len(sys.argv) > 1 else 512
pk, msg, sig, exp = synth.verify_batch_inputs(ctx, n, every=10**9, fast=True)
t0 = time.time(); prog = G.verify_program(pk[:48].tobytes(), msg[:32].tobytes(), sig[:96].tobytes()); nvars = prog["nvars"]; print("program s", round(time.time() - t0, 1), "nvars", nvars, "levels", prog["level_ptr"].size - 1)
h = ctx.witness_load(prog); print('split', ctx.witness_shape(h))
d_pk, d_msg, d_sig = (torch.from_numpy(x).to(dev) for x in (pk, msg, sig))
z = torch.empty(n * nvars * 48, dtype=torch.uint8, device=dev); st = torch.empty(n, dtype=torch.uint8, device=dev)
ctx.set_pointer_mode(True)
for rep in range(2):
  e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
  e0.record(stream); ctx.witness_gen_ptr(h, d_pk.data_ptr(), d_msg.data_ptr(), d_sig.data_ptr(), n, z.data_ptr(), st.data_ptr()); e1.record(stream); torch.cuda.synchronize()
  ms = e0.elapsed_time(e1); print(f"witness_gen n={n}: {ms:.1f} ms = {n / (ms * 1e-3):.0f} assignments/s")
if len(sys.argv) > 2:      # fused generation + check (the packed 0/1 view is live in this path)
    c = G.verify_circuit(pk[:48].tobytes(), msg[:32].tobytes(), sig[:96].tobytes()); mats = c.matrices(); ctx.set_pointer_mode(False)
    rh = ctx.r1cs_load([m[0] for m in mats], [m[1] for m in mats], [m[2] for m in mats], c.nrows, c.ncols); ctx.set_pointer_mode(True)
    bits = torch.zeros(n * ((c.nrows + 63) // 64), dtype=torch.int64, device=dev); al = torch.zeros(n, dtype=torch.uint8, device=dev)
    for rep in range(2):
      e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
      e0.record(stream); ctx.witness_check_ptr(h, rh, d_pk.data_ptr(), d_msg.data_ptr(), d_sig.data_ptr(), n, bits.data_ptr(), al.data_ptr(), st.data_ptr()); e1.record(stream); torch.cuda.synchronize()
      ms = e0.elapsed_time(e1); print(f"witness_check n={n}: {ms:.1f} ms = {n / (ms * 1e-3):.0f} assignments/s; all satisfied: {bool(al.all().item())}")
assert int(st.sum().item()) == 0
# check a couple against the host
zh, res = G.verify_witnesses([(pk[48*i:48*i+48].tobytes(), msg[32*i:32*i+32].tobytes(), sig[96*i:96*i+96].tobytes()) for i in (0, n - 1)], ncols=nvars)
zz = z.reshape(n, nvars * 48); assert np.array_equal(zz[0].cpu().numpy(), zh[0]) and np.array_equal(zz[n - 1].cpu().numpy(), zh[1]); print("matches host synthesis")
