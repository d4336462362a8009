#!/bin/bash
# Alternating A/B of the verify benchmark (profiles/r03_sig_subgroup.md): the parent commit's library, this tree's, and this tree's
# built with -DBLS_MINB_DG2=3, three rounds, each run on the same seeded inputs with its outputs compared to the first run's.
# Expects build_var/parent.so (nvcc of the parent commit's bls_verify_gadget_b200/csrc/blsgpu.cu with _lib.NVCC_FLAGS),
# build_var/minb3.so (this tree, the same flags plus -DBLS_MINB_DG2=3) and the built tree; writes under out/ab.
mkdir -p out/ab
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee out/ab/gpu.txt
for r in 1 2 3; do
  for v in parent new minb3; do
    case $v in parent) so=build_var/parent.so;; new) so=bls_verify_gadget_b200/libblsgpu.so;; minb3) so=build_var/minb3.so;; esac
    BLSGPU_SO=$PWD/$so python bench.py --skip-extra --no-cpu --dump-outputs out/ab/dump_${v}_$r > out/ab/${v}_$r.out 2> out/ab/${v}_$r.err
    echo "$v round $r rc=$?"
    python -c "
import numpy as np, os, shutil
d, ref = 'out/ab/dump_${v}_$r', 'out/ab/dump_ref'
if not os.path.isdir(ref): shutil.copytree(d, ref)
print('  status / ok / gt identical to the first run:', all(np.array_equal(np.load(os.path.join(d, k + '.npy')), np.load(os.path.join(ref, k + '.npy'))) for k in ('status', 'ok', 'gt')))
shutil.rmtree(d)"
  done
done
python - <<'P'
import glob, json, os
for f in sorted(glob.glob("out/ab/*_[123].out")):
    j = json.loads([l for l in open(f) if l.startswith("{")][-1]); s = j["stage_ms"]
    print("%-10s value=%10.1f decode_g2=%7.2f miller=%7.2f sm=%s MHz" % (os.path.basename(f)[:-4], j["value"], s["decode_g2"], s["miller"], j["clocks"]["sm_mhz"]))
P
