# round-2 final measurements on one GPU (the commands behind profiles/*_r02*)
set -x
( time python -m pytest tests -x -q -m gpu 2>&1 | tail -4 ) 2>&1
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
python bench.py > gpurun_out/bench_r02.json 2> gpurun_out/bench_r02.err; tail -2 gpurun_out/bench_r02.err; cut -c1-300 gpurun_out/bench_r02.json
python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/bench_reference_arm_r02.json 2>/dev/null; cut -c1-200 gpurun_out/bench_reference_arm_r02.json
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/launches_r02.csv python bench.py --steps 2 --warmup 1 --skip-extra --no-cpu > gpurun_out/launches_r02.log 2>&1; tail -1 gpurun_out/launches_r02.log | cut -c1-120
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"k_r1cs|k_witness" -c 200 --csv --log-file gpurun_out/launches_r1cs_r02.csv python bench_r1cs.py --steps 1 --warmup 1 --per-gpu 128 --no-cpu > gpurun_out/launches_r1cs_r02.log 2>&1; tail -1 gpurun_out/launches_r1cs_r02.log | cut -c1-120
mkdir -p /tmp/ncu
ncu --set full --clock-control none --import-source on -k regex:"^k_decode_g1|^k_decode_g2|^k_hash_to_g2|^k_miller$|^k_final_exp" -c 6 -o /tmp/ncu/stage python bench.py --n 65536 --lanes 1 --steps 1 --warmup 3 --skip-extra --no-cpu > /dev/null 2>&1
python profiles/tools/ncu_executed.py 65536 /tmp/ncu/stage.ncu-rep > gpurun_out/ncu_r02_executed.json; grep -c imad_wide gpurun_out/ncu_r02_executed.json
ncu -i /tmp/ncu/stage.ncu-rep --page raw --csv > gpurun_out/ncu_r02_stage_raw.csv 2>/dev/null
ncu --set full --clock-control none --import-source on -k regex:"k_r1cs_long_rows|k_r1cs_transpose|k_r1cs_lut$|k_r1cs_rows_list|k_witness_light|k_witness_levels" -c 8 -o /tmp/ncu/r1 python bench_r1cs.py --steps 1 --warmup 1 --per-gpu 64 --no-cpu > /dev/null 2>&1
ncu -i /tmp/ncu/r1.ncu-rep --page raw --csv > gpurun_out/ncu_r02_r1cs_raw.csv 2>/dev/null
python bench_configs.py --cfg 2r,5 --steps 2 > gpurun_out/bench_configs_r02.jsonl 2>/dev/null; cut -c1-200 gpurun_out/bench_configs_r02.jsonl
python profiles/tools/wit_bench.py 2048 2>&1 | grep -E "witness_|matches" | tail -2
ls -la gpurun_out | head -30
