set -x
python -m pytest tests -x -q -m gpu -k "witness or r1cs" 2>&1 | tail -3
BLSGPU_SO=build_var/wit_trace.so python profiles/tools/wit_trace.py 512 2>&1 | tail -24
python profiles/tools/wit_bench.py 512 fused 2>&1 | grep -E "witness_" | tail -3
echo "== default"; python bench_configs.py --cfg 5r --steps 3 --scale 0.5 2>&1 | python -c "import json,sys; d=json.loads(sys.stdin.readlines()[-1]); print(d['ms'], d['value'])"
for v in rows4 rows5; do echo "== r1_$v"; BLSGPU_SO=build_var/r1_$v.so python bench_configs.py --cfg 5r --steps 3 --scale 0.5 2>&1 | python -c "import json,sys; d=json.loads(sys.stdin.readlines()[-1]); print(d['ms'], d['value'])"; done
