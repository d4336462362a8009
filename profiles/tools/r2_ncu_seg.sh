ncu --set full --clock-control none --import-source on -k regex:k_r1cs_rows_list -s 2 -c 2 -o gpurun_out/r2_rows_a python bench_configs.py --cfg 5r --steps 1 --scale 0.25 > gpurun_out/r2_ncu_rows.log 2>&1; tail -2 gpurun_out/r2_ncu_rows.log
ls -la gpurun_out/
