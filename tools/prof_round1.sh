set -x
ncu --set full --clock-control none -k regex:k_euclid_tiles -c 1 -o gpurun_out/prof_euclid_r1 python tools/bench_configs.py --quick --only euclid > gpurun_out/ncu_euclid.log 2>&1
ncu --set full --clock-control none -k regex:"k_mash_filter|k_mash_pairs" -c 2 -o gpurun_out/prof_mash_r1 python tools/bench_configs.py --only mash > gpurun_out/ncu_mash.log 2>&1
ncu --set full --clock-control none -k regex:k_count -c 1 -o gpurun_out/prof_count_k8_r1 python bench.py --steps 1 --warmup 0 --no-e2e --no-cpu-baseline --k 8 --n 20 > gpurun_out/ncu_count_k8.log 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none -s 3 -c 900 --csv --log-file gpurun_out/launches_r1_final.csv python bench.py --steps 1 --warmup 0 --no-e2e --no-cpu-baseline > gpurun_out/ncu_bench_final.log 2>&1
ls -la gpurun_out | tail -8
