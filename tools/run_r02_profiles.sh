#!/bin/bash
# Round-2 evidence in one gpurun call: GPU tests, the bench line, the ncu launch list of the same bench command and one
# ncu --set full capture of the dominant kernel (conv_ru2_kernel) plus the training step's SnakeBeta backward.
mkdir -p gpurun_out
python -m pytest tests -m gpu -x -q > gpurun_out/r02_gputest.log 2>&1; echo "pytest rc=$?"; tail -3 gpurun_out/r02_gputest.log
python bench.py --steps 20 --warmup 5 > gpurun_out/r02_bench.json 2> gpurun_out/r02_bench.err; echo "bench rc=$?"
python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/r02_bench_reference.json 2> gpurun_out/r02_bench_reference.err; echo "ref rc=$?"
ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file gpurun_out/r02_bench_launches_ncu.csv \
    python bench.py --steps 2 --warmup 1 --no-cpu-baseline --main-only > gpurun_out/r02_bench_under_ncu.log 2>&1; echo "ncu list rc=$?"
ncu --set full --clock-control none --import-source on -k regex:conv_ru2_kernel --launch-skip 30 --launch-count 1 \
    -o gpurun_out/r02_conv_ru2_bench_shape_B16 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --main-only > gpurun_out/r02_ncu_ru2.log 2>&1; echo "ncu ru2 rc=$?"
ncu --set full --clock-control none -k regex:snake_bwd_stream --launch-skip 130 --launch-count 1 \
    -o gpurun_out/r02_snake_bwd_stream python tools/prof_train.py 4 2 > gpurun_out/r02_ncu_sbs.log 2>&1; echo "ncu sbs rc=$?"
ncu --set full --clock-control none --import-source on -k regex:conv_umma2_kernel --launch-skip 41 --launch-count 1 \
    -o gpurun_out/r02_k1_c256_B16_fast python tools/prof_dec_once.py 16 > gpurun_out/r02_ncu_k1.log 2>&1; echo "ncu k1 rc=$?"
PROF_STEPS=1 python tools/prof_sao_b16.py 16 > gpurun_out/r02_step_profile_sao_b16.txt 2>&1
python tools/prof_o12_b1.py 128 1 > gpurun_out/r02_step_profile_o12_b1.txt 2>&1
python tools/prof_o12_b1.py 96 1 >> gpurun_out/r02_step_profile_o12_b1.txt 2>&1
python bench.py --workload train --steps 10 --warmup 3 > gpurun_out/r02_bench_train_n1.json 2>/dev/null
python bench.py --workload stream --steps 30 --warmup 5 > gpurun_out/r02_bench_stream.json 2>/dev/null
python bench.py --workload bigvgan --steps 6 > gpurun_out/r02_bench_bigvgan.json 2>/dev/null
nvidia-smi --query-gpu=name,clocks.max.sm,power.limit --format=csv > gpurun_out/r02_gpu_info.csv
