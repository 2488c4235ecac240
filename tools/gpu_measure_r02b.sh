#!/bin/bash
# Second measurement pass of round 2: small-frame scheduling, the one-pair ncu table, training kernels.
mkdir -p gpurun_out
P=gpurun_out
python -m pytest tests/test_gpu_unet.py tests/test_gpu_train_step.py tests/test_gpu_conv_layers.py -q -s 2>&1 | grep -E "gradient rel|passed|failed|FAILED|Error|assert" | tail -30 > $P/r02b_pytest.log
python tools/profile_small.py > $P/r02_small_profile.json 2> $P/small.err
python tools/profile_small.py --bilinear > $P/r02_small_profile_bilinear.json 2>> $P/small.err
python bench.py --workload api256 --no-cpu-baseline > $P/r02_api256.json 2> $P/r02_api256.err
python bench.py --steps 20 --no-cpu-baseline > $P/r02b_bench.json 2> $P/r02b_bench.err
ncu --set full --clock-control none -k regex:"conv_|stem_mma" -c 22 -f -o /tmp/prof_fwd_r02 \
  python bench.py --steps 1 --warmup 0 --pairs 1 --no-cpu-baseline > $P/ncu_fwd.log 2>&1
python tools/summarize_ncu.py /tmp/prof_fwd_r02.ncu-rep > $P/r02_kernels_ncu_full.csv 2>> $P/ncu_fwd.log
ncu --set full --clock-control none -k regex:"wgrad_kernel|bn_relu_bwd" -c 40 -f -o /tmp/prof_trainb_r02 \
  python tools/bench_train.py --steps 1 --warmup 0 --skip-torch > $P/ncu_trainb.log 2>&1
python tools/summarize_ncu.py /tmp/prof_trainb_r02.ncu-rep > $P/r02_train_bwd_ncu_full.csv 2>> $P/ncu_trainb.log
du -sh $P; cat $P/r02b_pytest.log
