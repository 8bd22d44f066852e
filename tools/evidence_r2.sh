#!/bin/bash
# Round-2 final evidence on ONE B200: GPU tests, bench lines of every BASELINE config that fits one GPU
# (C4 / C5 as their per-GPU shard), the reference arm, ncu launch lists and `--set full` captures of the tcgen05 kernels.
# Outputs land in $OUT/r2f_* (default evidence_out/).
set -x
OUT=${OUT:-evidence_out}
mkdir -p "$OUT"
python -m pytest tests -q -m gpu -p no:cacheprovider > $OUT/r2f_pytest.txt 2>&1
tail -3 $OUT/r2f_pytest.txt
python bench.py --steps 60 --warmup 5 > $OUT/r2f_bench_c2.json 2> $OUT/r2f_bench_c2.err
python bench.py --steps 20 --warmup 5 --no-cpu-baseline > $OUT/r2f_bench_c2_steps20.json 2> /dev/null
SBR_NO_SIDE_STREAM=1 python bench.py --steps 20 --warmup 5 --no-cpu-baseline > $OUT/r2f_bench_c2_no_side_stream.json 2> /dev/null
python bench.py --impl reference --steps 3 --warmup 1 > $OUT/r2f_ref_c2.json 2> $OUT/r2f_ref_c2.err
python bench.py --config c3 --steps 10 --warmup 3 > $OUT/r2f_bench_c3.json 2> $OUT/r2f_bench_c3.err
python bench.py --config c4 --steps 8 --warmup 3 --no-cpu-baseline > $OUT/r2f_bench_c4_shard.json 2> $OUT/r2f_bench_c4.err
python bench.py --config c5 --steps 5 --warmup 3 --no-cpu-baseline > $OUT/r2f_bench_c5_shard.json 2> $OUT/r2f_bench_c5.err
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/r2f_launches_c2.csv \
    python bench.py --steps 3 --warmup 3 --no-cpu-baseline > /dev/null 2> $OUT/r2f_ncu1.err
timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -c 300 --csv --log-file $OUT/r2f_launches_c3.csv \
    python bench.py --config c3 --steps 2 --warmup 3 --no-cpu-baseline > /dev/null 2> $OUT/r2f_ncu2.err
timeout 600 ncu --set full --clock-control none --import-source on -k regex:"rnn_.*_tc_kernel|wgrad_tc|tc_gemm_kernel" -s 12 -c 7 -f -o $OUT/r2f_full_c2 \
    python bench.py --steps 3 --warmup 3 --no-cpu-baseline > /dev/null 2> $OUT/r2f_ncu3.err
SBR_SCAN_NO_COOP=1 timeout 900 ncu --set full --clock-control none --import-source on -k regex:"tc_scan_.*_kernel" -s 4 -c 4 -f -o $OUT/r2f_full_c3_scans \
    python bench.py --config c3 --steps 2 --warmup 3 --no-cpu-baseline > /dev/null 2> $OUT/r2f_ncu4.err
ls -la $OUT/ | grep r2f
for f in $OUT/r2f_bench_c2.json $OUT/r2f_bench_c2_steps20.json $OUT/r2f_bench_c2_no_side_stream.json $OUT/r2f_ref_c2.json $OUT/r2f_bench_c3.json $OUT/r2f_bench_c4_shard.json $OUT/r2f_bench_c5_shard.json; do echo $f; cut -c1-1400 $f; done

# Multi-GPU lines of the round (each on a machine with N B200s):
#   N=2: python -m pytest tests/test_gpu_e2e.py -k "two_rank or nccl"; torchrun --nproc-per-node 2 bench.py --gpus 2 --steps 20 --warmup 5 --no-cpu-baseline
#   N=4: torchrun --nproc-per-node 4 bench.py --gpus 4 [--config c4 --steps 8 --warmup 3] --no-cpu-baseline
#   N=8: torchrun --nproc-per-node 8 bench.py --gpus 8 [--config c5 --steps 5 --warmup 3] --no-cpu-baseline
#        (with NCCL_DEBUG=INFO for the NVLS line kept in profiles/r2f_nccl_info_8gpu.txt; NCCL prints to stdout)
# with torchrun = python -m torch.distributed.run --nnodes=1 --master-addr 127.0.0.1 --master-port <P>
