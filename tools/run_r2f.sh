set -x
mkdir -p gpurun_out
nvidia-smi -L
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/r2f_pytest.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2f_pytest.log
tail -5 gpurun_out/r2f_pytest.log
GMSB_TC_TRACE=1 timeout 300 python tools/e2e_trace.py --scale 24 --reps 2 --orient 1 > gpurun_out/r2f_e2e_trace.jsonl 2> gpurun_out/r2f_e2e_trace.err
cat gpurun_out/r2f_e2e_trace.jsonl; grep -A12 "rep 1" gpurun_out/r2f_e2e_trace.err
timeout 600 python bench.py --steps 5 --warmup 3 --kclique '4,5' > gpurun_out/r2f_bench_1gpu.json 2> gpurun_out/r2f_bench_1gpu.err; tail -3 gpurun_out/r2f_bench_1gpu.err
cut -c1-1500 gpurun_out/r2f_bench_1gpu.json
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus 2 --steps 5 --warmup 3 --kclique '4,5' > gpurun_out/r2f_bench_2gpu.json 2> gpurun_out/r2f_bench_2gpu.err; tail -3 gpurun_out/r2f_bench_2gpu.err
cut -c1-600 gpurun_out/r2f_bench_2gpu.json
GMSB_DEVICES=0,1 timeout 300 oracle/_ref/dropin_tc -g kronecker 18 --deg 16 -n 2 -v > gpurun_out/r2f_dropin_2gpu.log 2>&1; grep "@@@\|devices" gpurun_out/r2f_dropin_2gpu.log
