set -x
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/r2h_pytest.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2h_pytest.log
tail -5 gpurun_out/r2h_pytest.log
timeout 400 python tools/setops_bench.py --scale 22 --cpu-seconds 10 > gpurun_out/r2h_setops.jsonl 2> gpurun_out/r2h_setops.err; cat gpurun_out/r2h_setops.jsonl | cut -c1-420
timeout 600 ncu --set full --clock-control none -k regex:"k_kclique_lane_pair|k_kclique_lane_mid" -c 6 -o gpurun_out/r2h_prof_kc python tools/kc_prof.py 16 7 > gpurun_out/r2h_prof_kc.log 2>&1
ls -la gpurun_out/r2h_prof_kc.ncu-rep
timeout 300 python bench.py --steps 10 --warmup 3 --kclique '' > gpurun_out/r2h_bench_1gpu.json 2> gpurun_out/r2h_bench_1gpu.err; cut -c1-300 gpurun_out/r2h_bench_1gpu.json
