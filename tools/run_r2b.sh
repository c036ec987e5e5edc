set -x
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/r2b_pytest.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2b_pytest.log
tail -5 gpurun_out/r2b_pytest.log
export GMSB_KCLIQUE_TRACE=1
timeout 300 python tools/kc_prof.py 22 5 > gpurun_out/r2b_kc_s22_k5.log 2>&1
timeout 300 python tools/kc_prof.py 22 6 > gpurun_out/r2b_kc_s22_k6.log 2>&1
timeout 400 python tools/kc_prof.py 20 7 > gpurun_out/r2b_kc_s20_k7.log 2>&1
unset GMSB_KCLIQUE_TRACE
timeout 600 ncu --set full --clock-control none --import-source on -k regex:"k_plan_scatter|k_plan_count|k_sort_mid|k_sort_big|k_relabel_count|k_emit_sorted" -c 6 \
    -o gpurun_out/r2b_prof_prep python tools/e2e_trace.py --scale 24 --reps 1 > gpurun_out/r2b_prof_prep.log 2>&1
ls -la gpurun_out/r2b_prof_prep.ncu-rep
