set -x
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/r2c_pytest.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2c_pytest.log
tail -5 gpurun_out/r2c_pytest.log
export GMSB_KCLIQUE_TRACE=1
timeout 300 python tools/kc_prof.py 22 6 > gpurun_out/r2c_kc_s22_k6.log 2>&1
timeout 400 python tools/kc_prof.py 20 7 > gpurun_out/r2c_kc_s20_k7.log 2>&1
unset GMSB_KCLIQUE_TRACE
