set -x
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/r2e_pytest.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2e_pytest.log
tail -5 gpurun_out/r2e_pytest.log
