#!/bin/bash
# Round-2 GPU session: conv-stack check (timeline), full GPU test suite with the NEW kernels selected, bench
mkdir -p gpurun_out
TAG=${1:-r2h}
export SNB200_GENERATOR_BACKWARD=cuda
timeout -k 10 200 python tools/check_conv_stack.py > gpurun_out/${TAG}_check_cs.txt 2>&1; echo "check rc=$?"
timeout -k 10 1500 python -m pytest tests -m gpu -q --tb=short --timeout 300 -p no:cacheprovider > gpurun_out/${TAG}_pytest.log 2>&1; echo "pytest rc=$?" | tee -a gpurun_out/${TAG}_pytest.log
grep "MISMATCH\|ALL OK\|FAILED\|Error\|error" gpurun_out/${TAG}_check_cs.txt | head; grep -v "^b=" gpurun_out/${TAG}_check_cs.txt | grep "barrier done\|generator\|scale\|head"
tail -60 gpurun_out/${TAG}_pytest.log
