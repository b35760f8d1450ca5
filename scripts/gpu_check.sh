#!/bin/bash
# Run the GPU test groups as separate processes (a trapping kernel kills its CUDA context, not the others),
# then a short bench.  Logs land in gpurun_out/.
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
nvidia-smi --query-gpu=name,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
run() { name=$1; shift; timeout 900 python -m pytest tests -m gpu -q --timeout 600 -k "$@" > gpurun_out/test_$name.log 2>&1; echo "$name exit $?" >> gpurun_out/summary.txt; tail -3 gpurun_out/test_$name.log >> gpurun_out/summary.txt; }
: > gpurun_out/summary.txt
run raytile "sample_coarse or composite or resample"
run ops "positional or index_operator or resnetfc_operator or gather_encode"
run field_fp32 "field and fp32"
run field_bf16 "field and bf16"
run render "render or full_image"
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "smoke exit $?" >> gpurun_out/summary.txt
timeout 900 python bench.py --steps 5 --warmup 3 > gpurun_out/bench.log 2> gpurun_out/bench.err; echo "bench exit $?" >> gpurun_out/summary.txt
tail -1 gpurun_out/bench.log >> gpurun_out/summary.txt
cat gpurun_out/summary.txt
