#!/bin/bash
# end-of-round check: full GPU test-suite, smoke, benches (default, ViT-L, inference, reference arm)
mkdir -p gpurun_out
O=gpurun_out
timeout 1200 python -m pytest tests -q -m gpu -x --timeout 900 > $O/pytest_gpu_all.log 2>&1; echo "pytest -m gpu rc=$?"; tail -3 $O/pytest_gpu_all.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1; echo "smoke rc=$?"; tail -2 $O/smoke.log
timeout 400 python bench.py > $O/bench.json 2> $O/bench.err; echo "bench rc=$?"; cut -c1-260 $O/bench.json
timeout 300 python bench.py --config vitl384 --steps 10 --warmup 3 --no-cpu-baseline > $O/bench_vitl.json 2> $O/bench_vitl.err; echo "vitl rc=$?"; cut -c1-200 $O/bench_vitl.json
timeout 300 python bench.py --config vitb224-infer --steps 20 --warmup 3 > $O/bench_infer.json 2> $O/bench_infer.err; echo "infer rc=$?"
timeout 300 python bench.py --impl reference --steps 3 --warmup 1 > $O/bench_ref.json 2> $O/bench_ref.err; echo "reference rc=$?"; cut -c1-200 $O/bench_ref.json
