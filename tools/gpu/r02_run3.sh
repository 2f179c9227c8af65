# round 2, run 3 (after the container was re-created): whole GPU suite, smoke, default bench
mkdir -p gpurun_out/r02
timeout 1500 python -m pytest tests -m gpu -x -q > gpurun_out/r02/pytest_run3.log 2>&1; echo "pytest rc=$?"
tail -15 gpurun_out/r02/pytest_run3.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python bench.py > gpurun_out/r02/bench_n1.json 2> gpurun_out/r02/bench_n1.err; echo "bench rc=$?"
tail -5 gpurun_out/r02/bench_n1.err
cut -c1-3000 gpurun_out/r02/bench_n1.json
