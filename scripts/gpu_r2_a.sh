# round 2, first GPU pass: parity suite + device A* tests + A* micro-benchmarks
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,memory.total --format=csv,noheader; nproc; free -g | head -2
make -C oracle -s 2>&1 | tail -3
timeout 900 python -m pytest tests/test_gpu_astar.py -x -q 2>&1 | tail -15
timeout 1500 python -m pytest tests -m gpu -x -q --deselect tests/test_gpu_astar.py 2>&1 | tail -8
for args in "300 1024 44850 host" "300 1024 44850 gpu" "1000 1024 60000 host" "1000 1024 60000 gpu" "1000 4096 60000 gpu"; do
  timeout 600 python scripts/astar_bench.py $args 2>&1 | tail -1 | tee -a gpurun_out/astar_bench_a.jsonl
done
