cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
timeout 600 python -m pytest tests/test_gpu_matcher.py -x -q 2>&1 | tail -40
timeout 900 python scripts/diag_tuples.py cfg4_sparse 2>&1 | tail -40
