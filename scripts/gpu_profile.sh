cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
BENCH_ARGS="--no-overlap" bash scripts/gpu_bench1.sh 2>&1 | grep -v "^+" | tail -9
python scripts/profile_wave.py 1184
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/launches_wave.csv python scripts/profile_wave.py 1184 > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:k5_fallback_score -s 9 -c 2 -o gpurun_out/prof_k5 python scripts/profile_wave.py 1184 > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:"k3_decompose|k2_fivept|k1_score" -s 3 -c 3 -o gpurun_out/prof_k123 python scripts/profile_wave.py 1184 > /dev/null 2>&1
ls -la gpurun_out/
