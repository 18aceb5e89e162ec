cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
timeout 600 python -m pytest tests/test_gpu_astar.py -x -q 2>&1 | tail -5
timeout 600 python scripts/astar_bench.py 1000 2048 150000 check 2>&1 | tail -1 | cut -c1-600
run() { # name, env..., -- args
  name=$1; shift
  timeout 1500 env "$@" > gpurun_out/$name.json 2> gpurun_out/$name.err
  echo "== $name rc=$?"; python - <<P
import json
try:
    d=json.load(open("gpurun_out/$name.json"))
    print({k:d.get(k) for k in ("value","ms_per_step")}, d["e2e"]["value"], d.get("host_s_per_step"), {k:d["host_counters"][k] for k in ("astar_runs","astar_pops","astar_pushes","sec_astar","gpu_searches","gpu_search_redo","sec_search_gpu","sec_search_host_part","waves")}, d.get("search_stats_last_step"), d.get("verify"))
except Exception as e:
    print("no json", e); print(open("gpurun_out/$name.err").read()[-2000:])
P
}
run i_cfg3_w2048_hybrid python bench.py --config cfg3_1000v --steps 1 --warmup 0 --wave 2048 --cpu-sample 256
