# round 2, second GPU pass: device A* in the real pipeline (cfg2 A/B, wave sizes), then cfg3 once
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
timeout 600 python -m pytest tests/test_gpu_astar.py tests/test_gpu_scene.py -x -q 2>&1 | tail -5
run() { # name, env..., args
  name=$1; shift
  timeout 900 env "$@" > gpurun_out/$name.json 2> gpurun_out/$name.err
  echo "== $name rc=$?"; python - <<P
import json
try:
    d=json.load(open("gpurun_out/$name.json"))
    print({k:d.get(k) for k in ("value","ms_per_step")}, d["e2e"]["value"], d.get("host_s_per_step"), {k:d["host_counters"][k] for k in ("astar_runs","astar_pops","astar_pushes","sec_astar","sec_visibility","sec_commit","gpu_searches","gpu_search_redo","sec_search_gpu","waves")}, d.get("search_stats"))
except Exception as e:
    print("no json", e); print(open("gpurun_out/$name.err").read()[-2000:])
P
}
run cfg2_host python bench.py --config cfg2_300v --steps 2 --warmup 1 --cpu-sample 256
run cfg2_gpu256 python bench.py --config cfg2_300v --steps 2 --warmup 1 --cpu-sample 256
run cfg2_gpu1024 python bench.py --config cfg2_300v --steps 2 --warmup 1 --cpu-sample 256 --wave 1024
run cfg2_gpu4096 python bench.py --config cfg2_300v --steps 2 --warmup 1 --cpu-sample 256 --wave 4096
run cfg3_gpu2048 python bench.py --config cfg3_1000v --steps 1 --warmup 1 --cpu-sample 256 --wave 2048
