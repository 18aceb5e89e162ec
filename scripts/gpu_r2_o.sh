cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
run() { # name, env..., -- args
  name=$1; shift
  timeout 1700 env "$@" > gpurun_out/$name.json 2> gpurun_out/$name.err
  echo "== $name rc=$?"; python - <<P
import json
try:
    d=json.load(open("gpurun_out/$name.json"))
    print({k:d.get(k) for k in ("value","ms_per_step")}, d["e2e"]["value"], d.get("host_s_per_step"), {k:d["host_counters"].get(k) for k in ("astar_runs","astar_pushes","sec_astar","waves","floor_retries")}, "cpu", d["cpu_baseline"]["value"])
except Exception as e:
    print("no json", e); print(open("gpurun_out/$name.err").read()[-2000:])
P
}
run o_cfg3_floor X=1 python bench.py --config cfg3_1000v --steps 1 --warmup 1 --cpu-sample 512 --verify 0
run o_cfg2_floor X=1 python bench.py --config cfg2_300v --steps 2 --warmup 1 --verify 0
