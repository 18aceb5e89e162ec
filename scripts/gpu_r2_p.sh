cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
timeout 600 python -m pytest tests -m gpu -q 2>&1 | tail -5
cp pose_graph_initialization_b200/libpgi.so /tmp/libpgi_A.so
TAG=A timeout 120 python scripts/k1_probe.py 2>&1 | tail -1
for v in B C D; do
  cp gpurun_variants/libpgi_$v.so pose_graph_initialization_b200/libpgi.so
  TAG=$v timeout 120 python scripts/k1_probe.py 2>&1 | tail -1
done
cp /tmp/libpgi_A.so pose_graph_initialization_b200/libpgi.so
run() { # name, env..., -- args
  name=$1; shift
  timeout 800 env "$@" > gpurun_out/$name.json 2> gpurun_out/$name.err
  echo "== $name rc=$?"; python - <<P
import json
try:
    d=json.load(open("gpurun_out/$name.json"))
    print({k:d.get(k) for k in ("value","ms_per_step")}, d["e2e"]["value"], d.get("host_s_per_step"), {k:d["host_counters"].get(k) for k in ("astar_runs","astar_pushes","sec_astar","waves","floor_retries","stale_spared")}, "cpu", d["cpu_baseline"]["value"], "verify", json.dumps(d.get("verify"))[:300])
except Exception as e:
    print("no json", e); print(open("gpurun_out/$name.err").read()[-2000:])
P
}
run p_cfg2 X=1 python bench.py --config cfg2_300v --steps 2 --warmup 1 --verify 4000
run p_cfg2_w512 X=1 python bench.py --config cfg2_300v --steps 2 --warmup 1 --wave 512 --cpu-sample 64
run p_cfg3 X=1 python bench.py --config cfg3_1000v --steps 1 --warmup 1 --verify 2000 --verify-replay 5000
