cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
timeout 900 python -m pytest tests/test_gpu_k1_stream.py tests/test_gpu_parity.py tests/test_gpu_edge_cases.py -x -q 2>&1 | tail -8
run() { # name, env..., -- args
  name=$1; shift
  timeout 1500 env "$@" > gpurun_out/$name.json 2> gpurun_out/$name.err
  echo "== $name rc=$?"; python - <<P
import json
try:
    d=json.load(open("gpurun_out/$name.json"))
    print({k:d.get(k) for k in ("value","ms_per_step")}, d["e2e"]["value"], d.get("host_s_per_step"), {k:d["host_counters"][k] for k in ("astar_runs","astar_pushes","sec_astar","gpu_searches","sec_search_gpu","sec_search_host_part","waves")}, d.get("roofline_k1_scoring"))
except Exception as e:
    print("no json", e); print(open("gpurun_out/$name.err").read()[-2000:])
P
}
run j_cfg3_w256_host python bench.py --config cfg3_1000v --steps 1 --warmup 0 --wave 256 --cpu-sample 64 --host-search
run j_cfg3_w512_hybrid python bench.py --config cfg3_1000v --steps 1 --warmup 0 --wave 512 --cpu-sample 64 --search-min-batch 128
run j_cfg3_w512_host python bench.py --config cfg3_1000v --steps 1 --warmup 0 --wave 512 --cpu-sample 64 --host-search
