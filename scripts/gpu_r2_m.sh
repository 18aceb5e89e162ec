cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
make -C oracle -s 2>&1 | tail -3
timeout 1500 python -m pytest tests -m gpu -x -q 2>&1 | tail -6
timeout 900 python scripts/diag_tuples.py cfg4_sparse 36805 2>&1 | tail -12
run() { # name, env..., -- args
  name=$1; shift
  timeout 1700 env "$@" > gpurun_out/$name.json 2> gpurun_out/$name.err
  echo "== $name rc=$?"; python - <<P
import json
try:
    d=json.load(open("gpurun_out/$name.json"))
    print({k:d.get(k) for k in ("value","ms_per_step")}, d["e2e"]["value"], d.get("host_s_per_step"), {k:d["host_counters"][k] for k in ("astar_runs","astar_pushes","sec_astar","waves")}, d.get("branch_mix"), "K1", d["roofline_k1_scoring"]["frac"], "verify", json.dumps(d.get("verify"))[:400], "cpu", d["cpu_baseline"]["value"])
except Exception as e:
    print("no json", e); print(open("gpurun_out/$name.err").read()[-2000:])
P
}
run m_cfg2_tma1 python bench.py --config cfg2_300v --steps 2 --warmup 1
run m_cfg4 X=1 python bench.py --config cfg4_sparse --steps 2 --warmup 1 --verify 0
