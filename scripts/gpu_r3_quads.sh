#!/bin/bash
# Quad scan evidence in one GPU session: tensor-memory load rates, quads on/off A/B on the benchmark (alternating, dumped hit
# lists compared), per-length scan throughput both ways, the GPU suite, smoke() and one full bench run.
# Reads the card's name, power limit and max SM clock; changes no settings.
# usage: scripts/gpu_r3_quads.sh OUTDIR   (every result goes under OUTDIR)
O=${1:?usage: scripts/gpu_r3_quads.sh OUTDIR}
mkdir -p "$O"
export O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/gpu.txt
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o /tmp/tmem_rate profiles/microbench/tmem_rate.cu && timeout 120 /tmp/tmem_rate | tee $O/tmem_rate.txt
echo "tmem_rate exit ${PIPESTATUS[0]}"
timeout 600 python -m pytest -q tests/test_scan_quads.py 2>&1 | tail -5
BENCH="python bench.py --no-secondary --no-cpu --no-libmarv --steps 10 --warmup 3"
for i in 1 2 3; do
    timeout 600 $BENCH --dump-outputs $O/dump_quads_$i > $O/bench_quads_$i.json 2> $O/bench_quads_$i.err
    B200_SCAN_NO_QUADS=1 timeout 600 $BENCH --dump-outputs $O/dump_noquads_$i > $O/bench_noquads_$i.json 2> $O/bench_noquads_$i.err
done
python - <<'PY'
import json, os, numpy as np
O = os.environ["O"]
def val(f):
    try: return json.loads(open(f).read().strip().splitlines()[-1])["value"]
    except Exception as e: return "ERR %s" % e
for i in (1, 2, 3):
    a, b = val(f"{O}/bench_quads_{i}.json"), val(f"{O}/bench_noquads_{i}.json")
    same = True
    da, db = f"{O}/dump_quads_{i}", f"{O}/dump_noquads_{i}"
    files = sorted(os.listdir(da)) if os.path.isdir(da) else []
    for f in files:
        same &= os.path.exists(os.path.join(db, f)) and np.array_equal(np.load(os.path.join(da, f)), np.load(os.path.join(db, f)))
    print(f"pair {i}: quads {a}  no_quads {b}  ratio {a / b if isinstance(a, float) and isinstance(b, float) else 'n/a'}  dumps identical {same} ({len(files)} files)")
PY
timeout 600 python scripts/scan_classes.py 2>&1 | tail -16 | tee $O/scan_classes_quads.txt
B200_SCAN_NO_QUADS=1 timeout 600 python scripts/scan_classes.py 2>&1 | tail -16 | tee $O/scan_classes_noquads.txt
timeout 1500 python -m pytest -q -m gpu tests 2>&1 | tail -5
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python bench.py --steps 10 --warmup 3 > $O/r03_bench_n1.json 2> $O/r03_bench_n1.err; echo "bench exit $?"
python - <<'PY'
import json, os
d = json.loads(open(os.path.join(os.environ["O"], "r03_bench_n1.json")).read().strip().splitlines()[-1])
print("value %.0f e2e %.0f binding frac %.3f" % (d["value"], d["e2e"]["value"], d["roofline"]["binding_resource"]["frac"]))
print({k: d.get("cpu_baseline", {}).get(k) for k in ("value", "scan_identical_to_gpu", "hit_lists_identical_to_gpu")})
PY
