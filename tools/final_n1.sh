# usage: bash tools/final_n1.sh OUTDIR      GPU tests, bench N=1 (line + per-step times from its stderr detail), reference arm
OUT=${1:?usage: bash tools/final_n1.sh OUTDIR}
mkdir -p "$OUT"
timeout 500 python -m pytest tests -m gpu -q -x 2>&1 | tail -3
timeout 400 python bench.py --steps 20 --warmup 5 > "$OUT/r02_bench_n1.json" 2> "$OUT/r02_bench_n1.err"; echo "bench rc $?"; python - "$OUT" <<'PY'
import json, os, sys
line = json.loads(open(os.path.join(sys.argv[1], "r02_bench_n1.json")).read().splitlines()[-1])
tag = "[bench detail] "
detail = json.loads([l for l in open(os.path.join(sys.argv[1], "r02_bench_n1.err")) if l.startswith(tag)][-1][len(tag):])
print([round(x,2) for x in detail["step_ms_rank0"]])
print([round(x,2) for x in detail["e2e_step_ms_rank0"]])
print(line["value"], line["ms_per_step"], line["e2e"]["ms_per_step"], line["clocks"], line["b1"])
PY
timeout 300 python bench.py --impl reference --steps 5 --warmup 1 > "$OUT/r02_bench_reference_n1.json" 2>/dev/null; tail -c 150 "$OUT/r02_bench_reference_n1.json"
echo final_n1_done
