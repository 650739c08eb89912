#!/bin/bash
# Groth16 verification: the new tests, the whole GPU suite, smoke, tools/prof_groth16.py (-> profiles/r3a_groth16_rates.txt)
# and one bench run on the final tree.  Usage: tools/gpu_r3a.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3a.sh OUTDIR}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3a_build.log" 2>&1 || { tail -30 "$OUT/r3a_build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3a_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider >> "$OUT/r3a_pytest_gpu.log" 2>&1
tail -15 "$OUT/r3a_pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3a_smoke.log" 2>&1; tail -2 "$OUT/r3a_smoke.log"
timeout 600 python tools/prof_groth16.py 18 3 > "$OUT/r3a_groth16_rates.txt" 2>&1; cat "$OUT/r3a_groth16_rates.txt"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3a_bench_2p20.json" 2> "$OUT/r3a_bench.err"; tail -c 600 "$OUT/r3a_bench_2p20.json"
