#!/bin/bash
# EIP-7594 cells: the build, the new tests, the whole GPU suite, smoke, tools/prof_kzg_cells.py (-> r3f_kzg_cells_rates.txt)
# and one bench run on the final tree.
# Usage: tools/gpu_r3f.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3f.sh OUTDIR}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3f_build.log" 2>&1 || { tail -30 "$OUT/r3f_build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3f_pytest_kzg_cells.log"
timeout 900 python -m pytest -q tests/test_kzg_cells.py -p no:cacheprovider >> "$OUT/r3f_pytest_kzg_cells.log" 2>&1
tail -15 "$OUT/r3f_pytest_kzg_cells.log"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3f_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider >> "$OUT/r3f_pytest_gpu.log" 2>&1
tail -15 "$OUT/r3f_pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3f_smoke.log" 2>&1; tail -2 "$OUT/r3f_smoke.log"
timeout 900 python tools/prof_kzg_cells.py 2 > "$OUT/r3f_kzg_cells_rates.txt" 2> "$OUT/r3f_kzg_cells_rates.err"; cat "$OUT/r3f_kzg_cells_rates.txt"; tail -5 "$OUT/r3f_kzg_cells_rates.err"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3f_bench_2p20.json" 2> "$OUT/r3f_bench.err"; tail -c 600 "$OUT/r3f_bench_2p20.json"
