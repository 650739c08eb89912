#!/bin/bash
# EIP-4844 blob verification: the build, the new tests, the whole GPU suite, smoke, tools/prof_kzg_blob.py
# (-> r3c_kzg_blob_rates.txt), tools/prof_kzg.py (-> r3c_kzg_rates.txt) and one bench run on the final tree.
# Usage: tools/gpu_r3c.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3c.sh OUTDIR}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3c_build.log" 2>&1 || { tail -30 "$OUT/r3c_build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3c_pytest_kzg_blob.log"
timeout 900 python -m pytest -q tests/test_kzg_blob.py -p no:cacheprovider >> "$OUT/r3c_pytest_kzg_blob.log" 2>&1
tail -15 "$OUT/r3c_pytest_kzg_blob.log"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3c_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider >> "$OUT/r3c_pytest_gpu.log" 2>&1
tail -15 "$OUT/r3c_pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3c_smoke.log" 2>&1; tail -2 "$OUT/r3c_smoke.log"
timeout 900 python tools/prof_kzg_blob.py 3 > "$OUT/r3c_kzg_blob_rates.txt" 2> "$OUT/r3c_kzg_blob_rates.err"; cat "$OUT/r3c_kzg_blob_rates.txt"
timeout 900 python tools/prof_kzg.py 20 3 > "$OUT/r3c_kzg_rates.txt" 2> "$OUT/r3c_kzg_rates.err"; cat "$OUT/r3c_kzg_rates.txt"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3c_bench_2p20.json" 2> "$OUT/r3c_bench.err"; tail -c 600 "$OUT/r3c_bench_2p20.json"
