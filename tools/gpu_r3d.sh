#!/bin/bash
# EIP-4844 commitments and proofs: the build, the new tests, the whole GPU suite, smoke, tools/prof_kzg_prove.py
# (-> r3d_kzg_prove_rates.txt) and one bench run on the final tree.
# Usage: tools/gpu_r3d.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3d.sh OUTDIR}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3d_build.log" 2>&1 || { tail -30 "$OUT/r3d_build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3d_pytest_kzg_prove.log"
timeout 900 python -m pytest -q tests/test_kzg_prove.py -p no:cacheprovider >> "$OUT/r3d_pytest_kzg_prove.log" 2>&1
tail -15 "$OUT/r3d_pytest_kzg_prove.log"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3d_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider >> "$OUT/r3d_pytest_gpu.log" 2>&1
tail -15 "$OUT/r3d_pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3d_smoke.log" 2>&1; tail -2 "$OUT/r3d_smoke.log"
timeout 900 python tools/prof_kzg_prove.py 3 > "$OUT/r3d_kzg_prove_rates.txt" 2> "$OUT/r3d_kzg_prove_rates.err"; cat "$OUT/r3d_kzg_prove_rates.txt"; tail -5 "$OUT/r3d_kzg_prove_rates.err"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3d_bench_2p20.json" 2> "$OUT/r3d_bench.err"; tail -c 600 "$OUT/r3d_bench_2p20.json"
