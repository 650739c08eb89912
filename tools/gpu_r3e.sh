#!/bin/bash
# MSM branch coverage and Fr on the device: the build, the new and extended test files, the whole GPU suite, smoke and
# one bench run on the final tree.
# Usage: tools/gpu_r3e.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3e.sh OUTDIR}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3e_build.log" 2>&1 || { tail -30 "$OUT/r3e_build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3e_pytest_msm_fr.log"
timeout 900 python -m pytest -q tests/test_kzg_msm_edges.py tests/test_device_bounds.py -p no:cacheprovider >> "$OUT/r3e_pytest_msm_fr.log" 2>&1
tail -15 "$OUT/r3e_pytest_msm_fr.log"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3e_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider >> "$OUT/r3e_pytest_gpu.log" 2>&1
tail -15 "$OUT/r3e_pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3e_smoke.log" 2>&1; tail -2 "$OUT/r3e_smoke.log"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3e_bench_2p20.json" 2> "$OUT/r3e_bench.err"; tail -c 600 "$OUT/r3e_bench_2p20.json"
