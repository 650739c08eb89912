#!/bin/bash
# EIP-7594 cell recovery: the build, the cluster probe, the new tests, the whole GPU suite, smoke,
# tools/prof_kzg_recover.py (-> r3g_kzg_recover_rates.txt) and one bench run on the final tree.
# Usage: tools/gpu_r3g.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3g.sh OUTDIR}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3g_build.log" 2>&1 || { tail -30 "$OUT/r3g_build.log"; exit 1; }
[ -x build/recover_cluster_probe ] || nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --threads 0 -o build/recover_cluster_probe \
    tools/recover_cluster_probe.cu zkvm_pairings_b200/csrc/pairing_kernel.cu zkvm_pairings_b200/csrc/fe_kernel.cu
build/recover_cluster_probe > "$OUT/r3g_recover_clusters.txt" 2>&1; cat "$OUT/r3g_recover_clusters.txt"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3g_pytest_kzg_recover.log"
timeout 900 python -m pytest -q tests/test_kzg_recover.py -p no:cacheprovider >> "$OUT/r3g_pytest_kzg_recover.log" 2>&1
tail -15 "$OUT/r3g_pytest_kzg_recover.log"
timeout 600 python tools/prof_kzg_recover.py 3 > "$OUT/r3g_kzg_recover_rates.txt" 2> "$OUT/r3g_kzg_recover_rates.err"; cat "$OUT/r3g_kzg_recover_rates.txt"; tail -5 "$OUT/r3g_kzg_recover_rates.err"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3g_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider >> "$OUT/r3g_pytest_gpu.log" 2>&1
tail -15 "$OUT/r3g_pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3g_smoke.log" 2>&1; tail -2 "$OUT/r3g_smoke.log"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3g_bench_2p20.json" 2> "$OUT/r3g_bench.err"; tail -c 300 "$OUT/r3g_bench_2p20.json"
