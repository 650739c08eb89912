#!/bin/bash
# Multi-scalar multiplication over caller-given points: the build, the new tests, the whole GPU suite, smoke,
# tools/prof_msm.py (-> r3i_msm_rates.txt, with a torch.profiler pass whose traces stay in OUTDIR) and one bench run.
# Usage: tools/gpu_r3i.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3i.sh OUTDIR}"
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3i_build.log" 2>&1 || { tail -30 "$OUT/r3i_build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3i_pytest_msm.log"
timeout 1200 python -m pytest -q tests/test_msm.py -p no:cacheprovider -rs >> "$OUT/r3i_pytest_msm.log" 2>&1
tail -15 "$OUT/r3i_pytest_msm.log"
timeout 900 python tools/prof_msm.py 3 --profile "$OUT" > "$OUT/r3i_msm_rates.txt" 2> "$OUT/r3i_msm_rates.err"; cat "$OUT/r3i_msm_rates.txt"; tail -5 "$OUT/r3i_msm_rates.err"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > "$OUT/r3i_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider -rs >> "$OUT/r3i_pytest_gpu.log" 2>&1
tail -12 "$OUT/r3i_pytest_gpu.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3i_smoke.log" 2>&1; tail -2 "$OUT/r3i_smoke.log"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3i_bench_2p20.json" 2> "$OUT/r3i_bench.err"; tail -c 400 "$OUT/r3i_bench_2p20.json"
