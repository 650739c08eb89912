#!/bin/bash
# Host-buffer pipeline refactor: the A/B of every host-buffer call against the parent build (default defines, and
# small chunks with forced staging), the whole GPU suite, alternating parent / new timings of the pinned e2e pairing
# path, the pageable multi-Miller product and blob verification at the shipped chunk, smoke and one bench run.
# Expects build/libzkpair_parent.so and build/libzkpair_parent_small.so (the parent commit's sources, default defines
# and SMALL below) and build/libzkpair_new_small.so (this tree, SMALL).
# Usage: tools/gpu_r3h.sh OUTDIR
OUT="${1:?usage: tools/gpu_r3h.sh OUTDIR}"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee "$OUT/r3h_gpu.txt"
NGPU=$(nvidia-smi --query-gpu=name --format=csv,noheader | wc -l)
python -c "import __graft_entry__ as g; g.build()" > "$OUT/r3h_build.log" 2>&1 || { tail -30 "$OUT/r3h_build.log"; exit 1; }
cp zkvm_pairings_b200/libzkpair.so build/libzkpair_new.so
for pair in "parent new" "parent_small new_small"; do
  set -- $pair
  timeout 900 python tools/ab_host_calls.py build/libzkpair_$1.so build/libzkpair_$2.so > "$OUT/r3h_ab_$2.txt" 2>&1
  echo "A/B $1 vs $2: exit $? : $(tail -1 "$OUT/r3h_ab_$2.txt")"
  if [ "$NGPU" -ge 2 ]; then
    timeout 900 python tools/ab_host_calls.py build/libzkpair_$1.so build/libzkpair_$2.so --devices 2 > "$OUT/r3h_ab_$2_2dev.txt" 2>&1
    echo "A/B $1 vs $2, 2 devices: exit $? : $(tail -1 "$OUT/r3h_ab_$2_2dev.txt")"
  fi
done
cp "$OUT/r3h_gpu.txt" "$OUT/r3h_pytest_gpu.log"
timeout 1500 python -m pytest -q -m gpu tests -p no:cacheprovider -rs >> "$OUT/r3h_pytest_gpu.log" 2>&1
tail -12 "$OUT/r3h_pytest_gpu.log"
cp "$OUT/r3h_gpu.txt" "$OUT/r3h_speed_ab.txt"
for rep in 1 2 3; do
  for v in parent new; do
    export ZKPAIR_LIB=$PWD/build/libzkpair_$v.so
    echo "$v rep=$rep e2e: $(timeout 300 python tools/prof_e2e.py 20 6 2>&1 | tail -1)"
    echo "$v rep=$rep product: $(timeout 300 python tools/prof_product.py 20 2>&1 | tail -1)"
    echo "$v rep=$rep blob: $(timeout 300 python tools/prof_kzg_blob_chunk.py --measure 15 3 2>&1 | tail -1)"
  done
done >> "$OUT/r3h_speed_ab.txt"
unset ZKPAIR_LIB
cat "$OUT/r3h_speed_ab.txt"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3h_smoke.log" 2>&1; tail -2 "$OUT/r3h_smoke.log"
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 2 > "$OUT/r3h_bench_2p20.json" 2> "$OUT/r3h_bench.err"; tail -c 400 "$OUT/r3h_bench_2p20.json"
