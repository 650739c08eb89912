#!/bin/bash
# k_kzg_msm at one resident block per SM (ZKP_MSM_MIN_BLOCKS=1, 164 registers) against two (the default, 128 registers):
# the library is built with each bound into a temporary directory and tools/prof_kzg_prove.py runs at 2^12 blobs,
# alternating the two builds twice.  Usage: tools/prof_kzg_msm_bounds.sh OUTFILE
OUT="${1:?usage: tools/prof_kzg_msm_bounds.sh OUTFILE}"
TMP=$(mktemp -d)
for mb in 1 2; do
    python -c "from zkvm_pairings_b200 import build; build.build(force=True, defines=['-DZKP_MSM_MIN_BLOCKS=$mb'], out='$TMP/libzkpair_mb$mb.so')" || exit 1
done
: > "$OUT"
for rep in 1 2; do
    for mb in 1 2; do
        echo "== ZKP_MSM_MIN_BLOCKS=$mb (pass $rep)" >> "$OUT"
        ZKPAIR_LIB="$TMP/libzkpair_mb$mb.so" timeout 600 python tools/prof_kzg_prove.py 3 12 >> "$OUT" 2>&1
    done
done
rm -rf "$TMP"
cat "$OUT"
