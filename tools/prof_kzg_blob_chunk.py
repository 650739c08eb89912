#!/usr/bin/env python3
"""Host pipeline chunk bound of zkp_kzg_verify_blob_batch on one GPU: for each chunk size 2^C, libzkpair.so is built
with -DZKP_BLOB_CHUNK=2^C into BUILD_DIR (kept while the sources are unchanged: the build is keyed by a hash of them),
and a fresh process (ZKPAIR_LIB pointing at that build) verifies 2^LOG2 blobs from pinned and from pageable host
memory, best of REPS, verdicts checked against the construction.  The card's name and power limit are read first.
Usage: python tools/prof_kzg_blob_chunk.py BUILD_DIR [LOG2=15] [REPS=3] [C ...]   (default C: 10 11 12 13 14)"""
import hashlib
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def measure(log2, reps):
    import numpy as np
    import torch

    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    n = 1 << log2
    eng = z.PairingEngine([0])
    w = workloads.kzg_blob_proofs(eng, n, seed=0x4844, distinct=128)
    pb = torch.from_numpy(w["blobs"]).pin_memory().numpy()
    pp = torch.from_numpy(w["proofs"].view(np.int64)).pin_memory().numpy().view(np.uint64)
    out = []
    with eng.kzg_setup(w["tau_g2"]) as s:
        for name, blobs, proofs in (("pinned", pb, pp), ("pageable", w["blobs"], w["proofs"])):
            assert np.array_equal(eng.kzg_verify_blob_batch(s, blobs, proofs), w["expect"]), name   # also the warm-up
            best = None
            for _ in range(reps):
                t0 = time.perf_counter()
                eng.kzg_verify_blob_batch(s, blobs, proofs)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            out.append("%s %.1f k blobs/s (%.3f ms, %.1f GB/s of blobs)" % (name, n / best / 1e3, best * 1e3, n * 131072 / best / 1e9))
    eng.close()
    print("   ".join(out))


def main():
    if sys.argv[1] == "--measure":
        measure(int(sys.argv[2]), int(sys.argv[3]))
        return
    from zkvm_pairings_b200 import build
    bdir = os.path.abspath(sys.argv[1])
    log2 = int(sys.argv[2]) if len(sys.argv) > 2 else 15
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    chunks = [int(v) for v in sys.argv[4:]] or [10, 11, 12, 13, 14]
    os.makedirs(bdir, exist_ok=True)
    h = hashlib.sha256()
    for f in build.SOURCES + build.HEADERS:
        h.update(open(os.path.join(build.CSRC, f), "rb").read())
    key = h.hexdigest()[:16]
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip())
    for c in chunks:
        so = os.path.join(bdir, "libzkpair_blobchunk%d_%s.so" % (c, key))
        if not os.path.exists(so):
            build.build(force=True, defines=["-DZKP_BLOB_CHUNK=%du" % (1 << c)], out=so)
        env = dict(os.environ, ZKPAIR_LIB=so)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--measure", str(log2), str(reps)], env=env, capture_output=True,
                           text=True)
        line = r.stdout.strip().splitlines()[-1] if r.returncode == 0 else "failed: " + r.stderr.strip()[-400:]
        print("chunk 2^%d  n=2^%d  %s" % (c, log2, line), flush=True)


if __name__ == "__main__":
    main()
