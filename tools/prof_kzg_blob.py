#!/usr/bin/env python3
"""EIP-4844 blob verification rate on one GPU: zkp_kzg_verify_blob_dev over 2^10, 2^12 and 2^14 device-resident blobs
(CUDA events), alternated in the same process with zkp_kzg_verify_dev on the derived z | y of the same proofs (the
point-evaluation remainder); the kernel times of k_blob_challenge and k_blob_eval from a torch.profiler pass of its
own; and the host end-to-end rate of zkp_kzg_verify_blob_batch from pinned memory at the largest size, with the
host-to-device bandwidth that rate implies.  The card's name and power limit are read first.
Usage: python tools/prof_kzg_blob.py [REPS=3] [LOG2 ...]"""
import os
import subprocess
import sys
import time
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import zkvm_pairings_b200 as z
from zkvm_pairings_b200 import workloads

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
sizes = [int(v) for v in sys.argv[2:]] or [10, 12, 14]
nmax = 1 << max(sizes)
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
eng = z.PairingEngine([0])
dev = torch.device("cuda", 0)
s = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(s)
st = s.cuda_stream

w = workloads.kzg_blob_proofs(eng, nmax, seed=0x4844, distinct=128)
setup = eng.kzg_setup(w["tau_g2"])
db = torch.from_numpy(w["blobs"]).to(dev)
dp = torch.from_numpy(w["proofs"].view(np.int64)).to(dev)
dz = torch.from_numpy(np.ascontiguousarray(w["zy"]).view(np.int64)).to(dev)
status = torch.empty(nmax, dtype=torch.uint8, device=dev)
zy_out = torch.empty((nmax, 8), dtype=torch.int64, device=dev)
scratch = torch.empty(eng.kzg_blob_scratch_bytes(nmax), dtype=torch.uint8, device=dev)
torch.cuda.synchronize()


def blob(n):
    eng.kzg_verify_blob_dev(setup, db, dp, n, status, scratch, d_out_zy=zy_out, stream=st)


def point(n):
    eng.kzg_verify_dev(setup, dp, dz, n, status, scratch, stream=st)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


for lg in sizes:   # warm-up, and the verdicts and z | y at every timed size
    n = 1 << lg
    point(n)
    blob(n)
    torch.cuda.synchronize()
    assert np.array_equal(status[:n].cpu().numpy(), w["expect"][:n]), lg
    assert np.array_equal(zy_out[:n].cpu().numpy().view(np.uint64), w["zy"][:n]), lg
print("verdicts and z | y equal the construction at n = %s" % ", ".join("2^%d" % lg for lg in sizes))

kt = {}
warnings.filterwarnings("ignore", message=".*Profiler clears events.*")   # one profiled call per context: nothing to keep
for lg in sizes:   # kernel times, one profiled call per size
    n = 1 << lg
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        blob(n)
        torch.cuda.synchronize()
    t = {"k_blob_challenge": 0.0, "k_blob_eval": 0.0}
    for e in prof.key_averages():
        for k in t:
            if k in e.key:
                t[k] += getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3
    kt[lg] = t

for lg in sizes:
    n = 1 << lg
    tb, tp = [], []
    for r in range(reps):
        tp.append(timed(lambda: point(n)))
        tb.append(timed(lambda: blob(n)))
    b, p = min(tb), min(tp)
    c, e = kt[lg]["k_blob_challenge"], kt[lg]["k_blob_eval"]
    print("n=2^%d  blob verify_dev best %.3f ms  %.1f k blobs/s  = %.2f x verify_dev (%.3f ms)   k_blob_challenge %.3f ms (%.0f %%)"
          "  k_blob_eval %.3f ms (%.0f %%)  point evaluation %.0f %%   (all: %s | %s)"
          % (lg, b, n / b, b / p, p, c, 100 * c / b, e, 100 * e / b, 100 * p / b, " ".join("%.2f" % v for v in tb),
             " ".join("%.2f" % v for v in tp)))

# host end to end, pinned buffers, the largest size
pb = torch.from_numpy(w["blobs"]).pin_memory().numpy()
pp = torch.from_numpy(w["proofs"].view(np.int64)).pin_memory().numpy().view(np.uint64)
eng.kzg_verify_blob_batch(setup, pb, pp)
best = None
for r in range(reps):
    t0 = time.perf_counter()
    got = eng.kzg_verify_blob_batch(setup, pb, pp)
    dt = time.perf_counter() - t0
    best = dt if best is None else min(best, dt)
assert np.array_equal(got, w["expect"])
print("blob verify_batch host pinned n=2^%d  best %.3f ms  %.1f k blobs/s  = %.1f GB/s of blobs host to device"
      % (max(sizes), best * 1e3, nmax / best / 1e3, nmax * 131072 / best / 1e9))
setup.close()
eng.close()
