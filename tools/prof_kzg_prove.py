#!/usr/bin/env python3
"""EIP-4844 prover rates on one GPU: the prover setup's creation time and resident bytes; zkp_kzg_blob_to_commitment_dev
and zkp_kzg_compute_blob_proof_dev over 2^10, 2^12 and 2^14 device-resident blobs (CUDA events, alternated in the same
process); the kernel times of k_kzg_prove_challenge, k_kzg_quotient and k_kzg_msm in the blob proofs from a
torch.profiler pass of its own; and the host end-to-end rates of the _batch calls from pinned memory at the largest size.  A sample of the proofs
is checked with zkp_kzg_verify_blob_batch.  The card's name and power limit are read first.
Usage: python tools/prof_kzg_prove.py [REPS=3] [LOG2 ...]"""
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

tau, tg, lag = workloads.kzg_lagrange_setup(eng, seed=0x4844)
torch.cuda.synchronize()
free0 = torch.cuda.mem_get_info(dev)[0]
t0 = time.perf_counter()
setup = eng.kzg_setup(tg, lag)
t_setup = time.perf_counter() - t0
free1 = torch.cuda.mem_get_info(dev)[0]
t0 = time.perf_counter()
plain = eng.kzg_setup(tg)
t_plain = time.perf_counter() - t0
plain.close()
print("prover setup: created in %.1f ms (verifier-only setup %.1f ms); device memory taken %.1f MiB"
      % (t_setup * 1e3, t_plain * 1e3, (free0 - free1) / 2 ** 20))

blobs = np.random.default_rng(0x4844).integers(0, 256, size=(nmax, workloads.BLOB_BYTES), dtype=np.uint8)
blobs.reshape(nmax, workloads.BLOB_N, 32)[:, :, 0] &= 0x3F   # every element < 2^254 < r
db = torch.from_numpy(blobs).to(dev)
dc = torch.empty((nmax, 12), dtype=torch.int64, device=dev)
dci = torch.empty(nmax, dtype=torch.uint8, device=dev)
dp = torch.empty((nmax, 12), dtype=torch.int64, device=dev)
dpi = torch.empty(nmax, dtype=torch.uint8, device=dev)
dst = torch.empty(nmax, dtype=torch.uint8, device=dev)
scratch = torch.empty(eng.kzg_prover_scratch_bytes(nmax), dtype=torch.uint8, device=dev)
torch.cuda.synchronize()


def commit(n):
    eng.kzg_blob_to_commitment_dev(setup, db, n, dc, dci, dst, stream=st)


def prove(n):
    eng.kzg_compute_blob_proof_dev(setup, db, dc, n, dp, dpi, dst, scratch, d_commitment_inf=dci, stream=st)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


commit(nmax)
prove(nmax)
torch.cuda.synchronize()
assert not dst.cpu().numpy().any()
k = np.array([0, 1, nmax // 2, nmax - 1])
c, ci, p, pi = (t.cpu().numpy() for t in (dc, dci, dp, dpi))
ver = eng.kzg_verify_blob_batch(setup, blobs[k], np.concatenate([c.view(np.uint64)[k], p.view(np.uint64)[k]], axis=1),
                                np.stack([ci[k], pi[k]], axis=1))
assert not ver.any(), ver
print("statuses VALID at n = 2^%d; a sample of %d proofs verifies" % (max(sizes), len(k)))

names = ("k_kzg_prove_challenge", "k_kzg_quotient", "k_kzg_msm")
kt = {}
warnings.filterwarnings("ignore", message=".*Profiler clears events.*")
for lg in sizes:   # kernel times, one profiled pass per size
    n = 1 << lg
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        prove(n)
        torch.cuda.synchronize()
    t = {k_: 0.0 for k_ in names}
    for e in prof.key_averages():
        for k_ in t:
            if k_ in e.key:
                t[k_] += getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3
    kt[lg] = t

for lg in sizes:
    n = 1 << lg
    tc, tp = [], []
    for r in range(reps):
        tc.append(timed(lambda: commit(n)))
        tp.append(timed(lambda: prove(n)))
    c_, p_ = min(tc), min(tp)
    t = kt[lg]
    msm_prove = t["k_kzg_msm"]
    print("n=2^%d  commitments_dev best %.3f ms  %.1f k/s   blob proofs_dev best %.3f ms  %.1f k/s   proof kernels: challenge %.3f ms "
          "(%.0f %%)  quotient %.3f ms (%.0f %%)  msm %.3f ms (%.0f %%)   (all: %s | %s)"
          % (lg, c_, n / c_, p_, n / p_, t["k_kzg_prove_challenge"], 100 * t["k_kzg_prove_challenge"] / p_, t["k_kzg_quotient"],
             100 * t["k_kzg_quotient"] / p_, msm_prove, 100 * msm_prove / p_, " ".join("%.2f" % v for v in tc),
             " ".join("%.2f" % v for v in tp)))

# host end to end, pinned buffers, the largest size
pb = torch.from_numpy(blobs).pin_memory().numpy()
c, ci, _ = eng.kzg_blob_to_commitment_batch(setup, pb)
pc, pci = torch.from_numpy(c.view(np.int64)).pin_memory().numpy().view(np.uint64), torch.from_numpy(ci).pin_memory().numpy()
for name, fn in (("commitments", lambda: eng.kzg_blob_to_commitment_batch(setup, pb)),
                 ("blob proofs", lambda: eng.kzg_compute_blob_proof_batch(setup, pb, pc, pci))):
    fn()
    best = None
    for r in range(reps):
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    print("%s _batch host pinned n=2^%d  best %.3f ms  %.1f k/s" % (name, max(sizes), best * 1e3, nmax / best / 1e3))
setup.close()
eng.close()
