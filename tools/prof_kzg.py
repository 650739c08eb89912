#!/usr/bin/env python3
"""KZG point-evaluation verification rate on one GPU: zkp_kzg_verify_dev over 2^18 and 2^LOG2 device-resident proofs
(CUDA events), alternated in the same process with the bare prepared 2-pair check (multi_pairing_prepared_dev,
k = kf = 2) over the same number of checks; the front end's share of the step (step time minus the pairing kernels'
event-timed share: k_kzg_prepare plus the one-byte verdict kernel); and the host end-to-end rate of
zkp_kzg_verify_batch from pinned memory at 2^LOG2.
Usage: python tools/prof_kzg.py [LOG2=20] [REPS=3]"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import zkvm_pairings_b200 as z
from zkvm_pairings_b200 import workloads

log2 = int(sys.argv[1]) if len(sys.argv) > 1 else 20
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
sizes = sorted({18, log2})
nmax = 1 << sizes[-1]
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
eng = z.PairingEngine([0])
dev = torch.device("cuda", 0)
s = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(s)
st = s.cuda_stream


def dev_u64(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).to(dev)


# 2^14 constructed proofs tiled to the largest size (verdicts known), device resident; smaller sizes use a prefix
m = 1 << 14
w = workloads.kzg_proofs(eng, m, seed=0x4844)
proofs, zy, expect = np.tile(w["proofs"], (nmax // m, 1)), np.tile(w["zy"], (nmax // m, 1)), np.tile(w["expect"], nmax // m)
setup = eng.kzg_setup(w["tau_g2"])
dp, dz = dev_u64(proofs), dev_u64(zy)
scratch = torch.empty(eng.kzg_scratch_bytes(nmax), dtype=torch.uint8, device=dev)
status = torch.empty(nmax, dtype=torch.uint8, device=dev)

# the bare prepared 2-pair check over the same number of checks: seeded G1 points, both G2 points from tables
k = 2
g1 = torch.empty((nmax * k, 12), dtype=torch.int64, device=dev)
g2 = torch.empty((nmax * k, 24), dtype=torch.int64, device=dev)
i1 = torch.empty(nmax * k, dtype=torch.uint8, device=dev)
i2 = torch.empty(nmax * k, dtype=torch.uint8, device=dev)
out = torch.empty((nmax, 72), dtype=torch.int64, device=dev)
one = torch.empty(nmax, dtype=torch.uint8, device=dev)
eng.gen_points_dev(13, 0, nmax * k, g1, i1, g2, i2, stream=st)
tab = torch.empty((k, eng.G2_PREPARED_U64), dtype=torch.int64, device=dev)
eng.g2_prepare_dev(g2[:k].contiguous(), k, tab, stream=st)
del g2, i2
torch.cuda.synchronize()


def checks2(n):
    eng.multi_pairing_prepared_dev(out, g1, None, n, k, tab, k, is_one=one, stream=st)


def verify(n):
    eng.kzg_verify_dev(setup, dp, dz, n, status, scratch, stream=st)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


for lg in sizes:   # warm-up, and the verdicts at every timed size
    n = 1 << lg
    checks2(n)
    verify(n)
    torch.cuda.synchronize()
    assert np.array_equal(status[:n].cpu().numpy(), expect[:n]), lg
print("verdicts equal the construction at n = %s" % ", ".join("2^%d" % lg for lg in sizes))

for lg in sizes:
    n = 1 << lg
    ref, res = [], []
    for r in range(reps):
        ref.append(timed(lambda: checks2(n)))
        res.append(timed(lambda: verify(n)))
    c2, t = min(ref), min(res)
    eng.set_kernel_timing(True)
    eng.last_kernel_ms()
    step = timed(lambda: verify(n))
    pair_ms, _ = eng.last_kernel_ms()
    eng.set_kernel_timing(False)
    print("checks2 prepared   n=2^%d  best %.3f ms  %.3f M checks/s   (all: %s)" % (lg, c2, n / c2 / 1e3, " ".join("%.2f" % v for v in ref)))
    print("kzg verify_dev     n=2^%d  best %.3f ms  %.3f M proofs/s  = %.3f x checks2 time   front end %.1f %% of the step"
          " (step %.3f ms, pairing %.3f ms)   (all: %s)" % (lg, t, n / t / 1e3, t / c2, 100.0 * (step - pair_ms) / step, step, pair_ms,
                                                          " ".join("%.2f" % v for v in res)))

# host end to end, pinned buffers, the largest size
pp = torch.from_numpy(proofs.view(np.int64)).pin_memory().numpy().view(np.uint64)
pz = torch.from_numpy(np.ascontiguousarray(zy).view(np.int64)).pin_memory().numpy().view(np.uint64)
eng.kzg_verify_batch(setup, pp, pz)
best = None
for r in range(reps):
    t0 = time.perf_counter()
    got = eng.kzg_verify_batch(setup, pp, pz)
    dt = time.perf_counter() - t0
    best = dt if best is None else min(best, dt)
assert np.array_equal(got, expect)
print("kzg verify_batch host pinned n=2^%d  best %.3f ms  %.3f M proofs/s" % (sizes[-1], best * 1e3, nmax / best / 1e6))
setup.close()
eng.close()
