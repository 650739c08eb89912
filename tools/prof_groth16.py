#!/usr/bin/env python3
"""Groth16 verification rate on one GPU: zkp_groth16_verify_dev over 2^LOG2 device-resident proofs for
l in {1, 2, 8, 32} public inputs (CUDA events), alternated in the same process with the prepared 4-pair launch of
tools/prof_checks4.py over the same number of checks; the front end's share of the step (step time minus the
pairing kernels' event-timed share: k_groth16_prepare plus the one-byte verdict kernel); and the host end-to-end
rate of zkp_groth16_verify_batch from pinned memory at l = 2.
Usage: python tools/prof_groth16.py [LOG2=18] [REPS=3]"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import zkvm_pairings_b200 as z
from zkvm_pairings_b200 import workloads

log2 = int(sys.argv[1]) if len(sys.argv) > 1 else 18
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
n = 1 << log2
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
eng = z.PairingEngine([0])
dev = torch.device("cuda", 0)
s = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(s)
st = s.cuda_stream


def dev_u64(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).to(dev)


# per l: a distinct key, 2^14 constructed proofs tiled to n (verdicts known), device resident
cases = {}
for lp in (1, 2, 8, 32):
    m = min(n, 1 << 14)
    w = workloads.groth16_proofs(eng, m, lp, seed=0x9000 + lp)
    reps_t = n // m
    proofs, inputs, expect = np.tile(w["proofs"], (reps_t, 1)), np.tile(w["inputs"], (reps_t, 1, 1)), np.tile(w["expect"], reps_t)
    vk = eng.groth16_prepare_vk(w["alpha"], w["beta"], w["gamma"], w["delta"], w["ic"])
    cases[lp] = (vk, dev_u64(proofs), dev_u64(inputs), expect, proofs, inputs)
scratch = torch.empty(eng.groth16_scratch_bytes(n), dtype=torch.uint8, device=dev)
status = torch.empty(n, dtype=torch.uint8, device=dev)

# the prepared 4-pair check of tools/prof_checks4.py over n checks
k, kf = 4, 3
g1 = torch.empty((n * k, 12), dtype=torch.int64, device=dev)
g2 = torch.empty((n * k, 24), dtype=torch.int64, device=dev)
i1 = torch.empty(n * k, dtype=torch.uint8, device=dev)
i2 = torch.empty(n * k, dtype=torch.uint8, device=dev)
out = torch.empty((n, 72), dtype=torch.int64, device=dev)
one = torch.empty(n, dtype=torch.uint8, device=dev)
eng.gen_points_dev(11, 0, n * k, g1, i1, g2, i2, stream=st)
tab = torch.empty((kf, eng.G2_PREPARED_U64), dtype=torch.int64, device=dev)
eng.g2_prepare_dev(g2[:kf].contiguous(), kf, tab, stream=st)
var = g2.view(n, k, 24)[:, 0, :].contiguous()
torch.cuda.synchronize()


def checks4():
    eng.multi_pairing_prepared_dev(out, g1, var, n, k, tab, kf, is_one=one, stream=st)


def verify(lp):
    vk, dp, dx = cases[lp][:3]
    eng.groth16_verify_dev(vk, dp, dx, n, status, scratch, stream=st)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


checks4()
for lp in cases:   # warm-up, and the verdicts at the timed size
    verify(lp)
    torch.cuda.synchronize()
    assert np.array_equal(status.cpu().numpy(), cases[lp][3]), lp
print("verdicts at n=2^%d equal the construction for l = %s" % (log2, sorted(cases)))

res = {lp: [] for lp in cases}
ref = []
for r in range(reps):
    ref.append(timed(checks4))
    for lp in cases:
        res[lp].append(timed(lambda: verify(lp)))
c4 = min(ref)
print("checks4 prepared  n=2^%d  best %.3f ms  %.3f M checks/s   (all: %s)" % (log2, c4, n / c4 / 1e3, " ".join("%.2f" % v for v in ref)))
for lp in cases:
    t = min(res[lp])
    eng.set_kernel_timing(True)
    eng.last_kernel_ms()
    step = timed(lambda: verify(lp))
    pair_ms, _ = eng.last_kernel_ms()
    eng.set_kernel_timing(False)
    print("groth16 verify_dev l=%-3d n=2^%d  best %.3f ms  %.3f M proofs/s  = %.3f x checks4 time   front end %.1f %% of the step"
          " (step %.3f ms, pairing %.3f ms)   (all: %s)" % (lp, log2, t, n / t / 1e3, t / c4, 100.0 * (step - pair_ms) / step, step,
                                                          pair_ms, " ".join("%.2f" % v for v in res[lp])))

# host end to end, pinned buffers, l = 2
vk, _, _, expect, proofs, inputs = cases[2]
pp = torch.from_numpy(proofs.view(np.int64)).pin_memory().numpy().view(np.uint64)
px = torch.from_numpy(np.ascontiguousarray(inputs).view(np.int64)).pin_memory().numpy().view(np.uint64)
eng.groth16_verify_batch(vk, pp, px)
best = None
for r in range(reps):
    t0 = time.perf_counter()
    got = eng.groth16_verify_batch(vk, pp, px)
    dt = time.perf_counter() - t0
    best = dt if best is None else min(best, dt)
assert np.array_equal(got, expect)
print("groth16 verify_batch host pinned l=2 n=2^%d  best %.3f ms  %.3f M proofs/s" % (log2, best * 1e3, n / best / 1e6))
for c in cases.values():
    c[0].close()
eng.close()
