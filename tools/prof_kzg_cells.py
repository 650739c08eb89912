#!/usr/bin/env python3
"""EIP-7594 cell rates on one GPU: the cells setup's creation time and resident bytes; zkp_kzg_compute_cells_dev over 2^8
and 2^12 device-resident blobs, zkp_kzg_compute_cells_and_proofs_dev over 2^6 and 2^8 blobs and zkp_kzg_verify_cell_dev
over 2^14, 2^16 and 2^18 cells (CUDA events, best of REPS); the kernel shares of each from a torch.profiler pass of its
own; and the host end-to-end rate of zkp_kzg_compute_cells_and_proofs_batch from pinned memory.  The statuses are
checked: every cell of the batches verifies.  The card's name and power limit are read first.
Usage: python tools/prof_kzg_cells.py [REPS=2]"""
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

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 2
CELLS, CB = z.CELLS_PER_EXT_BLOB, z.CELL_BYTES
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
eng = z.PairingEngine([0])
dev = torch.device("cuda", 0)
s = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(s)
st = s.cuda_stream

tau, g2m, g1m, lag = workloads.kzg_cell_setup(eng, seed=0x7594)
torch.cuda.synchronize()
free0 = torch.cuda.mem_get_info(dev)[0]
t0 = time.perf_counter()
setup = eng.kzg_setup_cells(g2m, g1m, lag)
t_setup = time.perf_counter() - t0
free1 = torch.cuda.mem_get_info(dev)[0]
print("cells setup with Lagrange points: created in %.1f ms; device memory taken %.1f MiB" % (t_setup * 1e3, (free0 - free1) / 2 ** 20))

nb = 1 << 12
blobs = np.random.default_rng(0x7594).integers(0, 256, size=(nb, workloads.BLOB_BYTES), dtype=np.uint8)
blobs.reshape(nb, workloads.BLOB_N, 32)[:, :, 0] &= 0x3F   # every element < 2^254 < r
db = torch.from_numpy(blobs).to(dev)
dcells = torch.empty((nb, CELLS, CB), dtype=torch.uint8, device=dev)
dst = torch.empty(nb, dtype=torch.uint8, device=dev)
npb = 1 << 8
dp = torch.empty((npb, CELLS, 12), dtype=torch.int64, device=dev)
dpi = torch.empty((npb, CELLS), dtype=torch.uint8, device=dev)
pscratch = torch.empty(eng.kzg_cells_proofs_scratch_bytes(npb), dtype=torch.uint8, device=dev)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def shares(fn, names):
    warnings.filterwarnings("ignore", message=".*Profiler clears events.*")
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    t = {}
    for e in prof.key_averages():
        dt = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3
        if dt <= 0:
            continue
        key = next((k for k in names if k in e.key), "other")
        t[key] = t.get(key, 0.0) + dt
    tot = sum(t.values())
    return " ".join("%s %.2f ms (%.0f %%)" % (k, v, 100 * v / tot) for k, v in sorted(t.items(), key=lambda kv: -kv[1]))


def cells(n):
    eng.kzg_compute_cells_dev(setup, db, n, dcells, dst, stream=st)


def proofs(n):
    eng.kzg_compute_cells_and_proofs_dev(setup, db, n, dcells, dp, dpi, dst, pscratch, stream=st)


cells(nb)
torch.cuda.synchronize()
assert not dst.cpu().numpy().any()
for lg in (8, 12):
    n = 1 << lg
    t = [timed(lambda: cells(n)) for _ in range(reps)]
    print("compute_cells_dev n=2^%d blobs  best %.3f ms  %.1f blobs/s   (all: %s)" % (lg, min(t), n / min(t) * 1e3, " ".join("%.2f" % v for v in t)))
print("  kernel shares at 2^12:", shares(lambda: cells(nb), ("k_cells_extend",)))

proofs(npb)
torch.cuda.synchronize()
assert not dst[:npb].cpu().numpy().any()
for lg in (6, 8):
    n = 1 << lg
    t = [timed(lambda: proofs(n)) for _ in range(reps)]
    print("compute_cells_and_proofs_dev n=2^%d blobs  best %.1f ms  %.1f blobs/s  %.1f us per proof row   (all: %s)"
          % (lg, min(t), n / min(t) * 1e3, min(t) * 1e3 / (n * CELLS), " ".join("%.1f" % v for v in t)))
print("  kernel shares at 2^8:", shares(lambda: proofs(npb), ("k_cells_extend", "k_cells_quotient", "k_kzg_msm")))

# verification: every cell of the 2^8 blobs, tiled to 2^18 cells
hc, hp, hpi = dcells[:npb].cpu().numpy(), dp.cpu().numpy().view(np.uint64), dpi.cpu().numpy()
cpts, cinf, cst = eng.kzg_blob_to_commitment_batch(setup, blobs[:npb])
assert not cst.any()
nv = 1 << 18
rep = nv // (npb * CELLS)
C = np.repeat(cpts, CELLS, axis=0)
Ci = np.repeat(cinf, CELLS)
K = np.tile(np.arange(CELLS, dtype=np.uint64), npb)
X = hc.reshape(npb * CELLS, CB)
P, Pi = hp.reshape(npb * CELLS, 12), hpi.reshape(npb * CELLS)
dC, dCi, dK, dX, dP, dPi = (torch.from_numpy(np.ascontiguousarray(np.tile(a, (rep,) + (1,) * (a.ndim - 1))).view(dt)).to(dev)
                            for a, dt in ((C, np.int64), (Ci, np.uint8), (K, np.int64), (X, np.uint8), (P, np.int64), (Pi, np.uint8)))
dvs = torch.empty(nv, dtype=torch.uint8, device=dev)
vscratch = torch.empty(eng.kzg_verify_cell_scratch_bytes(nv), dtype=torch.uint8, device=dev)


def verify(n):
    eng.kzg_verify_cell_dev(setup, dC, dK, dX, dP, n, dvs, vscratch, d_commitment_inf=dCi, d_proof_inf=dPi, stream=st)


verify(nv)
torch.cuda.synchronize()
assert not dvs.cpu().numpy().any(), "a computed cell does not verify"
print("every one of the %d cells and proofs verifies" % nv)
for lg in (14, 16, 18):
    n = 1 << lg
    t = [timed(lambda: verify(n)) for _ in range(reps)]
    print("verify_cell_dev n=2^%d cells  best %.3f ms  %.1f k cells/s   (all: %s)" % (lg, min(t), n / min(t), " ".join("%.2f" % v for v in t)))
print("  kernel shares at 2^18:", shares(lambda: verify(nv), ("k_cells_interp", "k_cells_prepare", "k_pairing", "k_groth16_verdict")))

pb = torch.from_numpy(blobs[:npb]).pin_memory().numpy()
eng.kzg_compute_cells_and_proofs_batch(setup, pb[:2])
t0 = time.perf_counter()
eng.kzg_compute_cells_and_proofs_batch(setup, pb)
dt = time.perf_counter() - t0
print("compute_cells_and_proofs_batch host pinned n=2^8 blobs  %.1f ms  %.1f blobs/s" % (dt * 1e3, npb / dt))
setup.close()
eng.close()
