#!/usr/bin/env python3
"""EIP-7594 cell recovery rates on one GPU: zkp_kzg_recover_cells_dev over 2^8, 2^10 and 2^12 device-resident blobs with
64 and with 127 cells present (a different random erasure per blob), next to zkp_kzg_compute_cells_dev (k_cells_extend)
on the same blobs; zkp_kzg_recover_cells_and_proofs_dev over 2^6 and 2^8 blobs; the host rate of
zkp_kzg_recover_cells_batch over 2^12 blobs from pinned memory (CUDA events / a host clock around synchronised work,
best of REPS).  Every recovered cell is compared with compute_cells' and every status must be 0.  The card's name and
power limit are read first.
Usage: python tools/prof_kzg_recover.py [REPS=3]"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import zkvm_pairings_b200 as z
from zkvm_pairings_b200 import workloads

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
CELLS, CB = z.CELLS_PER_EXT_BLOB, z.CELL_BYTES
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
eng = z.PairingEngine([0])
dev = torch.device("cuda", 0)
s = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(s)
st = s.cuda_stream
tau, g2m, g1m, lag = workloads.kzg_cell_setup(eng, seed=0x7594)
setup = eng.kzg_setup_cells(g2m, g1m, lag)

nb = 1 << 12
blobs = np.random.default_rng(0x7594).integers(0, 256, size=(nb, workloads.BLOB_BYTES), dtype=np.uint8)
blobs.reshape(nb, workloads.BLOB_N, 32)[:, :, 0] &= 0x3F   # every element < 2^254 < r
db = torch.from_numpy(blobs).to(dev)
full = torch.empty((nb, CELLS, CB), dtype=torch.uint8, device=dev)
dst = torch.empty(nb, dtype=torch.uint8, device=dev)
eng.kzg_compute_cells_dev(setup, db, nb, full, dst, stream=st)
torch.cuda.synchronize()
assert not dst.any()


def timed(fn):
    best = None
    for _ in range(reps + 1):   # the first pass warms up
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None or ms < best else best
    return best


def erasure(n, m, seed):
    """Per blob a random set of m present cells (ascending), their cells, and the counts."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    idx = torch.rand((n, CELLS), generator=g).argsort(dim=1)[:, :m].sort(dim=1).values.to(dev)
    didx = torch.zeros((n, CELLS), dtype=torch.int64, device=dev)
    didx[:, :m] = idx
    dcl = torch.zeros((n, CELLS, CB), dtype=torch.uint8, device=dev)
    dcl[:, :m] = torch.gather(full[:n], 1, idx[:, :, None].expand(n, m, CB))
    return didx, dcl, torch.full((n,), m, dtype=torch.int64, device=dev)


out = torch.empty((nb, CELLS, CB), dtype=torch.uint8, device=dev)
for n in (1 << 8, 1 << 10, 1 << 12):
    ext = timed(lambda: eng.kzg_compute_cells_dev(setup, db, n, out, dst, stream=st))
    for m in (64, 127):
        didx, dcl, dnum = erasure(n, m, n + m)
        out.zero_()
        ms = timed(lambda: eng.kzg_recover_cells_dev(setup, didx, dcl, dnum, n, out, dst, stream=st))
        ok = torch.equal(out[:n], full[:n]) and not dst[:n].any()
        print("recover_cells 2^%d blobs, %3d cells present: %8.3f ms  %9.0f blobs/s  (k_cells_extend on the same blobs %7.3f ms, "
              "%9.0f blobs/s; ratio %.2f)  cells equal compute_cells: %s" % (n.bit_length() - 1, m, ms, n / ms * 1e3, ext, n / ext * 1e3,
                                                                             ms / ext, ok))
        assert ok

for n in (1 << 6, 1 << 8):
    didx, dcl, dnum = erasure(n, 64, 7 * n)
    dp = torch.empty((n, CELLS, 12), dtype=torch.int64, device=dev)
    dpi = torch.empty((n, CELLS), dtype=torch.uint8, device=dev)
    scratch = torch.empty(eng.kzg_cells_proofs_scratch_bytes(n), dtype=torch.uint8, device=dev)
    ms = timed(lambda: eng.kzg_recover_cells_and_proofs_dev(setup, didx, dcl, dnum, n, out, dp, dpi, dst, scratch, stream=st))
    ok = torch.equal(out[:n], full[:n]) and not dst[:n].any()
    print("recover_cells_and_kzg_proofs 2^%d blobs, 64 cells present: %9.1f ms  %7.1f blobs/s  cells equal: %s" % (
        n.bit_length() - 1, ms, n / ms * 1e3, ok))
    assert ok
    del dp, dpi, scratch

didx, dcl, dnum = erasure(nb, 64, 99)
pin = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in (didx, dcl, dnum)]
for p, t in zip(pin, (didx, dcl, dnum)):
    p.copy_(t)
hidx, hcl, hnum = pin[0].numpy().view(np.uint64), pin[1].numpy(), pin[2].numpy().view(np.uint64)
best = None
for _ in range(reps + 1):
    t0 = time.perf_counter()
    cells, hst = eng.kzg_recover_cells_batch(setup, hidx, hcl, hnum)
    dt = time.perf_counter() - t0
    best = dt if best is None or dt < best else best
ok = np.array_equal(cells, full.cpu().numpy()) and not hst.any()
print("recover_cells host path, 2^12 blobs from pinned memory (output pageable): %.1f ms  %.0f blobs/s  cells equal: %s" % (
    best * 1e3, nb / best, ok))
assert ok
setup.close()
eng.close()
