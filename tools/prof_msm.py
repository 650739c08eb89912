#!/usr/bin/env python3
"""Multi-scalar multiplication rates on one GPU (zkp_g1_msm / zkp_g2_msm):
- device-resident points/s of the _dev forms at 2^16 .. 2^22 (G1 also 2^24), CUDA events, warmed, best of REPS;
- host points/s from pinned memory (a host clock around the synchronous call), best of REPS;
- the window-width table: G1 at 2^16, 2^20 and 2^22 under forced widths (ZKPAIR_MSM_WINDOW), and the rule's pick;
- all scalars equal against random scalars, G1 at 2^20;
- the path without an MSM at 2^16: g1_mul_batch, then a pairwise g1_add_batch tree;
- kernel shares of one G1 and one G2 MSM at 2^20 from a separate torch.profiler pass.
Points are zkp_gen_points' [e_i]G and every MSM result is checked against [sum k_i e_i mod r]G.  The card's name and
power limit are read first.
Usage: python tools/prof_msm.py [REPS=3] [--profile DIR]"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np
import torch

import zkvm_pairings_b200 as z

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
args = [a for a in sys.argv[1:] if not a.startswith("--")]
reps = int(args[0]) if args else 3
prof_dir = sys.argv[sys.argv.index("--profile") + 1] if "--profile" in sys.argv else None
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0], flush=True)
eng = z.PairingEngine([0])
dev = torch.device("cuda", 0)
s = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(s)
st = s.cuda_stream
SEED = 0x4D534D

import test_msm as tm   # the discrete logs of zkp_gen_points and the exact sum sum k_i e_i mod r

g1_all, _, g2_all, _ = eng.gen_points(SEED, 0, 1 << 22)
a_all, b_all = tm._dlogs(SEED, 0, 1 << 22)
rng = np.random.default_rng(SEED)


def points(group, n):
    """n points of known discrete log (G1 beyond 2^22 repeats the first 2^22)."""
    rows, e = (g1_all, a_all) if group == "g1" else (g2_all, b_all)
    reps_ = (n + rows.shape[0] - 1) // rows.shape[0]
    return np.tile(rows, (reps_, 1))[:n], np.tile(e, reps_)[:n]


def expected(group, k, e):
    sgen = tm._dot_mod_r(k, e) * pow(int(e[0]), -1, R) % R
    base = (g1_all if group == "g1" else g2_all)[:1]
    ref, rinf = (eng.g1_mul_batch if group == "g1" else eng.g2_mul_batch)(base, tm._fr([sgen]))
    return ref[0], int(rinf[0])


def dev_rate(group, n, k=None, check=True):
    rows, e = points(group, n)
    if k is None:
        k = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64, endpoint=False)
    dp = torch.from_numpy(rows.view(np.int64)).to(dev)
    dk = torch.from_numpy(np.ascontiguousarray(k).view(np.int64)).to(dev)
    nbytes = (eng.g1_msm_scratch_bytes if group == "g1" else eng.g2_msm_scratch_bytes)(n)
    scr = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = torch.zeros(rows.shape[1], dtype=torch.int64, device=dev)
    oinf, ost, err = (torch.zeros(1, dtype=torch.uint8, device=dev), torch.zeros(1, dtype=torch.uint8, device=dev),
                      torch.zeros(1, dtype=torch.int32, device=dev))
    fn = eng.g1_msm_dev if group == "g1" else eng.g2_msm_dev
    fn(dp, dk, n, out, oinf, ost, scr, err=err, stream=st)
    torch.cuda.synchronize()
    if check:
        want, winf = expected(group, k, e)
        assert np.array_equal(out.cpu().numpy().view(np.uint64), want) and int(oinf.item()) == winf and int(ost.item()) == 0
    best = 1e9
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        fn(dp, dk, n, out, oinf, ost, scr, err=err, stream=st)
        e1.record(s)
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / 1e3)
    del scr, dp, dk
    torch.cuda.empty_cache()
    return best


def host_rate(group, n):
    rows, e = points(group, n)
    pr = torch.empty(rows.shape, dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
    pk = torch.empty((n, 4), dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
    pr[...] = rows
    pk[...] = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64, endpoint=False)
    fn = eng.g1_msm if group == "g1" else eng.g2_msm
    out, inf, stt = fn(pr, pk)
    want, winf = expected(group, pk, e)
    assert np.array_equal(out, want) and inf == winf and stt == 0
    best = 1e9
    for _ in range(reps):
        t0 = time.perf_counter()
        fn(pr, pk)
        best = min(best, time.perf_counter() - t0)
    return best


print("\n# rates (points/s; device-resident = _dev form on CUDA events; host = pinned buffers, host clock)")
print("%-4s %-6s %-6s %12s %14s %12s %14s" % ("grp", "log2n", "width", "dev ms", "dev pts/s", "host ms", "host pts/s"))
for group, logs in (("g1", (12, 16, 18, 20, 22, 24)), ("g2", (12, 16, 18, 20, 22))):
    for lg in logs:
        n = 1 << lg
        td = dev_rate(group, n)
        th = host_rate(group, n) if lg <= 22 else float("nan")
        c = 8 if n < (1 << 13) else 10 if n < (1 << 18) else 14 if n < (1 << 21) else 15
        print("%-4s %-6d %-6d %12.3f %14.4g %12.3f %14.4g" % (group, lg, c, td * 1e3, n / td, th * 1e3, n / th), flush=True)

print("\n# window widths, G1 device-resident ms (ZKPAIR_MSM_WINDOW forced; * = the rule's pick)")
for lg, widths in ((16, (9, 10, 11, 12)), (20, (13, 14, 15, 16)), (22, (14, 15, 16, 17))):
    cells = []
    for c in widths:
        os.environ["ZKPAIR_MSM_WINDOW"] = str(c)
        t = dev_rate("g1", 1 << lg)
        pick = {16: 10, 20: 14, 22: 15}[lg]
        cells.append("c=%d%s %.3f" % (c, "*" if c == pick else "", t * 1e3))
    os.environ.pop("ZKPAIR_MSM_WINDOW")
    print("2^%d: %s" % (lg, "  ".join(cells)), flush=True)

print("\n# all scalars equal vs random, G1 2^20, device-resident")
n = 1 << 20
kk = rng.integers(0, 1 << 64, size=(1, 4), dtype=np.uint64, endpoint=False)
t_eq = dev_rate("g1", n, np.tile(kk, (n, 1)))
t_rnd = dev_rate("g1", n)
print("equal %.3f ms  random %.3f ms  ratio %.2f" % (t_eq * 1e3, t_rnd * 1e3, t_eq / t_rnd), flush=True)

print("\n# without an MSM, G1 2^16: g1_mul_batch + pairwise g1_add_batch tree (host buffers)")
n = 1 << 16
rows, e = points("g1", n)
k = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64, endpoint=False)
best = 1e9
for _ in range(reps):
    t0 = time.perf_counter()
    p, pinf = eng.g1_mul_batch(rows, k)
    while p.shape[0] > 1:
        h = p.shape[0] // 2
        q, f = eng.g1_add_batch(p[:h], p[h:2 * h], pinf[:h], pinf[h:2 * h])
        p, pinf = (np.concatenate([q, p[2 * h:]]), np.concatenate([f & 1, pinf[2 * h:]]))
    best = min(best, time.perf_counter() - t0)
want, _ = expected("g1", k, e)
assert np.array_equal(p[0], want)
t_msm = host_rate("g1", n)
print("mul+tree %.3f ms (%.4g pts/s)  g1_msm %.3f ms (%.4g pts/s)  speed-up %.1fx" % (best * 1e3, n / best, t_msm * 1e3, n / t_msm, best / t_msm))

if prof_dir:
    from torch.profiler import ProfilerActivity, profile
    print("\n# kernel shares, one MSM at 2^20 (torch.profiler)")
    for group in ("g1", "g2"):
        dev_rate(group, 1 << 20, check=False)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            dev_rate(group, 1 << 20, check=False)
        tot = {}
        for ev in prof.key_averages():
            if ev.device_time_total > 0 and "msm" in ev.key:
                tot[ev.key] = ev.device_time_total
        allt = sum(tot.values())
        print(group, "  ".join("%s %.1f%%" % (k.split("(")[0].replace("void ", "")[:40], 100 * v / allt)
                                 for k, v in sorted(tot.items(), key=lambda kv: -kv[1])))
        prof.export_chrome_trace(os.path.join(prof_dir, "msm_%s_trace.json" % group))
eng.close()
