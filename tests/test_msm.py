"""Multi-scalar multiplication over caller-given points (zkp_g1_msm / zkp_g2_msm and their _dev forms): the step functions
of csrc/msm.cuh through the CPU dev simulation at small window widths (crowded buckets, segments that cross them), and
the GPU entry points against independent oracles: the C oracle's [k_i]P_i summed under its group law, [sum k_i e_i]G
for points of known discrete log, and the exact integer-scalar sums of points with small-order components."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import util
from test_small_order_points import Fp, Fp2, G1, G2, R, P, add, dec, enc_rows, mul, neg, points

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M64 = (1 << 64) - 1
MSM_CHUNK = 1 << 22   # ZKP_MSM_CHUNK (kernels.cu)
P_LIMBS = np.array([(P >> (64 * k)) & M64 for k in range(6)], np.uint64)   # a limb vector >= p


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _fr(vals):
    return np.array([[(v >> (64 * k)) & M64 for k in range(4)] for v in vals], np.uint64).reshape(-1, 4)


def _ints(k):
    return [sum(int(row[j]) << (64 * j) for j in range(4)) for row in k]


def _msum(F, pts, ks):
    """sum_i [k_i]P_i on Python integers (None = the identity)."""
    acc = None
    for a, k in zip(pts, ks):
        acc = add(F, acc, mul(F, a, k))
    return acc


def _splitmix(seed, idx):
    """SplitMix64 output idx + 1 of seed, vectorised (util.scalars_for's generator)."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (idx.astype(np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def _dlogs(seed, first, n):
    """The discrete logs (a_i for G1, b_i for G2) of zkp_gen_points(seed, first, n), as util.scalars_for."""
    i = np.arange(first, first + n, dtype=np.uint64)
    a, b = _splitmix(seed, 2 * i), _splitmix(seed, 2 * i + np.uint64(1))
    a[a == 0] = 1
    b[b == 0] = 1
    return a, b


def _dot_mod_r(k, e):
    """sum_i k_i e_i mod r for (n,4) u64 scalars k and u64 e, in 16-bit pieces so that numpy sums never overflow."""
    kp = [((k[:, j] >> np.uint64(16 * h)) & np.uint64(0xFFFF)).astype(np.uint64) for j in range(4) for h in range(4)]
    ep = [((e >> np.uint64(16 * h)) & np.uint64(0xFFFF)).astype(np.uint64) for h in range(4)]
    tot = 0
    for a, ka in enumerate(kp):
        for b, eb in enumerate(ep):
            tot += int(np.sum(ka * eb, dtype=np.uint64)) << (16 * (a + b))
    return tot % R


# ---------------------------------------------------------------- CPU: the dev simulation of msm.cuh

@pytest.fixture(scope="module")
def sim():
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_msm.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, f) for f in ("sim_msm.cpp", "sim.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", so, src[0]])
    return ctypes.CDLL(so)


def _sim_msm(sim, F, rows, flags, ks, c, seg, ranges=2):
    n = len(ks)
    w = 12 if F is Fp else 24
    rows = np.ascontiguousarray(np.asarray(rows, np.uint64).reshape(-1, w))
    flags = None if flags is None else np.ascontiguousarray(np.asarray(flags, np.uint8))
    k = np.ascontiguousarray(_fr(ks)) if n else np.zeros((0, 4), np.uint64)
    out, oinf, st, err = np.zeros(w, np.uint64), np.zeros(1, np.uint8), np.zeros(1, np.uint8), np.zeros(1, np.uint32)
    sim.sim_msm(ctypes.c_int(F is Fp2), _p(rows), _p(flags), _p(k), ctypes.c_size_t(n), ctypes.c_int(c), ctypes.c_int(seg),
                ctypes.c_int(ranges), _p(out), _p(oinf), _p(st), _p(err))
    return out, int(oinf[0]), int(st[0]), int(err[0])


def _expect(F, out, inf, a):
    if a is None:
        assert inf == 1
        assert dec(F, out) == ((0, 1) if F is Fp else ((0, 0), (1, 0)))
    else:
        assert inf == 0
        assert dec(F, out) == a


EDGE_SCALARS = [0, 1, R - 1, R, R + 1, 1 << 255, (1 << 256) - 1, 2 * R]


@pytest.mark.parametrize("c", [3, 4, 5, 8, 12, 16])
def test_recoding_reconstructs_every_scalar(sim, c):
    rng = random.Random(c)
    ks = list(EDGE_SCALARS)
    # every window rounds up (its bits exceed 2^(c-1)), so the carry runs out of the top window
    ks.append(sum(((1 << c) - 1) << (c * w) for w in range(256 // c)) & ((1 << 256) - 1))
    ks.append(sum(((1 << (c - 1)) + 1) << (c * w) for w in range(256 // c)) & ((1 << 256) - 1))
    ks += [rng.getrandbits(256) for _ in range(40)]
    digits = (ctypes.c_int32 * 128)()
    for k in ks:
        nw = sim.sim_msm_recode(_p(_fr([k])), c, digits)
        assert nw == 256 // c + 1
        ds = list(digits[:nw])
        assert all(-(1 << (c - 1)) < d <= (1 << (c - 1)) for d in ds)
        assert sum(d << (c * w) for w, d in enumerate(ds)) == k


def test_window_rule(sim):
    ns = (1, (1 << 13) - 1, 1 << 13, (1 << 18) - 1, 1 << 18, (1 << 21) - 1, 1 << 21, 1 << 22)
    assert [sim.sim_msm_window(ctypes.c_size_t(n)) for n in ns] == [8, 8, 10, 10, 14, 14, 15, 15]


def _subgroup_points(coracle, n, seed, group="g1"):
    """n subgroup points [e_i]G with their discrete logs, from the C oracle."""
    rng = random.Random(seed)
    e = [rng.randrange(1, R) for _ in range(n)]
    if group == "g1":
        rows, flags = coracle.g1_mul_batch(util.scalar_matrix(e))
    else:
        rows, flags = coracle.g2_mul_batch(util.scalar_matrix(e))
    return rows, e


@pytest.mark.parametrize("n", [1, 2, 3, 37, 1000])
def test_sim_g1_msm_matches_the_sum(sim, coracle, n):
    rows, e = _subgroup_points(coracle, n, 0x3100 + n)
    rng = random.Random(n)
    ks = [rng.choice(EDGE_SCALARS) if rng.random() < 0.2 else rng.getrandbits(256) for _ in range(n)]
    want = mul(Fp, G1, sum(k * x for k, x in zip(ks, e)) % R)
    for c, seg in ((3, 1), (4, 3), (5, 7)) if n <= 37 else ((4, 5),):
        out, inf, st, err = _sim_msm(sim, Fp, rows, None, ks, c, seg)
        assert (st, err) == (0, 0)
        _expect(Fp, out, inf, want)


@pytest.mark.parametrize("n", [1, 3, 12])
def test_sim_g2_msm_matches_the_sum(sim, coracle, n):
    rows, e = _subgroup_points(coracle, n, 0x3200 + n, "g2")
    rng = random.Random(n)
    ks = [rng.getrandbits(256) for _ in range(n)]
    ks[0] = (1 << 256) - 1
    want = mul(Fp2, G2, sum(k * x for k, x in zip(ks, e)) % R)
    out, inf, st, err = _sim_msm(sim, Fp2, rows, None, ks, 4, 3)
    assert (st, err) == (0, 0)
    _expect(Fp2, out, inf, want)


def test_sim_degenerate_inputs(sim, coracle):
    n = 40
    rows, e = _subgroup_points(coracle, n, 0x3300)
    rng = random.Random(7)
    k = rng.getrandbits(256)
    # all scalars equal: one bucket per window holds every point, over many segments (length 1, 3) or one (longer than n)
    for seg in (1, 3, n + 5):
        out, inf, st, _ = _sim_msm(sim, Fp, rows, None, [k] * n, 4, seg)
        _expect(Fp, out, inf, mul(Fp, G1, k * sum(e) % R))
    # all zero
    out, inf, st, _ = _sim_msm(sim, Fp, rows, None, [0] * n, 4, 3)
    _expect(Fp, out, inf, None)
    # P and -P under equal scalars: the inverse meets inside a bucket
    pts = [mul(Fp, G1, x) for x in e[:6]]
    both = pts + [neg(Fp, a) for a in pts]
    r2, f2 = enc_rows(Fp, both)
    ks = [rng.getrandbits(256) for _ in pts]
    out, inf, st, _ = _sim_msm(sim, Fp, r2, f2, ks + ks, 3, 2)
    _expect(Fp, out, inf, None)
    # one point repeated: the doubling case inside a bucket
    ks = [rng.getrandbits(256) for _ in range(n)]
    out, inf, st, _ = _sim_msm(sim, Fp, np.stack([rows[0]] * n), None, ks, 3, 4)
    _expect(Fp, out, inf, mul(Fp, G1, sum(ks) * e[0] % R))
    # flagged points contribute the identity
    flags = np.array([i % 3 == 0 for i in range(n)], np.uint8)
    out, inf, st, _ = _sim_msm(sim, Fp, rows, flags, ks, 5, 2)
    _expect(Fp, out, inf, mul(Fp, G1, sum(kk * x for kk, x, f in zip(ks, e, flags) if not f) % R))


def test_sim_small_order_components_and_statuses(sim):
    rng = random.Random(11)
    for F, key in ((Fp, "g1"), (Fp2, "g2")):
        pts = [a for _, a, q in points()[key]][:6]
        ks = [R + rng.getrandbits(200) for _ in pts]
        ks[0] = (1 << 256) - 1
        rows, flags = enc_rows(F, pts)
        out, inf, st, err = _sim_msm(sim, F, rows, flags, ks, 4, 3)
        assert (st, err) == (0, 0)
        _expect(F, out, inf, _msum(F, pts, ks))
        # off the curve: status 1, zero limbs, the flag set
        bad = rows.copy()
        bad[1, 0] ^= np.uint64(1)
        out, inf, st, err = _sim_msm(sim, F, bad, flags, ks, 4, 3)
        assert (st, inf, err) == (1, 1, 0) and not out.any()
        # a flagged off-curve point is ignored
        f2 = flags.copy()
        f2[1] = 1
        out, inf, st, err = _sim_msm(sim, F, bad, f2, ks, 4, 3)
        assert (st, err) == (0, 0)
        _expect(F, out, inf, _msum(F, [a for i, a in enumerate(pts) if i != 1], [k for i, k in enumerate(ks) if i != 1]))
        # a limb >= p: the error word
        nc = rows.copy()
        nc[2, :6] = P_LIMBS
        _, _, _, err = _sim_msm(sim, F, nc, flags, ks, 4, 3)
        assert err == 1


# ---------------------------------------------------------------- GPU

def _gpu_sum_oracle(coracle, group, rows, flags, ks):
    """The C oracle's [k_i]P_i, summed under its group law."""
    mulf = coracle.g1_mul_batch if group == "g1" else coracle.g2_mul_batch
    prods, pinf = mulf(_fr(ks), base=rows, binf=flags)
    w = rows.shape[1]
    acc, ainf = np.zeros(w, np.uint64), 1
    for j in range(len(ks)):
        if pinf[j]:
            continue
        if ainf:
            acc, ainf = prods[j].copy(), 0
            continue
        if np.array_equal(acc[: w // 2], prods[j][: w // 2]) and not np.array_equal(acc[w // 2:], prods[j][w // 2:]):
            acc, ainf = np.zeros(w, np.uint64), 1   # P + (-P)
            continue
        acc, f = coracle.group_op(group, "add", acc, 0, prods[j], 0)
        ainf = f & 1
    return acc, ainf


def _engine_msm(engine, group, rows, ks, flags=None):
    return (engine.g1_msm if group == "g1" else engine.g2_msm)(rows, ks, flags)


def _neg_rows(rows):
    """-P for every row: each y coordinate's Fp to (p - y) mod p."""
    out = rows.copy()
    w = rows.shape[1] // 2
    for i in range(rows.shape[0]):
        for c in range(w // 6):
            lo = w + 6 * c
            y = sum(int(rows[i, lo + j]) << (64 * j) for j in range(6))
            out[i, lo:lo + 6] = [((P - y) % P >> (64 * j)) & M64 for j in range(6)]
    return out


def _identity_rows(group):
    w = 12 if group == "g1" else 24
    r = np.zeros(w, np.uint64)
    r[w // 2] = 1
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["g1", "g2"])
def test_gpu_msm_n0_n1(engine, coracle, group):
    w = 12 if group == "g1" else 24
    out, inf, st = _engine_msm(engine, group, np.zeros((0, w), np.uint64), np.zeros((0, 4), np.uint64))
    assert (inf, st) == (1, 0) and np.array_equal(out, _identity_rows(group))
    g1, i1, g2, i2 = engine.gen_points(0x51, 0, 1)
    rows = g1 if group == "g1" else g2
    for k in EDGE_SCALARS:
        out, inf, st = _engine_msm(engine, group, rows, _fr([k]))
        ref, rinf = (engine.g1_mul_batch if group == "g1" else engine.g2_mul_batch)(rows, _fr([k]))
        assert st == 0 and inf == rinf[0] and np.array_equal(out, ref[0])


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["g1", "g2"])
@pytest.mark.parametrize("n", [2, 255, 4097, (1 << 16) + 3])
def test_gpu_msm_equals_the_oracle_sum(engine, coracle, group, n):
    g1, _, g2, _ = util.oracle_points(coracle, 0x5200 + n, 0, n)
    rows = g1 if group == "g1" else g2
    rng = random.Random(n)
    ks = [rng.getrandbits(256) for _ in range(n)]
    flags = np.array([rng.random() < 0.05 for _ in range(n)], np.uint8)
    want, winf = _gpu_sum_oracle(coracle, group, rows, flags, ks)
    out, inf, st = _engine_msm(engine, group, rows, _fr(ks), flags)
    assert st == 0 and inf == winf and np.array_equal(out, want)


def _known_dlog_case(engine, group, n, seed, pinned=False):
    g1, _, g2, _ = engine.gen_points(seed, 0, n)
    a, b = _dlogs(seed, 0, n)
    rows, e = (g1, a) if group == "g1" else (g2, b)
    k = np.random.default_rng(seed).integers(0, 1 << 63, size=(n, 4), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    if pinned:
        import torch
        pr = torch.empty(rows.shape, dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
        pk = torch.empty(k.shape, dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
        pr[...] = rows
        pk[...] = k
        rows, k = pr, pk
    s = _dot_mod_r(k, e)
    gen = g1[:1] if group == "g1" else g2[:1]
    # [s]G from the first point [e_0]G: s / e_0 mod r
    ref, rinf = (engine.g1_mul_batch if group == "g1" else engine.g2_mul_batch)(gen, _fr([s * pow(int(e[0]), -1, R) % R]))
    return rows, k, ref[0], int(rinf[0])


@pytest.mark.gpu
@pytest.mark.parametrize("group,n", [("g1", 1 << 20), ("g1", 1 << 22), ("g2", 1 << 18), ("g2", 1 << 20)])
def test_gpu_msm_known_discrete_logs(engine, group, n):
    rows, k, want, winf = _known_dlog_case(engine, group, n, 0x5300 + n)
    out, inf, st = _engine_msm(engine, group, rows, k)
    assert st == 0 and inf == winf and np.array_equal(out, want)


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_gpu_msm_across_the_chunk_boundary(engine, pinned):
    n = MSM_CHUNK + 77
    rows, k, want, winf = _known_dlog_case(engine, "g1", n, 0x5400, pinned)
    out, inf, st = engine.g1_msm(rows, k)
    assert st == 0 and inf == winf and np.array_equal(out, want)


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["g1", "g2"])
def test_gpu_msm_degenerate_distributions(engine, group):
    n = 1 << 16
    g1, _, g2, _ = engine.gen_points(0x55, 0, n)
    a, b = _dlogs(0x55, 0, n)
    rows, e = (g1, a) if group == "g1" else (g2, b)
    mulf = engine.g1_mul_batch if group == "g1" else engine.g2_mul_batch
    gen_inv = pow(int(e[0]), -1, R)

    def check(pts, ks, s, flags=None):
        out, inf, st = _engine_msm(engine, group, pts, _fr(ks) if isinstance(ks, list) else ks, flags)
        ref, rinf = mulf(rows[:1], _fr([s * gen_inv % R]))
        assert st == 0 and inf == rinf[0] and np.array_equal(out, ref[0])

    rng = random.Random(5)
    kk = rng.getrandbits(256)
    allk = np.tile(_fr([kk]), (n, 1))
    check(rows, allk, kk * sum(int(x) for x in e) % R)                   # all scalars equal: one bucket per window
    check(rows, np.zeros((n, 4), np.uint64), 0)                          # all zero
    half = n // 2
    negs = _neg_rows(rows[:half])
    ks = np.random.default_rng(1).integers(0, M64, size=(half, 4), dtype=np.uint64, endpoint=True)
    check(np.concatenate([rows[:half], negs]), np.concatenate([ks, ks]), 0)   # P and -P under equal scalars
    ks = np.random.default_rng(2).integers(0, M64, size=(n, 4), dtype=np.uint64, endpoint=True)
    check(np.tile(rows[:1], (n, 1)), ks, sum(_ints(ks)) * int(e[0]) % R)     # one point repeated
    flags = (np.arange(n) % 7 == 3).astype(np.uint8)
    check(rows, ks, sum(k * int(x) for k, x, f in zip(_ints(ks), e, flags) if not f) % R, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["g1", "g2"])
def test_gpu_msm_small_order_components(engine, group):
    F = Fp if group == "g1" else Fp2
    rng = random.Random(0x56)
    named = points()[group]
    pts = [a for _, a, q in named]
    ks = [R + rng.getrandbits(255) for _ in pts]
    ks[0] = (1 << 256) - 1
    rows, flags = enc_rows(F, pts)
    out, inf, st = _engine_msm(engine, group, rows, _fr(ks))
    assert st == 0
    _expect(F, out, inf, _msum(F, pts, ks))
    # subgroup points: k and k + r give the same sum
    sub = [a for _, a, q in named if q == 1]
    rs, _ = enc_rows(F, sub)
    k0 = [rng.randrange(R) for _ in sub]
    o1 = _engine_msm(engine, group, rs, _fr(k0))
    o2 = _engine_msm(engine, group, rs, _fr([k + R for k in k0]))
    assert np.array_equal(o1[0], o2[0]) and o1[1:] == o2[1:]
    _expect(F, o1[0], o1[1], _msum(F, sub, k0))


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["g1", "g2"])
def test_gpu_msm_errors_and_statuses(engine, group):
    import zkvm_pairings_b200 as z
    g1, _, g2, _ = engine.gen_points(0x57, 0, 300)
    rows = (g1 if group == "g1" else g2).copy()
    ks = np.random.default_rng(3).integers(0, M64, size=(300, 4), dtype=np.uint64, endpoint=True)
    bad = rows.copy()
    bad[17, 0] ^= np.uint64(1)
    out, inf, st = _engine_msm(engine, group, bad, ks)
    assert (st, inf) == (1, 1) and not out.any()
    nc = rows.copy()
    nc[5, :6] = P_LIMBS
    with pytest.raises(z.NonCanonicalError):
        _engine_msm(engine, group, nc, ks)
    lib = engine._lib
    fn = lib.zkp_g1_msm if group == "g1" else lib.zkp_g2_msm
    o, b1, b2 = np.zeros(24, np.uint64), np.zeros(1, np.uint8), np.zeros(1, np.uint8)
    assert fn(engine._ctx, None, None, _p(ks), 300, _p(o), _p(b1), _p(b2)) == z._lib.ZKP_ERR_INVALID_ARG
    assert fn(engine._ctx, _p(rows), None, _p(ks), 300, None, _p(b1), _p(b2)) == z._lib.ZKP_ERR_INVALID_ARG
    assert fn(None, _p(rows), None, _p(ks), 300, _p(o), _p(b1), _p(b2)) == z._lib.ZKP_ERR_INVALID_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["g1", "g2"])
def test_gpu_msm_dev_equals_host(engine, group):
    import torch
    import zkvm_pairings_b200 as z
    n = 70001
    g1, _, g2, _ = engine.gen_points(0x58, 0, n)
    rows = g1 if group == "g1" else g2
    w = rows.shape[1]
    ks = np.random.default_rng(4).integers(0, M64, size=(n, 4), dtype=np.uint64, endpoint=True)
    flags = (np.arange(n) % 11 == 0).astype(np.uint8)
    want = _engine_msm(engine, group, rows, ks, flags)
    dev = torch.device("cuda", 0)
    d_pts = torch.from_numpy(rows.view(np.int64)).to(dev)
    d_k = torch.from_numpy(ks.view(np.int64)).to(dev)
    d_inf = torch.from_numpy(flags).to(dev)
    nbytes = (engine.g1_msm_scratch_bytes if group == "g1" else engine.g2_msm_scratch_bytes)(n)
    d_scr = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_out = torch.zeros(w, dtype=torch.int64, device=dev)
    d_oinf, d_st, d_err = (torch.zeros(1, dtype=torch.uint8, device=dev), torch.zeros(1, dtype=torch.uint8, device=dev),
                           torch.zeros(1, dtype=torch.int32, device=dev))
    fn = engine.g1_msm_dev if group == "g1" else engine.g2_msm_dev
    s = torch.cuda.Stream(device=dev)
    before = torch.cuda.current_device()
    fn(d_pts, d_k, n, d_out, d_oinf, d_st, d_scr, d_inf=d_inf, err=d_err, stream=s.cuda_stream)
    s.synchronize()
    assert torch.cuda.current_device() == before
    assert np.array_equal(d_out.cpu().numpy().view(np.uint64), want[0])
    assert (int(d_oinf.item()), int(d_st.item()), int(d_err.item())) == (want[1], want[2], 0)
    # n = 0: the identity
    fn(d_pts, d_k, 0, d_out, d_oinf, d_st, d_scr, err=d_err, stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(d_out.cpu().numpy().view(np.uint64), _identity_rows(group)) and int(d_oinf.item()) == 1
    # a limb >= p: bit 0 of d_err, no error code
    nc = rows.copy()
    nc[9, :6] = P_LIMBS
    d_nc = torch.from_numpy(nc.view(np.int64)).to(dev)
    fn(d_nc, d_k, n, d_out, d_oinf, d_st, d_scr, err=d_err, stream=s.cuda_stream)
    s.synchronize()
    assert int(d_err.item()) & 1
    with pytest.raises(z.ZkpError):
        fn(d_pts, d_k, n, d_out, d_oinf, d_st, None, stream=s.cuda_stream)


@pytest.mark.gpu
def test_gpu_msm_multi_device_equals_single(engine):
    import zkvm_pairings_b200 as z
    if z.PairingEngine is None or engine._lib.zkp_device_count() < 2:
        pytest.skip("needs two GPUs")
    multi = z.PairingEngine([0, 1])
    try:
        for group, n in (("g1", (1 << 20) + 5), ("g2", (1 << 16) + 9)):
            rows, k, want, winf = _known_dlog_case(engine, group, n, 0x5900)
            a = _engine_msm(engine, group, rows, k)
            b = _engine_msm(multi, group, rows, k)
            assert np.array_equal(a[0], b[0]) and a[1:] == b[1:] and np.array_equal(a[0], want)
    finally:
        multi.close()
