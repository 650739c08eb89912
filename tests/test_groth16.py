"""Groth16 verification (zkp_groth16_*): the front end's bodies bit-exact against the oracle through the CPU dev
simulation of csrc/groth16.cuh, and the GPU entry points against the trapdoor construction of
workloads.groth16_proofs, the C oracle and the existing prepared multi-pairing path."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
TABLE_U64 = 32 * 255 * 2 * 6


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _fr(vals):
    return np.array([[(v >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)] for v in vals], dtype=np.uint64).reshape(-1, 4)


@pytest.fixture(scope="module")
def sim():
    """The dev simulation with the Groth16 front end (its own build: the staleness list covers groth16.cuh)."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_g16.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, "sim_groth16.cpp"), os.path.join(d, "sim.cpp"), os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    return ctypes.CDLL(so)


def _g1_points(coracle, scalars):
    """k G1 for each k (None = the identity) -> (points (n, 12), inf (n,))."""
    ks = [0 if k is None else k % R for k in scalars]
    pts, inf = coracle.g1_mul_batch(_fr(ks))
    return pts, inf


def _neg_g2(q):
    q = q.copy().reshape(-1, 24)
    for k in (12, 18):
        y = util.arr_fp(q[:, k:k + 6])
        q[:, k:k + 6] = np.stack([util.fp_arr([(-v) % util.o.P]) for v in y])
    return q


class SimKey:
    """A verifying key run through the simulated front end: IC_j = u_j G1 (u_j None = the identity)."""

    def __init__(self, sim, coracle, us, alpha=5):
        self.sim, self.us, self.n_public = sim, us, len(us) - 1
        self.ic, inf = _g1_points(coracle, us)
        self.ic_inf = np.array([1 if u is None else 0 for u in us], np.uint8)
        assert np.array_equal(inf, self.ic_inf)
        self.alpha = _g1_points(coracle, [alpha])[0][0]
        self.tables = np.zeros(max(1, self.n_public) * TABLE_U64, np.uint64)
        sim.sim_g16_tables(_p(self.ic), _p(self.ic_inf), self.n_public, _p(self.tables))

    def prepare(self, proofs, xs, proof_inf=None):
        n = proofs.shape[0]
        x = np.ascontiguousarray(np.array(xs, dtype=np.uint64).reshape(n, self.n_public * 4)) if self.n_public else np.zeros((n, 1), np.uint64)
        g1, g1inf = np.full((n, 48), 7, np.uint64), np.full((n, 4), 9, np.uint8)
        g2, g2inf, st = np.full((n, 24), 7, np.uint64), np.full(n, 9, np.uint8), np.full(n, 9, np.uint8)
        pi = None if proof_inf is None else np.ascontiguousarray(proof_inf, dtype=np.uint8)
        self.sim.sim_g16_prepare(_p(self.alpha), _p(self.ic[0]), _p(self.ic_inf), _p(self.tables), self.n_public, _p(proofs), _p(pi),
                                 _p(x), ctypes.c_size_t(n), _p(g1), _p(g1inf), _p(g2), _p(g2inf), _p(st))
        return g1, g1inf, g2, g2inf, st


def _valid_proof(coracle, seed=3):
    g1, _, g2, _ = util.oracle_points(coracle, seed, 0, 2)
    return np.concatenate([g1[0], g2[0], g1[1]])


# ---------------------------------------------------------------- CPU: dev simulation of the device bodies

def test_sim_window_table_entries(sim, coracle, pyref):
    """Entry (w, d) of IC_j's table is d 2^(8w) IC_j, for sampled windows and digits (the last one included)."""
    u = 0x1234567890ABCDEF1234567890ABCDEF
    key = SimKey(sim, coracle, [None, 77, u])
    ic = (util.arr_fp(key.ic[2][:6])[0], util.arr_fp(key.ic[2][6:])[0], False)
    for w, d in ((0, 1), (0, 2), (0, 255), (1, 1), (7, 128), (16, 3), (30, 254), (31, 255)):
        xy = np.zeros(12, np.uint64)
        sim.sim_g16_table_entry(_p(key.tables), 1, w, d, _p(xy))
        e = pyref.g1_mul(ic, d << (8 * w))
        assert not e[2] and list(xy) == pyref.fp_to_u64(e[0]) + pyref.fp_to_u64(e[1]), (w, d)
    xy = np.zeros(12, np.uint64)
    sim.sim_g16_table_entry(_p(key.tables), 0, 31, 255, _p(xy))
    assert np.array_equal(xy, coracle.g1_mul_batch(_fr([(255 << 248) * 77 % R]))[0][0])


def _check_accumulation(sim, coracle, us, xs, proof):
    key = SimKey(sim, coracle, us)
    n = len(xs)
    proofs = np.tile(proof, (n, 1))
    g1, g1inf, g2, g2inf, st = key.prepare(proofs, [_fr(x) if x else np.zeros((0, 4), np.uint64) for x in xs])
    assert not st.any()
    ls = [(us[0] or 0) + sum(xj * (uj or 0) for xj, uj in zip(x, us[1:])) for x in xs]
    exp, einf = _g1_points(coracle, ls)
    for i in range(n):
        assert g1inf[i, 2] == einf[i], i
        if einf[i]:
            assert list(g1[i, 24:36]) == [0] * 6 + [1] + [0] * 5        # the identity as (0, 1)
        else:
            assert np.array_equal(g1[i, 24:36], exp[i]), i
        assert np.array_equal(g1[i, :12], proof[:12]) and np.array_equal(g1[i, 12:24], key.alpha)
        assert np.array_equal(g1[i, 36:], proof[36:]) and np.array_equal(g2[i], proof[12:36])
        assert list(g1inf[i, [0, 1, 3]]) == [0, 0, 0] and g2inf[i] == 0
    return ls


def test_sim_accumulation_edge_scalars(sim, coracle):
    """L = IC_0 + sum x_j IC_j for l in {0, 1, 2, 5}, scalars 0, 1, r - 1 and ones with all-zero and all-0xFF windows."""
    rng = random.Random(0x616)
    proof = _valid_proof(coracle)
    ff = int("ff" * 31, 16)                     # windows 0..30 = 0xff, window 31 = 0
    alt = int("00ff" * 15 + "ff", 16)           # alternating zero / 0xff windows
    edges = [0, 1, R - 1, ff, alt, 1 << 248, 0xff << 240, rng.randrange(R)]
    for lp in (0, 1, 2, 5):
        us = [rng.randrange(1, R) for _ in range(lp + 1)]
        xs = [[edges[(i + j) % len(edges)] for j in range(lp)] for i in range(len(edges) if lp else 1)]
        _check_accumulation(sim, coracle, us, xs, proof)


def test_sim_accumulation_identity_ic_and_partial_sum_branches(sim, coracle):
    """An identity IC_j contributes nothing; the final addition of the two lanes' partial sums (even lane:
    IC_0 + the even windows, odd lane: the odd windows) meets each of its branches: equal operands (doubling),
    opposite operands (identity), an operand at infinity; and the shapes IC_1 = IC_2 with x_1 = x_2,
    x_2 = r - x_1 and IC_0 = -sum (L the identity, flag set)."""
    rng = random.Random(0x617)
    proof = _valid_proof(coracle, seed=5)
    u1 = rng.randrange(1, R)
    x = rng.randrange(R)
    _check_accumulation(sim, coracle, [rng.randrange(1, R), u1, None], [[x, rng.randrange(R)], [0, 5]], proof)
    # even partial = IC_0 = 2^8 IC_1, odd partial = window 1 of x_1 = 1  ->  equal: doubling
    _check_accumulation(sim, coracle, [256 * u1 % R, u1], [[0x100]], proof)
    # IC_0 = -2^8 IC_1: opposite partial sums -> L = identity
    ls = _check_accumulation(sim, coracle, [(-256 * u1) % R, u1], [[0x100]], proof)
    assert ls[0] % R == 0
    # odd partial at infinity (x only in even windows, or zero); even partial at infinity (IC_0 identity, odd windows only)
    _check_accumulation(sim, coracle, [rng.randrange(1, R), u1], [[0], [0xff00ff], [0x42]], proof)
    _check_accumulation(sim, coracle, [None, u1], [[0x100], [0xff00ff00], [0]], proof)
    # the shapes of an input-split accumulation
    _check_accumulation(sim, coracle, [None, u1, u1], [[x, x], [x, R - x]], proof)
    s = (x * u1 + 3 * u1) % R
    ls = _check_accumulation(sim, coracle, [(-s) % R, u1, u1], [[x, 3]], proof)
    assert ls[0] % R == 0


def rejection_cases(pyref, coracle, proof, x, seed=0x618):
    """(proofs, proof_inf, inputs, front-end status) rows around one proof with inputs x: the unchanged row first,
    then one row per rejection class, then rows the front end passes that are no longer solutions (x_1 = r - 1,
    A replaced by the identity)."""
    g1b, _, e1, g2b, _, e2 = util.group_check_cases(pyref, coracle, seed=seed)
    off1, tor1 = g1b[list(e1).index(1)], g1b[list(e1).index(2)]
    tor2 = g2b[list(e2).index(2)]                # on E'(Fp2), lifted with fp2_sqrt, not in G2
    rows = []

    def add(pr, xs, st, inf=(0, 0, 0)):
        rows.append((pr, np.array(inf, np.uint8), list(xs), st))
    add(proof, x, 0)
    for off in (0, 12 + 18, 36 + 6):             # a limb vector >= p: A.x, B.y.c1, C.y
        pr = proof.copy()
        big = sum(int(t) << (64 * k) for k, t in enumerate(proof[off:off + 6])) + pyref.P
        pr[off:off + 6] = [(big >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(6)]
        add(pr, x, 2)
    pr = proof.copy(); pr[:12] = off1; add(pr, x, 2)          # A off the curve
    pr = proof.copy(); pr[12:36] = tor2; add(pr, x, 2)        # B on E'(Fp2), not in G2
    pr = proof.copy(); pr[36:] = tor1; add(pr, x, 2)          # C on E(Fp), not torsion free
    if x:
        add(proof, [R] + x[1:], 3)
        add(proof, x[:-1] + [(1 << 256) - 1], 3)
        pr = proof.copy(); pr[36:] = tor1; add(pr, [R] + x[1:], 2)   # a bad point takes precedence
        add(proof, [R - 1] + x[1:], 0)
    pr = proof.copy(); pr[:12] = 0; pr[6] = 1
    add(pr, x, 0, inf=(1, 0, 0))                 # A = identity: a valid group element
    proofs = np.stack([r[0] for r in rows])
    pinf = np.stack([r[1] for r in rows])
    xs = np.stack([_fr(r[2]) if x else np.zeros((0, 4), np.uint64) for r in rows])
    return proofs, pinf, xs, np.array([r[3] for r in rows], np.uint8)


def test_sim_prepare_statuses_and_canonical_rejected_slots(sim, coracle, pyref):
    key = SimKey(sim, coracle, [11, 13])
    proof = _valid_proof(coracle, seed=9)
    proofs, pinf, xs, exp = rejection_cases(pyref, coracle, proof, [1])
    g1, g1inf, g2, g2inf, st = key.prepare(proofs, xs, pinf)
    assert list(st) == list(exp)
    for i in np.nonzero(exp)[0]:
        assert not g1[i].any() and not g2[i].any() and g1inf[i].all() and g2inf[i] == 1
    for i in np.nonzero(exp == 0)[0]:
        assert g1inf[i, 0] == pinf[i, 0] and g1inf[i, 1] == 0 and g2inf[i] == 0


def test_no_gpu_fails_loudly():
    """The key and verify calls check their arguments on the host and never compute on the CPU."""
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import _lib, build
    build.build()
    lib = _lib.load()
    pt = np.zeros(24, np.uint64)
    out = ctypes.c_void_p()
    assert lib.zkp_groth16_vk_create(None, _p(pt), _p(pt), _p(pt), _p(pt), _p(pt), None, 0, ctypes.byref(out)) == -1
    assert lib.zkp_groth16_vk_create(None, _p(pt), _p(pt), _p(pt), _p(pt), _p(pt), None, 0, None) == -1
    st = np.zeros(1, np.uint8)
    assert lib.zkp_groth16_verify_batch(None, None, _p(pt), None, None, 1, _p(st)) == -1
    assert lib.zkp_groth16_verify_dev(None, 0, None, None, None, None, 0, None, None, None) == -1
    assert lib.zkp_groth16_scratch_bytes(1 << 10) >= (1 << 10) * (384 + 192 + 576 + 6)
    if z.device_count() == 0:
        with pytest.raises(z.ZkpError) as ei:
            z.PairingEngine()
        assert ei.value.code == -4


# ---------------------------------------------------------------- GPU

def _key(engine, w):
    return engine.groth16_prepare_vk(w["alpha"], w["beta"], w["gamma"], w["delta"], w["ic"])


def _oracle_is_one(coracle, w, idx):
    """The C oracle's 4-pair product (A, alpha, L, C) x (B, -beta, -gamma, -delta) for the proofs idx."""
    pr = w["proofs"][idx]
    L, linf = coracle.g1_mul_batch(w["l"][idx])
    n = len(idx)
    g1 = np.stack([pr[:, :12], np.tile(w["alpha"], (n, 1)), L, pr[:, 36:]], axis=1).reshape(-1, 12)
    i1 = np.stack([np.zeros(n, np.uint8), np.zeros(n, np.uint8), linf, np.zeros(n, np.uint8)], axis=1).reshape(-1)
    fixed = _neg_g2(np.stack([w["beta"], w["gamma"], w["delta"]]))
    g2 = np.concatenate([pr[:, None, 12:36], np.tile(fixed[None], (n, 1, 1))], axis=1).reshape(-1, 24)
    return coracle.multi_pairing_batch(g1, i1, g2, None, 4)[1]


@pytest.mark.gpu
def test_groth16_512_proofs_match_construction_and_oracle(engine, coracle):
    from zkvm_pairings_b200 import workloads
    w = workloads.groth16_proofs(engine, 512, 3, seed=0x512, corrupt_every=10)
    with _key(engine, w) as vk:
        assert vk.n_public == 3
        st = engine.groth16_verify_batch(vk, w["proofs"], w["inputs"])
    assert np.array_equal(st, w["expect"]) and w["expect"].sum() > 0
    one = _oracle_is_one(coracle, w, np.arange(512))
    assert np.array_equal(one, 1 - w["expect"])


@pytest.mark.gpu
def test_groth16_every_rejection_class_in_one_batch(engine, coracle, pyref):
    """Every rejection class among valid proofs, which stay valid; the call returns ZKP_OK."""
    from zkvm_pairings_b200 import workloads
    w = workloads.groth16_proofs(engine, 64, 2, seed=0x519, corrupt_every=0)
    x0 = [sum(int(t) << (64 * k) for k, t in enumerate(v)) for v in w["inputs"][0]]
    proofs, pinf, xs, exp = rejection_cases(pyref, coracle, w["proofs"][0], x0)
    exp[1:][exp[1:] == 0] = 1                    # passed the front end, no longer a solution: the equation decides
    allp = np.concatenate([w["proofs"][:32], proofs, w["proofs"][32:]])
    alli = np.concatenate([np.zeros((32, 3), np.uint8), pinf, np.zeros((32, 3), np.uint8)])
    allx = np.concatenate([w["inputs"][:32], xs, w["inputs"][32:]])
    with _key(engine, w) as vk:
        st = engine.groth16_verify_batch(vk, allp, allx, alli)
    assert list(st) == [0] * 32 + list(exp) + [0] * 32


@pytest.mark.gpu
def test_groth16_identity_a_accepted(engine):
    """A = identity is a valid group element: with a = 0 the proof C = -(alpha beta + l gamma) / delta G1 verifies."""
    rng = random.Random(1)
    alpha, beta, gamma, delta = (rng.randrange(1, R) for _ in range(4))
    u = [rng.randrange(1, R) for _ in range(2)]
    g1gen, g2gen = util.g1_to_arr(util.o.G1_GENERATOR), util.g2_to_arr(util.o.G2_GENERATOR)
    k1, _ = engine.g1_mul_batch(np.tile(g1gen, (3, 1)), _fr([alpha] + u))
    k2, _ = engine.g2_mul_batch(np.tile(g2gen, (3, 1)), _fr([beta, gamma, delta]))
    x = [R - 1, 0, 12345]
    cs = [(-(alpha * beta) - (u[0] + xi * u[1]) * gamma) * pow(delta, -1, R) % R for xi in x]
    C, _ = engine.g1_mul_batch(np.tile(g1gen, (3, 1)), _fr(cs))
    B, _ = engine.g2_mul_batch(np.tile(g2gen, (3, 1)), _fr([7, 8, 9]))
    A = np.zeros((3, 12), np.uint64)
    A[:, 6] = 1
    proofs = np.concatenate([A, B, C], axis=1)
    pinf = np.array([[1, 0, 0]] * 3, np.uint8)
    with engine.groth16_prepare_vk(k1[0], k2[0], k2[1], k2[2], k1[1:]) as vk:
        st = engine.groth16_verify_batch(vk, proofs, _fr(x).reshape(3, 1, 4), pinf)
        assert list(st) == [0, 0, 0]
        pinf[1, 0] = 0                               # the same limbs without the flag: (0, 1) is not a curve point
        assert list(engine.groth16_verify_batch(vk, proofs, _fr(x).reshape(3, 1, 4), pinf)) == [0, 2, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("n_public", [0, 1, 2, 16, 256])
def test_groth16_public_input_counts(engine, n_public):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    assert z.GROTH16_MAX_PUBLIC == 256
    w = workloads.groth16_proofs(engine, 96, n_public, seed=0x520 + n_public, corrupt_every=7)
    with _key(engine, w) as vk:
        st = engine.groth16_verify_batch(vk, w["proofs"], w["inputs"])
    assert np.array_equal(st, w["expect"])


@pytest.mark.gpu
def test_groth16_full_size_2p18(engine, coracle):
    """2^18 proofs, l = 2, 1 % corrupted: the verdicts equal the construction, and the is_one of the existing
    prepared 4-pair call on the same pairs -- L from g1_mul_batch + g1_add_batch -- agrees, plus an oracle sample."""
    from zkvm_pairings_b200 import workloads
    n = 1 << 18
    w = workloads.groth16_proofs(engine, n, 2, seed=0x218)
    with _key(engine, w) as vk:
        st = engine.groth16_verify_batch(vk, w["proofs"], w["inputs"])
    assert np.array_equal(st, w["expect"]) and int(w["expect"].sum()) == n // 100 + (1 if n % 100 > 7 else 0)
    ic = w["ic"]
    p1, i1 = engine.g1_mul_batch(np.tile(ic[1], (n, 1)), w["inputs"][:, 0])
    p2, i2 = engine.g1_mul_batch(np.tile(ic[2], (n, 1)), w["inputs"][:, 1])
    s, f = engine.g1_add_batch(p1, p2, i1, i2)
    L, fl = engine.g1_add_batch(s, np.tile(ic[0], (n, 1)), f & 1, None)
    pr = w["proofs"]
    g1 = np.stack([pr[:, :12], np.tile(w["alpha"], (n, 1)), L, pr[:, 36:]], axis=1).reshape(-1, 12)
    g1inf = np.zeros((n, 4), np.uint8)
    g1inf[:, 2] = fl & 1
    tabs = engine.g2_prepare_batch(_neg_g2(np.stack([w["beta"], w["gamma"], w["delta"]])))
    _, one = engine.multi_pairing_prepared_batch(g1, pr[:, 12:36], 4, tabs, g1_inf=g1inf.reshape(-1))
    assert np.array_equal(one, (st == 0).astype(np.uint8))
    idx = np.arange(3, n, 4099)
    assert np.array_equal(_oracle_is_one(coracle, w, idx), 1 - w["expect"][idx])


@pytest.mark.gpu
def test_groth16_host_and_dev_paths_agree(engine):
    """Pageable and pinned host buffers, ragged n across the l-dependent chunk boundary (8192 proofs per chunk at
    l = 256), n = 0, and the _dev form on the default stream: identical statuses, caller's device untouched."""
    import torch
    from zkvm_pairings_b200 import workloads
    n = 8192 + 37
    w = workloads.groth16_proofs(engine, n, 256, seed=0x521, corrupt_every=50)
    with _key(engine, w) as vk:
        st = engine.groth16_verify_batch(vk, w["proofs"], w["inputs"])
        assert np.array_equal(st, w["expect"])
        pp = torch.from_numpy(w["proofs"].view(np.int64)).pin_memory()
        px = torch.from_numpy(np.ascontiguousarray(w["inputs"]).view(np.int64)).pin_memory()
        st2 = engine.groth16_verify_batch(vk, pp.numpy().view(np.uint64), px.numpy().view(np.uint64))
        assert np.array_equal(st2, st)
        assert engine.groth16_verify_batch(vk, w["proofs"][:0], w["inputs"][:0]).shape == (0,)
        before = torch.cuda.current_device()
        assert torch.cuda.current_stream().cuda_stream == 0
        big = torch.zeros((1 << 26,), dtype=torch.int64, device="cuda")      # keeps the default stream busy first
        big += 1
        dp = pp.cuda(non_blocking=True)
        dx = px.cuda(non_blocking=True)
        ds = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
        scratch = torch.empty(engine.groth16_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        engine.groth16_verify_dev(vk, dp, dx, n, ds, scratch, stream=0)
        engine.groth16_verify_dev(vk, dp, dx, 0, ds, scratch, stream=0)
        host = ds.cpu().numpy()                                                 # default-stream consumer, no sync call
        assert torch.cuda.current_device() == before
        assert np.array_equal(host, st)


@pytest.mark.gpu
def test_groth16_vk_checks(engine, coracle, pyref):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    w = workloads.groth16_proofs(engine, 8, 2, seed=0x522, corrupt_every=0)
    g1b, _, e1, g2b, _, e2 = util.group_check_cases(pyref, coracle, seed=0x523)
    off1, tor1, off2, tor2 = g1b[list(e1).index(1)], g1b[list(e1).index(2)], g2b[list(e2).index(1)], g2b[list(e2).index(2)]
    base = dict(alpha=w["alpha"], beta=w["beta"], gamma=w["gamma"], delta=w["delta"], ic=w["ic"])

    def bad(code, name, **kw):
        args = dict(base, **kw)
        with pytest.raises(z.ZkpError) as ei:
            engine.groth16_prepare_vk(**args)
        assert ei.value.code == code
        if name:
            assert name in str(ei.value), str(ei.value)
    big = w["alpha"].copy()
    big[5] = 0xFFFFFFFFFFFFFFFF
    bad(-3, None, alpha=big)
    bad(-1, "alpha_g1", alpha=off1)
    bad(-1, "beta_g2", beta=off2)
    bad(-1, "gamma_g2", gamma=tor2)
    bad(-1, "delta_g2", delta=off2)
    ic = w["ic"].copy()
    ic[1] = tor1
    bad(-1, "ic_g1[1]", ic=ic)
    bad(-1, "n_public", ic=np.tile(w["ic"][0], (258, 1)))
    other = z.PairingEngine([0])
    try:
        with _key(engine, w) as vk:
            with pytest.raises(z.ZkpError) as ei:
                other.groth16_verify_batch(vk, w["proofs"], w["inputs"])
            assert ei.value.code == -1 and "another context" in str(ei.value)
            assert list(engine.groth16_verify_batch(vk, w["proofs"], w["inputs"])) == [0] * 8
    finally:
        other.close()


@pytest.mark.gpu
def test_groth16_multi_device_matches_single(engine):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    if z.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    w = workloads.groth16_proofs(engine, 3001, 2, seed=0x524)
    multi = z.PairingEngine()
    try:
        with _key(engine, w) as vk1, _key(multi, w) as vkm:
            assert np.array_equal(engine.groth16_verify_batch(vk1, w["proofs"], w["inputs"]),
                                  multi.groth16_verify_batch(vkm, w["proofs"], w["inputs"]))
    finally:
        multi.close()
