"""KZG point-evaluation verification (zkp_kzg_*): the front end's body bit-exact against pyref through the CPU dev
simulation of csrc/kzg.cuh, and the GPU entry points against the trapdoor construction of workloads.kzg_proofs, the C
oracle, a real SRS and the existing group-op + prepared multi-pairing path."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
X2 = 0xd201000000010000 ** 2
TABLE_U64 = 32 * 255 * 2 * 6
IDENTITY_XY = [0] * 6 + [1] + [0] * 5


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _fr(vals):
    return np.array([[(v >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)] for v in vals], dtype=np.uint64).reshape(-1, 4)


def _int(limbs):
    return sum(int(t) << (64 * k) for k, t in enumerate(limbs))


def _neg_g2(q):
    q = q.copy().reshape(-1, 24)
    for k in (12, 18):
        y = util.arr_fp(q[:, k:k + 6])
        q[:, k:k + 6] = np.stack([util.fp_arr([(-v) % util.o.P]) for v in y])
    return q


def _g1(coracle, ks):
    """k G1 for each k -> (points (n, 12), inf (n,)); k = 0 gives the identity as (0, 1)."""
    return coracle.g1_mul_batch(_fr([k % R for k in ks]))


@pytest.fixture(scope="module")
def sim(pyref):
    """The dev simulation with the KZG front end (its own build: the staleness list covers kzg.cuh) and the generator's
    window table it reads."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_kzg.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, "sim_kzg.cpp"), os.path.join(d, "sim.cpp"), os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    lib = ctypes.CDLL(so)
    table = np.zeros(TABLE_U64, np.uint64)
    lib.sim_kzg_table(_p(util.g1_to_arr(pyref.G1_GENERATOR)), _p(table))
    return lib, table


def _prepare(sim, proofs, zy, proof_inf=None):
    lib, table = sim
    proofs = np.ascontiguousarray(proofs, dtype=np.uint64).reshape(-1, 24)
    zy = np.ascontiguousarray(zy, dtype=np.uint64).reshape(-1, 8)
    n = proofs.shape[0]
    g1, g1inf, st = np.full((n, 24), 7, np.uint64), np.full((n, 2), 9, np.uint8), np.full(n, 9, np.uint8)
    pi = None if proof_inf is None else np.ascontiguousarray(proof_inf, dtype=np.uint8)
    lib.sim_kzg_prepare(_p(table), _p(proofs), _p(pi), _p(zy), ctypes.c_size_t(n), _p(g1), _p(g1inf), _p(st))
    return g1, g1inf, st


def _pt(a, inf=False):
    v = util.arr_fp(a)
    return (v[0], v[1], bool(inf))


def _check_p(sim, pyref, cases):
    """cases: (C (12,), C_inf, pi (12,), pi_inf, z, y).  The P slot equals pyref's C + [z]pi - [y]G1 and the pi slot
    passes pi through, with the flags; every status is 0."""
    proofs = np.stack([np.concatenate([c, q]) for c, _, q, _, _, _ in cases])
    pinf = np.array([[ci, qi] for _, ci, _, qi, _, _ in cases], np.uint8)
    zy = np.concatenate([_fr([cs[4] for cs in cases]), _fr([cs[5] for cs in cases])], axis=1)
    g1, g1inf, st = _prepare(sim, proofs, zy, pinf)
    assert not st.any()
    infs = []
    for i, (c, ci, q, qi, z, y) in enumerate(cases):
        e = pyref.g1_add(pyref.g1_add(_pt(c, ci), pyref.g1_mul(_pt(q, qi), z)), pyref.g1_neg(pyref.g1_mul(pyref.G1_GENERATOR, y)))
        assert g1inf[i, 0] == (1 if e[2] else 0), i
        want = IDENTITY_XY if e[2] else pyref.fp_to_u64(e[0]) + pyref.fp_to_u64(e[1])
        assert list(g1[i, :12]) == want, (i, hex(z), hex(y))
        assert np.array_equal(g1[i, 12:], q) and g1inf[i, 1] == qi
        infs.append(bool(e[2]))
    return infs


# ---------------------------------------------------------------- CPU: dev simulation of the device body

def test_sim_glv_split_and_endomorphism(sim, pyref):
    """z = z_hi x^2 + z_lo with z_lo < x^2 and both halves < 2^128 across the edges, and [x^2]P = (beta x, -y) on G1."""
    lib, _ = sim
    rng = random.Random(0x4841)
    for z in (0, 1, X2 - 1, X2, X2 + 1, rng.randrange(1 << 127) * X2, (1 << 128) - 1, R - 1, rng.randrange(R)):
        hi, lo = np.zeros(2, np.uint64), np.zeros(2, np.uint64)
        lib.sim_kzg_glv_split(_p(_fr([z])[0]), _p(hi), _p(lo))
        assert (_int(hi), _int(lo)) == divmod(z, X2), hex(z)
        assert _int(hi) < 1 << 128
    p = pyref.g1_mul(pyref.G1_GENERATOR, rng.randrange(1, R))
    q = pyref.g1_mul(p, X2)
    assert (q[0], q[1]) == (pyref.fp_mul(pyref.BETA, p[0]), pyref.fp_neg(p[1]))


def test_sim_p_for_edge_scalars(sim, coracle, pyref):
    """P = C + [z]pi - [y]G1 for z in {0, 1, x^2 - 1, x^2, x^2 + 1, k x^2, 2^128 - 1, r - 1, random} crossed with
    y in {0, 1, r - 1, all-0xff windows, alternating windows, random}."""
    rng = random.Random(0x4842)
    zs = [0, 1, X2 - 1, X2, X2 + 1, rng.randrange(1, 1 << 127) * X2, (1 << 128) - 1, R - 1, rng.randrange(R)]
    ys = [0, 1, R - 1, int("ff" * 31, 16), int("00ff" * 15 + "ff", 16), rng.randrange(R)]
    pts, _ = _g1(coracle, [rng.randrange(1, R) for _ in range(2 * len(zs))])
    cases = [(pts[2 * i], 0, pts[2 * i + 1], 0, z, y) for i, z in enumerate(zs) for y in ys]
    _check_p(sim, pyref, cases)


def test_sim_every_branch_of_the_partial_sums(sim, coracle, pyref):
    """The even lane's C + [z_lo]pi and the final addition of the two lanes' partial sums meet each branch: equal
    operands (doubling), opposite operands (identity, flag set), and an operand at infinity."""
    rng = random.Random(0x4843)
    q = rng.randrange(1, R)
    zh, zl = rng.randrange(1, 1 << 127), rng.randrange(1, X2)
    pi = _g1(coracle, [q])[0][0]

    def c(k):
        return _g1(coracle, [k])[0][0]
    z = zh * X2
    cases = [
        (c(z * q), 0, pi, 0, z, 0),             # y = 0, z_lo = 0: C = [z_hi] phi'(pi), the partial sums are equal
        (c(-z * q), 0, pi, 0, z, 0),            # C = -[z_hi] phi'(pi): P is the identity
        (c(7), 0, pi, 0, zl, 0),                # z_hi = 0, y = 0: the odd partial sum is the identity
        (c(-zl * q), 0, pi, 0, z + zl, 0),      # C = -[z_lo] pi: the even partial sum is the identity (mixed add: opposite)
        (c(zl * q), 0, pi, 0, z + zl, 0x100),   # C = [z_lo] pi: the mixed addition doubles
        (c(5), 1, pi, 0, 0, 0),                 # both partial sums at infinity (C flagged)
        (c(-zl * q + 1), 0, pi, 0, zl, 1),      # windows of r - 1 in both lanes, opposite partial sums: P = identity
    ]
    infs = _check_p(sim, pyref, cases)
    assert infs == [False, True, False, False, False, True, True]


def test_sim_identity_c_and_pi(sim, coracle, pyref):
    """An identity C or pi is a valid group element: it contributes nothing to P, and an identity pi's slot is flagged."""
    rng = random.Random(0x4844)
    pts, _ = _g1(coracle, [rng.randrange(1, R) for _ in range(2)])
    ident = np.array(IDENTITY_XY, np.uint64)
    z, y = rng.randrange(R), rng.randrange(R)
    _check_p(sim, pyref, [(ident, 1, pts[1], 0, z, y), (pts[0], 0, ident, 1, z, y), (ident, 1, ident, 1, z, y),
                          (pts[0], 0, np.zeros(12, np.uint64), 1, z, 0)])


def rejection_cases(pyref, coracle, proof, zy, seed=0x4845):
    """(proofs, proof_inf, zy, front-end status) rows around one proof: the unchanged row first, then one row per
    rejection class, then rows the front end passes (z = r - 1, y = 0, pi the identity)."""
    g1b, _, e1, _, _, _ = util.group_check_cases(pyref, coracle, seed=seed)
    off1, tor1 = g1b[list(e1).index(1)], g1b[list(e1).index(2)]
    z, y = _int(zy[:4]), _int(zy[4:])
    rows = []

    def add(pr, zz, yy, st, inf=(0, 0)):
        rows.append((pr, np.array(inf, np.uint8), np.concatenate([_fr([zz])[0], _fr([yy])[0]]), st))
    add(proof, z, y, 0)
    for off in (0, 12 + 6):                      # a limb vector >= p: C.x, pi.y
        pr = proof.copy()
        big = _int(proof[off:off + 6]) + pyref.P
        pr[off:off + 6] = [(big >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(6)]
        add(pr, z, y, 2)
    pr = proof.copy(); pr[:12] = off1; add(pr, z, y, 2)           # C off the curve
    pr = proof.copy(); pr[12:] = tor1; add(pr, z, y, 2)           # pi on the curve, not torsion free
    add(proof, R, y, 3)                                           # z = r
    add(proof, z, (1 << 256) - 1, 3)                              # y = 2^256 - 1
    pr = proof.copy(); pr[12:] = tor1; add(pr, R, y, 2)           # a bad point takes precedence over a bad scalar
    add(proof, R - 1, y, 0)
    add(proof, z, 0, 0)
    pr = proof.copy(); pr[12:] = 0; pr[18] = 1
    add(pr, z, y, 0, inf=(0, 1))                                  # pi = identity
    return (np.stack([r[0] for r in rows]), np.stack([r[1] for r in rows]), np.stack([r[2] for r in rows]),
            np.array([r[3] for r in rows], np.uint8))


def test_sim_statuses_and_canonical_rejected_slots(sim, coracle, pyref):
    pts, _ = _g1(coracle, [11, 13])
    proof = np.concatenate([pts[0], pts[1]])
    proofs, pinf, zy, exp = rejection_cases(pyref, coracle, proof, np.concatenate([_fr([5])[0], _fr([7])[0]]))
    g1, g1inf, st = _prepare(sim, proofs, zy, pinf)
    assert list(st) == list(exp)
    for i in np.nonzero(exp)[0]:
        assert not g1[i].any() and g1inf[i].all()
    for i in np.nonzero(exp == 0)[0]:
        assert g1inf[i, 1] == pinf[i, 1] and np.array_equal(g1[i, 12:], proofs[i, 12:])


def test_no_gpu_fails_loudly():
    """The setup and verify calls check their arguments on the host and never compute on the CPU."""
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import _lib, build
    build.build()
    lib = _lib.load()
    pt = np.zeros(24, np.uint64)
    out = ctypes.c_void_p()
    assert lib.zkp_kzg_setup_create(None, _p(pt), ctypes.byref(out)) == -1
    assert lib.zkp_kzg_setup_create(None, _p(pt), None) == -1
    st = np.zeros(1, np.uint8)
    assert lib.zkp_kzg_verify_batch(None, None, _p(pt), None, _p(pt), 1, _p(st)) == -1
    assert lib.zkp_kzg_verify_dev(None, 0, None, None, None, None, 0, None, None, None) == -1
    assert lib.zkp_kzg_scratch_bytes(1 << 10) >= (1 << 10) * (192 + 576 + 3)
    assert (z.KZG_VALID, z.KZG_INVALID, z.KZG_BAD_POINT, z.KZG_BAD_SCALAR) == (0, 1, 2, 3)
    if z.device_count() == 0:
        with pytest.raises(z.ZkpError) as ei:
            z.PairingEngine()
        assert ei.value.code == -4


# ---------------------------------------------------------------- GPU

def _oracle_is_one(coracle, w, idx):
    """The C oracle's 2-pair product (P, pi) x (G2, -[tau]G2) for the proofs idx."""
    P, pinf = coracle.g1_mul_batch(w["p"][idx])
    n = len(idx)
    g1 = np.stack([P, w["proofs"][idx, 12:]], axis=1).reshape(-1, 12)
    i1 = np.stack([pinf, np.zeros(n, np.uint8)], axis=1).reshape(-1)
    g2 = np.tile(np.concatenate([util.g2_to_arr(util.o.G2_GENERATOR)[None], _neg_g2(w["tau_g2"])]), (n, 1))
    return coracle.multi_pairing_batch(g1, i1, g2, None, 2)[1]


@pytest.mark.gpu
def test_kzg_512_proofs_match_construction_and_oracle(engine, coracle):
    from zkvm_pairings_b200 import workloads
    w = workloads.kzg_proofs(engine, 512, seed=0x512, corrupt_every=10)
    with engine.kzg_setup(w["tau_g2"]) as s:
        st = engine.kzg_verify_batch(s, w["proofs"], w["zy"])
    assert np.array_equal(st, w["expect"]) and w["expect"].sum() > 0
    assert np.array_equal(_oracle_is_one(coracle, w, np.arange(512)), 1 - w["expect"])


@pytest.mark.gpu
def test_kzg_every_rejection_class_in_one_batch(engine, coracle, pyref):
    """Every rejection class among valid proofs, which stay valid; the call returns ZKP_OK."""
    from zkvm_pairings_b200 import workloads
    w = workloads.kzg_proofs(engine, 64, seed=0x519, corrupt_every=0)
    proofs, pinf, zy, exp = rejection_cases(pyref, coracle, w["proofs"][0], w["zy"][0])
    exp[1:][exp[1:] == 0] = 1                    # passed the front end, no longer an opening: the equation decides
    allp = np.concatenate([w["proofs"][:32], proofs, w["proofs"][32:]])
    alli = np.concatenate([np.zeros((32, 2), np.uint8), pinf, np.zeros((32, 2), np.uint8)])
    allzy = np.concatenate([w["zy"][:32], zy, w["zy"][32:]])
    with engine.kzg_setup(w["tau_g2"]) as s:
        st = engine.kzg_verify_batch(s, allp, allzy, alli)
    assert list(st) == [0] * 32 + list(exp) + [0] * 32


def _sum_rows(engine, pts, inf):
    """Row sums of a (n, m, 12) point array with flags (n, m) through g1_add_batch, pairwise."""
    while pts.shape[1] > 1:
        if pts.shape[1] % 2:
            pts = np.concatenate([pts, np.tile(np.array(IDENTITY_XY, np.uint64), (pts.shape[0], 1, 1))], axis=1)
            inf = np.concatenate([inf, np.ones((inf.shape[0], 1), np.uint8)], axis=1)
        n, m = pts.shape[0], pts.shape[1] // 2
        s, f = engine.g1_add_batch(pts[:, 0::2].reshape(-1, 12), pts[:, 1::2].reshape(-1, 12), inf[:, 0::2].reshape(-1),
                                   inf[:, 1::2].reshape(-1))
        pts, inf = s.reshape(n, m, 12), (f & 1).reshape(n, m)
    return pts[:, 0], inf[:, 0]


@pytest.mark.gpu
def test_kzg_real_srs_openings(engine):
    """A degree-15 polynomial committed with the SRS [tau^i]G1 (g1_mul_batch / g1_add_batch), 32 openings with pi from
    the quotient by synthetic division: all verify, and one wrong y is rejected."""
    rng = random.Random(0x5125)
    tau = rng.randrange(1, R)
    f = [rng.randrange(R) for _ in range(16)]
    g1gen, g2gen = util.g1_to_arr(util.o.G1_GENERATOR), util.g2_to_arr(util.o.G2_GENERATOR)
    srs, srs_inf = engine.g1_mul_batch(np.tile(g1gen, (16, 1)), _fr([pow(tau, i, R) for i in range(16)]))
    tg, _ = engine.g2_mul_batch(g2gen[None], _fr([tau]))
    cm, ci = engine.g1_mul_batch(srs, _fr(f), srs_inf)
    C, cinf = _sum_rows(engine, cm[None], ci[None])
    zs = [rng.randrange(R) for _ in range(32)]
    ys, quots = [], []
    for z in zs:
        qs, acc = [0] * 15, f[15]
        for i in range(14, -1, -1):              # synthetic division by (X - z): f = q (X - z) + f(z)
            qs[i] = acc
            acc = (acc * z + f[i]) % R
        ys.append(acc)
        quots.append(qs)
    pm, pmi = engine.g1_mul_batch(np.tile(srs[:15], (32, 1)), _fr([c for qs in quots for c in qs]), np.tile(srs_inf[:15], 32))
    pi, pinf = _sum_rows(engine, pm.reshape(32, 15, 12), pmi.reshape(32, 15))
    proofs = np.concatenate([np.tile(C, (32, 1)), pi], axis=1)
    flags = np.stack([np.repeat(cinf, 32), pinf], axis=1)
    zy = np.concatenate([_fr(zs), _fr(ys)], axis=1)
    zy[5, 4:] = _fr([(ys[5] + 3) % R])[0]
    with engine.kzg_setup(tg[0]) as s:
        st = engine.kzg_verify_batch(s, proofs, zy, flags)
    assert list(st) == [0] * 5 + [1] + [0] * 26


@pytest.mark.gpu
def test_kzg_full_size_and_every_path(engine, coracle):
    """2^18 + 37 proofs (one chunk boundary), 1 % corrupted: the verdicts equal the construction and the is_one of the
    existing path on the same data (P from g1_mul_batch + g1_add_batch, then the prepared 2-pair multi-pairing), an
    oracle sample agrees; pageable, pinned, n = 0 and the _dev form on the default stream give the same statuses, and
    the caller's device is left unchanged."""
    import torch
    from zkvm_pairings_b200 import workloads
    n = (1 << 18) + 37
    w = workloads.kzg_proofs(engine, n, seed=0x218)
    pr, zy = w["proofs"], w["zy"]
    with engine.kzg_setup(w["tau_g2"]) as s:
        st = engine.kzg_verify_batch(s, pr, zy)
        assert np.array_equal(st, w["expect"]) and int(w["expect"].sum()) == n // 100 + (1 if n % 100 > 7 else 0)

        g1gen = util.g1_to_arr(util.o.G1_GENERATOR)
        ny = _fr([(R - _int(v)) % R for v in zy[:, 4:]])
        zp, zi = engine.g1_mul_batch(pr[:, 12:], zy[:, :4])
        yg, yi = engine.g1_mul_batch(np.tile(g1gen, (n, 1)), ny)
        t, ti = engine.g1_add_batch(pr[:, :12], zp, None, zi)
        P, pf = engine.g1_add_batch(t, yg, ti & 1, yi)
        g1 = np.stack([P, pr[:, 12:]], axis=1).reshape(-1, 12)
        g1inf = np.stack([pf & 1, np.zeros(n, np.uint8)], axis=1).reshape(-1)
        tabs = engine.g2_prepare_batch(np.concatenate([util.g2_to_arr(util.o.G2_GENERATOR)[None], _neg_g2(w["tau_g2"])]))
        _, one = engine.multi_pairing_prepared_batch(g1, None, 2, tabs, g1_inf=g1inf)
        assert np.array_equal(one, (st == 0).astype(np.uint8))
        idx = np.arange(3, n, 4099)
        assert np.array_equal(_oracle_is_one(coracle, w, idx), 1 - w["expect"][idx])

        pp = torch.from_numpy(pr.view(np.int64)).pin_memory()
        pz = torch.from_numpy(np.ascontiguousarray(zy).view(np.int64)).pin_memory()
        assert np.array_equal(engine.kzg_verify_batch(s, pp.numpy().view(np.uint64), pz.numpy().view(np.uint64)), st)
        assert engine.kzg_verify_batch(s, pr[:0], zy[:0]).shape == (0,)
        before = torch.cuda.current_device()
        assert torch.cuda.current_stream().cuda_stream == 0
        big = torch.zeros((1 << 26,), dtype=torch.int64, device="cuda")      # keeps the default stream busy first
        big += 1
        dp = pp.cuda(non_blocking=True)
        dz = pz.cuda(non_blocking=True)
        ds = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
        scratch = torch.empty(engine.kzg_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        engine.kzg_verify_dev(s, dp, dz, n, ds, scratch, stream=0)
        engine.kzg_verify_dev(s, dp, dz, 0, ds, scratch, stream=0)
        host = ds.cpu().numpy()                                                 # default-stream consumer, no sync call
        assert torch.cuda.current_device() == before
        assert np.array_equal(host, st)


@pytest.mark.gpu
def test_kzg_setup_checks(engine, coracle, pyref):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    w = workloads.kzg_proofs(engine, 8, seed=0x522, corrupt_every=0)
    _, _, _, g2b, _, e2 = util.group_check_cases(pyref, coracle, seed=0x523)
    big = w["tau_g2"].copy()
    big[5] = 0xFFFFFFFFFFFFFFFF
    with pytest.raises(z.NonCanonicalError) as ei:
        engine.kzg_setup(big)
    assert ei.value.code == -3
    for bad in (g2b[list(e2).index(1)], g2b[list(e2).index(2)]):
        with pytest.raises(z.ZkpError) as ei:
            engine.kzg_setup(bad)
        assert ei.value.code == -1 and "tau_g2" in str(ei.value), str(ei.value)
    other = z.PairingEngine([0])
    try:
        with engine.kzg_setup(w["tau_g2"]) as s:
            with pytest.raises(z.ZkpError) as ei:
                other.kzg_verify_batch(s, w["proofs"], w["zy"])
            assert ei.value.code == -1 and "another context" in str(ei.value)
            assert list(engine.kzg_verify_batch(s, w["proofs"], w["zy"])) == [0] * 8
        with pytest.raises(ValueError):
            engine.kzg_verify_batch(s, w["proofs"], w["zy"])
    finally:
        other.close()


@pytest.mark.gpu
def test_kzg_multi_device_matches_single(engine):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    if z.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    w = workloads.kzg_proofs(engine, 3001, seed=0x524)
    multi = z.PairingEngine()
    try:
        with engine.kzg_setup(w["tau_g2"]) as s1, multi.kzg_setup(w["tau_g2"]) as sm:
            assert np.array_equal(engine.kzg_verify_batch(s1, w["proofs"], w["zy"]), multi.kzg_verify_batch(sm, w["proofs"], w["zy"]))
    finally:
        multi.close()
