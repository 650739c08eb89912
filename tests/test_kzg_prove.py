"""EIP-4844 commitments and proofs (zkp_kzg_setup_create_prover, zkp_kzg_blob_to_commitment_*, zkp_kzg_compute_proof_*,
zkp_kzg_compute_blob_proof_*): the signed-digit recoding, the window tables and the quotient rows bit-exact against
pyref and a line-by-line restatement of the consensus specs through the CPU dev simulation of csrc/kzg_prove.cuh, and
the GPU entry points against oracles independent of the MSM: [p(tau)]G1 and [q(tau)]G1 through g1_mul_batch, and the
existing verification calls."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
N = 4096
BLOB_BYTES = 32 * N
RF = (1 << 256) % R
M64 = (1 << 64) - 1


# ---------------------------------------------------------------- the consensus specs (deneb polynomial-commitments.md)

def _roots_brp():
    w = pow(7, (R - 1) // N, R)
    roots = [pow(w, k, R) for k in range(N)]
    return [roots[int(format(i, "012b")[::-1], 2)] for i in range(N)]


ROOTS_BRP = _roots_brp()


def evaluate_polynomial_in_evaluation_form(polynomial, z):
    if z in ROOTS_BRP:
        return polynomial[ROOTS_BRP.index(z)]
    result = 0
    for i in range(N):
        result += polynomial[i] * ROOTS_BRP[i] % R * pow((z - ROOTS_BRP[i]) % R, -1, R)
    return result % R * ((pow(z, N, R) - 1) * pow(N, -1, R) % R) % R


def compute_quotient_eval_within_domain(z, polynomial, y):
    result = 0
    for i, omega_i in enumerate(ROOTS_BRP):
        if omega_i == z:
            continue
        f_i = (polynomial[i] - y) % R
        numerator = f_i * omega_i % R
        denominator = z * (z - omega_i) % R
        result += numerator * pow(denominator, -1, R)
    return result % R


def compute_kzg_proof_impl_quotient(polynomial, z):
    """The quotient polynomial and y of compute_kzg_proof_impl (before its g1_lincomb)."""
    y = evaluate_polynomial_in_evaluation_form(polynomial, z)
    q = [0] * N
    for i, (p, x) in enumerate(zip(polynomial, ROOTS_BRP)):
        b = (x - z) % R
        q[i] = compute_quotient_eval_within_domain(ROOTS_BRP[i], polynomial, y) if b == 0 else (p - y) * pow(b, -1, R) % R
    return q, y


# ---------------------------------------------------------------- helpers

def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _fr(vals):
    return np.array([[(v >> (64 * k)) & M64 for k in range(4)] for v in vals], dtype=np.uint64).reshape(-1, 4)


def _int(limbs):
    return sum(int(t) << (64 * k) for k, t in enumerate(limbs))


def _blob(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "big") for v in vals), dtype=np.uint8).copy()


def _row_ints(row):
    b = bytes(row)
    return [int.from_bytes(b[32 * i:32 * i + 32], "big") for i in range(N)]


def _random_blobs(seed, n):
    """n blobs of seeded random elements < 2^254 < r (numpy, for large batches)."""
    b = np.random.default_rng(seed).integers(0, 256, size=(n, N, 32), dtype=np.uint8)
    b[:, :, 0] &= 0x3F
    return b.reshape(n, BLOB_BYTES)


@pytest.fixture(scope="module")
def sim():
    """The dev simulation with the prover front end (its own build: the staleness list covers every device header)."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_kzg_prove.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, "sim_kzg_prove.cpp"), os.path.join(d, "sim_kzg_blob.cpp"), os.path.join(d, "sim.cpp"),
           os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    return ctypes.CDLL(so)


def _domain(sim):
    d = np.zeros((N, 4), np.uint64)
    sim.sim_blob_domain(_p(d))
    return d


def _digits(sim, s):
    out = np.zeros(33, np.int32)
    sim.sim_msm_digits(_p(np.frombuffer(s.to_bytes(32, "big"), np.uint8).copy()), _p(out))
    return [int(v) for v in out[:32]], int(out[32])


def _quotient(sim, blobs, zs):
    """k_kzg_quotient's body for compute_kzg_proof: (rows as ints, y, status) per blob."""
    blobs = np.ascontiguousarray(blobs, np.uint8).reshape(-1, BLOB_BYTES)
    n = blobs.shape[0]
    zy, y, st = np.zeros((n, 8), np.uint64), np.zeros((n, 4), np.uint64), np.zeros(n, np.uint8)
    rows = np.zeros((n, BLOB_BYTES), np.uint8)
    sim.sim_kzg_quotient(_p(blobs), _p(_domain(sim)), _p(_fr(zs)), ctypes.c_size_t(n), _p(zy), _p(y), _p(rows), None, _p(st))
    return [(_row_ints(rows[b]), _int(y[b]), int(st[b])) for b in range(n)]


# ---------------------------------------------------------------- CPU: dev simulation of the device bodies

def test_sim_signed_digits_at_the_edges(sim):
    """The recoding gives digits in [-127, 128] that sum back to the scalar: 0, 1, r - 1, bytes 0x80 (digit 128, no
    carry), 0x81 and 0xff (negative digits and carries), 2^256 - 1 (the carry out of the top window) and random values;
    no scalar < r carries out of the top window."""
    rng = random.Random(0xD161)
    assert _digits(sim, 0) == ([0] * 32, 0)
    assert _digits(sim, 1) == ([1] + [0] * 31, 0)
    assert _digits(sim, 0x80) == ([128] + [0] * 31, 0)
    assert _digits(sim, 0x81) == ([-127, 1] + [0] * 30, 0)
    assert _digits(sim, 0xFF) == ([-1, 1] + [0] * 30, 0)
    assert _digits(sim, (1 << 256) - 1) == ([-1] + [0] * 31, 1)
    assert _digits(sim, int("80" * 32, 16)) == ([128] * 32, 0)
    vals = [R - 1, R - 2, (1 << 255) - 1, int("ff" * 31, 16), int("7f" * 32, 16), int("81" * 32, 16), int("ff" * 16 + "00" * 16, 16)]
    vals += [rng.getrandbits(256) for _ in range(40)] + [rng.randrange(R) for _ in range(40)]
    for s in vals:
        d, carry = _digits(sim, s)
        assert all(-127 <= x <= 128 for x in d), hex(s)
        assert sum(x << (8 * w) for w, x in enumerate(d)) + (carry << 256) == s, hex(s)
        if s < R:
            assert carry == 0 and d[31] >= 0, hex(s)


def test_sim_window_table_entries_match_pyref(sim, pyref):
    """Entries d 2^(8w) P, d = 1 .. 128, of windows 0, 1, 17 and 31 for a random subgroup point, bit-exact against the
    Python oracle's affine arithmetic."""
    rng = random.Random(0x7AB1)
    P = pyref.g1_mul(pyref.G1_GENERATOR, rng.randrange(1, R))
    xy = util.g1_to_arr(P)
    for w in (0, 1, 17, 31):
        out = np.zeros((128, 12), np.uint64)
        sim.sim_msm_table(_p(xy), ctypes.c_int(w), _p(out))
        Q = P
        for _ in range(8 * w):
            Q = pyref.g1_double(Q)
        acc = Q
        for d in range(1, 129):
            assert np.array_equal(out[d - 1], util.g1_to_arr(acc)), (w, d)
            acc = pyref.g1_add(acc, Q)


def test_sim_quotient_rows_match_the_spec(sim):
    """The quotient row and y of compute_kzg_proof_impl, bit-exact, for random z and for z = roots_brp[m] with m in
    {0, 1, 2047, 4095} (q_m by compute_quotient_eval_within_domain, y = p_m); a constant blob has q = 0."""
    rng = random.Random(0x9071)
    polys = [[rng.randrange(R) for _ in range(N)] for _ in range(2)]
    blobs, zs, polys_of = [], [], []
    for k, p in enumerate(polys):
        for z in (rng.randrange(R),) + tuple(ROOTS_BRP[m] for m in ((0, 2047) if k == 0 else (1, 4095))):
            blobs.append(_blob(p)); zs.append(z); polys_of.append(p)
    c = rng.randrange(R)
    blobs.append(_blob([c] * N)); zs.append(rng.randrange(R)); polys_of.append([c] * N)
    got = _quotient(sim, np.stack(blobs), zs)
    for (rows, y, st), p, z in zip(got, polys_of, zs):
        q, want_y = compute_kzg_proof_impl_quotient(p, z)
        assert st == 0 and y == want_y
        assert rows == q
    assert got[1][1] == polys[0][0] and got[2][1] == polys[0][2047] and got[-1][0] == [0] * N


def test_sim_quotient_rejections(sim):
    """z >= r, and an element >= r at positions 0 and 4095, give ZKP_KZG_BAD_SCALAR with y = 0."""
    rng = random.Random(0xBAD2)
    p = [rng.randrange(R) for _ in range(N)]
    blobs, zs = [_blob(p), _blob(p)], [R, (1 << 256) - 1]
    for pos in (0, N - 1):
        q = list(p)
        q[pos] = R
        blobs.append(_blob(q)); zs.append(rng.randrange(R))
    got = _quotient(sim, np.stack(blobs), zs)
    assert [(y, st) for _, y, st in got] == [(0, 3)] * 4


def test_sim_blob_proof_front(sim, coracle):
    """compute_blob_kzg_proof's front: z is the verifier's challenge, and C off the curve or with a limb >= p is
    ZKP_KZG_BAD_POINT; the identity C is valid."""
    from zkvm_pairings_b200 import workloads
    rng = random.Random(0xF407)
    pts, _ = coracle.g1_mul_batch(_fr([rng.randrange(1, R) for _ in range(2)]))
    blob = _blob([rng.randrange(R) for _ in range(N)])
    off = pts[1].copy(); off[6] ^= 1
    nonc = pts[1].copy(); nonc[:6] = [(util.o.P >> (64 * k)) & M64 for k in range(6)]
    ident = np.array([0] * 6 + [1] + [0] * 5, np.uint64)
    cs = np.stack([pts[0], off, nonc, ident])
    cinf = np.array([0, 0, 0, 1], np.uint8)
    blobs = np.stack([blob] * 4)
    zy, st = np.zeros((4, 8), np.uint64), np.zeros(4, np.uint8)
    sim.sim_kzg_prove_challenge(_p(blobs), _p(cs), _p(cinf), ctypes.c_size_t(4), _p(zy), _p(st))
    assert list(st) == [0, 2, 2, 0]
    for i in (0, 3):
        assert _int(zy[i, :4]) == workloads.blob_challenge(blob.tobytes(), workloads.g1_compressed(cs[i], bool(cinf[i])))


def test_no_gpu_argument_checks():
    """The prover calls check their arguments on the host and never compute on the CPU."""
    from zkvm_pairings_b200 import _lib, build
    build.build()
    lib = _lib.load()
    buf = np.zeros(BLOB_BYTES, np.uint8)
    pt, z = np.zeros(12, np.uint64), np.zeros(4, np.uint64)
    st = np.zeros(1, np.uint8)
    tg = np.zeros(24, np.uint64)
    h = ctypes.c_void_p()
    assert lib.zkp_kzg_setup_create_prover(None, _p(tg), _p(buf), ctypes.byref(h)) == -1 and not h.value
    assert lib.zkp_kzg_setup_create_prover(None, _p(tg), None, ctypes.byref(h)) == -1
    assert lib.zkp_kzg_setup_create_prover(None, _p(tg), _p(buf), None) == -1
    assert lib.zkp_kzg_blob_to_commitment_batch(None, None, _p(buf), 1, _p(pt), _p(st), _p(st)) == -1
    assert lib.zkp_kzg_compute_proof_batch(None, None, _p(buf), _p(z), 1, _p(pt), _p(st), _p(z), _p(st)) == -1
    assert lib.zkp_kzg_compute_blob_proof_batch(None, None, _p(buf), _p(pt), None, 1, _p(pt), _p(st), _p(st), None) == -1
    assert lib.zkp_kzg_blob_to_commitment_dev(None, 0, None, None, 0, None, None, None, None) == -1
    assert lib.zkp_kzg_compute_proof_dev(None, 0, None, None, None, 0, None, None, None, None, None, None) == -1
    assert lib.zkp_kzg_compute_blob_proof_dev(None, 0, None, None, None, None, 0, None, None, None, None, None, None) == -1
    assert lib.zkp_kzg_prover_scratch_bytes(1 << 10) == (1 << 10) * BLOB_BYTES + (1 << 10) * 64
    assert lib.zkp_kzg_prover_scratch_bytes(3) == 3 * BLOB_BYTES + 256


# ---------------------------------------------------------------- GPU

def _limbs6(v):
    return np.array([(v >> (64 * k)) & M64 for k in range(6)], np.uint64)


def _g1gen():
    return util.g1_to_arr(util.o.G1_GENERATOR)


@pytest.fixture(scope="module")
def prover(engine):
    """A seeded trusted setup, its prover setup and the Lagrange coefficients at tau in bit-reversed order."""
    from zkvm_pairings_b200 import workloads
    tau, tg, lag = workloads.kzg_lagrange_setup(engine, seed=0x9E0F)
    s = engine.kzg_setup(tg, lag)
    yield dict(tau=tau, tau_g2=tg, lag=lag, s=s, lag_brp=workloads.lagrange_at(tau, workloads.blob_domain()))
    s.close()


def _p_tau(pr, poly):
    return sum(v * l for v, l in zip(poly, pr["lag_brp"])) % R


def _times_g1(engine, vals):
    return engine.g1_mul_batch(np.tile(_g1gen(), (len(vals), 1)), _fr(vals))


@pytest.mark.gpu
def test_commitments_equal_p_tau(engine, prover):
    """C = [p(tau)]G1 (g1_mul_batch of p(tau) computed in Python) for the zero blob (the identity, (0, 1) with the
    flag), all r - 1, one non-zero element at index 0 and at 4095, and random blobs; an element >= r gives
    ZKP_KZG_BAD_SCALAR with a zeroed, flagged slot."""
    rng = random.Random(0xC0A1)
    polys = [[0] * N, [R - 1] * N, [rng.randrange(1, R)] + [0] * (N - 1), [0] * (N - 1) + [rng.randrange(1, R)]]
    polys += [[rng.randrange(R) for _ in range(N)] for _ in range(4)]
    blobs = [_blob(p) for p in polys]
    bad = blobs[5].copy(); bad[32 * 100:32 * 101] = 0xFF
    blobs.append(bad)
    c, ci, st = engine.kzg_blob_to_commitment_batch(prover["s"], np.stack(blobs))
    assert list(st) == [0] * len(polys) + [3]
    want, winf = _times_g1(engine, [_p_tau(prover, p) for p in polys])
    assert np.array_equal(c[:len(polys)], want) and np.array_equal(ci[:len(polys)], winf)
    assert ci[0] == 1 and np.array_equal(c[0], np.array([0] * 6 + [1] + [0] * 5, np.uint64))
    assert ci[-1] == 1 and not c[-1].any()


@pytest.mark.gpu
def test_blob_proofs_verify(engine, prover):
    """Every pi of compute_blob_kzg_proof verifies as VALID through zkp_kzg_verify_blob_batch, with the same z | y; for a
    sample pi = [q(tau)]G1 with q(tau) = (p(tau) - y) / (tau - z).  The identity commitment of the zero blob proves too."""
    rng = random.Random(0xB10F)
    coef = [rng.randrange(R) for _ in range(8)]
    polys = [[rng.randrange(R) for _ in range(N)] for _ in range(5)] + [[sum(k * pow(w, e, R) for e, k in enumerate(coef)) % R for w in ROOTS_BRP]]
    polys.append([0] * N)
    blobs = np.stack([_blob(p) for p in polys])
    s = prover["s"]
    c, ci, st = engine.kzg_blob_to_commitment_batch(s, blobs)
    assert not st.any()
    pi, pinf, st, zy = engine.kzg_compute_blob_proof_batch(s, blobs, c, ci, return_zy=True)
    assert not st.any()
    vst, vzy = engine.kzg_verify_blob_batch(s, blobs, np.concatenate([c, pi], axis=1), np.stack([ci, pinf], axis=1), return_zy=True)
    assert list(vst) == [0] * len(polys)
    assert np.array_equal(zy, vzy)
    tau = prover["tau"]
    qs = []
    for k in (0, 5):
        z, y = _int(zy[k, :4]), _int(zy[k, 4:])
        qs.append((_p_tau(prover, polys[k]) - y) * pow((tau - z) % R, -1, R) % R)
    want, _ = _times_g1(engine, qs)
    assert np.array_equal(pi[[0, 5]], want)
    assert pinf[-1] == 1


@pytest.mark.gpu
def test_compute_proof_random_and_in_domain(engine, prover):
    """(pi, y) of compute_kzg_proof verifies through zkp_kzg_verify_batch for random z and for z = roots_brp[m],
    m in {0, 1, 2047, 4095}, where y = p_m; z >= r and an element >= r give ZKP_KZG_BAD_SCALAR with y = 0 and a zeroed,
    flagged slot."""
    rng = random.Random(0x2C0F)
    polys = [[rng.randrange(R) for _ in range(N)] for _ in range(2)]
    ms = (0, 1, 2047, 4095)
    blobs, zs, exp_y = [], [], []
    for k, p in enumerate(polys):
        for z in (rng.randrange(R), rng.randrange(R)):
            blobs.append(_blob(p)); zs.append(z); exp_y.append(None)
        for m in ms[2 * k:2 * k + 2]:
            blobs.append(_blob(p)); zs.append(ROOTS_BRP[m]); exp_y.append(p[m])
    nv = len(blobs)
    bad = _blob(polys[0]); bad[32 * 4095:] = 0xFF
    blobs += [_blob(polys[0]), bad]
    zs += [R, rng.randrange(R)]
    s = prover["s"]
    blobs = np.stack(blobs)
    c, ci, _ = engine.kzg_blob_to_commitment_batch(s, blobs)
    pi, pinf, y, st = engine.kzg_compute_proof_batch(s, blobs, _fr(zs))
    assert list(st) == [0] * nv + [3, 3]
    assert not y[nv:].any() and not pi[nv:].any() and list(pinf[nv:]) == [1, 1]
    for k in range(nv):
        if exp_y[k] is not None:
            assert _int(y[k]) == exp_y[k]
    vzy = np.concatenate([_fr(zs[:nv]), y[:nv]], axis=1)
    vst = engine.kzg_verify_batch(s, np.concatenate([c[:nv], pi[:nv]], axis=1), vzy, np.stack([ci[:nv], pinf[:nv]], axis=1))
    assert list(vst) == [0] * nv
    # a wrong y fails the equation: the proofs are bound to their openings
    vzy[0, 4] ^= 1
    assert engine.kzg_verify_batch(s, np.concatenate([c[:1], pi[:1]], axis=1), vzy[:1])[0] == 1


@pytest.mark.gpu
def test_blob_proof_bad_commitments(engine, prover, pyref):
    """A commitment with a limb >= p, off the curve, of order 3, or a valid C plus a point of order 3 gives
    ZKP_KZG_BAD_POINT with a zeroed, flagged slot, also together with an element >= r (BAD_POINT precedes)."""
    rng = random.Random(0xBAD3)
    s = prover["s"]
    blob = _blob([rng.randrange(R) for _ in range(N)])
    c, ci, _ = engine.kzg_blob_to_commitment_batch(s, blob[None])
    C = (_int(c[0, :6]), _int(c[0, 6:]), False)
    nonc = c[0].copy(); nonc[:6] = _limbs6(_int(c[0, :6]) + pyref.P)
    off = c[0].copy(); off[6] ^= 1
    t3 = util.g1_to_arr((0, 2))
    ct3 = util.g1_to_arr(pyref.g1_add(C, (0, 2, False)))
    bad_blob = blob.copy(); bad_blob[:32] = 0xFF
    cs = np.stack([c[0], nonc, off, t3, ct3, off])
    blobs = np.stack([blob] * 5 + [bad_blob])
    pi, pinf, st = engine.kzg_compute_blob_proof_batch(s, blobs, cs)
    assert list(st) == [0, 2, 2, 2, 2, 2]
    assert not pi[1:].any() and list(pinf[1:]) == [1] * 5


@pytest.mark.gpu
def test_prover_setup_rejections(engine, prover):
    """Setup creation rejects a limb >= p (NonCanonicalError), an off-curve point (naming its index), and, as
    inconsistent with tau_g2, two swapped points, a wrong tau and the points in bit-reversed order.  A setup without
    Lagrange points cannot prove, and a setup is refused by another context."""
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    lag, tg = prover["lag"], prover["tau_g2"]
    bad = lag.copy(); bad[5, :6] = _limbs6(util.o.P)
    with pytest.raises(z.NonCanonicalError):
        engine.kzg_setup(tg, bad)
    bad = lag.copy(); bad[17, 6] ^= 1
    with pytest.raises(z.ZkpError) as ei:
        engine.kzg_setup(tg, bad)
    assert ei.value.code == -1 and "g1_lagrange[17]" in str(ei.value) and "not on the curve" in str(ei.value)
    swapped = lag.copy(); swapped[[3, 4]] = lag[[4, 3]]
    _, other_tg, _ = workloads.kzg_lagrange_setup(engine, seed=0x9E10)
    brp = lag[[int(format(i, "012b")[::-1], 2) for i in range(N)]]
    for t, l in ((tg, swapped), (other_tg, lag), (tg, brp)):
        with pytest.raises(z.ZkpError) as ei:
            engine.kzg_setup(t, l)
        assert ei.value.code == -1 and "inconsistent with tau_g2" in str(ei.value)
    blob = np.zeros((1, BLOB_BYTES), np.uint8)
    with engine.kzg_setup(tg) as plain:
        with pytest.raises(z.ZkpError) as ei:
            engine.kzg_blob_to_commitment_batch(plain, blob)
        assert ei.value.code == -1 and "no Lagrange points" in str(ei.value)
        with pytest.raises(z.ZkpError):
            engine.kzg_compute_proof_batch(plain, blob, _fr([1]))
        with pytest.raises(z.ZkpError):
            engine.kzg_compute_blob_proof_batch(plain, blob, np.zeros((1, 12), np.uint64), np.ones(1, np.uint8))
    other = z.PairingEngine([0])
    try:
        with pytest.raises(z.ZkpError) as ei:
            other.kzg_blob_to_commitment_batch(prover["s"], blob)
        assert ei.value.code == -1 and "another context" in str(ei.value)
    finally:
        other.close()


@pytest.mark.gpu
def test_chunk_paths_agree(engine, prover):
    """One chunk bound (2^14 blobs) + 3: pageable, pinned and _dev calls agree for commitments, proofs at z and blob
    proofs, and n = 0 works; a sample of the blob proofs verifies."""
    import torch
    rng = random.Random(0xC4C4)
    n = (1 << 14) + 3
    s = prover["s"]
    blobs = _random_blobs(0xC4C4, n)
    zs = _fr([rng.randrange(R) for _ in range(n)])
    c, ci, cst = engine.kzg_blob_to_commitment_batch(s, blobs)
    pz, pzi, y, zst = engine.kzg_compute_proof_batch(s, blobs, zs)
    pb, pbi, bst, zy = engine.kzg_compute_blob_proof_batch(s, blobs, c, ci, return_zy=True)
    assert not cst.any() and not zst.any() and not bst.any()
    tb = torch.from_numpy(blobs).pin_memory()
    hb = tb.numpy()
    for got, want in zip(engine.kzg_blob_to_commitment_batch(s, hb), (c, ci, cst)):
        assert np.array_equal(got, want)
    for got, want in zip(engine.kzg_compute_proof_batch(s, hb, zs), (pz, pzi, y, zst)):
        assert np.array_equal(got, want)
    for got, want in zip(engine.kzg_compute_blob_proof_batch(s, hb, c, ci, return_zy=True), (pb, pbi, bst, zy)):
        assert np.array_equal(got, want)
    for got in engine.kzg_blob_to_commitment_batch(s, blobs[:0]) + engine.kzg_compute_blob_proof_batch(s, blobs[:0], c[:0]):
        assert got.shape[0] == 0
    before = torch.cuda.current_device()
    db = tb.cuda()
    dc = torch.zeros((n, 12), dtype=torch.int64, device="cuda")
    dci = torch.zeros(n, dtype=torch.uint8, device="cuda")
    dst = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    engine.kzg_blob_to_commitment_dev(s, db, n, dc, dci, dst)
    assert np.array_equal(dc.cpu().numpy().view(np.uint64), c) and np.array_equal(dci.cpu().numpy(), ci) and not dst.cpu().numpy().any()
    scratch = torch.empty(engine.kzg_prover_scratch_bytes(n), dtype=torch.uint8, device="cuda")
    dz = torch.from_numpy(zs.view(np.int64)).cuda()
    dp = torch.zeros((n, 12), dtype=torch.int64, device="cuda")
    dpi = torch.zeros(n, dtype=torch.uint8, device="cuda")
    dy = torch.zeros((n, 4), dtype=torch.int64, device="cuda")
    dst.fill_(9)
    engine.kzg_compute_proof_dev(s, db, dz, n, dp, dpi, dy, dst, scratch)
    assert np.array_equal(dp.cpu().numpy().view(np.uint64), pz) and np.array_equal(dpi.cpu().numpy(), pzi)
    assert np.array_equal(dy.cpu().numpy().view(np.uint64), y) and not dst.cpu().numpy().any()
    dzy = torch.zeros((n, 8), dtype=torch.int64, device="cuda")
    dst.fill_(9)
    engine.kzg_compute_blob_proof_dev(s, db, dc, n, dp, dpi, dst, scratch, d_commitment_inf=dci, d_out_zy=dzy)
    engine.kzg_compute_blob_proof_dev(s, db, dc, 0, dp, dpi, dst, scratch)
    assert np.array_equal(dp.cpu().numpy().view(np.uint64), pb) and np.array_equal(dpi.cpu().numpy(), pbi)
    assert np.array_equal(dzy.cpu().numpy().view(np.uint64), zy) and not dst.cpu().numpy().any()
    assert torch.cuda.current_device() == before
    k = np.array([0, 1, (1 << 14) - 1, 1 << 14, n - 1])
    vst = engine.kzg_verify_blob_batch(s, blobs[k], np.concatenate([c[k], pb[k]], axis=1), np.stack([ci[k], pbi[k]], axis=1))
    assert list(vst) == [0] * len(k)


@pytest.mark.gpu
def test_prover_multi_device_matches_single(engine, prover):
    import zkvm_pairings_b200 as z
    if z.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    blobs = _random_blobs(0xC6C6, 301)
    multi = z.PairingEngine()
    try:
        with multi.kzg_setup(prover["tau_g2"], prover["lag"]) as sm:
            a = engine.kzg_blob_to_commitment_batch(prover["s"], blobs)
            b = multi.kzg_blob_to_commitment_batch(sm, blobs)
            assert all(np.array_equal(x, y) for x, y in zip(a, b))
            pa = engine.kzg_compute_blob_proof_batch(prover["s"], blobs, a[0], a[1], return_zy=True)
            pm = multi.kzg_compute_blob_proof_batch(sm, blobs, a[0], a[1], return_zy=True)
            assert all(np.array_equal(x, y) for x, y in zip(pa, pm))
    finally:
        multi.close()
