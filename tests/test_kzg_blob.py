"""EIP-4844 blob verification (zkp_kzg_verify_blob_*): the Fr arithmetic, the domain table, the transcript and the
barycentric evaluation bit-exact against a line-by-line restatement of the consensus specs (below) through the CPU dev
simulation of csrc/fr.cuh and csrc/blob.cuh, and the GPU entry points against the trapdoor construction of
workloads.kzg_blob_proofs, an honest prover over a Lagrange-basis SRS and the existing point-evaluation call."""
import ctypes
import hashlib
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
N = 4096
BLOB_BYTES = 32 * N
RF = (1 << 256) % R
IDENTITY_XY = [0] * 6 + [1] + [0] * 5


# ---------------------------------------------------------------- the consensus specs (deneb polynomial-commitments.md)

BLS_MODULUS = R
FIELD_ELEMENTS_PER_BLOB = N
PRIMITIVE_ROOT_OF_UNITY = 7
FIAT_SHAMIR_PROTOCOL_DOMAIN = b"FSBLOBVERIFY_V1_"


def reverse_bits(n, order):
    return int(("{:0" + str(order.bit_length() - 1) + "b}").format(n)[::-1], 2)


def bit_reversal_permutation(sequence):
    return [sequence[reverse_bits(i, len(sequence))] for i in range(len(sequence))]


def compute_roots_of_unity(order):
    assert (BLS_MODULUS - 1) % order == 0
    root_of_unity = pow(PRIMITIVE_ROOT_OF_UNITY, (BLS_MODULUS - 1) // order, BLS_MODULUS)
    roots, current = [], 1
    for _ in range(order):
        roots.append(current)
        current = current * root_of_unity % BLS_MODULUS
    return roots


ROOTS_BRP = bit_reversal_permutation(compute_roots_of_unity(FIELD_ELEMENTS_PER_BLOB))


def g1_to_bytes48(x, y, inf):
    """The standard compressed encoding of a G1 point (ZCash serialisation): x big-endian with the compression flag,
    the sign of y (y > (p - 1) / 2) and the infinity flag in the top three bits."""
    if inf:
        return bytes([0xC0]) + bytes(47)
    out = bytearray(x.to_bytes(48, "big"))
    out[0] |= 0x80
    if y > (util.o.P - 1) // 2:
        out[0] |= 0x20
    return bytes(out)


def hash_to_bls_field(data):
    return int.from_bytes(hashlib.sha256(data).digest(), "big") % BLS_MODULUS


def compute_challenge(blob, commitment):
    degree_poly = int.to_bytes(FIELD_ELEMENTS_PER_BLOB, 16, "big")
    return hash_to_bls_field(FIAT_SHAMIR_PROTOCOL_DOMAIN + degree_poly + blob + commitment)


def blob_to_polynomial(blob):
    poly = [int.from_bytes(blob[32 * i:32 * i + 32], "big") for i in range(FIELD_ELEMENTS_PER_BLOB)]
    assert all(v < BLS_MODULUS for v in poly)
    return poly


def evaluate_polynomial_in_evaluation_form(polynomial, z):
    width = len(polynomial)
    inverse_width = pow(width, -1, BLS_MODULUS)
    if z in ROOTS_BRP:
        return polynomial[ROOTS_BRP.index(z)]
    result = 0
    for i in range(width):
        a = polynomial[i] * ROOTS_BRP[i] % BLS_MODULUS
        b = (z - ROOTS_BRP[i]) % BLS_MODULUS
        result += a * pow(b, -1, BLS_MODULUS)
    r = (pow(z, width, BLS_MODULUS) - 1) * inverse_width % BLS_MODULUS
    return result % BLS_MODULUS * r % BLS_MODULUS


# ---------------------------------------------------------------- helpers

def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _fr(vals):
    return np.array([[(v >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)] for v in vals], dtype=np.uint64).reshape(-1, 4)


def _int(limbs):
    return sum(int(t) << (64 * k) for k, t in enumerate(limbs))


def _blob(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "big") for v in vals), dtype=np.uint8).copy()


def _pt_ints(a):
    return _int(a[:6]), _int(a[6:12])


@pytest.fixture(scope="module")
def sim():
    """The dev simulation with the blob front end (its own build: the staleness list covers every device header)."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_kzg_blob.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, "sim_kzg_blob.cpp"), os.path.join(d, "sim.cpp"), os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    return ctypes.CDLL(so)


def _challenge(sim, blobs, proofs, pinf=None):
    blobs = np.ascontiguousarray(blobs, np.uint8).reshape(-1, BLOB_BYTES)
    n = blobs.shape[0]
    proofs = np.ascontiguousarray(proofs, np.uint64).reshape(n, 24)
    dg, zy = np.zeros((n, 8), np.uint32), np.zeros((n, 8), np.uint64)
    pi = None if pinf is None else np.ascontiguousarray(pinf, np.uint8).reshape(n, 2)
    sim.sim_blob_challenge(_p(blobs), _p(proofs), _p(pi), ctypes.c_size_t(n), _p(dg), _p(zy))
    return dg, zy


def _domain(sim):
    d = np.zeros((N, 4), np.uint64)
    sim.sim_blob_domain(_p(d))
    return d


def _eval(sim, blobs, zs):
    """k_blob_eval's body: y for each blob at z (canonical), or (z, y) = (r, 0) for a blob with an element >= r."""
    blobs = np.ascontiguousarray(blobs, np.uint8).reshape(-1, BLOB_BYTES)
    n = blobs.shape[0]
    zy = np.zeros((n, 8), np.uint64)
    zy[:, :4] = _fr(zs)
    sim.sim_blob_eval(_p(blobs), _p(_domain(sim)), _p(zy), ctypes.c_size_t(n))
    return [(_int(r[:4]), _int(r[4:])) for r in zy]


def _proof_for(c_xy):
    pr = np.zeros(24, np.uint64)
    pr[:12] = c_xy
    return pr


# ---------------------------------------------------------------- CPU: dev simulation of the device bodies

def test_generated_fr_constants():
    text = open(os.path.join(ROOT, "zkvm_pairings_b200", "csrc", "consts.cuh")).read()

    def arr8(name):
        m = re.search(r"%s\[8\] = \{(.*?)\};" % name, text, re.S)
        w = [int(x, 16) for x in re.findall(r"0x([0-9a-f]{8})u", m.group(1))]
        return sum(v << (32 * j) for j, v in enumerate(w))
    n0 = int(re.search(r"#define ZKP_FR_N0INV 0x([0-9a-f]+)u", text).group(1), 16)
    assert (n0 * R + 1) % (1 << 32) == 0
    assert arr8("ZKP_FR_ONE") == RF and arr8("ZKP_FR_R2") == RF * RF % R and arr8("ZKP_FR_R3") == RF ** 3 % R
    assert arr8("ZKP_FR_INV_N") == pow(N, -1, R) * RF % R
    w = compute_roots_of_unity(N)[1]
    assert arr8("ZKP_FR_OMEGA") == w * RF % R
    assert pow(w, N, R) == 1 and pow(w, N // 2, R) == R - 1


def test_sim_domain_table(sim):
    """The setup's 4096 entries (Montgomery) against roots_brp; roots_brp[0] = 1, roots_brp[1] = r - 1."""
    d = _domain(sim)
    rinv = pow(RF, -1, R)
    got = [_int(row) * rinv % R for row in d]
    assert got == ROOTS_BRP
    assert got[0] == 1 and got[1] == R - 1
    assert len(set(got)) == N


def test_sim_fr_ops_at_the_corners(sim):
    """add / sub / mul / inv at {0, 1, 2, r - 2, r - 1} crossed with random values, against Python ints; every product
    passes the simulation's operand-bound assertion."""
    rng = random.Random(0xF12)
    corners = [0, 1, 2, R - 2, R - 1]
    vals = corners + [rng.randrange(R) for _ in range(6)]
    a = [x for x in vals for _ in vals]
    b = [y for _ in vals for y in vals]
    A, B = _fr(a), _fr(b)
    for op, fn in ((0, lambda x, y: (x + y) % R), (1, lambda x, y: (x - y) % R), (2, lambda x, y: x * y % R),
                   (3, lambda x, y: pow(x, -1, R) if x else 0)):
        out = np.zeros_like(A)
        sim.sim_fr_op(op, _p(A), _p(B), _p(out), ctypes.c_size_t(len(a)))
        assert [_int(r) for r in out] == [fn(x, y) for x, y in zip(a, b)], op


def test_sim_fr_operand_bound_is_asserted(sim):
    """A representative >= r handed to fr_add, fr_sub or fr_mul aborts the simulation (ZKP_SIM_ASSERT)."""
    big = tuple((R >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4))
    for op, what in ((0, "fr_add"), (1, "fr_sub"), (2, "fr_mul")):
        code = ("import ctypes, numpy as np; l = ctypes.CDLL(%r); a = np.array([1, 0, 0, 0], np.uint64); "
                "b = np.array([%d, %d, %d, %d], np.uint64); o = np.zeros(4, np.uint64); "
                "l.sim_fr_raw(%d, a.ctypes.data_as(ctypes.c_void_p), b.ctypes.data_as(ctypes.c_void_p), o.ctypes.data_as(ctypes.c_void_p))"
                % ((sim._name,) + big + (op,)))
        p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
        assert p.returncode != 0 and what + " operand bound" in p.stderr, what


def test_sim_commitment_encoding(sim, coracle, pyref):
    """The compressed encoding of C from its limbs: the G1 generator, the identity and one point of each y-sign."""
    def enc(xy, inf=0):
        out = np.zeros(12, np.uint32)
        sim.sim_g1_compress(_p(np.ascontiguousarray(xy, np.uint64)), ctypes.c_uint8(inf), _p(out))
        return b"".join(int(w).to_bytes(4, "big") for w in out)
    g = util.g1_to_arr(pyref.G1_GENERATOR)
    assert enc(g).hex() == ("97f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb")
    assert enc(np.array(IDENTITY_XY, np.uint64), 1) == bytes([0xC0]) + bytes(47)
    rng = random.Random(0xC48)
    pts, _ = coracle.g1_mul_batch(_fr([rng.randrange(1, R) for _ in range(16)]))
    signs = set()
    for pt in pts:
        x, y = _pt_ints(pt)
        e = enc(pt)
        assert e == g1_to_bytes48(x, y, False)
        signs.add(bool(e[0] & 0x20))
    assert signs == {False, True}


def test_sim_transcript_digest_and_z(sim, coracle):
    """SHA-256 of the transcript and z = digest mod r against hashlib for random blobs, the zero blob, the all-(r - 1)
    blob and blobs found by search whose digest is >= r and >= 2r (both subtractions of the reduction)."""
    rng = random.Random(0x7A5)
    pts, _ = coracle.g1_mul_batch(_fr([rng.randrange(1, R) for _ in range(2)]))
    blobs = [_blob([rng.randrange(R) for _ in range(N)]) for _ in range(2)] + [_blob([0] * N), _blob([R - 1] * N)]
    infs = [0, 0, 1, 0]
    found = {}
    base = _blob([rng.randrange(R) for _ in range(N)])
    for s in range(1000):
        b = base.copy()
        b[-8:] = np.frombuffer(s.to_bytes(8, "big"), np.uint8)
        d = int.from_bytes(hashlib.sha256(FIAT_SHAMIR_PROTOCOL_DOMAIN + N.to_bytes(16, "big") + b.tobytes() +
                                          g1_to_bytes48(*_pt_ints(pts[0]), False)).digest(), "big")
        k = 2 if d >= 2 * R else 1 if d >= R else 0
        found.setdefault(k, b)
        if len(found) == 3:
            break
    assert len(found) == 3
    blobs += [found[1], found[2]]
    infs += [0, 0]
    proofs = np.stack([_proof_for(pts[i % 2] if not infs[i] else np.array(IDENTITY_XY, np.uint64)) for i in range(len(blobs))])
    pinf = np.array([[f, 0] for f in infs], np.uint8)
    dg, zy = _challenge(sim, np.stack(blobs), proofs, pinf)
    for i, b in enumerate(blobs):
        c48 = g1_to_bytes48(*_pt_ints(proofs[i, :12]), bool(infs[i]))
        data = FIAT_SHAMIR_PROTOCOL_DOMAIN + N.to_bytes(16, "big") + b.tobytes() + c48
        assert b"".join(int(w).to_bytes(4, "big") for w in dg[i]) == hashlib.sha256(data).digest(), i
        assert _int(zy[i, :4]) == compute_challenge(b.tobytes(), c48), i
    assert int.from_bytes(b"".join(int(w).to_bytes(4, "big") for w in dg[-1]), "big") >= 2 * R


def test_sim_evaluation(sim):
    """y against the spec for random blobs at random z; z in the domain at indices 0, 1, 2, 4095 and a random one gives
    p_j; a constant blob gives y = c everywhere, and the evaluations of a degree-15 polynomial give its value at z."""
    rng = random.Random(0xE7A)
    polys = [[rng.randrange(R) for _ in range(N)] for _ in range(2)]
    blobs, zs, want = [], [], []
    for p in polys:
        for z in (rng.randrange(R), rng.randrange(R)):
            blobs.append(_blob(p)); zs.append(z); want.append(evaluate_polynomial_in_evaluation_form(p, z))
    for j in (0, 1, 2, N - 1, rng.randrange(N)):
        blobs.append(_blob(polys[0])); zs.append(ROOTS_BRP[j]); want.append(polys[0][j])
    c = rng.randrange(R)
    for z in (0, 1, rng.randrange(R), ROOTS_BRP[77]):
        blobs.append(_blob([c] * N)); zs.append(z); want.append(c)
    coef = [rng.randrange(R) for _ in range(16)]
    f = lambda x: sum(k * pow(x, e, R) for e, k in enumerate(coef)) % R
    low = [f(w) for w in ROOTS_BRP]
    for z in (rng.randrange(R), 0, rng.randrange(R)):
        blobs.append(_blob(low)); zs.append(z); want.append(f(z))
    got = _eval(sim, np.stack(blobs), zs)
    assert got == list(zip(zs, want))


def test_sim_element_range_check(sim):
    """An element r - 1 passes; r, 2^256 - 1, and an element >= r at positions 0, 2048 and 4095 give z = r, y = 0."""
    rng = random.Random(0xBAD)
    p = [rng.randrange(R) for _ in range(N)]
    blobs, zs, want = [], [], []
    ok = list(p)
    ok[5] = R - 1
    z = rng.randrange(R)
    blobs.append(_blob(ok)); zs.append(z); want.append((z, evaluate_polynomial_in_evaluation_form(ok, z)))
    for pos, v in ((5, R), (5, (1 << 256) - 1), (0, R + 1), (2048, R), (N - 1, (1 << 256) - 1)):
        q = list(p)
        q[pos] = v
        blobs.append(_blob(q)); zs.append(z); want.append((R, 0))
    q = list(p)
    q[9] = R
    blobs.append(_blob(q)); zs.append(ROOTS_BRP[9]); want.append((R, 0))   # also when z is in the domain
    assert _eval(sim, np.stack(blobs), zs) == want


def test_no_gpu_fails_loudly():
    """The blob calls check their arguments on the host and never compute on the CPU."""
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import _lib, build
    build.build()
    lib = _lib.load()
    buf = np.zeros(BLOB_BYTES, np.uint8)
    pr = np.zeros(24, np.uint64)
    st = np.zeros(1, np.uint8)
    assert lib.zkp_kzg_verify_blob_batch(None, None, _p(buf), _p(pr), None, 1, _p(st), None) == -1
    assert lib.zkp_kzg_verify_blob_dev(None, 0, None, None, None, None, 0, None, None, None, None) == -1
    assert lib.zkp_kzg_blob_scratch_bytes(1 << 10) == (1 << 10) * 64 + lib.zkp_kzg_scratch_bytes(1 << 10)
    assert z.BLOB_BYTES == BLOB_BYTES


# ---------------------------------------------------------------- GPU

def _bad_points(pyref, coracle):
    g1b, _, e1, _, _, _ = util.group_check_cases(pyref, coracle, seed=0xB10B)
    return g1b[list(e1).index(1)], g1b[list(e1).index(2)]


@pytest.mark.gpu
def test_blob_verdicts_in_one_batch(engine, coracle, pyref):
    """Valid blobs; a flipped blob byte (z changes) and proofs swapped between blobs fail the equation; an element
    >= r is 3; C or pi off the curve or not torsion free is 2, also together with a bad element; the zero blob with
    C = pi = identity is valid.  out_zy matches the spec."""
    from zkvm_pairings_b200 import workloads
    w = workloads.kzg_blob_proofs(engine, 8, seed=0xB1, distinct=8, corrupt_every=0)
    off, tor = _bad_points(pyref, coracle)
    blobs, proofs = [w["blobs"][i].copy() for i in range(8)], [w["proofs"][i].copy() for i in range(8)]
    infs, exp = [[0, 0]] * 8, [0] * 8

    def add(b, pr, e, inf=(0, 0)):
        blobs.append(b); proofs.append(pr); infs.append(list(inf)); exp.append(e)
    b = w["blobs"][0].copy(); b[32 * 9 + 31] ^= 1; add(b, w["proofs"][0], 1)
    pr = w["proofs"][1].copy(); pr[12:] = w["proofs"][2][12:]; add(w["blobs"][1], pr, 1)
    pr = w["proofs"][2].copy(); pr[12:] = w["proofs"][1][12:]; add(w["blobs"][2], pr, 1)
    bad = w["blobs"][3].copy(); bad[32 * 100:32 * 101] = 0xFF
    add(bad, w["proofs"][3], 3)
    pr = w["proofs"][4].copy(); pr[:12] = off; add(w["blobs"][4], pr, 2)
    pr = w["proofs"][4].copy(); pr[12:] = tor; add(w["blobs"][4], pr, 2)
    pr = w["proofs"][5].copy(); pr[:12] = tor; add(bad, pr, 2)
    zero = np.zeros(24, np.uint64); zero[6] = 1; zero[18] = 1
    add(np.zeros(BLOB_BYTES, np.uint8), zero, 0, (1, 1))
    with engine.kzg_setup(w["tau_g2"]) as s:
        st, zy = engine.kzg_verify_blob_batch(s, np.stack(blobs), np.stack(proofs), np.array(infs, np.uint8), return_zy=True)
        assert list(st) == exp
        assert np.array_equal(zy[:8], w["zy"])
        assert _int(zy[11, :4]) == R and _int(zy[11, 4:]) == 0
        for i in (0, 8, len(blobs) - 1):
            c = proofs[i][:12]
            c48 = g1_to_bytes48(*_pt_ints(c), bool(infs[i][0]))
            zz = compute_challenge(blobs[i].tobytes(), c48)
            assert (_int(zy[i, :4]), _int(zy[i, 4:])) == (zz, evaluate_polynomial_in_evaluation_form(blob_to_polynomial(blobs[i].tobytes()), zz))
        assert np.array_equal(engine.kzg_verify_batch(s, np.stack(proofs), zy, np.array(infs, np.uint8)), st)


def _msm(engine, bases, scalars):
    """sum_i scalars[j][i] bases[i] for each row j, through g1_mul_batch and a g1_add_batch tree."""
    m, nb = len(scalars), bases.shape[0]
    pts, inf = engine.g1_mul_batch(np.tile(bases, (m, 1)), _fr([v for row in scalars for v in row]))
    pts, inf = pts.reshape(m, nb, 12), inf.reshape(m, nb)
    while pts.shape[1] > 1:
        s, f = engine.g1_add_batch(pts[:, 0::2].reshape(-1, 12), pts[:, 1::2].reshape(-1, 12), inf[:, 0::2].reshape(-1),
                                   inf[:, 1::2].reshape(-1))
        pts, inf = s.reshape(m, -1, 12), (f & 1).reshape(m, -1)
    return pts[:, 0], inf[:, 0]


@pytest.mark.gpu
def test_blob_honest_prover(engine):
    """blob_to_kzg_commitment and compute_kzg_proof_impl over a Lagrange-basis SRS [l_i(tau)]G1 in bit-reversed order
    (multi-scalar products through g1_mul_batch / g1_add_batch, no trapdoor shortcut in the combination): four blobs,
    one of low degree, all verify; a flipped byte in each, and each blob with the next one's proof, fail."""
    rng = random.Random(0x5125)
    tau = rng.randrange(1, R)
    scale = (pow(tau, N, R) - 1) * pow(N, -1, R) % R
    lag = [scale * w * pow(tau - w, -1, R) % R for w in ROOTS_BRP]
    g1gen = util.g1_to_arr(util.o.G1_GENERATOR)
    srs, srs_inf = engine.g1_mul_batch(np.tile(g1gen, (N, 1)), _fr(lag))
    assert not srs_inf.any()
    tg, _ = engine.g2_mul_batch(util.g2_to_arr(util.o.G2_GENERATOR)[None], _fr([tau]))
    coef = [rng.randrange(R) for _ in range(8)]
    polys = [[rng.randrange(R) for _ in range(N)] for _ in range(3)] + [[sum(k * pow(w, e, R) for e, k in enumerate(coef)) % R for w in ROOTS_BRP]]
    C, cinf = _msm(engine, srs, polys)
    quots = []
    for k, p in enumerate(polys):
        z = compute_challenge(_blob(p).tobytes(), g1_to_bytes48(*_pt_ints(C[k]), bool(cinf[k])))
        y = evaluate_polynomial_in_evaluation_form(p, z)
        quots.append([(pk - y) * pow((w - z) % R, -1, R) % R for pk, w in zip(p, ROOTS_BRP)])
    PI, pinf = _msm(engine, srs, quots)
    blobs = [_blob(p) for p in polys]
    proofs = [np.concatenate([C[k], PI[k]]) for k in range(4)]
    flags = [[cinf[k], pinf[k]] for k in range(4)]
    for k in range(4):
        b = blobs[k].copy(); b[32 * 17 + 31] ^= 2
        blobs.append(b); proofs.append(proofs[k]); flags.append(flags[k])
    for k in range(4):
        blobs.append(blobs[k]); proofs.append(np.concatenate([C[k], PI[(k + 1) % 4]])); flags.append([cinf[k], pinf[(k + 1) % 4]])
    with engine.kzg_setup(tg[0]) as s:
        st = engine.kzg_verify_blob_batch(s, np.stack(blobs), np.stack(proofs), np.array(flags, np.uint8))
    assert list(st) == [0] * 4 + [1] * 8


@pytest.mark.gpu
def test_blob_chunks_and_every_path(engine):
    """Two chunks plus a tail: the verdicts equal the construction, (proofs, out_zy) through kzg_verify_batch gives
    the same verdict in every slot, and pageable, pinned, _dev (with and without out_zy) and n = 0 agree."""
    import torch
    from zkvm_pairings_b200 import workloads
    n = 2 * (1 << 14) + 37                          # ZKP_BLOB_CHUNK = 2^14 blobs per host chunk
    w = workloads.kzg_blob_proofs(engine, n, seed=0xC4, distinct=48)
    w["blobs"][n - 5, 32 * 7:32 * 8] = 0xFF          # an element >= r in the tail
    expect = w["expect"].copy()
    expect[n - 5] = 3
    with engine.kzg_setup(w["tau_g2"]) as s:
        st, zy = engine.kzg_verify_blob_batch(s, w["blobs"], w["proofs"], return_zy=True)
        assert np.array_equal(st, expect) and expect.sum() > 80
        keep = np.ones(n, bool)
        keep[n - 5] = False
        assert np.array_equal(zy[keep], w["zy"][keep])
        assert np.array_equal(engine.kzg_verify_batch(s, w["proofs"], zy), st)

        pb = torch.from_numpy(w["blobs"]).pin_memory()
        pp = torch.from_numpy(w["proofs"].view(np.int64)).pin_memory()
        assert np.array_equal(engine.kzg_verify_blob_batch(s, pb.numpy(), pp.numpy().view(np.uint64)), st)
        assert engine.kzg_verify_blob_batch(s, w["blobs"][:0], w["proofs"][:0]).shape == (0,)
        before = torch.cuda.current_device()
        db, dp = pb.cuda(), pp.cuda()
        ds = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
        dzy = torch.zeros((n, 8), dtype=torch.int64, device="cuda")
        scratch = torch.empty(engine.kzg_blob_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        engine.kzg_verify_blob_dev(s, db, dp, n, ds, scratch, d_out_zy=dzy)
        assert np.array_equal(ds.cpu().numpy(), st)
        assert np.array_equal(dzy.cpu().numpy().view(np.uint64), zy)
        ds.fill_(9)
        engine.kzg_verify_blob_dev(s, db, dp, n, ds, scratch)
        engine.kzg_verify_blob_dev(s, db, dp, 0, ds, scratch)
        assert np.array_equal(ds.cpu().numpy(), st)
        assert torch.cuda.current_device() == before


@pytest.mark.gpu
def test_blob_context_check(engine):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    w = workloads.kzg_blob_proofs(engine, 4, seed=0xC5, corrupt_every=0)
    other = z.PairingEngine([0])
    try:
        with engine.kzg_setup(w["tau_g2"]) as s:
            with pytest.raises(z.ZkpError) as ei:
                other.kzg_verify_blob_batch(s, w["blobs"], w["proofs"])
            assert ei.value.code == -1 and "another context" in str(ei.value)
            assert list(engine.kzg_verify_blob_batch(s, w["blobs"], w["proofs"])) == [0] * 4
    finally:
        other.close()


@pytest.mark.gpu
def test_blob_multi_device_matches_single(engine):
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    if z.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    w = workloads.kzg_blob_proofs(engine, 301, seed=0xC6, distinct=16)
    multi = z.PairingEngine()
    try:
        with engine.kzg_setup(w["tau_g2"]) as s1, multi.kzg_setup(w["tau_g2"]) as sm:
            a = engine.kzg_verify_blob_batch(s1, w["blobs"], w["proofs"], return_zy=True)
            b = multi.kzg_verify_blob_batch(sm, w["blobs"], w["proofs"], return_zy=True)
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[0], w["expect"])
    finally:
        multi.close()
