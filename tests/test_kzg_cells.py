"""EIP-7594 cells and cell proofs (zkp_kzg_setup_create_cells, zkp_kzg_compute_cells_*, zkp_kzg_compute_cells_and_proofs_*,
zkp_kzg_verify_cell_*): the extension, the quotient rows and the interpolation bit-exact against a restatement of the
consensus specs (fulu polynomial-commitments-sampling.md) through the CPU dev simulation of csrc/kzg_cells.cuh, and the
GPU entry points against oracles independent of the MSM: [q_k(tau)]G1 through g1_mul_batch at the trapdoor tau, and
the verdicts of changed cells, indices, proofs and commitments."""
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
EXT = 2 * N
CELLS = 128
PER_CELL = 64
CELL_BYTES = 32 * PER_CELL
BLOB_BYTES = 32 * N
M64 = (1 << 64) - 1


# ---------------------------------------------------------------- the consensus specs (fulu polynomial-commitments-sampling.md)

def _brp(i, bits):
    return int(format(i, "0%db" % bits)[::-1], 2)


def compute_roots_of_unity(order):
    w = pow(7, (R - 1) // order, R)
    out = [1] * order
    for i in range(1, order):
        out[i] = out[i - 1] * w % R
    return out


ROOTS_EXT = compute_roots_of_unity(EXT)
ROOTS_EXT_BRP = [ROOTS_EXT[_brp(i, 13)] for i in range(EXT)]
ROOTS_BRP = [ROOTS_EXT[2 * _brp(i, 12)] for i in range(N)]   # roots_brp of the 4096 domain


def coset_for_cell(cell_index):
    return ROOTS_EXT_BRP[PER_CELL * cell_index:PER_CELL * (cell_index + 1)]


def _ntt(a, w):
    """sum_t a_t w^(t k) for k < len(a), natural order in and out (recursive radix 2)."""
    n = len(a)
    if n == 1:
        return list(a)
    ev, od = _ntt(a[0::2], w * w % R), _ntt(a[1::2], w * w % R)
    out, t = [0] * n, 1
    for k in range(n // 2):
        v = od[k] * t % R
        out[k], out[k + n // 2] = (ev[k] + v) % R, (ev[k] - v) % R
        t = t * w % R
    return out


def polynomial_eval_to_coeff(values_brp):
    """The coefficients of the blob's polynomial from its values at roots_brp (an inverse NTT)."""
    nat = [0] * N
    for i, v in enumerate(values_brp):
        nat[_brp(i, 12)] = v
    inv_n, w_inv = pow(N, -1, R), pow(ROOTS_EXT[2], -1, R)
    return [v * inv_n % R for v in _ntt(nat, w_inv)]


def compute_cells(values_brp):
    """compute_cells by the NTT route: the coefficients, evaluated over the 8192 roots (one NTT) in bit-reversed order."""
    coeff = polynomial_eval_to_coeff(values_brp)
    ext = _ntt(coeff + [0] * N, ROOTS_EXT[1])
    ys = [ext[_brp(i, 13)] for i in range(EXT)]
    return [ys[PER_CELL * k:PER_CELL * (k + 1)] for k in range(CELLS)], coeff


def evaluate_polynomialcoeff(coeff, z):
    y = 0
    for c in reversed(coeff):
        y = (y * z + c) % R
    return y


def divide_by_vanishing(coeff, c):
    """p = q (X^64 - c) + rem: the quotient q (4032 coefficients) and the remainder I (64) by long division."""
    a = list(coeff)
    q = [0] * (N - PER_CELL)
    for j in range(N - 1, PER_CELL - 1, -1):
        q[j - PER_CELL] = a[j]
        a[j - PER_CELL] = (a[j - PER_CELL] + c * a[j]) % R
        a[j] = 0
    return q, a[:PER_CELL]


def _c_k(k):
    return pow(coset_for_cell(k)[0], PER_CELL, R)


# ---------------------------------------------------------------- helpers

def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _fr(vals):
    return np.array([[(v >> (64 * k)) & M64 for k in range(4)] for v in vals], dtype=np.uint64).reshape(-1, 4)


def _ints(b):
    b = bytes(b)
    return [int.from_bytes(b[32 * i:32 * i + 32], "big") for i in range(len(b) // 32)]


def _bytes(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "big") for v in vals), dtype=np.uint8).copy()


def _coeff_ints(a):
    return [sum(int(a[i, k]) << (64 * k) for k in range(4)) for i in range(a.shape[0])]


def _edge_blobs(rng):
    """(name, values) of the edge blobs; the low-degree one has quotients that are all zero."""
    low = [rng.randrange(R) for _ in range(PER_CELL - 1)]
    return [("zero", [0] * N), ("r-1", [R - 1] * N), ("constant", [rng.randrange(R)] * N),
            ("first", [rng.randrange(1, R)] + [0] * (N - 1)), ("last", [0] * (N - 1) + [rng.randrange(1, R)]),
            ("degree<64", [evaluate_polynomialcoeff(low, x) for x in ROOTS_BRP])]


@pytest.fixture(scope="module")
def sim():
    """The dev simulation with the cell bodies (its own build: the staleness list covers every device header)."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_kzg_cells.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, f) for f in ("sim_kzg_cells.cpp", "sim_kzg_prove.cpp", "sim_kzg_blob.cpp", "sim.cpp")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def pw(sim):
    out = np.zeros((EXT, 4), np.uint64)
    sim.sim_cells_powers(_p(out))
    return out


def _sim_extend(sim, pw, blobs):
    blobs = np.ascontiguousarray(blobs, np.uint8).reshape(-1, BLOB_BYTES)
    n = blobs.shape[0]
    cells, coeffs, st = np.zeros((n, CELLS, CELL_BYTES), np.uint8), np.zeros((n, N, 4), np.uint64), np.zeros(n, np.uint8)
    sim.sim_cells_extend(_p(blobs), ctypes.c_size_t(n), _p(pw), _p(cells), _p(coeffs), _p(st))
    return cells, coeffs, st


# ---------------------------------------------------------------- CPU: the oracle and the dev simulation

def test_oracle_facts_and_ntt_route():
    """The extended domain's layout (cells 0 .. 63 on roots_brp, cells 64 .. 127 on omega_8192 roots_brp, cell k's
    points h_k omega_64^brp6(j), c_k = omega_128^brp7(k)), and the NTT route of compute_cells against Horner at the
    literal cosets on sampled cells of a random blob."""
    assert pow(ROOTS_EXT[1], N, R) == R - 1
    assert ROOTS_EXT_BRP[:N] == ROOTS_BRP
    assert ROOTS_EXT_BRP[N:] == [ROOTS_EXT[1] * x % R for x in ROOTS_BRP]
    w64, w128 = ROOTS_EXT[EXT // 64], ROOTS_EXT[EXT // 128]
    for k in range(CELLS):
        h = ROOTS_EXT[_brp(k, 7)]
        assert coset_for_cell(k) == [h * pow(w64, _brp(j, 6), R) % R for j in range(PER_CELL)]
        assert _c_k(k) == pow(w128, _brp(k, 7), R)
    rng = random.Random(0xCE11)
    vals = [rng.randrange(R) for _ in range(N)]
    cells, coeff = compute_cells(vals)
    assert [evaluate_polynomialcoeff(coeff, x) for x in ROOTS_BRP[:8]] == vals[:8]
    for k in (0, 63, 64, 65, 127, rng.randrange(CELLS)):
        xs = coset_for_cell(k)
        for j in (0, 1, 31, 63):
            assert cells[k][j] == evaluate_polynomialcoeff(coeff, xs[j]), (k, j)
    assert [v for c in cells[:64] for v in c] == vals


def test_sim_extension_matches_the_oracle(sim, pw):
    """k_cells_extend's body: every cell byte for byte and the coefficients, for seeded and edge blobs; an element >= r
    at index 0 or 4095 gives ZKP_KZG_BAD_SCALAR with zero cells."""
    rng = random.Random(0xE7E7)
    blobs = [("random%d" % i, [rng.randrange(R) for _ in range(N)]) for i in range(2)] + _edge_blobs(rng)
    cells, coeffs, st = _sim_extend(sim, pw, np.stack([_bytes(v) for _, v in blobs]))
    assert not st.any()
    for b, (name, vals) in enumerate(blobs):
        want, coeff = compute_cells(vals)
        assert _coeff_ints(coeffs[b]) == coeff, name
        assert cells[b].tobytes() == b"".join(_bytes(c).tobytes() for c in want), name
    bad = []
    for pos in (0, N - 1):
        v = list(blobs[0][1]); v[pos] = R
        bad.append(_bytes(v))
    big = bytearray(_bytes(blobs[1][1]).tobytes()); big[32 * 7:32 * 8] = b"\xff" * 32
    bad.append(np.frombuffer(bytes(big), np.uint8))
    cells, _, st = _sim_extend(sim, pw, np.stack(bad))
    assert list(st) == [3, 3, 3] and not cells.any()


def test_sim_quotients_match_the_division(sim, pw):
    """k_cells_quotient's chains: the rows of cosets 0, 1, 63, 64, 127 and a random one equal the quotient of the long
    division (top 64 entries zero) and q (X^64 - c_k) + I = p at random points; a degree < 64 blob has zero quotients."""
    rng = random.Random(0x9D1F)
    blobs = [[rng.randrange(R) for _ in range(N)], _edge_blobs(rng)[-1][1]]
    _, coeffs, _ = _sim_extend(sim, pw, np.stack([_bytes(v) for v in blobs]))
    ks = [0, 1, 63, 64, 127, rng.randrange(CELLS)]
    for b, vals in enumerate(blobs):
        rows = np.zeros((len(ks), BLOB_BYTES), np.uint8)
        sim.sim_cells_quotient(_p(np.ascontiguousarray(coeffs[b])), _p(pw), _p(np.array(ks, np.int32)), ctypes.c_size_t(len(ks)), _p(rows))
        coeff = _coeff_ints(coeffs[b])
        for r, k in enumerate(ks):
            q, rem = divide_by_vanishing(coeff, _c_k(k))
            got = _ints(rows[r])
            assert got == q + [0] * PER_CELL, (b, k)
            if b == 1:
                assert not any(q)
            for x in (rng.randrange(R), rng.randrange(R)):
                lhs = (evaluate_polynomialcoeff(q, x) * (pow(x, PER_CELL, R) - _c_k(k)) + evaluate_polynomialcoeff(rem, x)) % R
                assert lhs == evaluate_polynomialcoeff(coeff, x)


def test_sim_interpolation_matches_the_remainder(sim, pw):
    """k_cells_interp's steps: I_k of every cell of a random blob and of sampled cells of the edge blobs is the remainder
    of p by X^64 - c_k; an index >= 128 or an element >= r gives ZKP_KZG_BAD_SCALAR."""
    rng = random.Random(0x1E7F)
    blobs = [[rng.randrange(R) for _ in range(N)]] + [v for _, v in _edge_blobs(rng)]
    cells_in, idx, want = [], [], []
    for b, vals in enumerate(blobs):
        cells, coeff = compute_cells(vals)
        for k in (range(CELLS) if b == 0 else (0, 64, 127)):
            cells_in.append(_bytes(cells[k])); idx.append(k); want.append(divide_by_vanishing(coeff, _c_k(k))[1])
    cells_in += [cells_in[3], cells_in[3]]
    idx += [CELLS, 1 << 63]
    bad = cells_in[5].copy(); bad[32 * 9:32 * 10] = _bytes([R]); cells_in.append(bad); idx.append(5)
    n = len(idx)
    rows, st = np.zeros((n, CELL_BYTES), np.uint8), np.zeros(n, np.uint8)
    sim.sim_cells_interp(_p(np.stack(cells_in)), _p(np.array(idx, np.uint64)), ctypes.c_size_t(n), _p(pw), _p(rows), _p(st))
    assert list(st) == [0] * len(want) + [3, 3, 3]
    for c, w in enumerate(want):
        assert _ints(rows[c]) == w, c


def test_no_gpu_argument_checks():
    """The cells calls check their arguments on the host and never compute on the CPU."""
    from zkvm_pairings_b200 import _lib, build
    build.build()
    lib = _lib.load()
    buf = np.zeros(BLOB_BYTES, np.uint8)
    pt, st = np.zeros(12, np.uint64), np.zeros(1, np.uint8)
    g2 = np.zeros(65 * 24, np.uint64)
    h = ctypes.c_void_p()
    assert lib.zkp_kzg_setup_create_cells(None, _p(g2), _p(buf), None, ctypes.byref(h)) == -1 and not h.value
    assert lib.zkp_kzg_setup_create_cells(None, _p(g2), _p(buf), None, None) == -1
    assert lib.zkp_kzg_compute_cells_batch(None, None, _p(buf), 1, _p(buf), _p(st)) == -1
    assert lib.zkp_kzg_compute_cells_and_proofs_batch(None, None, _p(buf), 1, _p(buf), _p(pt), _p(st), _p(st)) == -1
    assert lib.zkp_kzg_verify_cell_batch(None, None, _p(pt), None, _p(pt), _p(buf), _p(pt), None, 1, _p(st)) == -1
    assert lib.zkp_kzg_compute_cells_dev(None, 0, None, None, 0, None, None, None) == -1
    assert lib.zkp_kzg_compute_cells_and_proofs_dev(None, 0, None, None, 0, None, None, None, None, None, None) == -1
    assert lib.zkp_kzg_verify_cell_dev(None, 0, None, None, None, None, None, None, None, 0, None, None, None) == -1
    assert lib.zkp_kzg_cells_proofs_scratch_bytes(2) == 2 * N * 32 + 2 * CELLS * BLOB_BYTES + 256
    assert lib.zkp_kzg_verify_cell_scratch_bytes(1) == lib.zkp_kzg_scratch_bytes(1) + 512


# ---------------------------------------------------------------- GPU

def _g1gen():
    return util.g1_to_arr(util.o.G1_GENERATOR)


def _limbs6(v):
    return np.array([(v >> (64 * k)) & M64 for k in range(6)], np.uint64)


@pytest.fixture(scope="module")
def cells_setup(engine):
    """A seeded EIP-7594 trusted setup and its cells setup, with the Lagrange points."""
    from zkvm_pairings_b200 import workloads
    tau, g2m, g1m, lag = workloads.kzg_cell_setup(engine, seed=0x7594)
    s = engine.kzg_setup_cells(g2m, g1m, lag)
    yield dict(tau=tau, g2m=g2m, g1m=g1m, lag=lag, s=s)
    s.close()


def _times_g1(engine, vals):
    return engine.g1_mul_batch(np.tile(_g1gen(), (len(vals), 1)), _fr(vals))


def _cell_bytes(vals):
    cells, _ = compute_cells(vals)
    return np.stack([_bytes(c) for c in cells])


@pytest.mark.gpu
def test_cells_match_the_oracle(engine, cells_setup):
    """Every cell byte for byte at n = 1, n = 3 and across the 2^11-blob chunk boundary (five distinct seeded blobs
    tiled over 2^11 + 3 slots); an element >= r gives ZKP_KZG_BAD_SCALAR and zero cells."""
    rng = random.Random(0xC311)
    vals = [[rng.randrange(R) for _ in range(N)] for _ in range(5)]
    want = np.stack([_cell_bytes(v) for v in vals])
    blobs = np.stack([_bytes(v) for v in vals])
    s = cells_setup["s"]
    for sel in ([0], [1, 2, 3]):
        cells, st = engine.kzg_compute_cells_batch(s, blobs[sel])
        assert not st.any() and np.array_equal(cells, want[sel])
    n = (1 << 11) + 3
    idx = np.arange(n) % 5
    cells, st = engine.kzg_compute_cells_batch(s, blobs[idx])
    assert not st.any() and np.array_equal(cells, want[idx])
    bad = blobs[:2].copy(); bad[1, 32 * 4095:] = 0xFF
    cells, st = engine.kzg_compute_cells_batch(s, bad)
    assert list(st) == [0, 3] and np.array_equal(cells[0], want[0]) and not cells[1].any()


def _q_tau(tau, coeff, k):
    """q_k(tau) = (p(tau) - I_k(tau)) / (tau^64 - c_k)."""
    rem = divide_by_vanishing(coeff, _c_k(k))[1]
    num = (evaluate_polynomialcoeff(coeff, tau) - evaluate_polynomialcoeff(rem, tau)) % R
    return num * pow((pow(tau, PER_CELL, R) - _c_k(k)) % R, -1, R) % R


@pytest.mark.gpu
def test_proofs_equal_q_tau(engine, cells_setup):
    """With the trapdoor tau every proof is [q_k(tau)]G1: all 128 proofs of two blobs, and a sample of 2^7 + 1 blobs
    (across the proof chunk boundary); the cells come out as from compute_cells.  A degree < 64 blob has identity
    proofs."""
    rng = random.Random(0x9707)
    tau = cells_setup["tau"]
    vals = [[rng.randrange(R) for _ in range(N)] for _ in range(2)] + [_edge_blobs(rng)[-1][1]]
    blobs = np.stack([_bytes(v) for v in vals])
    cells, pr, pi, st = engine.kzg_compute_cells_and_proofs_batch(cells_setup["s"], blobs)
    assert not st.any()
    coeffs = [polynomial_eval_to_coeff(v) for v in vals]
    for b in range(2):
        assert np.array_equal(cells[b], _cell_bytes(vals[b]))
        want, winf = _times_g1(engine, [_q_tau(tau, coeffs[b], k) for k in range(CELLS)])
        assert np.array_equal(pr[b], want) and np.array_equal(pi[b], winf)
    assert pi[2].all() and np.array_equal(pr[2], np.tile(np.array([0] * 6 + [1] + [0] * 5, np.uint64), (CELLS, 1)))
    n = (1 << 7) + 1
    idx = np.arange(n) % 2
    cells, pr, pi, st = engine.kzg_compute_cells_and_proofs_batch(cells_setup["s"], blobs[idx])
    assert not st.any()
    ks = [(b, k) for b in (0, 1, 127, 128) for k in (0, 63, 64, 127, rng.randrange(CELLS))]
    want, winf = _times_g1(engine, [_q_tau(tau, coeffs[idx[b]], k) for b, k in ks])
    for (b, k), w, wi in zip(ks, want, winf):
        assert np.array_equal(pr[b, k], w) and pi[b, k] == wi, (b, k)
        assert np.array_equal(cells[b], cells[idx[b]])


def _cells_and_proofs(engine, cs, vals):
    blobs = np.stack([_bytes(v) for v in vals])
    cells, pr, pi, st = engine.kzg_compute_cells_and_proofs_batch(cs["s"], blobs)
    c, ci, cst = engine.kzg_blob_to_commitment_batch(cs["s"], blobs)
    assert not st.any() and not cst.any()
    return cells, pr, pi, c, ci


def _flat(cells, pr, pi, c, ci, blobs_idx):
    """Every cell of the given blobs as verifier rows: (C, C_inf, index, cell, pi, pi_inf)."""
    rows = [(c[b], ci[b], k, cells[b, k], pr[b, k], pi[b, k]) for b in blobs_idx for k in range(CELLS)]
    return [np.stack([r[i] for r in rows]) for i in range(6)]


@pytest.mark.gpu
def test_cells_verify_and_changes_fail(engine, cells_setup):
    """All cells and proofs computed on the GPU verify against the commitment of kzg_blob_to_commitment_batch (the
    Lagrange points with the same tau; it equals [p(tau)]G1), the degree < 64 blob with its identity proofs too.  A
    changed element, a swapped cell index, a proof of another cell and another blob's commitment give INVALID."""
    rng = random.Random(0xF3F3)
    vals = [[rng.randrange(R) for _ in range(N)] for _ in range(2)] + [_edge_blobs(rng)[-1][1]]
    cells, pr, pi, c, ci = _cells_and_proofs(engine, cells_setup, vals)
    want, _ = _times_g1(engine, [evaluate_polynomialcoeff(polynomial_eval_to_coeff(v), cells_setup["tau"]) for v in vals])
    assert np.array_equal(c, want)
    C, Ci, K, X, P, Pi = _flat(cells, pr, pi, c, ci, range(3))
    st = engine.kzg_verify_cell_batch(cells_setup["s"], C, K, X, P, Ci, Pi)
    assert not st.any()
    X2 = X.copy(); X2[5, 40] ^= 1                               # a changed element
    K2 = K.copy(); K2[[7, 8]] = K[[8, 7]]                        # swapped indices
    P2 = P.copy(); P2[9] = P[10]                                 # the proof of another cell
    C2 = C.copy(); C2[11] = C[CELLS + 11]                        # another blob's commitment
    st = engine.kzg_verify_cell_batch(cells_setup["s"], C2, K2, X2, P2, Ci, Pi)
    bad = {5, 7, 8, 9, 11}
    assert [int(v) for v in st] == [1 if i in bad else 0 for i in range(len(st))]


@pytest.mark.gpu
def test_cell_rejections(engine, cells_setup, pyref, coracle):
    """An element >= r or an index >= 128 gives BAD_SCALAR; a non-canonical, off-curve or non-subgroup C or pi gives
    BAD_POINT, which takes precedence over BAD_SCALAR."""
    rng = random.Random(0xBAD7)
    cells, pr, pi, c, ci = _cells_and_proofs(engine, cells_setup, [[rng.randrange(R) for _ in range(N)]])
    g1b, _, e1, _, _, _ = util.group_check_cases(pyref, coracle)
    off, tor = g1b[list(e1).index(1)], g1b[list(e1).index(2)]
    rows = []

    def add(k, cc=None, cell=None, p=None, idx=None, want=0):
        rows.append((c[0] if cc is None else cc, k if idx is None else idx, cells[0, k] if cell is None else cell,
                     pr[0, k] if p is None else p, want))

    add(3)
    big = cells[0, 4].copy(); big[:32] = 0xFF
    add(4, cell=big, want=3)
    add(5, cell=np.concatenate([cells[0, 5][:32 * 63], _bytes([R])]), want=3)
    add(6, idx=CELLS, want=3)
    add(6, idx=(1 << 64) - 1, want=3)
    nc = c[0].copy(); nc[:6] = _limbs6(sum(int(v) << (64 * i) for i, v in enumerate(c[0][:6])) + util.o.P)
    add(7, cc=nc, want=2)
    add(8, p=off, want=2)
    add(9, cc=tor, want=2)
    add(10, p=tor, want=2)
    add(11, p=tor, idx=CELLS, want=2)
    add(12, cc=off, cell=big, want=2)
    C, X, P = (np.stack([r[i] for r in rows]) for i in (0, 2, 3))
    K = np.array([r[1] for r in rows], np.uint64)   # straight to uint64: 2^64 - 1 survives no float conversion
    st = engine.kzg_verify_cell_batch(cells_setup["s"], C, K, X, P)
    assert [int(v) for v in st] == [r[4] for r in rows]


@pytest.mark.gpu
def test_cells_setup_rejections(engine, cells_setup):
    """Setup creation rejects a limb >= p, an off-curve point (naming its index), two swapped monomial points, a wrong
    g2_monomial[64] and g1_monomial[0] != G1; the cells calls refuse a setup made without monomial points."""
    import zkvm_pairings_b200 as z
    g2m, g1m = cells_setup["g2m"], cells_setup["g1m"]
    bad = g1m.copy(); bad[9, :6] = _limbs6(util.o.P)
    with pytest.raises(z.NonCanonicalError):
        engine.kzg_setup_cells(g2m, bad)
    bad = g1m.copy(); bad[17, 6] ^= 1
    with pytest.raises(z.ZkpError) as ei:
        engine.kzg_setup_cells(g2m, bad)
    assert ei.value.code == -1 and "g1_monomial[17]" in str(ei.value) and "not on the curve" in str(ei.value)
    cases = []
    sw = g1m.copy(); sw[[300, 301]] = g1m[[301, 300]]
    cases.append((g2m, sw, "g1_monomial[300] is inconsistent"))
    wrong = g2m.copy(); wrong[64] = g2m[63]
    cases.append((wrong, g1m, "g2_monomial[64] is inconsistent"))
    first = g1m.copy(); first[0] = g1m[1]
    cases.append((g2m, first, "g1_monomial[0] is not the G1 generator"))
    for a, b, msg in cases:
        with pytest.raises(z.ZkpError) as ei:
            engine.kzg_setup_cells(a, b)
        assert ei.value.code == -1 and msg in str(ei.value), str(ei.value)
    blob = np.zeros((1, BLOB_BYTES), np.uint8)
    with engine.kzg_setup(g2m[1]) as plain:
        with pytest.raises(z.ZkpError) as ei:
            engine.kzg_compute_cells_batch(plain, blob)
        assert ei.value.code == -1 and "no monomial points" in str(ei.value)


@pytest.mark.gpu
def test_dev_forms_equal_host_forms(engine, cells_setup):
    """The _dev forms on device-resident tensors give the host forms' cells, proofs and verdicts, n = 0 included."""
    import torch
    rng = random.Random(0xDE77)
    s = cells_setup["s"]
    vals = [[rng.randrange(R) for _ in range(N)] for _ in range(3)]
    blobs = np.stack([_bytes(v) for v in vals])
    cells, pr, pi, st = engine.kzg_compute_cells_and_proofs_batch(s, blobs)
    c, ci, _ = engine.kzg_blob_to_commitment_batch(s, blobs)
    n = 3
    db = torch.from_numpy(blobs).cuda()
    dcells = torch.zeros((n, CELLS, CELL_BYTES), dtype=torch.uint8, device="cuda")
    dst = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    engine.kzg_compute_cells_dev(s, db, n, dcells, dst)
    assert np.array_equal(dcells.cpu().numpy(), cells) and not dst.cpu().numpy().any()
    dcells.zero_(); dst.fill_(9)
    dp = torch.zeros((n, CELLS, 12), dtype=torch.int64, device="cuda")
    dpi = torch.zeros((n, CELLS), dtype=torch.uint8, device="cuda")
    scratch = torch.empty(engine.kzg_cells_proofs_scratch_bytes(n), dtype=torch.uint8, device="cuda")
    engine.kzg_compute_cells_and_proofs_dev(s, db, n, dcells, dp, dpi, dst, scratch)
    engine.kzg_compute_cells_and_proofs_dev(s, db, 0, dcells, dp, dpi, dst, scratch)
    assert np.array_equal(dcells.cpu().numpy(), cells) and np.array_equal(dp.cpu().numpy().view(np.uint64), pr)
    assert np.array_equal(dpi.cpu().numpy(), pi) and not dst.cpu().numpy().any()
    C, Ci, K, X, P, Pi = _flat(cells, pr, pi, c, ci, range(n))
    X[17, 3] ^= 1
    host = engine.kzg_verify_cell_batch(s, C, K, X, P, Ci, Pi)
    m = len(K)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).cuda()
    dvs = torch.full((m,), 9, dtype=torch.uint8, device="cuda")
    vscratch = torch.empty(engine.kzg_verify_cell_scratch_bytes(m), dtype=torch.uint8, device="cuda")
    engine.kzg_verify_cell_dev(s, t(C, np.int64), t(K.astype(np.uint64), np.int64), t(X, np.uint8), t(P, np.int64), m, dvs, vscratch,
                               d_commitment_inf=t(Ci, np.uint8), d_proof_inf=t(Pi, np.uint8))
    assert np.array_equal(dvs.cpu().numpy(), host) and int(host[17]) == 1 and host.sum() == 1


@pytest.mark.gpu
def test_cells_multi_device_matches_single(engine, cells_setup):
    import zkvm_pairings_b200 as z
    if z.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    rng = random.Random(0x3D3D)
    blobs = np.stack([_bytes([rng.randrange(R) for _ in range(N)]) for _ in range(5)])
    multi = z.PairingEngine()
    try:
        with multi.kzg_setup_cells(cells_setup["g2m"], cells_setup["g1m"], cells_setup["lag"]) as sm:
            a = engine.kzg_compute_cells_and_proofs_batch(cells_setup["s"], blobs)
            b = multi.kzg_compute_cells_and_proofs_batch(sm, blobs)
            assert all(np.array_equal(x, y) for x, y in zip(a, b))
            c, ci, _ = engine.kzg_blob_to_commitment_batch(cells_setup["s"], blobs)
            C, Ci, K, X, P, Pi = _flat(a[0], a[1], a[2], c, ci, range(5))
            assert np.array_equal(engine.kzg_verify_cell_batch(cells_setup["s"], C, K, X, P, Ci, Pi),
                                  multi.kzg_verify_cell_batch(sm, C, K, X, P, Ci, Pi))
    finally:
        multi.close()
