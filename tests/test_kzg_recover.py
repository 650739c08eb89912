"""EIP-7594 cell recovery (zkp_kzg_recover_cells_*, zkp_kzg_recover_cells_and_proofs_*): the two-block cluster of
csrc/kzg_recover.cuh bit-exact against a literal restatement of the spec's recover_polynomialcoeff (consensus specs, fulu
polynomial-commitments-sampling.md) through the CPU dev simulation, for consistent and inconsistent cells, and the GPU
entry points against compute_cells / compute_cells_and_kzg_proofs, the trapdoor tau and the cell verifier."""
import ctypes
import os
import random
import re
import subprocess

import numpy as np
import pytest

# the spec restatement, helpers and the module-scoped cells_setup fixture of the cells tests
from test_kzg_cells import (BLOB_BYTES, CELL_BYTES, CELLS, EXT, N, PER_CELL, R, ROOTS_EXT, _brp, _bytes, _coeff_ints, _edge_blobs, _ints,
                            _ntt, _p, _q_tau, _times_g1, cells_setup, compute_roots_of_unity, polynomial_eval_to_coeff)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_CELLS, BAD_SCALAR = 4, 3
RF = (1 << 256) % R   # Fr Montgomery radix

# ---------------------------------------------------------------- the consensus specs (fulu polynomial-commitments-sampling.md)

def fft_field(vals, inv=False):
    if inv:
        inv_n = pow(len(vals), -1, R)
        return [v * inv_n % R for v in _ntt(vals, pow(ROOTS_EXT[1], -1, R))]
    return _ntt(vals, ROOTS_EXT[1])


def shift_vals(vals, factor):
    out, s = [], 1
    for v in vals:
        out.append(v * s % R)
        s = s * factor % R
    return out


def coset_fft_field(vals, inv=False):
    """PRIMITIVE_ROOT_OF_UNITY = 7 is the shift."""
    if inv:
        return shift_vals(fft_field(vals, inv=True), pow(7, -1, R))
    return fft_field(shift_vals(vals, 7))


def vanishing_polynomialcoeff(xs):
    p = [1]
    for x in xs:
        q = [0] * (len(p) + 1)
        for i, c in enumerate(p):
            q[i] = (q[i] - x * c) % R
            q[i + 1] = (q[i + 1] + c) % R
        p = q
    return p


def construct_vanishing_polynomial(missing_cell_indices):
    reduced = compute_roots_of_unity(CELLS)
    short = vanishing_polynomialcoeff([reduced[_brp(m, 7)] for m in missing_cell_indices])
    z = [0] * EXT
    for i, c in enumerate(short):
        z[i * PER_CELL] = c
    return z


def recover_polynomialcoeff(cell_indices, cells):
    e_rbo = [0] * EXT
    for k, cell in zip(cell_indices, cells):
        e_rbo[k * PER_CELL:(k + 1) * PER_CELL] = cell
    e = [e_rbo[_brp(i, 13)] for i in range(EXT)]
    zpoly = construct_vanishing_polynomial([k for k in range(CELLS) if k not in cell_indices])
    ez = fft_field([a * b % R for a, b in zip(fft_field(zpoly), e)], inv=True)
    over = coset_fft_field(ez)
    zover = coset_fft_field(zpoly)
    return coset_fft_field([a * pow(b, -1, R) % R for a, b in zip(over, zover)], inv=True)[:N]


def cells_of_coeff(coeff):
    """compute_cells_and_kzg_proofs_polynomialcoeff's cells: the coefficients over the 8192 roots, bit-reversed."""
    ext = _ntt(list(coeff) + [0] * N, ROOTS_EXT[1])
    ys = [ext[_brp(i, 13)] for i in range(EXT)]
    return [ys[PER_CELL * k:PER_CELL * (k + 1)] for k in range(CELLS)]


def spec_accepts(cell_indices, cells):
    """The asserts of recover_cells_and_kzg_proofs (cell_to_coset_evals rejects an element >= r)."""
    return (CELLS // 2 <= len(cell_indices) <= CELLS and len(set(cell_indices)) == len(cell_indices)
            and list(cell_indices) == sorted(cell_indices) and all(k < CELLS for k in cell_indices)
            and all(v < R for c in cells for v in c))


# ---------------------------------------------------------------- helpers

def _patterns(rng):
    """(name, the present cell indices) of the erasure patterns."""
    return [("first64", list(range(64))), ("last64", list(range(64, 128))), ("even", list(range(0, 128, 2))),
            ("odd", list(range(1, 128, 2))), ("random64", sorted(rng.sample(range(CELLS), 64))),
            ("random100", sorted(rng.sample(range(CELLS), 100))), ("127", sorted(rng.sample(range(CELLS), 127))),
            ("all", list(range(CELLS)))]


def _inputs(rows):
    """rows = [(indices, cells (len(indices), CELL_BYTES) uint8)] -> the padded (idx, cells, num) arrays of the ABI."""
    n = len(rows)
    idx, cl, num = np.zeros((n, CELLS), np.uint64), np.zeros((n, CELLS, CELL_BYTES), np.uint8), np.zeros(n, np.uint64)
    for b, (ks, c) in enumerate(rows):
        m = len(ks)
        num[b] = m
        idx[b, :min(m, CELLS)] = np.array(ks[:CELLS], np.uint64)
        cl[b, :min(m, CELLS)] = c[:CELLS]
    return idx, cl, num


def _cells_bytes(cells):
    return np.stack([_bytes(c) for c in cells])


@pytest.fixture(scope="module")
def rsim():
    """The dev simulation with the recovery bodies (its own build: the staleness list covers every device header)."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_kzg_recover.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, f) for f in ("sim_kzg_recover.cpp", "sim_kzg_cells.cpp", "sim_kzg_prove.cpp", "sim_kzg_blob.cpp", "sim.cpp")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def rpw(rsim):
    out = np.zeros((EXT, 4), np.uint64)
    rsim.sim_cells_powers(_p(out))
    return out


def _sim_recover(rsim, pw, rows, raw=None):
    """The simulated k_cells_recover over rows (see _inputs), or over raw = (idx, cells, num) -> (cells, coefficients,
    statuses, z and 1 / zc (n, 2, 128, 4) Montgomery)."""
    idx, cl, num = raw if raw is not None else _inputs(rows)
    n = idx.shape[0]
    out, coeffs, st = np.zeros((n, CELLS, CELL_BYTES), np.uint8), np.zeros((n, N, 4), np.uint64), np.zeros(n, np.uint8)
    van = np.zeros((n, 2, CELLS, 4), np.uint64)
    rsim.sim_cells_recover(_p(idx), _p(cl), _p(num), ctypes.c_size_t(n), _p(pw), _p(out), _p(coeffs), _p(st), _p(van))
    return out, coeffs, st, van


def _sim_extend(rsim, pw, blobs):
    blobs = np.ascontiguousarray(blobs, np.uint8).reshape(-1, BLOB_BYTES)
    n = blobs.shape[0]
    cells, coeffs, st = np.zeros((n, CELLS, CELL_BYTES), np.uint8), np.zeros((n, N, 4), np.uint64), np.zeros(n, np.uint8)
    rsim.sim_cells_extend(_p(blobs), ctypes.c_size_t(n), _p(pw), _p(cells), _p(coeffs), _p(st))
    return cells, coeffs, st


def _canon(words):
    """A Montgomery Fr (4 u64) -> its value."""
    return sum(int(w) << (64 * i) for i, w in enumerate(words)) * pow(RF, -1, R) % R


def _random_cells(rng, ks):
    return [[rng.randrange(R) for _ in range(PER_CELL)] for _ in ks]


# ---------------------------------------------------------------- CPU: the oracle and the dev simulation

def test_vanishing_scalars_and_constants(rsim, rpw):
    """The kernel's z_k and 1 / zc_k equal fft_field and coset_fft_field of construct_vanishing_polynomial at every slot
    of cell k (slot j = 64 k + t of the bit-reversed domain); zc_k is never zero; the recovery constants of consts.cuh
    hold their values."""
    rng = random.Random(0x2E50)
    for present in (sorted(rng.sample(range(CELLS), 64)), sorted(rng.sample(range(CELLS), 127)), list(range(CELLS))):
        _, _, st, van = _sim_recover(rsim, rpw, [(present, _cells_bytes(_random_cells(rng, present)))])
        assert st[0] == 0
        zpoly = construct_vanishing_polynomial([k for k in range(CELLS) if k not in present])
        ze, zc = fft_field(zpoly), coset_fft_field(zpoly)
        z = [_canon(van[0, 0, k]) for k in range(CELLS)]
        zci = [_canon(van[0, 1, k]) for k in range(CELLS)]
        for j in range(EXT):
            i, k = _brp(j, 13), j // PER_CELL
            assert ze[i] == z[k] and zc[i] * zci[k] % R == 1, (j, len(present))
        assert all(zc) and all((z[k] == 0) == (k not in present) for k in range(CELLS))
    text = open(os.path.join(ROOT, "zkvm_pairings_b200", "csrc", "consts.cuh")).read()

    def const(name):
        words = re.search(r"%s\[8\] = \{\s*([^}]*)\}" % name, text).group(1).replace("u", "").split(",")
        return sum(int(w, 16) << (32 * i) for i, w in enumerate(w for w in words if w.strip()))
    want = {"ZKP_FR_INV_EXT_N": pow(EXT, -1, R), "ZKP_FR_SHIFT": 7, "ZKP_FR_SHIFT_INV": pow(7, -1, R), "ZKP_FR_SHIFT_64": pow(7, 64, R),
            "ZKP_FR_SHIFT_512": pow(7, 512, R), "ZKP_FR_SHIFT_INV_512": pow(7, -512, R), "ZKP_FR_SHIFT_4096": pow(7, 4096, R)}
    for name, v in want.items():
        assert const(name) == v * RF % R, name


def test_sim_matches_the_spec(rsim, rpw):
    """The simulated cluster is bit-exact to the literal recover_polynomialcoeff (coefficients and the cells of
    compute_cells_and_kzg_proofs_polynomialcoeff) on inconsistent random cells for every erasure pattern, and on the
    consistent cells of a random blob and an edge blob."""
    rng = random.Random(0x5EC7)
    rows = [(ks, _random_cells(rng, ks)) for _, ks in _patterns(rng) if len(ks) < CELLS]
    vals = [rng.randrange(R) for _ in range(N)]
    for blob, ks in ((vals, sorted(rng.sample(range(CELLS), 64))), (_edge_blobs(rng)[1][1], list(range(1, 128, 2)))):
        full = cells_of_coeff(polynomial_eval_to_coeff(blob))
        rows.append((ks, [full[k] for k in ks]))
    out, coeffs, st, _ = _sim_recover(rsim, rpw, [(ks, _cells_bytes(c)) for ks, c in rows])
    assert not st.any()
    for b, (ks, c) in enumerate(rows):
        coeff = recover_polynomialcoeff(ks, c)
        assert _coeff_ints(coeffs[b]) == coeff, b
        assert out[b].tobytes() == _cells_bytes(cells_of_coeff(coeff)).tobytes(), b


def test_sim_round_trip(rsim, rpw):
    """recover(erase(compute_cells(blob))) == compute_cells(blob), and the coefficients are the blob's, for two random
    blobs and the edge blobs (zero, r - 1, constant, single first / last, degree < 64) under every erasure pattern."""
    rng = random.Random(0x7219)
    blobs = [[rng.randrange(R) for _ in range(N)] for _ in range(2)] + [v for _, v in _edge_blobs(rng)]
    cells, coeffs, st = _sim_extend(rsim, rpw, np.stack([_bytes(v) for v in blobs]))
    assert not st.any()
    pats = _patterns(rng)
    rows = [(ks, cells[b][ks]) for b in range(len(blobs)) for _, ks in pats]
    out, rc, st, _ = _sim_recover(rsim, rpw, rows)
    assert not st.any()
    for i in range(len(rows)):
        b = i // len(pats)
        assert np.array_equal(out[i], cells[b]), (b, pats[i % len(pats)][0])
        assert np.array_equal(rc[i], coeffs[b]), (b, pats[i % len(pats)][0])


def _status_rows(rng, cells):
    """(name, indices, cells, want) of malformed inputs around one blob's cells, with the spec's verdict checked."""
    ks = sorted(rng.sample(range(CELLS), 80))
    big = cells[ks].copy(); big[3, 32 * 5:32 * 6] = _bytes([R])
    big_hi = cells[ks].copy(); big_hi[-1, -32:] = 0xFF
    rows = [("valid", ks, cells[ks], 0),
            ("63 cells", ks[:63], cells[ks[:63]], BAD_CELLS),
            ("duplicate", ks[:40] + [ks[40]] + ks[40:79], cells[ks[:40] + [ks[40]] + ks[40:79]], BAD_CELLS),
            ("descending", ks[:10] + [ks[11], ks[10]] + ks[12:], cells[ks[:10] + [ks[11], ks[10]] + ks[12:]], BAD_CELLS),
            ("index 128", ks[:-1] + [CELLS], cells[ks], BAD_CELLS),
            ("element >= r, rank 0", ks, big, BAD_SCALAR),
            ("element >= r, rank 1", ks, big_hi, BAD_SCALAR),
            ("duplicate and element >= r", ks[:40] + [ks[40]] + ks[40:79], np.concatenate([big[:41], big[40:79]]), BAD_CELLS)]
    for name, i, c, want in rows:
        assert spec_accepts(i, [_ints(x) for x in c]) == (want == 0), name
    return rows


def test_sim_statuses(rsim, rpw):
    """63 cells, a count of 129, a duplicate, a descending pair and index 128 give BAD_CELLS; an element >= r gives
    BAD_SCALAR (in either block's half), BAD_CELLS wins over it; a rejected blob gets zero cells; an entry beyond
    num_cells is ignored."""
    rng = random.Random(0xBAD5)
    cells, _, _ = _sim_extend(rsim, rpw, _bytes([rng.randrange(R) for _ in range(N)]))
    cells = cells[0]
    rows = _status_rows(rng, cells)
    idx, cl, num = _inputs([(i, c) for _, i, c, _ in rows])
    extra = _inputs([(list(range(CELLS)), cells)])   # count 129: 128 entries that would be valid
    idx = np.concatenate([idx, extra[0]]); cl = np.concatenate([cl, extra[1]]); num = np.concatenate([num, np.array([CELLS + 1], np.uint64)])
    ign = _inputs([(rows[0][1], rows[0][2])])        # an element >= r and index 0 beyond num_cells
    ign[0][0, 80] = 0; ign[1][0, 80, :32] = 0xFF
    idx = np.concatenate([idx, ign[0]]); cl = np.concatenate([cl, ign[1]]); num = np.concatenate([num, ign[2]])
    out, _, st, _ = _sim_recover(rsim, rpw, None, raw=(idx, cl, num))
    want = [w for _, _, _, w in rows] + [BAD_CELLS, 0]
    assert list(st) == want
    for b, w in enumerate(want):
        assert np.array_equal(out[b], cells) if w == 0 else not out[b].any(), b


def test_no_gpu_argument_checks():
    """The recovery calls check their arguments on the host and never compute on the CPU."""
    from zkvm_pairings_b200 import _lib, build
    build.build()
    lib = _lib.load()
    buf, idx, st = np.zeros(CELL_BYTES, np.uint8), np.zeros(CELLS, np.uint64), np.zeros(1, np.uint8)
    pt = np.zeros(12, np.uint64)
    assert lib.zkp_kzg_recover_cells_batch(None, None, _p(idx), _p(buf), _p(idx), 1, _p(buf), _p(st)) == -1
    assert lib.zkp_kzg_recover_cells_and_proofs_batch(None, None, _p(idx), _p(buf), _p(idx), 1, _p(buf), _p(pt), _p(st), _p(st)) == -1
    assert lib.zkp_kzg_recover_cells_dev(None, 0, None, None, None, None, 0, None, None, None) == -1
    assert lib.zkp_kzg_recover_cells_and_proofs_dev(None, 0, None, None, None, None, 0, None, None, None, None, None, None) == -1


# ---------------------------------------------------------------- GPU

def _erase(rng, full, m=None):
    """A random erasure of one blob's cells (128, CELL_BYTES): (indices, cells) with m (default: random 64 .. 128) present."""
    ks = sorted(rng.sample(range(CELLS), m if m is not None else rng.randrange(64, CELLS + 1)))
    return ks, full[ks]


@pytest.fixture(scope="module")
def base(engine, cells_setup):
    """Five seeded blobs, their cells and proofs from compute_cells_and_kzg_proofs, and their commitments."""
    rng = random.Random(0x8EC0)
    vals = [[rng.randrange(R) for _ in range(N)] for _ in range(5)]
    blobs = np.stack([_bytes(v) for v in vals])
    cells, pr, pi, st = engine.kzg_compute_cells_and_proofs_batch(cells_setup["s"], blobs)
    c, ci, cst = engine.kzg_blob_to_commitment_batch(cells_setup["s"], blobs)
    assert not st.any() and not cst.any()
    return dict(vals=vals, blobs=blobs, cells=cells, pr=pr, pi=pi, c=c, ci=ci)


@pytest.mark.gpu
def test_round_trip_matches_compute_cells(engine, cells_setup, base):
    """Byte for byte against kzg_compute_cells_batch at n = 1, n = 3 and across the 2^11-blob chunk boundary, with a
    different random erasure (64 .. 128 cells) in every slot and the named patterns among them."""
    rng = random.Random(0x2071)
    s, full = cells_setup["s"], base["cells"]
    pats = _patterns(rng)
    for sel in ([0], [1, 2, 3]):
        rows = [(pats[i][1], full[b][pats[i][1]]) for i, b in enumerate(sel)]
        out, st = engine.kzg_recover_cells_batch(s, *_inputs(rows))
        assert not st.any() and np.array_equal(out, full[sel])
    n = (1 << 11) + 3
    which = np.arange(n) % 5
    rows = [(pats[i][1], full[which[i]][pats[i][1]]) if i < len(pats) else _erase(rng, full[which[i]]) for i in range(n)]
    out, st = engine.kzg_recover_cells_batch(s, *_inputs(rows))
    assert not st.any() and np.array_equal(out, full[which])


@pytest.mark.gpu
def test_inconsistent_cells_match_the_simulation(engine, cells_setup, rsim, rpw):
    """Cells that belong to no one blob: the GPU's cells (and, with proofs, the proofs of the same coefficients) equal
    the simulation, which is bit-exact to the spec."""
    rng = random.Random(0x1C0E)
    rows = [(ks, _cells_bytes(_random_cells(rng, ks))) for _, ks in _patterns(rng)]
    want, _, wst, _ = _sim_recover(rsim, rpw, rows)
    out, st = engine.kzg_recover_cells_batch(cells_setup["s"], *_inputs(rows))
    assert not wst.any() and not st.any() and np.array_equal(out, want)


@pytest.mark.gpu
def test_proofs_equal_compute_cells_and_proofs(engine, cells_setup, base):
    """All cells and proofs of two blobs equal kzg_compute_cells_and_proofs_batch, as does a sample across the 2^7-blob
    proof chunk boundary; with the trapdoor a sample is [q_k(tau)]G1; every recovered cell and proof verifies against the
    blob's commitment."""
    rng = random.Random(0x9F00)
    s, full = cells_setup["s"], base["cells"]
    rows = [_erase(rng, full[b], 64) for b in (0, 1)]
    out, pr, pi, st = engine.kzg_recover_cells_and_proofs_batch(s, *_inputs(rows))
    assert not st.any()
    assert np.array_equal(out, full[:2]) and np.array_equal(pr, base["pr"][:2]) and np.array_equal(pi, base["pi"][:2])
    n = (1 << 7) + 1
    which = np.arange(n) % 5
    out, pr, pi, st = engine.kzg_recover_cells_and_proofs_batch(s, *_inputs([_erase(rng, full[which[i]]) for i in range(n)]))
    assert not st.any()
    ks = [(b, k) for b in (0, 1, 127, 128) for k in (0, 63, 64, 127, rng.randrange(CELLS))]
    for b, k in ks:
        assert np.array_equal(out[b], full[which[b]]), b
        assert np.array_equal(pr[b, k], base["pr"][which[b], k]) and pi[b, k] == base["pi"][which[b], k], (b, k)
    coeffs = {w: polynomial_eval_to_coeff(base["vals"][w]) for w in set(int(which[b]) for b, _ in ks)}
    want, winf = _times_g1(engine, [_q_tau(cells_setup["tau"], coeffs[int(which[b])], k) for b, k in ks])
    for (b, k), w, wi in zip(ks, want, winf):
        assert np.array_equal(pr[b, k], w) and pi[b, k] == wi, (b, k)
    sel = [0, 1]
    C = np.repeat(base["c"][which[sel]], CELLS, axis=0); Ci = np.repeat(base["ci"][which[sel]], CELLS)
    K = np.tile(np.arange(CELLS, dtype=np.uint64), len(sel))
    vst = engine.kzg_verify_cell_batch(s, C, K, out[sel].reshape(-1, CELL_BYTES), pr[sel].reshape(-1, 12), Ci, pi[sel].reshape(-1))
    assert not vst.any()


@pytest.mark.gpu
def test_rejected_blobs_among_valid_ones(engine, cells_setup, base, rsim, rpw):
    """Malformed blobs among valid ones get their status, zero cells and zero-limb proofs with the flag set; the
    neighbours are unaffected."""
    rng = random.Random(0x4E1E)
    full = base["cells"]
    rows = _status_rows(rng, full[0])
    idx, cl, num = _inputs([(i, c) for _, i, c, _ in rows])
    want = [w for _, _, _, w in rows]
    out, st = engine.kzg_recover_cells_batch(cells_setup["s"], idx, cl, num)
    assert list(st) == want
    out2, pr, pi, st2 = engine.kzg_recover_cells_and_proofs_batch(cells_setup["s"], idx, cl, num)
    assert list(st2) == want and np.array_equal(out, out2)
    for b, w in enumerate(want):
        if w:
            assert not out[b].any() and not pr[b].any() and pi[b].all(), b
        else:
            assert np.array_equal(out[b], full[0]) and np.array_equal(pr[b], base["pr"][0]) and np.array_equal(pi[b], base["pi"][0])


@pytest.mark.gpu
def test_dev_forms_pinned_and_default_stream(engine, cells_setup, base):
    """The _dev forms equal the host forms (queued on the default stream after the uploads, the caller's device left
    current), n = 0 included; pinned and pageable host inputs give the same results."""
    import torch
    rng = random.Random(0xDE70)
    s, full = cells_setup["s"], base["cells"]
    n = 3
    idx, cl, num = _inputs([_erase(rng, full[b]) for b in range(n)])
    cells, pr, pi, st = engine.kzg_recover_cells_and_proofs_batch(s, idx, cl, num)
    assert not st.any() and np.array_equal(cells, full[:n])
    dev_before = torch.cuda.current_device()
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).cuda()
    di, dc, dn = t(idx, np.int64), t(cl, np.uint8), t(num, np.int64)
    dout = torch.zeros((n, CELLS, CELL_BYTES), dtype=torch.uint8, device="cuda")
    dst = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    engine.kzg_recover_cells_dev(s, di, dc, dn, n, dout, dst)
    assert np.array_equal(dout.cpu().numpy(), cells) and not dst.cpu().numpy().any()
    dout.zero_(); dst.fill_(9)
    dp = torch.zeros((n, CELLS, 12), dtype=torch.int64, device="cuda")
    dpi = torch.zeros((n, CELLS), dtype=torch.uint8, device="cuda")
    scratch = torch.empty(engine.kzg_cells_proofs_scratch_bytes(n), dtype=torch.uint8, device="cuda")
    engine.kzg_recover_cells_and_proofs_dev(s, di, dc, dn, n, dout, dp, dpi, dst, scratch)
    engine.kzg_recover_cells_and_proofs_dev(s, di, dc, dn, 0, dout, dp, dpi, dst, scratch)
    assert np.array_equal(dout.cpu().numpy(), cells) and np.array_equal(dp.cpu().numpy().view(np.uint64), pr)
    assert np.array_equal(dpi.cpu().numpy(), pi) and not dst.cpu().numpy().any()
    assert torch.cuda.current_device() == dev_before
    pins = [torch.empty(a.shape, dtype=torch.uint8 if a.dtype == np.uint8 else torch.int64, pin_memory=True) for a in (idx, cl, num)]
    for p, a in zip(pins, (idx, cl, num)):
        p.numpy()[...] = a.view(p.numpy().dtype)
    out, st2 = engine.kzg_recover_cells_batch(s, pins[0].numpy().view(np.uint64), pins[1].numpy(), pins[2].numpy().view(np.uint64))
    assert np.array_equal(out, cells) and not st2.any()


@pytest.mark.gpu
def test_recover_multi_device_matches_single(engine, cells_setup, base):
    import zkvm_pairings_b200 as z
    if z.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    rng = random.Random(0x3D3E)
    inp = _inputs([_erase(rng, base["cells"][b % 5]) for b in range(7)])
    multi = z.PairingEngine()
    try:
        with multi.kzg_setup_cells(cells_setup["g2m"], cells_setup["g1m"], cells_setup["lag"]) as sm:
            a = engine.kzg_recover_cells_and_proofs_batch(cells_setup["s"], *inp)
            b = multi.kzg_recover_cells_and_proofs_batch(sm, *inp)
            assert all(np.array_equal(x, y) for x, y in zip(a, b))
            assert all(np.array_equal(x, y) for x, y in zip(engine.kzg_recover_cells_batch(cells_setup["s"], *inp),
                                                             multi.kzg_recover_cells_batch(sm, *inp)))
    finally:
        multi.close()
