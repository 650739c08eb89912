"""The device arithmetic at the limits it is designed for.

fp.cuh / tower.cuh accept Montgomery representatives anywhere in [0, 2p] (one mont_mul operand up to 4p, unreduced
Fp6 recombinations up to 68 p^2), but the C ABI converts canonical inputs at load time and never delivers a
representative above ~1.1 p.  tests/device_harness/bodies.cuh runs the bodies on RAW representatives instead:
compiled with nvcc once per define set a shipped unit uses (harness.cu, built into a temporary directory) and as plain
C++ in the dev simulation (tests/host_sim/sim.cpp, sim_body).  Every body is checked with Python big integers or
the C oracle at the corners of its operand box, and the device's raw output words must equal the simulation's.

The binary-GCD inversion (tower.cuh fp_inv) runs a fixed 2 * 381 - 1 iterations, and its result depends on all but
the last of them: the internal value 3 * 2^379 makes its last swap in iteration 760 (2^380 runs all 761 to a = 0).
Canonical 3/32 and 1/16 load as exactly these values (R = 2^384), so the worst cases are reachable through the C ABI
too; those rows go through zkp_tower_op_batch and the simulation.

Fr (fr.cuh) keeps every value in [0, r) (4r > 2^256 rules out a redundant form), so its bodies run at the corners of
that range: 0, 1, 2, r - 1, r - 2, the long carry patterns, and sums of exactly r and 2r - 2; the range checks
(fr_geq_r, fr_reduce_once, blob_element) also at r, r + 1, 2r - 1 and 2^256 - 1.  fr_inv runs a fixed 2 * 255 - 1
iterations: the internal value 3 * 2^253 (canonical 3/8) makes its last swap in iteration 508.  blob_element and
store_be32 read and write bytes through uint4 and __byte_perm on the device and through byte loops in the
simulation, so their device words are compared with the simulation's too.

Last, the multi-pairing entry points at every check width 1..8 and the prepared-table path at (pairs, prepared)
combinations the other tests do not use, with points at infinity in the first, the last and every pair of a check."""
import ctypes
import hashlib
import os
import random
import re
import subprocess
import tempfile
import zlib

import numpy as np
import pytest

import pyref
import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
HARNESS_DIR = os.path.join(ROOT, "tests", "device_harness")
HEADERS = [os.path.join(CSRC, f) for f in ("fp.cuh", "tower.cuh", "pairing.cuh", "ops.cuh", "consts.cuh", "fr.cuh", "blob.cuh",
                                           "kzg.cuh", "groth16.cuh", "kzg_prove.cuh")]

P = pyref.P
R = 1 << 384
RINV = pow(R, -1, P)
W768 = (1 << 768) - 1
SLOTS = 16                   # Fp2 slots per element (bodies.cuh BODY_SLOTS)
U64 = 12 * SLOTS


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _body_codes():
    text = open(os.path.join(HARNESS_DIR, "bodies.cuh")).read()
    enum = re.search(r"enum Body \{(.*?)\};", text, re.S).group(1)
    enum = re.sub(r"//[^\n]*", "", enum)
    codes, nxt = {}, 0
    for item in (s.strip() for s in enum.split(",")):
        if not item:
            continue
        name, _, val = item.partition("=")
        nxt = int(val) if val.strip() else nxt
        codes[name.strip()[2:].lower()] = nxt
        nxt += 1
    return codes


BODY = _body_codes()
assert SLOTS == int(re.search(r"#define BODY_SLOTS (\d+)", open(os.path.join(HARNESS_DIR, "bodies.cuh")).read()).group(1))


def _define(unit, name):
    m = re.search(r"#define %s (\d+)\b" % name, open(os.path.join(CSRC, unit)).read())
    return int(m.group(1))


def define_sets():
    """name -> (nvcc -D flags, ZKP_LAZY of that set): the three shipped units' sets, read from their sources, and the
    measured-but-unshipped everywhere-lazy ZKP_LAZY = 7"""
    pk = open(os.path.join(CSRC, "pairing_kernel.cu")).read()
    fe = open(os.path.join(CSRC, "fe_kernel.cu")).read()
    kern = open(os.path.join(CSRC, "kernels.cu")).read()
    assert "#define ZKP_LOOP_SYNC ZKP_MILLER_SYNC" in pk and "#define ZKP_LAZY ZKP_MILLER_LAZY" in pk and "#define ZKP_CONVERGED 1" in pk
    assert "#define ZKP_LOOP_SYNC ZKP_FE_SYNC" in fe and "#define ZKP_CONVERGED 1" in fe and "ZKP_LAZY" not in fe
    assert not re.search(r"#define ZKP_(LAZY|CONVERGED|LOOP_SYNC)\b", kern)
    ms, ml, fs = _define("pairing_kernel.cu", "ZKP_MILLER_SYNC"), _define("pairing_kernel.cu", "ZKP_MILLER_LAZY"), _define("fe_kernel.cu", "ZKP_FE_SYNC")
    return {
        "kernels": ([], 0),
        "pairing": (["-DZKP_CONVERGED", "-DZKP_LOOP_SYNC=%d" % ms, "-DZKP_LAZY=%d" % ml], ml),
        "fe": (["-DZKP_CONVERGED", "-DZKP_LOOP_SYNC=%d" % fs], 0),
        "lazy7": (["-DZKP_LAZY=7"], 7),
    }


VARIANTS = sorted(define_sets())


def _cached_build(kind, srcs, cmd):
    """build once per distinct source set and command: the .so lands in a per-user temporary directory under a name
    hashed from both, so the suite also runs from a read-only tree and a changed header always rebuilds"""
    h = hashlib.sha256(" ".join(cmd).encode())
    for f in srcs:
        h.update(open(f, "rb").read())
    d = os.path.join(tempfile.gettempdir(), "zkpair-test-builds-%d" % os.getuid())
    os.makedirs(d, mode=0o700, exist_ok=True)
    so = os.path.join(d, "%s-%s.so" % (kind, h.hexdigest()[:20]))
    if not os.path.exists(so):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call(cmd + ["-o", tmp, srcs[0]])
        os.replace(tmp, so)
    return so


def build_harness(name):
    """the device harness (harness.cu) compiled with one define set's flags"""
    from zkvm_pairings_b200 import build
    srcs = [os.path.join(HARNESS_DIR, "harness.cu"), os.path.join(HARNESS_DIR, "bodies.cuh")] + HEADERS
    cmd = [build.nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
           "-shared"] + define_sets()[name][0]
    return _cached_build("harness-" + name, srcs, cmd)


def build_sim(lazy):
    """the dev simulation (sim.cpp, with sim_body) built with -DZKP_LAZY=lazy"""
    srcs = [os.path.join(ROOT, "tests", "host_sim", "sim.cpp"), os.path.join(HARNESS_DIR, "bodies.cuh")] + HEADERS
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-DZKP_LAZY=%d" % lazy]
    return ctypes.CDLL(_cached_build("sim-lazy%d" % lazy, srcs, cmd))


# ---------------------------------------------------------------- marshalling: raw representatives

def pack(vals):
    """flat list of n * 2 * SLOTS ints (element, slot, lane) -> (n, U64) uint64"""
    return np.frombuffer(b"".join(v.to_bytes(48, "little") for v in vals), np.uint64).reshape(-1, U64).copy()


def unpack(a):
    b = a.tobytes()
    return [int.from_bytes(b[48 * k:48 * k + 48], "little") for k in range(len(b) // 48)]


def run_sim(sim, body, vals):
    a = pack(vals)
    out = np.zeros_like(a)
    sim.sim_body(BODY[body], _p(a), _p(out), ctypes.c_size_t(a.shape[0]))
    return out


def run_dev(lib, body, vals):
    a = pack(vals)
    out = np.zeros_like(a)
    assert lib.harness_run(BODY[body], a.shape[0], _p(a), _p(out)) == 0
    return out


def fp_cases(cases):
    """Fp-level cases (tuples of per-slot ints), two per element (even / odd lane) -> flat values"""
    if len(cases) % 2:
        cases = cases + [cases[-1]]
    vals = []
    for e in range(0, len(cases), 2):
        for j in range(SLOTS):
            for lane in (0, 1):
                c = cases[e + lane]
                vals.append(c[j] if j < len(c) else 0)
    return vals


def fp_results(out, ncases):
    """(n, U64) -> per case, the list of its SLOTS output values"""
    v = unpack(out)
    return [[v[(c // 2) * 2 * SLOTS + 2 * j + (c & 1)] for j in range(SLOTS)] for c in range(ncases)]


def split768(t):
    return (t & (R - 1), t >> 384)


# ---------------------------------------------------------------- operand sets at the bounds

def operand_set(bound, inclusive):
    """0, 1, 2^32k - 1, p - 1, p, p + 1, 2p - 1, 2p, 2p + 1, B - 1, B (inclusive bound), and the top word of B minus one
    with all ones below (the longest carry chains)"""
    s = {0, 1, P - 1, P, P + 1, 2 * P - 1, 2 * P, 2 * P + 1, bound - 1}
    s |= {(1 << (32 * k)) - 1 for k in range(1, 13)}
    s.add((((bound >> 352) - 1) << 352) | ((1 << 352) - 1))
    if inclusive:
        s.add(bound)
    return sorted(x for x in s if x < bound or (inclusive and x == bound))


def wide_set(limit):
    """unreduced values below `limit` (exclusive): the limit - 1 itself and the 768-bit analogue of the carry pattern"""
    s = {0, 1, P - 1, P, P * P, R - 1, R, 8 * P * P, 16 * P * P, limit - 1}
    s.add((((limit >> 736) - 1) << 736) | ((1 << 736) - 1))
    return sorted(x for x in s if x < limit)


S2, S4, S8 = operand_set(2 * P, True), operand_set(4 * P, True), operand_set(8 * P, False)
N_RANDOM = 2000


def fp_body_cases(rng):
    """body -> list of operand tuples.  All pairs of the fixed sets, plus seeded random tuples in the box."""
    r2 = lambda: rng.randint(0, 2 * P)
    r4 = lambda: rng.randint(0, 4 * P)
    cases = {}
    cases["mont_mul"] = [(a, b) for a in S4 for b in S2] + [(a, b) for a in S2 for b in S4] + \
        [(r4(), r2()) for _ in range(N_RANDOM)] + [(r2(), r4()) for _ in range(N_RANDOM)]
    cases["mont_mul2"] = [t for a in S2 for b in S2 for t in ((a, b, a, b), (a, b, b, a))] + \
        [(r2(), r2(), r2(), r2()) for _ in range(N_RANDOM)]
    cases["mul_wide"] = [(a, b) for a in S4 for b in S2] + [(r4(), r2()) for _ in range(N_RANDOM)]
    cases["mul_wide2"] = [(a, b, a, b) for a in S4 for b in S2] + [(a, b, b, a) for a in S2 for b in S2] + \
        [(r4(), r2(), r4(), r2()) for _ in range(N_RANDOM)]
    t29, t68 = wide_set(29 * P * P), wide_set(68 * P * P)
    w29 = t29 + [rng.randrange(29 * P * P) for _ in range(N_RANDOM)]
    w68 = t68 + [rng.randrange(68 * P * P) for _ in range(N_RANDOM)]
    cases["mont_redc"] = [split768(t) for t in w29 + w68]
    cases["fp2_redc0"] = [split768(t) for t in w29]
    cases["fp2_redc1"] = [split768(t) for t in w68]
    cases["fp_correct"] = [(a,) for a in S4] + [(r4(),) for _ in range(N_RANDOM)]
    cases["fp_correct8"] = [(a,) for a in S8] + [(rng.randrange(8 * P),) for _ in range(N_RANDOM)]
    cases["fp_add"] = [(a, b) for a in S2 for b in S2] + [(r2(), r2()) for _ in range(N_RANDOM)]
    cases["fp_sub"] = list(cases["fp_add"])
    cases["fp_neg"] = [(a,) for a in S2] + [(r2(),) for _ in range(N_RANDOM)]
    ws = [0, 1, W768, R - 1, R, 68 * P * P - 1, 96 * P * P, (W768 >> 32) << 32] + [rng.getrandbits(768) for _ in range(8)]
    cases["fpw_mul_nr"] = [split768(x) + split768(y) for x in ws for y in ws]   # (X lo, X hi, Y lo, Y hi)
    z = sorted(set(S2 + [P - 1, P + 1, 2 * P - 1]))
    cases["fp_to_words"] = [(a,) for a in z] + [(r2(),) for _ in range(N_RANDOM)]
    cases["fp_is_zero"] = list(cases["fp_to_words"])
    cases["fp_inv"] = [(a,) for a in INV_EDGE_REPS + S2] + [(r2(),) for _ in range(200)]
    return cases


# representatives whose inversion runs the binary GCD's full 2 * 381 - 1 iterations (and the neighbours)
INV_EDGE_REPS = [1 << 380, 3 << 379, (1 << 380) + P, (3 << 379) + P, 1 << 379, 0, P, 2 * P]


def gcd_trace(y, m=P):
    """tower.cuh fp_inv's loop (fr.cuh fr_inv's for m = r) for y = the representative reduced mod m: (iterations until
    a = 0, the iteration of the last swap).  v, the result, changes only in swap iterations, so the loop count must
    reach the last swap."""
    a, b, it, last = y, m, 0, 0
    while a:
        it += 1
        if a & 1:
            if a < b:
                a, b, last = b - a, a, it
            else:
                a = a - b
        a >>= 1
    return it, last


def loaded_rep(c):
    """the representative fp_from_words produces for canonical c: REDC(c * R^2 mod p) without its final correction"""
    r2 = R * R % P
    t = c * r2
    m = (t * (-pow(P, -1, R))) % R
    return (t + m * P) >> 384


def check_fp_body(name, case, res):
    """the reference of one Fp-level case; raises AssertionError with the case on a mismatch"""
    msg = (name, [hex(x) for x in case], [hex(x) for x in res[:2]])
    o = res[0]
    if name == "mont_mul":
        assert o < 2 * P and o % P == case[0] * case[1] * RINV % P, msg
    elif name == "mont_mul2":
        assert o < 2 * P and o % P == (case[0] * case[1] + case[2] * case[3]) * RINV % P, msg
    elif name == "mul_wide":
        assert o | (res[1] << 384) == case[0] * case[1], msg
    elif name == "mul_wide2":
        assert o | (res[1] << 384) == case[0] * case[1] + case[2] * case[3], msg
    elif name in ("mont_redc", "fp2_redc0", "fp2_redc1"):
        t = case[0] | (case[1] << 384)
        assert o % P == t * RINV % P, msg
        if name == "mont_redc":
            assert o * R < t + (P + 1) * R, msg                      # < T / 2^384 + p + 1
            assert o < (4 * P if t < 29 * P * P else 8 * P), msg     # what fp2_redc<0> / <1> rely on
        else:
            assert o <= 2 * P, msg
    elif name in ("fp_correct", "fp_correct8"):
        assert o <= 2 * P and o % P == case[0] % P, msg
    elif name == "fp_add":
        assert o <= 2 * P and o % P == (case[0] + case[1]) % P, msg
    elif name == "fp_sub":
        assert o <= 2 * P and o % P == (case[0] - case[1]) % P, msg
    elif name == "fp_neg":
        assert o <= 2 * P and o % P == -case[0] % P, msg
    elif name == "fp_to_words":
        assert o == case[0] * RINV % P, msg
    elif name == "fp_is_zero":
        assert o == (1 if case[0] % P == 0 else 0), msg
    elif name == "fp_inv":
        x = case[0] % P
        assert o <= 2 * P and o % P == (0 if x == 0 else R * R * pow(x, -1, P) % P), msg
    else:
        raise KeyError(name)


def fpw_mul_nr_check(case_even, case_odd, res_even, res_odd):
    x = case_even[0] | (case_even[1] << 384)
    y = case_odd[0] | (case_odd[1] << 384)
    assert res_even[0] | (res_even[1] << 384) == (x - y) & W768
    assert res_odd[0] | (res_odd[1] << 384) == (x + y) & W768


def fpw_mul_nr_cases(cases):
    """the lane pair holds (X, Y): the even lane's case is X, the odd lane's Y"""
    flat = []
    for c in cases:
        flat += [c[:2], c[2:]]
    return flat


def batch_inv_cases(rng):
    """runs of 1, 7 and 16 values with zero representatives (0, p, 2p) inside; in every run but the random ones the
    product of the nonzero values is 3/32, so the one inversion inside sees the internal value 3 * 2^379"""
    runs = {1: [[1 << 380], [3 << 379], [(3 << 379) + P], [0], [P], [2 * P], [rng.randint(1, 2 * P)]]}
    for n, zeros in ((7, (0, 3, 6)), (16, (1, 5, 9, 15))):
        runs[n] = []
        for variant in range(6):
            vals, zero_reps = [], [0, P, 2 * P]
            for i in range(n):
                vals.append(zero_reps[(i + variant) % 3] if (i in zeros and variant < 5) else rng.randint(1, P - 1) + (P if rng.random() < 0.5 else 0))
            if variant < 5:                       # make the product of the nonzero values exactly 3/32
                nz = [i for i in range(n) if vals[i] % P]
                q = 1
                for i in nz[:-1]:
                    q = q * vals[i] * RINV % P
                last = 3 * pow(32 * q, -1, P) % P  # canonical value of the last nonzero element
                vals[nz[-1]] = last * R % P + (P if variant & 1 else 0)
            runs[n].append(vals)
    return runs


def batch_inv_product_rep(vals):
    """the value acc that fp_batch_inv hands to fp_inv, reduced mod p: (prod of the nonzero X_i) R"""
    q = 1
    for v in vals:
        if v % P:
            q = q * v * RINV % P
    return q * R % P


# ---------------------------------------------------------------- tower bodies at the vertices

# body -> (Fp2 operand slots, C-oracle op or None, Fp2 result slots)
TOWER = {
    "fp2_mul": (2, "fp2_mul", 1), "fp2_sqr": (1, "fp2_sqr", 1), "fp2_mul_nr": (1, "fp2_mul_nr", 1), "fp2_inv": (1, "fp2_inv", 1),
    "fp6_mul": (6, "fp6_mul", 3), "fp6_sqr": (3, "fp6_sqr", 3), "fp6_mul_by_1": (4, "fp6_mul_by_1", 3),
    "fp6_mul_by_01": (5, "fp6_mul_by_01", 3), "fp6_mul_sums": (6, None, 3), "fp4_square": (2, None, 2),
    "fp12_mul": (12, "fp12_mul", 6), "fp12_sqr": (6, "fp12_sqr", 6), "fp12_sqr_inplace": (6, "fp12_sqr", 6),
    "fp12_mul_by_014": (9, "fp12_mul_by_014", 6), "fp12_mul_by_014_inplace": (9, "fp12_mul_by_014", 6),
    "fp12_cyc_sqr": (6, "fp12_cyc_sqr", 6), "fp12_inv": (6, "fp12_inv", 6),
}
SAMPLED = 1 << 14      # corners per body whose box has more vertices than EXHAUSTIVE
EXHAUSTIVE = 1 << 12


def vertex_inputs(name, rng, limit=None):
    """flat values of the corner inputs of a tower body, and the count / kind of the coverage.  Every Fp slot is
    d or 2p - d, d < 2^20 (vertex = bit of the combination); boxes with at most 2^12 vertices run all of them twice (d = 0
    and random d), larger ones SAMPLED seeded combinations (every fourth with d = 0).  Fp2-level bodies add the class
    where every slot is d, p - d, p + d or 2p - d (zero representatives included)."""
    k = TOWER[name][0]
    nf = 2 * k
    if 1 << nf <= EXHAUSTIVE:
        combos = [(c, False) for c in range(1 << nf)] + [(c, True) for c in range(1 << nf)]
        kind = "exhaustive"
    else:
        combos = [(rng.getrandbits(nf), i % 4 != 0) for i in range(SAMPLED)]
        kind = "sampled"
    rows = []
    for c, rand_d in combos:
        row = []
        for s in range(nf):
            d = rng.getrandbits(20) if rand_d else 0
            row.append(2 * P - d if (c >> s) & 1 else d)
        rows.append(row)
    if k <= 2:
        for _ in range(4 ** nf if 4 ** nf <= 256 else 256):
            row = []
            for s in range(nf):
                d = rng.getrandbits(20) if rng.random() < 0.75 else 0
                row.append(rng.choice((d, P - d, P + d, 2 * P - d)))
            rows.append(row)
    if limit is not None:
        rows = rows[:limit]
    vals = []
    for row in rows:                # slot s // 2, lane s % 2 (c0 in the even lane, c1 in the odd lane)
        vals += row + [0] * (2 * SLOTS - nf)
    return vals, len(rows), kind


def canon(v):
    return v * RINV % P


def canon_matrix(vals, n, first, count):
    """canonical u64 matrix (n, 12 * count) of Fp2 slots first .. first + count - 1"""
    rows = []
    for e in range(n):
        base = e * 2 * SLOTS
        rows += [canon(vals[base + 2 * first + i]) for i in range(2 * count)]
    return util.fp_arr(rows).reshape(n, 12 * count)


def tower_expected(coracle, name, vals, n):
    k, op, nr = TOWER[name]
    if name == "fp4_square":
        exp = []
        for e in range(n):
            a = (canon(vals[e * 2 * SLOTS]), canon(vals[e * 2 * SLOTS + 1]))
            b = (canon(vals[e * 2 * SLOTS + 2]), canon(vals[e * 2 * SLOTS + 3]))
            c0 = pyref.fp2_add(pyref.fp2_mul(a, a), pyref.fp2_mul_by_nonresidue(pyref.fp2_mul(b, b)))
            c1 = pyref.fp2_add(pyref.fp2_mul(a, b), pyref.fp2_mul(a, b))
            exp += [c0[0], c0[1], c1[0], c1[1]]
        return util.fp_arr(exp).reshape(n, 24)
    if name == "fp6_mul_sums":        # (a0 + a1) (a0.c0 + xi a1.c2, a0.c1 + a1.c0, a0.c2 + a1.c1)
        s, b = [], []
        for e in range(n):
            f = [(canon(vals[e * 2 * SLOTS + 2 * j]), canon(vals[e * 2 * SLOTS + 2 * j + 1])) for j in range(6)]
            a0, a1 = f[:3], f[3:]
            for j in range(3):
                s += list(pyref.fp2_add(a0[j], a1[j]))
            b += list(pyref.fp2_add(a0[0], pyref.fp2_mul_by_nonresidue(a1[2]))) + list(pyref.fp2_add(a0[1], a1[0])) + \
                list(pyref.fp2_add(a0[2], a1[1]))
        return coracle.tower_op("fp6_mul", util.fp_arr(s).reshape(n, 36), util.fp_arr(b).reshape(n, 36))
    na = {"fp6_mul_by_1": 3, "fp6_mul_by_01": 3, "fp12_mul_by_014": 6, "fp12_mul_by_014_inplace": 6}.get(name, nr)
    a = canon_matrix(vals, n, 0, na)
    b = canon_matrix(vals, n, na, k - na) if k > na else None
    return coracle.tower_op(op, a, b)


def check_tower(name, out, expected, n):
    nr = TOWER[name][2]
    raw = unpack(out)
    got = []
    for e in range(n):
        for i in range(2 * nr):
            v = raw[e * 2 * SLOTS + i]
            assert v <= 2 * P, (name, e, i, hex(v))            # every output coefficient 2p-redundant
            got.append(canon(v))
    got = util.fp_arr(got).reshape(n, 12 * nr)
    bad = np.nonzero(~np.all(got == expected, axis=1))[0]
    assert len(bad) == 0, (name, "mismatching corners", bad[:8].tolist(), len(bad))


# ---------------------------------------------------------------- CPU: models, builds, simulation

def test_gcd_iteration_count_is_tight():
    """The Python model of fp_inv's loop: the fixed count 2 * 381 - 1 is reached, and the inputs the tests below use
    hit it through the C ABI (canonical 1/16 and 3/32 load as 2^380 and 3 * 2^379; the norm of (1/4, 0) is 1/16)."""
    assert 2 * 381 - 1 == 761
    assert gcd_trace(1 << 380) == (761, 381) and gcd_trace(3 << 379) == (761, 760) and gcd_trace(1 << 379) == (760, 380)
    # the last iteration takes a from b to 0 and never swaps, so 760 iterations would give the same results; 3 * 2^379
    # swaps in iteration 760, so one iteration fewer than that gives a wrong inverse
    rng = random.Random(7)
    assert max(gcd_trace(rng.randrange(1, P))[1] for _ in range(2000)) < 700
    inv16, c3_32 = pow(16, -1, P), 3 * pow(32, -1, P) % P
    assert loaded_rep(inv16) == 1 << 380 and loaded_rep(c3_32) == 3 << 379
    quarter = pow(4, -1, P)
    assert (quarter * quarter) * R % P == 1 << 380           # the internal value of the norm of (1/4, 0) and (0, 1/4)
    rows, _ = abi_fp2_inverse_rows()
    a, b = util.arr_fp(rows[2:3].reshape(-1, 6))
    assert (a * a + b * b) * R % P == 3 << 379               # ... and of the third fp2_inv row
    for run in batch_inv_cases(random.Random(3))[7][:5] + batch_inv_cases(random.Random(3))[16][:5]:
        assert gcd_trace(batch_inv_product_rep(run)) == (761, 760)


def test_loaded_representatives_stay_far_below_2p():
    """Why the ABI cannot test the operand bounds: fp_from_words returns (c R^2 + m p) / 2^384 < p (1 + p / 2^384)."""
    bound = P + P * P // R + 1
    assert bound < 1.102 * P
    rng = random.Random(11)
    for c in [P - k for k in range(1, 2001)] + list(range(2000)) + [rng.randrange(P) for _ in range(2000)]:
        rep = loaded_rep(c)
        assert rep < bound and rep % P == c * R % P


@pytest.mark.parametrize("variant", VARIANTS)
def test_harness_builds_for_every_define_set(variant):
    so = build_harness(variant)
    assert os.path.getsize(so) > 0
    assert b"sm_100a" in open(so, "rb").read()


def test_sim_body_bound_cases():
    """Fp-level bodies on the simulation (which also asserts the operand bounds inside): every case's reference."""
    sim = build_sim(0)
    cases = fp_body_cases(random.Random(0xB0))
    for name, cs in cases.items():
        if name == "fpw_mul_nr":
            flat = fpw_mul_nr_cases(cs)
            res = fp_results(run_sim(sim, name, fp_cases(flat)), len(flat))
            for i in range(0, len(flat), 2):
                fpw_mul_nr_check(flat[i], flat[i + 1], res[i], res[i + 1])
            continue
        res = fp_results(run_sim(sim, name, fp_cases(cs)), len(cs))
        for c, r in zip(cs, res):
            check_fp_body(name, c, r)


def check_batch_inv(runner, lib):
    for n, runs in batch_inv_cases(random.Random(0xBA7)).items():
        body = "batch_inv%d" % n
        res = fp_results(runner(lib, body, fp_cases(runs)), len(runs))
        for vals, out in zip(runs, res):
            for v, o in zip(vals, out[:n]):
                assert o <= 2 * P, (n, hex(v), hex(o))
                assert o % P == (0 if v % P == 0 else R * R * pow(v, -1, P) % P), (n, hex(v), hex(o))


def test_sim_inversions_at_the_iteration_limit():
    sim = build_sim(0)
    cs = [(x,) for x in INV_EDGE_REPS]
    for c, r in zip(cs, fp_results(run_sim(sim, "fp_inv", fp_cases(cs)), len(cs))):
        check_fp_body("fp_inv", c, r)
    check_batch_inv(run_sim, sim)


def test_sim_abi_inversion_at_the_iteration_limit(coracle):
    """zkp_tower_op_batch's fp_inv / fp2_inv rows whose inversion needs all 761 iterations, in the simulation."""
    sim = build_sim(0)
    from zkvm_pairings_b200 import TOWER_OPS
    a, exp = abi_inverse_rows()
    out, st = np.zeros_like(a), np.zeros(a.shape[0], np.uint8)
    sim.sim_tower_op(TOWER_OPS["fp_inv"], _p(a), None, _p(out), _p(st), ctypes.c_size_t(a.shape[0]))
    assert util.arr_fp(out) == exp and not st.any()
    a2, exp2 = abi_fp2_inverse_rows()
    out2, st2 = np.zeros_like(a2), np.zeros(a2.shape[0], np.uint8)
    sim.sim_tower_op(TOWER_OPS["fp2_inv"], _p(a2), None, _p(out2), _p(st2), ctypes.c_size_t(a2.shape[0]))
    assert util.arr_fp(out2) == exp2 and not st2.any()
    assert np.array_equal(out2, coracle.tower_op("fp2_inv", a2))


def abi_inverse_rows():
    inv16, c3_32 = pow(16, -1, P), 3 * pow(32, -1, P) % P
    return util.fp_arr([inv16, c3_32]).reshape(-1, 6), [16, 32 * pow(3, -1, P) % P]


def abi_fp2_inverse_rows():
    """(1/4, 0) and (0, 1/4), norm 1/16; (a, b) with norm a^2 + b^2 = 3/32.  Inverse: (a, -b) / norm."""
    q, n3 = pow(4, -1, P), 3 * pow(32, -1, P) % P
    a = 1
    while pow((n3 - a * a) % P, (P - 1) // 2, P) != 1:
        a += 1
    b = pow((n3 - a * a) % P, (P + 1) // 4, P)
    assert (a * a + b * b) % P == n3
    ni = pow(n3, -1, P)
    return util.fp_arr([q, 0, 0, q, a, b]).reshape(-1, 12), [4, 0, 0, P - 4, a * ni % P, -b * ni % P]


# lanes' work in the simulation is slow (two host threads per lane pair): the CPU tests take a prefix of every body's
# corner inputs; the GPU tests run all of them on the device
SIM_CORNERS = 256


@pytest.mark.parametrize("lazy", sorted({v[1] for v in define_sets().values()}))
def test_sim_tower_bodies_at_the_vertices(coracle, lazy):
    """Tower bodies of the simulation with every Fp slot at a corner of [0, 2p] (a prefix of the device's inputs),
    against the C oracle, for every ZKP_LAZY a define set uses."""
    sim = build_sim(lazy)
    for name in TOWER:
        vals, n, _ = vertex_inputs(name, random.Random(zlib.crc32(name.encode())), limit=SIM_CORNERS)
        check_tower(name, run_sim(sim, name, vals), tower_expected(coracle, name, vals, n), n)


# ---------------------------------------------------------------- Fr bodies (fr.cuh, the byte paths of blob.cuh / kzg_prove.cuh)

FR = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
FR_MONT = 1 << 256
FR_MINV = pow(FR_MONT, -1, FR)
W256 = FR_MONT - 1

# internal values whose inversion runs fr_inv's full 2 * 255 - 1 iterations (canonical 3/8 and 1/4), and neighbours
FR_INV_EDGE = [3 << 253, 1 << 254, 1 << 253, (3 << 253) - 1, (3 << 253) + 1, (1 << 254) - 1, (1 << 254) + 1,
               (1 << 253) - 1, (1 << 253) + 1, 0, 1, FR - 1]


def fr_operand_set():
    """0, 1, 2, r - 2, r - 1, 2^32k - 1 below r, and the top word of r minus one with all ones below"""
    s = {0, 1, 2, FR - 2, FR - 1, (((FR >> 224) - 1) << 224) | ((1 << 224) - 1)}
    s |= {(1 << (32 * k)) - 1 for k in range(1, 8)}
    return sorted(x for x in s if x < FR)


def fr_body_cases(rng):
    """body -> list of operand tuples: the corners and seeded random values of each body's input range"""
    s = fr_operand_set()
    rr = lambda: rng.randrange(FR)
    wide = s + [FR, FR + 1, 2 * FR - 2, 2 * FR - 1, W256, 1 << 255, W256 - (1 << 32)]
    pairs = [(a, b) for a in s for b in s]
    pairs += [(a, FR - a) for a in s if a] + [(FR - 1, FR - 1)]          # sums of exactly r and 2r - 2
    pairs += [(a, FR - a) for a in (rr() for _ in range(50))] + [(a, a) for a in (rr() for _ in range(50))]
    pairs += [(rr(), rr()) for _ in range(N_RANDOM)]
    cases = {"fr_add": pairs, "fr_sub": list(pairs), "fr_mul": list(pairs)}
    cases["fr_reduce_once"] = [(a,) for a in sorted(set(s + [FR + a for a in s] + [2 * FR - 1]))] + \
        [(rng.randrange(2 * FR),) for _ in range(N_RANDOM)]
    cases["fr_geq_r"] = [(a,) for a in wide] + [(rng.getrandbits(256),) for _ in range(N_RANDOM)]
    cases["blob_element"] = list(cases["fr_geq_r"])
    cases["fr_to_mont"] = [(a,) for a in s] + [(rr(),) for _ in range(N_RANDOM)]
    cases["fr_from_mont"] = list(cases["fr_to_mont"])
    cases["fr_inv"] = [(a,) for a in FR_INV_EDGE + s] + [(rr(),) for _ in range(200)]
    cases["store_be32"] = [(a,) for a in s] + [(rr(),) for _ in range(N_RANDOM)]
    return cases


def check_fr_body(name, case, res):
    """the reference of one Fr-level case; the words above the low 256 bits of every result must stay zero"""
    a = case[0]
    o = res[0]
    msg = (name, [hex(x) for x in case], [hex(x) for x in res[:2]])
    assert o >> 256 == 0 and res[1] >> 256 == 0, msg
    if name == "fr_add":
        assert o == (a + case[1]) % FR, msg
    elif name == "fr_sub":
        assert o == (a - case[1]) % FR, msg
    elif name == "fr_mul":
        assert o == a * case[1] * FR_MINV % FR, msg
    elif name == "fr_reduce_once":
        assert o == (a - FR if a >= FR else a), msg
    elif name == "fr_geq_r":
        assert o == (1 if a >= FR else 0), msg
    elif name == "fr_to_mont":
        assert o == a * FR_MONT % FR, msg
    elif name == "fr_from_mont":
        assert o == a * FR_MINV % FR, msg
    elif name == "fr_inv":
        assert o == (0 if a == 0 else FR_MONT * FR_MONT * pow(a, -1, FR) % FR), msg
    elif name == "blob_element":
        assert (o, res[1]) == ((a, 1) if a < FR else (0, 0)), msg
    elif name == "store_be32":
        assert o.to_bytes(48, "little")[:32] == a.to_bytes(32, "big"), msg
    else:
        raise KeyError(name)


def check_fr_bodies(runner, lib):
    """every Fr body's cases through runner (run_sim / run_dev) against the references; returns {body: (values, out)}"""
    done = {}
    for name, cs in fr_body_cases(random.Random(0xF4)).items():
        vals = fp_cases(cs)
        out = runner(lib, name, vals)
        for c, r in zip(cs, fp_results(out, len(cs))):
            check_fr_body(name, c, r)
        done[name] = (vals, out)
    return done


def test_fr_inv_iteration_count_is_tight():
    """The Python model of fr_inv's loop: the fixed count 2 * 255 - 1 is reached, 3 * 2^253 swaps in its last
    iteration but one, and canonical 3/8 and 1/4 load as 3 * 2^253 and 2^254 (RF = 2^256); random inputs stop
    swapping long before, so only the edge values notice a shorter loop."""
    assert 2 * 255 - 1 == 509
    assert gcd_trace(3 << 253, FR) == (509, 508) and gcd_trace(1 << 254, FR) == (509, 255)
    assert 3 * pow(8, -1, FR) * FR_MONT % FR == 3 << 253 and pow(4, -1, FR) * FR_MONT % FR == 1 << 254
    rng = random.Random(0x1F4)
    assert max(gcd_trace(rng.randrange(1, FR), FR)[1] for _ in range(2000)) < 450


def test_sim_fr_bodies_at_the_bounds():
    """Fr bodies of the simulation (which asserts the operand bound of every sum, difference and product) at the
    corners of their input ranges: Python big-int references."""
    check_fr_bodies(run_sim, build_sim(0))


# ---------------------------------------------------------------- GPU: the device builds

@pytest.fixture(scope="module", params=VARIANTS)
def device_variant(request):
    lib = ctypes.CDLL(build_harness(request.param))
    lib.harness_run.restype = ctypes.c_int
    lib.harness_run.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    return request.param, lib, build_sim(define_sets()[request.param][1])


SIM_COMPARE = 512      # elements per body the simulation recomputes for the raw comparison with the device


@pytest.mark.gpu
def test_device_fp_bodies_at_the_bounds(device_variant):
    """Fp-level bodies on the device at the operand bounds: Python big-int references, and raw output words equal to
    the simulation's (a correction step that differs would hide behind congruence)."""
    name_v, lib, sim = device_variant
    cases = fp_body_cases(random.Random(0xB0))
    for name, cs in cases.items():
        flat = fpw_mul_nr_cases(cs) if name == "fpw_mul_nr" else cs
        vals = fp_cases(flat)
        out = run_dev(lib, name, vals)
        res = fp_results(out, len(flat))
        if name == "fpw_mul_nr":
            for i in range(0, len(flat), 2):
                fpw_mul_nr_check(flat[i], flat[i + 1], res[i], res[i + 1])
        else:
            for c, r in zip(flat, res):
                check_fp_body(name, c, r)
        idx, sub = spread(vals, out.shape[0], SIM_COMPARE)
        assert np.array_equal(out[idx], run_sim(sim, name, sub)), (name_v, name)
    check_batch_inv(run_dev, lib)
    for n, runs in batch_inv_cases(random.Random(0xBA7)).items():
        vals = fp_cases(runs)
        assert np.array_equal(run_dev(lib, "batch_inv%d" % n, vals), run_sim(sim, "batch_inv%d" % n, vals)), (name_v, n)


_TOWER_CASES = {}


def tower_case(coracle, name):
    """the corner inputs of a body and their expected results, shared by the four device builds"""
    if name not in _TOWER_CASES:
        vals, n, _ = vertex_inputs(name, random.Random(zlib.crc32(name.encode())))
        _TOWER_CASES[name] = (vals, n, tower_expected(coracle, name, vals, n))
    return _TOWER_CASES[name]


def spread(vals, n, m):
    """m elements spread evenly over the n of a flat value list: (their indices, their values)"""
    idx = np.unique(np.linspace(0, n - 1, min(n, m)).astype(int))
    return idx, [v for i in idx for v in vals[i * 2 * SLOTS:(i + 1) * 2 * SLOTS]]


@pytest.mark.gpu
def test_device_tower_bodies_at_the_vertices(device_variant, coracle):
    """Tower bodies on the device with every Fp slot at a corner of [0, 2p]: canonical results equal the C oracle's
    (pyref formulas for fp4_square, fp6_mul for fp6_mul_sums), every output coefficient <= 2p, and the raw words of
    SIM_COMPARE corners spread over the inputs equal the simulation's with the same ZKP_LAZY."""
    name_v, lib, sim = device_variant
    for name in TOWER:
        vals, n, expected = tower_case(coracle, name)
        out = run_dev(lib, name, vals)
        check_tower(name, out, expected, n)
        idx, sub = spread(vals, n, SIM_COMPARE)
        assert np.array_equal(out[idx], run_sim(sim, name, sub)), (name_v, name)


@pytest.mark.gpu
def test_device_fr_bodies_at_the_bounds(device_variant):
    """Fr bodies on the device at the corners of their input ranges: Python big-int references, and every raw output
    word equal to the simulation's (blob_element and store_be32 take the device's uint4 / __byte_perm paths there)."""
    name_v, lib, sim = device_variant
    for name, (vals, out) in check_fr_bodies(run_dev, lib).items():
        assert np.array_equal(out, run_sim(sim, name, vals)), (name_v, name)


# ---------------------------------------------------------------- GPU: the C ABI at its reachable edges

@pytest.mark.gpu
def test_abi_inversion_at_the_iteration_limit(engine, coracle):
    a, exp = abi_inverse_rows()
    out, st = engine.tower_op("fp_inv", a, return_status=True)
    assert util.arr_fp(out) == exp and not st.any()
    assert np.array_equal(out, coracle.tower_op("fp_inv", a))
    a2, exp2 = abi_fp2_inverse_rows()
    out2, st2 = engine.tower_op("fp2_inv", a2, return_status=True)
    assert util.arr_fp(out2) == exp2 and not st2.any()
    assert np.array_equal(out2, coracle.tower_op("fp2_inv", a2))


def _checks_with_infinities(coracle, k, nchk, seed):
    g1, i1, g2, i2 = util.oracle_points(coracle, seed, 0, nchk * k)
    i1[0] = 1                              # first pair of check 0
    i2[2 * k - 1] = 1                      # last pair of check 1
    i1[2 * k: 3 * k: 2] = 1                # every pair of check 2 (alternating sides)
    i2[2 * k + 1: 3 * k: 2] = 1
    return g1, i1, g2, i2


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(1, 9))
def test_multi_pairing_every_check_width(engine, coracle, pyref, k):
    """pairs_per_check 1..8 (6 and 7 run the 8-wide kernel with idle pair slots), ragged check counts, points at
    infinity in the first pair, the last pair and every pair of a check."""
    nchk = 5 + 2 * k
    g1, i1, g2, i2 = _checks_with_infinities(coracle, k, nchk, 0x900 + k)
    out, one = engine.multi_pairing_batch(g1, g2, k, i1, i2)
    exp, eone = coracle.multi_pairing_batch(g1, i1, g2, i2, k)
    assert np.array_equal(out, exp) and np.array_equal(one, eone)
    assert one[2] == 1 and util.arr_to_fp12(out[2]) == pyref.FP12_ONE
    mm = engine.multi_miller_loop_batch(g1, g2, k, i1, i2)
    assert np.array_equal(mm, coracle.multi_miller_batch(g1, i1, g2, i2, k))


@pytest.mark.gpu
@pytest.mark.parametrize("k,kf", [(8, 1), (8, 7), (8, 8), (6, 3), (7, 7), (5, 0), (1, 1)])
def test_prepared_tables_at_more_widths(engine, coracle, k, kf):
    """multi_pairing_prepared_batch with the last kf pairs from shared tables, one of them flagged as the point at
    infinity: equal to the unprepared call and to the oracle."""
    nc = 9
    g1, i1, g2all, _ = util.oracle_points(coracle, 0x7AB + 16 * k + kf, 0, nc * k)
    i1[k - 1] = 1
    fixed = g2all[:kf].copy()
    g2 = g2all.reshape(nc, k, 24).copy()
    g2[:, k - kf:, :] = fixed
    ti = np.zeros(kf, np.uint8)
    if kf:
        ti[kf // 2] = 1
    i2 = np.zeros((nc, k), np.uint8)
    i2[:, k - kf:] = ti
    tab = engine.g2_prepare_batch(fixed) if kf else np.zeros((0, engine.G2_PREPARED_U64), np.uint64)
    var = np.ascontiguousarray(g2[:, :k - kf, :]).reshape(-1, 24) if kf < k else None
    gt, one = engine.multi_pairing_prepared_batch(g1, var, k, tab, g1_inf=i1, tables_inf=ti if kf else None)
    ref, ref_one = engine.multi_pairing_batch(g1, g2.reshape(-1, 24), k, i1, i2.reshape(-1))
    assert np.array_equal(gt, ref) and np.array_equal(one, ref_one)
    exp, eone = coracle.multi_pairing_batch(g1, i1, g2.reshape(-1, 24), i2.reshape(-1), k)
    assert np.array_equal(gt, exp) and np.array_equal(one, eone)
