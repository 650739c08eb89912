"""Points with small-order components: the subgroup checks, the group kernels and the Groth16 / KZG front ends on
P + T with T of small order, judged by the definition of the subgroups, [r]P = O.

The pairing cannot tell P + T from P when T has small order in G1 (e(T, Q) = 1), so the subgroup checks are what
keeps such a point from a valid verdict.  The expected values here come from an affine group law on Python integers
(no endomorphism, no Montgomery form), not from the formulas the kernels and the oracles share (-[x^2]P == (beta x, y),
psi(Q) == -[|x|]Q).  Small-order bases also drive the double-and-add ladder through every branch of its mixed
addition (acc == Q, acc == -Q, acc at infinity), which subgroup points reach only at special scalars."""
import ctypes
import functools
import os
import random
import subprocess

import numpy as np
import pytest

import pyref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P, R = pyref.P, pyref.R_ORDER
BLS_X = -pyref.X                        # the curve parameter x = -0xd201000000010000
M64 = (1 << 64) - 1
H1 = (BLS_X - 1) ** 2 // 3              # #E(Fp) = H1 r
H2 = (BLS_X ** 8 - 4 * BLS_X ** 7 + 5 * BLS_X ** 6 - 4 * BLS_X ** 4 + 6 * BLS_X ** 3 - 4 * BLS_X ** 2 - 4 * BLS_X + 13) // 9   # #E'(Fp2) = H2 r
TILED = (1 << 18) + 37                  # one host pipeline chunk (2^18 rows) and a ragged remainder


# ---------------------------------------------------------------- reference: affine group law on Python integers

class Fp:
    zero, one, b = 0, 1, 4

    @staticmethod
    def add(a, b):
        return (a + b) % P

    @staticmethod
    def sub(a, b):
        return (a - b) % P

    @staticmethod
    def mul(a, b):
        return a * b % P

    @staticmethod
    def inv(a):
        return pow(a, -1, P)

    @staticmethod
    def small(k):
        return k % P

    @staticmethod
    def random(rng):
        return rng.randrange(P)

    @staticmethod
    def sqrt(a):                        # p = 3 mod 4
        s = pow(a, (P + 1) // 4, P)
        return s if s * s % P == a % P else None

    @staticmethod
    def limbs(a):
        return [(a >> (64 * k)) & M64 for k in range(6)]


class Fp2:
    """Fp[u] / (u^2 + 1), elements (c0, c1)."""
    zero, one, b = (0, 0), (1, 0), (4, 4)

    @staticmethod
    def add(a, b):
        return ((a[0] + b[0]) % P, (a[1] + b[1]) % P)

    @staticmethod
    def sub(a, b):
        return ((a[0] - b[0]) % P, (a[1] - b[1]) % P)

    @staticmethod
    def mul(a, b):
        return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)

    @staticmethod
    def inv(a):
        n = pow(a[0] * a[0] + a[1] * a[1], -1, P)
        return (a[0] * n % P, -a[1] * n % P)

    @staticmethod
    def small(k):
        return (k % P, 0)

    @staticmethod
    def random(rng):
        return (rng.randrange(P), rng.randrange(P))

    @staticmethod
    def sqrt(a):
        """A square root of a, or None: the norm's root s gives x0^2 = (a0 +- s) / 2 and x1 = a1 / (2 x0)."""
        if a[1] == 0:
            s = Fp.sqrt(a[0])
            if s is not None:
                return (s, 0)
            s = Fp.sqrt(-a[0] % P)
            return None if s is None else (0, s)
        s = Fp.sqrt(a[0] * a[0] + a[1] * a[1])
        if s is None:
            return None
        for t in (a[0] + s, a[0] - s):
            x0 = Fp.sqrt(t * pow(2, -1, P) % P)
            if x0:
                r = (x0, a[1] * pow(2 * x0, -1, P) % P)
                assert Fp2.mul(r, r) == a
                return r
        return None

    @staticmethod
    def limbs(a):
        return Fp.limbs(a[0]) + Fp.limbs(a[1])


def on_curve(F, a):
    return a is None or F.mul(a[1], a[1]) == F.add(F.mul(F.mul(a[0], a[0]), a[0]), F.b)


def neg(F, a):
    return None if a is None else (a[0], F.sub(F.zero, a[1]))


def add(F, a, b):
    """a + b for curve points; None is the identity."""
    if a is None:
        return b
    if b is None:
        return a
    (x1, y1), (x2, y2) = a, b
    if x1 == x2:
        if F.add(y1, y2) == F.zero:
            return None
        lam = F.mul(F.mul(F.small(3), F.mul(x1, x1)), F.inv(F.add(y1, y1)))
    else:
        lam = F.mul(F.sub(y2, y1), F.inv(F.sub(x2, x1)))
    x3 = F.sub(F.sub(F.mul(lam, lam), x1), x2)
    return (x3, F.sub(F.mul(lam, F.sub(x1, x3)), y1))


def mul(F, a, k):
    """[k]a by double-and-add over every bit of k >= 0."""
    acc = None
    for i in range(k.bit_length() - 1, -1, -1):
        acc = add(F, acc, acc)
        if (k >> i) & 1:
            acc = add(F, acc, a)
    return acc


def in_subgroup(F, a):
    return mul(F, a, R) is None


def add_flag(F, a, b):
    """The flag the group-addition kernels write: bit0 the sum is the identity, bit1 P + (-P) of two finite points."""
    s = add(F, a, b)
    opposite = a is not None and b is not None and a[0] == b[0] and F.add(a[1], b[1]) == F.zero
    return (1 if s is None else 0) | (2 if opposite else 0)


def curve_point(F, rng):
    while True:
        x = F.random(rng)
        y = F.sqrt(F.add(F.mul(F.mul(x, x), x), F.b))
        if y is not None:
            return (x, y)


def point_of_order(F, rng, q):
    """A point of order exactly q (q prime): [#E / q^v]R (q^v the q-part of #E) for random curve points R until it is not
    the identity, then multiplied by q while that is not the identity.  The q-part need not be cyclic (E(Fp) has
    11^2), so [#E / q]R can be the identity for every R."""
    n = (H1 if F is Fp else H2) * R
    while n % q == 0:
        n //= q
    while True:
        t = mul(F, curve_point(F, rng), n)
        if t is not None:
            while mul(F, t, q) is not None:
                t = mul(F, t, q)
            assert on_curve(F, t)
            return t


def enc(F, a):
    """(limbs, infinity flag) in the library's layout; the identity as (0, 1) with the flag."""
    if a is None:
        return np.array(F.limbs(F.zero) + F.limbs(F.one), np.uint64), 1
    return np.array(F.limbs(a[0]) + F.limbs(a[1]), np.uint64), 0


def dec(F, row):
    v = [sum(int(row[6 * i + k]) << (64 * k) for k in range(6)) for i in range(len(row) // 6)]
    return (v[0], v[1]) if F is Fp else ((v[0], v[1]), (v[2], v[3]))


def enc_rows(F, pts):
    e = [enc(F, a) for a in pts]
    return np.stack([x for x, _ in e]), np.array([f for _, f in e], np.uint8)


def fr(vals):
    return np.array([[(v >> (64 * k)) & M64 for k in range(4)] for v in vals], np.uint64).reshape(-1, 4)


G1 = (pyref.G1_X, pyref.G1_Y)
G2 = ((pyref.G2_X0, pyref.G2_X1), (pyref.G2_Y0, pyref.G2_Y1))


# ---------------------------------------------------------------- the points, built once per module

@functools.lru_cache(maxsize=None)
def points():
    """Named points of G1 = E(Fp) and of E'(Fp2), with the order of their small component (1 for subgroup points),
    plus the torsion points, a trapdoor KZG proof and Groth16 proof on which they are used."""
    rng = random.Random(0x7031)
    t3, t11, t10177 = (point_of_order(Fp, rng, q) for q in (3, 11, 10177))
    t13, t23, t2713 = (point_of_order(Fp2, rng, q) for q in (13, 23, 2713))
    p = mul(Fp, G1, rng.randrange(1, R))
    q = mul(Fp2, G2, rng.randrange(1, R))
    tau, z, y, w = (rng.randrange(1, R) for _ in range(4))
    kzg = dict(tau=tau, z=z, y=y, pi=mul(Fp, G1, w), c=mul(Fp, G1, (y + w * (tau - z)) % R), tau_g2=mul(Fp2, G2, tau))
    al, be, ga, de, u0, u1, a, b, x1 = (rng.randrange(1, R) for _ in range(9))
    l = (u0 + x1 * u1) % R
    c = (a * b - al * be - l * ga) * pow(de, -1, R) % R
    g16 = dict(alpha=mul(Fp, G1, al), beta=mul(Fp2, G2, be), gamma=mul(Fp2, G2, ga), delta=mul(Fp2, G2, de),
               ic=[mul(Fp, G1, u0), mul(Fp, G1, u1)], x=[x1], l=mul(Fp, G1, l), a=mul(Fp, G1, a), b=mul(Fp2, G2, b),
               c=mul(Fp, G1, c))
    pt3 = add(Fp, p, t3)
    g1 = [("G1", G1, 1), ("P", p, 1), ("(0,2)", (0, 2), 3), ("(0,p-2)", (0, P - 2), 3), ("T3", t3, 3), ("T11", t11, 11),
          ("T10177", t10177, 10177), ("P+T3", pt3, 3), ("-(P+T3)", neg(Fp, pt3), 3), ("P+T11", add(Fp, p, t11), 11),
          ("-(P+T11)", neg(Fp, add(Fp, p, t11)), 11), ("P+T10177", add(Fp, p, t10177), 10177),
          ("T3+T11", add(Fp, t3, t11), 33), ("kzg.pi+T3", add(Fp, kzg["pi"], t3), 3),
          ("g16.C+T3", add(Fp, g16["c"], t3), 3)]
    g2 = [("G2", G2, 1), ("Q", q, 1), ("T13", t13, 13), ("T23", t23, 23), ("T2713", t2713, 2713), ("Q+T13", add(Fp2, q, t13), 13),
          ("Q+T23", add(Fp2, q, t23), 23), ("-(Q+T23)", neg(Fp2, add(Fp2, q, t23)), 23), ("Q+T2713", add(Fp2, q, t2713), 2713),
          ("tauG2+T13", add(Fp2, kzg["tau_g2"], t13), 13)]
    return dict(g1=g1, g2=g2, t3=t3, t11=t11, t13=t13, t23=t23, p=p, q=q, kzg=kzg, g16=g16)


def scalars_for(q, rng):
    """Scalars for a base whose small component has order q: 1 .. 7 and the multiples of q around q (where the ladder's
    mixed addition meets acc == Q, acc == -Q and restarts from the identity), multiples of r, 2^256 - 1 (2r is the
    largest multiple of r below 2^256), and two 247-bit k with a top part m and a set bit below it where 2m = +-1 mod q:
    the accumulator equals the base or its negative deep in the ladder."""
    ks = list(range(1, 8)) + [q - 1, q, q + 1, 2 * q, 2 * q + 1, R, R + 1, R + 2, 2 * R, (1 << 256) - 1]
    if q > 2:
        for target in (1, q - 1):
            m = rng.getrandbits(170) | (1 << 169)
            m += (target * pow(2, -1, q) - m) % q
            ks.append((m << 76) | (1 << 75) | rng.getrandbits(75))
    return ks


def mul_rows(F):
    """(bases, scalars, names) over the G1 or G2 points with a small component, each crossed with its scalars."""
    rng = random.Random(0x7032 if F is Fp else 0x7033)
    rows = []
    for name, a, q in points()["g1" if F is Fp else "g2"]:
        if q > 1:
            rows += [(name, a, k) for k in scalars_for(q, rng)]
    return rows


def add_rows(F):
    """(name, a, b): T + T, T + (-T), T3 + 2 T3 (= T3 + (-T3)), P + T and T + P, T + P + T, P + (-(P + T))."""
    pts = points()
    if F is Fp:
        p, ts = pts["p"], [("T3", pts["t3"]), ("T11", pts["t11"])]
        t3 = pts["t3"]
        extra = [("T3+2T3", t3, mul(Fp, t3, 2)), ("(0,2)+(0,p-2)", (0, 2), (0, P - 2)), ("(0,2)+(0,2)", (0, 2), (0, 2))]
    else:
        p, ts = pts["q"], [("T13", pts["t13"]), ("T23", pts["t23"])]
        extra = []
    rows = []
    for n, t in ts:
        pt = add(F, p, t)
        rows += [(n + "+" + n, t, t), (n + "-" + n, t, neg(F, t)), ("P+" + n, p, t), (n + "+P", t, p), ("(P+T)+T " + n, pt, t),
                 ("(P+T)+(P+T) " + n, pt, pt), ("P-(P+T) " + n, p, neg(F, pt)), ("(P+T)-(P+T) " + n, pt, neg(F, pt)),
                 ("T+identity " + n, t, None), ("identity+T " + n, None, t)]
    return rows + extra


# ---------------------------------------------------------------- CPU: the reference and the suite's oracle

def test_reference_cofactors_and_orders():
    """#E(Fp) = H1 r and #E'(Fp2) = H2 r with the known factorisations; both within the Hasse bound, annihilating random
    curve points, and the generators in their subgroups."""
    assert (BLS_X - 1) ** 2 % 3 == 0 and H1 == 3 * 11 ** 2 * 10177 ** 2 * 859267 ** 2 * 52437899 ** 2
    assert P + 1 - H1 * R == BLS_X + 1                                       # the trace of Frobenius is x + 1
    small = 13 ** 2 * 23 ** 2 * 2713 * 11953 * 262069
    rest = H2 // small
    assert H2 % small == 0 and rest.bit_length() == 448 and rest % 13 and rest % 23 and H2 % 3
    assert abs(P * P + 1 - H2 * R) <= 2 * P
    rng = random.Random(0x7034)
    for F, n, g in ((Fp, H1 * R, G1), (Fp2, H2 * R, G2)):
        assert on_curve(F, g) and in_subgroup(F, g) and mul(F, g, R - 1) == neg(F, g)
        for _ in range(2):
            a = curve_point(F, rng)
            assert mul(F, a, n) is None and not in_subgroup(F, a)
    assert mul(Fp, (0, 2), 3) is None and mul(Fp, (0, 2), 2) == (0, P - 2)


def test_points_are_what_they_are_named():
    """Every named point is on its curve; subgroup points are killed by r, points with a small component are not, and the
    component's order is q: [r q]P = O and [r]P != O."""
    pts = points()
    for F, key in ((Fp, "g1"), (Fp2, "g2")):
        for name, a, q in pts[key]:
            assert on_curve(F, a), name
            assert in_subgroup(F, a) == (q == 1), name
            if q > 1:
                assert mul(F, a, R * q) is None, name
    kzg, g16 = pts["kzg"], pts["g16"]
    for F, a in ((Fp, kzg["c"]), (Fp, kzg["pi"]), (Fp2, kzg["tau_g2"]), (Fp, g16["a"]), (Fp2, g16["b"]), (Fp, g16["c"])):
        assert in_subgroup(F, a)


def test_pyref_endomorphism_checks_agree_with_the_definition():
    """The suite's oracle decides membership by the same endomorphism identities as the kernels; on every named point its
    verdict equals [r]P = O."""
    pts = points()
    for name, a, _ in pts["g1"]:
        assert pyref.g1_is_torsion_free((a[0], a[1], False)) == in_subgroup(Fp, a), name
    for name, a, _ in pts["g2"]:
        assert pyref.g2_is_torsion_free((a[0], a[1], False)) == in_subgroup(Fp2, a), name


# ---------------------------------------------------------------- CPU: dev simulation of the device code

def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _sim_lib(name, main):
    """A dev-simulation build of the device headers (tests/host_sim/<main>), rebuilt when a source is newer."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, name)
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, main), os.path.join(d, "sim.cpp"), os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def sim():
    """The KZG front end's simulation; it also exports sim.cpp's group ops and pairings."""
    return _sim_lib("libzkpair_sim_kzg.so", "sim_kzg.cpp")


@pytest.fixture(scope="module")
def sim_g16():
    return _sim_lib("libzkpair_sim_g16.so", "sim_groth16.cpp")


def _group(F):
    return (Fp, "g1", 0, 2, 4) if F is Fp else (Fp2, "g2", 1, 3, 5)


def _sim_check(sim, F, pts):
    _, _, gop, _, _ = _group(F)
    xy, inf = enc_rows(F, pts)
    st = np.full(len(pts), 9, np.uint8)
    assert sim.sim_group_op(gop, _p(xy), _p(inf), None, None, _p(st), ctypes.c_size_t(len(pts))) == 0
    return st


def _sim_mul(sim, F, bases, ks):
    _, _, _, gop, _ = _group(F)
    xy, inf = enc_rows(F, bases)
    k = fr(ks)
    out, flag = np.full_like(xy, 7), np.full(len(ks), 9, np.uint8)
    assert sim.sim_group_op(gop, _p(xy), _p(inf), _p(k), _p(out), _p(flag), ctypes.c_size_t(len(ks))) == 0
    return out, flag


def _sim_add(sim, F, a, b):
    _, _, _, _, gop = _group(F)
    axy, ainf = enc_rows(F, a)
    bxy, binf = enc_rows(F, b)
    out, flag = np.full_like(axy, 7), np.full(len(a), 9, np.uint8)
    assert sim.sim_group_add(gop, _p(axy), _p(ainf), _p(bxy), _p(binf), _p(out), _p(flag), ctypes.c_size_t(len(a))) == 0
    return out, flag


def _expect_mul(F, rows):
    return enc_rows(F, [mul(F, a, k) for _, a, k in rows])


def _expect_add(F, rows):
    xy, inf = enc_rows(F, [add(F, a, b) for _, a, b in rows])
    return xy, np.array([add_flag(F, a, b) for _, a, b in rows], np.uint8)


def _assert_rows(names, out, flag, exp, eflag):
    for i, name in enumerate(names):
        assert flag[i] == eflag[i] and np.array_equal(out[i], exp[i]), (i, name, flag[i], eflag[i])


@pytest.mark.parametrize("group", ["g1", "g2"])
def test_sim_subgroup_checks_match_the_definition(sim, group):
    """Status 0 for the subgroup points, 2 (not torsion free) for every point with a small component."""
    F = Fp if group == "g1" else Fp2
    named = points()[group]
    st = _sim_check(sim, F, [a for _, a, _ in named])
    assert [(n, int(s)) for (n, _, _), s in zip(named, st)] == [(n, 0 if in_subgroup(F, a) else 2) for n, a, _ in named]


@pytest.mark.parametrize("group", ["g1", "g2"])
def test_sim_scalar_mul_on_small_order_bases(sim, group):
    """[k]B bit-exact for small-order and mixed-order bases across the ladder's branches; identities as (0, 1), flag 1."""
    F = Fp if group == "g1" else Fp2
    rows = mul_rows(F)
    out, flag = _sim_mul(sim, F, [a for _, a, _ in rows], [k for _, _, k in rows])
    exp, einf = _expect_mul(F, rows)
    _assert_rows(["%s * %#x" % (n, k) for n, _, k in rows], out, flag, exp, einf)
    assert 0 < einf.sum() < len(rows)


@pytest.mark.parametrize("group", ["g1", "g2"])
def test_sim_addition_with_small_order_points(sim, group):
    F = Fp if group == "g1" else Fp2
    rows = add_rows(F)
    out, flag = _sim_add(sim, F, [a for _, a, _ in rows], [b for _, _, b in rows])
    exp, eflag = _expect_add(F, rows)
    _assert_rows([n for n, _, _ in rows], out, flag, exp, eflag)
    assert (eflag == 3).sum() >= 4


def _shifted(F, a, t):
    return enc(F, add(F, a, t))[0]


def kzg_shift_rows(proof, t3, t11):
    """(name, proof row (24,)) for one KZG proof C | pi: unshifted, then C or pi plus T3 or T11."""
    c, pi = dec(Fp, proof[:12]), dec(Fp, proof[12:])
    rows = [("valid", proof)]
    for tn, t in (("T3", t3), ("T11", t11)):
        rows.append(("C+" + tn, np.concatenate([_shifted(Fp, c, t), proof[12:]])))
        rows.append(("pi+" + tn, np.concatenate([proof[:12], _shifted(Fp, pi, t)])))
    return rows


def kzg_p(proof, z, y):
    """P = C + [z]pi - [y]G1 of a KZG check, from the reference."""
    c, pi = dec(Fp, proof[:12]), dec(Fp, proof[12:])
    return add(Fp, add(Fp, c, mul(Fp, pi, z)), neg(Fp, mul(Fp, G1, y)))


def _kzg_oracle_is_one(coracle, rows, z, y, tau_g2):
    g1, g1inf = enc_rows(Fp, [a for pr in rows for a in (kzg_p(pr, z, y), dec(Fp, pr[12:]))])
    g2 = np.tile(np.stack([enc(Fp2, G2)[0], enc(Fp2, neg(Fp2, tau_g2))[0]]), (len(rows), 1))
    return coracle.multi_pairing_batch(g1, g1inf, g2, None, 2)[1]


def test_sim_kzg_front_end_rejects_shifted_points(sim, coracle):
    """A KZG proof whose C or pi is shifted by a point of order 3 or 11 still satisfies the pairing equation (C oracle),
    and the front end gives it BAD_POINT with zeroed, flagged slots; the unshifted proof passes."""
    pts = points()
    kzg = pts["kzg"]
    proof = np.concatenate([enc(Fp, kzg["c"])[0], enc(Fp, kzg["pi"])[0]])
    rows = kzg_shift_rows(proof, pts["t3"], pts["t11"])
    assert list(_kzg_oracle_is_one(coracle, [r for _, r in rows], kzg["z"], kzg["y"], kzg["tau_g2"])) == [1] * len(rows)
    table = np.zeros(32 * 255 * 2 * 6, np.uint64)
    sim.sim_kzg_table(_p(enc(Fp, G1)[0]), _p(table))
    proofs = np.stack([r for _, r in rows])
    n = len(rows)
    zy = np.tile(np.concatenate([fr([kzg["z"]])[0], fr([kzg["y"]])[0]]), (n, 1))
    g1, g1inf, st = np.full((n, 24), 7, np.uint64), np.full((n, 2), 9, np.uint8), np.full(n, 9, np.uint8)
    sim.sim_kzg_prepare(_p(table), _p(proofs), None, _p(zy), ctypes.c_size_t(n), _p(g1), _p(g1inf), _p(st))
    assert [(nm, int(s)) for (nm, _), s in zip(rows, st)] == [(nm, 0 if nm == "valid" else 2) for nm, _ in rows]
    assert np.array_equal(g1[0, :12], enc(Fp, kzg_p(proof, kzg["z"], kzg["y"]))[0]) and np.array_equal(g1[0, 12:], proof[12:])
    assert not g1[1:].any() and g1inf[1:].all() and not g1inf[0].any()


def g16_shift_rows(proof, t3, t11, t13):
    """(name, proof row (48,)) for one Groth16 proof A | B | C: unshifted, A + T3, C + T11, B + T13."""
    a, b, c = dec(Fp, proof[:12]), dec(Fp2, proof[12:36]), dec(Fp, proof[36:])
    return [("valid", proof),
            ("A+T3", np.concatenate([_shifted(Fp, a, t3), proof[12:]])),
            ("C+T3", np.concatenate([proof[:36], _shifted(Fp, c, t3)])),
            ("C+T11", np.concatenate([proof[:36], _shifted(Fp, c, t11)])),
            ("B+T13", np.concatenate([proof[:12], _shifted(Fp2, b, t13), proof[36:]]))]


def _g16_oracle_is_one(coracle, rows, alpha, ls, beta, gamma, delta):
    """The C oracle's 4-pair product (A, alpha, L, C) x (B, -beta, -gamma, -delta) per proof row, L = ls[i]."""
    g1, g1inf = enc_rows(Fp, [a for pr, l in zip(rows, ls) for a in (dec(Fp, pr[:12]), alpha, l, dec(Fp, pr[36:]))])
    fixed = [enc(Fp2, neg(Fp2, v))[0] for v in (beta, gamma, delta)]
    g2 = np.stack([np.concatenate([pr[12:36]] + fixed) for pr in rows])
    return coracle.multi_pairing_batch(g1, g1inf, g2.reshape(-1, 24), None, 4)[1]


# e(A, B + T13) for B + T13 outside G2: the Miller loop's value is not e(A, B) times a pairing of T13, and the product
# of the four pairings is not one (the C oracle, on the proof of points() and on the GPU test's proofs)
B_SHIFT_EQUATION_HOLDS = False


def test_sim_groth16_front_end_rejects_shifted_points(sim_g16, coracle):
    """A Groth16 proof with A or C shifted by a point of order 3 or 11 still satisfies the pairing equation (C oracle);
    with B + T13 it does not.  The front end gives every shifted proof BAD_POINT with zeroed, flagged slots."""
    pts = points()
    g = pts["g16"]
    proof = np.concatenate([enc(Fp, g["a"])[0], enc(Fp2, g["b"])[0], enc(Fp, g["c"])[0]])
    rows = g16_shift_rows(proof, pts["t3"], pts["t11"], pts["t13"])
    one = _g16_oracle_is_one(coracle, [r for _, r in rows], g["alpha"], [g["l"]] * len(rows), g["beta"], g["gamma"], g["delta"])
    assert list(one) == [1, 1, 1, 1, int(B_SHIFT_EQUATION_HOLDS)]
    ic, ic_inf = enc_rows(Fp, g["ic"])
    tables = np.zeros(32 * 255 * 2 * 6, np.uint64)
    sim_g16.sim_g16_tables(_p(ic), _p(ic_inf), 1, _p(tables))
    proofs = np.stack([r for _, r in rows])
    n = len(rows)
    x = np.tile(fr(g["x"]), (n, 1))
    g1, g1inf = np.full((n, 48), 7, np.uint64), np.full((n, 4), 9, np.uint8)
    g2, g2inf, st = np.full((n, 24), 7, np.uint64), np.full(n, 9, np.uint8), np.full(n, 9, np.uint8)
    sim_g16.sim_g16_prepare(_p(enc(Fp, g["alpha"])[0]), _p(ic[0]), _p(ic_inf), _p(tables), 1, _p(proofs), None, _p(x),
                            ctypes.c_size_t(n), _p(g1), _p(g1inf), _p(g2), _p(g2inf), _p(st))
    assert [(nm, int(s)) for (nm, _), s in zip(rows, st)] == [(nm, 0 if nm == "valid" else 2) for nm, _ in rows]
    assert np.array_equal(g1[0, 24:36], enc(Fp, g["l"])[0]) and not g1inf[0].any() and g2inf[0] == 0
    assert not g1[1:].any() and not g2[1:].any() and g1inf[1:].all() and g2inf[1:].all()


def test_sim_pairing_with_g1_outside_the_subgroup(sim, coracle):
    """e(P + T, Q) for T of order 3, 11 and 33 through the simulated Miller loop and final exponentiation: bit-exact with
    the C oracle, equal to e(P, Q), and e(T3, Q) = 1."""
    pts = points()
    p, q, t3, t11 = pts["p"], pts["q"], pts["t3"], pts["t11"]
    g1, i1 = enc_rows(Fp, [add(Fp, p, t3), add(Fp, p, t11), add(Fp, add(Fp, p, t3), t11), t3, p])
    g2 = np.tile(enc(Fp2, q)[0], (5, 1))
    gt = np.zeros((5, 72), np.uint64)
    assert sim.sim_pairing(3, _p(g1), _p(i1), _p(g2), None, ctypes.c_size_t(5), 1, None, _p(gt), None) == 0
    assert np.array_equal(gt, coracle.pairing_batch(g1, i1, g2, None))
    one = np.array(pyref.fp12_to_u64(pyref.FP12_ONE), np.uint64)
    assert np.array_equal(gt[0], gt[4]) and np.array_equal(gt[1], gt[4]) and np.array_equal(gt[2], gt[4]) and np.array_equal(gt[3], one)


# ---------------------------------------------------------------- GPU

def _tiled(n_distinct):
    return np.arange(TILED) % n_distinct


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["g1", "g2"])
def test_gpu_checks_mul_add_tiled_past_a_chunk(engine, group):
    """The check, multiplication and addition rows of the CPU tests through the batch entry points, tiled to 2^18 + 37
    rows: every distinct row equals the reference, every tiled copy its first occurrence."""
    F = Fp if group == "g1" else Fp2
    check = engine.g1_check_batch if F is Fp else engine.g2_check_batch
    mulb = engine.g1_mul_batch if F is Fp else engine.g2_mul_batch
    addb = engine.g1_add_batch if F is Fp else engine.g2_add_batch

    named = points()[group]
    xy, inf = enc_rows(F, [a for _, a, _ in named])
    idx = _tiled(len(named))
    st = check(xy[idx], inf[idx])
    assert [(n, int(s)) for (n, _, _), s in zip(named, st)] == [(n, 0 if in_subgroup(F, a) else 2) for n, a, _ in named]
    assert np.array_equal(st, st[idx])

    rows = mul_rows(F)
    bxy, binf = enc_rows(F, [a for _, a, _ in rows])
    k = fr([k for _, _, k in rows])
    idx = _tiled(len(rows))
    out, flag = mulb(bxy[idx], k[idx], binf[idx])
    exp, einf = _expect_mul(F, rows)
    _assert_rows(["%s * %#x" % (n, k) for n, _, k in rows], out, flag, exp, einf)
    assert np.array_equal(out, out[idx]) and np.array_equal(flag, flag[idx])

    rows = add_rows(F)
    axy, ainf = enc_rows(F, [a for _, a, _ in rows])
    bxy, binf = enc_rows(F, [b for _, _, b in rows])
    idx = _tiled(len(rows))
    out, flag = addb(axy[idx], bxy[idx], ainf[idx], binf[idx])
    exp, eflag = _expect_add(F, rows)
    _assert_rows([n for n, _, _ in rows], out, flag, exp, eflag)
    assert np.array_equal(out, out[idx]) and np.array_equal(flag, flag[idx])


def _neg_rows(F, rows):
    return np.stack([enc(F, neg(F, dec(F, r)))[0] for r in rows])


@pytest.mark.gpu
def test_gpu_kzg_shifted_proofs_hold_the_equation_and_are_rejected(engine):
    """KZG proofs with C or pi shifted by T3 or T11 satisfy the bare prepared 2-pair check (is_one = 1), and
    kzg_verify_batch gives them BAD_POINT while the unshifted proofs in the same batch stay VALID."""
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    pts = points()
    w = workloads.kzg_proofs(engine, 4, seed=0x7035, corrupt_every=0)
    proofs, exp, g1, g1inf = [], [], [], []
    for i in range(4):
        zz, yy = (sum(int(v) << (64 * k) for k, v in enumerate(w["zy"][i, h:h + 4])) for h in (0, 4))
        for name, pr in kzg_shift_rows(w["proofs"][i], pts["t3"], pts["t11"]):
            proofs.append(pr)
            exp.append(z.KZG_VALID if name == "valid" else z.KZG_BAD_POINT)
            e, f = enc_rows(Fp, [kzg_p(pr, zz, yy), dec(Fp, pr[12:])])
            g1.append(e)
            g1inf.append(f)
    n = len(proofs)
    tabs = engine.g2_prepare_batch(np.stack([enc(Fp2, G2)[0], _neg_rows(Fp2, [w["tau_g2"]])[0]]))
    _, one = engine.multi_pairing_prepared_batch(np.concatenate(g1), None, 2, tabs, g1_inf=np.concatenate(g1inf))
    assert list(one) == [1] * n
    zy = np.repeat(w["zy"], n // 4, axis=0)
    with engine.kzg_setup(w["tau_g2"]) as s:
        st = engine.kzg_verify_batch(s, np.stack(proofs), zy)
    assert list(st) == exp


@pytest.mark.gpu
def test_gpu_groth16_shifted_proofs_and_their_verdicts(engine, coracle):
    """Groth16 proofs with A or C shifted by T3 (or C by T11) satisfy the bare prepared 4-pair check (is_one = 1); B
    shifted by T13 does not (C oracle).  groth16_verify_batch gives every shifted proof BAD_POINT and the unshifted
    ones VALID, in one batch."""
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    pts = points()
    w = workloads.groth16_proofs(engine, 4, 1, seed=0x7036, corrupt_every=0)
    alpha, beta, gamma, delta = dec(Fp, w["alpha"]), dec(Fp2, w["beta"]), dec(Fp2, w["gamma"]), dec(Fp2, w["delta"])
    proofs, names = [], []
    for i in range(4):
        for name, pr in g16_shift_rows(w["proofs"][i], pts["t3"], pts["t11"], pts["t13"]):
            proofs.append(pr)
            names.append((i, name))
    proofs = np.stack(proofs)
    n = len(proofs)
    ls = [mul(Fp, G1, sum(int(v) << (64 * k) for k, v in enumerate(w["l"][i]))) for i, _ in names]
    g1 = np.stack([np.concatenate([pr[:12], w["alpha"], enc(Fp, l)[0], pr[36:]]) for pr, l in zip(proofs, ls)])
    g1inf = np.array([[0, 0, 1 if l is None else 0, 0] for l in ls], np.uint8)
    tabs = engine.g2_prepare_batch(_neg_rows(Fp2, [w["beta"], w["gamma"], w["delta"]]))
    g1_lifted = [i for i, (_, nm) in enumerate(names) if nm != "B+T13"]
    _, one = engine.multi_pairing_prepared_batch(g1[g1_lifted].reshape(-1, 12), proofs[g1_lifted, 12:36], 4, tabs,
                                                 g1_inf=g1inf[g1_lifted].reshape(-1))
    assert list(one) == [1] * len(g1_lifted)
    b_shift = [i for i, (_, nm) in enumerate(names) if nm == "B+T13"]
    one = _g16_oracle_is_one(coracle, proofs[b_shift], alpha, [ls[i] for i in b_shift], beta, gamma, delta)
    assert list(one) == [int(B_SHIFT_EQUATION_HOLDS)] * len(b_shift)
    with engine.groth16_prepare_vk(w["alpha"], w["beta"], w["gamma"], w["delta"], w["ic"]) as vk:
        st = engine.groth16_verify_batch(vk, proofs, np.repeat(w["inputs"], n // 4, axis=0))
    assert list(st) == [z.G16_VALID if nm == "valid" else z.G16_BAD_POINT for _, nm in names]


@pytest.mark.gpu
def test_gpu_setup_and_key_reject_shifted_points(engine):
    """kzg_setup([tau]G2 + T13) and groth16_prepare_vk with IC_1 + T3 or delta + T13 raise INVALID_ARG naming the point;
    the unshifted setup and key are accepted."""
    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import workloads
    pts = points()
    w = workloads.kzg_proofs(engine, 2, seed=0x7037, corrupt_every=0)
    with engine.kzg_setup(w["tau_g2"]) as s:
        assert list(engine.kzg_verify_batch(s, w["proofs"], w["zy"])) == [0, 0]
    with pytest.raises(z.ZkpError) as ei:
        engine.kzg_setup(_shifted(Fp2, dec(Fp2, w["tau_g2"]), pts["t13"]))
    assert ei.value.code == -1 and "tau_g2" in str(ei.value), str(ei.value)
    g = workloads.groth16_proofs(engine, 2, 2, seed=0x7038, corrupt_every=0)
    key = dict(alpha=g["alpha"], beta=g["beta"], gamma=g["gamma"], delta=g["delta"], ic=g["ic"])
    with engine.groth16_prepare_vk(**key) as vk:
        assert list(engine.groth16_verify_batch(vk, g["proofs"], g["inputs"])) == [0, 0]
    ic = g["ic"].copy()
    ic[1] = _shifted(Fp, dec(Fp, ic[1]), pts["t3"])
    for name, bad in (("ic_g1[1]", dict(key, ic=ic)), ("delta_g2", dict(key, delta=_shifted(Fp2, dec(Fp2, g["delta"]), pts["t13"])))):
        with pytest.raises(z.ZkpError) as ei:
            engine.groth16_prepare_vk(**bad)
        assert ei.value.code == -1 and name in str(ei.value), str(ei.value)


@pytest.mark.gpu
def test_gpu_pairing_with_g1_outside_the_subgroup(engine, coracle):
    """e(P + T, Q) for T of order 3, 11 and 33, and e(T3, Q): pairing_batch and final_exp(miller_loop) bit-exact with the
    C oracle (the header defines the pairing for curve points; G2 arguments stay in G2)."""
    pts = points()
    p, q, t3, t11 = pts["p"], pts["q"], pts["t3"], pts["t11"]
    g1, i1 = enc_rows(Fp, [add(Fp, p, t3), neg(Fp, add(Fp, p, t3)), add(Fp, p, t11), add(Fp, add(Fp, p, t3), t11), t3, (0, P - 2), p])
    n = len(g1)
    g2 = np.tile(enc(Fp2, q)[0], (n, 1))
    exp = coracle.pairing_batch(g1, i1, g2, None)
    assert np.array_equal(engine.pairing_batch(g1, g2, i1), exp)
    assert np.array_equal(engine.miller_loop_batch(g1, g2, i1), coracle.miller_loop_batch(g1, i1, g2, None))
    assert np.array_equal(engine.final_exponentiation_batch(engine.miller_loop_batch(g1, g2, i1)), exp)
    one = np.array(pyref.fp12_to_u64(pyref.FP12_ONE), np.uint64)
    assert np.array_equal(exp[0], exp[6]) and np.array_equal(exp[2], exp[6]) and np.array_equal(exp[4], one)
