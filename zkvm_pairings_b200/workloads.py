"""Synthetic workloads of BASELINE.json's configs, built with the engine itself (GPU) and Python integers.

Nothing here touches the oracle: tests and bench.py use these generators for the INPUTS and the expected
verdicts, and compare Gt values with the oracle separately.

Config 3 ("Groth16-style 4-pair multi-pairing product checks, shared final exponentiation per check"):
every check is the verification equation of a Groth16-shaped verifier with a fixed verifying key
(beta, gamma, delta in G2) and per-proof points A, C, L, X in G1 and B in G2,

    e(A, B) * e(X, beta G2) * e(C, -delta G2) * e(L, -gamma G2) == 1,

with A = a G1, B = b G2, C = c G1, L = l G1 from 64-bit seeded scalars and X = s G1 where
s = (c delta + l gamma - a b) / beta mod r makes the product one.  A seeded 1 % of the checks is corrupted
(s + 1), so the expected verdict vector is known without running a pairing.
"""
from __future__ import annotations

import numpy as np

# BLS12-381 group order and generators (the curve's standard constants; the reference carries them in
# src/common.rs:69-157)
R_ORDER = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
G1_GEN = (
    0x17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb,
    0x08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3edd03cc744a2888ae40caa232946c5e7e1,
)
G2_GEN = (
    (0x024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8,
     0x13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e),
    (0x0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c923ac9cc3baca289e193548608b82801,
     0x0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab3f370d275cec1da1aaa9075ff05f79be),
)
VK_SEED = 0x6716_0B20_0


def _limbs(v: int, n: int):
    return [(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(n)]


def _fp_row(vals):
    return np.array([x for v in vals for x in _limbs(v, 6)], dtype=np.uint64)


def splitmix64_at(seed: int, idx: np.ndarray) -> np.ndarray:
    """Output number idx+1 of the SplitMix64 stream seeded with `seed` (vectorised; the scalars
    zkp_gen_points uses, csrc/ops.cuh splitmix64_at)."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed & 0xFFFFFFFFFFFFFFFF) + (idx.astype(np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def gen_scalars(seed: int, first: int, n: int):
    """(a_i, b_i) of zkp_gen_points(seed, first, n): zero mapped to one."""
    i = np.arange(first, first + n, dtype=np.uint64)
    a = splitmix64_at(seed, np.uint64(2) * i)
    b = splitmix64_at(seed, np.uint64(2) * i + np.uint64(1))
    a[a == 0] = 1
    b[b == 0] = 1
    return a, b


def scalar_matrix(ks) -> np.ndarray:
    """Python ints -> (n, 4) little-endian u64 limbs (the limbs of an Fr)."""
    return np.array([_limbs(int(k), 4) for k in ks], dtype=np.uint64).reshape(-1, 4)


def groth16_checks(engine, n_checks: int, seed: int = 0x6716, corrupt_every: int = 100, corrupt_at: int = 7):
    """BASELINE config 3 inputs.  Returns a dict:
         g1 (n*4, 12)   A, X, C, L per check            g2 (n*4, 24)  B, beta, -delta, -gamma per check
         g2_var (n, 24) B only (prepared variant)        fixed (3, 24) beta G2, -delta G2, -gamma G2
         expect_one (n,) bool                            pairs_per_check = 4, prepared_pairs = 3
    """
    n = int(n_checks)
    vk = splitmix64_at(VK_SEED, np.arange(12, dtype=np.uint64))
    beta, gamma, delta = (int.from_bytes(vk[4 * j:4 * j + 4].tobytes(), "little") % R_ORDER or 1 for j in range(3))
    g2gen = np.tile(_fp_row([G2_GEN[0][0], G2_GEN[0][1], G2_GEN[1][0], G2_GEN[1][1]]), (3, 1))
    fixed, finf = engine.g2_mul_batch(g2gen, scalar_matrix([beta, R_ORDER - delta, R_ORDER - gamma]))
    assert not finf.any()
    # per-proof points from the seeded generator: (A, B), C, L
    gA, _, gB, _ = engine.gen_points(seed, 0, n)
    gC, _, _, _ = engine.gen_points(seed + 1, 0, n)
    gL, _, _, _ = engine.gen_points(seed + 2, 0, n)
    a, b = gen_scalars(seed, 0, n)
    c, _ = gen_scalars(seed + 1, 0, n)
    l, _ = gen_scalars(seed + 2, 0, n)
    beta_inv = pow(beta, -1, R_ORDER)
    corrupt = np.zeros(n, dtype=bool)
    if corrupt_every:
        corrupt[corrupt_at % corrupt_every::corrupt_every] = True
    s = np.empty((n, 4), dtype=np.uint64)
    for i in range(n):
        v = ((int(c[i]) * delta + int(l[i]) * gamma - int(a[i]) * int(b[i])) * beta_inv + (1 if corrupt[i] else 0)) % R_ORDER
        s[i, 0] = v & 0xFFFFFFFFFFFFFFFF
        s[i, 1] = (v >> 64) & 0xFFFFFFFFFFFFFFFF
        s[i, 2] = (v >> 128) & 0xFFFFFFFFFFFFFFFF
        s[i, 3] = v >> 192
    g1gen = np.broadcast_to(_fp_row([G1_GEN[0], G1_GEN[1]]), (n, 12))
    gX, xinf = engine.g1_mul_batch(np.ascontiguousarray(g1gen), s)
    assert not xinf.any()
    g1 = np.empty((n, 4, 12), dtype=np.uint64)
    g1[:, 0], g1[:, 1], g1[:, 2], g1[:, 3] = gA, gX, gC, gL
    g2 = np.empty((n, 4, 24), dtype=np.uint64)
    g2[:, 0] = gB
    g2[:, 1:] = fixed[None]
    return {"g1": g1.reshape(-1, 12), "g2": g2.reshape(-1, 24), "g2_var": np.ascontiguousarray(gB), "fixed": fixed,
            "expect_one": ~corrupt, "pairs_per_check": 4, "prepared_pairs": 3}


def _fr_matrix(vals) -> np.ndarray:
    """Python ints (< 2^256) -> (n, 4) little-endian u64 limbs, vectorised over 64-bit slices."""
    vals = list(vals)
    m = np.empty((len(vals), 4), dtype=np.uint64)
    for k in range(4):
        m[:, k] = np.array([(v >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for v in vals], dtype=np.uint64)
    return m


def groth16_proofs(engine, n: int, n_public: int, seed: int = 0x6716, corrupt_every: int = 100, corrupt_at: int = 7):
    """Groth16 verifying key, proofs and public inputs with known verdicts, from the trapdoor construction.

    Seeded alpha, beta, gamma, delta and u_0 .. u_l give the key alpha G1, beta G2, gamma G2, delta G2 and
    IC_j = u_j G1.  Per proof: random a, b and full-width inputs x_j < r, l = u_0 + sum_j x_j u_j and
    c = (a b - alpha beta - l gamma) / delta mod r; A = a G1, B = b G2, C = c G1 (engine.g1_mul_batch /
    g2_mul_batch).  The verifier sees only the equation, so these proofs exercise it as a prover's would.  A seeded
    1 % is corrupted as x_1 + 1 (C + G1 when there is no public input), so the expected verdicts are known without
    running a pairing.  Returns a dict:
        alpha (12,), beta / gamma / delta (24,), ic (l + 1, 12)      the verifying key
        proofs (n, 48) A | B | C, inputs (n, l, 4)                  what the verifier receives
        l (n, 4) the discrete log of the L the verifier derives    expect (n,) uint8 ZKP_G16_VALID / ZKP_G16_INVALID
    """
    import random
    rng = random.Random(seed)
    n, lp = int(n), int(n_public)
    alpha, beta, gamma, delta = (rng.randrange(1, R_ORDER) for _ in range(4))
    u = [rng.randrange(1, R_ORDER) for _ in range(lp + 1)]
    g1gen, g2gen = _fp_row([G1_GEN[0], G1_GEN[1]]), _fp_row([G2_GEN[0][0], G2_GEN[0][1], G2_GEN[1][0], G2_GEN[1][1]])
    k1, _ = engine.g1_mul_batch(np.tile(g1gen, (lp + 2, 1)), _fr_matrix([alpha] + u))
    k2, _ = engine.g2_mul_batch(np.tile(g2gen, (3, 1)), _fr_matrix([beta, gamma, delta]))
    corrupt = np.zeros(n, dtype=bool)
    if corrupt_every:
        corrupt[corrupt_at % corrupt_every::corrupt_every] = True
    a = [rng.randrange(1, R_ORDER) for _ in range(n)]
    b = [rng.randrange(1, R_ORDER) for _ in range(n)]
    x = [[rng.randrange(R_ORDER) for _ in range(lp)] for _ in range(n)]
    ab_ = alpha * beta
    dinv = pow(delta, -1, R_ORDER)
    ls, cs = [], []
    for i in range(n):
        l = (u[0] + sum(xj * uj for xj, uj in zip(x[i], u[1:]))) % R_ORDER
        c = (a[i] * b[i] - ab_ - l * gamma) * dinv % R_ORDER
        if corrupt[i] and lp:
            x[i][0] = (x[i][0] + 1) % R_ORDER
            l = (l + u[1]) % R_ORDER
        elif corrupt[i]:
            c = (c + 1) % R_ORDER
        ls.append(l)
        cs.append(c)
    gA, _ = engine.g1_mul_batch(np.tile(g1gen, (n, 1)), _fr_matrix(a))
    gB, _ = engine.g2_mul_batch(np.tile(g2gen, (n, 1)), _fr_matrix(b))
    gC, _ = engine.g1_mul_batch(np.tile(g1gen, (n, 1)), _fr_matrix(cs))
    inputs = _fr_matrix([v for row in x for v in row]).reshape(n, lp, 4)
    return {"alpha": k1[0], "beta": k2[0], "gamma": k2[1], "delta": k2[2], "ic": k1[1:],
            "proofs": np.concatenate([gA, gB, gC], axis=1), "inputs": inputs, "l": _fr_matrix(ls),
            "expect": corrupt.astype(np.uint8)}


def kzg_proofs(engine, n: int, seed: int = 0x4844, corrupt_every: int = 100, corrupt_at: int = 7):
    """KZG point-evaluation setup and proofs with known verdicts, from the trapdoor construction.

    A seeded tau gives the setup [tau]G2.  Per proof: random z, y and q < r, pi = q G1 and C = (y + q (tau - z)) G1
    (engine.g1_mul_batch), so C - y G1 = q (tau - z) G1 opens the committed polynomial at z to y.  A seeded 1 % of the
    claimed values is corrupted as y + 1 mod r, so the expected verdicts are known without running a pairing.
    Returns a dict:
        tau_g2 (24,)                                  the setup
        proofs (n, 24) C | pi, zy (n, 8) z | y          what the verifier receives
        p (n, 4) the discrete log of P = C + z pi - y G1 the verifier derives
        expect (n,) uint8 ZKP_KZG_VALID / ZKP_KZG_INVALID
    """
    import random
    rng = random.Random(seed)
    n = int(n)
    tau = rng.randrange(1, R_ORDER)
    g1gen, g2gen = _fp_row([G1_GEN[0], G1_GEN[1]]), _fp_row([G2_GEN[0][0], G2_GEN[0][1], G2_GEN[1][0], G2_GEN[1][1]])
    tg, _ = engine.g2_mul_batch(g2gen[None], _fr_matrix([tau]))
    corrupt = np.zeros(n, dtype=bool)
    if corrupt_every:
        corrupt[corrupt_at % corrupt_every::corrupt_every] = True
    z = [rng.randrange(R_ORDER) for _ in range(n)]
    y = [rng.randrange(R_ORDER) for _ in range(n)]
    q = [rng.randrange(1, R_ORDER) for _ in range(n)]
    c = [(yi + qi * (tau - zi)) % R_ORDER for zi, yi, qi in zip(z, y, q)]
    y = [(yi + 1) % R_ORDER if bad else yi for yi, bad in zip(y, corrupt)]
    p = [(ci - yi + zi * qi) % R_ORDER for ci, yi, zi, qi in zip(c, y, z, q)]
    pts, _ = engine.g1_mul_batch(np.tile(g1gen, (2 * n, 1)), _fr_matrix(c + q))
    return {"tau_g2": tg[0], "proofs": np.concatenate([pts[:n], pts[n:]], axis=1),
            "zy": np.concatenate([_fr_matrix(z), _fr_matrix(y)], axis=1), "p": _fr_matrix(p),
            "expect": corrupt.astype(np.uint8)}


BLOB_N = 4096                # EIP-4844 FIELD_ELEMENTS_PER_BLOB
BLOB_BYTES = 32 * BLOB_N
P_BASE = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab


def _roots_of_unity():
    """The 4096th roots of unity of Fr, omega^k for k = 0 .. 4095 (omega = 7^((r - 1) / 4096))."""
    w = pow(7, (R_ORDER - 1) // BLOB_N, R_ORDER)
    roots = [1] * BLOB_N
    for i in range(1, BLOB_N):
        roots[i] = roots[i - 1] * w % R_ORDER
    return roots


def blob_domain():
    """roots_brp: the 4096th roots of unity of Fr (generator 7^((r - 1) / 4096)) in bit-reversed order."""
    roots = _roots_of_unity()
    return [roots[int(format(i, "012b")[::-1], 2)] for i in range(BLOB_N)]


def _batch_inv(vals):
    pre, acc = [], 1
    for v in vals:
        pre.append(acc)
        acc = acc * v % R_ORDER
    inv, out = pow(acc, -1, R_ORDER), [0] * len(vals)
    for i in range(len(vals) - 1, -1, -1):
        out[i] = inv * pre[i] % R_ORDER
        inv = inv * vals[i] % R_ORDER
    return out


def lagrange_at(tau, roots):
    """The Lagrange basis of the domain `roots` at tau: l_k(tau) = (tau^N - 1) / N * w_k / (tau - w_k), for tau outside
    the domain."""
    scale = (pow(tau, BLOB_N, R_ORDER) - 1) * pow(BLOB_N, -1, R_ORDER) % R_ORDER
    return [scale * w % R_ORDER * i % R_ORDER for w, i in zip(roots, _batch_inv([(tau - w) % R_ORDER for w in roots]))]


def kzg_lagrange_setup(engine, seed: int = 0x4844):
    """A trusted setup from a seeded tau: (tau, [tau]G2 (24,), g1_lagrange (4096, 12)), g1_lagrange in the natural order
    of a setup file, L_k = [l_k(tau)]G1 at omega^k (engine.g1_mul_batch of the Lagrange coefficients)."""
    import random
    rng = random.Random(seed)
    tau = rng.randrange(1, R_ORDER)
    g1gen, g2gen = _fp_row([G1_GEN[0], G1_GEN[1]]), _fp_row([G2_GEN[0][0], G2_GEN[0][1], G2_GEN[1][0], G2_GEN[1][1]])
    tg, _ = engine.g2_mul_batch(g2gen[None], _fr_matrix([tau]))
    lag, _ = engine.g1_mul_batch(np.tile(g1gen, (BLOB_N, 1)), _fr_matrix(lagrange_at(tau, _roots_of_unity())))
    return tau, tg[0], lag


def kzg_cell_setup(engine, seed: int = 0x7594):
    """An EIP-7594 trusted setup from a seeded tau: (tau, g2_monomial (65, 24) = [tau^i]G2 for i <= 64, g1_monomial
    (4096, 12) = [tau^i]G1, g1_lagrange (4096, 12) as kzg_lagrange_setup gives it), by engine.g1_mul_batch /
    g2_mul_batch of the powers of tau."""
    import random
    rng = random.Random(seed)
    tau = rng.randrange(1, R_ORDER)
    powers = [pow(tau, i, R_ORDER) for i in range(BLOB_N)]
    g1gen, g2gen = _fp_row([G1_GEN[0], G1_GEN[1]]), _fp_row([G2_GEN[0][0], G2_GEN[0][1], G2_GEN[1][0], G2_GEN[1][1]])
    g2m, _ = engine.g2_mul_batch(np.tile(g2gen, (65, 1)), _fr_matrix(powers[:65]))
    g1m, _ = engine.g1_mul_batch(np.tile(g1gen, (BLOB_N, 1)), _fr_matrix(powers))
    lag, _ = engine.g1_mul_batch(np.tile(g1gen, (BLOB_N, 1)), _fr_matrix(lagrange_at(tau, _roots_of_unity())))
    return tau, g2m, g1m, lag


def blob_eval(poly, z, roots):
    """The blob's polynomial (values at roots) at z, barycentric (the value itself when z is a root)."""
    if z in roots:
        return poly[roots.index(z)]
    inv = _batch_inv([(z - w) % R_ORDER for w in roots])
    s = sum(p * w % R_ORDER * i for p, w, i in zip(poly, roots, inv)) % R_ORDER
    return s * (pow(z, BLOB_N, R_ORDER) - 1) * pow(BLOB_N, -1, R_ORDER) % R_ORDER


def g1_compressed(xy, inf=False) -> bytes:
    """The 48-byte compressed encoding of a G1 point given as canonical limbs x | y (12 u64)."""
    if inf:
        return b"\xc0" + bytes(47)
    x = sum(int(v) << (64 * k) for k, v in enumerate(xy[:6]))
    y = sum(int(v) << (64 * k) for k, v in enumerate(xy[6:12]))
    b = bytearray(x.to_bytes(48, "big"))
    b[0] |= 0x80 | (0x20 if y > (P_BASE - 1) // 2 else 0)
    return bytes(b)


def blob_challenge(blob: bytes, c48: bytes) -> int:
    """compute_challenge: SHA-256 of the Fiat-Shamir transcript as a big-endian integer mod r."""
    import hashlib
    data = b"FSBLOBVERIFY_V1_" + BLOB_N.to_bytes(16, "big") + blob + c48
    return int.from_bytes(hashlib.sha256(data).digest(), "big") % R_ORDER


def kzg_blob_proofs(engine, n: int, seed: int = 0x4844, distinct: int = 64, corrupt_every: int = 100, corrupt_at: int = 7):
    """EIP-4844 blobs, commitments and proofs with known verdicts, from the trapdoor construction.

    A seeded tau gives the setup [tau]G2.  Per distinct blob: random elements p_i < r, c = p(tau) from the Lagrange
    coefficients at tau, C = c G1 (engine.g1_mul_batch), z from the transcript of the blob and C, y = p(z), and
    pi = q G1 with q = (c - y) / (tau - z).  Python costs about 10 ms per distinct blob, so at most `distinct` blobs
    are built and tiled over the n slots.  A seeded 1 % of the slots gets pi = (q + 1) G1, so the expected verdicts are
    known without running a pairing.  Returns a dict:
        tau_g2 (24,)                                    the setup
        blobs (n, BLOB_BYTES) uint8, proofs (n, 24) C | pi   what the verifier receives
        zy (n, 8) the z | y the verifier derives         expect (n,) uint8 ZKP_KZG_VALID / ZKP_KZG_INVALID
    """
    import random
    rng = random.Random(seed)
    n = int(n)
    m = max(1, min(n, int(distinct)))
    tau = rng.randrange(1, R_ORDER)
    roots = blob_domain()
    g1gen, g2gen = _fp_row([G1_GEN[0], G1_GEN[1]]), _fp_row([G2_GEN[0][0], G2_GEN[0][1], G2_GEN[1][0], G2_GEN[1][1]])
    tg, _ = engine.g2_mul_batch(g2gen[None], _fr_matrix([tau]))
    lag = lagrange_at(tau, roots)
    polys = [[rng.randrange(R_ORDER) for _ in range(BLOB_N)] for _ in range(m)]
    blobs = np.frombuffer(b"".join(v.to_bytes(32, "big") for p in polys for v in p), dtype=np.uint8).reshape(m, BLOB_BYTES)
    cs = [sum(p * l for p, l in zip(poly, lag)) % R_ORDER for poly in polys]
    cpts, cinf = engine.g1_mul_batch(np.tile(g1gen, (m, 1)), _fr_matrix(cs))
    zs, ys, qs = [], [], []
    for k in range(m):
        z = blob_challenge(blobs[k].tobytes(), g1_compressed(cpts[k], cinf[k]))
        y = blob_eval(polys[k], z, roots)
        zs.append(z)
        ys.append(y)
        qs.append((cs[k] - y) * pow((tau - z) % R_ORDER, -1, R_ORDER) % R_ORDER)
    corrupt = np.zeros(n, dtype=bool)
    if corrupt_every:
        corrupt[corrupt_at % corrupt_every::corrupt_every] = True
    idx = np.arange(n) % m
    pis, _ = engine.g1_mul_batch(np.tile(g1gen, (n, 1)), _fr_matrix([(qs[k] + int(b)) % R_ORDER for k, b in zip(idx, corrupt)]))
    zy = np.concatenate([_fr_matrix(zs), _fr_matrix(ys)], axis=1)
    return {"tau_g2": tg[0], "blobs": blobs[idx], "proofs": np.concatenate([cpts[idx], pis], axis=1), "zy": zy[idx],
            "expect": corrupt.astype(np.uint8)}
