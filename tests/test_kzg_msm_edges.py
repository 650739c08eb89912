"""The prover's fixed-base MSM (csrc/kzg_prove.cuh msm_partial, msm_tree_add, msm_finish; kernel k_kzg_msm) on the
branches of its additions that random scalars never reach.

Every addition inside the MSM either starts from the identity or adds two points that are neither equal nor opposite,
unless the scalars are related through tau: doubling (h = 0, rr = 0) and cancellation to the identity (h = 0, rr != 0),
in the mixed additions of the threads' partial sums and in the tree that combines them, and a non-zero row whose sum is
the identity.  With the trapdoor tau known, the Lagrange coefficients l_i = l_i(tau) give every point of the setup as
a multiple of G1, so rows that reach each of those branches can be built on purpose.

A scalar model of the MSM works on these discrete logs in the kernel's order (thread t owns the bases t + 256 k, k
ascending; windows up with the signed-digit recoding; tree levels 128 .. 1) and labels every addition.  The tests use
it to check that each constructed row reaches the branch it was built for, that the rows together reach every label,
and for the expected scalar of each row.  The CPU dev simulation (tests/host_sim/sim_kzg_msm.cpp) runs the kernel's
body on the sparse rows; on the GPU, every row goes through the commitment entry points, and proofs that are the
identity go through the verifiers."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
N = 4096
TPB = 256
WINDOWS = 32
BLOB_BYTES = 32 * N
M64 = (1 << 64) - 1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BRP = [int(format(i, "012b")[::-1], 2) for i in range(N)]
IDENTITY = np.array([0] * 6 + [1] + [0] * 5, np.uint64)   # (0, 1) with the flag: the identity as the ABI writes it
VALID, BAD_POINT, BAD_SCALAR = 0, 2, 3

PARTIAL_LABELS = ("from-identity", "generic", "double", "cancel")
TREE_LABELS = ("both-identity", "p-identity", "q-identity", "generic", "double", "cancel")


# ---------------------------------------------------------------- the scalar model

def msm_digits(s):
    """kzg_prove.cuh msm_digit over the 32 windows of s < 2^256: digits in [-127, 128]"""
    out, carry = [], 0
    for w in range(WINDOWS):
        d = ((s >> (8 * w)) & 0xFF) + carry
        carry = 1 if d > 128 else 0
        out.append(d - 256 if carry else d)
    return out


def _add(p, q):
    """p + q for discrete logs (None = the identity), with the branch jac_add / jac_add_affine takes for two points
    that are not the identity"""
    if p == q:
        return 2 * p % R, "double"
    if (p + q) % R == 0:
        return None, "cancel"
    return (p + q) % R, "generic"


def msm_model(scalars, lag):
    """The MSM of one row (4096 ints, any 256-bit values) over the bases l_i G1, in the kernel's order of additions.
    Returns a dict: partial = [(thread, base, window, label)], tree = [(level, thread, label)], value = the row's sum
    (None = the identity), status, finish = "identity" when a valid row's sum is the identity (msm_finish writes
    (0, 1) with the flag)."""
    partial, tree, acc = [], [], []
    bad = any(s >= R for s in scalars)
    for t in range(TPB):
        a = None
        for k in range(N // TPB):
            i = t + TPB * k
            s = scalars[i]
            if not s or s >= R:            # blob_element reads an element >= r as 0
                continue
            for w, d in enumerate(msm_digits(s)):
                if not d:
                    continue
                e = d * (1 << (8 * w)) * lag[i] % R
                if a is None:
                    a, label = e, "from-identity"
                else:
                    a, label = _add(a, e)
                partial.append((t, i, w, label))
        acc.append(a)
    w = TPB // 2
    while w >= 1:
        for t in range(w):
            p, q = acc[t], acc[t + w]
            if p is None:
                acc[t], label = q, ("both-identity" if q is None else "p-identity")
            elif q is None:
                label = "q-identity"
            else:
                acc[t], label = _add(p, q)
            tree.append((w, t, label))
        w //= 2
    value = acc[0]
    if not bad:
        assert (value or 0) == sum(s * l for s, l in zip(scalars, lag)) % R
    return dict(partial=partial, tree=tree, value=value, status=BAD_SCALAR if bad else VALID,
                finish="identity" if value is None and not bad else None)


def labels_of(m):
    got = {("partial", e[3]) for e in m["partial"]} | {("tree", e[2]) for e in m["tree"]}
    if m["finish"]:
        got.add(("finish", m["finish"]))
    return got


ALL_LABELS = {("partial", x) for x in PARTIAL_LABELS} | {("tree", x) for x in TREE_LABELS} | {("finish", "identity")}


# ---------------------------------------------------------------- rows built from the trapdoor

def _div(a, b):
    return a * pow(b, -1, R) % R


def _sparse(entries):
    s = [0] * N
    for i, v in entries.items():
        s[i] = v
    return s


def edge_rows(lag, rng):
    """name -> (scalars, the model's check of the row's branch).  The constructed bases sit at threads 0, 1, 127, 128
    and 255, so that the first and the last tree levels do the work."""
    rows = {}

    # a. double at window 0: thread 0's sum over base 0 equals the first entry it adds for base 256
    rows["a_double_window0"] = (_sparse({0: _div(lag[256], lag[0]), 256: 1}),
                                lambda m: (0, 256, 0, "double") in m["partial"])

    # b. double at a late window with a negative digit: thread 127, base j = 383 random, base 127 such that the sum
    # before window W of base j is d_W 2^(8W) l_j
    j = 127 + TPB
    while True:
        sj = rng.randrange(R)
        ds = msm_digits(sj)
        late = [w for w in range(16, WINDOWS - 1) if ds[w] < 0]
        if late:
            break
    W = late[0]
    low = sum(ds[w] << (8 * w) for w in range(W))
    rows["b_double_late_negative"] = (_sparse({127: _div((ds[W] * (1 << (8 * W)) - low) * lag[j], lag[127]), j: sj}),
                                      lambda m, W=W: (127, 383, W, "double") in m["partial"])

    # c. cancel, then continue: thread 128's sum is the identity after base 384, then base 640 starts it again
    def check_c(m):
        ev = [e for e in m["partial"] if e[0] == 128]
        k = ev.index((128, 384, 0, "cancel"))
        return ev[k + 1][1] == 640 and ev[k + 1][3] == "from-identity" and m["value"] is not None
    rows["c_cancel_then_continue"] = (_sparse({128: (-_div(lag[384], lag[128])) % R, 384: 1, 640: rng.randrange(R)}), check_c)

    # c'. cancel at a thread's last addition: thread 255's scalars are non-zero, its partial sum is the identity; base 1
    # keeps the row's sum non-zero
    s511 = rng.randrange(R)
    last_w = max(w for w, d in enumerate(msm_digits(s511)) if d)

    def check_c2(m):
        ev = [e for e in m["partial"] if e[0] == 255]
        return ev[-1] == (255, 511, last_w, "cancel") and m["value"] is not None and ("tree", "both-identity") in labels_of(m)
    rows["c2_cancel_last"] = (_sparse({1: rng.randrange(R), 255: (-_div(s511 * lag[511], lag[255])) % R, 511: s511}), check_c2)

    # d. the tree doubles at level 1 (threads 0 and 1), and cancels at level 128 (threads 127 and 255: a non-zero row
    # whose sum is the identity)
    s0 = rng.randrange(1, R)
    rows["d_tree_double"] = (_sparse({0: s0, 1: _div(s0 * lag[0], lag[1])}), lambda m: (1, 0, "double") in m["tree"])
    s127 = rng.randrange(1, R)
    rows["d_tree_cancel"] = (_sparse({127: s127, 255: (-_div(s127 * lag[127], lag[255])) % R}),
                             lambda m: (128, 127, "cancel") in m["tree"] and m["finish"] == "identity")

    # f, sparse: structured scalars at the five threads (negative digits and carries in every window)
    rows["f_structured_sparse"] = (_sparse({0: R - 1, 1: (1 << 254) - 1, 127: int("80" * 31, 16), 128: int("81" * 31, 16),
                                            255: R - 2, 256 + 255: (1 << 254) - 1}),
                                   lambda m: m["value"] is not None and (128, 0, "generic") in m["tree"])
    return rows


STRUCTURED = {"r-1": R - 1, "2^254-1": (1 << 254) - 1, "80": int("80" * 31, 16), "81": int("81" * 31, 16)}


def solved_blob(lag, rng, minus=None):
    """random elements with one solved so that p(tau) = 0, or p(tau) = p(z) when minus = the Lagrange basis at z"""
    c = [(a - b) % R for a, b in zip(lag, minus)] if minus else lag
    s = [rng.randrange(R) for _ in range(N)]
    k = rng.randrange(N)
    s[k] = 0
    s[k] = (-_div(sum(v * l for v, l in zip(s, c)), c[k])) % R
    return s


# ---------------------------------------------------------------- helpers

def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _fr(vals):
    return np.array([[(v >> (64 * k)) & M64 for k in range(4)] for v in vals], dtype=np.uint64).reshape(-1, 4)


def _int(limbs):
    return sum(int(t) << (64 * k) for k, t in enumerate(limbs))


def _blob(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "big") for v in vals), dtype=np.uint8).copy()


def _expected(coracle, models):
    """[value]G1 through the C oracle for each model: (points (n, 12), flags (n,)); rejected rows zeroed and flagged"""
    pts, inf = coracle.g1_mul_batch(_fr([m["value"] or 0 for m in models]))
    pts, inf = pts.copy(), inf.copy()
    for k, m in enumerate(models):
        if m["status"] != VALID:
            pts[k], inf[k] = 0, 1
    return pts, inf


@pytest.fixture(scope="module")
def sim():
    """The dev simulation with the MSM body (its own build: the staleness list covers every device header)."""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_kzg_msm.so")
    csrc = os.path.join(ROOT, "zkvm_pairings_b200", "csrc")
    src = [os.path.join(d, f) for f in ("sim_kzg_msm.cpp", "sim_kzg_prove.cpp", "sim_kzg_blob.cpp", "sim.cpp")] + \
        [os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")] + \
        [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src[0]])
    return ctypes.CDLL(so)


def run_sim_msm(sim, lag_points_brp, rows, pre=None):
    """k_kzg_msm's body over the rows (lists of 4096 ints): (points (n, 12), flags (n,), status (n,))"""
    blobs = np.stack([_blob(s) for s in rows])
    n = len(rows)
    out, inf, st = np.zeros((n, 12), np.uint64), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    pre = None if pre is None else np.asarray(pre, np.uint8)
    assert sim.sim_kzg_msm(_p(np.ascontiguousarray(lag_points_brp)), _p(blobs), _p(pre), ctypes.c_size_t(n), _p(out), _p(inf), _p(st)) == 0
    return out, inf, st


def _used_points(coracle, lag, rows):
    """the Lagrange points (bit-reversed order) of the bases the rows use, through the C oracle; zero elsewhere"""
    used = sorted({i for s in rows for i in range(N) if s[i]})
    pts = np.zeros((N, 12), np.uint64)
    got, inf = coracle.g1_mul_batch(_fr([lag[i] for i in used]))
    assert not inf.any()
    pts[used] = got
    return pts


def _cpu_setup():
    from zkvm_pairings_b200 import workloads
    tau = random.Random(0x35E7).randrange(1, R)
    return workloads.lagrange_at(tau, workloads.blob_domain())


# ---------------------------------------------------------------- CPU

def test_model_reaches_every_branch():
    """Each constructed row reaches the branch it was built for, and the rows together reach every label of the
    partial sums, the tree and the finish."""
    lag = _cpu_setup()
    rows = edge_rows(lag, random.Random(0xED6E))
    got = set()
    for name, (s, check) in rows.items():
        m = msm_model(s, lag)
        assert check(m), name
        got |= labels_of(m)
    assert got == ALL_LABELS, ALL_LABELS - got


def test_model_digits_sum_back():
    """The model's recoding is the kernel's: digits in [-127, 128] that sum back, no carry out of the top window."""
    rng = random.Random(0xD1)
    for s in list(STRUCTURED.values()) + [0, 1, 0x80, 0x81, 0xFF] + [rng.randrange(R) for _ in range(200)]:
        d = msm_digits(s)
        assert all(-127 <= x <= 128 for x in d) and sum(x << (8 * w) for w, x in enumerate(d)) == s
    assert msm_digits((1 << 254) - 1) == [-1] + [0] * 30 + [64]        # a carry out of every window below the top
    assert msm_digits(int("81" * 31, 16)) == [-127] + [-126] * 30 + [1]
    assert msm_digits(int("80" * 31, 16)) == [128] * 31 + [0]


def test_sim_msm_edge_rows_match_the_oracle(sim, coracle):
    """The MSM body of the simulation on the constructed rows, an element >= r and an earlier rejection, bit-exact
    against [model scalar]G1 from the C oracle: the identity as (0, 1) with the flag, rejected rows zeroed and
    flagged."""
    lag = _cpu_setup()
    rng = random.Random(0xED6E)
    rows = [s for s, _ in edge_rows(lag, rng).values()]
    bad = _sparse({0: rng.randrange(R), 5: R})
    rows += [bad, rows[0]]
    pre = [0] * (len(rows) - 1) + [BAD_POINT]
    models = [msm_model(s, lag) for s in rows]
    want, winf = _expected(coracle, models)
    got, inf, st = run_sim_msm(sim, _used_points(coracle, lag, rows), rows, pre)
    assert list(st) == [m["status"] for m in models[:-1]] + [BAD_POINT]
    want[-1], winf[-1] = 0, 1
    assert np.array_equal(got, want) and np.array_equal(inf, winf)
    identities = [k for k, m in enumerate(models) if m["finish"] == "identity"]
    assert identities and all(np.array_equal(got[k], IDENTITY) and inf[k] == 1 for k in identities)


# ---------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def prover(engine):
    """A seeded trusted setup with its prover setup, the Lagrange coefficients at tau in bit-reversed order and the
    setup's points in that order."""
    from zkvm_pairings_b200 import workloads
    tau, tg, lag = workloads.kzg_lagrange_setup(engine, seed=0xED6E)
    s = engine.kzg_setup(tg, lag)
    yield dict(tau=tau, s=s, lag=workloads.lagrange_at(tau, workloads.blob_domain()), points_brp=lag[BRP])
    s.close()


def _gpu_rows(lag):
    """(name -> scalars, name -> check): the constructed rows, the structured blobs, a blob with p(tau) = 0, random
    blobs and one with an element >= r"""
    rng = random.Random(0x6E0)
    edges = edge_rows(lag, rng)
    rows, checks = {k: v[0] for k, v in edges.items()}, {k: v[1] for k, v in edges.items()}
    for k, v in STRUCTURED.items():
        rows["f_full_" + k] = [v] * N
    rows["e_p_tau_zero"] = solved_blob(lag, rng)
    for k in range(2):
        rows["random%d" % k] = [rng.randrange(R) for _ in range(N)]
    bad = [rng.randrange(R) for _ in range(N)]
    bad[2049] = R + 5
    rows["element_ge_r"] = bad
    return rows, checks


@pytest.mark.gpu
def test_commitments_at_every_branch(engine, prover, coracle, sim):
    """Every row in one kzg_blob_to_commitment_batch equals [model scalar]G1 (C oracle), the rows together reach every
    label of the model, the sparse rows equal the simulation word for word, and the _dev entry point agrees."""
    import torch
    rows, checks = _gpu_rows(prover["lag"])
    names = list(rows)
    models = [msm_model(rows[k], prover["lag"]) for k in names]
    got = set()
    for k, m in zip(names, models):
        assert k not in checks or checks[k](m), k
        got |= labels_of(m)
    assert got == ALL_LABELS, ALL_LABELS - got
    e = names.index("e_p_tau_zero")
    assert models[e]["finish"] == "identity"
    blobs = np.stack([_blob(rows[k]) for k in names])
    c, ci, st = engine.kzg_blob_to_commitment_batch(prover["s"], blobs)
    want, winf = _expected(coracle, models)
    assert list(st) == [m["status"] for m in models] and st[-1] == BAD_SCALAR
    assert np.array_equal(c, want) and np.array_equal(ci, winf)
    assert np.array_equal(c[e], IDENTITY) and ci[e] == 1
    sparse = [k for k, n in enumerate(names) if n[0] in "abcd" or n == "f_structured_sparse"]
    sc, sci, sst = run_sim_msm(sim, prover["points_brp"], [rows[names[k]] for k in sparse])
    assert np.array_equal(sc, c[sparse]) and np.array_equal(sci, ci[sparse]) and np.array_equal(sst, st[sparse])
    n = len(names)
    db = torch.from_numpy(blobs).cuda()
    dc = torch.zeros((n, 12), dtype=torch.int64, device="cuda")
    dci = torch.zeros(n, dtype=torch.uint8, device="cuda")
    dst = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    engine.kzg_blob_to_commitment_dev(prover["s"], db, n, dc, dci, dst)
    torch.cuda.synchronize()
    assert np.array_equal(dc.cpu().numpy().view(np.uint64), c) and np.array_equal(dci.cpu().numpy(), ci)
    assert np.array_equal(dst.cpu().numpy(), st)


@pytest.mark.gpu
def test_proofs_that_are_the_identity(engine, prover, coracle):
    """compute_kzg_proof on a blob with p(tau) = p(z) has q(tau) = 0: pi is (0, 1) with the flag and verifies.
    compute_blob_kzg_proof on a blob with p(tau) = 0 hashes the identity commitment's 0xc0 encoding into z, and its
    proof [-y / (tau - z)]G1 verifies through the blob verifier."""
    from zkvm_pairings_b200 import workloads
    rng = random.Random(0x1DE7)
    s, lag, tau = prover["s"], prover["lag"], prover["tau"]
    domain = workloads.blob_domain()
    z = rng.randrange(R)
    lz = workloads.lagrange_at(z, domain)
    poly = solved_blob(lag, rng, minus=lz)
    y = sum(v * l for v, l in zip(poly, lz)) % R
    assert y == sum(v * l for v, l in zip(poly, lag)) % R
    blob = _blob(poly)[None]
    c, ci, cst = engine.kzg_blob_to_commitment_batch(s, blob)
    pi, pinf, py, st = engine.kzg_compute_proof_batch(s, blob, _fr([z]))
    assert cst[0] == VALID and st[0] == VALID and _int(py[0]) == y
    assert pinf[0] == 1 and np.array_equal(pi[0], IDENTITY)
    vst = engine.kzg_verify_batch(s, np.concatenate([c, pi], axis=1), np.concatenate([_fr([z]), py], axis=1),
                                  np.stack([ci, pinf], axis=1))
    assert vst[0] == VALID

    e = solved_blob(lag, rng)
    eb = _blob(e)[None]
    c, ci, cst = engine.kzg_blob_to_commitment_batch(s, eb)
    assert cst[0] == VALID and ci[0] == 1 and np.array_equal(c[0], IDENTITY)
    pi, pinf, st, zy = engine.kzg_compute_blob_proof_batch(s, eb, c, ci, return_zy=True)
    assert st[0] == VALID
    z = _int(zy[0, :4])
    assert z == workloads.blob_challenge(eb.tobytes(), b"\xc0" + bytes(47))
    y = workloads.blob_eval(e, z, domain)
    assert _int(zy[0, 4:]) == y
    want, winf = coracle.g1_mul_batch(_fr([(-y) * pow((tau - z) % R, -1, R) % R]))
    assert np.array_equal(pi, want) and np.array_equal(pinf, winf)
    vst = engine.kzg_verify_blob_batch(s, eb, np.concatenate([c, pi], axis=1), np.stack([ci, pinf], axis=1))
    assert vst[0] == VALID
