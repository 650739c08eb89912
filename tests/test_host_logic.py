"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/zkpair.h
declares, fails loudly without a GPU (no CPU fallback), the generated constants agree with the
oracle, and the device code -- compiled as plain C++ with the PTX carry flag emulated
(tests/host_sim/sim.cpp, a DEV SIMULATION, never part of the product) -- is bit-exact against the
oracle for every tower op, the Miller loop, the final exponentiation and the point generator."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def lib():
    from zkvm_pairings_b200 import _lib, build
    build.build()
    return _lib.load()


def test_abi_exports_every_declared_symbol(lib):
    from zkvm_pairings_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "zkpair.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(zkp_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.zkp_version()


def test_no_cuda_device_fails_loudly(lib):
    """Without a GPU the product path must raise -- never fall back to a CPU implementation."""
    import zkvm_pairings_b200 as z
    if z.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(z.ZkpError) as ei:
        z.PairingEngine()
    assert ei.value.code == -4


def test_precompile_shaped_calls_have_no_cpu_path(lib):
    """zkp_sys_bigint / zkp_syscall_fp_mulmod (the reference's zkVM precompile FFI, src/fp.rs:126,376,443): argument
    checks happen on the host; without a GPU the process-wide context cannot be created and the call fails with
    ZKP_ERR_NO_DEVICE -- it never computes on the CPU."""
    import zkvm_pairings_b200 as z
    a = np.arange(1, 13, dtype=np.uint32)
    out = np.zeros(12, dtype=np.uint32)
    assert lib.zkp_sys_bigint(None, None, 0, _p(a), _p(a)) == -1
    assert lib.zkp_sys_bigint(None, _p(out), 7, _p(a), _p(a)) == -1 and b"op" in lib.zkp_last_error()
    assert lib.zkp_syscall_fp_mulmod(None, None, _p(a)) == -1
    if z.device_count() == 0:
        assert lib.zkp_sys_bigint(None, _p(out), 0, _p(a), _p(a)) == -4
        assert lib.zkp_syscall_fp_mulmod(None, _p(out), _p(a)) == -4
        assert not out.any()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "zkvm_pairings_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "coracle" not in text and "pyref" not in text and "zkp_oracle" not in text, f
                assert "host_sim" not in text or f in ("fp.cuh", "ops.cuh"), f   # only comments pointing at the test sim


def test_generated_constants_match_oracle(pyref, coracle):
    o = pyref
    text = open(os.path.join(ROOT, "zkvm_pairings_b200", "csrc", "consts.cuh")).read()

    def arr(name):
        m = re.search(r"%s\[\d+\] = \{(.*?)\};" % name, text, re.S)
        w = [int(x, 16) for x in re.findall(r"0x([0-9a-f]{8})u", m.group(1))]
        return [sum(w[12 * i + j] << (32 * j) for j in range(12)) for i in range(len(w) // 12)]

    R = o.R_MONT                   # the device Montgomery radix is the reference's R = 2^384 mod p (src/common.rs:150-157)
    assert R == (1 << 384) % o.P
    assert arr("ZKP_P") == [o.P] and arr("ZKP_ONE") == [R] and arr("ZKP_R2") == [R * R % o.P]
    assert arr("ZKP_2P") == [2 * o.P] and arr("ZKP_2P1") == [2 * o.P + 1] and arr("ZKP_4P1") == [4 * o.P + 1]
    n0 = int(re.search(r"#define ZKP_N0INV 0x([0-9a-f]+)u", text).group(1), 16)
    assert (n0 * o.P + 1) % (1 << 32) == 0
    r2, f61, f62, f121 = coracle.constants()
    assert util.arr_fp(r2)[0] == o.R_MONT * o.R_MONT % o.P
    frob = arr("ZKP_FROB")
    unmont = lambda v: v * pow(R, -1, o.P) % o.P
    g = [(unmont(frob[2 * i]), unmont(frob[2 * i + 1])) for i in range(15)]
    assert g[0] == o.FROB12_C1 and g[1] == o.FROB6_C1 and g[3] == o.FROB6_C2      # gamma_{1,1}, gamma_{1,2}, gamma_{1,4}
    assert tuple(util.arr_fp(f121)) == g[0] and tuple(util.arr_fp(f61)) == g[1] and tuple(util.arr_fp(f62)) == g[3]
    for k in (1, 2, 3):
        base = o.fp2_pow_vartime((1, 1), o._to_limbs((o.P ** k - 1) // 6, 6 * k))
        acc = o.FP2_ONE
        for i in range(5):
            acc = o.fp2_mul(acc, base)
            assert g[5 * (k - 1) + i] == acc
    assert [unmont(v) for v in arr("ZKP_G1_GEN")] == [o.G1_X, o.G1_Y]
    assert [unmont(v) for v in arr("ZKP_G2_GEN")] == [o.G2_X0, o.G2_X1, o.G2_Y0, o.G2_Y1]
    assert [unmont(v) for v in arr("ZKP_PSI")] == [o.PSI_COEFF_X[0], o.PSI_COEFF_X[1], o.PSI_COEFF_Y[0], o.PSI_COEFF_Y[1]]
    assert [unmont(v) for v in arr("ZKP_BETA")] == [o.BETA]


def test_op_widths():
    from zkvm_pairings_b200 import op_widths
    assert op_widths("fp_mul") == (1, 1, 1) and op_widths("fp_inv") == (1, 0, 1)
    assert op_widths("fp12_mul_by_014") == (12, 6, 12) and op_widths("fp6_mul_by_01") == (6, 4, 6)
    assert op_widths("fp12_frob2") == (12, 0, 12) and op_widths("fp2_mul_nr") == (2, 0, 2)
    assert op_widths("fp12_pow") == (12, 1, 12) and op_widths("fp_sqrt") == (1, 0, 1)


# ---------------------------------------------------------------- dev simulation of the device code

@pytest.fixture(scope="module")
def sim():
    d = os.path.join(ROOT, "tests", "host_sim")
    # ZKP_SIM_DEFINES="-DNAME ..." runs the same tests against a build variant of the device headers
    defs = os.environ.get("ZKP_SIM_DEFINES", "").split()
    so = os.path.join(d, "libzkpair_sim%s.so" % ("_" + re.sub(r"\W+", "_", "".join(defs)) if defs else ""))
    src = [os.path.join(d, "sim.cpp")] + [os.path.join(ROOT, "zkvm_pairings_b200", "csrc", f)
                                          for f in ("fp.cuh", "tower.cuh", "pairing.cuh", "ops.cuh", "consts.cuh")] + \
        [os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared"] + defs + ["-o", so, src[0]])
    return ctypes.CDLL(so)


def test_integration_doc_lists_every_entry_point():
    """INTEGRATION.md section 3 (the Rust `extern "C"` block a maintainer pastes) is the output of
    tools/gen_rust_ffi.py for the current header: every declared entry point, with its current signature."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_rust_ffi.py")], capture_output=True, text=True, check=True).stdout
    doc = re.sub(r"\s+", " ", open(os.path.join(ROOT, "INTEGRATION.md")).read())
    lines = [l.strip() for l in out.splitlines() if l.strip().startswith("pub fn")]
    assert len(lines) >= 39
    for l in lines:
        assert re.sub(r"\s+", " ", l) in doc, l


def test_sim_tower_ops_bit_exact(sim, coracle, pyref):
    from zkvm_pairings_b200 import TOWER_OPS, op_widths
    for name, code in TOWER_OPS.items():
        na, nb, nr = op_widths(name)
        if name in util.POW_OPS:
            n = {"fp_pow": 8, "fp2_pow": 6, "fp12_pow": 2, "fp_sqrt": 8}[name]
            a, b, exp, exp_status = util.pow_sqrt_case(pyref, name, n, seed=code)
            out, st = np.zeros((n, 6 * nr), np.uint64), np.zeros(n, np.uint8)
            sim.sim_tower_op(code, _p(a), _p(b), _p(out), _p(st), ctypes.c_size_t(n))
            assert np.array_equal(st, exp_status), name
            if name == "fp_sqrt":
                assert all(r is None or g in (r, pyref.P - r) for g, r in zip(util.arr_fp(out), exp))
            else:
                assert np.array_equal(out, exp), name
            continue
        n = 14
        a = util.random_fp_matrix(n, na, seed=code + 1)
        b = util.random_fp_matrix(n, nb, seed=code + 101) if nb else None
        out = np.zeros((n, 6 * nr), np.uint64)
        st = np.zeros(n, np.uint8)
        sim.sim_tower_op(code, _p(a), _p(b), _p(out), _p(st), ctypes.c_size_t(n))
        if name in ("fp12_frob2", "fp12_frob3"):
            exp = a
            for _ in range(int(name[-1])):
                exp = coracle.tower_op("fp12_frob", exp)
        else:
            exp = coracle.tower_op(name, a, b)
        assert np.array_equal(out, exp), name
        assert not (st & 1).any()
        if name.endswith("_inv"):
            assert st[0] == 2 and not st[3:].any()   # row 0 is all-zero: inverse of zero flagged


def test_sim_montgomery_edge_operands(sim, coracle, pyref):
    """Operands at the bounds the lazy-reduction analysis in fp.cuh relies on."""
    P = pyref.P
    vals = [0, 1, P - 1, P - 2, (1 << 381) - 1 if (1 << 381) - 1 < P else P - 3, pyref.R_MONT, P // 2, P // 3]
    a = util.fp_arr([x for x in vals for _ in vals]).reshape(-1, 6)
    b = util.fp_arr([y for _ in vals for y in vals]).reshape(-1, 6)
    out = np.zeros_like(a)
    sim.sim_tower_op(3, _p(a), _p(b), _p(out), None, ctypes.c_size_t(a.shape[0]))
    assert util.arr_fp(out) == [x * y % P for x in vals for y in vals]


def test_sim_rejects_noncanonical(sim, pyref):
    a = util.fp_arr([pyref.P, pyref.P + 5, (1 << 384) - 1, pyref.P - 1]).reshape(-1, 6)
    out, st = np.zeros_like(a), np.zeros(4, np.uint8)
    sim.sim_tower_op(2, _p(a), None, _p(out), _p(st), ctypes.c_size_t(4))
    assert list(st & 1) == [1, 1, 1, 0]


def test_sim_pairing_golden_vectors(sim, pyref):
    vec = util.golden("pairing_vectors.json")
    cases = vec["pairings"]
    g1 = np.stack([util.g1_to_arr(util.hex_g1(c["g1"])) for c in cases])
    g2 = np.stack([util.g2_to_arr(util.hex_g2(c["g2"])) for c in cases])
    i1 = np.array([c["g1"]["inf"] for c in cases], dtype=np.uint8)
    i2 = np.array([c["g2"]["inf"] for c in cases], dtype=np.uint8)
    n = len(cases)
    ml, gt = np.zeros((n, 72), np.uint64), np.zeros((n, 72), np.uint64)
    assert sim.sim_pairing(1, _p(g1), _p(i1), _p(g2), _p(i2), ctypes.c_size_t(n), 1, None, _p(ml), None) == 0
    assert sim.sim_pairing(3, _p(g1), _p(i1), _p(g2), _p(i2), ctypes.c_size_t(n), 1, None, _p(gt), None) == 0
    fe = np.zeros((n, 72), np.uint64)
    assert sim.sim_pairing(2, None, None, None, None, ctypes.c_size_t(n), 1, _p(ml), _p(fe), None) == 0
    for k, c in enumerate(cases):
        assert util.arr_to_fp12(ml[k]) == util.hex_fp12(c["miller_loop"]), k
        assert util.arr_to_fp12(gt[k]) == util.hex_fp12(c["pairing"]), k
    assert np.array_equal(fe, gt)
    assert pyref.fp12_sha256(util.arr_to_fp12(gt[0])) != ""
    for chk in vec["multi"]:
        a1 = np.stack([util.g1_to_arr(util.hex_g1(x["g1"])) for x in chk["pairs"]])
        a2 = np.stack([util.g2_to_arr(util.hex_g2(x["g2"])) for x in chk["pairs"]])
        out, one = np.zeros((1, 72), np.uint64), np.zeros(1, np.uint8)
        assert sim.sim_pairing(3, _p(a1), None, _p(a2), None, ctypes.c_size_t(1), 4, None, _p(out), _p(one)) == 0
        assert util.arr_to_fp12(out[0]) == util.hex_fp12(chk["gt"]) and bool(one[0]) == chk["is_one"]


def test_sim_point_generator_matches_oracle(sim, coracle):
    seed, first, n = 0x5EED, 7, 6
    a, b = util.scalars_for(seed, first, n)
    sim.sim_splitmix64_at.restype = ctypes.c_uint64
    assert sim.sim_splitmix64_at(ctypes.c_uint64(seed), ctypes.c_uint64(2 * first)) == a[0]
    k1, k2 = np.array(a, np.uint64), np.array(b, np.uint64)
    g1, g2 = np.zeros((n, 12), np.uint64), np.zeros((n, 24), np.uint64)
    i1, i2 = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    sim.sim_gen_points(_p(k1), _p(k2), ctypes.c_size_t(n), _p(g1), _p(i1), _p(g2), _p(i2))
    e1, ei1, e2, ei2 = util.oracle_points(coracle, seed, first, n)
    assert np.array_equal(g1, e1) and np.array_equal(g2, e2) and not i1.any() and not i2.any()
    for j in range(n):
        assert coracle.group_op("g1", "on_curve", g1[j]) and coracle.group_op("g2", "on_curve", g2[j])
    assert coracle.group_op("g2", "torsion_free", g2[0]) and coracle.group_op("g1", "torsion_free", g1[0])


def test_sim_group_checks_and_scalar_mul(sim, coracle, pyref):
    """SURVEY 8f rows: G1/G2 is_valid semantics (src/g1.rs:49-62, src/g2.rs:57-69) and scalar
    multiplication (src/g1.rs:130-153, src/g2.rs:185-208) of the device code vs the oracle."""
    g1, i1, e1, g2, i2, e2 = util.group_check_cases(pyref, coracle)
    st1, st2 = np.full(len(e1), 9, np.uint8), np.full(len(e2), 9, np.uint8)
    assert sim.sim_group_op(0, _p(g1), _p(i1), None, None, _p(st1), ctypes.c_size_t(len(e1))) == 0
    assert sim.sim_group_op(1, _p(g2), _p(i2), None, None, _p(st2), ctypes.c_size_t(len(e2))) == 0
    assert list(st1) == list(e1) and list(st2) == list(e2)
    for j in range(len(e1)):      # the C oracle agrees with the expectation the Python oracle produced
        if not i1[j]:
            assert coracle.group_op("g1", "on_curve", g1[j]) == (e1[j] != 1)
    n = 9
    k = util.random_scalars(n, seed=5)
    b1, bi1, b2, bi2 = util.oracle_points(coracle, 0xBEEF, 3, n)
    bi1[2] = 1                                      # identity base stays the identity
    o1, f1 = np.zeros((n, 12), np.uint64), np.zeros(n, np.uint8)
    o2, f2 = np.zeros((n, 24), np.uint64), np.zeros(n, np.uint8)
    assert sim.sim_group_op(2, _p(b1), _p(bi1), _p(k), _p(o1), _p(f1), ctypes.c_size_t(n)) == 0
    assert sim.sim_group_op(3, _p(b2), _p(bi2), _p(k), _p(o2), _p(f2), ctypes.c_size_t(n)) == 0
    x1, xf1 = coracle.g1_mul_batch(k, b1, bi1)
    x2, xf2 = coracle.g2_mul_batch(k, b2, bi2)
    assert np.array_equal(f1, xf1) and np.array_equal(f2, xf2)
    assert np.array_equal(o1[f1 == 0], x1[xf1 == 0]) and np.array_equal(o2[f2 == 0], x2[xf2 == 0])
    assert f1[0] == 1 and f1[2] == 1 and f1[5] == 1 and f2[5] == 1     # k = 0, identity base, k = r


def test_sim_prepared_g2_tables(sim, coracle):
    """SURVEY 8f-4: Miller loop over prepared line tables == the plain multi-pairing, bit for bit
    (k = 4 with the last 3 pairs prepared, k = 2 all prepared, a prepared pair at infinity)."""
    nc, k, kf = 3, 4, 3
    g1, _, g2all, _ = util.oracle_points(coracle, 0xABCD, 0, nc * k)
    fixed = g2all[:kf].copy()                                   # the shared "verifying-key" points
    g2 = g2all.reshape(nc, k, 24).copy()
    g2[:, k - kf:, :] = fixed                                   # every check ends with the same kf G2 points
    tab = np.zeros((kf, 68 * 3 * 12), np.uint64)
    sim.sim_g2_prepare(_p(fixed), ctypes.c_size_t(kf), _p(tab))
    var = np.ascontiguousarray(g2[:, :k - kf, :]).reshape(-1, 24)
    out, one = np.zeros((nc, 72), np.uint64), np.zeros(nc, np.uint8)
    assert sim.sim_pairing_prepared(_p(g1), None, _p(var), None, ctypes.c_size_t(nc), k, _p(tab), None, kf, _p(out), _p(one)) == 0
    exp, exp_one = coracle.multi_pairing_batch(g1, None, g2.reshape(-1, 24), None, k)
    assert np.array_equal(out, exp) and np.array_equal(one, exp_one)
    # all pairs prepared, one table flagged as the point at infinity
    ti = np.array([0, 1], np.uint8)
    out2 = np.zeros((1, 72), np.uint64)
    assert sim.sim_pairing_prepared(_p(g1[:2]), None, None, None, ctypes.c_size_t(1), 2, _p(tab[:2]), _p(ti), 2, _p(out2), None) == 0
    exp2, _ = coracle.multi_pairing_batch(g1[:2], None, fixed[:2], ti, 2)
    assert np.array_equal(out2, exp2)


def test_sim_group_addition(sim, coracle):
    """`&G1Affine + &G1Affine` / `&G2Affine + &G2Affine` (src/g1.rs:155-187, src/g2.rs:210-242): every branch of the
    affine law in the device code vs the oracle; P + (-P), where the reference panics, is flagged."""
    for gop, group, (a, ai, b, bi) in zip((4, 5), ("g1", "g2"), util.group_add_cases(coracle)):
        n, w = a.shape
        out, flag = np.zeros((n, w), np.uint64), np.full(n, 9, np.uint8)
        assert sim.sim_group_add(gop, _p(a), _p(ai), _p(b), _p(bi), _p(out), _p(flag), ctypes.c_size_t(n)) == 0
        exp, einf, pan = util.oracle_group_add(coracle, group, a, ai, b, bi)
        assert np.array_equal(flag & 1, einf) and np.array_equal((flag & 2) != 0, pan)
        keep = einf == 0
        assert np.array_equal(out[keep], exp[keep])
        assert pan.sum() == 1 and einf.sum() == 2       # P + (-P) and identity + identity


def test_sim_final_exponentiation_edge_inputs(sim, coracle, pyref):
    """The staged final exponentiation (compressed squarings, factorised hard part) on inputs that are not
    Miller-loop outputs -- zero, one, subfield elements (degenerate decompression), random Fp12 -- against the
    C oracle's plain Granger-Scott chain, and against the big-int oracle on two of them."""
    f = util.final_exp_edge_inputs()
    n = f.shape[0]
    out = np.zeros((n, 72), np.uint64)
    one = np.zeros(n, np.uint8)
    assert sim.sim_pairing(2, None, None, None, None, ctypes.c_size_t(n), 1, _p(f), _p(out), _p(one)) == 0
    exp = coracle.final_exp_batch(f)
    assert np.array_equal(out, exp)
    assert not out[0].any()                                   # zero maps to zero
    assert list(one[:6]) == [0, 1, 1, 1, 1, 1]                # subfield elements die in the easy part
    for j in (7, n - 1):
        assert util.arr_to_fp12(out[j]) == pyref.final_exponentiation(util.arr_to_fp12(f[j]))


def test_sim_batch_inversion(sim, coracle, pyref):
    """fp_batch_inv (Montgomery's trick, used between the two final-exponentiation launches): equal to
    element-wise Fermat inversion, zeros stay zero and do not poison their run, ragged last run."""
    n = 37
    a = util.random_fp_matrix(n, 1, seed=77)
    a[0] = 0
    a[5] = 0
    a[16] = util.fp_arr([1]).reshape(-1, 6)[0]
    a[36] = util.fp_arr([pyref.P - 1]).reshape(-1, 6)[0]
    out = np.zeros_like(a)
    sim.sim_batch_inv(_p(a), _p(out), ctypes.c_size_t(n), 16)
    vals = util.arr_fp(a)
    assert util.arr_fp(out) == [pow(v, pyref.P - 2, pyref.P) for v in vals]
    assert util.arr_fp(out)[0] == 0 and util.arr_fp(out)[16] == 1


def _sim_variant(defs):
    """the dev simulation built with extra -D flags (a build variant of the device headers)"""
    d = os.path.join(ROOT, "tests", "host_sim")
    so = os.path.join(d, "libzkpair_sim_%s.so" % re.sub(r"\W+", "_", "".join(defs)))
    src = [os.path.join(d, "sim.cpp")] + [os.path.join(ROOT, "zkvm_pairings_b200", "csrc", f)
                                          for f in ("fp.cuh", "tower.cuh", "pairing.cuh", "ops.cuh", "consts.cuh")] + \
        [os.path.join(ROOT, "tests", "device_harness", "bodies.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared"] + list(defs) + ["-o", so, src[0]])
    return ctypes.CDLL(so)


def test_sim_fp6_bodies_at_the_vertices_of_the_operand_box(sim):
    """fp6_mul / fp6_mul_by_01 / fp4_square with every operand representative next to 0 or next to 2p (all 2^12 / 2^10 /
    2^4 combinations) against the schoolbook formulas: the operand-bound asserts inside must hold at the extremes."""
    for what in (0, 1, 2):
        assert sim.sim_vertex_check(what) == 0


MILLER_MACS_LAZY3 = 1841352   # wide + narrow MACs of one Miller loop with ZKP_LAZY = 3 (both lanes; reduced forms: 2041032)


def test_sim_lazy_reduction_variant(coracle, pyref):
    """The lazy-reduction build variant (-DZKP_LAZY=7, tower.cuh: unreduced Fp2 products recombined as 768-bit integers,
    3 / 3 / 2 reductions per Fp6 product / sparse product / Fp4 square) computes the same field elements: worst-case
    operand vertices (where its bounds are tight), tower ops, golden pairing vectors, and the work it saves."""
    lazy = _sim_variant(["-DZKP_LAZY=7"])
    for what in (0, 1, 2):
        assert lazy.sim_vertex_check(what) == 0
    from zkvm_pairings_b200 import TOWER_OPS, op_widths
    for name in ("fp6_mul", "fp6_mul_by_01", "fp6_sqr", "fp12_mul", "fp12_sqr", "fp12_mul_by_014", "fp12_inv", "fp12_cyclotomic_sqr"):
        if name not in TOWER_OPS:
            continue
        code = TOWER_OPS[name]
        na, nb, nr = op_widths(name)
        n = 10
        a = util.random_fp_matrix(n, na, seed=code + 7)
        b = util.random_fp_matrix(n, nb, seed=code + 107) if nb else None
        out, st = np.zeros((n, 6 * nr), np.uint64), np.zeros(n, np.uint8)
        lazy.sim_tower_op(code, _p(a), _p(b), _p(out), _p(st), ctypes.c_size_t(n))
        assert np.array_equal(out, coracle.tower_op(name, a, b)), name
    g1, i1, g2, i2 = util.oracle_points(coracle, 0x5EED, 0, 3)
    ml, gt = np.zeros((3, 72), np.uint64), np.zeros((3, 72), np.uint64)
    assert lazy.sim_pairing(1, _p(g1), _p(i1), _p(g2), _p(i2), ctypes.c_size_t(3), 1, None, _p(ml), None) == 0
    assert lazy.sim_pairing(3, _p(g1), _p(i1), _p(g2), _p(i2), ctypes.c_size_t(3), 1, None, _p(gt), None) == 0
    assert np.array_equal(ml, coracle.miller_loop_batch(g1, i1, g2, i2)) and np.array_equal(gt, coracle.pairing_batch(g1, i1, g2, i2))
    lazy.sim_take_mac_count.restype = ctypes.c_uint64
    lazy.sim_take_mac_count()
    lazy.sim_pairing(1, _p(g1), None, _p(g2), None, ctypes.c_size_t(1), 1, None, _p(ml), None)
    miller = lazy.sim_take_mac_count()
    lazy.sim_pairing(2, None, None, None, None, ctypes.c_size_t(1), 1, _p(ml), _p(gt), None)
    fexp = lazy.sim_take_mac_count()
    assert (miller, fexp) == (MILLER_MACS_LAZY3, 1534416)   # reduced forms: 2041032 / 1829256 (test_sim_executed_mac_count)
    # the SHIPPED combination (pairing_kernel.cu ZKP_MILLER_LAZY = 3: lazy Fp6 products and line products in the Miller unit,
    # reduced forms in the final-exponentiation unit) executes 1841352 + 1829256 wide MACs per pairing in this accounting
    lazy3 = _sim_variant(["-DZKP_LAZY=3"])
    lazy3.sim_take_mac_count.restype = ctypes.c_uint64
    lazy3.sim_take_mac_count()
    ml3 = np.zeros((3, 72), np.uint64)
    assert lazy3.sim_pairing(1, _p(g1), _p(i1), _p(g2), _p(i2), ctypes.c_size_t(3), 1, None, _p(ml3), None) == 0
    assert lazy3.sim_take_mac_count() == 3 * MILLER_MACS_LAZY3 and np.array_equal(ml3, coracle.miller_loop_batch(g1, i1, g2, i2))
    src = open(os.path.join(ROOT, "zkvm_pairings_b200", "csrc", "pairing_kernel.cu")).read()
    assert re.search(r"#define ZKP_MILLER_LAZY 3\b", src) and "#define ZKP_LAZY ZKP_MILLER_LAZY" in src


def test_sim_executed_mac_count(sim, coracle):
    """Work accounting behind bench.py's `executed_macs_per_pairing`: the dev simulation counts the
    32x32->64 MACs both lanes issue (300 per Montgomery product, 444 per two-product form)."""
    sim.sim_take_mac_count.restype = ctypes.c_uint64
    g1, _, g2, _ = util.oracle_points(coracle, 0x5EED, 0, 4)
    out, ml = np.zeros((1, 72), np.uint64), np.zeros((1, 72), np.uint64)
    sim.sim_take_mac_count()
    sim.sim_pairing(1, _p(g1), None, _p(g2), None, ctypes.c_size_t(1), 1, None, _p(ml), None)
    miller = sim.sim_take_mac_count()
    sim.sim_pairing(2, None, None, None, None, ctypes.c_size_t(1), 1, _p(ml), _p(out), None)
    fexp = sim.sim_take_mac_count()
    sim.sim_pairing(3, _p(g1), None, _p(g2), None, ctypes.c_size_t(1), 4, None, _p(out), None)
    check4 = sim.sim_take_mac_count()
    # the one-call path runs its six Fp inversions in the lane: binary-GCD inversions (tower.cuh fp_inv) issue no
    # multiplications except the one product that takes the result back to Montgomery form
    # (check4 runs the FUSED path: homogeneous line steps, 2 Fp2 squarings fewer per doubling step than SURVEY 9.1's)
    assert (miller, fexp, check4) == (2041032, 1829256, 7742640)
    fused_saving = 63 * 2 * 600 + 5 * ((7 * 888 + 8 * 600) - (11 * 888 + 2 * 600))   # per pair: 63 doublings, 5 additions
    assert 8046000 - check4 == 4 * fused_saving
    a, o, st = util.random_fp_matrix(1, 1, seed=3), np.zeros((1, 6), np.uint64), np.zeros(1, np.uint8)
    sim.sim_tower_op(5, _p(a), None, _p(o), _p(st), ctypes.c_size_t(1))
    assert sim.sim_take_mac_count() == 600           # both lanes: one Montgomery product each (the Fermat ladder was 2 x 608 x 300)
    # bench.py's `executed_macs_per_pairing` is now an ncu opcode count of the shipped build (profiles/executed_work.json,
    # written by tools/ncu_executed_work.py); the simulation's arithmetic must agree with that counter: the staged GPU path
    # replaces the six in-lane ladders by batched inversions (12,300 MACs per pairing each) and 288 of every 300 MACs of a
    # Montgomery product are wide (the other 12 are the 32-bit m = t0 * n0' products)
    import json
    prof = json.load(open(os.path.join(ROOT, "profiles", "executed_work.json")))
    # staged GPU path: the six in-lane inversions (600 each) become batched ones (Montgomery's trick over runs of 16:
    # 45 products + one inversion per run = 46 x 300 / 16 per pairing), plus 20 boundary conversions
    # (the SHIPPED Miller unit runs the lazy forms, pairing_kernel.cu ZKP_MILLER_LAZY = 3: MILLER_MACS_LAZY3 instead of `miller`;
    # test_sim_lazy_reduction_variant pins that count on the variant build and checks the define)
    model = (MILLER_MACS_LAZY3 - fused_saving + fexp - 6 * 600 + 6 * 46 * 300 // 16 + 6000) * 288.0 / 300.0
    assert abs(prof["executed_wide_macs_per_pairing"] / model - 1.0) < 0.05, (prof["executed_wide_macs_per_pairing"], model)


def test_sim_operand_bounds_are_asserted(sim):
    """The dev simulation aborts (ZKP_SIM_ASSERT) when a Montgomery product is handed an operand
    above the bound fp.cuh documents; every other sim test therefore also proves that no call site
    of the tower / pairing code exceeds those bounds on its inputs (the bounds depend on the call
    sites, not on the data: every add/sub corrects to [0, 2p])."""
    text = open(os.path.join(ROOT, "zkvm_pairings_b200", "csrc", "fp.cuh")).read()
    assert text.count("ZKP_SIM_ASSERT(") >= 3


def test_pyref_splitmix_matches_util(pyref):
    st, out = pyref.splitmix64(0x5EED)
    a, _ = util.scalars_for(0x5EED, 0, 1)
    assert out == a[0]


def test_groth16_workload_generator_against_oracle(coracle):
    """zkvm_pairings_b200.workloads.groth16_checks (BASELINE config 3 inputs) with the ORACLE standing in for the
    engine's point generator / scalar multiplications: valid checks multiply to one, the seeded corrupted ones do
    not, and the SplitMix scalars mirror zkp_gen_points."""
    import numpy as np

    import util
    from zkvm_pairings_b200 import workloads as w

    class OracleEngine:
        def gen_points(self, seed, first, n):
            return util.oracle_points(coracle, seed, first, n)

        def g1_mul_batch(self, pts, scalars, inf=None):
            return coracle.g1_mul_batch(scalars, pts, inf)

        def g2_mul_batch(self, pts, scalars, inf=None):
            return coracle.g2_mul_batch(scalars, pts, inf)

    a, b = w.gen_scalars(0x5EED, 1000, 50)
    ea, eb = util.scalars_for(0x5EED, 1000, 50)
    assert [int(x) for x in a] == ea and [int(x) for x in b] == eb
    wl = w.groth16_checks(OracleEngine(), 24, seed=0x77, corrupt_every=5, corrupt_at=2)
    assert wl["g1"].shape == (96, 12) and wl["g2"].shape == (96, 24) and wl["fixed"].shape == (3, 24)
    assert list(np.nonzero(~wl["expect_one"])[0]) == [2, 7, 12, 17, 22]
    gt, one = coracle.multi_pairing_batch(wl["g1"], None, wl["g2"], None, 4)
    assert np.array_equal(one.astype(bool), wl["expect_one"])
    # generators embedded in the workload module are the curve's (and the oracle's) generators
    import pyref
    assert w.G1_GEN == pyref.G1_GENERATOR[:2] and w.G2_GEN == pyref.G2_GENERATOR[:2] and w.R_ORDER == pyref.R_ORDER
