"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI
(libzkpair.so), against the CPU oracle on identical seeded inputs, against the committed golden
vectors, and -- at BASELINE.json's full batch sizes -- through size-independent properties
(bilinearity, product checks, Miller-product consistency).  Bit-exact everywhere (integer path)."""
import os

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

VEC = util.golden("pairing_vectors.json")
FULL = int(os.environ.get("ZKP_TEST_FULL_LOG2", "16"))     # BASELINE config[1]: 2^16 pairings


def _cases():
    cases = VEC["pairings"]
    g1 = np.stack([util.g1_to_arr(util.hex_g1(c["g1"])) for c in cases])
    g2 = np.stack([util.g2_to_arr(util.hex_g2(c["g2"])) for c in cases])
    i1 = np.array([c["g1"]["inf"] for c in cases], dtype=np.uint8)
    i2 = np.array([c["g2"]["inf"] for c in cases], dtype=np.uint8)
    return cases, g1, i1, g2, i2


def test_native_library_is_the_one_loaded(engine):
    from zkvm_pairings_b200 import _lib
    assert os.path.samefile(_lib.lib_path(), os.path.join(os.path.dirname(_lib.__file__), "libzkpair.so"))
    with open("/proc/self/maps") as f:
        assert "libzkpair.so" in f.read()
    assert "sm_100a" in engine.version()
    before = engine.launch_count
    engine.fp_mul_batch(util.fp_arr([3]), util.fp_arr([5]))
    assert engine.launch_count == before + 1


def test_fp_mul_known_answers(engine, pyref):
    P = pyref.P
    vals = [0, 1, 2, P - 1, P - 2, pyref.R_MONT, P // 2, (1 << 380) + 12345]
    a = util.fp_arr([x for x in vals for _ in vals]).reshape(-1, 6)
    b = util.fp_arr([y for _ in vals for y in vals]).reshape(-1, 6)
    out = engine.fp_mul_batch(a, b)
    assert util.arr_fp(out) == [x * y % P for x in vals for y in vals]


@pytest.mark.parametrize("name", sorted(__import__("zkvm_pairings_b200").TOWER_OPS))
def test_tower_op_matches_oracle(engine, coracle, pyref, name):
    from zkvm_pairings_b200 import TOWER_OPS, op_widths
    na, nb, nr = op_widths(name)
    if name in util.POW_OPS:
        n = {"fp_pow": 24, "fp2_pow": 12, "fp12_pow": 6, "fp_sqrt": 40}[name]
        a, b, exp, exp_status = util.pow_sqrt_case(pyref, name, n, seed=TOWER_OPS[name])
        out, status = engine.tower_op(name, a, b, return_status=True)
        assert np.array_equal(status, exp_status)
        if name == "fp_sqrt":      # a root where one exists (the reference returns Err(()) otherwise)
            got = util.arr_fp(out)
            assert all(r is None or g in (r, pyref.P - r) for g, r in zip(got, exp))
            assert got[0] == 0x025e51146a92917731d9d66d63f8c24ed8cae114e7c9d188e3eaa1e79bb19769f5877f9443e03723d9ed1eebbf92df98
        else:
            assert np.array_equal(out, exp)
        return
    n = 1000 if not name.endswith(("_inv", "cyc_exp")) else 200
    a = util.random_fp_matrix(n, na, seed=TOWER_OPS[name] + 1)
    b = util.random_fp_matrix(n, nb, seed=TOWER_OPS[name] + 101) if nb else None
    out, status = engine.tower_op(name, a, b, return_status=True)
    if name in ("fp12_frob2", "fp12_frob3"):
        exp = a
        for _ in range(int(name[-1])):
            exp = coracle.tower_op("fp12_frob", exp)
    else:
        exp = coracle.tower_op(name, a, b)
    assert np.array_equal(out, exp)
    assert not (status & 1).any()
    if name.endswith("_inv"):
        assert status[0] == 2 and not status[3:].any()


def test_empty_and_ragged_batches(engine, coracle):
    assert engine.fp_mul_batch(np.zeros((0, 6), np.uint64), np.zeros((0, 6), np.uint64)).shape == (0, 6)
    assert engine.pairing_batch(np.zeros((0, 12), np.uint64), np.zeros((0, 24), np.uint64)).shape == (0, 72)
    for n in (1, 31, 33, 129):     # not multiples of the warp / block size
        g1, i1, g2, i2 = util.oracle_points(coracle, 99, 0, n)
        assert np.array_equal(engine.miller_loop_batch(g1, g2), coracle.miller_loop_batch(g1, None, g2, None))
    with pytest.raises(ValueError):
        engine.multi_pairing_batch(np.zeros((5, 12), np.uint64), np.zeros((5, 24), np.uint64), 4)


def test_noncanonical_inputs_rejected(engine, pyref):
    from zkvm_pairings_b200 import NonCanonicalError
    g1 = util.g1_to_arr(pyref.G1_GENERATOR)[None].copy()
    g2 = util.g2_to_arr(pyref.G2_GENERATOR)[None]
    g1[0, 6:12] = util.fp_arr([pyref.P])
    with pytest.raises(NonCanonicalError):
        engine.pairing_batch(g1, g2)
    out, status = engine.tower_op("fp_neg", util.fp_arr([pyref.P - 1]), return_status=True)
    assert status[0] == 0
    with pytest.raises(NonCanonicalError):
        engine.tower_op("fp_neg", util.fp_arr([pyref.P]))
    # the context stays usable after an error
    assert util.arr_fp(engine.fp_mul_batch(util.fp_arr([3]), util.fp_arr([5]))) == [15]


def test_pairing_golden_vectors(engine, pyref):
    cases, g1, i1, g2, i2 = _cases()
    ml = engine.miller_loop_batch(g1, g2, i1, i2)
    gt = engine.pairing_batch(g1, g2, i1, i2)
    for k, c in enumerate(cases):
        assert util.arr_to_fp12(ml[k]) == util.hex_fp12(c["miller_loop"]), k
        assert util.arr_to_fp12(gt[k]) == util.hex_fp12(c["pairing"]), k
    gen = util.golden("pairing_vectors.json")["generators"]
    e = engine.pairing_batch(util.g1_to_arr(pyref.G1_GENERATOR), util.g2_to_arr(pyref.G2_GENERATOR))
    assert pyref.fp12_sha256(util.arr_to_fp12(e[0])) == gen["pairing_sha256"] == "06fa588b89fdfb034dbc1c163ecb3dfac228f552b643c7294cc5f2c4dc170b84"
    m = engine.miller_loop_batch(util.g1_to_arr(pyref.G1_GENERATOR), util.g2_to_arr(pyref.G2_GENERATOR))
    assert pyref.fp12_sha256(util.arr_to_fp12(m[0])) == "eceb6467936a62ed011881c3efceb3b9f05b6017afd264fa0caeebf4f8437115"
    assert np.array_equal(engine.final_exponentiation_batch(ml), gt)
    # infinity on either side gives Gt one (last two golden cases)
    assert util.arr_to_fp12(gt[-1]) == pyref.FP12_ONE and util.arr_to_fp12(gt[-2]) == pyref.FP12_ONE


def test_bilinearity_config0(engine, pyref):
    """BASELINE config[0]: e(aP, bQ) == e(P, Q)^(ab), with aP, bQ made by the ORACLE."""
    o = pyref
    e = util.arr_to_fp12(engine.pairing_batch(util.g1_to_arr(o.G1_GENERATOR), util.g2_to_arr(o.G2_GENERATOR))[0])
    for a, b in ((6, 11), (5, 7), (2, 3)):
        p, q = o.g1_mul(o.G1_GENERATOR, a), o.g2_mul(o.G2_GENERATOR, b)
        got = util.arr_to_fp12(engine.pairing_batch(util.g1_to_arr(p), util.g2_to_arr(q))[0])
        assert got == o.fp12_pow_int(e, a * b)


def test_point_generator_matches_oracle(engine, coracle):
    n = 300
    g1, i1, g2, i2 = engine.gen_points(0x5EED, 1000, n)
    e1, ei1, e2, ei2 = util.oracle_points(coracle, 0x5EED, 1000, n)
    assert np.array_equal(g1, e1) and np.array_equal(g2, e2)
    assert not i1.any() and not i2.any()


def test_batch_matches_oracle_seeded(engine, coracle):
    n = 2048
    g1, i1, g2, i2 = util.oracle_points(coracle, 0xC0FFEE, 0, n)
    i1[5] = 1
    i2[9] = 1
    assert np.array_equal(engine.miller_loop_batch(g1, g2, i1, i2), coracle.miller_loop_batch(g1, i1, g2, i2))
    gt = engine.pairing_batch(g1, g2, i1, i2)
    assert np.array_equal(gt, coracle.pairing_batch(g1, i1, g2, i2))


def test_multi_pairing_checks(engine, coracle, pyref):
    for chk in VEC["multi"]:
        a1 = np.stack([util.g1_to_arr(util.hex_g1(x["g1"])) for x in chk["pairs"]])
        a2 = np.stack([util.g2_to_arr(util.hex_g2(x["g2"])) for x in chk["pairs"]])
        out, one = engine.multi_pairing_batch(a1, a2, 4)
        assert util.arr_to_fp12(out[0]) == util.hex_fp12(chk["gt"]) and bool(one[0]) == chk["is_one"]
        mm = engine.multi_miller_loop_batch(a1, a2, 4)
        assert util.arr_to_fp12(mm[0]) == util.hex_fp12(chk["multi_miller"])
    # random checks of every supported width, with some infinities, vs the oracle
    for k in (1, 2, 3, 4, 5, 8):
        nchk = 40
        g1, i1, g2, i2 = util.oracle_points(coracle, 1234 + k, 0, nchk * k)
        i1[3] = 1
        out, one = engine.multi_pairing_batch(g1, g2, k, i1, i2)
        exp, eone = coracle.multi_pairing_batch(g1, i1, g2, i2, k)
        assert np.array_equal(out, exp) and np.array_equal(one, eone), k
    from zkvm_pairings_b200 import ZkpError
    with pytest.raises(ZkpError):
        engine.multi_pairing_batch(np.zeros((9, 12), np.uint64), np.zeros((9, 24), np.uint64), 9)


def test_groth16_style_checks_config3_small(engine, coracle, pyref):
    """4-pair checks e(A,B) e(-alpha,beta) e(-C,delta) e(-L,gamma): valid => one; 1% corrupted."""
    o = pyref
    nchk = 256
    rng = np.random.default_rng(3)
    sc = rng.integers(1, 1 << 20, size=(nchk, 6)).astype(object)
    k1, k2, bad = [], [], []
    for i in range(nchk):
        a, b, c, d, l, g = (int(x) for x in sc[i])
        # choose alpha*beta so the exponents cancel:  a*b - al*be - c*d - l*g = 0  (mod r)
        al, be = 1, (a * b - c * d - l * g) % o.R_ORDER
        corrupt = (i % 100) == 7
        bad.append(corrupt)
        if corrupt:
            l += 1
        k1 += [a, o.R_ORDER - al, o.R_ORDER - c, o.R_ORDER - l]
        k2 += [b, be, d, g]
    g1, i1 = coracle.g1_mul_batch(util.scalar_matrix(k1))
    g2, i2 = coracle.g2_mul_batch(util.scalar_matrix(k2))
    out, one = engine.multi_pairing_batch(g1, g2, 4, i1, i2)
    assert [not bool(x) for x in one] == bad
    exp, eone = coracle.multi_pairing_batch(g1, i1, g2, i2, 4)
    assert np.array_equal(out, exp) and np.array_equal(one, eone)


def test_multi_miller_product(engine, coracle):
    n = 700
    g1, i1, g2, i2 = util.oracle_points(coracle, 77, 0, n)
    ml, gt = engine.multi_miller_product(g1, g2)
    eml, egt = coracle.miller_product(g1, None, g2, None)
    assert np.array_equal(ml, eml) and np.array_equal(gt, egt)


def test_full_size_config1_bit_exact(engine, coracle):
    """BASELINE config[1]: 2^16 independent pairings, every Gt bit-exact against the oracle."""
    n = 1 << FULL
    g1, i1, g2, i2 = engine.gen_points(0x5EED5EED, 0, n)
    gt = engine.pairing_batch(g1, g2)
    step = max(1, n // (1 << 13)) if coracle.ncores() < 16 else 1    # whole batch when the host has the cores
    idx = np.arange(0, n, step)
    assert np.array_equal(gt[idx], coracle.pairing_batch(g1[idx], None, g2[idx], None))
    # size-independent property over the WHOLE batch: product of all Miller loops through the sharded
    # product path equals the product of the per-pair outputs
    ml = engine.miller_loop_batch(g1, g2)
    prod, gt_prod = engine.multi_miller_product(g1, g2)
    import torch
    d_in = torch.from_numpy(ml.view(np.int64)).cuda()
    scratch = torch.empty(engine.product_scratch_elems(n) * 72, dtype=torch.int64, device="cuda")
    d_out = torch.empty(72, dtype=torch.int64, device="cuda")
    engine.fp12_product_dev(d_in, n, scratch, d_out, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(d_out.cpu().numpy().view(np.uint64), prod)
    assert np.array_equal(engine.final_exponentiation_batch(prod[None])[0], gt_prod)


def test_metric_batch_2p20_properties(engine, coracle):
    """The metric's batch (2^20 pairings on one GPU) through size-independent properties, every element checked:
    bilinearity e([2]P, Q) == e(P, Q)^2 with [2]P from the group kernel and the square from the tower kernel,
    "checksum of checksums" prod_i e(P_i, Q_i) == final_exp(prod_i miller(P_i, Q_i)) through the product
    kernels, and a strided sample against the oracle."""
    import torch
    n = 1 << int(os.environ.get("ZKP_TEST_METRIC_LOG2", "20"))
    g1, i1, g2, i2 = engine.gen_points(0x2B200, 0, n)
    gt = engine.pairing_batch(g1, g2)
    two = np.zeros((n, 4), np.uint64)
    two[:, 0] = 2
    g1x2, inf2 = engine.g1_mul_batch(g1, two)
    assert not inf2.any()
    gt2 = engine.pairing_batch(g1x2, g2)
    assert np.array_equal(gt2, engine.tower_op("fp12_sqr", gt))
    idx = np.arange(0, n, n // 64)
    assert np.array_equal(gt[idx], coracle.pairing_batch(np.ascontiguousarray(g1[idx]), None, np.ascontiguousarray(g2[idx]), None))
    _, gt_prod = engine.multi_miller_product(g1, g2)
    st = torch.cuda.current_stream().cuda_stream
    d_in = torch.from_numpy(gt.view(np.int64)).cuda()
    scratch = torch.empty(engine.product_scratch_elems(n) * 72, dtype=torch.int64, device="cuda")
    d_out = torch.empty(72, dtype=torch.int64, device="cuda")
    engine.fp12_product_dev(d_in, n, scratch, d_out, stream=st)
    torch.cuda.synchronize()
    assert np.array_equal(d_out.cpu().numpy().view(np.uint64), gt_prod)


def test_full_size_final_exp_config2_properties(engine, coracle, pyref):
    """BASELINE config[2] shape (final exponentiation only) at 2^16 here: outputs lie in the order-r
    subgroup (checked on a sample via the oracle) and f -> f^2 commutes with the map."""
    n = 1 << min(FULL, 16)
    g1, i1, g2, i2 = engine.gen_points(0xABCDEF, 0, n)
    ml = engine.miller_loop_batch(g1, g2)
    fe = engine.final_exponentiation_batch(ml)
    sq = engine.tower_op("fp12_sqr", ml)
    fe_sq = engine.final_exponentiation_batch(sq)
    assert np.array_equal(fe_sq, engine.tower_op("fp12_sqr", fe))
    for j in (0, n // 2, n - 1):
        assert pyref.fp12_pow_int(util.arr_to_fp12(fe[j]), pyref.R_ORDER) == pyref.FP12_ONE
    idx = np.arange(0, n, max(1, n // 512))
    assert np.array_equal(fe[idx], coracle.final_exp_batch(ml[idx]))


def test_final_exponentiation_edge_inputs(engine, coracle, pyref):
    """Staged final exponentiation on inputs that are not Miller-loop outputs: zero, one, subfield elements
    (every decompression takes its degenerate branch), random Fp12; a ragged batch so that tail lanes and the
    two-stream split boundary are exercised too."""
    f = util.final_exp_edge_inputs(n_random=23)
    out = engine.final_exponentiation_batch(f)
    assert np.array_equal(out, coracle.final_exp_batch(f))
    assert not out[0].any()
    assert util.arr_to_fp12(out[1]) == pyref.FP12_ONE and util.arr_to_fp12(out[5]) == pyref.FP12_ONE
    # the same rows tiled past the split threshold (2^15 checks): both halves, odd size
    n = (1 << 15) + 77
    big = np.ascontiguousarray(np.tile(f, (n // f.shape[0] + 1, 1))[:n])
    outb = engine.final_exponentiation_batch(big)
    assert np.array_equal(outb[: f.shape[0]], out) and np.array_equal(outb[-f.shape[0]:], coracle.final_exp_batch(big[-f.shape[0]:]))
    assert np.array_equal(outb[n // 2 - 40: n // 2 + 40], coracle.final_exp_batch(big[n // 2 - 40: n // 2 + 40]))


def test_device_resident_path(engine, coracle):
    import torch
    n = 512
    g1, i1, g2, i2 = util.oracle_points(coracle, 4242, 0, n)
    st = torch.cuda.current_stream().cuda_stream
    dg1, dg2 = torch.from_numpy(g1.view(np.int64)).cuda(), torch.from_numpy(g2.view(np.int64)).cuda()
    out = torch.empty((n, 72), dtype=torch.int64, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    engine.pairing_dev(3, out, g1=dg1, g2=dg2, err=err, stream=st)
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    assert np.array_equal(out.cpu().numpy().view(np.uint64), coracle.pairing_batch(g1, None, g2, None))
    # generator on device == generator through host buffers
    a1 = torch.empty((n, 12), dtype=torch.int64, device="cuda")
    a2 = torch.empty((n, 24), dtype=torch.int64, device="cuda")
    f1 = torch.empty(n, dtype=torch.uint8, device="cuda")
    f2 = torch.empty(n, dtype=torch.uint8, device="cuda")
    engine.gen_points_dev(4242, 0, n, a1, f1, a2, f2, stream=st)
    torch.cuda.synchronize()
    assert np.array_equal(a1.cpu().numpy().view(np.uint64), g1) and np.array_equal(a2.cpu().numpy().view(np.uint64), g2)


def test_prepared_g2_tables(engine, coracle):
    """SURVEY 8f-4: G2Prepared-style line tables: Groth16-shaped checks (4 pairs, 3 verifying-key G2 points
    prepared once) equal the unprepared results and the oracle bit for bit, including corrupted checks."""
    nc, k, kf = 257, 4, 3
    g1, _, g2all, _ = engine.gen_points(0x6716, 0, nc * k)
    fixed = g2all[:kf].copy()
    g2 = g2all.reshape(nc, k, 24).copy()
    g2[:, k - kf:, :] = fixed
    tab = engine.g2_prepare_batch(fixed)
    assert tab.shape == (kf, 68 * 3 * 12)
    var = np.ascontiguousarray(g2[:, :k - kf, :]).reshape(-1, 24)
    gt, one = engine.multi_pairing_prepared_batch(g1, var, k, tab)
    ref, ref_one = engine.multi_pairing_batch(g1, g2.reshape(-1, 24), k)
    assert np.array_equal(gt, ref) and np.array_equal(one, ref_one)
    exp, _ = coracle.multi_pairing_batch(g1[:16 * k], None, g2.reshape(-1, 24)[:16 * k], None, k)
    assert np.array_equal(gt[:16], exp)
    # all pairs prepared (k = kf = 2), second table flagged infinite
    gt2, _ = engine.multi_pairing_prepared_batch(g1[:10], None, 2, tab[:2], tables_inf=np.array([0, 1], np.uint8))
    exp2, _ = coracle.multi_pairing_batch(g1[:10], None, np.tile(fixed[:2], (5, 1)), np.tile(np.array([0, 1], np.uint8), 5), 2)
    assert np.array_equal(gt2, exp2)


def test_fp_byte_serialisation(engine, pyref):
    """SURVEY 8f-2: Fp::from_bytes / to_bytes (src/fp.rs:165-207): big-endian, canonical check, round trip."""
    P = pyref.P
    vals = [0, 1, P - 1, P, P + 1, (1 << 384) - 1, 0x0102030405060708090a0b0c0d0e0f101112131415161718191a1b1c1d1e1f202122232425262728292a2b2c2d2e2f30]
    rng = np.random.default_rng(5)
    data = np.concatenate([np.frombuffer(b"".join(v.to_bytes(48, "big") for v in vals), np.uint8).reshape(-1, 48),
                           rng.integers(0, 256, size=(1000, 48), dtype=np.uint8)])
    limbs, ok = engine.fp_from_bytes_batch(data)
    for row, lim, k in zip(data, limbs, ok):
        v = int.from_bytes(row.tobytes(), "big")
        assert sum(int(x) << (64 * i) for i, x in enumerate(lim)) == v
        assert bool(k) == (pyref.fp_from_bytes(row.tobytes()) is not None) == (v < P)
    back = engine.fp_to_bytes_batch(limbs)
    assert np.array_equal(back, data)
    assert engine.fp_to_bytes_batch(util.fp_arr([5]).reshape(-1, 6)).tobytes() == pyref.fp_to_bytes(5)
    assert engine.fp_from_bytes_batch(np.zeros((0, 48), np.uint8))[0].shape == (0, 6)


def test_group_validity_checks(engine, coracle, pyref):
    """SURVEY 8f-1: G1Affine::is_valid / G2Affine::is_valid (src/g1.rs:49-62, src/g2.rs:57-69) batched."""
    g1, i1, e1, g2, i2, e2 = util.group_check_cases(pyref, coracle, n_valid=40)
    assert list(engine.g1_check_batch(g1, i1)) == list(e1)
    assert list(engine.g2_check_batch(g2, i2)) == list(e2)
    # a larger batch of valid points, ragged size, no infinity array
    a, _, b, _ = engine.gen_points(0x77, 0, 333)
    assert not engine.g1_check_batch(a).any() and not engine.g2_check_batch(b).any()
    b[17, 0] ^= np.uint64(1)
    st = engine.g2_check_batch(b)
    assert st[17] == 1 and st.sum() == 1
    from zkvm_pairings_b200 import ZkpError
    with pytest.raises(ZkpError):
        bad = a.copy()
        bad[3, :6] = util.fp_arr([pyref.P]).reshape(-1, 6)[0]
        engine.g1_check_batch(bad)


def test_group_scalar_mul_matches_oracle(engine, coracle):
    """SURVEY 8f-3: [k]P for 256-bit scalars (src/g1.rs:130-153 done correctly, src/g2.rs:185-208)."""
    n = 77
    k = util.random_scalars(n, seed=11)
    b1, bi1, b2, bi2 = util.oracle_points(coracle, 0xC0FFEE, 5, n)
    bi2[4] = 1
    o1, f1 = engine.g1_mul_batch(b1, k, bi1)
    o2, f2 = engine.g2_mul_batch(b2, k, bi2)
    x1, xf1 = coracle.g1_mul_batch(k, b1, bi1)
    x2, xf2 = coracle.g2_mul_batch(k, b2, bi2)
    assert np.array_equal(f1, xf1) and np.array_equal(f2, xf2)
    assert np.array_equal(o1[f1 == 0], x1[xf1 == 0]) and np.array_equal(o2[f2 == 0], x2[xf2 == 0])
    # bilinearity through the engine's own scalar multiplication: e([a]P, Q) == e(P, [a]Q)
    gt1 = engine.pairing_batch(o1[7:20], b2[7:20])
    gt2 = engine.pairing_batch(b1[7:20], o2[7:20])
    assert np.array_equal(gt1, gt2)


def test_group_addition_matches_oracle(engine, coracle):
    """zkp_g1_add_batch / zkp_g2_add_batch: every branch of the reference's affine law, and [2]P + P == [3]P
    against the scalar-multiplication kernel on a larger batch."""
    for group, add, (a, ai, b, bi) in zip(("g1", "g2"), (engine.g1_add_batch, engine.g2_add_batch), util.group_add_cases(coracle)):
        out, flag = add(a, b, ai, bi)
        exp, einf, pan = util.oracle_group_add(coracle, group, a, ai, b, bi)
        assert np.array_equal(flag & 1, einf) and np.array_equal((flag & 2) != 0, pan)
        assert np.array_equal(out[einf == 0], exp[einf == 0])
    n = 777
    g1, _, g2, _ = engine.gen_points(0x3A, 0, n)
    two, three = np.zeros((n, 4), np.uint64), np.zeros((n, 4), np.uint64)
    two[:, 0], three[:, 0] = 2, 3
    for pts, mul, add in ((g1, engine.g1_mul_batch, engine.g1_add_batch), (g2, engine.g2_mul_batch, engine.g2_add_batch)):
        dbl, _ = mul(pts, two)
        tri, _ = mul(pts, three)
        s, flag = add(dbl, pts)
        assert not flag.any() and np.array_equal(s, tri)
        d2, flag = add(pts, pts)                      # the tangent branch
        assert not flag.any() and np.array_equal(d2, dbl)


def test_config3_full_size_2p18_checks(engine, coracle):
    """BASELINE config[3] at its stated size: 2^18 Groth16-shaped 4-pair checks with a shared final
    exponentiation, a seeded 1 % of them corrupted.  Every is_one flag against the construction, the prepared
    (G2Prepared line tables for the three verifying-key points) path bit-identical to the plain one over the
    whole batch, and a strided sample of Gt values against the C oracle."""
    from zkvm_pairings_b200 import workloads
    n = 1 << int(os.environ.get("ZKP_TEST_CONFIG3_LOG2", "18"))
    wl = workloads.groth16_checks(engine, n)
    gt, one = engine.multi_pairing_batch(wl["g1"], wl["g2"], 4)
    assert np.array_equal(one.astype(bool), wl["expect_one"])
    assert wl["expect_one"].sum() == n - len(range(7, n, 100))
    tab = engine.g2_prepare_batch(wl["fixed"])
    gtp, onep = engine.multi_pairing_prepared_batch(wl["g1"], wl["g2_var"], 4, tab)
    assert np.array_equal(gtp, gt) and np.array_equal(onep, one)
    idx = np.unique(np.concatenate([np.arange(0, n, max(1, n // 48)), np.arange(7, n, max(100, 100 * (n // 1600)))]))
    g1s = np.ascontiguousarray(wl["g1"].reshape(n, 4, 12)[idx]).reshape(-1, 12)
    g2s = np.ascontiguousarray(wl["g2"].reshape(n, 4, 24)[idx]).reshape(-1, 24)
    exp, eone = coracle.multi_pairing_batch(g1s, None, g2s, None, 4)
    assert np.array_equal(gt[idx], exp) and np.array_equal(one[idx], eone)
    assert not eone.all() and eone.any()          # the sample holds valid and corrupted checks


def test_config2_full_size_2p20_final_exp_only(engine, coracle):
    """BASELINE config[2] at its stated size: the final exponentiation alone over 2^20 Miller-loop outputs:
    every element equal to the one-call pairing of the same points, a strided sample against the C oracle."""
    n = 1 << int(os.environ.get("ZKP_TEST_CONFIG2_LOG2", "20"))
    g1, _, g2, _ = engine.gen_points(0xFE20, 0, n)
    ml = engine.miller_loop_batch(g1, g2)
    fe = engine.final_exponentiation_batch(ml)
    assert np.array_equal(fe, engine.pairing_batch(g1, g2))
    idx = np.arange(0, n, n // 64)
    assert np.array_equal(fe[idx], coracle.final_exp_batch(np.ascontiguousarray(ml[idx])))
    assert np.array_equal(ml[idx], coracle.miller_loop_batch(np.ascontiguousarray(g1[idx]), None, np.ascontiguousarray(g2[idx]), None))


def test_multi_miller_product_grouping_and_chunks(engine, coracle):
    """zkp_multi_miller_product streams 2^18-pair chunks through two buffer sets and runs FOUR pairs per
    shared-accumulator Miller loop: sizes that leave a ragged group (n % 4 != 0), cross a chunk boundary, and
    carry points at infinity must give the same field element as the product of the per-pair outputs."""
    import torch
    for n, seed in ((1, 5), (3, 6), (6, 7), (1029, 8), ((1 << 18) + 5, 9)):
        g1, i1, g2, i2 = engine.gen_points(seed, 0, n)
        if n > 4:
            i1[2] = 1
            i2[n - 1] = 1
        prod, gt = engine.multi_miller_product(g1, g2, i1, i2)
        if n <= 2048:
            eml, egt = coracle.miller_product(g1, i1, g2, i2)
            assert np.array_equal(prod, eml) and np.array_equal(gt, egt), n
        ml = engine.miller_loop_batch(g1, g2, i1, i2)
        d_in = torch.from_numpy(ml.view(np.int64)).cuda()
        scratch = torch.empty(engine.product_scratch_elems(n) * 72, dtype=torch.int64, device="cuda")
        d_out = torch.empty(72, dtype=torch.int64, device="cuda")
        engine.fp12_product_dev(d_in, n, scratch, d_out, stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(d_out.cpu().numpy().view(np.uint64), prod), n
        assert np.array_equal(engine.final_exponentiation_batch(prod[None])[0], gt), n
        # Gt only: the Miller loops run with free line scaling (cheaper homogeneous line steps), same Gt bit for bit
        none, gt_only = engine.multi_miller_product(g1, g2, i1, i2, want_miller_product=False)
        assert none is None and np.array_equal(gt_only, gt), n


def test_miller_mode_with_free_line_scaling(engine, coracle):
    """mode 5 (Miller loop whose output only feeds a final exponentiation): differs from SURVEY 9.1's Miller value
    by a subfield factor, gives the same Gt bit for bit, alone and inside shared-accumulator checks."""
    import torch
    import zkvm_pairings_b200 as z
    n, k = 512, 4
    g1, i1, g2, i2 = util.oracle_points(coracle, 555, 0, n)
    st = torch.cuda.current_stream().cuda_stream
    dg1, dg2 = torch.from_numpy(g1.view(np.int64)).cuda(), torch.from_numpy(g2.view(np.int64)).cuda()
    for kk in (1, k):
        nc = n // kk
        m5 = torch.empty((nc, 72), dtype=torch.int64, device="cuda")
        gt = torch.empty((nc, 72), dtype=torch.int64, device="cuda")
        engine.pairing_dev(z.MODE_MILLER_FOR_FINAL_EXP, m5, g1=dg1, g2=dg2, n_checks=nc, pairs_per_check=kk, stream=st)
        engine.pairing_dev(z.MODE_FINAL_EXP, gt, in_fp12=m5, n_checks=nc, stream=st)
        torch.cuda.synchronize()
        exp, _ = coracle.multi_pairing_batch(g1, None, g2, None, kk)
        assert np.array_equal(gt.cpu().numpy().view(np.uint64), exp)
        m1 = coracle.multi_miller_batch(g1, None, g2, None, kk)
        assert not np.array_equal(m5.cpu().numpy().view(np.uint64), m1)      # a different representative ...
    from zkvm_pairings_b200 import ZkpError
    with pytest.raises(ZkpError):
        engine.pairing_dev(4, gt, g1=dg1, g2=dg2, stream=st)


def test_default_stream_ordering_and_device_restored(engine, coracle):
    """*_dev calls with stream = 0 run on the legacy default stream, i.e. ordered after torch's default-stream
    work that produced their inputs and before the torch work that consumes their outputs -- no explicit
    synchronisation in between; the caller's current device is untouched."""
    import torch
    assert torch.cuda.current_stream().cuda_stream == 0
    n = 4096
    g1, _, g2, _ = util.oracle_points(coracle, 31337, 0, 64)
    reps = n // 64
    before = torch.cuda.current_device()
    big = torch.zeros((1 << 26,), dtype=torch.int64, device="cuda")          # keeps the default stream busy first
    big += 1
    dg1 = torch.from_numpy(np.tile(g1, (reps, 1)).view(np.int64)).cuda(non_blocking=True)
    dg2 = torch.from_numpy(np.tile(g2, (reps, 1)).view(np.int64)).cuda(non_blocking=True)
    out = torch.zeros((n, 72), dtype=torch.int64, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    engine.pairing_dev(3, out, g1=dg1, g2=dg2, err=err, stream=0)
    host = out.cpu()                                                          # default-stream consumer, no sync call
    assert torch.cuda.current_device() == before
    exp = coracle.pairing_batch(g1, None, g2, None)
    assert np.array_equal(host.numpy().view(np.uint64)[:64], exp) and np.array_equal(host.numpy().view(np.uint64)[-64:], exp)
    assert int(err.item()) == 0


def _all_devices_engine():
    import zkvm_pairings_b200 as z
    if z.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    return z.PairingEngine()


def test_multi_device_context_matches_single_device(engine, coracle):
    """The in-library multi-device paths (one host thread + two streams per device, contiguous slices; the
    576-byte Fp12 partial gather of zkp_multi_miller_product over peer copies): bit-identical to the
    single-device engine and the oracle, for sizes that do not divide evenly and for n < 2 * devices."""
    import torch
    multi = _all_devices_engine()
    try:
        nd = multi.num_devices
        assert nd >= 2
        before = torch.cuda.current_device()
        for n in (1, nd + 1, 2 * nd - 1, 5003, (1 << 18) + 77):
            g1, i1, g2, i2 = engine.gen_points(0xD0 + n, 0, n)
            if n > 8:
                i1[3] = 1
            gt = multi.pairing_batch(g1, g2, i1, i2)
            assert np.array_equal(gt, engine.pairing_batch(g1, g2, i1, i2)), n
            if n <= 5003:
                assert np.array_equal(gt, coracle.pairing_batch(g1, i1, g2, i2)), n
            prod, pgt = multi.multi_miller_product(g1, g2, i1, i2)
            sprod, sgt = engine.multi_miller_product(g1, g2, i1, i2)
            assert np.array_equal(prod, sprod) and np.array_equal(pgt, sgt), n
            if n <= 5003:
                eml, egt = coracle.miller_product(g1, i1, g2, i2)
                assert np.array_equal(prod, eml) and np.array_equal(pgt, egt), n
        n = 4 * 1001
        g1, i1, g2, i2 = engine.gen_points(0xD4, 0, n)
        out, one = multi.multi_pairing_batch(g1, g2, 4, i1, i2)
        sout, sone = engine.multi_pairing_batch(g1, g2, 4, i1, i2)
        assert np.array_equal(out, sout) and np.array_equal(one, sone)
        exp, eone = coracle.multi_pairing_batch(g1[:400], None, g2[:400], None, 4)
        assert np.array_equal(out[:100], exp)
        assert torch.cuda.current_device() == before      # the context never leaves the caller on another device
    finally:
        multi.close()


def test_config5_sharded_2p24_with_product_gather(engine, coracle):
    """BASELINE config[4] ("2^24 independent pairings sharded across 2/4/8 B200 with Fp12 partial-product
    gather"): one multi-device context, pageable host buffers.  Independent Gt outputs: a sample of every
    device's slice against the C oracle; the global product through the gather equals the final exponentiation
    of the product of all per-pair Miller outputs folded on ONE device."""
    import torch
    multi = _all_devices_engine()
    try:
        nd = multi.num_devices
        n = 1 << int(os.environ.get("ZKP_TEST_CONFIG5_LOG2", "24"))
        g1, _, g2, _ = multi.gen_points(0xC5, 0, n)
        gt = multi.pairing_batch(g1, g2)
        idx = np.concatenate([np.arange(d * n // nd, d * n // nd + 8) for d in range(nd)] + [np.arange(n - 8, n)])
        assert np.array_equal(gt[idx], coracle.pairing_batch(np.ascontiguousarray(g1[idx]), None, np.ascontiguousarray(g2[idx]), None))
        prod, pgt = multi.multi_miller_product(g1, g2)
        # single-device fold of the per-pair Miller outputs, chunk by chunk (2^22 pairs = 2.4 GB at a time)
        parts = []
        step = 1 << 22
        for lo in range(0, n, step):
            ml = engine.miller_loop_batch(g1[lo:lo + step], g2[lo:lo + step])
            d_in = torch.from_numpy(ml.view(np.int64)).cuda()
            scratch = torch.empty(engine.product_scratch_elems(len(ml)) * 72, dtype=torch.int64, device="cuda")
            d_out = torch.empty(72, dtype=torch.int64, device="cuda")
            engine.fp12_product_dev(d_in, len(ml), scratch, d_out, stream=0)
            parts.append(d_out.cpu().numpy().view(np.uint64))
        acc = parts[0]
        for p in parts[1:]:
            acc = engine.fp12_mul_batch(acc[None], p[None])[0]
        assert np.array_equal(acc, prod)
        assert np.array_equal(engine.final_exponentiation_batch(prod[None])[0], pgt)
    finally:
        multi.close()


def test_precompile_shaped_scalar_calls(engine, pyref):
    """zkp_sys_bigint / zkp_syscall_fp_mulmod: the argument meaning of the reference's zkVM precompile FFI
    (src/fp.rs:126,376,443) -- twelve little-endian u32 limbs, op 0 = mul, 1 = add, canonical in and out --
    on the engine's context and on the process-wide one (ctx = NULL), aliasing allowed, limbs >= p rejected."""
    import random
    import zkvm_pairings_b200 as z
    rng = random.Random(0xB16)
    to32 = lambda v: np.array([(v >> (32 * i)) & 0xFFFFFFFF for i in range(12)], dtype=np.uint32)
    from32 = lambda a: sum(int(x) << (32 * i) for i, x in enumerate(a))
    P = pyref.P
    cases = [(0, 0), (1, P - 1), (P - 1, P - 1), (P - 1, 1), (2, (P + 1) // 2)] + [(rng.randrange(P), rng.randrange(P)) for _ in range(6)]
    for k, (a, b) in enumerate(cases):
        dflt = bool(k & 1)
        assert from32(engine.sys_bigint(0, to32(a), to32(b), use_default_ctx=dflt)) == a * b % P
        assert from32(engine.sys_bigint(1, to32(a), to32(b), use_default_ctx=dflt)) == (a + b) % P
        lhs = to32(a)
        engine.syscall_fp_mulmod(lhs, to32(b), use_default_ctx=dflt)
        assert from32(lhs) == a * b % P
    # `result` may alias an operand (the crate's mul_assign passes lhs as the output, src/fp.rs:118-130)
    lib, x = engine._lib, to32(cases[-1][0])
    assert lib.zkp_sys_bigint(None, x.ctypes.data, 1, x.ctypes.data, x.ctypes.data) == 0
    assert from32(x) == 2 * cases[-1][0] % P
    with pytest.raises(z.ZkpError) as ei:
        engine.sys_bigint(0, to32(P), to32(1))
    assert ei.value.code == -3
    with pytest.raises(z.ZkpError):
        engine.sys_bigint(2, to32(1), to32(1))


def test_imad_peak_probe(engine):
    wide = engine.imad_peak(0)
    lo = engine.imad_peak(1)
    chain = engine.imad_peak(2)
    assert 1e12 < wide < 1e14 and 1e12 < lo < 1e14 and 1e12 < chain < 1e14
