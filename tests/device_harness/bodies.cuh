// Test bodies over RAW Montgomery representatives, shared by the device harness (harness.cu, nvcc) and the dev
// simulation (tests/host_sim/sim.cpp, sim_body).  TEST INFRASTRUCTURE ONLY: never part of libzkpair.so.
//
// The C ABI converts canonical inputs at load time, so every representative it delivers is below ~1.1 p; the
// arithmetic of fp.cuh / tower.cuh is written for representatives anywhere in [0, 2p] (one mont_mul operand up to
// 4p, unreduced sums up to 68 p^2).  These bodies take the representatives as they are -- no conversion, no bound
// check -- so that the tests can put every operand at the corners of the box the code is designed for.
//
// Layout of one element (host and device): BODY_SLOTS Fp2 slots in, BODY_SLOTS out, 12 u64 each; slot j holds the
// even lane's Fp at u64 12 j and the odd lane's at 12 j + 6 (six u64 = the twelve 32-bit words of Fp, low first).
// Fp-level bodies run lane-locally, so each element carries two independent Fp cases (one per lane); an FpW value
// takes two consecutive slots (low half, high half).  Fp6 / Fp12 operands are consecutive Fp2 slots in struct order.
// Fr-level bodies (fr.cuh, and the byte paths of blob.cuh / kzg_prove.cuh) also run lane-locally and read and write the
// low 256 bits of the lane's Fp in a slot (eight words, low first); the bits above stay zero in the results.
#pragma once
#include "../../zkvm_pairings_b200/csrc/ops.cuh"
#include "../../zkvm_pairings_b200/csrc/kzg_prove.cuh"

#define BODY_SLOTS 16
#define BODY_U64 (12 * BODY_SLOTS)

namespace zkp {

enum Body {
    // Fp level, per lane: x_j / r_j = this lane's Fp in slot j
    B_MONT_MUL = 0,       // r0 = mont_mul(x0, x1)
    B_MONT_MUL2,          // r0 = mont_mul2(x0, x1, x2, x3)
    B_MUL_WIDE,           // r0|r1 = mul_wide(x0, x1)
    B_MUL_WIDE2,          // r0|r1 = mul_wide2(x0, x1, x2, x3)
    B_MONT_REDC,          // r0 = mont_redc(x0|x1)
    B_FP2_REDC0,          // r0 = fp2_redc<0>(x0|x1)
    B_FP2_REDC1,          // r0 = fp2_redc<1>(x0|x1)
    B_FP_CORRECT,         // r0 = fp_correct(x0)
    B_FP_CORRECT8,        // r0 = fp_correct8(x0)
    B_FP_ADD,             // r0 = fp_add(x0, x1)
    B_FP_SUB,             // r0 = fp_sub(x0, x1)
    B_FP_NEG,             // r0 = fp_neg(x0)
    B_FPW_MUL_NR,         // r0|r1 = fpw_mul_nr(x0|x1)   (lane pair: the even lane holds c0, the odd lane c1)
    B_FP_TO_WORDS,        // r0 = fp_to_words(x0)
    B_FP_IS_ZERO,         // r0 = fp_is_zero(x0) (0 / 1)
    B_FP_INV,             // r0 = fp_inv(x0)
    B_BATCH_INV1,         // r0..r(n-1) = fp_batch_inv(x0..x(n-1)), n = 1 / 7 / 16
    B_BATCH_INV7,
    B_BATCH_INV16,
    // tower level, lane-split Fp2 slots
    B_FP2_MUL = 32,       // r0 = x0 * x1
    B_FP2_SQR,            // r0 = x0^2
    B_FP2_MUL_NR,         // r0 = xi x0
    B_FP2_INV,            // r0 = 1 / x0
    B_FP6_MUL,            // r0..2 = (x0..2) (x3..5)
    B_FP6_SQR,            // r0..2 = (x0..2)^2
    B_FP6_MUL_BY_1,       // r0..2 = (x0..2) (0, x3, 0)
    B_FP6_MUL_BY_01,      // r0..2 = (x0..2) (x3, x4, 0)
    B_FP6_MUL_SUMS,       // r0..2 = fp6_mul_sums(x0..2, x3..5)
    B_FP4_SQUARE,         // r0, r1 = fp4_square(x0, x1)
    B_FP12_MUL,           // r0..5 = (x0..5) (x6..11)
    B_FP12_SQR,           // r0..5 = (x0..5)^2
    B_FP12_SQR_INPLACE,   // the same by fp12_sqr_inplace
    B_FP12_MUL_BY_014,    // r0..5 = (x0..5) (x6 + x7 v + x8 v w)
    B_FP12_MUL_BY_014_INPLACE,
    B_FP12_CYC_SQR,       // r0..5 = fp12_cyclotomic_sqr(x0..5)
    B_FP12_INV,           // r0..5 = 1 / (x0..5)
    // Fr level, per lane: x_j / r_j = the low 256 bits of this lane's Fp in slot j
    B_FR_ADD = 64,        // r0 = fr_add(x0, x1)
    B_FR_SUB,             // r0 = fr_sub(x0, x1)
    B_FR_MUL,             // r0 = fr_mul(x0, x1)
    B_FR_REDUCE_ONCE,     // r0 = fr_reduce_once(x0)
    B_FR_GEQ_R,           // r0 = fr_geq_r(x0) (0 / 1)
    B_FR_TO_MONT,         // r0 = fr_to_mont(x0)
    B_FR_FROM_MONT,       // r0 = fr_from_mont(x0)
    B_FR_INV,             // r0 = fr_inv(x0)
    B_BLOB_ELEMENT,       // r0 = the element, r1 = ok (0 / 1): blob_element of x0 as 32 big-endian bytes
    B_STORE_BE32,         // r0 = the 32 bytes store_be32 writes for x0, in memory order
};

ZKP_HD Fp raw_fp(const uint64_t *s) {
    Fp r;
    for (int i = 0; i < 6; i++) {
        r.l[2 * i] = (uint32_t)s[i];
        r.l[2 * i + 1] = (uint32_t)(s[i] >> 32);
    }
    return r;
}
ZKP_HD void raw_store(uint64_t *d, const Fp &a) {
    for (int i = 0; i < 6; i++) d[i] = (uint64_t)a.l[2 * i] | ((uint64_t)a.l[2 * i + 1] << 32);
}
ZKP_HD FpW raw_w(const Fp &lo, const Fp &hi) {
    FpW t;
    for (int i = 0; i < ZKP_NL; i++) {
        t.l[i] = lo.l[i];
        t.l[ZKP_NL + i] = hi.l[i];
    }
    return t;
}
ZKP_HD void split_w(Fp &lo, Fp &hi, const FpW &t) {
    for (int i = 0; i < ZKP_NL; i++) {
        lo.l[i] = t.l[i];
        hi.l[i] = t.l[ZKP_NL + i];
    }
}
ZKP_HD Fr low_fr(const Fp &a) {
    Fr r;
    for (int i = 0; i < ZKP_FR_NL; i++) r.l[i] = a.l[i];
    return r;
}
ZKP_HD Fp fr_slot(const Fr &a) {
    Fp r = fp_zero();
    for (int i = 0; i < ZKP_FR_NL; i++) r.l[i] = a.l[i];
    return r;
}

// One element, executed by a lane pair (both lanes make the same calls).  `live` = store the result (tail lanes of
// the converged builds recompute the last element and store nothing).
ZKP_HD void body_one(int body, const uint64_t *in, uint64_t *out, bool live) {
    Fp2 x[BODY_SLOTS], r[BODY_SLOTS];
    for (int j = 0; j < BODY_SLOTS; j++) {
        x[j].c = raw_fp(in + 12 * j + 6 * lane_par());
        r[j].c = fp_zero();
    }
    Fp6 *x6 = (Fp6 *)x, *r6 = (Fp6 *)r;
    Fp12 *x12 = (Fp12 *)x, *r12 = (Fp12 *)r;
    switch (body) {
        case B_MONT_MUL: r[0].c = mont_mul(x[0].c, x[1].c); break;
        case B_MONT_MUL2: r[0].c = mont_mul2(x[0].c, x[1].c, x[2].c, x[3].c); break;
        case B_MUL_WIDE: split_w(r[0].c, r[1].c, mul_wide(x[0].c, x[1].c)); break;
        case B_MUL_WIDE2: split_w(r[0].c, r[1].c, mul_wide2(x[0].c, x[1].c, x[2].c, x[3].c)); break;
        case B_MONT_REDC: r[0].c = mont_redc(raw_w(x[0].c, x[1].c)); break;
        case B_FP2_REDC0: r[0] = fp2_redc<0>(raw_w(x[0].c, x[1].c)); break;
        case B_FP2_REDC1: r[0] = fp2_redc<1>(raw_w(x[0].c, x[1].c)); break;
        case B_FP_CORRECT: r[0].c = fp_correct(x[0].c); break;
        case B_FP_CORRECT8: r[0].c = fp_correct8(x[0].c); break;
        case B_FP_ADD: r[0].c = fp_add(x[0].c, x[1].c); break;
        case B_FP_SUB: r[0].c = fp_sub(x[0].c, x[1].c); break;
        case B_FP_NEG: r[0].c = fp_neg(x[0].c); break;
        case B_FPW_MUL_NR: split_w(r[0].c, r[1].c, fpw_mul_nr(raw_w(x[0].c, x[1].c))); break;
        case B_FP_TO_WORDS: fp_to_words(r[0].c.l, x[0].c); break;
        case B_FP_IS_ZERO: r[0].c.l[0] = fp_is_zero(x[0].c) ? 1u : 0u; break;
        case B_FP_INV: r[0].c = fp_inv(x[0].c); break;
        case B_BATCH_INV1:
        case B_BATCH_INV7:
        case B_BATCH_INV16: {
            const int n = body == B_BATCH_INV1 ? 1 : body == B_BATCH_INV7 ? 7 : 16;
            Fp v[16], pre[16];
            for (int j = 0; j < n; j++) v[j] = x[j].c;
            fp_batch_inv(v, pre, n);
            for (int j = 0; j < n; j++) r[j].c = v[j];
        } break;
        case B_FP2_MUL: r[0] = fp2_mul(x[0], x[1]); break;
        case B_FP2_SQR: r[0] = fp2_sqr(x[0]); break;
        case B_FP2_MUL_NR: r[0] = fp2_mul_nr(x[0]); break;
        case B_FP2_INV: r[0] = fp2_inv(x[0]); break;
        case B_FP6_MUL: fp6_mul(r6[0], x6[0], x6[1]); break;
        case B_FP6_SQR: fp6_sqr(r6[0], x6[0]); break;
        case B_FP6_MUL_BY_1: fp6_mul_by_1(r6[0], x6[0], x[3]); break;
        case B_FP6_MUL_BY_01: fp6_mul_by_01(r6[0], x6[0], x[3], x[4]); break;
        case B_FP6_MUL_SUMS: fp6_mul_sums(r6[0], x6[0], x6[1]); break;
        case B_FP4_SQUARE: fp4_square(r[0], r[1], x[0], x[1]); break;
        case B_FP12_MUL: fp12_mul(r12[0], x12[0], x12[1]); break;
        case B_FP12_SQR: fp12_sqr(r12[0], x12[0]); break;
        case B_FP12_SQR_INPLACE: {
            Fp6 t;
            r12[0] = x12[0];
            fp12_sqr_inplace(r12[0], t);
        } break;
        case B_FP12_MUL_BY_014: r12[0] = x12[0]; fp12_mul_by_014(r12[0], x[6], x[7], x[8]); break;
        case B_FP12_MUL_BY_014_INPLACE: {
            Fp6 t;
            r12[0] = x12[0];
            fp12_mul_by_014_inplace(r12[0], t, x[6], x[7], x[8]);
        } break;
        case B_FP12_CYC_SQR: fp12_cyclotomic_sqr(r12[0], x12[0]); break;
        case B_FP12_INV: fp12_inv(r12[0], x12[0]); break;
        case B_FR_ADD: r[0].c = fr_slot(fr_add(low_fr(x[0].c), low_fr(x[1].c))); break;
        case B_FR_SUB: r[0].c = fr_slot(fr_sub(low_fr(x[0].c), low_fr(x[1].c))); break;
        case B_FR_MUL: r[0].c = fr_slot(fr_mul(low_fr(x[0].c), low_fr(x[1].c))); break;
        case B_FR_REDUCE_ONCE: r[0].c = fr_slot(fr_reduce_once(low_fr(x[0].c))); break;
        case B_FR_GEQ_R: r[0].c.l[0] = fr_geq_r(low_fr(x[0].c)) ? 1u : 0u; break;
        case B_FR_TO_MONT: r[0].c = fr_slot(fr_to_mont(low_fr(x[0].c))); break;
        case B_FR_FROM_MONT: r[0].c = fr_slot(fr_from_mont(low_fr(x[0].c))); break;
        case B_FR_INV: r[0].c = fr_slot(fr_inv(low_fr(x[0].c))); break;
        case B_BLOB_ELEMENT: {
            // element 1 of a 16-byte aligned two-element row, as blob_element reads a blob (uint4 loads on the device)
            alignas(16) uint8_t row[64];
            const Fr v = low_fr(x[0].c);
            for (int k = 0; k < 32; k++) {
                row[k] = 0;
                row[63 - k] = (uint8_t)(v.l[k >> 2] >> (8 * (k & 3)));
            }
            Fr e;
            const bool ok = blob_element(row, 1, e);
            r[0].c = fr_slot(e);
            r[1].c.l[0] = ok ? 1u : 0u;
        } break;
        case B_STORE_BE32: {
            alignas(16) uint8_t row[32];
            store_be32(row, low_fr(x[0].c));
            for (int k = 0; k < 8; k++)
                r[0].c.l[k] = (uint32_t)row[4 * k] | ((uint32_t)row[4 * k + 1] << 8) | ((uint32_t)row[4 * k + 2] << 16) |
                              ((uint32_t)row[4 * k + 3] << 24);
        } break;
        default: break;
    }
    if (live)
        for (int j = 0; j < BODY_SLOTS; j++) raw_store(out + 12 * j + 6 * lane_par(), r[j].c);
}

}  // namespace zkp
