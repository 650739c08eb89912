// KZG point-evaluation verification front end (EIP-4844 verify_kzg_proof(C, z, y, pi)): the per-proof body that
// validates C and pi, range-checks z and y, computes P = C + [z]pi + [r - y]G1 and assembles the 2-pair check
// e(P, G2) e(pi, -[tau]G2) == 1 for the prepared pairing path (pairs [P, pi] x two prepared tables).
//
// Shared by the CUDA kernels (kernels.cu) and the CPU dev simulation of the not-gpu tests.
#pragma once
#include "groth16.cuh"

namespace zkp {

#ifndef ZKP_KZG_VALID   /* same values as include/zkpair.h (and as ZKP_G16_*, so k_groth16_verdict applies) */
#define ZKP_KZG_VALID 0
#define ZKP_KZG_INVALID 1
#define ZKP_KZG_BAD_POINT 2
#define ZKP_KZG_BAD_SCALAR 3
#endif

// GLV split of a scalar z < r over the G1 endomorphism [x^2]P = (beta x_P, -y_P) (the identity g1_check_one tests):
// z = hi x^2 + lo with lo < x^2 < 2^128, and hi < 2^128 because r < 2^128 x^2.  Shift-and-subtract long division;
// the remainder stays below x^2, and the one bit a shift can push past 2^128 is kept in `top`.
ZKP_HD void kzg_glv_split(const uint64_t *z, uint64_t *hi, uint64_t *lo) {
    typedef unsigned __int128 u128;
    const u128 d = (u128)ZKP_BLS_X * ZKP_BLS_X;
    u128 rem = 0, q = 0;
#pragma unroll 1
    for (int i = 255; i >= 0; i--) {
        const bool top = (rem >> 127) != 0;
        rem = (rem << 1) | (u128)((z[i >> 6] >> (i & 63)) & 1);
        q <<= 1;
        if (top || rem >= d) {
            rem -= d;
            q |= 1;
        }
    }
    hi[0] = (uint64_t)q;
    hi[1] = (uint64_t)(q >> 64);
    lo[0] = (uint64_t)rem;
    lo[1] = (uint64_t)(rem >> 64);
}

// r - y for y < r, and 0 for y = 0: the fixed-base scalar of -[y]G1
ZKP_HD void fr_neg(const uint64_t *y, uint64_t *out) {
    const bool zero = (y[0] | y[1] | y[2] | y[3]) == 0;
    uint64_t borrow = 0;
    for (int i = 0; i < 4; i++) {
        const uint64_t r = ((uint64_t)ZKP_R_ORDER[2 * i + 1] << 32) | ZKP_R_ORDER[2 * i];
        const uint64_t t = r - y[i];
        const uint64_t b = (r < y[i]) | (t < borrow);
        out[i] = zero ? 0 : t - borrow;
        borrow = b;
    }
}

// One proof, executed by a lane pair.  proof = C.x|C.y | pi.x|pi.y (24 u64); pinf = 2 flags (C, pi) or NULL;
// zy = z | y (8 u64); g1_table = the generator's window table (groth16_window_table layout, ZKP_G16_TABLE_FP Fp).
// Writes the check's two G1 slots [P, pi] (g1, g1inf) and returns the status (both lanes).  A rejected proof's
// slots hold zeros with both infinity flags set, so the pairing that follows never sees a non-canonical limb.
//
// Lane split (all of it Fp-level work): the even lane checks C and the odd lane pi.  With z = z_hi x^2 + z_lo the
// even lane computes [z_lo]pi + C and the odd lane [z_hi](beta x_pi, -y_pi), one 128-bit ladder each.  Each lane
// then adds the windows of its own parity of r - y from the table (at most 16 mixed additions).  The two partial
// sums meet in one general Jacobian addition, followed by one inversion.
ZKP_HD uint8_t kzg_prepare_one(const Fp *g1_table, const uint64_t *proof, const uint8_t *pinf, const uint64_t *zy, uint64_t *g1,
                               uint8_t *g1inf) {
    const int par = lane_par();
    const uint8_t cinf = pinf ? pinf[0] : 0, qinf = pinf ? pinf[1] : 0;
    bool bad = false;
    const uint8_t sp = g1_check_one(proof + (par ? 12 : 0), par ? qinf : cinf, bad);
    const bool bad_point = lane_or(bad | (sp != ZKP_POINT_OK));
    const bool bad_scalar = !fr_canonical(zy) | !fr_canonical(zy + 4);
    const uint8_t st = bad_point ? ZKP_KZG_BAD_POINT : bad_scalar ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
    const bool rej = st != ZKP_KZG_VALID;   // the same in both lanes

    Jac<OpsFp> acc;
    acc.x = fp_zero(); acc.y = fp_one(); acc.z = fp_zero();
    if (!rej) {
        bool b = false;
        if (!qinf) {
            uint64_t zh[2], zl[2];
            kzg_glv_split(zy, zh, zl);
            Fp qx = load_fp(proof + 12, b), qy = load_fp(proof + 18, b);
            if (par) {
                qx = fmul(qx, fp_const(ZKP_BETA));
                qy = fp_neg(qy);
            }
            scalar_mul_jac<OpsFp>(acc, qx, qy, par ? zh : zl, 128);
        }
        if (par == 0 && !cinf) jac_add_affine(acc, acc, load_fp(proof, b), load_fp(proof + 6, b));
        uint64_t yn[4];
        fr_neg(zy + 4, yn);
        for (int w = par; w < ZKP_G16_WINDOWS; w += 2) {
            uint32_t d = (uint32_t)(yn[w >> 3] >> (8 * (w & 7))) & 0xffu;
            if (!d) continue;
            const Fp *e = g1_table + 2 * (w * ZKP_G16_DIGITS + (int)d - 1);
            jac_add_affine(acc, acc, e[0], e[1]);
        }
    }
    // both lanes form even + odd in the same order, so they hold the same representative
    Jac<OpsFp> pe, po, p;
    pe.x = fp_bcast<0>(acc.x); pe.y = fp_bcast<0>(acc.y); pe.z = fp_bcast<0>(acc.z);
    po.x = fp_bcast<1>(acc.x); po.y = fp_bcast<1>(acc.y); po.z = fp_bcast<1>(acc.z);
    jac_add(p, pe, po);
    const bool p_inf = fp_is_zero(p.z);
    Fp px = fp_zero(), py = fp_one();
    if (!p_inf) {
        Fp zi = fp_inv(p.z), zi2 = fsqr(zi);
        px = fmul(p.x, zi2);
        py = fmul(p.y, fmul(zi2, zi));
    }
    if (rej) { px = fp_zero(); py = fp_zero(); }
    if (par == 0) {
        store_fp(g1, px, nullptr);                 // P.x
        copy_u64(g1 + 12, proof + 12, 6, rej);     // pi.x
        g1inf[0] = rej ? 1 : (p_inf ? 1 : 0);
        g1inf[1] = rej ? 1 : qinf;
    } else {
        store_fp(g1 + 6, py, nullptr);             // P.y
        copy_u64(g1 + 18, proof + 18, 6, rej);     // pi.y
    }
    return st;
}

}  // namespace zkp
