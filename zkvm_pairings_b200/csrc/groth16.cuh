// Groth16 verification front end: fixed-base window tables of the verifying key's IC points and the
// per-proof body that validates a proof, accumulates L = IC_0 + sum_j x_j IC_j from those tables and
// assembles the 4-pair check e(A,B) e(alpha,-beta) e(L,-gamma) e(C,-delta) == 1 for the prepared
// pairing path (pairs [A, alpha, L, C] x [B | three prepared tables]).
//
// Shared by the CUDA kernels (kernels.cu) and the CPU dev simulation of the not-gpu tests.
#pragma once
#include "ops.cuh"

namespace zkp {

#define ZKP_G16_WINDOWS 32      // 8-bit windows of a 256-bit scalar
#define ZKP_G16_DIGITS 255      // non-zero digits per window
// Fp per IC_j table: [window][digit - 1] affine (x, y), Montgomery form (32 * 255 * 2 * 48 B = 765 KB)
#define ZKP_G16_TABLE_FP (ZKP_G16_WINDOWS * ZKP_G16_DIGITS * 2)

#ifndef ZKP_G16_VALID   /* same values as include/zkpair.h */
#define ZKP_G16_VALID 0
#define ZKP_G16_INVALID 1
#define ZKP_G16_BAD_POINT 2
#define ZKP_G16_BAD_INPUT 3
#endif

// General Jacobian addition (add-2007-bl).  Either operand may be the identity (z == 0); equal
// operands double, opposite operands give the identity.
template <class O>
ZKP_NOINLINE void jac_add(Jac<O> &r, const Jac<O> &p, const Jac<O> &q) {
    typedef typename O::T T;
    if (O::is_zero(p.z)) { r = q; return; }
    if (O::is_zero(q.z)) { r = p; return; }
    T z1z1 = O::sqr(p.z), z2z2 = O::sqr(q.z);
    T u1 = O::mul(p.x, z2z2), u2 = O::mul(q.x, z1z1);
    T s1 = O::mul(O::mul(p.y, q.z), z2z2), s2 = O::mul(O::mul(q.y, p.z), z1z1);
    T h = O::sub(u2, u1), rr = O::sub(s2, s1);
    if (O::is_zero(h)) {
        if (O::is_zero(rr)) { jac_double(r, p); return; }
        r.x = O::zero(); r.y = O::one(); r.z = O::zero(); return;
    }
    T i = O::add(h, h);
    i = O::sqr(i);
    T j = O::mul(h, i);
    rr = O::add(rr, rr);
    T v = O::mul(u1, i);
    T x3 = O::sub(O::sub(O::sqr(rr), j), O::add(v, v));
    T t = O::mul(s1, j);
    T y3 = O::sub(O::mul(rr, O::sub(v, x3)), O::add(t, t));
    T z3 = O::mul(O::sub(O::sub(O::sqr(O::add(p.z, q.z)), z1z1), z2z2), h);
    r.x = x3; r.y = y3; r.z = z3;
}

// Window table of ONE (IC_j, window w), built by one thread: entry d - 1 = d 2^(8w) IC_j for d = 1..digits
// (255, or 128 for the signed digits of kzg_prove.cuh), affine.  A Jacobian chain P, 2P, .., digits P from
// P = 2^(8w) IC_j (8w doublings, one inversion), then Montgomery's trick over the chain's Z.  IC_j is a
// validated subgroup point, so no entry is the identity (d 2^(8w) < r is never a multiple of the prime r).
// zs / pre: scratch of `digits` Fp each.
ZKP_HD void groth16_window_table(const uint64_t *ic_xy, int w, Fp *out, Fp *zs, Fp *pre, int digits = ZKP_G16_DIGITS) {
    bool bad = false;
    Jac<OpsFp> p;
    p.x = load_fp(ic_xy, bad);
    p.y = load_fp(ic_xy + 6, bad);
    p.z = fp_one();
    for (int i = 0; i < 8 * w; i++) jac_double(p, p);
    Fp zi = fp_inv(p.z), zi2 = fsqr(zi);
    Fp px = fmul(p.x, zi2), py = fmul(p.y, fmul(zi2, zi));
    Jac<OpsFp> e;
    e.x = px; e.y = py; e.z = fp_one();
    for (int d = 0; d < digits; d++) {
        if (d) jac_add_affine(e, e, px, py);
        out[2 * d] = e.x;
        out[2 * d + 1] = e.y;
        zs[d] = e.z;
    }
    fp_batch_inv(zs, pre, digits);
    for (int d = 0; d < digits; d++) {
        Fp z2 = fsqr(zs[d]);
        out[2 * d] = fmul(out[2 * d], z2);
        out[2 * d + 1] = fmul(out[2 * d + 1], fmul(z2, zs[d]));
    }
}

// The verifying key as the per-proof body reads it (device pointers on the GPU).
struct G16Key {
    const uint64_t *alpha;   // canonical x|y
    const uint64_t *ic0;     // canonical x|y of IC_0
    const uint8_t *ic_inf;   // n_public + 1 flags: IC_0 .. IC_l at infinity (no table is built for those)
    const Fp *tables;        // n_public x ZKP_G16_TABLE_FP, for IC_1 .. IC_l
    int n_public;
};

// x < r for a scalar of four little-endian u64 limbs
ZKP_HD bool fr_canonical(const uint64_t *x) {
    for (int i = 3; i >= 0; i--) {
        uint64_t r = ((uint64_t)ZKP_R_ORDER[2 * i + 1] << 32) | ZKP_R_ORDER[2 * i];
        if (x[i] != r) return x[i] < r;
    }
    return false;
}

ZKP_HD void copy_u64(uint64_t *dst, const uint64_t *src, int n, bool zero) {
    for (int i = 0; i < n; i++) dst[i] = zero ? 0 : src[i];
}

// One proof, executed by a lane pair.  proof = A.x|A.y | B (24 u64) | C.x|C.y; pinf = 3 flags (A, B, C) or
// NULL; x = n_public scalars.  Writes the check's four G1 slots [A, alpha, L, C] (g1, g1inf) and its one G2
// slot [B] (g2, g2inf) and returns the status (both lanes).  A rejected proof's slots hold zeros with every
// infinity flag set, so the pairing that follows never sees a non-canonical limb.
//
// Lane split: B's check is Fp2 work, split over the pair as everywhere; the G1 work is Fp-level, so the
// even lane checks A and the odd lane C, and for L each lane accumulates the windows of its own parity
// (even lane: IC_0 + the windows 0, 2, .., 30 of every x_j; odd lane: windows 1, 3, .., 31), at most
// 16 mixed additions per input and lane; the two partial sums meet in one general Jacobian addition.
ZKP_HD uint8_t groth16_prepare_one(const G16Key &vk, const uint64_t *proof, const uint8_t *pinf, const uint64_t *x,
                                   uint64_t *g1, uint8_t *g1inf, uint64_t *g2, uint8_t *g2inf) {
    const int par = lane_par();
    const uint8_t ainf = pinf ? pinf[0] : 0, binf = pinf ? pinf[1] : 0, cinf = pinf ? pinf[2] : 0;
    bool bad = false;
    uint8_t sb = g2_check_one(proof + 12, binf, bad);
    uint8_t sac = g1_check_one(proof + (par ? 36 : 0), par ? cinf : ainf, bad);
    const bool bad_point = lane_or(bad | (sb != ZKP_POINT_OK) | (sac != ZKP_POINT_OK));

    bool bad_input = false;
    Jac<OpsFp> acc;
    acc.x = fp_zero(); acc.y = fp_one(); acc.z = fp_zero();
    if (par == 0 && !vk.ic_inf[0]) {
        bool b0 = false;
        acc.x = load_fp(vk.ic0, b0);
        acc.y = load_fp(vk.ic0 + 6, b0);
        acc.z = fp_one();
    }
    for (int j = 0; j < vk.n_public; j++) {
        const uint64_t *s = x + 4 * j;
        bad_input |= !fr_canonical(s);
        if (vk.ic_inf[j + 1]) continue;
        const Fp *t = vk.tables + (size_t)j * ZKP_G16_TABLE_FP;
        for (int w = par; w < ZKP_G16_WINDOWS; w += 2) {
            uint32_t d = (uint32_t)(s[w >> 3] >> (8 * (w & 7))) & 0xffu;
            if (!d) continue;
            const Fp *e = t + 2 * (w * ZKP_G16_DIGITS + (int)d - 1);
            jac_add_affine(acc, acc, e[0], e[1]);
        }
    }
    // both lanes form even + odd in the same order, so they hold the same representative
    Jac<OpsFp> pe, po, l;
    pe.x = fp_bcast<0>(acc.x); pe.y = fp_bcast<0>(acc.y); pe.z = fp_bcast<0>(acc.z);
    po.x = fp_bcast<1>(acc.x); po.y = fp_bcast<1>(acc.y); po.z = fp_bcast<1>(acc.z);
    jac_add(l, pe, po);
    const bool linf = fp_is_zero(l.z);
    Fp lx = fp_zero(), ly = fp_one();
    if (!linf) {
        Fp zi = fp_inv(l.z), zi2 = fsqr(zi);
        lx = fmul(l.x, zi2);
        ly = fmul(l.y, fmul(zi2, zi));
    }

    const uint8_t st = bad_point ? ZKP_G16_BAD_POINT : bad_input ? ZKP_G16_BAD_INPUT : ZKP_G16_VALID;
    const bool rej = st != ZKP_G16_VALID;
    if (rej) { lx = fp_zero(); ly = fp_zero(); }
    if (par == 0) {
        copy_u64(g1, proof, 12, rej);              // A
        copy_u64(g1 + 12, vk.alpha, 12, rej);      // alpha
        store_fp(g1 + 24, lx, nullptr);            // L.x
        g1inf[0] = rej ? 1 : ainf;
        g1inf[1] = rej ? 1 : 0;
        g1inf[2] = rej ? 1 : (linf ? 1 : 0);
        g1inf[3] = rej ? 1 : cinf;
        *g2inf = rej ? 1 : binf;
    } else {
        store_fp(g1 + 30, ly, nullptr);            // L.y
        copy_u64(g1 + 36, proof + 36, 12, rej);    // C
        copy_u64(g2, proof + 12, 24, rej);         // B
    }
    return st;
}

}  // namespace zkp
