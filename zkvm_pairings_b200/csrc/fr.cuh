// Fr: the BLS12-381 scalar field (the group order r < 2^255) -- 8 saturated 32-bit limbs, Montgomery form RF = 2^256.
//
// Built on the carry primitives of fp.cuh, so the CPU dev simulation runs the same code.  fp.cuh's 2p-redundant
// representation does not carry over (4r > 2^256), so every Fr that leaves a function of this file is a value in
// [0, r): a CIOS product of two such values is below 2r and needs one conditional subtraction, a sum of two is below
// 2r < 2^256 and needs one as well.  The dev simulation asserts the operand bound on every product, sum and difference
// (ZKP_SIM_ASSERT).
// The EIP-4844 blob path (blob.cuh) is the user; the bit ladders of the group code take canonical Fr limbs directly.
#pragma once
#include "fp.cuh"

namespace zkp {

#define ZKP_FR_NL 8

struct alignas(16) Fr {
    uint32_t l[ZKP_FR_NL];
};

ZKP_HD Fr fr_const(const uint32_t *k) {
    Fr r;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) r.l[i] = k[i];
    return r;
}
ZKP_HD Fr fr_one() { return fr_const(ZKP_FR_ONE); }   // Montgomery one
ZKP_HD Fr fr_zero() {
    Fr r;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) r.l[i] = 0;
    return r;
}
ZKP_HD bool fr_is_zero(const Fr &a) {
    uint32_t z = 0;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) z |= a.l[i];
    return z == 0;
}
ZKP_HD bool fr_eq(const Fr &a, const Fr &b) {
    uint32_t z = 0;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) z |= a.l[i] ^ b.l[i];
    return z == 0;
}
ZKP_HD Fr fr_select(bool c, const Fr &a, const Fr &b) {
    Fr r;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) r.l[i] = c ? a.l[i] : b.l[i];
    return r;
}
// a >= r ?  (ZKP_R_ORDER holds r in its low eight words)
ZKP_HD bool fr_geq_r(const Fr &a) {
    sub_cc(a.l[0], ZKP_R_ORDER[0]);
#pragma unroll
    for (int i = 1; i < ZKP_FR_NL; i++) subc_cc(a.l[i], ZKP_R_ORDER[i]);
    return subc(0, 0) == 0;
}
// a in [0, 2r) -> [0, r)
ZKP_HD Fr fr_reduce_once(const Fr &a) {
    Fr d;
    d.l[0] = sub_cc(a.l[0], ZKP_R_ORDER[0]);
#pragma unroll
    for (int i = 1; i < ZKP_FR_NL; i++) d.l[i] = subc_cc(a.l[i], ZKP_R_ORDER[i]);
    const bool lt = subc(0, 0) != 0;
    return fr_select(lt, a, d);
}
// (a + b) mod r for a, b < r: the sum is below 2r < 2^256, no carry out
ZKP_HD Fr fr_add(const Fr &a, const Fr &b) {
#ifndef ZKP_DEVICE_BUILD
    ZKP_SIM_ASSERT(!fr_geq_r(a) && !fr_geq_r(b), "fr_add operand bound");
#endif
    Fr s;
    s.l[0] = add_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < ZKP_FR_NL - 1; i++) s.l[i] = addc_cc(a.l[i], b.l[i]);
    s.l[ZKP_FR_NL - 1] = addc(a.l[ZKP_FR_NL - 1], b.l[ZKP_FR_NL - 1]);
    return fr_reduce_once(s);
}
// (a - b) mod r for a, b < r
ZKP_HD Fr fr_sub(const Fr &a, const Fr &b) {
#ifndef ZKP_DEVICE_BUILD
    ZKP_SIM_ASSERT(!fr_geq_r(a) && !fr_geq_r(b), "fr_sub operand bound");
#endif
    Fr d;
    d.l[0] = sub_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < ZKP_FR_NL; i++) d.l[i] = subc_cc(a.l[i], b.l[i]);
    const uint32_t mneg = subc(0, 0) != 0 ? 0xffffffffu : 0u;   // a < b: add r back
    d.l[0] = add_cc(d.l[0], ZKP_R_ORDER[0] & mneg);
#pragma unroll
    for (int i = 1; i < ZKP_FR_NL - 1; i++) d.l[i] = addc_cc(d.l[i], ZKP_R_ORDER[i] & mneg);
    d.l[ZKP_FR_NL - 1] = addc(d.l[ZKP_FR_NL - 1], ZKP_R_ORDER[ZKP_FR_NL - 1] & mneg);
    return d;
}

// t[0..9] += a * b: one chain over the low halves of the eight products, one over the high halves.  With t < 2r before
// a CIOS row and a, b < 2^256 the sum stays below 2^289, so t[9] never carries out.
ZKP_HD void fr_row(uint32_t *t, const uint32_t *a, uint32_t b) {
    t[0] = mad_lo_cc(a[0], b, t[0]);
#pragma unroll
    for (int j = 1; j < ZKP_FR_NL; j++) t[j] = madc_lo_cc(a[j], b, t[j]);
    t[8] = addc_cc(t[8], 0);
    t[9] = addc(t[9], 0);
    add_cc(0, 0);   // clears the carry flag for the high chain
#pragma unroll
    for (int j = 0; j < ZKP_FR_NL; j++) t[j + 1] = madc_hi_cc(a[j], b, t[j + 1]);
    t[9] = addc(t[9], 0);
}
// a * b / 2^256 mod r in [0, r) for a, b < r (CIOS: the running sum stays below 2r, one final subtraction)
ZKP_HD Fr fr_mul(const Fr &a, const Fr &b) {
#ifndef ZKP_DEVICE_BUILD
    ZKP_SIM_ASSERT(!fr_geq_r(a) && !fr_geq_r(b), "fr_mul operand bound");
#endif
    uint32_t t[ZKP_FR_NL + 2];
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL + 2; i++) t[i] = 0;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) {
        fr_row(t, a.l, b.l[i]);
        fr_row(t, ZKP_R_ORDER, t[0] * ZKP_FR_N0INV);   // clears t[0]
#pragma unroll
        for (int k = 0; k < ZKP_FR_NL + 1; k++) t[k] = t[k + 1];
        t[ZKP_FR_NL + 1] = 0;
    }
    Fr r;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) r.l[i] = t[i];
    return fr_reduce_once(r);
}
ZKP_HD Fr fr_mul_const(const Fr &a, const uint32_t *k) { return fr_mul(a, fr_const(k)); }
ZKP_HD Fr fr_sqr(const Fr &a) { return fr_mul(a, a); }

// canonical value < r -> Montgomery, and back
ZKP_HD Fr fr_to_mont(const Fr &a) { return fr_mul_const(a, ZKP_FR_R2); }
ZKP_HD Fr fr_from_mont(const Fr &a) {
    Fr one = fr_zero();
    one.l[0] = 1;
    return fr_mul(a, one);
}

// 1/x for a Montgomery x in [1, r) (0 maps to 0): the binary extended GCD of tower.cuh's fp_inv on eight words,
// 2 * 255 - 1 branch-free iterations of shifts, subtractions and selects; the result v = X^-1 R^-1 is taken back to
// Montgomery form with one product by R^3.
ZKP_NOINLINE Fr fr_inv(Fr x) {
    uint32_t a[ZKP_FR_NL], b[ZKP_FR_NL], u[ZKP_FR_NL], v[ZKP_FR_NL];
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) {
        a[i] = x.l[i];
        b[i] = ZKP_R_ORDER[i];
        u[i] = i == 0 ? 1u : 0u;
        v[i] = 0;
    }
#pragma unroll 1
    for (int it = 0; it < 2 * 255 - 1; it++) {
        const bool odd = (a[0] & 1u) != 0;
        uint32_t d[ZKP_FR_NL], nd[ZKP_FR_NL], w[ZKP_FR_NL];
        d[0] = sub_cc(a[0], b[0]);
#pragma unroll
        for (int i = 1; i < ZKP_FR_NL; i++) d[i] = subc_cc(a[i], b[i]);
        const bool lt = subc(0, 0) != 0;   // a < b
        const bool sw = odd & lt;          // the pair (a, u) <-> (b, v) changes roles
        nd[0] = sub_cc(0, d[0]);
#pragma unroll
        for (int i = 1; i < ZKP_FR_NL - 1; i++) nd[i] = subc_cc(0, d[i]);
        nd[ZKP_FR_NL - 1] = subc(0, d[ZKP_FR_NL - 1]);
#pragma unroll
        for (int i = 0; i < ZKP_FR_NL; i++) {
            uint32_t na = odd ? (lt ? nd[i] : d[i]) : a[i];
            b[i] = sw ? a[i] : b[i];
            a[i] = na;
        }
#pragma unroll
        for (int i = 0; i < ZKP_FR_NL - 1; i++) a[i] = (a[i] >> 1) | (a[i + 1] << 31);
        a[ZKP_FR_NL - 1] >>= 1;
#pragma unroll
        for (int i = 0; i < ZKP_FR_NL; i++) {
            uint32_t tu = sw ? v[i] : u[i];
            v[i] = sw ? u[i] : v[i];
            u[i] = tu;
        }
        // u <- odd ? (u - v mod r) : u
        w[0] = sub_cc(u[0], v[0]);
#pragma unroll
        for (int i = 1; i < ZKP_FR_NL; i++) w[i] = subc_cc(u[i], v[i]);
        const uint32_t mneg = subc(0, 0) != 0 ? 0xffffffffu : 0u;
        w[0] = add_cc(w[0], ZKP_R_ORDER[0] & mneg);
#pragma unroll
        for (int i = 1; i < ZKP_FR_NL - 1; i++) w[i] = addc_cc(w[i], ZKP_R_ORDER[i] & mneg);
        w[ZKP_FR_NL - 1] = addc(w[ZKP_FR_NL - 1], ZKP_R_ORDER[ZKP_FR_NL - 1] & mneg);
#pragma unroll
        for (int i = 0; i < ZKP_FR_NL; i++) u[i] = odd ? w[i] : u[i];
        // u <- u / 2 mod r: (u + r) / 2 when u is odd; u + r < 2^256 (r < 2^255), no carry out of the top word
        const uint32_t modd = (u[0] & 1u) ? 0xffffffffu : 0u;
        w[0] = add_cc(u[0], ZKP_R_ORDER[0] & modd);
#pragma unroll
        for (int i = 1; i < ZKP_FR_NL - 1; i++) w[i] = addc_cc(u[i], ZKP_R_ORDER[i] & modd);
        w[ZKP_FR_NL - 1] = addc(u[ZKP_FR_NL - 1], ZKP_R_ORDER[ZKP_FR_NL - 1] & modd);
#pragma unroll
        for (int i = 0; i < ZKP_FR_NL - 1; i++) u[i] = (w[i] >> 1) | (w[i + 1] << 31);
        u[ZKP_FR_NL - 1] = w[ZKP_FR_NL - 1] >> 1;
    }
    Fr r;
#pragma unroll
    for (int i = 0; i < ZKP_FR_NL; i++) r.l[i] = v[i];
    return fr_mul_const(r, ZKP_FR_R3);
}

}  // namespace zkp
