// Multi-scalar multiplication sum_i [k_i]P_i over caller-given G1 or G2 points (zkp_g1_msm / zkp_g2_msm): Pippenger with
// signed c-bit digits.  The scalars are 256-bit integers, not reduced mod r, and no endomorphism is used, so the sum is
// exact for any points on the curve, in the prime-order subgroup or not.
//
//   1. check   one thread (G1) or lane pair (G2) per point: canonical limbs, on the curve; the Montgomery affine point
//   2. count   one thread per point: the scalar's signed digits; a histogram of (window, |digit|) buckets
//   3. scan    one block: exclusive prefix sums of the histogram (bucket offsets in the sorted list)
//   4. scatter one thread per point: the digits again, each non-zero one placed at its bucket's next slot as
//              (key = window * M + |d| - 1, value = point index | sign << 31)
//   5. levels  fixed-length segments of the sorted list, one thread (G1) or lane pair (G2) each: the segment's runs of
//              equal key are summed; a run that starts in the segment is added into its bucket, the first run of a
//              segment that began in an earlier segment leaves its partial (and key) in the next level's list.  That
//              list is sorted by key again and 1/ZKP_MSM_SEG as long, and the same step runs over it until one segment
//              remains.  No thread sums more than ZKP_MSM_SEG entries per level, whatever the scalars are.
//   6. reduce  one block per window: ranges of buckets give their running sum R and weighted sum S; the window's
//              sum_j j B_j is the sum over ranges of S + (a - 1) R (a = the range's first digit), by a tree
//   7. combine one thread (G1) or lane pair (G2): Horner over the windows, c doublings per window
//
// Shared by the CUDA kernels (kernels.cu) and the CPU dev simulation of the not-gpu tests: every step is a function of
// a thread index over plain arrays.  Jacobian and affine values live in Fp arrays: a G1 coordinate is one Fp, a G2
// coordinate two (c0, c1), of which each lane of the pair reads and writes its own (tower.cuh's lane split).
#pragma once
#include "groth16.cuh"

namespace zkp {

#define ZKP_MSM_SEG 32          // entries per segment of the bucket accumulation (one thread or lane pair each)
#define ZKP_MSM_RANGES 128      // bucket ranges per window in the reduction (one block per window)
#define ZKP_MSM_SCAN_TPB 1024   // threads of the one-block histogram scan

// The window width for a chunk of n points, in steps from the widths measured fastest on a B200 (DESIGN.md section
// 3.9): c = 10 at 2^16 points, 14 at 2^20, 15 at 2^22.  The per-window bucket reduction is the reason they sit below
// the additions-only optimum ((ceil(256 / c) + 1) (n + 2^c) additions: 12, 16, 17).
ZKP_HOSTDEV int msm_window(size_t n) {
    return n < ((size_t)1 << 13) ? 8 : n < ((size_t)1 << 18) ? 10 : n < ((size_t)1 << 21) ? 14 : 15;
}
// windows of c-bit signed digits of a 256-bit integer: one more than the 256 bits need when c divides 256, for the
// carry out of the top window; otherwise the top window has fewer than c bits and never carries
ZKP_HOSTDEV int msm_windows(int c) { return 256 / c + 1; }
// accumulation levels for a sorted list of at most m entries: until one segment remains
ZKP_HOSTDEV int msm_levels(size_t m) {
    int lv = 0;
    do {
        m = (m + ZKP_MSM_SEG - 1) / ZKP_MSM_SEG;
        lv++;
    } while (m > 1);
    return lv;
}

// c bits of the 256-bit integer k (four little-endian u64) from bit pos; bits at 256 and above read as 0
ZKP_HD uint32_t msm_bits(const uint64_t *k, int pos, int c) {
    if (pos >= 256) return 0;
    const int li = pos >> 6, sh = pos & 63;
    uint64_t v = k[li] >> sh;
    if (sh + c > 64 && li < 3) v |= k[li + 1] << (64 - sh);
    return (uint32_t)(v & (((uint64_t)1 << c) - 1));
}
// msm_digit's rule at width c: window w's bits plus the carry of window w - 1; a sum above 2^(c-1) becomes sum - 2^c
// and carries 1 into window w + 1.  Digits lie in [-(2^(c-1) - 1), 2^(c-1)], and sum_w d_w 2^(c w) = k.
ZKP_HD int msm_digit_c(const uint64_t *k, int w, int c, uint32_t &carry) {
    const int d = (int)msm_bits(k, c * w, c) + (int)carry;
    carry = d > (1 << (c - 1)) ? 1u : 0u;
    return carry ? d - (1 << c) : d;
}

// ------------------------------------------------------------------ Fp-array storage of both groups' coordinates

ZKP_HD void msm_ld(Fp &r, const Fp *p, size_t k) { r = p[k]; }
ZKP_HD void msm_ld(Fp2 &r, const Fp *p, size_t k) { r.c = p[2 * k + lane_par()]; }
ZKP_HD void msm_st(Fp *p, size_t k, const Fp &v) { p[k] = v; }
ZKP_HD void msm_st(Fp *p, size_t k, const Fp2 &v) { p[2 * k + lane_par()] = v.c; }
template <class O>
ZKP_HD void msm_ldj(Jac<O> &r, const Fp *p, size_t k) {
    msm_ld(r.x, p, 3 * k);
    msm_ld(r.y, p, 3 * k + 1);
    msm_ld(r.z, p, 3 * k + 2);
}
template <class O>
ZKP_HD void msm_stj(Fp *p, size_t k, const Jac<O> &v) {
    msm_st(p, 3 * k, v.x);
    msm_st(p, 3 * k + 1, v.y);
    msm_st(p, 3 * k + 2, v.z);
}
template <class O>
ZKP_HD void msm_id(Jac<O> &p) {
    p.x = O::zero();
    p.y = O::one();
    p.z = O::zero();
}
// Fp per coordinate (W) and limbs of a boundary point (U64)
template <class O> struct MsmWidth { enum { W = 1, U64 = 12 }; };
template <> struct MsmWidth<OpsFp2> { enum { W = 2, U64 = 24 }; };
// the lane that writes a point's bytes and flags: every G1 thread, the even lane of a G2 pair
template <class O>
ZKP_HD bool msm_writer() { return MsmWidth<O>::W == 1 || lane_par() == 0; }

ZKP_HD void msm_or(uint32_t *p, uint32_t v) {
#ifdef ZKP_DEVICE_BUILD
    atomicOr(p, v);
#else
    *p |= v;
#endif
}

// A slot of ctr[key] for this thread (live) among all threads that claim from the same key: *ctr grows by the number
// of claims.  On the device the lanes of a warp with equal keys are served by one atomic (the all-equal-scalars case
// would otherwise serialise on one address); every lane of the warp must call it together.
ZKP_HD uint32_t msm_claim(uint32_t *ctr, uint32_t key, bool live) {
#ifdef ZKP_DEVICE_BUILD
    const unsigned peers = __match_any_sync(0xffffffffu, live ? key : 0xffffffffu);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    uint32_t base = 0;
    if (live && lane == leader) base = atomicAdd(ctr + key, (uint32_t)__popc(peers));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (uint32_t)__popc(peers & ((1u << lane) - 1u));
#else
    return live ? (*(ctr + key))++ : 0;
#endif
}

// ------------------------------------------------------------------ step 1: check

ZKP_HD void msm_load_affine(Fp &x, Fp &y, const uint64_t *xy, bool &bad) {
    x = load_fp(xy, bad);
    y = load_fp(xy + 6, bad);
}
ZKP_HD void msm_load_affine(Fp2 &x, Fp2 &y, const uint64_t *xy, bool &bad) {
    x = load_fp2(xy, bad);
    y = load_fp2(xy + 12, bad);
    bad = lane_or(bad);
}
// b of y^2 = x^3 + b: 4 on G1, 4 + 4u on G2 (both components 4)
ZKP_HD void msm_curve_b(Fp &b) { b = fp_const(ZKP_B1); }
ZKP_HD void msm_curve_b(Fp2 &b) { b.c = fp_const(ZKP_B1); }

// Point i: its Montgomery affine coordinates into pts (2 coordinates), valid[i] = 1 when it takes part (canonical,
// not flagged, on the curve).  A limb >= p ORs 1 into *err, an unflagged point off the curve 1 into *off.
template <class O>
ZKP_HD void msm_check(size_t i, const uint64_t *xy, const uint8_t *inf, Fp *pts, uint8_t *valid, uint32_t *off, uint32_t *err) {
    typedef typename O::T T;
    bool bad = false;
    T x, y, b;
    msm_load_affine(x, y, xy + (size_t)MsmWidth<O>::U64 * i, bad);
    msm_curve_b(b);
    const bool flagged = inf && inf[i];
    const bool on = O::is_zero(O::sub(O::sqr(y), O::add(O::mul(O::sqr(x), x), b)));
    msm_st(pts, 2 * i, x);
    msm_st(pts, 2 * i + 1, y);
    if (msm_writer<O>()) {
        valid[i] = (!bad && !flagged && on) ? 1 : 0;
        if (bad && err) msm_or(err, 1u);
        if (!bad && !flagged && !on) msm_or(off, 1u);
    }
}

// ------------------------------------------------------------------ steps 2 and 4: digits

// Thread i (every thread of the launch, i >= n included: the claims are warp-wide): the digits of scalar i, each
// non-zero one claiming a slot of its bucket in ctr.  Counting pass: keys == NULL, ctr = the histogram.  Scatter pass:
// ctr = the cursors (the offsets of step 3), and the entry is written at its slot.
ZKP_HD void msm_digits(size_t i, size_t n, const uint64_t *scalars, const uint8_t *valid, int c, uint32_t *ctr, uint32_t *keys,
                       uint32_t *vals) {
    const bool live = i < n && valid[i] != 0;
    const uint64_t *k = scalars + 4 * (live ? i : 0);
    const int nw = msm_windows(c), m = 1 << (c - 1);
    uint32_t carry = 0;
#pragma unroll 1
    for (int w = 0; w < nw; w++) {
        const int d = live ? msm_digit_c(k, w, c, carry) : 0;
        const uint32_t key = (uint32_t)(w * m + (d < 0 ? -d : d) - 1);
        const uint32_t slot = msm_claim(ctr, key, d != 0);
        if (keys && d != 0) {
            keys[slot] = key;
            vals[slot] = (uint32_t)i | (d < 0 ? 0x80000000u : 0u);
        }
    }
}

// ------------------------------------------------------------------ step 3: scan (one block of T threads)

// Step 3a, thread t: the sum of its range of the nb counts into part[t]
ZKP_HD void msm_scan_sum(int t, int T, const uint32_t *cnt, uint32_t nb, uint32_t *part) {
    const uint32_t lo = (uint32_t)((uint64_t)nb * t / T), hi = (uint32_t)((uint64_t)nb * (t + 1) / T);
    uint32_t s = 0;
    for (uint32_t j = lo; j < hi; j++) s += cnt[j];
    part[t] = s;
}
// Step 3b, one thread: part[] to exclusive prefix sums; the total (the sorted list's length) into *total and *len
ZKP_HD void msm_scan_prefix(int T, uint32_t *part, uint32_t *total, uint32_t *len) {
    uint32_t s = 0;
    for (int t = 0; t < T; t++) {
        const uint32_t v = part[t];
        part[t] = s;
        s += v;
    }
    *total = s;
    *len = s;
}
// Step 3c, thread t: the offsets of its range, into off and cur (the scatter's cursors)
ZKP_HD void msm_scan_write(int t, int T, const uint32_t *cnt, uint32_t nb, const uint32_t *part, uint32_t *off, uint32_t *cur) {
    const uint32_t lo = (uint32_t)((uint64_t)nb * t / T), hi = (uint32_t)((uint64_t)nb * (t + 1) / T);
    uint32_t s = part[t];
    for (uint32_t j = lo; j < hi; j++) {
        off[j] = s;
        cur[j] = s;
        s += cnt[j];
    }
}

// ------------------------------------------------------------------ step 5: bucket accumulation

// Segment s of a level's list of *len_in entries, seg entries long.  AFF (the first level): entry j is the affine point
// pts[vals[j] & 0x7fffffff], negated when bit 31 is set; otherwise the Jacobian point src[j].  Every run of equal keys
// that starts in the segment is added into buckets[key]; the segment's first run, when it began in an earlier segment,
// goes to (fkey[s], fval[s]) instead, and otherwise fval[s] is the identity under that run's key.  Exactly one run of a
// key starts in a list, so no two threads touch one bucket.  Segment 0 writes the next level's length.
template <class O, bool AFF>
ZKP_HD void msm_segment(size_t s, int seg, const uint32_t *len_in, uint32_t *len_out, const uint32_t *keys, const uint32_t *vals,
                        const Fp *src, Fp *buckets, uint32_t *fkey, Fp *fval) {
    const size_t m = *len_in, lo = s * (size_t)seg;
    if (s == 0 && msm_writer<O>()) *len_out = (uint32_t)((m + seg - 1) / seg);
    if (lo >= m) return;
    const size_t hi = lo + seg < m ? lo + seg : m;
    size_t j = lo;
    bool first = true;
#pragma unroll 1
    while (j < hi) {
        const uint32_t k = keys[j];
        const bool start = j == 0 || keys[j - 1] != k;
        Jac<O> acc;
        msm_id(acc);
#pragma unroll 1
        do {
            if (AFF) {
                const uint32_t v = vals[j];
                typename O::T x, y;
                msm_ld(x, src, 2 * (size_t)(v & 0x7fffffffu));
                msm_ld(y, src, 2 * (size_t)(v & 0x7fffffffu) + 1);
                if (v >> 31) y = O::sub(O::zero(), y);
                jac_add_affine(acc, acc, x, y);
            } else {
                Jac<O> e;
                msm_ldj(e, src, j);
                jac_add(acc, acc, e);
            }
            j++;
        } while (j < hi && keys[j] == k);
        if (first && msm_writer<O>()) fkey[s] = k;
        if (first && !start) {
            msm_stj(fval, s, acc);
        } else {
            if (first) {
                Jac<O> z;
                msm_id(z);
                msm_stj(fval, s, z);
            }
            Jac<O> b;
            msm_ldj(b, buckets, k);
            jac_add(b, b, acc);
            msm_stj(buckets, k, b);
        }
        first = false;
    }
}

// ------------------------------------------------------------------ step 6: bucket reduction

// Range q < R of window w (M buckets, digits 1 .. M; R divides M): with a = its first digit, the range's
// sum_j (j - a + 1) B_j by running sums, plus (a - 1) times its plain sum, into out.
template <class O>
ZKP_HD void msm_range(int w, int q, int R, int M, const Fp *buckets, Jac<O> &out) {
    const int per = M / R, a = q * per + 1;
    Jac<O> run, sum, t;
    msm_id(run);
    msm_id(sum);
    msm_id(t);
#pragma unroll 1
    for (int j = a + per - 1; j >= a; j--) {
        Jac<O> b;
        msm_ldj(b, buckets, (size_t)w * M + j - 1);
        jac_add(run, run, b);
        jac_add(sum, sum, run);
    }
    const uint32_t f = (uint32_t)(a - 1);
#pragma unroll 1
    for (int bit = 31; bit >= 0; bit--) {
        jac_double(t, t);
        if ((f >> bit) & 1) jac_add(t, t, run);
    }
    jac_add(out, sum, t);
}
// Tree step over the ranges' results sh[] (Fp-array storage): sh[q] += sh[q + h]
template <class O>
ZKP_HD void msm_tree_step(Fp *sh, int q, int h) {
    Jac<O> a, b;
    msm_ldj(a, sh, q);
    msm_ldj(b, sh, q + h);
    jac_add(a, a, b);
    msm_stj(sh, q, a);
}

// ------------------------------------------------------------------ step 7 and the folds

// Horner over the nw window sums: sum_w 2^(c w) W_w, into part (one Jacobian point)
template <class O>
ZKP_HD void msm_combine(int nw, int c, const Fp *wsum, Fp *part) {
    Jac<O> acc;
    msm_id(acc);
#pragma unroll 1
    for (int w = nw - 1; w >= 0; w--) {
#pragma unroll 1
        for (int i = 0; i < c; i++) jac_double(acc, acc);
        Jac<O> e;
        msm_ldj(e, wsum, w);
        jac_add(acc, acc, e);
    }
    msm_stj(part, 0, acc);
}
// the sum of np Jacobian points into out (a device's chunk partials)
template <class O>
ZKP_HD void msm_sum(const Fp *parts, int np, Fp *out) {
    Jac<O> acc;
    msm_id(acc);
    for (int i = 0; i < np; i++) {
        Jac<O> e;
        msm_ldj(e, parts, i);
        jac_add(acc, acc, e);
    }
    msm_stj(out, 0, acc);
}

ZKP_HD void msm_store_affine(uint64_t *xy, const Fp &x, const Fp &y) {
    store_fp(xy, x, nullptr);
    store_fp(xy + 6, y, nullptr);
}
ZKP_HD void msm_store_affine(uint64_t *xy, const Fp2 &x, const Fp2 &y) {
    store_fp2(xy, x, nullptr);
    store_fp2(xy + 12, y, nullptr);
}
// The call's result from np partials (one per device) and noff off-curve words: canonical affine limbs and the flag.
// The identity is (0, 1) with the flag set; a point off the curve gives zero limbs with the flag set and
// ZKP_POINT_NOT_ON_CURVE.  Returns the status.
template <class O>
ZKP_HD uint8_t msm_final(const Fp *parts, int np, const uint32_t *offs, int noff, uint64_t *out_xy, uint8_t *out_inf) {
    typedef typename O::T T;
    Jac<O> acc;
    msm_id(acc);
    for (int i = 0; i < np; i++) {
        Jac<O> e;
        msm_ldj(e, parts, i);
        jac_add(acc, acc, e);
    }
    bool off = false;
    for (int i = 0; i < noff; i++) off |= offs[i] != 0;
    const bool p_inf = O::is_zero(acc.z);
    T x = O::zero(), y = O::one();
    if (!p_inf) {
        T zi = O::inv(acc.z), zi2 = O::sqr(zi);
        x = O::mul(acc.x, zi2);
        y = O::mul(acc.y, O::mul(zi2, zi));
    }
    if (off) y = O::zero();
    if (off) x = O::zero();
    msm_store_affine(out_xy, x, y);
    if (msm_writer<O>()) *out_inf = (off || p_inf) ? 1 : 0;
    return off ? ZKP_POINT_NOT_ON_CURVE : ZKP_POINT_OK;
}

}  // namespace zkp
