// DEV SIMULATION of the multi-scalar multiplication (zkvm_pairings_b200/csrc/msm.cuh) for the CPU tests of
// tests/test_msm.py: every step of zkp_g1_msm / zkp_g2_msm, run here in a loop over the thread indices where the kernels
// launch one thread (G1) or lane pair (G2) per index, at window widths, segment lengths and range counts the caller
// chooses (small ones crowd the buckets and make segments cross them; a segment length of 1 applies to the first level,
// the later ones take 2).  TEST INFRASTRUCTURE ONLY, built into
// tests/host_sim/libzkpair_sim_msm.so.
#include "sim.cpp"

#include <vector>

#include "../../zkvm_pairings_b200/csrc/msm.cuh"

template <class O>
static void sim_msm_run(const uint64_t *xy, const uint8_t *inf, const uint64_t *scalars, size_t n, int c, int seg, int R, uint64_t *out_xy,
                        uint8_t *out_inf, uint8_t *status, uint32_t *err) {
    const int W = MsmWidth<O>::W, nw = msm_windows(c), M = 1 << (c - 1);
    const size_t nb = (size_t)nw * M, emax = (size_t)nw * n, s0 = (emax + seg - 1) / seg + 1;
    std::vector<Fp> pts(2 * W * n + 1), buckets(3 * W * nb), wsum(3 * W * nw), part(3 * W), fval[2] = {std::vector<Fp>(3 * W * s0), std::vector<Fp>(3 * W * s0)};
    std::vector<uint8_t> valid(n + 1);
    std::vector<uint32_t> cnt(nb), off(nb + 1), cur(nb), keys(emax + 1), vals(emax + 1), fkey[2] = {std::vector<uint32_t>(s0), std::vector<uint32_t>(s0)};
    std::vector<uint32_t> lens(64);
    uint32_t off_curve = 0;
    auto lanes = [&](auto f) {
        if (W == 2) {
            run_pair(f);
        } else {
            zkp_sim_par = 0;
            f();
        }
    };
    lanes([&]() {
        for (size_t i = 0; i < n; i++) msm_check<O>(i, xy, inf, pts.data(), valid.data(), &off_curve, err);
    });
    zkp_sim_par = 0;
    for (size_t i = 0; i < n; i++) msm_digits(i, n, scalars, valid.data(), c, cnt.data(), nullptr, nullptr);
    const int T = 7;   // scan threads (a count that does not divide the buckets)
    uint32_t part_sums[T];
    for (int t = 0; t < T; t++) msm_scan_sum(t, T, cnt.data(), (uint32_t)nb, part_sums);
    msm_scan_prefix(T, part_sums, &off[nb], &lens[0]);
    for (int t = 0; t < T; t++) msm_scan_write(t, T, cnt.data(), (uint32_t)nb, part_sums, off.data(), cur.data());
    for (size_t i = 0; i < n; i++) msm_digits(i, n, scalars, valid.data(), c, cur.data(), keys.data(), vals.data());
    lanes([&]() {
        size_t m = emax;
        for (int lv = 0; m > 1 || lv == 0; lv++) {
            const int sl = lv == 0 || seg > 1 ? seg : 2;   // a list shrinks only under segments of 2 or more
            const size_t nseg = (m + sl - 1) / sl;
            const int o = lv & 1, i = o ^ 1;
            for (size_t s = 0; s < nseg; s++) {
                if (lv == 0)
                    msm_segment<O, true>(s, sl, &lens[0], &lens[1], keys.data(), vals.data(), pts.data(), buckets.data(), fkey[0].data(),
                                         fval[0].data());
                else
                    msm_segment<O, false>(s, sl, &lens[lv], &lens[lv + 1], fkey[i].data(), nullptr, fval[i].data(), buckets.data(),
                                          fkey[o].data(), fval[o].data());
            }
            m = nseg;
        }
        int T2 = 1;
        while (T2 < R) T2 <<= 1;
        std::vector<Fp> sh(3 * W * T2);
        for (int w = 0; w < nw; w++) {
            for (int q = 0; q < T2; q++) {
                Jac<O> r;
                msm_id(r);
                if (q < R) msm_range<O>(w, q, R, M, buckets.data(), r);
                msm_stj(sh.data(), q, r);
            }
            for (int h = T2 / 2; h >= 1; h >>= 1)
                for (int q = 0; q < h; q++) msm_tree_step<O>(sh.data(), q, h);
            Jac<O> r;
            msm_ldj(r, sh.data(), 0);
            msm_stj(wsum.data(), w, r);
        }
        msm_combine<O>(nw, c, wsum.data(), part.data());
        const uint8_t st = msm_final<O>(part.data(), 1, &off_curve, 1, out_xy, out_inf);
        if (msm_writer<O>()) *status = st;
    });
}

extern "C" {
// the signed digits of one scalar at width c (msm_digits' recoding); returns the number of windows
int sim_msm_recode(const uint64_t *k, int c, int32_t *digits) {
    uint32_t carry = 0;
    const int nw = msm_windows(c);
    for (int w = 0; w < nw; w++) digits[w] = msm_digit_c(k, w, c, carry);
    return nw;
}
// the window width the library picks for a chunk of n points (ZKPAIR_MSM_WINDOW aside)
int sim_msm_window(size_t n) { return msm_window(n); }
// sum_i [k_i]P_i (g2: G2 points) through every step of the kernels; R ranges per window (R divides 2^(c-1))
void sim_msm(int g2, const uint64_t *xy, const uint8_t *inf, const uint64_t *scalars, size_t n, int c, int seg, int R, uint64_t *out_xy,
             uint8_t *out_inf, uint8_t *status, uint32_t *err) {
    if (g2) sim_msm_run<OpsFp2>(xy, inf, scalars, n, c, seg, R, out_xy, out_inf, status, err);
    else sim_msm_run<OpsFp>(xy, inf, scalars, n, c, seg, R, out_xy, out_inf, status, err);
}
}
