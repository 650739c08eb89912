// DEV SIMULATION of the EIP-4844 prover front end (zkvm_pairings_b200/csrc/kzg_prove.cuh) for the CPU tests of
// tests/test_kzg_prove.py: the simulation of sim_kzg_blob.cpp plus the signed-digit recoding and window tables of the
// fixed-base MSM, the front of compute_blob_kzg_proof and the block-wide quotient of k_kzg_quotient, whose steps run
// here in a loop over the thread indices where the kernel separates them with __syncthreads().  TEST INFRASTRUCTURE
// ONLY, built into tests/host_sim/libzkpair_sim_kzg_prove.so.
#include "sim_kzg_blob.cpp"

#include "../../zkvm_pairings_b200/csrc/kzg_prove.cuh"

extern "C" {
// the 32 signed digits of a scalar given as 32 big-endian bytes (any 256-bit value), then the carry out of the top window
void sim_msm_digits(const uint8_t *be32, int32_t *digits) {
    uint32_t w[8], s[8], carry = 0;
    load_be16(be32, w);
    load_be16(be32 + 16, w + 4);
    for (int k = 0; k < 8; k++) s[k] = w[7 - k];
    for (int i = 0; i < ZKP_MSM_WINDOWS; i++) digits[i] = msm_digit(s, i, carry);
    digits[ZKP_MSM_WINDOWS] = (int32_t)carry;
}
// the window table of one base (canonical x|y) and window w as the setup stores it, converted to canonical x|y limbs:
// entry d - 1 = d 2^(8w) P for d = 1 .. 128
void sim_msm_table(const uint64_t *xy, int w, uint64_t *out) {
    std::vector<Fp> tab(2 * ZKP_MSM_DIGITS), zs(2 * ZKP_MSM_DIGITS);
    groth16_window_table(xy, w, tab.data(), zs.data(), zs.data() + ZKP_MSM_DIGITS, ZKP_MSM_DIGITS);
    for (int d = 0; d < 2 * ZKP_MSM_DIGITS; d++) store_fp(out + 6 * d, tab[d], nullptr);
}
// the body of k_kzg_prove_challenge over n blobs (commitments n x 12, flags or NULL)
void sim_kzg_prove_challenge(const uint8_t *blobs, const uint64_t *c, const uint8_t *cinf, size_t n, uint64_t *zy, uint8_t *status) {
    for (size_t i = 0; i < n; i++) status[i] = prove_challenge_one(blobs + i * ZKP_BLOB_BYTES_, c + 12 * i, cinf ? cinf[i] : 0, zy + 8 * i);
}
// the body of k_kzg_quotient over n blobs: z from z_in (or NULL: already in zy), y to y_out (or NULL), the quotient
// rows (n x 4096 x 32 big-endian bytes), the statuses (pre = earlier rejections or NULL); roots = the domain as stored
void sim_kzg_quotient(const uint8_t *blobs, const uint64_t *roots, const uint64_t *z_in, size_t n, uint64_t *zy, uint64_t *y_out,
                      uint8_t *rows, const uint8_t *pre, uint8_t *status) {
    const Fr *rt = (const Fr *)roots;
    std::vector<BlobLane> lanes(ZKP_BLOB_TPB);
    QuotShared *sh = new QuotShared;
    for (size_t b = 0; b < n; b++) {
        const uint8_t *blob = blobs + b * ZKP_BLOB_BYTES_;
        uint8_t *row = rows + b * ZKP_BLOB_BYTES_;
        uint64_t *o = zy + 8 * b;
        const uint8_t p = pre ? pre[b] : 0;
        quot_init(*sh, z_in ? z_in + 4 * b : nullptr, o);
        const Fr zm = sh->zm;
        for (int t = 0; t < ZKP_BLOB_TPB; t++) blob_eval_prefix(t, rt, zm, sh->b, lanes[t]);
        for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1)
            for (int t = 0; t < w; t++) blob_tree_mul(sh->b.tree, w + t);
        blob_tree_invert_root(sh->b.tree);
        for (int w = 1; w < ZKP_BLOB_TPB; w <<= 1)
            for (int t = 0; t < w; t++) blob_tree_inv(sh->b.tree, w + t);
        for (int t = 0; t < ZKP_BLOB_TPB; t++) blob_eval_terms<true>(t, blob, rt, zm, sh->b, lanes[t], (Fr *)row);
        for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1)
            for (int t = 0; t < w; t++) blob_tree_add(sh->b.tree, w + t);
        blob_eval_finish(sh->b, zm, o);
        status[b] = quot_status(*sh, p, o, y_out ? y_out + 4 * b : nullptr);
        for (int t = 0; t < ZKP_BLOB_TPB; t++) quot_terms(t, blob, rt, *sh, row);
        if (sh->b.hit) {
            for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1)
                for (int t = 0; t < w; t++) blob_tree_add(sh->b.tree, w + t);
            quot_within_domain(*sh, row);
        }
    }
    delete sh;
}
}
