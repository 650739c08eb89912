// DEV SIMULATION of the EIP-4844 blob front end (zkvm_pairings_b200/csrc/fr.cuh, blob.cuh) for the CPU tests of
// tests/test_kzg_blob.py: the simulation of sim.cpp plus the Fr arithmetic, the setup's domain body, the transcript of
// k_blob_challenge and the block-wide evaluation of k_blob_eval, whose steps run here in a loop over the thread indices
// where the kernel separates them with __syncthreads().  TEST INFRASTRUCTURE ONLY, built into
// tests/host_sim/libzkpair_sim_kzg_blob.so.
#include "sim.cpp"

#include <vector>

#include "../../zkvm_pairings_b200/csrc/blob.cuh"

static Fr fr_load(const uint64_t *a) {
    Fr r;
    for (int i = 0; i < 4; i++) {
        r.l[2 * i] = (uint32_t)a[i];
        r.l[2 * i + 1] = (uint32_t)(a[i] >> 32);
    }
    return r;
}
static void fr_store(uint64_t *o, const Fr &a) {
    for (int i = 0; i < 4; i++) o[i] = ((uint64_t)a.l[2 * i + 1] << 32) | a.l[2 * i];
}

extern "C" {
// canonical a, b < r (four u64 limbs each) -> canonical op(a, b): 0 add, 1 sub, 2 mul, 3 inv (b unused); the operands
// go through fr_to_mont and the result through fr_from_mont, as on the device
void sim_fr_op(int op, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n) {
    for (size_t i = 0; i < n; i++) {
        Fr x = fr_to_mont(fr_load(a + 4 * i)), y = fr_to_mont(fr_load(b + 4 * i)), r;
        switch (op) {
            case 0: r = fr_add(x, y); break;
            case 1: r = fr_sub(x, y); break;
            case 2: r = fr_mul(x, y); break;
            default: r = fr_inv(x); break;
        }
        fr_store(out + 4 * i, fr_from_mont(r));
    }
}
// op (0 add, 1 sub, 2 mul) on two raw representatives (the operand bound is asserted: a representative >= r aborts)
void sim_fr_raw(int op, const uint64_t *a, const uint64_t *b, uint64_t *out) {
    const Fr x = fr_load(a), y = fr_load(b);
    fr_store(out, op == 0 ? fr_add(x, y) : op == 1 ? fr_sub(x, y) : fr_mul(x, y));
}
// the body of k_blob_domain: the 4096 entries of roots_brp as stored (Montgomery)
void sim_blob_domain(uint64_t *out) {
    for (int i = 0; i < ZKP_BLOB_N; i++) fr_store(out + 4 * i, blob_root(i));
}
// the 48-byte compressed encoding the transcript hashes, as 12 big-endian words
void sim_g1_compress(const uint64_t *xy, uint8_t inf, uint32_t *out) { g1_compress_words(xy, inf, out); }
// the body of k_blob_challenge over n blobs: digest (8 words, H0 first) and z
void sim_blob_challenge(const uint8_t *blobs, const uint64_t *proofs, const uint8_t *proof_inf, size_t n, uint32_t *digest,
                        uint64_t *zy) {
    for (size_t i = 0; i < n; i++)
        blob_challenge_one(blobs + i * ZKP_BLOB_BYTES_, proofs + 24 * i, proof_inf ? proof_inf[2 * i] : 0, digest + 8 * i, zy + 8 * i);
}
// the body of k_blob_eval over n blobs, z read from and y (or r | 0) written to zy; roots = the domain as stored
void sim_blob_eval(const uint8_t *blobs, const uint64_t *roots, uint64_t *zy, size_t n) {
    const Fr *rt = (const Fr *)roots;
    std::vector<BlobLane> lanes(ZKP_BLOB_TPB);
    BlobShared *sh = new BlobShared;
    for (size_t b = 0; b < n; b++) {
        const uint8_t *blob = blobs + b * ZKP_BLOB_BYTES_;
        uint64_t *o = zy + 8 * b;
        const Fr zm = blob_z_mont(o);
        blob_eval_init(*sh);
        for (int t = 0; t < ZKP_BLOB_TPB; t++) blob_eval_prefix(t, rt, zm, *sh, lanes[t]);
        for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1)
            for (int t = 0; t < w; t++) blob_tree_mul(sh->tree, w + t);
        blob_tree_invert_root(sh->tree);
        for (int w = 1; w < ZKP_BLOB_TPB; w <<= 1)
            for (int t = 0; t < w; t++) blob_tree_inv(sh->tree, w + t);
        for (int t = 0; t < ZKP_BLOB_TPB; t++) blob_eval_terms(t, blob, rt, zm, *sh, lanes[t]);
        for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1)
            for (int t = 0; t < w; t++) blob_tree_add(sh->tree, w + t);
        blob_eval_finish(*sh, zm, o);
    }
    delete sh;
}
}
