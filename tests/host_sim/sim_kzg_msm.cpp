// DEV SIMULATION of the prover's fixed-base MSM (zkvm_pairings_b200/csrc/kzg_prove.cuh: msm_partial, msm_tree_add,
// msm_finish; kernel k_kzg_msm) for the CPU tests of tests/test_kzg_msm_edges.py: the simulation of
// sim_kzg_prove.cpp plus the body of k_kzg_msm, whose steps run here in a loop over the thread indices where the kernel
// separates them with __syncthreads().  TEST INFRASTRUCTURE ONLY, built into tests/host_sim/libzkpair_sim_kzg_msm.so.
#include "sim_kzg_prove.cpp"

#include <stdlib.h>

extern "C" {
// The body of k_kzg_msm over n scalar rows (n x 4096 x 32 big-endian bytes; pre = earlier rejections or NULL).
// lag_brp = the Lagrange points in bit-reversed order, 4096 x 12 canonical limbs: only the bases with a non-zero
// element in some row are read, and only their window tables are built (128 signed digits, as k_kzg_lagrange_tables
// builds them).  The tables live in one zero-filled allocation of the full device layout, so the pages of unused bases
// are never touched: msm_partial reads a table only for a non-zero digit.  Returns -1 when that allocation fails.
int sim_kzg_msm(const uint64_t *lag_brp, const uint8_t *rows, const uint8_t *pre, size_t n, uint64_t *out, uint8_t *out_inf,
                uint8_t *status) {
    zkp_sim_par = 0;
    Fp *tables = (Fp *)calloc((size_t)ZKP_BLOB_N * ZKP_MSM_TABLE_FP, sizeof(Fp));
    if (!tables) return -1;
    std::vector<Fp> zs(2 * ZKP_MSM_DIGITS);
    for (int i = 0; i < ZKP_BLOB_N; i++) {
        bool used = false;
        for (size_t b = 0; b < n && !used; b++)
            for (int k = 0; k < 32; k++) used |= rows[b * ZKP_BLOB_BYTES_ + 32 * (size_t)i + k] != 0;
        if (!used) continue;
        for (int w = 0; w < ZKP_MSM_WINDOWS; w++)
            groth16_window_table(lag_brp + 12 * i, w, tables + (size_t)i * ZKP_MSM_TABLE_FP + (size_t)w * ZKP_MSM_DIGITS * 2,
                                 zs.data(), zs.data() + ZKP_MSM_DIGITS, ZKP_MSM_DIGITS);
    }
    MsmShared *sh = new MsmShared;
    for (size_t b = 0; b < n; b++) {
        const uint8_t p = pre ? pre[b] : 0;
        msm_init(*sh);
        for (int t = 0; t < ZKP_MSM_TPB; t++) msm_partial(t, tables, rows + b * ZKP_BLOB_BYTES_, p != 0, *sh);
        for (int w = ZKP_MSM_TPB / 2; w >= 1; w >>= 1)
            for (int t = 0; t < w; t++) msm_tree_add(*sh, t, w);
        status[b] = msm_finish(*sh, p, out + 12 * b, out_inf + b);
    }
    delete sh;
    free(tables);
    return 0;
}
}
