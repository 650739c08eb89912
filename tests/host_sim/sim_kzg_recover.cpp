// DEV SIMULATION of cell recovery (zkvm_pairings_b200/csrc/kzg_recover.cuh) for the CPU tests of
// tests/test_kzg_recover.py: the simulation of sim_kzg_cells.cpp plus the body of k_cells_recover over the two halves
// of a cluster, each step in a loop over the ranks and thread indices where the kernel separates steps with
// __syncthreads() or a cluster barrier.  TEST INFRASTRUCTURE ONLY, built into tests/host_sim/libzkpair_sim_kzg_recover.so.
#include "sim_kzg_cells.cpp"

#include "../../zkvm_pairings_b200/csrc/kzg_recover.cuh"

extern "C" {
// the body of k_cells_recover over n blobs: cell_indices (n x 128 u64), cells (n x 128 x 2048 bytes), num_cells (n)
// -> out (n x 128 x 2048 bytes), coeffs (n x 4096 x 4 u64 canonical, or NULL) and the statuses; vanish (n x 2 x 128 x
// 4 u64 Montgomery, or NULL) receives z_k and 1 / zc_k of every cell
void sim_cells_recover(const uint64_t *idx, const uint8_t *cells, const uint64_t *num, size_t n, const uint64_t *pw, uint8_t *out,
                       uint64_t *coeffs, uint8_t *status, uint64_t *vanish) {
    std::vector<Fr> x0(ZKP_RECOVER_HALF), x1(ZKP_RECOVER_HALF);
    Fr *half[2] = {x0.data(), x1.data()};
    RecoverShared sh[2];
    const Fr *w = (const Fr *)pw;
    for (size_t b = 0; b < n; b++) {
        const uint64_t *bi = idx + b * ZKP_CELLS_PER_BLOB;
        const uint8_t *bc = cells + b * ZKP_CELLS_PER_BLOB * ZKP_CELL_BYTES_;
        for (int r = 0; r < 2; r++) {
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_init(t, num[b], sh[r]);
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_index(t, num[b], bi, sh[r]);
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_vanish_part(r, t, w, sh[r], half[r]);
            for (int t = 0; t < ZKP_CELL_N; t++) recover_vanish(t, half[r], sh[r]);
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_load(r, t, bc, sh[r], half[r]);
            if (vanish)
                for (int c = 0; c < ZKP_CELL_N; c++) {
                    ((Fr *)vanish)[(2 * b) * ZKP_CELLS_PER_BLOB + ZKP_CELL_N * r + c] = sh[r].z[c];
                    ((Fr *)vanish)[(2 * b + 1) * ZKP_CELLS_PER_BLOB + ZKP_CELL_N * r + c] = sh[r].zci[c];
                }
        }
        const bool rej = sh[0].bad_cells || sh[0].bad || sh[1].bad;
        for (int r = 0; r < 2; r++)
            for (int h = 1; h < ZKP_RECOVER_HALF; h <<= 1)
                for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_dit_pass(t, half[r], w, h);
        for (int r = 0; r < 2; r++)
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_cross_a(r, t, w, half);
        for (int r = 0; r < 2; r++) {
            for (int h = ZKP_RECOVER_HALF / 2; h >= 1; h >>= 1)
                for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_dif_pass(t, half[r], w, h);
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_divide(t, sh[r], half[r]);
            for (int h = 1; h < ZKP_RECOVER_HALF; h <<= 1)
                for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_dit_pass(t, half[r], w, h);
        }
        for (int r = 0; r < 2; r++)
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_cross_b(r, t, w, half, coeffs ? (Fr *)coeffs + b * ZKP_BLOB_N : nullptr);
        for (int r = 0; r < 2; r++) {
            for (int h = ZKP_RECOVER_HALF / 2; h >= 1; h >>= 1)
                for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_dif_pass(t, half[r], w, h);
            for (int t = 0; t < ZKP_CELLS_TPB; t++) recover_store(r, t, half[r], rej, out + b * 2 * ZKP_BLOB_BYTES_);
        }
        status[b] = recover_status(sh[0], sh[1].bad != 0);
    }
}
}
