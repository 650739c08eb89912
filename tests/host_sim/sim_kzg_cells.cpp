// DEV SIMULATION of the EIP-7594 cell bodies (zkvm_pairings_b200/csrc/kzg_cells.cuh) for the CPU tests of
// tests/test_kzg_cells.py: the simulation of sim_kzg_prove.cpp plus the twiddle table, the block-wide extension of
// k_cells_extend, the chains of k_cells_quotient and the interpolation of k_cells_interp, whose steps run here in a
// loop over the thread indices where the kernels separate them with __syncthreads().  TEST INFRASTRUCTURE ONLY, built
// into tests/host_sim/libzkpair_sim_kzg_cells.so.
#include "sim_kzg_prove.cpp"

#include "../../zkvm_pairings_b200/csrc/kzg_cells.cuh"

extern "C" {
// pw[e] = omega_8192^e (Montgomery, 8192 x 4 u64), as k_cells_powers stores it
void sim_cells_powers(uint64_t *pw) {
    for (int e = 0; e < ZKP_CELLS_EXT_N; e++) ((Fr *)pw)[e] = cells_power(e);
}
// the body of k_cells_extend over n blobs: cells (n x 128 x 2048 bytes), coeffs (n x 4096 x 4 u64 canonical, or NULL)
// and the statuses
void sim_cells_extend(const uint8_t *blobs, size_t n, const uint64_t *pw, uint8_t *cells, uint64_t *coeffs, uint8_t *status) {
    std::vector<Fr> x(ZKP_BLOB_N);
    const Fr *w = (const Fr *)pw;
    for (size_t b = 0; b < n; b++) {
        const uint8_t *blob = blobs + b * ZKP_BLOB_BYTES_;
        uint32_t bad = 0;
        for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_load(t, blob, x.data(), &bad);
        for (int h = 1; h < ZKP_BLOB_N; h <<= 1)
            for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_dit_pass(t, x.data(), w, h);
        for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_scale(t, x.data(), w, coeffs ? (Fr *)coeffs + b * ZKP_BLOB_N : nullptr);
        for (int h = ZKP_BLOB_N / 2; h >= 1; h >>= 1)
            for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_dif_pass(t, x.data(), w, h);
        for (int t = 0; t < ZKP_CELLS_TPB; t++) cells_store(t, blob, x.data(), bad != 0, cells + b * 2 * ZKP_BLOB_BYTES_);
        status[b] = bad ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
    }
}
// the chains of k_cells_quotient for the cosets ks[0 .. nk) of one blob: rows (nk x 4096 x 32 bytes)
void sim_cells_quotient(const uint64_t *coeffs, const uint64_t *pw, const int32_t *ks, size_t nk, uint8_t *rows) {
    for (size_t r = 0; r < nk; r++)
        for (int m = 0; m < ZKP_CELL_N; m++) cells_quotient_chain(ks[r], m, (const Fr *)coeffs, (const Fr *)pw, rows + r * ZKP_BLOB_BYTES_);
}
// the interpolation steps of k_cells_interp over n cells: I_k's coefficients as big-endian rows (n x 2048 bytes) and
// the status of the front (ZKP_KZG_BAD_SCALAR for an element >= r or an index >= 128)
void sim_cells_interp(const uint8_t *cells, const uint64_t *idx, size_t n, const uint64_t *pw, uint8_t *rows, uint8_t *status) {
    CellShared *sh = new CellShared;
    for (size_t c = 0; c < n; c++) {
        cell_init(*sh, idx[c]);
        for (int t = 0; t < ZKP_CELL_N; t++) cell_load(t, cells + c * ZKP_CELL_BYTES_, *sh);
        for (int h = 1; h < ZKP_CELL_N; h <<= 1)
            for (int t = 0; t < ZKP_CELL_N / 2; t++) cells_dit(sh->x, (const Fr *)pw, t, h);
        for (int t = 0; t < ZKP_CELL_N; t++) cell_interp_scale(t, idx[c], (const Fr *)pw, *sh);
        memcpy(rows + c * ZKP_CELL_BYTES_, sh->row, ZKP_CELL_BYTES_);
        status[c] = sh->bad ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
    }
    delete sh;
}
}
