// DEV SIMULATION of the KZG front end (zkvm_pairings_b200/csrc/kzg.cuh) for the CPU tests of tests/test_kzg.py: the
// simulation of sim.cpp (lane pairs as two host threads in lock-step) plus the bodies of k_g16_window_tables (for the
// G1 generator) and k_kzg_prepare.  TEST INFRASTRUCTURE ONLY, built into tests/host_sim/libzkpair_sim_kzg.so.
#include "sim.cpp"

#include "../../zkvm_pairings_b200/csrc/kzg.cuh"

extern "C" {
// The setup's window table of g1 (canonical x|y): ZKP_G16_TABLE_FP Montgomery Fp, as on the device
void sim_kzg_table(const uint64_t *g1, uint64_t *table) {
    zkp_sim_par = 0;
    static Fp zs[ZKP_G16_DIGITS], pre[ZKP_G16_DIGITS];
    for (int w = 0; w < ZKP_G16_WINDOWS; w++) groth16_window_table(g1, w, (Fp *)table + (size_t)w * ZKP_G16_DIGITS * 2, zs, pre);
}
// z -> (z_hi, z_lo), z = z_hi x^2 + z_lo
void sim_kzg_glv_split(const uint64_t *z, uint64_t *hi, uint64_t *lo) { kzg_glv_split(z, hi, lo); }
// the per-proof body of k_kzg_prepare over n proofs
void sim_kzg_prepare(const uint64_t *table, const uint64_t *proofs, const uint8_t *proof_inf, const uint64_t *zy, size_t n, uint64_t *g1,
                     uint8_t *g1inf, uint8_t *status) {
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            uint8_t s = kzg_prepare_one((const Fp *)table, proofs + 24 * i, proof_inf ? proof_inf + 2 * i : nullptr, zy + 8 * i, g1 + 24 * i,
                                        g1inf + 2 * i);
            if (lane_par() == 0) status[i] = s;
        }
    });
}
}
