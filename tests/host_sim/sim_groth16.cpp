// DEV SIMULATION of the Groth16 front end (zkvm_pairings_b200/csrc/groth16.cuh) for the CPU tests of
// tests/test_groth16.py: the simulation of sim.cpp (lane pairs as two host threads in lock-step) plus the bodies of
// k_g16_window_tables and k_groth16_prepare.  TEST INFRASTRUCTURE ONLY, built into tests/host_sim/libzkpair_sim_g16.so.
#include "sim.cpp"

#include "../../zkvm_pairings_b200/csrc/groth16.cuh"

extern "C" {
// Window tables of IC_1 .. IC_l (ic = IC_0 .. IC_l): the body of k_g16_window_tables, one simulated thread per
// (IC_j, window); tables = n_public x ZKP_G16_TABLE_FP Montgomery Fp, as on the device.
void sim_g16_tables(const uint64_t *ic, const uint8_t *ic_inf, int n_public, uint64_t *tables) {
    zkp_sim_par = 0;
    static Fp zs[ZKP_G16_DIGITS], pre[ZKP_G16_DIGITS];
    for (int j = 0; j < n_public; j++) {
        if (ic_inf && ic_inf[j + 1]) continue;
        for (int w = 0; w < ZKP_G16_WINDOWS; w++)
            groth16_window_table(ic + 12 * (j + 1), w, (Fp *)tables + (size_t)j * ZKP_G16_TABLE_FP + (size_t)w * ZKP_G16_DIGITS * 2, zs, pre);
    }
}
// entry (IC_j, window w, digit d) of such tables as canonical x|y
void sim_g16_table_entry(const uint64_t *tables, int j, int w, int d, uint64_t *xy) {
    zkp_sim_par = 0;
    const Fp *e = (const Fp *)tables + (size_t)j * ZKP_G16_TABLE_FP + 2 * (w * ZKP_G16_DIGITS + d - 1);
    store_fp(xy, e[0], nullptr);
    store_fp(xy + 6, e[1], nullptr);
}
// the per-proof body of k_groth16_prepare over n proofs
void sim_g16_prepare(const uint64_t *alpha, const uint64_t *ic0, const uint8_t *ic_inf, const uint64_t *tables, int n_public,
                     const uint64_t *proofs, const uint8_t *proof_inf, const uint64_t *x, size_t n, uint64_t *g1, uint8_t *g1inf,
                     uint64_t *g2, uint8_t *g2inf, uint8_t *status) {
    G16Key vk = {alpha, ic0, ic_inf, (const Fp *)tables, n_public};
    run_pair([&]() {
        for (size_t i = 0; i < n; i++) {
            uint8_t s = groth16_prepare_one(vk, proofs + 48 * i, proof_inf ? proof_inf + 3 * i : nullptr, x + (size_t)n_public * 4 * i,
                                            g1 + 48 * i, g1inf + 4 * i, g2 + 24 * i, g2inf + i);
            if (lane_par() == 0) status[i] = s;
        }
    });
}
}
