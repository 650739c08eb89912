// EIP-7594 cells (compute_cells, compute_cells_and_kzg_proofs and the per-cell check of verify_cell_kzg_proof_batch of
// the consensus specs, fulu polynomial-commitments-sampling.md).
//
// The extended domain is the 8192nd roots of unity in 13-bit bit-reversed order, and cell k holds its entries
// [64 k, 64 k + 64).  Entries 0 .. 4095 are the blob domain roots_brp, so cells 0 .. 63 are the blob's own bytes;
// entries 4096 + i are omega_8192 roots_brp[i], so cells 64 .. 127 are the size-4096 NTT of a_t omega_8192^t in
// bit-reversed order, a = the blob's coefficients.  The blob is in bit-reversed order already, so a decimation-in-time
// inverse NTT reads it as it is and gives natural-order coefficients; a decimation-in-frequency forward NTT of natural
// input gives bit-reversed output.  No permutation runs anywhere.
//
// Cell k's points are h_k omega_64^brp6(j), h_k = omega_8192^brp7(k), and its vanishing polynomial is X^64 - c_k with
// c_k = h_k^64 = omega_128^brp7(k).  Its proof is [q_k(tau)]G1 over the monomial setup, q_k = p div (X^64 - c_k), and
// the verifier checks e(C + [c_k]pi - [I_k(tau)]G1, G2) e(pi, -[tau^64]G2) == 1, I_k = the cell's interpolation
// polynomial (the remainder of that division).
//
// Every twiddle is an entry of one table pw[e] = omega_8192^e, e < 8192 (Montgomery), resident in a cells setup.
// Values stay canonical: a canonical value times a Montgomery twiddle is canonical.
//
// Shared by the CUDA kernels (kernels.cu) and the CPU dev simulation of the not-gpu tests.  As in blob.cuh, the
// block-wide steps are functions of one thread index over shared memory: the kernel calls them between
// __syncthreads(), the simulation in a loop over the thread indices.
#pragma once
#include "kzg_prove.cuh"

namespace zkp {

#define ZKP_CELLS_EXT_N 8192             // the extended domain
#define ZKP_CELLS_PER_BLOB 128           // CELLS_PER_EXT_BLOB (include/zkpair.h ZKP_CELLS_PER_EXT_BLOB)
#define ZKP_CELL_N 64                    // FIELD_ELEMENTS_PER_CELL
#define ZKP_CELL_BYTES_ (32 * ZKP_CELL_N)
#define ZKP_CELLS_TPB 512                // threads of one k_cells_extend block (one block per blob)
#define ZKP_CELLS_QUOT_TPB 256           // threads of one k_cells_quotient block (four cosets, one chain per thread)

// the 7-bit bit reversal of a cell index
ZKP_HD int cells_brp7(int k) {
    int e = 0;
    for (int b = 0; b < 7; b++) e |= ((k >> b) & 1) << (6 - b);
    return e;
}

// pw[e] = omega_8192^e (Montgomery), one entry; the setup's table is k_cells_powers over e < 8192
ZKP_HD Fr cells_power(int e) {
    Fr acc = fr_one(), base = fr_const(ZKP_FR_OMEGA_EXT);
    for (int b = 0; b < 13; b++) {
        if ((e >> b) & 1) acc = fr_mul(acc, base);
        base = fr_sqr(base);
    }
    return acc;
}

// One butterfly b < n/2 of the decimation-in-time inverse pass of half-length h (h = 1, 2, .. n/2 in turn): with
// lo = 2b - j, j = b mod h, x[lo], x[lo + h] <- x[lo] +- omega_2h^-j x[lo + h].
ZKP_HD void cells_dit(Fr *x, const Fr *pw, int b, int h) {
    const int j = b & (h - 1), lo = 2 * b - j;
    const Fr v = fr_mul(x[lo + h], pw[(ZKP_CELLS_EXT_N - j * (ZKP_CELLS_EXT_N / (2 * h))) & (ZKP_CELLS_EXT_N - 1)]);
    const Fr u = x[lo];
    x[lo] = fr_add(u, v);
    x[lo + h] = fr_sub(u, v);
}
// One butterfly of the decimation-in-frequency forward pass of half-length h (h = n/2, .. 2, 1 in turn):
// x[lo], x[lo + h] <- x[lo] + x[lo + h], (x[lo] - x[lo + h]) omega_2h^j.
ZKP_HD void cells_dif(Fr *x, const Fr *pw, int b, int h) {
    const int j = b & (h - 1), lo = 2 * b - j;
    const Fr u = x[lo], v = x[lo + h];
    x[lo] = fr_add(u, v);
    x[lo + h] = fr_mul(fr_sub(u, v), pw[j * (ZKP_CELLS_EXT_N / (2 * h))]);
}

// ------------------------------------------------------------------ k_cells_extend: compute_cells, one blob per block

// Step 1, thread t: its elements i = t + TPB k into x (an element >= r reads as 0 and sets *bad)
ZKP_HD void cells_load(int t, const uint8_t *blob, Fr *x, uint32_t *bad) {
    bool b = false;
    for (int k = 0; k < ZKP_BLOB_N / ZKP_CELLS_TPB; k++) {
        const int i = t + ZKP_CELLS_TPB * k;
        b |= !blob_element(blob, i, x[i]);
    }
    if (b) *bad = 1;
}
// Steps 2 (h = 1 .. 2048, the inverse NTT) and 4 (h = 2048 .. 1, the forward NTT), thread t: its butterflies t + TPB k
ZKP_HD void cells_dit_pass(int t, Fr *x, const Fr *pw, int h) {
    for (int k = 0; k < ZKP_BLOB_N / 2 / ZKP_CELLS_TPB; k++) cells_dit(x, pw, t + ZKP_CELLS_TPB * k, h);
}
ZKP_HD void cells_dif_pass(int t, Fr *x, const Fr *pw, int h) {
    for (int k = 0; k < ZKP_BLOB_N / 2 / ZKP_CELLS_TPB; k++) cells_dif(x, pw, t + ZKP_CELLS_TPB * k, h);
}
// Step 3, thread t: a_i = x_i / 4096 (the coefficients, also to coeffs when it is not NULL), then x_i = a_i omega_8192^i
ZKP_HD void cells_scale(int t, Fr *x, const Fr *pw, Fr *coeffs) {
    for (int k = 0; k < ZKP_BLOB_N / ZKP_CELLS_TPB; k++) {
        const int i = t + ZKP_CELLS_TPB * k;
        const Fr a = fr_mul_const(x[i], ZKP_FR_INV_N);
        if (coeffs) coeffs[i] = a;
        x[i] = fr_mul(a, pw[i]);
    }
}
// Step 5, thread t: the 128 cells of the blob (256 KiB at out, 16-byte aligned): its 32-byte entries of the first half
// copied from the blob, of the second half x in big-endian bytes.  A blob with an element >= r gets zero cells.
ZKP_HD void cells_store(int t, const uint8_t *blob, const Fr *x, bool bad, uint8_t *out) {
    for (int k = 0; k < ZKP_BLOB_N / ZKP_CELLS_TPB; k++) {
        const int i = t + ZKP_CELLS_TPB * k;
        Fr v = fr_zero(), p = fr_zero();
        if (!bad) {
            blob_element(blob, i, p);
            v = x[i];
        }
        store_be32(out + 32 * i, p);
        store_be32(out + ZKP_BLOB_BYTES_ + 32 * i, v);
    }
}

// ------------------------------------------------------------------ k_cells_quotient: the 128 quotient rows of a blob

// One chain, thread (k, m): the entries j = m + 64 s of q_k = p div (X^64 - c_k), q_j = a_{j+64} + c_k q_{j+64} from
// the top down, into the row of coset k (4096 x 32 big-endian bytes, entries 4032 .. 4095 zero: the layout of a blob,
// so that k_kzg_msm runs over it against the monomial tables).  a = the blob's coefficients (canonical).
ZKP_HD void cells_quotient_chain(int k, int m, const Fr *a, const Fr *pw, uint8_t *row) {
    const Fr c = pw[ZKP_CELL_N * cells_brp7(k)];
    Fr q = fr_zero();
    store_be32(row + 32 * (ZKP_BLOB_N - ZKP_CELL_N + m), q);
#pragma unroll 1
    for (int s = ZKP_BLOB_N / ZKP_CELL_N - 2; s >= 0; s--) {
        const int j = m + ZKP_CELL_N * s;
        q = fr_add(a[j + ZKP_CELL_N], fr_mul(q, c));
        store_be32(row + 32 * j, q);
    }
}

// ------------------------------------------------------------------ verifier front end, one cell per 64-thread block

struct CellShared {
    Fr x[ZKP_CELL_N];
    alignas(16) uint8_t row[ZKP_CELL_BYTES_];   // I_k's coefficients, big-endian: the scalar row of the 64-base MSM
    MsmSharedN<ZKP_CELL_N> msm;
    uint32_t bad;   // an element >= r or an index >= 128
};

ZKP_HD void cell_init(CellShared &sh, uint64_t k) {
    sh.bad = k >= ZKP_CELLS_PER_BLOB ? 1u : 0u;
    msm_init(sh.msm);
}
// Step 1, thread t < 64: element t of the cell
ZKP_HD void cell_load(int t, const uint8_t *cell, CellShared &sh) {
    if (!blob_element(cell, t, sh.x[t])) sh.bad = 1;
}
// Step 2, h = 1 .. 32, thread t < 32: the size-64 inverse NTT (the cell's points are h_k omega_64^brp6(j))
// Step 3, thread t < 64: I_t = x_t / 64 h_k^-t, big-endian into the row
ZKP_HD void cell_interp_scale(int t, uint64_t k, const Fr *pw, CellShared &sh) {
    const int e = sh.bad ? 0 : cells_brp7((int)k) * t;   // h_k^-t = omega_8192^(8192 - brp7(k) t)
    Fr inv64 = fr_const(ZKP_FR_INV_N);
    for (int s = 0; s < 6; s++) inv64 = fr_add(inv64, inv64);
    store_be32(sh.row + 32 * t, fr_mul(fr_mul(sh.x[t], inv64), pw[(ZKP_CELLS_EXT_N - e) & (ZKP_CELLS_EXT_N - 1)]));
}
// Steps 4 - 6 are msm_partial<64> over the first 64 monomial tables, msm_tree_add and msm_finish: [I_k(tau)]G1, with
// pre = ZKP_KZG_BAD_SCALAR for a rejected cell.

// One cell, executed by a lane pair after the interpolation: C and pi validated (the even lane checks C, the odd lane
// pi; ZKP_KZG_BAD_POINT precedes the interpolation's status pre), then P = C + [c_k]pi - [I_k(tau)]G1 with c_k split
// as in kzg_prepare_one: the even lane computes [lo]pi + C, the odd lane [hi](beta x_pi, -y_pi) - I, and the two meet
// in one Jacobian addition.  Writes the pairs [P, pi] (g1, g1inf) of the prepared 2-pair check against G2 and
// -[tau^64]G2 and returns the status (both lanes); a rejected cell's slots hold zeros with both flags set.
ZKP_HD uint8_t cell_prepare_one(const uint64_t *c, uint8_t cinf, const uint64_t *pi, uint8_t qinf, uint64_t k, const Fr *pw,
                                const uint64_t *ixy, uint8_t iinf, uint8_t pre, uint64_t *g1, uint8_t *g1inf) {
    const int par = lane_par();
    bool bad = false;
    const uint8_t sp = g1_check_one(par ? pi : c, par ? qinf : cinf, bad);
    const bool bad_point = lane_or(bad | (sp != ZKP_POINT_OK));
    const uint8_t st = bad_point ? ZKP_KZG_BAD_POINT : pre;
    const bool rej = st != ZKP_KZG_VALID;

    Jac<OpsFp> acc;
    acc.x = fp_zero(); acc.y = fp_one(); acc.z = fp_zero();
    if (!rej) {
        bool b = false;
        if (!qinf) {
            const Fr ck = fr_from_mont(pw[ZKP_CELL_N * cells_brp7((int)k)]);
            uint64_t z[4], zh[2], zl[2];
            for (int i = 0; i < 4; i++) z[i] = ((uint64_t)ck.l[2 * i + 1] << 32) | ck.l[2 * i];
            kzg_glv_split(z, zh, zl);
            Fp qx = load_fp(pi, b), qy = load_fp(pi + 6, b);
            if (par) {
                qx = fmul(qx, fp_const(ZKP_BETA));
                qy = fp_neg(qy);
            }
            scalar_mul_jac<OpsFp>(acc, qx, qy, par ? zh : zl, 128);
        }
        if (par == 0 && !cinf) jac_add_affine(acc, acc, load_fp(c, b), load_fp(c + 6, b));
        if (par == 1 && !iinf) jac_add_affine(acc, acc, load_fp(ixy, b), fp_neg(load_fp(ixy + 6, b)));
    }
    Jac<OpsFp> pe, po, p;
    pe.x = fp_bcast<0>(acc.x); pe.y = fp_bcast<0>(acc.y); pe.z = fp_bcast<0>(acc.z);
    po.x = fp_bcast<1>(acc.x); po.y = fp_bcast<1>(acc.y); po.z = fp_bcast<1>(acc.z);
    jac_add(p, pe, po);
    const bool p_inf = fp_is_zero(p.z);
    Fp px = fp_zero(), py = fp_one();
    if (!p_inf) {
        Fp zi = fp_inv(p.z), zi2 = fsqr(zi);
        px = fmul(p.x, zi2);
        py = fmul(p.y, fmul(zi2, zi));
    }
    if (rej) { px = fp_zero(); py = fp_zero(); }
    if (par == 0) {
        store_fp(g1, px, nullptr);           // P.x
        copy_u64(g1 + 12, pi, 6, rej);       // pi.x
        g1inf[0] = rej ? 1 : (p_inf ? 1 : 0);
        g1inf[1] = rej ? 1 : qinf;
    } else {
        store_fp(g1 + 6, py, nullptr);       // P.y
        copy_u64(g1 + 18, pi + 6, 6, rej);   // pi.y
    }
    return st;
}

}  // namespace zkp
