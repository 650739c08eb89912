// EIP-7594 cell recovery (recover_cells_and_kzg_proofs of the consensus specs, fulu polynomial-commitments-sampling.md):
// any 64 or more of a blob's 128 cells -> the blob's coefficients, then all cells (and, through k_cells_quotient and
// k_kzg_msm, all proofs) as compute_cells_and_kzg_proofs computes them.
//
// The spec's recover_polynomialcoeff, on the extended domain of kzg_cells.cuh (8192 slots in 13-bit bit-reversed
// order, cell k = slots [64 k, 64 k + 64)): E = the given cells with zeros where cells are missing, Z = the vanishing
// polynomial of the missing cells' cosets, D = ifft(fft(Z) E), then the coset evaluations of D at shift 7 divided by
// those of Z, and the coset inverse NTT truncated to 4096 coefficients.  Z depends on x^64 only, and at slot
// j = 64 k + t both x^64 (= c_k) and (7 x)^64 (= 7^64 c_k) depend on k only, so Z is one scalar per cell on either
// domain: z_k = prod_{missing m} (c_k - c_m), zero for a missing cell, and zc_k = prod_{missing m} (7^64 c_k - c_m),
// never zero (7^8192 != 1).  Recovery is four 8192-point NTTs with pointwise scales between them:
//   x_j = E_j z_k                      (bit-reversed; the inverse DIT reads it as it is)
//   d = inverse DIT NTT of x           (natural order), scaled by 7^t / 8192
//   forward DIF NTT                    (the coset evaluations, bit-reversed), slot j times 1 / zc_k
//   a = inverse DIT NTT                (natural order), scaled by 7^-t / 8192 and truncated to t < 4096
//   forward DIF NTT of (a, 0)          (the 128 cells, bit-reversed)
// The spec does not check that the given cells agree; for any input the result is bit-exact to its algorithm.
//
// One blob is one cluster of two blocks of ZKP_CELLS_TPB threads.  Rank r holds slots [4096 r, 4096 r + 4096) in its
// dynamic shared memory (128 KiB: one block cannot hold the 256 KiB of 8192 Fr).  Of the 13 stages of a radix-2
// transform only the one of half-length 4096 pairs slots of different ranks; the two of them that meet between
// transforms (the last inverse stage, the scale, the first forward stage) are fused into one cross pass over
// distributed shared memory, in which rank r does the pairs b in [2048 r, 2048 r + 2048).  The other 12 stages of each
// transform are cells_dit_pass / cells_dif_pass over the rank's half: with h <= 2048 a butterfly's twiddle depends on
// b mod h only, so the half runs the 4096-point stage sequence of k_cells_extend.
//
// As in kzg_cells.cuh, the block-wide steps are functions of (rank, thread index) over shared memory: the kernel calls
// them between __syncthreads() and cluster barriers, the CPU dev simulation in loops over the ranks and threads.
#pragma once
#include "kzg_cells.cuh"

namespace zkp {

#ifndef ZKP_KZG_BAD_CELLS   /* same value as include/zkpair.h */
#define ZKP_KZG_BAD_CELLS 4
#endif
#define ZKP_RECOVER_HALF 4096            // slots per rank
#define ZKP_RECOVER_PARTS (ZKP_CELLS_TPB / ZKP_CELL_N)   // partial products per cell in the vanishing step

// A block's state besides its half of the extended blob
struct RecoverShared {
    int16_t pos[ZKP_CELLS_PER_BLOB];     // cell index -> its position in the input, -1 when missing
    Fr z[ZKP_CELL_N];                    // z_k of the rank's cells 64 r + c (Montgomery)
    Fr zci[ZKP_CELL_N];                  // 1 / zc_k of the rank's cells (Montgomery)
    uint32_t bad_cells;                  // a count outside [64, 128], indices not strictly ascending or one >= 128
    uint32_t bad;                        // an element >= r in one of the rank's given cells
};

// base^e for 0 <= e < 4096 (Montgomery)
ZKP_HD Fr recover_pow(Fr base, int e) {
    Fr acc = fr_one();
    for (int b = 0; b < 12; b++) {
        if ((e >> b) & 1) acc = fr_mul(acc, base);
        base = fr_sqr(base);
    }
    return acc;
}

// Step 1, thread t (both ranks alike): the count check and an empty position table
ZKP_HD void recover_init(int t, uint64_t n, RecoverShared &sh) {
    if (t < ZKP_CELLS_PER_BLOB) sh.pos[t] = -1;
    if (t == 0) {
        sh.bad_cells = (n < ZKP_CELLS_PER_BLOB / 2 || n > ZKP_CELLS_PER_BLOB) ? 1u : 0u;
        sh.bad = 0;
    }
}
// Step 2, thread t < min(n, 128) (both ranks alike): input index t, checked (< 128, above index t - 1) and entered in
// the position table
ZKP_HD void recover_index(int t, uint64_t n, const uint64_t *idx, RecoverShared &sh) {
    if ((uint64_t)t >= n || t >= ZKP_CELLS_PER_BLOB) return;
    const uint64_t k = idx[t];
    if (k >= ZKP_CELLS_PER_BLOB || (t > 0 && idx[t - 1] >= k)) sh.bad_cells = 1;
    else sh.pos[k] = (int16_t)t;
}
// Step 3, thread t: the partial products of the rank's cell k = 64 r + (t mod 64) over the missing m in
// [16 (t / 64), 16 (t / 64) + 16): z into part[t], zc into part[TPB + t] (part: the first 1024 Fr of the rank's half)
ZKP_HD void recover_vanish_part(int r, int t, const Fr *pw, const RecoverShared &sh, Fr *part) {
    const int per = ZKP_CELLS_PER_BLOB / ZKP_RECOVER_PARTS, k = ZKP_CELL_N * r + (t % ZKP_CELL_N), m0 = (t / ZKP_CELL_N) * per;
    const Fr ck = pw[ZKP_CELL_N * cells_brp7(k)], sk = fr_mul_const(ck, ZKP_FR_SHIFT_64);
    Fr z = fr_one(), zc = fr_one();
    for (int m = m0; m < m0 + per; m++) {
        if (sh.pos[m] >= 0) continue;
        const Fr cm = pw[ZKP_CELL_N * cells_brp7(m)];
        z = fr_mul(z, fr_sub(ck, cm));
        zc = fr_mul(zc, fr_sub(sk, cm));
    }
    part[t] = z;
    part[ZKP_CELLS_TPB + t] = zc;
}
// Step 4, thread c < 64: z_k and 1 / zc_k of the rank's cell 64 r + c from the parts
ZKP_HD void recover_vanish(int c, const Fr *part, RecoverShared &sh) {
    Fr z = part[c], zc = part[ZKP_CELLS_TPB + c];
    for (int p = 1; p < ZKP_RECOVER_PARTS; p++) {
        z = fr_mul(z, part[ZKP_CELL_N * p + c]);
        zc = fr_mul(zc, part[ZKP_CELLS_TPB + ZKP_CELL_N * p + c]);
    }
    sh.z[c] = z;
    sh.zci[c] = fr_inv(zc);
}
// Step 5, thread t: the rank's slots i = t + TPB s (element i mod 64 of cell 64 r + i / 64) from the input cells
// (2048 bytes each, in input order) times z_k, zero for a missing cell; an element >= r reads as 0 and sets sh.bad
ZKP_HD void recover_load(int r, int t, const uint8_t *cells, RecoverShared &sh, Fr *x) {
    bool b = false;
    for (int s = 0; s < ZKP_RECOVER_HALF / ZKP_CELLS_TPB; s++) {
        const int i = t + ZKP_CELLS_TPB * s, c = i / ZKP_CELL_N, p = sh.pos[ZKP_CELL_N * r + c];
        Fr v = fr_zero();
        if (p >= 0) {
            b |= !blob_element(cells + (size_t)p * ZKP_CELL_BYTES_, i % ZKP_CELL_N, v);
            v = fr_mul(v, sh.z[c]);
        }
        x[i] = v;
    }
    if (b) sh.bad = 1;
}
// Steps 6, 8, 10 and 12 are the 12 local stages of a transform: cells_dit_pass (h = 1 .. 2048) or cells_dif_pass
// (h = 2048 .. 1) over the rank's half.

// Step 7, cross pass A, thread t of rank r (half[0], half[1]: the two ranks' halves, one of them remote): for the pairs
// b = 2048 r + t + 512 s, the last inverse stage (h = 4096), d_t = its outputs times 7^t / 8192 (t = b, 4096 + b),
// and the first forward stage (h = 4096) of d
ZKP_HD void recover_cross_a(int r, int t, const Fr *pw, Fr *const *half) {
    const int b0 = ZKP_CELLS_TPB * 4 * r + t;
    Fr sc = fr_mul_const(recover_pow(fr_const(ZKP_FR_SHIFT), b0), ZKP_FR_INV_EXT_N);
    for (int s = 0; s < ZKP_RECOVER_HALF / 2 / ZKP_CELLS_TPB; s++) {
        const int b = b0 + ZKP_CELLS_TPB * s;
        const Fr u = half[0][b], v = fr_mul(half[1][b], pw[(ZKP_CELLS_EXT_N - b) & (ZKP_CELLS_EXT_N - 1)]);
        const Fr d0 = fr_mul(fr_add(u, v), sc), d1 = fr_mul(fr_mul_const(fr_sub(u, v), ZKP_FR_SHIFT_4096), sc);
        half[0][b] = fr_add(d0, d1);
        half[1][b] = fr_mul(fr_sub(d0, d1), pw[b]);
        sc = fr_mul_const(sc, ZKP_FR_SHIFT_512);
    }
}
// Step 9, thread t: the rank's slot i (cell 64 r + i / 64) times 1 / zc_k
ZKP_HD void recover_divide(int t, const RecoverShared &sh, Fr *x) {
    for (int s = 0; s < ZKP_RECOVER_HALF / ZKP_CELLS_TPB; s++) {
        const int i = t + ZKP_CELLS_TPB * s;
        x[i] = fr_mul(x[i], sh.zci[i / ZKP_CELL_N]);
    }
}
// Step 11, cross pass B, thread t of rank r: for the pairs b as in step 7, the last inverse stage's lower output times
// 7^-b / 8192 is coefficient a_b of the blob (canonical; to coeffs when it is not NULL); the upper output is the
// truncated part.  Then the first forward stage of (a, 0): a_b and a_b omega_8192^b.
ZKP_HD void recover_cross_b(int r, int t, const Fr *pw, Fr *const *half, Fr *coeffs) {
    const int b0 = ZKP_CELLS_TPB * 4 * r + t;
    Fr sc = fr_mul_const(recover_pow(fr_const(ZKP_FR_SHIFT_INV), b0), ZKP_FR_INV_EXT_N);
    for (int s = 0; s < ZKP_RECOVER_HALF / 2 / ZKP_CELLS_TPB; s++) {
        const int b = b0 + ZKP_CELLS_TPB * s;
        const Fr a = fr_mul(fr_add(half[0][b], fr_mul(half[1][b], pw[(ZKP_CELLS_EXT_N - b) & (ZKP_CELLS_EXT_N - 1)])), sc);
        if (coeffs) coeffs[b] = a;
        half[0][b] = a;
        half[1][b] = fr_mul(a, pw[b]);
        sc = fr_mul_const(sc, ZKP_FR_SHIFT_INV_512);
    }
}
// Step 13, thread t: the rank's cells 64 r .. 64 r + 63 (its 128 KiB of the blob's 256 KiB at out) in big-endian
// bytes; a rejected blob gets zero cells
ZKP_HD void recover_store(int r, int t, const Fr *x, bool rej, uint8_t *out) {
    for (int s = 0; s < ZKP_RECOVER_HALF / ZKP_CELLS_TPB; s++) {
        const int i = t + ZKP_CELLS_TPB * s;
        store_be32(out + 32 * (ZKP_RECOVER_HALF * r + i), rej ? fr_zero() : x[i]);
    }
}
// The blob's status from its two blocks' states (BAD_CELLS precedes BAD_SCALAR)
ZKP_HD uint8_t recover_status(const RecoverShared &a, bool bad_other) {
    return a.bad_cells ? ZKP_KZG_BAD_CELLS : (a.bad || bad_other) ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
}

}  // namespace zkp
