// EIP-4844 prover front end (blob_to_kzg_commitment, compute_kzg_proof and compute_blob_kzg_proof of the consensus
// specs, deneb polynomial-commitments.md).  Commitments and proofs are one fixed-base multi-scalar multiplication over
// the setup's 4096 G1 Lagrange points in bit-reversed order, sum_i s_i L_brp(i): for a commitment s_i are the blob's
// elements, for a proof the quotient q_i = (p_i - y) / (omega_i - z) of compute_kzg_proof_impl, formed in evaluation
// form by the steps of blob.cuh.  Both scalar rows are 4096 x 32 big-endian bytes, the layout of a blob.
//
// Shared by the CUDA kernels (kernels.cu) and the CPU dev simulation of the not-gpu tests.  As in blob.cuh, the
// block-wide steps are functions of one thread index over a shared struct: the kernel calls them between
// __syncthreads(), the simulation in a loop over the thread indices.
#pragma once
#include "kzg.cuh"
#include "blob.cuh"

namespace zkp {

#define ZKP_MSM_WINDOWS 32   // signed 8-bit windows: every scalar is < r < 2^255, so the top window never carries out
#define ZKP_MSM_DIGITS 128   // table entries per window: |digit| = 1 .. 128, a negative digit negates y
// Fp per base: [window][|digit| - 1] affine (x, y), Montgomery form (32 * 128 * 96 B = 384 KiB; 1.5 GiB for 4096 bases)
#define ZKP_MSM_TABLE_FP (ZKP_MSM_WINDOWS * ZKP_MSM_DIGITS * 2)
#define ZKP_MSM_TPB 256      // threads of one k_kzg_msm block (one block per scalar row)

// the 12-bit bit reversal of a domain index
ZKP_HD int blob_brp(int i) {
    int e = 0;
    for (int b = 0; b < ZKP_BLOB_LOG_N; b++) e |= ((i >> b) & 1) << (ZKP_BLOB_LOG_N - 1 - b);
    return e;
}

// Signed-digit recoding, window w (w = 0 first) of a scalar given as eight little-endian 32-bit words: byte w plus the
// carry of window w - 1; a sum above 128 becomes sum - 256 and carries 1 into window w + 1.  Digits lie in [-127, 128]
// and sum_w d_w 2^(8w) + carry 2^(8 (w + 1)) is the scalar's value up to window w.
ZKP_HD int msm_digit(const uint32_t *s, int w, uint32_t &carry) {
    const int d = (int)((s[w >> 2] >> (8 * (w & 3))) & 0xffu) + (int)carry;
    carry = d > ZKP_MSM_DIGITS ? 1u : 0u;
    return carry ? d - 256 : d;
}

// v (canonical Fr words) as 32 big-endian bytes at p (16-byte aligned): the scalar-row layout
ZKP_HD void store_be32(uint8_t *p, const Fr &v) {
#ifdef ZKP_DEVICE_BUILD
    uint4 a, b;
    a.x = __byte_perm(v.l[7], 0, 0x0123); a.y = __byte_perm(v.l[6], 0, 0x0123);
    a.z = __byte_perm(v.l[5], 0, 0x0123); a.w = __byte_perm(v.l[4], 0, 0x0123);
    b.x = __byte_perm(v.l[3], 0, 0x0123); b.y = __byte_perm(v.l[2], 0, 0x0123);
    b.z = __byte_perm(v.l[1], 0, 0x0123); b.w = __byte_perm(v.l[0], 0, 0x0123);
    *(uint4 *)p = a;
    *(uint4 *)(p + 16) = b;
#else
    for (int k = 0; k < 8; k++)
        for (int j = 0; j < 4; j++) p[4 * k + j] = (uint8_t)(v.l[7 - k] >> (24 - 8 * j));
#endif
}

// ------------------------------------------------------------------ fixed-base MSM over the Lagrange tables

// Shared state of one row's block of TPB threads: each thread's Jacobian partial sum, then the tree of their sums in
// place.  k_kzg_msm runs 256 threads over 4096 bases; the cell verifier (kzg_cells.cuh) 64 threads over 64 bases.
template <int TPB>
struct MsmSharedN {
    Jac<OpsFp> acc[TPB];
    uint32_t bad;    // some scalar >= r
};
typedef MsmSharedN<ZKP_MSM_TPB> MsmShared;

template <int TPB>
ZKP_HD void msm_init(MsmSharedN<TPB> &sh) { sh.bad = 0; }
// Step 1, thread t: sum over the bases i = t + TPB k < NB and every window of d_w 2^(8w) L_brp(i), one table lookup and
// one mixed addition per non-zero digit, no doubling.  skip = the row is already rejected (the partial stays the
// identity).  The row holds NB scalars.
template <int NB = ZKP_BLOB_N, int TPB>
ZKP_HD void msm_partial(int t, const Fp *tables, const uint8_t *row, bool skip, MsmSharedN<TPB> &sh) {
    Jac<OpsFp> acc;
    acc.x = fp_zero(); acc.y = fp_one(); acc.z = fp_zero();
    bool bad = false;
    if (!skip) {
#pragma unroll 1
        for (int k = 0; k < NB / TPB; k++) {
            const int i = t + TPB * k;
            Fr s;
            bad |= !blob_element(row, i, s);
            const Fp *tb = tables + (size_t)i * ZKP_MSM_TABLE_FP;
            uint32_t carry = 0;
#pragma unroll 1
            for (int w = 0; w < ZKP_MSM_WINDOWS; w++) {
                const int d = msm_digit(s.l, w, carry);
                if (!d) continue;
                const Fp *e = tb + 2 * (w * ZKP_MSM_DIGITS + (d < 0 ? -d : d) - 1);
                jac_add_affine(acc, acc, e[0], d < 0 ? fp_neg(e[1]) : e[1]);
            }
        }
    }
    sh.acc[t] = acc;
    if (bad) sh.bad = 1;
}
// Step 2, level by level (t < w, w = TPB/2 .. 1): acc[t] += acc[t + w]
template <int TPB>
ZKP_HD void msm_tree_add(MsmSharedN<TPB> &sh, int t, int w) { jac_add(sh.acc[t], sh.acc[t], sh.acc[t + w]); }
// Step 3, one thread: the sum as canonical affine limbs and its flag; pre = an earlier rejection of this row (0 none).
// A rejected row (pre, or a scalar >= r: ZKP_KZG_BAD_SCALAR) gets zero limbs with the flag set; the identity is (0, 1)
// with the flag set.  Returns the row's status.
template <int TPB>
ZKP_HD uint8_t msm_finish(const MsmSharedN<TPB> &sh, uint8_t pre, uint64_t *xy, uint8_t *inf) {
    const uint8_t st = pre ? pre : sh.bad ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
    const Jac<OpsFp> &p = sh.acc[0];
    const bool p_inf = fp_is_zero(p.z);
    Fp x = fp_zero(), y = fp_one();
    if (!p_inf) {
        Fp zi = fp_inv(p.z), zi2 = fsqr(zi);
        x = fmul(p.x, zi2);
        y = fmul(p.y, fmul(zi2, zi));
    }
    if (st != ZKP_KZG_VALID) { x = fp_zero(); y = fp_zero(); }
    store_fp(xy, x, nullptr);
    store_fp(xy + 6, y, nullptr);
    *inf = (st != ZKP_KZG_VALID || p_inf) ? 1 : 0;
    return st;
}

// ------------------------------------------------------------------ quotient rows (compute_kzg_proof_impl)

// Shared state of one blob's quotient block: blob.cuh's evaluation state, then z, y and the in-domain index.
struct QuotShared {
    BlobShared b;
    Fr zm;           // z in Montgomery form (0 when z >= r)
    Fr y;            // canonical
    int m;           // z = omega_m (when b.hit)
    uint32_t zbad;   // z >= r
};

// Step 0, one thread: z from z_in (compute_kzg_proof; copied to zy) or already in zy (compute_blob_kzg_proof)
ZKP_HD void quot_init(QuotShared &sh, const uint64_t *z_in, uint64_t *zy) {
    if (z_in)
        for (int i = 0; i < 4; i++) zy[i] = z_in[i];
    sh.zbad = fr_canonical(zy) ? 0u : 1u;
    sh.zm = sh.zbad ? fr_zero() : blob_z_mont(zy);
    sh.m = 0;
    blob_eval_init(sh.b);
}
// Steps 1 - 7 are blob.cuh's, with blob_eval_terms<true> leaving 1/(z - omega_i) (Montgomery) in the row.
// Step 7b, one thread after blob_eval_finish: y (0 when z >= r) and the status; pre = an earlier rejection (0 none).
ZKP_HD uint8_t quot_status(QuotShared &sh, uint8_t pre, uint64_t *zy, uint64_t *y_out) {
    if (sh.zbad)
        for (int i = 0; i < 4; i++) zy[4 + i] = 0;
    for (int i = 0; i < 4; i++) {
        sh.y.l[2 * i] = (uint32_t)zy[4 + i];
        sh.y.l[2 * i + 1] = (uint32_t)(zy[4 + i] >> 32);
    }
    const uint8_t st = pre ? pre : (sh.b.bad || sh.zbad) ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
    if (y_out)
        for (int i = 0; i < 4; i++) y_out[i] = st == ZKP_KZG_VALID ? zy[4 + i] : 0;
    return st;
}
// Step 8, thread t: q_i = (y - p_i) (1/(z - omega_i)) over its elements, in place as big-endian bytes.  For z = omega_m
// the entry m is left for step 10, and the thread's partial sum of (p_i - y) omega_i / (z - omega_i), i != m, replaces
// its leaf of the tree.  p_i and y are canonical, omega_i and the inverses Montgomery, so every product is canonical.
ZKP_HD void quot_terms(int t, const uint8_t *blob, const Fr *roots, QuotShared &sh, uint8_t *row) {
    Fr sum = fr_zero();
#pragma unroll 1
    for (int k = 0; k < ZKP_BLOB_PER_THREAD; k++) {
        const int i = t + ZKP_BLOB_TPB * k;
        Fr p;
        blob_element(blob, i, p);
        const Fr inv = ((const Fr *)row)[i];
        if (sh.b.hit) {
            if (fr_eq(sh.zm, roots[i])) {
                sh.m = i;
                continue;
            }
            sum = fr_add(sum, fr_mul(fr_mul(fr_sub(p, sh.y), roots[i]), inv));
        }
        store_be32(row + 32 * i, fr_mul(fr_sub(sh.y, p), inv));
    }
    sh.b.tree[ZKP_BLOB_TPB + t] = sum;
}
// Step 9 (z in the domain only) is blob_tree_add.  Step 10, one thread: q_m = sum / z, compute_quotient_eval_within_domain.
ZKP_HD void quot_within_domain(const QuotShared &sh, uint8_t *row) {
    store_be32(row + 32 * sh.m, fr_mul(sh.b.tree[1], fr_inv(sh.zm)));
}

// compute_blob_kzg_proof's front, one thread: C validated (ZKP_KZG_BAD_POINT when it is non-canonical, off the curve
// or not torsion free) and z = the transcript's challenge into zy, computed for every blob as in the verifier.
ZKP_HD uint8_t prove_challenge_one(const uint8_t *blob, const uint64_t *c, uint8_t cinf, uint64_t *zy) {
    bool bad = false;
    const uint8_t sp = g1_check_one(c, cinf, bad);
    uint32_t digest[8];
    blob_challenge_one(blob, c, cinf, digest, zy);
    return (bad || sp != ZKP_POINT_OK) ? ZKP_KZG_BAD_POINT : ZKP_KZG_VALID;
}

}  // namespace zkp
