// EIP-4844 blob verification front end (verify_blob_kzg_proof(blob, C, pi) of the consensus specs, deneb
// polynomial-commitments.md): the Fiat-Shamir challenge z = SHA-256(transcript) mod r and the evaluation y = p(z) of
// the blob's polynomial, given in evaluation form over the bit-reversed 4096-point domain.  The point-evaluation
// check of z and y is kzg.cuh's, unchanged.
//
// Shared by the CUDA kernels (kernels.cu) and the CPU dev simulation of the not-gpu tests.  The block-wide steps of
// the evaluation are functions of one thread index over a shared struct: the kernel calls them between
// __syncthreads(), the simulation in a loop over the thread indices.
#pragma once
#include "fr.cuh"

namespace zkp {

#define ZKP_BLOB_N 4096                  // FIELD_ELEMENTS_PER_BLOB (include/zkpair.h ZKP_BLOB_FIELD_ELEMENTS)
#define ZKP_BLOB_LOG_N 12
#define ZKP_BLOB_BYTES_ (32 * ZKP_BLOB_N)
#define ZKP_BLOB_TPB 256                 // threads of one k_blob_eval block (one block per blob)
#define ZKP_BLOB_PER_THREAD (ZKP_BLOB_N / ZKP_BLOB_TPB)

// ------------------------------------------------------------------ SHA-256 (FIPS 180-4)
ZKP_CONST uint32_t ZKP_SHA256_K[64] = {
    0x428a2f98u, 0x71374491u, 0xb5c0fbcfu, 0xe9b5dba5u, 0x3956c25bu, 0x59f111f1u, 0x923f82a4u, 0xab1c5ed5u,
    0xd807aa98u, 0x12835b01u, 0x243185beu, 0x550c7dc3u, 0x72be5d74u, 0x80deb1feu, 0x9bdc06a7u, 0xc19bf174u,
    0xe49b69c1u, 0xefbe4786u, 0x0fc19dc6u, 0x240ca1ccu, 0x2de92c6fu, 0x4a7484aau, 0x5cb0a9dcu, 0x76f988dau,
    0x983e5152u, 0xa831c66du, 0xb00327c8u, 0xbf597fc7u, 0xc6e00bf3u, 0xd5a79147u, 0x06ca6351u, 0x14292967u,
    0x27b70a85u, 0x2e1b2138u, 0x4d2c6dfcu, 0x53380d13u, 0x650a7354u, 0x766a0abbu, 0x81c2c92eu, 0x92722c85u,
    0xa2bfe8a1u, 0xa81a664bu, 0xc24b8b70u, 0xc76c51a3u, 0xd192e819u, 0xd6990624u, 0xf40e3585u, 0x106aa070u,
    0x19a4c116u, 0x1e376c08u, 0x2748774cu, 0x34b0bcb5u, 0x391c0cb3u, 0x4ed8aa4au, 0x5b9cca4fu, 0x682e6ff3u,
    0x748f82eeu, 0x78a5636fu, 0x84c87814u, 0x8cc70208u, 0x90befffau, 0xa4506cebu, 0xbef9a3f7u, 0xc67178f2u,
};

ZKP_HD uint32_t rotr32(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }

// one compression of the 16 big-endian message words w (clobbered: the schedule runs in place)
ZKP_HD void sha256_compress(uint32_t *h, uint32_t *w) {
    uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], k = h[7];
#pragma unroll
    for (int i = 0; i < 64; i++) {
        if (i >= 16) {
            const uint32_t w15 = w[(i + 1) & 15], w2 = w[(i + 14) & 15];
            w[i & 15] += (rotr32(w15, 7) ^ rotr32(w15, 18) ^ (w15 >> 3)) + w[(i + 9) & 15] +
                         (rotr32(w2, 17) ^ rotr32(w2, 19) ^ (w2 >> 10));
        }
        const uint32_t t1 = k + (rotr32(e, 6) ^ rotr32(e, 11) ^ rotr32(e, 25)) + ((e & f) ^ (~e & g)) + ZKP_SHA256_K[i] + w[i & 15];
        const uint32_t t2 = (rotr32(a, 2) ^ rotr32(a, 13) ^ rotr32(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
        k = g; g = f; f = e; e = d + t1;
        d = c; c = b; b = a; a = t1 + t2;
    }
    h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += k;
}

// 16 bytes at p (16-byte aligned) -> four big-endian words
ZKP_HD void load_be16(const uint8_t *p, uint32_t *w) {
#ifdef ZKP_DEVICE_BUILD
    const uint4 v = *(const uint4 *)p;
    w[0] = __byte_perm(v.x, 0, 0x0123);
    w[1] = __byte_perm(v.y, 0, 0x0123);
    w[2] = __byte_perm(v.z, 0, 0x0123);
    w[3] = __byte_perm(v.w, 0, 0x0123);
#else
    for (int k = 0; k < 4; k++)
        w[k] = ((uint32_t)p[4 * k] << 24) | ((uint32_t)p[4 * k + 1] << 16) | ((uint32_t)p[4 * k + 2] << 8) | p[4 * k + 3];
#endif
}

// The compressed encoding of a G1 point (x | y canonical limbs, inf flag) as 12 big-endian words: x in 48 big-endian
// bytes with the top byte OR-ed with 0x80 (compressed), and with 0x20 when y > (p - 1) / 2; the identity is 0xc0
// followed by 47 zero bytes.  Only the transcript reads it.
ZKP_HD void g1_compress_words(const uint64_t *xy, uint8_t inf, uint32_t *c) {
    for (int k = 0; k < 6; k++) {
        c[2 * k] = inf ? 0u : (uint32_t)(xy[5 - k] >> 32);
        c[2 * k + 1] = inf ? 0u : (uint32_t)xy[5 - k];
    }
    // y > (p - 1) / 2 = p >> 1 (p is odd): (p >> 1) - y borrows
    uint32_t y[ZKP_NL], half[ZKP_NL];
    for (int i = 0; i < ZKP_NL; i++) {
        y[i] = (uint32_t)(xy[6 + i / 2] >> (32 * (i & 1)));
        half[i] = (ZKP_P[i] >> 1) | (i + 1 < ZKP_NL ? ZKP_P[i + 1] << 31 : 0u);
    }
    sub_cc(half[0], y[0]);
    for (int i = 1; i < ZKP_NL; i++) subc_cc(half[i], y[i]);
    const bool y_big = subc(0, 0) != 0;
    c[0] |= inf ? 0xc0000000u : (0x80000000u | (y_big ? 0x20000000u : 0u));
}

// compute_challenge(blob, C): digest = SHA-256(b"FSBLOBVERIFY_V1_" | N as 16 big-endian bytes | blob | C as 48 bytes),
// z = digest as a big-endian integer mod r (2^256 < 3r: at most two subtractions).  131 152 bytes, 2050 blocks; the
// blob is read in 16-byte aligned pieces (blob 16-byte aligned).  proof = C.x | C.y | ..., cinf = C's flag.
ZKP_HD void blob_challenge_one(const uint8_t *blob, const uint64_t *proof, uint8_t cinf, uint32_t *digest, uint64_t *z) {
    uint32_t h[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
    uint32_t c[12], w[16];
    g1_compress_words(proof, cinf, c);
    // block 0: the domain separator "FSBLOBVERIFY_V1_", N = 4096 in 16 bytes, the blob's first 32 bytes
    w[0] = 0x4653424cu; w[1] = 0x4f425645u; w[2] = 0x52494659u; w[3] = 0x5f56315fu;
    w[4] = 0; w[5] = 0; w[6] = 0; w[7] = (uint32_t)ZKP_BLOB_N;
    load_be16(blob, w + 8);
    load_be16(blob + 16, w + 12);
    sha256_compress(h, w);
    // blocks 1 .. 2047: blob bytes [64 b - 32, 64 b + 32)
#pragma unroll 1
    for (int b = 1; b < ZKP_BLOB_BYTES_ / 64; b++) {
        const uint8_t *p = blob + 64 * b - 32;
        load_be16(p, w);
        load_be16(p + 16, w + 4);
        load_be16(p + 32, w + 8);
        load_be16(p + 48, w + 12);
        sha256_compress(h, w);
    }
    // block 2048: the blob's last 32 bytes, the first 32 bytes of C
    load_be16(blob + ZKP_BLOB_BYTES_ - 32, w);
    load_be16(blob + ZKP_BLOB_BYTES_ - 16, w + 4);
    for (int i = 0; i < 8; i++) w[8 + i] = c[i];
    sha256_compress(h, w);
    // block 2049: the last 16 bytes of C, the padding and the message length in bits
    for (int i = 0; i < 4; i++) w[i] = c[8 + i];
    w[4] = 0x80000000u;
    for (int i = 5; i < 15; i++) w[i] = 0;
    w[15] = (uint32_t)((32 + ZKP_BLOB_BYTES_ + 48) * 8);
    sha256_compress(h, w);
    Fr v;
    for (int i = 0; i < 8; i++) {
        digest[i] = h[i];
        v.l[i] = h[7 - i];
    }
    v = fr_reduce_once(fr_reduce_once(v));   // each step subtracts r when v >= r
    for (int i = 0; i < 4; i++) z[i] = ((uint64_t)v.l[2 * i + 1] << 32) | v.l[2 * i];
}

// ------------------------------------------------------------------ evaluation at z (barycentric, in Fr)

// the domain's entry i, roots_brp[i] = omega^brp(i), in Montgomery form (brp = bit reversal of the 12-bit index)
ZKP_HD Fr blob_root(int i) {
    uint32_t e = 0;
    for (int b = 0; b < ZKP_BLOB_LOG_N; b++) e |= (uint32_t)((i >> b) & 1) << (ZKP_BLOB_LOG_N - 1 - b);
    Fr acc = fr_one(), base = fr_const(ZKP_FR_OMEGA);
    for (int b = 0; b < ZKP_BLOB_LOG_N; b++) {
        if ((e >> b) & 1) acc = fr_mul(acc, base);
        base = fr_sqr(base);
    }
    return acc;
}

// blob element i: 32 big-endian bytes -> the canonical value in Fr words; false (and 0) when it is >= r
ZKP_HD bool blob_element(const uint8_t *blob, int i, Fr &p) {
    uint32_t w[8];
    load_be16(blob + 32 * i, w);
    load_be16(blob + 32 * i + 16, w + 4);
    for (int k = 0; k < 8; k++) p.l[k] = w[7 - k];
    const bool ok = !fr_geq_r(p);
    p = fr_select(ok, p, fr_zero());
    return ok;
}

// Shared state of one blob's block.  tree is heap ordered (node k has children 2k and 2k + 1, thread t's leaf is
// TPB + t): first the product tree of the threads' denominator products and then, in place, their inverses; later the
// sum tree of the threads' partial sums.
struct BlobShared {
    Fr tree[2 * ZKP_BLOB_TPB];
    Fr pj;           // the element at z when z is a domain point
    uint32_t bad;    // some element >= r
    uint32_t hit;    // z is a domain point
};
struct BlobLane {    // one thread's prefix products of its denominators
    Fr pre[ZKP_BLOB_PER_THREAD];
};

// z (canonical, < r) -> Montgomery
ZKP_HD Fr blob_z_mont(const uint64_t *zy) {
    Fr z;
    for (int i = 0; i < 4; i++) {
        z.l[2 * i] = (uint32_t)zy[i];
        z.l[2 * i + 1] = (uint32_t)(zy[i] >> 32);
    }
    return fr_to_mont(z);
}

ZKP_HD void blob_eval_init(BlobShared &sh) {
    sh.bad = 0;
    sh.hit = 0;
    sh.pj = fr_zero();
}

// z - omega_i, with the one zero denominator of a z in the domain counted as 1
ZKP_HD Fr blob_denominator(const Fr &zm, const Fr &w) {
    const Fr d = fr_sub(zm, w);
    return fr_select(fr_is_zero(d), fr_one(), d);
}

// Step 1, thread t: the prefix products of the denominators z - omega_i of its elements i = t + TPB k (Montgomery)
// and their product at its leaf of the tree.
ZKP_HD void blob_eval_prefix(int t, const Fr *roots, const Fr &zm, BlobShared &sh, BlobLane &ln) {
    Fr acc = blob_denominator(zm, roots[t]);
    ln.pre[0] = acc;
#pragma unroll
    for (int k = 1; k < ZKP_BLOB_PER_THREAD; k++) {
        acc = fr_mul(acc, blob_denominator(zm, roots[t + ZKP_BLOB_TPB * k]));
        ln.pre[k] = acc;
    }
    sh.tree[ZKP_BLOB_TPB + t] = acc;
}
// Step 2, level by level from the leaves up (k = w + t for t < w, w = TPB/2 .. 1): node k = product of its children
ZKP_HD void blob_tree_mul(Fr *tr, int k) { tr[k] = fr_mul(tr[2 * k], tr[2 * k + 1]); }
// Step 3, one thread: the root's inverse (the one inversion of the blob)
ZKP_HD void blob_tree_invert_root(Fr *tr) { tr[1] = fr_inv(tr[1]); }
// Step 4, level by level from the root down (k = w + t for t < w, w = 1 .. TPB/2): node k holds 1/(L R), so its
// children get 1/L = R/(L R) and 1/R = L/(L R).  The leaves end up holding the inverse of each thread's product.
ZKP_HD void blob_tree_inv(Fr *tr, int k) {
    const Fr i = tr[k], l = tr[2 * k], r = tr[2 * k + 1];
    tr[2 * k] = fr_mul(i, r);
    tr[2 * k + 1] = fr_mul(i, l);
}
// Step 5, thread t: back-substitution from its leaf, 1/d_i = acc * pre[k - 1], acc *= d_i, and its partial sum of
// p_i omega_i / (z - omega_i), which replaces its leaf.  p_i enters canonical and omega_i and 1/d_i Montgomery, so
// each product p_i omega_i (1/d_i) comes out canonical: the conversion of p_i costs nothing.  ROW: 1/d_i is also
// stored at row[i] (the prover's quotient, kzg_prove.cuh).
template <bool ROW = false>
ZKP_HD void blob_eval_terms(int t, const uint8_t *blob, const Fr *roots, const Fr &zm, BlobShared &sh, const BlobLane &ln,
                            Fr *row = nullptr) {
    Fr acc = sh.tree[ZKP_BLOB_TPB + t], sum = fr_zero();
    bool bad = false;
#pragma unroll
    for (int k = ZKP_BLOB_PER_THREAD - 1; k >= 0; k--) {
        const int i = t + ZKP_BLOB_TPB * k;
        const Fr w = roots[i];
        Fr p;
        bad |= !blob_element(blob, i, p);
        const Fr d = fr_sub(zm, w);
        if (fr_is_zero(d)) {   // z = omega_i: y = p_i (at most one i per blob)
            sh.hit = 1;
            sh.pj = p;
        }
        const Fr inv = k ? fr_mul(acc, ln.pre[k - 1]) : acc;
        if (ROW) row[i] = inv;
        if (k) acc = fr_mul(acc, fr_select(fr_is_zero(d), fr_one(), d));
        sum = fr_add(sum, fr_mul(fr_mul(p, w), inv));
    }
    if (bad) sh.bad = 1;
    sh.tree[ZKP_BLOB_TPB + t] = sum;
}
// Step 6, level by level from the leaves up: node k = sum of its children
ZKP_HD void blob_tree_add(Fr *tr, int k) { tr[k] = fr_add(tr[2 * k], tr[2 * k + 1]); }
// Step 7, one thread: y = (z^N - 1) / N * sum (canonical), or p_j for z = omega_j; a blob with an element >= r gets
// z = r and y = 0, which the point-evaluation front end reports as ZKP_KZG_BAD_SCALAR (or BAD_POINT, which precedes).
ZKP_HD void blob_eval_finish(const BlobShared &sh, const Fr &zm, uint64_t *zy) {
    Fr zn = zm;
    for (int s = 0; s < ZKP_BLOB_LOG_N; s++) zn = fr_sqr(zn);
    Fr y = fr_mul(fr_mul_const(fr_sub(zn, fr_one()), ZKP_FR_INV_N), sh.tree[1]);
    if (sh.hit) y = sh.pj;
    if (sh.bad) {
        y = fr_zero();
        for (int i = 0; i < 4; i++) zy[i] = ((uint64_t)ZKP_R_ORDER[2 * i + 1] << 32) | ZKP_R_ORDER[2 * i];
    }
    for (int i = 0; i < 4; i++) zy[4 + i] = ((uint64_t)y.l[2 * i + 1] << 32) | y.l[2 * i];
}

}  // namespace zkp
