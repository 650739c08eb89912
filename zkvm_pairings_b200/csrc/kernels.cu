// libzkpair.so: CUDA kernels (sm_100a) + the C ABI declared in include/zkpair.h.
//
// This translation unit holds the C ABI, the host-side pipeline and the kernels whose lane pairs may
// diverge from each other (tower ops, products, point generation: pair-masked shuffles).  The
// pairing kernel itself is pairing_kernel.cu (warp-converged, full-mask shuffles).
//
// A LANE PAIR (two adjacent threads) owns one pairing check (k pairs -> shared-accumulator Miller
// loop -> final exponentiation): every Fp2 of the tower is split over the pair (tower.cuh), so a
// warp runs 16 independent checks in lock-step (the control flow is data independent) and the
// integer-multiply pipe is kept busy by the carry-chained 32-bit-limb Montgomery products of
// fp.cuh.  Independent checks shard in contiguous slices over the context's devices;
// the only cross-device traffic is the 576-byte Fp12 partial of zkp_multi_miller_product.
//
// There is deliberately no CPU implementation in this library: with no CUDA device every entry
// point fails with ZKP_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/zkpair.h"
#include "fe_scratch.cuh"   // ops.cuh + the context-owned helper objects of the final exponentiation
#include "groth16.cuh"
#include "kzg.cuh"
#include "blob.cuh"
#include "kzg_prove.cuh"
#include "kzg_cells.cuh"
#include "kzg_recover.cuh"
#include "msm.cuh"

#include <cooperative_groups.h>

#ifndef ZKP_TPB
#define ZKP_TPB 128           // threads per block of the pairing kernels
#endif
#ifndef ZKP_MIN_BLOCKS
#define ZKP_MIN_BLOCKS 2      // resident blocks per SM the register allocator must allow
#endif
#ifndef ZKP_PRODUCT_GROUP
#define ZKP_PRODUCT_GROUP 4   // pairs per shared-accumulator Miller loop in zkp_multi_miller_product (k_pairing<4>)
#endif
#ifndef ZKP_CHUNK
#define ZKP_CHUNK (1u << 18)  // checks per host<->device pipeline chunk (e2e at 2^20: 1.735 / 1.776 / 1.794 M/s for 2^16 / 2^17 / 2^18)
#endif

using namespace zkp;

// ================================================================== kernels

__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_tower_op(int op, const uint64_t *__restrict__ a, const uint64_t *__restrict__ b, uint64_t *__restrict__ out,
           uint8_t *__restrict__ status, uint32_t *err, size_t n) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;   // element = lane pair
    if (i >= n) return;
    int na, nb, nr;
    tower_op_shape(op, na, nb, nr);
    uint8_t s = tower_op_one(op, a + (size_t)6 * na * i, nb ? b + (size_t)6 * nb * i : nullptr, out + (size_t)6 * nr * i);
    if (lane_par() == 0) {
        if (status) status[i] = s;
        if ((s & 1) && err) atomicOr(err, 1u);
    }
}

// out[t] = in[t] * in[t+m] * in[t+2m] * ...   (t < m <= n), canonical limbs in and out
__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_fp12_product(const uint64_t *__restrict__ in, size_t n, uint64_t *__restrict__ out, size_t m, uint32_t *err) {
    size_t t = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (t >= m) return;
    bool bad = false;
    Fp12 acc, x;
    load_fp12(acc, in + 72 * t, bad);
    for (size_t j = t + m; j < n; j += m) {
        load_fp12(x, in + 72 * j, bad);
        fp12_mul(acc, acc, x);
    }
    store_fp12(out + 72 * t, acc);
    if (lane_or(bad) && err && lane_par() == 0) atomicOr(err, 1u);
}

__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_gen_points(uint64_t seed, uint64_t first, size_t n, uint64_t *__restrict__ g1, uint8_t *__restrict__ g1inf,
             uint64_t *__restrict__ g2, uint8_t *__restrict__ g2inf) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    uint64_t a = splitmix64_at(seed, 2 * (first + i));
    uint64_t b = splitmix64_at(seed, 2 * (first + i) + 1);
    if (a == 0) a = 1;
    if (b == 0) b = 1;
    gen_g1_one(a, g1 + 12 * i, g1inf + i);
    gen_g2_one(b, g2 + 24 * i, g2inf + i);
}

// G2Prepared-style line tables (SURVEY 8f-4): out = [point][68][3][lane parity] Montgomery Fp
__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_g2_prepare(const uint64_t *__restrict__ g2, Fp *__restrict__ out, uint32_t *err, size_t n) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    bool bad = false;
    G2A q;
    load_g2(q, g2 + 24 * i, bad);
    g2_prepare(q, out + i * (ZKP_LINE_STEPS * 3 * 2) + lane_par());
    if (lane_or(bad) && err && lane_par() == 0) atomicOr(err, 1u);
}

// Group-level batch ops (SURVEY 8f): subgroup/on-curve validation and scalar multiplication.
// gop = GroupOp; points are 12 (G1) or 24 (G2) u64 each; flag = status (checks), is_infinity (mul) or bit0 identity | bit1 undefined (add).
__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_group_op(int gop, const uint64_t *__restrict__ pts, const uint8_t *__restrict__ inf, const uint64_t *__restrict__ scalars,
           uint64_t *__restrict__ out_pts, uint8_t *__restrict__ flag, uint32_t *err, size_t n, const uint8_t *__restrict__ inf2) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    const int w = (gop & 1) ? 24 : 12;
    bool bad = false;
    uint8_t is_inf = inf ? inf[i] : 0, f = 0;
    switch (gop) {
        case GOP_G1_CHECK: f = g1_check_one(pts + (size_t)w * i, is_inf, bad); break;
        case GOP_G2_CHECK: f = g2_check_one(pts + (size_t)w * i, is_inf, bad); break;
        case GOP_G1_MUL: g1_mul_one(pts + (size_t)w * i, is_inf, scalars + 4 * i, out_pts + (size_t)w * i, flag + i, bad); break;
        case GOP_G2_MUL: g2_mul_one(pts + (size_t)w * i, is_inf, scalars + 4 * i, out_pts + (size_t)w * i, flag + i, bad); break;
        // additions: the second operand travels in `scalars` (w u64 per element), its flags in inf2
        case GOP_G1_ADD: g1_add_one(pts + (size_t)w * i, is_inf, scalars + (size_t)w * i, inf2 ? inf2[i] : 0, out_pts + (size_t)w * i, flag + i, bad); break;
        default: g2_add_one(pts + (size_t)w * i, is_inf, scalars + (size_t)w * i, inf2 ? inf2[i] : 0, out_pts + (size_t)w * i, flag + i, bad); break;
    }
    bad = lane_or(bad);
    if (lane_par() == 0) {
        if (gop <= GOP_G2_CHECK) flag[i] = f;
        if (bad && err) atomicOr(err, 1u);
    }
}

// ---- Groth16 verification front end (groth16.cuh)

// the verifying key's -beta, -gamma, -delta: negated here, then the prepared line tables of k_g2_prepare
__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_g16_neg_prepare(const uint64_t *__restrict__ g2, Fp *__restrict__ out, size_t n) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    bool bad = false;
    G2A q;
    load_g2(q, g2 + 24 * i, bad);
    q.y = fp2_neg(q.y);
    g2_prepare(q, out + i * (ZKP_LINE_STEPS * 3 * 2) + lane_par());
}

// one THREAD per (IC_j, window): Fp-level work only, no lane exchange.  ic = IC_0 .. IC_l (canonical);
// scratch: 2 * 255 Fp per thread
__global__ void __launch_bounds__(ZKP_TPB)
k_g16_window_tables(const uint64_t *__restrict__ ic, const uint8_t *__restrict__ ic_inf, int n_public, Fp *__restrict__ tables,
                    Fp *__restrict__ scratch) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)n_public * ZKP_G16_WINDOWS) return;
    int j = (int)(t / ZKP_G16_WINDOWS), w = (int)(t % ZKP_G16_WINDOWS);
    if (ic_inf[j + 1]) return;
    Fp *zs = scratch + t * 2 * ZKP_G16_DIGITS;
    groth16_window_table(ic + 12 * (j + 1), w, tables + (size_t)j * ZKP_G16_TABLE_FP + (size_t)w * ZKP_G16_DIGITS * 2, zs,
                         zs + ZKP_G16_DIGITS);
}

__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_groth16_prepare(G16Key vk, const uint64_t *__restrict__ proofs, const uint8_t *__restrict__ proof_inf, const uint64_t *__restrict__ x,
                  size_t n, uint64_t *__restrict__ g1, uint8_t *__restrict__ g1inf, uint64_t *__restrict__ g2,
                  uint8_t *__restrict__ g2inf, uint8_t *__restrict__ status) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    uint8_t s = groth16_prepare_one(vk, proofs + 48 * i, proof_inf ? proof_inf + 3 * i : nullptr, x + (size_t)vk.n_public * 4 * i,
                                    g1 + 48 * i, g1inf + 4 * i, g2 + 24 * i, g2inf + i);
    if (lane_par() == 0) status[i] = s;
}

// the verdict: a front-end rejection stands, otherwise the equation decides
__global__ void k_groth16_verdict(const uint8_t *__restrict__ is_one, uint8_t *__restrict__ status, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t s = status[i];
    status[i] = s ? s : (is_one[i] ? ZKP_G16_VALID : ZKP_G16_INVALID);
}

// ---- KZG point-evaluation verification front end (kzg.cuh)

// the canonical G1 generator at g1 (x|y) and G2 generator at g2 (x.c0|x.c1|y.c0|y.c1): one lane pair
__global__ void k_kzg_generators(uint64_t *__restrict__ g1, uint64_t *__restrict__ g2) {
    if (threadIdx.x >= 2) return;
    store_fp(g1 + 6 * lane_par(), fp_const(ZKP_G1_GEN + ZKP_NL * lane_par()), nullptr);
    store_fp2(g2, fp2_const(ZKP_G2_GEN), nullptr);
    store_fp2(g2 + 12, fp2_const(ZKP_G2_GEN + 2 * ZKP_NL), nullptr);
}

__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_kzg_prepare(const Fp *__restrict__ g1_table, const uint64_t *__restrict__ proofs, const uint8_t *__restrict__ proof_inf,
              const uint64_t *__restrict__ zy, size_t n, uint64_t *__restrict__ g1, uint8_t *__restrict__ g1inf,
              uint8_t *__restrict__ status) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    uint8_t s = kzg_prepare_one(g1_table, proofs + 24 * i, proof_inf ? proof_inf + 2 * i : nullptr, zy + 8 * i, g1 + 24 * i, g1inf + 2 * i);
    if (lane_par() == 0) status[i] = s;
}

// ---- EIP-4844 blob verification front end (blob.cuh)

#ifndef ZKP_BLOB_CHALLENGE_TPB
#define ZKP_BLOB_CHALLENGE_TPB 32   // one thread per blob: small blocks spread a small batch over more SMs
#endif

// the setup's domain table roots_brp (Montgomery), one thread per entry
__global__ void k_blob_domain(Fr *__restrict__ roots) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ZKP_BLOB_N) roots[i] = blob_root(i);
}

// z of every blob (canonical, zy[8 i .. 8 i + 4)): one thread per blob, 2050 dependent SHA-256 compressions
__global__ void __launch_bounds__(ZKP_BLOB_CHALLENGE_TPB)
k_blob_challenge(const uint8_t *__restrict__ blobs, const uint64_t *__restrict__ proofs, const uint8_t *__restrict__ proof_inf, size_t n,
                 uint64_t *__restrict__ zy) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t digest[8];
    blob_challenge_one(blobs + i * ZKP_BLOB_BYTES_, proofs + 24 * i, proof_inf ? proof_inf[2 * i] : 0, digest, zy + 8 * i);
}

// y = p(z) of every blob (zy[8 i + 4 .. 8 i + 8)), or z = r, y = 0 for a blob with an element >= r: one block per blob,
// thread t owning elements t + 256 k (a warp's 32-byte loads are contiguous); one inversion per blob
__global__ void __launch_bounds__(ZKP_BLOB_TPB)
k_blob_eval(const uint8_t *__restrict__ blobs, const Fr *__restrict__ roots, uint64_t *__restrict__ zy) {
    __shared__ BlobShared sh;
    const int t = threadIdx.x;
    const uint8_t *blob = blobs + (size_t)blockIdx.x * ZKP_BLOB_BYTES_;
    uint64_t *o = zy + 8 * (size_t)blockIdx.x;
    const Fr zm = blob_z_mont(o);
    BlobLane ln;
    if (t == 0) blob_eval_init(sh);
    blob_eval_prefix(t, roots, zm, sh, ln);
    __syncthreads();
    for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1) {
        if (t < w) blob_tree_mul(sh.tree, w + t);
        __syncthreads();
    }
    if (t == 0) blob_tree_invert_root(sh.tree);
    __syncthreads();
    for (int w = 1; w < ZKP_BLOB_TPB; w <<= 1) {
        if (t < w) blob_tree_inv(sh.tree, w + t);
        __syncthreads();
    }
    blob_eval_terms(t, blob, roots, zm, sh, ln);
    __syncthreads();
    for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1) {
        if (t < w) blob_tree_add(sh.tree, w + t);
        __syncthreads();
    }
    if (t == 0) blob_eval_finish(sh, zm, o);
}

// ---- EIP-4844 prover (kzg_prove.cuh)

// Signed-digit window tables of the setup points of bases [first, first + count): one THREAD per (base, window).
// permute: table i holds L_brp(i) (lag = the Lagrange points in the setup file's natural order); otherwise point i (the
// monomial points [tau^i]G1 of a cells setup).  scratch: 2 * ZKP_MSM_DIGITS Fp per thread.
__global__ void __launch_bounds__(ZKP_TPB)
k_kzg_lagrange_tables(const uint64_t *__restrict__ lag, int first, int count, bool permute, Fp *__restrict__ tables,
                      Fp *__restrict__ scratch) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count * ZKP_MSM_WINDOWS) return;
    const int i = first + t / ZKP_MSM_WINDOWS, w = t % ZKP_MSM_WINDOWS;
    Fp *zs = scratch + (size_t)t * 2 * ZKP_MSM_DIGITS;
    groth16_window_table(lag + 12 * (permute ? blob_brp(i) : i), w, tables + (size_t)i * ZKP_MSM_TABLE_FP + (size_t)w * ZKP_MSM_DIGITS * 2, zs,
                         zs + ZKP_MSM_DIGITS, ZKP_MSM_DIGITS);
}

// The setup's consistency rows: row 0 all ones (sum_k L_k) and row 1 roots_brp (sum_k omega^k L_k), big-endian
__global__ void k_kzg_check_rows(const Fr *__restrict__ roots, uint8_t *__restrict__ rows) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ZKP_BLOB_N) return;
    Fr one = fr_zero();
    one.l[0] = 1;
    store_be32(rows + 32 * i, one);
    store_be32(rows + ZKP_BLOB_BYTES_ + 32 * i, fr_from_mont(roots[i]));
}

#ifndef ZKP_MSM_MIN_BLOCKS
#define ZKP_MSM_MIN_BLOCKS 2   // resident k_kzg_msm blocks per SM: 128 registers, 16 % faster than one (profiles/r3d_kzg_msm_bounds.txt)
#endif

// sum_i s_i L_brp(i) for every scalar row (4096 x 32 big-endian bytes): one block per row, thread t owning the bases
// t + 256 k; a row with pre[b] != 0 is already rejected.  status may alias pre.
__global__ void __launch_bounds__(ZKP_MSM_TPB, ZKP_MSM_MIN_BLOCKS)
k_kzg_msm(const Fp *__restrict__ tables, const uint8_t *__restrict__ rows, const uint8_t *pre, uint64_t *__restrict__ out,
          uint8_t *__restrict__ out_inf, uint8_t *status) {
    __shared__ MsmShared sh;
    const int t = threadIdx.x;
    const size_t b = blockIdx.x;
    const uint8_t p = pre ? pre[b] : 0;
    if (t == 0) msm_init(sh);
    __syncthreads();
    msm_partial(t, tables, rows + b * ZKP_BLOB_BYTES_, p != 0, sh);
    __syncthreads();
    for (int w = ZKP_MSM_TPB / 2; w >= 1; w >>= 1) {
        if (t < w) msm_tree_add(sh, t, w);
        __syncthreads();
    }
    if (t == 0) status[b] = msm_finish(sh, p, out + 12 * b, out_inf + b);
}

// compute_blob_kzg_proof's front: C's check and z, one thread per blob (commitments = n x 12 u64)
__global__ void __launch_bounds__(ZKP_BLOB_CHALLENGE_TPB)
k_kzg_prove_challenge(const uint8_t *__restrict__ blobs, const uint64_t *__restrict__ c, const uint8_t *__restrict__ cinf, size_t n,
                      uint64_t *__restrict__ zy, uint8_t *__restrict__ status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    status[i] = prove_challenge_one(blobs + i * ZKP_BLOB_BYTES_, c + 12 * i, cinf ? cinf[i] : 0, zy + 8 * i);
}

// The quotient row of every blob (compute_kzg_proof_impl): y = p(z) by k_blob_eval's steps, then q_i in place of the
// inverses 1/(z - omega_i) that step 5 leaves in the row.  z from z_in (n x 4) or, when z_in is NULL, already in zy;
// y also to y_out (optional, n x 4; 0 for a rejected blob).  pre (may alias status): earlier rejections, or NULL.
__global__ void __launch_bounds__(ZKP_BLOB_TPB)
k_kzg_quotient(const uint8_t *__restrict__ blobs, const Fr *__restrict__ roots, const uint64_t *__restrict__ z_in, uint64_t *__restrict__ zy,
               uint64_t *__restrict__ y_out, uint8_t *__restrict__ rows, const uint8_t *pre, uint8_t *status) {
    __shared__ QuotShared sh;
    const int t = threadIdx.x;
    const size_t b = blockIdx.x;
    const uint8_t *blob = blobs + b * ZKP_BLOB_BYTES_;
    uint8_t *row = rows + b * ZKP_BLOB_BYTES_;
    uint64_t *o = zy + 8 * b;
    const uint8_t p = pre ? pre[b] : 0;
    BlobLane ln;
    if (t == 0) quot_init(sh, z_in ? z_in + 4 * b : nullptr, o);
    __syncthreads();
    const Fr zm = sh.zm;
    blob_eval_prefix(t, roots, zm, sh.b, ln);
    __syncthreads();
    for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1) {
        if (t < w) blob_tree_mul(sh.b.tree, w + t);
        __syncthreads();
    }
    if (t == 0) blob_tree_invert_root(sh.b.tree);
    __syncthreads();
    for (int w = 1; w < ZKP_BLOB_TPB; w <<= 1) {
        if (t < w) blob_tree_inv(sh.b.tree, w + t);
        __syncthreads();
    }
    blob_eval_terms<true>(t, blob, roots, zm, sh.b, ln, (Fr *)row);
    __syncthreads();
    for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1) {
        if (t < w) blob_tree_add(sh.b.tree, w + t);
        __syncthreads();
    }
    if (t == 0) {
        blob_eval_finish(sh.b, zm, o);
        status[b] = quot_status(sh, p, o, y_out ? y_out + 4 * b : nullptr);
    }
    __syncthreads();
    quot_terms(t, blob, roots, sh, row);
    __syncthreads();
    if (sh.b.hit) {   // z = omega_m: one more sum for the entry m
        for (int w = ZKP_BLOB_TPB / 2; w >= 1; w >>= 1) {
            if (t < w) blob_tree_add(sh.b.tree, w + t);
            __syncthreads();
        }
        if (t == 0) quot_within_domain(sh, row);
    }
}

// ---- EIP-7594 cells (kzg_cells.cuh)

// the cells setup's twiddle table pw[e] = omega_8192^e (Montgomery), one thread per entry
__global__ void k_cells_powers(Fr *__restrict__ pw) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < ZKP_CELLS_EXT_N) pw[e] = cells_power(e);
}

// The inputs of the cells setup's pairing checks from the monomial points M_i (mono, 4096 x 12) and G1 (g1, 12):
// chain[i] = [M_{i+1}, M_i] for i < 4095 (against G2, -[tau]G2), and pairs[i] = [-G1, M_i] for i <= 64 (against
// g2_monomial[i] in the per-check slot, then G2).  One lane pair per i.
__global__ void k_cells_setup_pairs(const uint64_t *__restrict__ mono, const uint64_t *__restrict__ g1, uint64_t *__restrict__ chain,
                                    uint64_t *__restrict__ pairs) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= ZKP_BLOB_N - 1) return;
    const int par = lane_par();
    copy_u64(chain + 24 * i + 6 * par, mono + 12 * (i + 1) + 6 * par, 6, false);
    copy_u64(chain + 24 * i + 12 + 6 * par, mono + 12 * i + 6 * par, 6, false);
    if (i <= ZKP_CELL_N) {
        bool b = false;
        const Fp v = load_fp(g1 + 6 * par, b);
        store_fp(pairs + 24 * i + 6 * par, par ? fp_neg(v) : v, nullptr);
        copy_u64(pairs + 24 * i + 12 + 6 * par, mono + 12 * i + 6 * par, 6, false);
    }
}

// compute_cells: the 128 cells of every blob (n x 256 KiB) and its status; coeffs (n x 4096 Fr, or NULL) receives the
// blob's coefficients for the proofs.  One block per blob, the blob's 4096 Fr in dynamic shared memory (128 KiB).
__global__ void __launch_bounds__(ZKP_CELLS_TPB)
k_cells_extend(const uint8_t *__restrict__ blobs, const Fr *__restrict__ pw, uint8_t *__restrict__ cells, Fr *__restrict__ coeffs,
               uint8_t *__restrict__ status) {
    extern __shared__ Fr cells_x[];
    __shared__ uint32_t bad;
    const int t = threadIdx.x;
    const size_t b = blockIdx.x;
    const uint8_t *blob = blobs + b * ZKP_BLOB_BYTES_;
    if (t == 0) bad = 0;
    __syncthreads();
    cells_load(t, blob, cells_x, &bad);
    __syncthreads();
    for (int h = 1; h < ZKP_BLOB_N; h <<= 1) {
        cells_dit_pass(t, cells_x, pw, h);
        __syncthreads();
    }
    cells_scale(t, cells_x, pw, coeffs ? coeffs + b * ZKP_BLOB_N : nullptr);
    __syncthreads();
    for (int h = ZKP_BLOB_N / 2; h >= 1; h >>= 1) {
        cells_dif_pass(t, cells_x, pw, h);
        __syncthreads();
    }
    cells_store(t, blob, cells_x, bad != 0, cells + b * 2 * ZKP_BLOB_BYTES_);
    if (t == 0) status[b] = bad ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
}

// The quotient rows of every blob's 128 cosets (n x 128 rows of 4096 x 32 bytes), one thread per (blob, coset, chain);
// row_status[128 b + k] = status[b], the rejection k_kzg_msm reads for the row
__global__ void __launch_bounds__(ZKP_CELLS_QUOT_TPB)
k_cells_quotient(const Fr *__restrict__ coeffs, const Fr *__restrict__ pw, const uint8_t *__restrict__ status, size_t n,
                 uint8_t *__restrict__ rows, uint8_t *__restrict__ row_status) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n * ZKP_CELLS_PER_BLOB * ZKP_CELL_N) return;
    const size_t r = g / ZKP_CELL_N, b = r / ZKP_CELLS_PER_BLOB;
    const int m = (int)(g % ZKP_CELL_N);
    const uint8_t st = status[b];
    if (m == 0) row_status[r] = st;
    if (st) return;
    cells_quotient_chain((int)(r % ZKP_CELLS_PER_BLOB), m, coeffs + b * ZKP_BLOB_N, pw, rows + r * ZKP_BLOB_BYTES_);
}

// recover_cells: one cluster of two blocks per blob (kzg_recover.cuh), rank r holding slots [4096 r, 4096 r + 4096) of
// the extended blob in dynamic shared memory (128 KiB).  idx (n x 128), cells (n x 128 x 2048 bytes) and num (n) are
// the input; out receives the 128 cells (n x 256 KiB), coeffs (n x 4096 Fr, or NULL) the coefficients for the proofs.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ZKP_CELLS_TPB, 1)
k_cells_recover(const uint64_t *__restrict__ idx, const uint8_t *__restrict__ cells, const uint64_t *__restrict__ num,
                const Fr *__restrict__ pw, uint8_t *__restrict__ out, Fr *__restrict__ coeffs, uint8_t *__restrict__ status) {
    namespace cg = cooperative_groups;
    extern __shared__ Fr rec_x[];
    __shared__ RecoverShared sh;
    cg::cluster_group cl = cg::this_cluster();
    const int r = (int)cl.block_rank(), t = threadIdx.x;
    const size_t b = blockIdx.x / 2;
    const uint64_t n = num[b];
    recover_init(t, n, sh);
    __syncthreads();
    recover_index(t, n, idx + b * ZKP_CELLS_PER_BLOB, sh);
    __syncthreads();
    recover_vanish_part(r, t, pw, sh, rec_x);
    __syncthreads();
    if (t < ZKP_CELL_N) recover_vanish(t, rec_x, sh);
    __syncthreads();
    recover_load(r, t, cells + b * ZKP_CELLS_PER_BLOB * ZKP_CELL_BYTES_, sh, rec_x);
    __syncthreads();
    for (int h = 1; h < ZKP_RECOVER_HALF; h <<= 1) {
        cells_dit_pass(t, rec_x, pw, h);
        __syncthreads();
    }
    cl.sync();   // both halves transformed (and both blocks' sh.bad final)
    Fr *half[2];
    half[r] = rec_x;
    half[r ^ 1] = cl.map_shared_rank(rec_x, r ^ 1);
    const bool bad_other = cl.map_shared_rank(&sh, r ^ 1)->bad != 0;
    const bool rej = sh.bad_cells || sh.bad || bad_other;
    recover_cross_a(r, t, pw, half);
    cl.sync();
    for (int h = ZKP_RECOVER_HALF / 2; h >= 1; h >>= 1) {
        cells_dif_pass(t, rec_x, pw, h);
        __syncthreads();
    }
    recover_divide(t, sh, rec_x);
    __syncthreads();
    for (int h = 1; h < ZKP_RECOVER_HALF; h <<= 1) {
        cells_dit_pass(t, rec_x, pw, h);
        __syncthreads();
    }
    cl.sync();
    recover_cross_b(r, t, pw, half, coeffs ? coeffs + b * ZKP_BLOB_N : nullptr);
    cl.sync();   // also: no block reads the other's shared memory after this
    for (int h = ZKP_RECOVER_HALF / 2; h >= 1; h >>= 1) {
        cells_dif_pass(t, rec_x, pw, h);
        __syncthreads();
    }
    recover_store(r, t, rec_x, rej, out + b * 2 * ZKP_BLOB_BYTES_);
    if (r == 0 && t == 0) status[b] = recover_status(sh, bad_other);
}

// The verifier's interpolation, one 64-thread block per cell: I_k from the cell, then [I_k(tau)]G1 over the first 64
// monomial tables (ixy / iinf), and the status (ZKP_KZG_BAD_SCALAR for an element >= r or an index >= 128)
__global__ void __launch_bounds__(ZKP_CELL_N)
k_cells_interp(const uint8_t *__restrict__ cells, const uint64_t *__restrict__ idx, const Fr *__restrict__ pw, const Fp *__restrict__ mono,
               uint64_t *__restrict__ ixy, uint8_t *__restrict__ iinf, uint8_t *__restrict__ status) {
    __shared__ CellShared sh;
    const int t = threadIdx.x;
    const size_t c = blockIdx.x;
    const uint64_t k = idx[c];
    if (t == 0) cell_init(sh, k);
    __syncthreads();
    cell_load(t, cells + c * ZKP_CELL_BYTES_, sh);
    __syncthreads();
    for (int h = 1; h < ZKP_CELL_N; h <<= 1) {
        if (t < ZKP_CELL_N / 2) cells_dit(sh.x, pw, t, h);
        __syncthreads();
    }
    cell_interp_scale(t, k, pw, sh);
    __syncthreads();
    const uint8_t pre = sh.bad ? ZKP_KZG_BAD_SCALAR : ZKP_KZG_VALID;
    msm_partial<ZKP_CELL_N>(t, mono, sh.row, pre != 0, sh.msm);
    __syncthreads();
    for (int w = ZKP_CELL_N / 2; w >= 1; w >>= 1) {
        if (t < w) msm_tree_add(sh.msm, t, w);
        __syncthreads();
    }
    if (t == 0) status[c] = msm_finish(sh.msm, pre, ixy + 12 * c, iinf + c);
}

// The verifier's pairs, one lane pair per cell (cell_prepare_one); status holds k_cells_interp's and is updated
__global__ void __launch_bounds__(ZKP_TPB, ZKP_MIN_BLOCKS)
k_cells_prepare(const uint64_t *__restrict__ c, const uint8_t *__restrict__ cinf, const uint64_t *__restrict__ idx,
                const uint64_t *__restrict__ pi, const uint8_t *__restrict__ piinf, const Fr *__restrict__ pw, const uint64_t *__restrict__ ixy,
                const uint8_t *__restrict__ iinf, size_t n, uint64_t *__restrict__ g1, uint8_t *__restrict__ g1inf, uint8_t *status) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    const uint8_t pre = status[i];   // both lanes read it before the lane exchanges of cell_prepare_one; the even lane writes last
    const uint8_t s = cell_prepare_one(c + 12 * i, cinf ? cinf[i] : 0, pi + 12 * i, piinf ? piinf[i] : 0, idx[i], pw, ixy + 12 * i, iinf[i],
                                       pre, g1 + 24 * i, g1inf + 2 * i);
    if (lane_par() == 0) status[i] = s;
}

// ---- multi-scalar multiplication over caller-given points (msm.cuh); O = OpsFp (G1, one thread per point or
// segment) or OpsFp2 (G2, one lane pair)

#define ZKP_MSM_KTPB 128   // threads per block of the per-point and per-segment kernels

template <class O>
__global__ void __launch_bounds__(ZKP_MSM_KTPB)
k_msm_check(const uint64_t *__restrict__ xy, const uint8_t *__restrict__ inf, size_t n, Fp *__restrict__ pts, uint8_t *__restrict__ valid,
            uint32_t *off, uint32_t *err) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / MsmWidth<O>::W;
    if (i >= n) return;
    msm_check<O>(i, xy, inf, pts, valid, off, err);
}

// every thread runs the window loop (the claims are warp-wide), also past n
__global__ void __launch_bounds__(ZKP_MSM_KTPB)
k_msm_digits(const uint64_t *__restrict__ scalars, const uint8_t *__restrict__ valid, size_t n, int c, uint32_t *ctr, uint32_t *keys,
             uint32_t *vals) {
    msm_digits((size_t)blockIdx.x * blockDim.x + threadIdx.x, n, scalars, valid, c, ctr, keys, vals);
}

__global__ void __launch_bounds__(ZKP_MSM_SCAN_TPB)
k_msm_scan(const uint32_t *__restrict__ cnt, uint32_t nb, uint32_t *__restrict__ off, uint32_t *__restrict__ cur, uint32_t *len) {
    __shared__ uint32_t part[ZKP_MSM_SCAN_TPB];
    const int t = threadIdx.x;
    msm_scan_sum(t, ZKP_MSM_SCAN_TPB, cnt, nb, part);
    __syncthreads();
    if (t == 0) msm_scan_prefix(ZKP_MSM_SCAN_TPB, part, off + nb, len);
    __syncthreads();
    msm_scan_write(t, ZKP_MSM_SCAN_TPB, cnt, nb, part, off, cur);
}

template <class O, bool AFF>
__global__ void __launch_bounds__(ZKP_MSM_KTPB)
k_msm_segment(const uint32_t *len_in, uint32_t *len_out, const uint32_t *__restrict__ keys, const uint32_t *__restrict__ vals,
              const Fp *__restrict__ src, Fp *buckets, uint32_t *__restrict__ fkey, Fp *__restrict__ fval, size_t nseg) {
    const size_t s = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / MsmWidth<O>::W;
    if (s >= nseg) return;
    msm_segment<O, AFF>(s, ZKP_MSM_SEG, len_in, len_out, keys, vals, src, buckets, fkey, fval);
}

// one block per window: R ranges (R <= ZKP_MSM_RANGES), then the tree over ZKP_MSM_RANGES slots
template <class O>
__global__ void __launch_bounds__(ZKP_MSM_RANGES * 2)
k_msm_reduce(const Fp *__restrict__ buckets, int M, int R, Fp *__restrict__ wsum) {
    __shared__ Fp sh[ZKP_MSM_RANGES * 3 * MsmWidth<O>::W];
    const int q = threadIdx.x / MsmWidth<O>::W, w = blockIdx.x;
    Jac<O> r;
    msm_id(r);
    if (q < R) msm_range<O>(w, q, R, M, buckets, r);
    msm_stj(sh, q, r);
    __syncthreads();
    for (int h = ZKP_MSM_RANGES / 2; h >= 1; h >>= 1) {
        if (q < h) msm_tree_step<O>(sh, q, h);
        __syncthreads();
    }
    if (q == 0) {
        msm_ldj(r, sh, 0);
        msm_stj(wsum, w, r);
    }
}

template <class O>
__global__ void k_msm_combine(int nw, int c, const Fp *__restrict__ wsum, Fp *__restrict__ part) {
    msm_combine<O>(nw, c, wsum, part);
}

template <class O>
__global__ void k_msm_sum(const Fp *__restrict__ parts, int np, Fp *__restrict__ out) {
    msm_sum<O>(parts, np, out);
}

template <class O>
__global__ void k_msm_final(const Fp *__restrict__ parts, int np, const uint32_t *__restrict__ offs, int noff, uint64_t *__restrict__ out_xy,
                            uint8_t *__restrict__ out_inf, uint8_t *__restrict__ status) {
    const uint8_t st = msm_final<O>(parts, np, offs, noff, out_xy, out_inf);
    if (msm_writer<O>()) *status = st;
}

// Byte (de)serialisation at the boundary (SURVEY 8f-2): 48 big-endian bytes <-> six little-endian u64
// limbs, Fp::from_bytes / Fp::to_bytes (src/fp.rs:165-207).  Pure byte shuffling, HBM bound: one
// thread moves one element with three 128-bit loads and three 128-bit stores (a warp covers 1536
// contiguous bytes on both sides).  dir 0: bytes -> limbs (+ canonical flag), dir 1: limbs -> bytes.
__device__ __forceinline__ uint64_t bswap64(uint64_t x) {
    uint32_t lo = __byte_perm((uint32_t)x, 0, 0x0123), hi = __byte_perm((uint32_t)(x >> 32), 0, 0x0123);
    return ((uint64_t)lo << 32) | hi;
}
__global__ void __launch_bounds__(256) k_fp_bytes(int dir, const uint4 *__restrict__ in, uint4 *__restrict__ out,
                                                  uint8_t *__restrict__ ok, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint4 a = in[3 * i], b = in[3 * i + 1], c = in[3 * i + 2];
    // reversing all 48 bytes: the three 16-byte chunks swap ends, each chunk is byte-reversed
    uint64_t w[6] = {((uint64_t)a.y << 32) | a.x, ((uint64_t)a.w << 32) | a.z, ((uint64_t)b.y << 32) | b.x,
                     ((uint64_t)b.w << 32) | b.z, ((uint64_t)c.y << 32) | c.x, ((uint64_t)c.w << 32) | c.z};
    uint64_t r[6];
#pragma unroll
    for (int k = 0; k < 6; k++) r[k] = bswap64(w[5 - k]);
    out[3 * i] = make_uint4((uint32_t)r[0], (uint32_t)(r[0] >> 32), (uint32_t)r[1], (uint32_t)(r[1] >> 32));
    out[3 * i + 1] = make_uint4((uint32_t)r[2], (uint32_t)(r[2] >> 32), (uint32_t)r[3], (uint32_t)(r[3] >> 32));
    out[3 * i + 2] = make_uint4((uint32_t)r[4], (uint32_t)(r[4] >> 32), (uint32_t)r[5], (uint32_t)(r[5] >> 32));
    if (dir == 0 && ok) {   // canonical: value < p (src/fp.rs:176-190)
        uint64_t borrow = 0;
#pragma unroll
        for (int k = 0; k < 6; k++) {
            uint64_t pk = ((uint64_t)ZKP_P[2 * k + 1] << 32) | ZKP_P[2 * k];
            uint64_t d = r[k] - pk;
            borrow = (r[k] < pk) | (d < borrow);
        }
        ok[i] = (uint8_t)borrow;   // 1 = canonical (Ok), 0 = Err(())
    }
}

// Integer-multiply roofline probe.  Every chain gets its own multiplier and the multiplicand changes
// every iteration, so nothing is loop invariant (ptxas would otherwise hoist the product and leave
// 64-bit adds).  KIND 0: 8 independent IMAD.WIDE.U32 accumulate chains per thread; KIND 1: 8
// independent 32-bit IMAD chains; KIND 2: the carry-chained wide MACs exactly as the Montgomery
// rows of fp.cuh issue them (row_mad: two 6-MAC carry chains per step).
template <int KIND>
__global__ void __launch_bounds__(512) k_imad_peak(uint32_t *sink, int iters) {
    uint32_t x = threadIdx.x * 2654435761u + 12345u, y = blockIdx.x * 40503u + 977u;
    uint32_t m = x;
    if (KIND == 0) {
        uint64_t acc[8];
        uint32_t ys[8];
#pragma unroll
        for (int c = 0; c < 8; c++) { acc[c] = x + c; ys[c] = y * (2 * c + 3) + sink[1]; }
        for (int it = 0; it < iters; it++) {
            asm volatile("shf.l.wrap.b32 %0, %0, %0, 7;" : "+r"(m));   // rotate + add (SHF, IADD3): only the counted MACs touch the multiply pipe
            m += 0x9E3779B9u;
#pragma unroll
            for (int c = 0; c < 8; c++) asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[c]) : "r"(m), "r"(ys[c]));
        }
        uint64_t s = 0;
#pragma unroll
        for (int c = 0; c < 8; c++) s ^= acc[c];
        if (s == 0x123456789abcdefull) sink[0] = (uint32_t)s;
    } else if (KIND == 1) {
        uint32_t acc[8], ys[8];
#pragma unroll
        for (int c = 0; c < 8; c++) { acc[c] = x + c; ys[c] = y * (2 * c + 3) + sink[1]; }
        for (int it = 0; it < iters; it++) {
            asm volatile("shf.l.wrap.b32 %0, %0, %0, 7;" : "+r"(m));   // rotate + add (SHF, IADD3): only the counted MACs touch the multiply pipe
            m += 0x9E3779B9u;
#pragma unroll
            for (int c = 0; c < 8; c++) asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(acc[c]) : "r"(m), "r"(ys[c]));
        }
        uint32_t s = 0;
#pragma unroll
        for (int c = 0; c < 8; c++) s ^= acc[c];
        if (s == 0x12345678u) sink[0] = s;
    } else {
        uint32_t ev[12], od[12], a[12];
#pragma unroll
        for (int c = 0; c < 12; c++) { ev[c] = x + c; od[c] = y + c; a[c] = x * (c + 3) + y + sink[1]; }
        for (int it = 0; it < iters; it++) {
            asm volatile("shf.l.wrap.b32 %0, %0, %0, 7;" : "+r"(m));   // rotate + add (SHF, IADD3): only the counted MACs touch the multiply pipe
            m += 0x9E3779B9u;
            row_mad(ev, od, a, m);
        }
        uint32_t s = 0;
#pragma unroll
        for (int c = 0; c < 12; c++) s ^= ev[c] ^ od[c];
        if (s == 0x12345678u) sink[0] = s;
    }
}

// ================================================================== host side

static thread_local std::string g_err;
static int32_t fail(int32_t code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(ZKP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));         \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// pinned host staging for user buffers that are pageable (a plain Vec / numpy array): an async copy to or
// from pageable memory blocks the issuing thread until it is done, which would serialise the two buffer
// sets of the pipeline; staged through these, the copies of one set overlap the kernels of the other
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};
struct PendingOut {   // staged device->host copy still to be moved into the caller's buffer
    void *user;
    const void *stage;
    size_t bytes;
};

enum { B_G1 = 0, B_G1INF, B_G2, B_G2INF, B_IN, B_OUT, B_FLAG, B_TAB, B_NBUF, B_TABINF = B_NBUF, B_NPIN };
#ifndef ZKP_STAGE_MIN
#define ZKP_STAGE_MIN ((size_t)256 << 10)   // smaller transfers go straight from / to the caller's memory
#endif

struct DevState {
    int id = 0;
    int sms = 0;
    cudaStream_t stream[2] = {nullptr, nullptr};
    // helper stream + fork/join events of the final exponentiation's two-stream split: one set per context
    // stream and a third for launches on caller streams (created once here, never in a call)
    ZkpFeAux fe_aux[3] = {};
    uint32_t *d_err = nullptr;
    cudaMemPool_t pool = nullptr;   // stream-ordered scratch of the final exponentiation (kept, never trimmed)
    DevBuf buf[2][B_NBUF];     // double-buffered pipeline scratch
    PinBuf pin_in[2][B_NPIN], pin_out[2][B_NPIN];   // pinned staging per buffer set (only for pageable user buffers)
    std::vector<PendingOut> pend[2];
    DevBuf scratch, partial;   // product reduction
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timers;
    double timed_ms = 0;
    uint64_t timed_launches = 0;
};

struct zkp_ctx {
    std::vector<DevState> devs;
    std::mutex mu;
    std::atomic<uint64_t> launches{0};
    bool timing = false;
};

// Entry points select the device they work on; the caller's current device is restored on every exit path
// (a torch process keeps allocating on ITS device after a call into a multi-device context).
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            cudaGetLastError();
            prev = -1;
        }
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};

// two threads (one lane pair) per element
static inline unsigned grid_for(size_t n) { return (unsigned)((2 * n + ZKP_TPB - 1) / ZKP_TPB); }

// the pairing kernels live in pairing_kernel.cu (compiled with warp-converged shuffles)
extern "C" size_t zkp_fe_scratch_bytes(size_t n);
cudaError_t zkp_launch_k_pairing(int mode, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                                 size_t n, int k, const uint64_t *in12, uint64_t *out, uint8_t *is_one, uint32_t *err,
                                 void *scratch, const void *tab, const uint8_t *tabinf, int kf, cudaStream_t st, const ZkpFeAux *aux,
                                 int *launches);

static cudaError_t launch_pairing(zkp_ctx *ctx, DevState &d, int mode, const uint64_t *g1, const uint8_t *g1inf,
                                  const uint64_t *g2, const uint8_t *g2inf, size_t n, int k, const uint64_t *in12,
                                  uint64_t *out, uint8_t *is_one, uint32_t *err, cudaStream_t st,
                                  const void *tab = nullptr, const uint8_t *tabinf = nullptr, int kf = 0) {
    if (n == 0) return cudaSuccess;
    // the final exponentiation parks its state between launches in stream-ordered scratch memory
    void *scratch = nullptr;
    if (mode & 2) {
        cudaError_t e = cudaMallocFromPoolAsync(&scratch, zkp_fe_scratch_bytes(n), d.pool, st);
        if (e != cudaSuccess) return e;
    }
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (ctx->timing) {   // (created after the only early return, so that no event is left behind)
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        cudaEventRecord(e0, st);
    }
    int nl = 0;
    const ZkpFeAux *aux = &d.fe_aux[st == d.stream[0] ? 0 : st == d.stream[1] ? 1 : 2];
    cudaError_t rc = zkp_launch_k_pairing(mode, g1, g1inf, g2, g2inf, n, k, in12, out, is_one, err, scratch, tab, tabinf, kf, st, aux, &nl);
    ctx->launches += nl;
    if (scratch) cudaFreeAsync(scratch, st);
    if (ctx->timing) {
        cudaEventRecord(e1, st);
        d.timers.emplace_back(e0, e1);
    }
    return rc;
}

// product of n canonical Fp12 at d_in -> d_out (1 element).  scratch: zkp_product_scratch_elems(n)
static const size_t PROD_M1 = 8192, PROD_M2 = 64;
extern "C" size_t zkp_product_scratch_elems(size_t n) {
    (void)n;
    return PROD_M1 + PROD_M2;
}
static cudaError_t launch_product(zkp_ctx *ctx, const uint64_t *d_in, size_t n, uint64_t *d_scratch, uint64_t *d_out,
                                  uint32_t *err, cudaStream_t st) {
    const uint64_t *cur = d_in;
    size_t cnt = n;
    uint64_t *s1 = d_scratch, *s2 = d_scratch + 72 * PROD_M1;
    if (cnt > PROD_M1) {
        k_fp12_product<<<grid_for(PROD_M1), ZKP_TPB, 0, st>>>(cur, cnt, s1, PROD_M1, err);
        ctx->launches++;
        cur = s1;
        cnt = PROD_M1;
    }
    if (cnt > PROD_M2) {
        k_fp12_product<<<grid_for(PROD_M2), ZKP_TPB, 0, st>>>(cur, cnt, s2, PROD_M2, err);
        ctx->launches++;
        cur = s2;
        cnt = PROD_M2;
    }
    k_fp12_product<<<1, ZKP_TPB, 0, st>>>(cur, cnt, d_out, 1, err);
    ctx->launches++;
    return cudaGetLastError();
}

// ---- Groth16 verification: resident verifying key and the per-batch launch sequence

static inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

struct G16Dev {   // one device's copy of a verifying key, in one allocation
    int id = 0;
    void *mem = nullptr;
    const Fp *prep = nullptr;   // prepared tables of -beta, -gamma, -delta
    G16Key key = {};
};
struct zkp_groth16_vk {
    zkp_ctx *ctx = nullptr;
    int n_public = 0;
    std::vector<G16Dev> devs;   // one per device of ctx, same order
};

// proofs per host pipeline chunk: at most 2^18, and at most 64 MB of public inputs (2^21 scalars)
static size_t g16_chunk(int n_public) {
    size_t c = n_public > 8 ? ((size_t)ZKP_CHUNK * 8) / (size_t)n_public : (size_t)ZKP_CHUNK;
    return c ? c : 1;
}

// Carves scratch into consecutive parts of the given sizes, each rounded up to 256 bytes: part[i] is where part i
// starts (NULL when base is NULL).  Returns the bytes of all parts.
template <size_t N> static size_t carve(void *base, const size_t (&sz)[N], uint8_t *(&part)[N]) {
    size_t o = 0;
    for (size_t i = 0; i < N; i++) {
        part[i] = base ? (uint8_t *)base + o : nullptr;
        o += align256(sz[i]);
    }
    return o;
}

// The prepared check of n assembled checks (k pairs each, the last kf of them from the tables prep), then the verdicts
// of the front end's status bytes.  The verifiers share it: Groth16 (k = 4, kf = 3), KZG and cells (k = kf = 2).
static cudaError_t launch_check_verdict(zkp_ctx *ctx, DevState &d, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2,
                                        const uint8_t *g2inf, size_t n, int k, const Fp *prep, int kf, uint64_t *gt, uint8_t *is_one,
                                        uint8_t *status, uint32_t *err, cudaStream_t st) {
    cudaError_t e = launch_pairing(ctx, d, 3, g1, g1inf, g2, g2inf, n, k, nullptr, gt, is_one, err, st, prep, nullptr, kf);
    if (e != cudaSuccess) return e;
    k_groth16_verdict<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(is_one, status, n);
    ctx->launches++;
    return cudaGetLastError();
}

// scratch of one batch of n proofs: assembled pairs [A, alpha, L, C] x [B], the Gt outputs and is_one
struct G16Scratch {
    uint64_t *g1, *g2, *gt;
    uint8_t *g1inf, *g2inf, *is_one;
};
static size_t g16_layout(size_t n, void *base, G16Scratch *s) {
    uint8_t *p[6];
    const size_t bytes = carve(base, {n * 4 * 96, n * 192, n * 576, n * 4, n, n}, p);
    if (s) *s = {(uint64_t *)p[0], (uint64_t *)p[1], (uint64_t *)p[2], p[3], p[4], p[5]};
    return bytes;
}

// front end -> prepared 4-pair check (k = 4, the last kf = 3 pairs from the key's tables) -> verdict
static cudaError_t launch_groth16(zkp_ctx *ctx, DevState &d, const G16Dev &k, const uint64_t *proofs, const uint8_t *proof_inf,
                                  const uint64_t *x, size_t n, uint8_t *status, void *scratch, uint32_t *err, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    G16Scratch s;
    g16_layout(n, scratch, &s);
    k_groth16_prepare<<<grid_for(n), ZKP_TPB, 0, st>>>(k.key, proofs, proof_inf, x, n, s.g1, s.g1inf, s.g2, s.g2inf, status);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_check_verdict(ctx, d, s.g1, s.g1inf, s.g2, s.g2inf, n, 4, k.prep, 3, s.gt, s.is_one, status, err, st);
}

// ---- KZG point-evaluation verification: resident setup and the per-batch launch sequence

struct KzgDev {   // one device's copy of a setup, in one allocation
    int id = 0;
    void *mem = nullptr;
    const Fp *prep = nullptr;    // prepared tables of G2 and -[tau]G2
    const Fp *table = nullptr;   // window table of G1 (ZKP_G16_TABLE_FP)
    const Fr *roots = nullptr;   // the blob domain roots_brp (ZKP_BLOB_N Fr, Montgomery)
    void *lag_mem = nullptr;     // prover setups only: the signed-digit window tables of L_brp(0) .. L_brp(4095)
    void *cell_mem = nullptr;    // cells setups only, one allocation of the three below
    const Fp *cell_prep = nullptr;   // prepared tables of G2 and -[tau^64]G2
    const Fr *pw = nullptr;          // omega_8192^e, e < 8192 (Montgomery)
    const Fp *mono = nullptr;        // the signed-digit window tables of [tau^i]G1, i < 4096
    int recover_clusters = 0;        // cudaOccupancyMaxActiveClusters of k_cells_recover; recovery needs >= 1
    cudaError_t recover_err = cudaSuccess;   // why that query failed
};
struct zkp_kzg_setup {
    zkp_ctx *ctx = nullptr;
    bool prover = false;        // has Lagrange tables: zkp_kzg_setup_create_prover, or zkp_kzg_setup_create_cells with g1_lagrange
    bool cells = false;         // made by zkp_kzg_setup_create_cells
    std::vector<KzgDev> devs;   // one per device of ctx, same order
};

// scratch of one batch of n proofs: assembled pairs [P, pi], their flags, the Gt outputs and is_one
struct KzgScratch {
    uint64_t *g1, *gt;
    uint8_t *g1inf, *is_one;
};
static size_t kzg_layout(size_t n, void *base, KzgScratch *s) {
    uint8_t *p[4];
    const size_t bytes = carve(base, {n * 2 * 96, n * 576, n * 2, n}, p);
    if (s) *s = {(uint64_t *)p[0], (uint64_t *)p[1], p[2], p[3]};
    return bytes;
}

// front end -> prepared 2-pair check (k = kf = 2: both G2 points from the setup's tables) -> verdict
static cudaError_t launch_kzg(zkp_ctx *ctx, DevState &d, const KzgDev &k, const uint64_t *proofs, const uint8_t *proof_inf,
                              const uint64_t *zy, size_t n, uint8_t *status, void *scratch, uint32_t *err, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    KzgScratch s;
    kzg_layout(n, scratch, &s);
    k_kzg_prepare<<<grid_for(n), ZKP_TPB, 0, st>>>(k.table, proofs, proof_inf, zy, n, s.g1, s.g1inf, status);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_check_verdict(ctx, d, s.g1, s.g1inf, nullptr, nullptr, n, 2, k.prep, 2, s.gt, s.is_one, status, err, st);
}

// ---- EIP-4844 blob verification: z by k_blob_challenge, y by k_blob_eval, then the point-evaluation check

#ifndef ZKP_BLOB_CHUNK
// blobs per host pipeline chunk: 2 GiB of blobs per buffer set.  Measured at 2^15 blobs (profiles/r3c_kzg_blob_chunk.txt,
// B200 at 1000 W), chunks of 2^10 .. 2^14 blobs: 42 / 71 / 108 / 146 / 171 k blobs/s from pinned and 31 / 44 / 56 / 64 /
// 69 k blobs/s from pageable memory; every launch sequence pays the fixed latency of the transcript (4.3 ms).
#define ZKP_BLOB_CHUNK (1u << 14)
#endif

// scratch of one batch of n blobs: z | y (n x 64 bytes), then the point-evaluation scratch
static size_t blob_zy_bytes(size_t n) { return align256(n * 64); }
extern "C" size_t zkp_kzg_blob_scratch_bytes(size_t n) { return blob_zy_bytes(n) + kzg_layout(n, nullptr, nullptr); }

// zy = the caller's z | y buffer, or NULL for the one in scratch
static cudaError_t launch_kzg_blob(zkp_ctx *ctx, DevState &d, const KzgDev &k, const uint8_t *blobs, const uint64_t *proofs,
                                   const uint8_t *proof_inf, size_t n, uint8_t *status, uint64_t *zy, void *scratch, uint32_t *err,
                                   cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    if (!zy) zy = (uint64_t *)scratch;
    k_blob_challenge<<<(unsigned)((n + ZKP_BLOB_CHALLENGE_TPB - 1) / ZKP_BLOB_CHALLENGE_TPB), ZKP_BLOB_CHALLENGE_TPB, 0, st>>>(
        blobs, proofs, proof_inf, n, zy);
    k_blob_eval<<<(unsigned)n, ZKP_BLOB_TPB, 0, st>>>(blobs, k.roots, zy);
    ctx->launches += 2;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_kzg(ctx, d, k, proofs, proof_inf, zy, n, status, (uint8_t *)scratch + blob_zy_bytes(n), err, st);
}

// ---- EIP-4844 prover: commitments by k_kzg_msm over the blobs, proofs by k_kzg_quotient then k_kzg_msm over the rows

// scratch of one batch of n proofs: the quotient rows (n x ZKP_BLOB_BYTES), then z | y (n x 64 bytes)
static size_t prove_rows_bytes(size_t n) { return align256(n * ZKP_BLOB_BYTES); }
extern "C" size_t zkp_kzg_prover_scratch_bytes(size_t n) { return prove_rows_bytes(n) + align256(n * 64); }

static cudaError_t launch_kzg_commit(zkp_ctx *ctx, const KzgDev &k, const uint8_t *blobs, size_t n, uint64_t *out, uint8_t *out_inf,
                                     uint8_t *status, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_kzg_msm<<<(unsigned)n, ZKP_MSM_TPB, 0, st>>>((const Fp *)k.lag_mem, blobs, nullptr, out, out_inf, status);
    ctx->launches++;
    return cudaGetLastError();
}

// z != NULL: compute_kzg_proof at z (n x 4), y to y_out.  z == NULL: compute_blob_kzg_proof for the commitments c
// (n x 12, flags cinf or NULL), z | y to zy (optional).
static cudaError_t launch_kzg_prove(zkp_ctx *ctx, const KzgDev &k, const uint8_t *blobs, const uint64_t *z, const uint64_t *c,
                                    const uint8_t *cinf, size_t n, uint64_t *out, uint8_t *out_inf, uint64_t *y_out, uint64_t *zy,
                                    uint8_t *status, void *scratch, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    uint8_t *rows = (uint8_t *)scratch;
    if (!zy) zy = (uint64_t *)(rows + prove_rows_bytes(n));
    const uint8_t *pre = nullptr;
    if (!z) {
        k_kzg_prove_challenge<<<(unsigned)((n + ZKP_BLOB_CHALLENGE_TPB - 1) / ZKP_BLOB_CHALLENGE_TPB), ZKP_BLOB_CHALLENGE_TPB, 0, st>>>(
            blobs, c, cinf, n, zy, status);
        ctx->launches++;
        pre = status;
    }
    k_kzg_quotient<<<(unsigned)n, ZKP_BLOB_TPB, 0, st>>>(blobs, k.roots, z, zy, y_out, rows, pre, status);
    k_kzg_msm<<<(unsigned)n, ZKP_MSM_TPB, 0, st>>>((const Fp *)k.lag_mem, rows, status, out, out_inf, status);
    ctx->launches += 2;
    return cudaGetLastError();
}

// ---- EIP-7594 cells: k_cells_extend (then k_cells_quotient and k_kzg_msm over the monomial tables for the proofs);
// verification by k_cells_interp and k_cells_prepare, then the prepared 2-pair check against G2 and -[tau^64]G2

#ifndef ZKP_CELLS_CHUNK
#define ZKP_CELLS_CHUNK (1u << 11)         // blobs per host chunk of compute_cells: 256 MiB of blobs, 512 MiB of cells per buffer set
#endif
#ifndef ZKP_CELL_PROOF_CHUNK
#define ZKP_CELL_PROOF_CHUNK (1u << 7)     // blobs per host chunk with proofs: 2 GiB of quotient rows per buffer set
#endif
#ifndef ZKP_CELLS_RECOVER_CHUNK
#define ZKP_CELLS_RECOVER_CHUNK (1u << 11) // blobs per host chunk of recovery: 512 MiB of cells in, 512 MiB out per buffer set
#endif
#ifndef ZKP_CELL_VERIFY_CHUNK
#define ZKP_CELL_VERIFY_CHUNK (1u << 16)   // cells per host chunk of verification: 128 MiB of cells per buffer set
#endif

// scratch of cells and proofs for n blobs: the coefficients (n x 4096 Fr), the quotient rows (n x 128 x ZKP_BLOB_BYTES),
// the rows' statuses (n x 128)
static size_t cells_coeff_bytes(size_t n) { return align256(n * ZKP_BLOB_N * sizeof(Fr)); }
static size_t cells_rows_bytes(size_t n) { return align256(n * ZKP_CELLS_PER_BLOB * ZKP_BLOB_BYTES); }
extern "C" size_t zkp_kzg_cells_proofs_scratch_bytes(size_t n) {
    return cells_coeff_bytes(n) + cells_rows_bytes(n) + align256(n * ZKP_CELLS_PER_BLOB);
}
// scratch of n cell checks: the point-evaluation pairs, then [I_k(tau)]G1 (n x 96 bytes) and its flags
extern "C" size_t zkp_kzg_verify_cell_scratch_bytes(size_t n) { return kzg_layout(n, nullptr, nullptr) + align256(n * 96) + align256(n); }

// the proofs of n blobs from their coefficients at the start of scratch: k_cells_quotient, then k_kzg_msm over the
// monomial tables (the launch errors are left to the caller's cudaGetLastError)
static void launch_cell_proofs(zkp_ctx *ctx, const KzgDev &k, const Fr *coeffs, size_t n, uint64_t *proofs, uint8_t *proof_inf,
                               uint8_t *status, void *scratch, cudaStream_t st) {
    uint8_t *rows = (uint8_t *)scratch + cells_coeff_bytes(n), *rst = rows + cells_rows_bytes(n);
    const size_t nt = n * ZKP_CELLS_PER_BLOB * ZKP_CELL_N;
    k_cells_quotient<<<(unsigned)((nt + ZKP_CELLS_QUOT_TPB - 1) / ZKP_CELLS_QUOT_TPB), ZKP_CELLS_QUOT_TPB, 0, st>>>(coeffs, k.pw, status, n,
                                                                                                                rows, rst);
    k_kzg_msm<<<(unsigned)(n * ZKP_CELLS_PER_BLOB), ZKP_MSM_TPB, 0, st>>>(k.mono, rows, rst, proofs, proof_inf, rst);
    ctx->launches += 2;
}

// proofs == NULL: cells only (no scratch)
static cudaError_t launch_cells(zkp_ctx *ctx, const KzgDev &k, const uint8_t *blobs, size_t n, uint8_t *cells, uint64_t *proofs,
                                uint8_t *proof_inf, uint8_t *status, void *scratch, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    Fr *coeffs = proofs ? (Fr *)scratch : nullptr;
    k_cells_extend<<<(unsigned)n, ZKP_CELLS_TPB, ZKP_BLOB_N * sizeof(Fr), st>>>(blobs, k.pw, cells, coeffs, status);
    ctx->launches++;
    if (proofs) launch_cell_proofs(ctx, k, coeffs, n, proofs, proof_inf, status, scratch, st);
    return cudaGetLastError();
}

// recover_cells (and, with proofs, as launch_cells from the recovered coefficients); proofs == NULL: cells only
static cudaError_t launch_cells_recover(zkp_ctx *ctx, const KzgDev &k, const uint64_t *idx, const uint8_t *cells, const uint64_t *num, size_t n,
                                        uint8_t *out, uint64_t *proofs, uint8_t *proof_inf, uint8_t *status, void *scratch, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    Fr *coeffs = proofs ? (Fr *)scratch : nullptr;
    k_cells_recover<<<(unsigned)(2 * n), ZKP_CELLS_TPB, ZKP_RECOVER_HALF * sizeof(Fr), st>>>(idx, cells, num, k.pw, out, coeffs, status);
    ctx->launches++;
    if (proofs) launch_cell_proofs(ctx, k, coeffs, n, proofs, proof_inf, status, scratch, st);
    return cudaGetLastError();
}

static cudaError_t launch_cells_verify(zkp_ctx *ctx, DevState &d, const KzgDev &k, const uint64_t *c, const uint8_t *cinf, const uint64_t *idx,
                                       const uint8_t *cells, const uint64_t *pi, const uint8_t *piinf, size_t n, uint8_t *status, void *scratch,
                                       uint32_t *err, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    KzgScratch s;
    uint64_t *ixy = (uint64_t *)((uint8_t *)scratch + kzg_layout(n, scratch, &s));
    uint8_t *iinf = (uint8_t *)ixy + align256(n * 96);
    k_cells_interp<<<(unsigned)n, ZKP_CELL_N, 0, st>>>(cells, idx, k.pw, k.mono, ixy, iinf, status);
    k_cells_prepare<<<grid_for(n), ZKP_TPB, 0, st>>>(c, cinf, idx, pi, piinf, k.pw, ixy, iinf, n, s.g1, s.g1inf, status);
    ctx->launches += 2;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return launch_check_verdict(ctx, d, s.g1, s.g1inf, nullptr, nullptr, n, 2, k.cell_prep, 2, s.gt, s.is_one, status, err, st);
}

// ---- multi-scalar multiplication over caller-given points: count, scan, scatter, accumulation levels, reduction, Horner
// (msm.cuh) for one batch of points, leaving one Jacobian partial on the device

#ifndef ZKP_MSM_CHUNK
#define ZKP_MSM_CHUNK (1u << 22)   // points per host chunk: 1.3 GiB (G1) / 2.1 GiB (G2) of scratch per buffer set (DESIGN.md 3.9)
#endif

// The window width for n points: msm_window's rule, or ZKPAIR_MSM_WINDOW (4 .. 20) when set, for measuring widths.
static int msm_width(size_t n) {
    const char *e = getenv("ZKPAIR_MSM_WINDOW");
    const int c = e ? atoi(e) : 0;
    return c >= 4 && c <= 20 ? c : msm_window(n);
}

struct MsmPlan {
    int c, nw, M, levels;
    size_t nb, emax, s0, s1;
};
static MsmPlan msm_plan(size_t n) {
    MsmPlan p;
    p.c = msm_width(n);
    p.nw = msm_windows(p.c);
    p.M = 1 << (p.c - 1);
    p.nb = (size_t)p.nw * p.M;
    p.emax = (size_t)p.nw * n;
    p.levels = msm_levels(p.emax);
    p.s0 = (p.emax + ZKP_MSM_SEG - 1) / ZKP_MSM_SEG;
    p.s1 = (p.s0 + ZKP_MSM_SEG - 1) / ZKP_MSM_SEG;
    return p;
}
// the largest batch one scratch holds: point indices take 31 bits and list positions 32
static bool msm_fits(size_t n) { return n < ((size_t)1 << 31) && (size_t)msm_windows(msm_width(n)) * n < ((size_t)1 << 32) - 1; }

struct MsmScratch {
    uint32_t *off_curve, *lens;   // header: the off-curve word, the levels' list lengths
    Fp *part;                     // header: the Jacobian result of the _dev forms
    Fp *pts, *buckets, *fval[2], *wsum;
    uint8_t *valid;
    uint32_t *cnt, *off, *cur, *keys, *vals, *fkey[2];
};
#define ZKP_MSM_HDR 1024   // off-curve word at 0, list lengths at 64, the Jacobian result at 256
static size_t msm_layout(size_t n, int w, void *base, MsmScratch *s) {
    const MsmPlan p = msm_plan(n);
    const size_t jb = 3 * (size_t)w * sizeof(Fp);   // bytes of one Jacobian point
    uint8_t *q[14];
    const size_t bytes = carve(base, {(size_t)ZKP_MSM_HDR, n * 2 * w * sizeof(Fp), n, p.nb * 4, (p.nb + 1) * 4, p.nb * 4, p.emax * 4,
                                      p.emax * 4, p.nb * jb, p.s0 * 4, p.s0 * jb, p.s1 * 4, p.s1 * jb, p.nw * jb}, q);
    if (s) {
        s->off_curve = (uint32_t *)q[0];
        s->lens = (uint32_t *)(q[0] + 64);
        s->part = (Fp *)(q[0] + 256);
        s->pts = (Fp *)q[1];
        s->valid = q[2];
        s->cnt = (uint32_t *)q[3];
        s->off = (uint32_t *)q[4];
        s->cur = (uint32_t *)q[5];
        s->keys = (uint32_t *)q[6];
        s->vals = (uint32_t *)q[7];
        s->buckets = (Fp *)q[8];
        s->fkey[0] = (uint32_t *)q[9];
        s->fval[0] = (Fp *)q[10];
        s->fkey[1] = (uint32_t *)q[11];
        s->fval[1] = (Fp *)q[12];
        s->wsum = (Fp *)q[13];
    }
    return bytes;
}
extern "C" size_t zkp_g1_msm_scratch_bytes(size_t n) { return msm_layout(n, 1, nullptr, nullptr); }
extern "C" size_t zkp_g2_msm_scratch_bytes(size_t n) { return msm_layout(n, 2, nullptr, nullptr); }

// sum_i [k_i]P_i over n > 0 device-resident points into the Jacobian point part; an unflagged point off the curve ORs 1
// into *off_curve (zeroed by the caller), a limb >= p 1 into *err
template <class O>
static cudaError_t launch_msm(zkp_ctx *ctx, const uint64_t *xy, const uint8_t *inf, const uint64_t *scalars, size_t n, void *scratch, Fp *part,
                              uint32_t *off_curve, uint32_t *err, cudaStream_t st) {
    const int w = MsmWidth<O>::W;
    const MsmPlan p = msm_plan(n);
    MsmScratch s;
    msm_layout(n, w, scratch, &s);
    cudaError_t e = cudaMemsetAsync(s.cnt, 0, p.nb * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(s.buckets, 0, p.nb * 3 * w * sizeof(Fp), st);   // z = 0: every bucket the identity
    if (e != cudaSuccess) return e;
    const unsigned gp = (unsigned)((n + ZKP_MSM_KTPB - 1) / ZKP_MSM_KTPB);
    k_msm_check<O><<<(unsigned)((n * w + ZKP_MSM_KTPB - 1) / ZKP_MSM_KTPB), ZKP_MSM_KTPB, 0, st>>>(xy, inf, n, s.pts, s.valid, off_curve, err);
    k_msm_digits<<<gp, ZKP_MSM_KTPB, 0, st>>>(scalars, s.valid, n, p.c, s.cnt, nullptr, nullptr);
    k_msm_scan<<<1, ZKP_MSM_SCAN_TPB, 0, st>>>(s.cnt, (uint32_t)p.nb, s.off, s.cur, s.lens);
    k_msm_digits<<<gp, ZKP_MSM_KTPB, 0, st>>>(scalars, s.valid, n, p.c, s.cur, s.keys, s.vals);
    ctx->launches += 4;
    size_t m = p.emax;   // the bound of each level's list length (the length itself is on the device)
    for (int lv = 0; lv < p.levels; lv++) {
        const size_t nseg = (m + ZKP_MSM_SEG - 1) / ZKP_MSM_SEG;
        const unsigned g = (unsigned)((nseg * w + ZKP_MSM_KTPB - 1) / ZKP_MSM_KTPB);
        const int o = lv & 1, i = o ^ 1;   // level lv writes list o and reads list i (the sorted entries at level 0)
        if (lv == 0)
            k_msm_segment<O, true><<<g, ZKP_MSM_KTPB, 0, st>>>(s.lens, s.lens + 1, s.keys, s.vals, s.pts, s.buckets, s.fkey[0], s.fval[0], nseg);
        else
            k_msm_segment<O, false><<<g, ZKP_MSM_KTPB, 0, st>>>(s.lens + lv, s.lens + lv + 1, s.fkey[i], nullptr, s.fval[i], s.buckets, s.fkey[o],
                                                                 s.fval[o], nseg);
        ctx->launches++;
        m = nseg;
    }
    const int R = p.M < ZKP_MSM_RANGES ? p.M : ZKP_MSM_RANGES;
    k_msm_reduce<O><<<(unsigned)p.nw, ZKP_MSM_RANGES * w, 0, st>>>(s.buckets, p.M, R, s.wsum);
    k_msm_combine<O><<<1, w, 0, st>>>(p.nw, p.c, s.wsum, part);
    ctx->launches += 2;
    return cudaGetLastError();
}

// Runs launch(d, st) for a device-resident entry point whose arguments passed their checks: under the context lock, on
// device dev of the context (the caller's current device is restored) and on the caller's stream (NULL = the legacy
// default stream, the CUDA convention).
template <class F> static int32_t on_device(zkp_ctx *ctx, int32_t dev, void *stream, F launch) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    DevState &d = ctx->devs[dev];
    DeviceGuard guard;
    CU(cudaSetDevice(d.id));
    return launch(d, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ host-buffer pipeline

// Split [0,n) into one contiguous slice per device.
static void slice_of(size_t n, size_t ndev, size_t d, size_t &lo, size_t &hi) {
    lo = n * d / ndev;
    hi = n * (d + 1) / ndev;
}

// The devices a call of n elements runs on, one slice_of slice each: the first alone when a slice would hold
// fewer than two elements.
static size_t fan_out(const zkp_ctx *ctx, size_t n) {
    const size_t nd = ctx->devs.size();
    return nd == 1 || n < 2 * nd ? 1 : nd;
}

// A failed CUDA call inside a host-buffer call: thrown by CUT, caught by run_slice, so that nothing after it is launched.
struct CudaFail {
    std::string msg;
};
#define CUT(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) throw CudaFail{std::string(#call) + ": " + cudaGetErrorString(e_)}; \
    } while (0)

// One chunk [c0, c0 + cn) of the slice [lo, hi) of device dev, on the stream and buffer set s.  Its copies go through
// the buffer slots B_* of that set; pageable host buffers of at least ZKP_STAGE_MIN bytes are staged through the
// set's pinned buffers (an async copy from or to pageable memory blocks the issuing thread, which would serialise
// the two sets), and the staged outputs reach the caller's buffers when the set's stream has drained.
struct Chunk {
    zkp_ctx *ctx;
    DevState &d;
    size_t dev, lo, hi, c0, cn;
    cudaStream_t st;
    int s;

    static bool pageable(const void *p) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
            cudaGetLastError();
            return true;
        }
        return a.type == cudaMemoryTypeUnregistered;
    }
    // slot with room for n elements
    template <class T> T *buf(int slot, size_t n) {
        CUT(d.buf[s][slot].ensure(n * sizeof(T)));
        return (T *)d.buf[s][slot].p;
    }
    // n elements from the host to dst (in slot's memory, or after it for B_TABINF)
    template <class T> void h2d(int slot, T *dst, const T *src, size_t n) {
        const size_t bytes = n * sizeof(T);
        if (bytes >= ZKP_STAGE_MIN && pageable(src)) {
            PinBuf &pb = d.pin_in[s][slot];
            CUT(pb.ensure(bytes));
            memcpy(pb.p, src, bytes);
            src = (const T *)pb.p;
        }
        CUT(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    }
    // elements [off, off + n) of the host buffer base in slot; NULL when base is NULL (an optional input)
    template <class T> T *in(int slot, const T *base, size_t off, size_t n) {
        if (!base) return nullptr;
        T *p = buf<T>(slot, n);
        h2d(slot, p, base + off, n);
        return p;
    }
    // n elements from the device to the host buffer dst
    template <class T> void out(int slot, T *dst, const T *src, size_t n) {
        const size_t bytes = n * sizeof(T);
        void *to = dst;
        if (bytes >= ZKP_STAGE_MIN && pageable(dst)) {
            PinBuf &pb = d.pin_out[s][slot];
            CUT(pb.ensure(bytes));
            d.pend[s].push_back(PendingOut{dst, pb.p, bytes});
            to = pb.p;
        }
        CUT(cudaMemcpyAsync(to, src, bytes, cudaMemcpyDeviceToHost, st));
    }
};
using ChunkBody = std::function<void(Chunk &)>;
using SliceFinish = std::function<void(DevState &, size_t lo, size_t hi)>;   // after the slice's streams have drained

// Runs elements [lo,hi) of a call on device dev, chunk elements at a time, on two streams and buffer sets in turn:
// the copies of one chunk overlap the kernels of the other.
static int32_t run_slice(zkp_ctx *ctx, size_t dev, size_t lo, size_t hi, size_t chunk, const ChunkBody &body, const SliceFinish &finish,
                         std::string &msg) {
    DevState &d = ctx->devs[dev];
    auto flush = [&](int set) {   // after that set's stream has drained
        for (const PendingOut &o : d.pend[set]) memcpy(o.user, o.stage, o.bytes);
        d.pend[set].clear();
    };
    try {
        DeviceGuard guard;
        CUT(cudaSetDevice(d.id));
        CUT(cudaMemsetAsync(d.d_err, 0, sizeof(uint32_t), d.stream[0]));
        CUT(cudaStreamSynchronize(d.stream[0]));
        d.pend[0].clear();   // (a call that failed half-way leaves nothing behind for the next one)
        d.pend[1].clear();
        int s = 0;
        for (size_t c0 = lo; c0 < hi; c0 += chunk, s ^= 1) {
            Chunk c{ctx, d, dev, lo, hi, c0, hi - c0 < chunk ? hi - c0 : chunk, d.stream[s], s};
            CUT(cudaStreamSynchronize(c.st));   // this buffer set's previous chunk is fully drained
            flush(s);
            body(c);
        }
        CUT(cudaStreamSynchronize(d.stream[0]));
        flush(0);
        CUT(cudaStreamSynchronize(d.stream[1]));
        flush(1);
        if (finish) finish(d, lo, hi);
        uint32_t herr = 0;
        CUT(cudaMemcpy(&herr, d.d_err, sizeof herr, cudaMemcpyDeviceToHost));
        if (herr & 1) {
            msg = "input limb vector >= p (non-canonical field element)";
            return ZKP_ERR_NONCANONICAL;
        }
        return ZKP_OK;
    } catch (const CudaFail &f) {
        msg = f.msg;
        return ZKP_ERR_CUDA;
    }
}

// Runs [0,n) over the fan_out devices, one thread per device; the first failing device's error is returned.
// The caller holds ctx->mu.
static int32_t run_slices(zkp_ctx *ctx, size_t n, size_t chunk, const ChunkBody &body, const SliceFinish &finish = nullptr) {
    const size_t nd = fan_out(ctx, n);
    std::vector<int32_t> rcs(nd, ZKP_OK);
    std::vector<std::string> msgs(nd);
    auto run = [&](size_t di) {
        size_t lo, hi;
        slice_of(n, nd, di, lo, hi);
        rcs[di] = run_slice(ctx, di, lo, hi, chunk, body, finish, msgs[di]);
    };
    if (nd == 1) {
        run(0);
    } else {
        std::vector<std::thread> th;
        for (size_t di = 0; di < nd; di++) th.emplace_back(run, di);
        for (auto &t : th) t.join();
    }
    for (size_t di = 0; di < nd; di++)
        if (rcs[di] != ZKP_OK) return fail(rcs[di], msgs[di]);
    return ZKP_OK;
}

static int32_t run_host_job(zkp_ctx *ctx, size_t n, size_t chunk, const ChunkBody &body) {
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (n == 0) return ZKP_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    return run_slices(ctx, n, chunk, body);
}

// One MSM over host buffers, in the shape of zkp_multi_miller_product: each device sums its slice chunk by chunk into
// Jacobian partials in d.partial (followed by the device's off-curve word), its finish step folds them into the slot
// after the last one, and the first device gathers one partial per device by peer copy, adds them and converts the sum
// to affine.
template <class O>
static int32_t msm_job(zkp_ctx *ctx, const uint64_t *xy, const uint8_t *inf, const uint64_t *scalars, size_t n, uint64_t *out_xy,
                       uint8_t *out_inf, uint8_t *out_status) {
    const int w = MsmWidth<O>::W;
    const size_t pw = MsmWidth<O>::U64, jb = 3 * w * sizeof(Fp);
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (!out_xy || !out_inf || !out_status || (n && (!xy || !scalars))) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (n == 0) {   // the identity (0, 1)
        memset(out_xy, 0, pw * sizeof(uint64_t));
        out_xy[pw / 2] = 1;
        *out_inf = 1;
        *out_status = ZKP_POINT_OK;
        return ZKP_OK;
    }
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard guard;
    const size_t chunk = ZKP_MSM_CHUNK;
    auto nchunks = [=](size_t lo, size_t hi) { return (hi - lo + chunk - 1) / chunk; };
    auto body = [=](Chunk &c) {
        DevState &d = c.d;
        const size_t nc = nchunks(c.lo, c.hi);
        if (c.c0 == c.lo) {   // the partials, their fold and the off-curve word, zeroed before any chunk runs
            CUT(d.partial.ensure((nc + 1) * jb + sizeof(uint32_t)));
            CUT(cudaMemsetAsync((uint8_t *)d.partial.p + (nc + 1) * jb, 0, sizeof(uint32_t), c.st));
            CUT(cudaStreamSynchronize(c.st));
        }
        const size_t ci = (c.c0 - c.lo) / chunk;
        const uint64_t *dxy = c.in(B_G1, xy, c.c0 * pw, c.cn * pw), *dsc = c.in(B_IN, scalars, c.c0 * 4, c.cn * 4);
        const uint8_t *dinf = c.in(B_G1INF, inf, c.c0, c.cn);
        void *scratch = c.buf<uint8_t>(B_TAB, msm_layout(c.cn, w, nullptr, nullptr));
        CUT(launch_msm<O>(ctx, dxy, dinf, dsc, c.cn, scratch, (Fp *)((uint8_t *)d.partial.p + ci * jb),
                          (uint32_t *)((uint8_t *)d.partial.p + (nc + 1) * jb), d.d_err, c.st));
    };
    auto fold = [=](DevState &d, size_t lo, size_t hi) {
        const size_t nc = nchunks(lo, hi);
        k_msm_sum<O><<<1, w, 0, d.stream[0]>>>((const Fp *)d.partial.p, (int)nc, (Fp *)((uint8_t *)d.partial.p + nc * jb));
        ctx->launches++;
        CUT(cudaGetLastError());
        CUT(cudaStreamSynchronize(d.stream[0]));
    };
    int32_t rc = run_slices(ctx, n, chunk, body, fold);
    if (rc != ZKP_OK) return rc;
    // gather: one partial and one off-curve word per device -> first device (peer copy over NVLink when available)
    const size_t nd = fan_out(ctx, n);
    DevState &d0 = ctx->devs[0];
    CU(cudaSetDevice(d0.id));
    DevBuf &G = d0.buf[1][B_IN];
    const size_t offs = align256(nd * jb), res = offs + align256(nd * 4);   // partials | off-curve words | x|y, flag, status
    CU(G.ensure(res + pw * sizeof(uint64_t) + 2));
    uint8_t *g = (uint8_t *)G.p;
    for (size_t di = 0; di < nd; di++) {
        DevState &d = ctx->devs[di];
        size_t lo, hi;
        slice_of(n, nd, di, lo, hi);
        const size_t nc = nchunks(lo, hi);
        const uint8_t *src = (const uint8_t *)d.partial.p;
        if (d.id == d0.id) {
            CU(cudaMemcpyAsync(g + di * jb, src + nc * jb, jb, cudaMemcpyDeviceToDevice, d0.stream[0]));
            CU(cudaMemcpyAsync(g + offs + 4 * di, src + (nc + 1) * jb, 4, cudaMemcpyDeviceToDevice, d0.stream[0]));
        } else {
            CU(cudaMemcpyPeerAsync(g + di * jb, d0.id, src + nc * jb, d.id, jb, d0.stream[0]));
            CU(cudaMemcpyPeerAsync(g + offs + 4 * di, d0.id, src + (nc + 1) * jb, d.id, 4, d0.stream[0]));
        }
    }
    uint64_t *rxy = (uint64_t *)(g + res);
    uint8_t *rflag = g + res + pw * sizeof(uint64_t);
    k_msm_final<O><<<1, w, 0, d0.stream[0]>>>((const Fp *)g, (int)nd, (const uint32_t *)(g + offs), (int)nd, rxy, rflag, rflag + 1);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out_xy, rxy, pw * sizeof(uint64_t), cudaMemcpyDeviceToHost, d0.stream[0]));
    CU(cudaMemcpyAsync(out_inf, rflag, 1, cudaMemcpyDeviceToHost, d0.stream[0]));
    CU(cudaMemcpyAsync(out_status, rflag + 1, 1, cudaMemcpyDeviceToHost, d0.stream[0]));
    CU(cudaStreamSynchronize(d0.stream[0]));
    return ZKP_OK;
}

// The _dev forms: the whole batch in one launch sequence on the caller's stream, the partial and the off-curve word in
// the scratch header.
template <class O>
static int32_t msm_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *xy, const uint8_t *inf, const uint64_t *scalars, size_t n, uint64_t *out_xy,
                       uint8_t *out_inf, uint8_t *status, uint32_t *err, void *scratch, void *stream) {
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (dev < 0 || dev >= (int)ctx->devs.size()) return fail(ZKP_ERR_INVALID_ARG, "device index out of range");
    if (!out_xy || !out_inf || !status || !scratch || (n && (!xy || !scalars))) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if ((uintptr_t)scratch & 15) return fail(ZKP_ERR_INVALID_ARG, "d_scratch is not 16-byte aligned");
    if (!msm_fits(n)) return fail(ZKP_ERR_INVALID_ARG, "n too large for one device-resident MSM");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        (void)d;
        MsmScratch s;
        msm_layout(n, MsmWidth<O>::W, scratch, &s);
        CU(cudaMemsetAsync(scratch, 0, ZKP_MSM_HDR, st));   // off-curve word 0, result the identity
        if (n) CU(launch_msm<O>(ctx, xy, inf, scalars, n, scratch, s.part, s.off_curve, err, st));
        k_msm_final<O><<<1, MsmWidth<O>::W, 0, st>>>(s.part, 1, s.off_curve, 1, out_xy, out_inf, status);
        ctx->launches++;
        CU(cudaGetLastError());
        return ZKP_OK;
    });
}

extern "C" {

const char *zkp_last_error(void) { return g_err.c_str(); }

extern "C" void zkp_miller_geometry(int *tpb, int *blocks, int *sync);   // pairing_kernel.cu
extern "C" void zkp_fe_geometry(int *tpb, int *blocks, int *sync);       // fe_kernel.cu
const char *zkp_version(void) {
    static char buf[224];
    int mt, mb, ms, ft, fb, fs;
    zkp_miller_geometry(&mt, &mb, &ms);
    zkp_fe_geometry(&ft, &fb, &fs);
    snprintf(buf, sizeof buf, "zkpair 0.3 (sm_100a, 2 lanes/pairing, 12x32 CIOS; miller %dx%d/SM sync %d, final exp %dx%d/SM sync %d, chunk=%u)",
             mt, mb, ms, ft, fb, fs, (unsigned)ZKP_CHUNK);
    return buf;
}

int32_t zkp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int32_t zkp_ctx_create(const int *devices, int n_devices, zkp_ctx **out) {
    if (!out) return fail(ZKP_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    int avail = zkp_device_count();
    if (avail <= 0) return fail(ZKP_ERR_NO_DEVICE, "no CUDA device available (libzkpair has no CPU path)");
    std::vector<int> ids;
    if (!devices || n_devices <= 0) {
        for (int i = 0; i < avail; i++) ids.push_back(i);
    } else {
        for (int i = 0; i < n_devices; i++) {
            if (devices[i] < 0 || devices[i] >= avail) return fail(ZKP_ERR_INVALID_ARG, "device index out of range");
            ids.push_back(devices[i]);
        }
    }
    DeviceGuard guard;
    zkp_ctx *c = new zkp_ctx();
    c->devs.resize(ids.size());
    for (size_t i = 0; i < ids.size(); i++) {
        DevState &d = c->devs[i];
        d.id = ids[i];
        cudaError_t e = cudaSetDevice(d.id);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d.stream[0], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d.stream[1], cudaStreamNonBlocking);
        for (int a = 0; a < 3 && e == cudaSuccess; a++) {
            e = cudaStreamCreateWithFlags(&d.fe_aux[a].s2, cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.fe_aux[a].fork, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.fe_aux[a].join, cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaMalloc(&d.d_err, 4 * sizeof(uint32_t));   // [0] error flag, [1] zero word read by the probes
        if (e == cudaSuccess) e = cudaMemset(d.d_err, 0, 4 * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, d.id);
        if (e == cudaSuccess) {
            // a private pool whose memory is never handed back at synchronisation points: the scratch
            // of one launch is reused by the next instead of being re-allocated (1.1 GB at 2^20)
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = d.id;
            e = cudaMemPoolCreate(&d.pool, &props);
            uint64_t keep = ~0ull;
            if (e == cudaSuccess) e = cudaMemPoolSetAttribute(d.pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        if (e != cudaSuccess) {
            std::string msg = std::string("device init failed: ") + cudaGetErrorString(e);
            zkp_ctx_destroy(c);
            return fail(ZKP_ERR_CUDA, msg);
        }
    }
    *out = c;
    return ZKP_OK;
}

void zkp_ctx_destroy(zkp_ctx *ctx) {
    if (!ctx) return;
    DeviceGuard guard;
    for (DevState &d : ctx->devs) {
        cudaSetDevice(d.id);
        cudaDeviceSynchronize();
        for (int a = 0; a < 3; a++) {
            if (d.fe_aux[a].fork) cudaEventDestroy(d.fe_aux[a].fork);
            if (d.fe_aux[a].join) cudaEventDestroy(d.fe_aux[a].join);
            if (d.fe_aux[a].s2) cudaStreamDestroy(d.fe_aux[a].s2);
        }
        for (auto &t : d.timers) {
            cudaEventDestroy(t.first);
            cudaEventDestroy(t.second);
        }
        for (int s = 0; s < 2; s++) {
            for (int b = 0; b < B_NBUF; b++) d.buf[s][b].release();
            for (int b = 0; b < B_NPIN; b++) {
                d.pin_in[s][b].release();
                d.pin_out[s][b].release();
            }
            if (d.stream[s]) cudaStreamDestroy(d.stream[s]);
        }
        d.scratch.release();
        d.partial.release();
        if (d.d_err) cudaFree(d.d_err);
        if (d.pool) {
            cudaDeviceSynchronize();
            cudaMemPoolDestroy(d.pool);
        }
    }
    delete ctx;
}

int32_t zkp_ctx_num_devices(const zkp_ctx *ctx) { return ctx ? (int32_t)ctx->devs.size() : 0; }
uint64_t zkp_launch_count(const zkp_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

int32_t zkp_set_kernel_timing(zkp_ctx *ctx, int32_t enabled) {
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->timing = enabled != 0;
    return ZKP_OK;
}

int32_t zkp_last_kernel_ms(zkp_ctx *ctx, int32_t dev, double *total_ms, uint64_t *launches) {
    if (!ctx || dev < 0 || dev >= (int)ctx->devs.size()) return fail(ZKP_ERR_INVALID_ARG, "bad ctx/dev");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DevState &d = ctx->devs[dev];
    DeviceGuard guard;
    CU(cudaSetDevice(d.id));
    for (auto &t : d.timers) {
        CU(cudaEventSynchronize(t.second));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, t.first, t.second));
        d.timed_ms += ms;
        d.timed_launches++;
        cudaEventDestroy(t.first);
        cudaEventDestroy(t.second);
    }
    d.timers.clear();
    if (total_ms) *total_ms = d.timed_ms;
    if (launches) *launches = d.timed_launches;
    d.timed_ms = 0;
    d.timed_launches = 0;
    return ZKP_OK;
}

// ------------------------------------------------------------------ device-resident entry points

static int32_t check_dev(zkp_ctx *ctx, int32_t dev) {
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (dev < 0 || dev >= (int)ctx->devs.size()) return fail(ZKP_ERR_INVALID_ARG, "device index out of range");
    return ZKP_OK;
}

int32_t zkp_pairing_dev(zkp_ctx *ctx, int32_t dev, int32_t mode, const uint64_t *d_g1_xy, const uint8_t *d_g1_inf,
                        const uint64_t *d_g2_xy, const uint8_t *d_g2_inf, size_t n_checks, int32_t pairs_per_check,
                        const uint64_t *d_in_fp12, uint64_t *d_out, uint8_t *d_is_one, uint32_t *d_err, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (!(mode == 1 || mode == 2 || mode == 3 || mode == 5) || !d_out) return fail(ZKP_ERR_INVALID_ARG, "bad mode / NULL output");
    if ((mode & 1) && (!d_g1_xy || !d_g2_xy || pairs_per_check < 1)) return fail(ZKP_ERR_INVALID_ARG, "NULL point buffers");
    if (!(mode & 1) && !d_in_fp12) return fail(ZKP_ERR_INVALID_ARG, "NULL Fp12 input");
    if (pairs_per_check > ZKP_MAX_PAIRS_PER_CHECK) return fail(ZKP_ERR_TOO_MANY_PAIRS, "pairs_per_check > 8");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_pairing(ctx, d, mode, d_g1_xy, d_g1_inf, d_g2_xy, d_g2_inf, n_checks, (mode & 1) ? pairs_per_check : 1,
                          d_in_fp12, d_out, d_is_one, d_err, st));
        return ZKP_OK;
    });
}

int32_t zkp_tower_op_dev(zkp_ctx *ctx, int32_t dev, int32_t op, const uint64_t *d_a, const uint64_t *d_b, uint64_t *d_out,
                         uint8_t *d_status, uint32_t *d_err, size_t n, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    int na, nb, nr;
    tower_op_shape(op, na, nb, nr);
    if (!d_a || !d_out || (nb && !d_b)) return fail(ZKP_ERR_INVALID_ARG, "NULL operand");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        if (n) {
            k_tower_op<<<grid_for(n), ZKP_TPB, 0, st>>>(op, d_a, d_b, d_out, d_status, d_err, n);
            ctx->launches++;
            CU(cudaGetLastError());
        }
        return ZKP_OK;
    });
}

int32_t zkp_fp12_product_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_in, size_t n, uint64_t *d_scratch,
                             uint64_t *d_out, uint32_t *d_err, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (!d_in || !d_out || !d_scratch || n == 0) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer or n == 0");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_product(ctx, d_in, n, d_scratch, d_out, d_err, st));
        return ZKP_OK;
    });
}

int32_t zkp_gen_points_dev(zkp_ctx *ctx, int32_t dev, uint64_t seed, uint64_t first, size_t n, uint64_t *d_g1_xy,
                           uint8_t *d_g1_inf, uint64_t *d_g2_xy, uint8_t *d_g2_inf, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (!d_g1_xy || !d_g1_inf || !d_g2_xy || !d_g2_inf) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        if (n) {
            k_gen_points<<<grid_for(n), ZKP_TPB, 0, st>>>(seed, first, n, d_g1_xy, d_g1_inf, d_g2_xy, d_g2_inf);
            ctx->launches++;
            CU(cudaGetLastError());
        }
        return ZKP_OK;
    });
}

// ------------------------------------------------------------------ host-buffer entry points

int32_t zkp_tower_op_batch(zkp_ctx *ctx, int32_t op, const uint64_t *a, const uint64_t *b, uint64_t *out, uint8_t *status, size_t n) {
    int na, nb, nr;
    tower_op_shape(op, na, nb, nr);
    bool known = (op >= 0 && op <= OP_FP_SQRT) || (op >= OP_FP2_ADD && op <= OP_FP2_POW) || (op >= OP_FP6_ADD && op <= OP_FP6_MUL_BY_01) ||
                 (op >= OP_FP12_ADD && op <= OP_FP12_POW);
    if (!known) return fail(ZKP_ERR_INVALID_ARG, "unknown tower op");
    if (n && (!a || !out || (nb && !b))) return fail(ZKP_ERR_INVALID_ARG, "NULL operand");
    return run_host_job(ctx, n, ZKP_CHUNK, [=](Chunk &c) {
        const uint64_t *da = c.in(B_IN, a, c.c0 * na * 6, c.cn * na * 6);
        uint64_t *dout = c.buf<uint64_t>(B_OUT, c.cn * nr * 6);
        uint8_t *dst = c.buf<uint8_t>(B_FLAG, c.cn);
        const uint64_t *db = c.in(B_G2, nb ? b : nullptr, c.c0 * nb * 6, c.cn * nb * 6);
        k_tower_op<<<grid_for(c.cn), ZKP_TPB, 0, c.st>>>(op, da, db, dout, dst, c.d.d_err, c.cn);
        ctx->launches++;
        CUT(cudaGetLastError());
        c.out(B_OUT, out + c.c0 * nr * 6, dout, c.cn * nr * 6);
        if (status) c.out(B_FLAG, status + c.c0, dst, c.cn);
    });
}
int32_t zkp_fp_mul_batch(zkp_ctx *ctx, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n) {
    return zkp_tower_op_batch(ctx, OP_FP_MUL, a, b, out, nullptr, n);
}
// The reference's zkVM precompile FFI, one Fp operation per call (src/fp.rs:126,376,443).  The precompiles carry no
// handle: ctx = NULL selects a process-wide context on device 0 created on first use (never destroyed).
static zkp_ctx *default_ctx(int32_t &rc) {
    static std::mutex mu;
    static zkp_ctx *ctx = nullptr;
    std::lock_guard<std::mutex> lk(mu);
    rc = ZKP_OK;
    if (!ctx) {
        int dev0 = 0;
        rc = zkp_ctx_create(&dev0, 1, &ctx);
        if (rc != ZKP_OK) ctx = nullptr;
    }
    return ctx;
}
int32_t zkp_sys_bigint(zkp_ctx *ctx, uint32_t *result, uint32_t op, const uint32_t *lhs, const uint32_t *rhs) {
    if (!result || !lhs || !rhs) return fail(ZKP_ERR_INVALID_ARG, "NULL limb pointer");
    if (op > 1) return fail(ZKP_ERR_INVALID_ARG, "op must be 0 (mul) or 1 (add)");
    if (!ctx) {
        int32_t rc;
        ctx = default_ctx(rc);
        if (!ctx) return rc;
    }
    // twelve u32 limbs = the little-endian [u64; 6] of src/fp.rs:24 (the crate transmutes, src/fp.rs:124-128)
    uint64_t a[6], b[6], o[6];
    memcpy(a, lhs, sizeof a);
    memcpy(b, rhs, sizeof b);
    int32_t rc = zkp_tower_op_batch(ctx, op == 0 ? OP_FP_MUL : OP_FP_ADD, a, b, o, nullptr, 1);
    if (rc == ZKP_OK) memcpy(result, o, sizeof o);
    return rc;
}
int32_t zkp_syscall_fp_mulmod(zkp_ctx *ctx, uint32_t *lhs, const uint32_t *rhs) { return zkp_sys_bigint(ctx, lhs, 0, lhs, rhs); }
int32_t zkp_fp12_mul_batch(zkp_ctx *ctx, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n) {
    return zkp_tower_op_batch(ctx, OP_FP12_MUL, a, b, out, nullptr, n);
}
int32_t zkp_fp12_mul_by_014_batch(zkp_ctx *ctx, const uint64_t *f, const uint64_t *c, uint64_t *out, size_t n) {
    return zkp_tower_op_batch(ctx, OP_FP12_MUL_BY_014, f, c, out, nullptr, n);
}

// launch_pairing over host buffers: mode 1 (Miller loops) or 3 (pairings) of n checks of k pairs, the last kf of
// each check from the kf shared prepared tables (flags tabinf), or mode 2 (final exponentiations of in12)
static int32_t pairs_job(zkp_ctx *ctx, int mode, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                         const uint64_t *in12, size_t n, int k, uint64_t *out, uint8_t *flags, const uint64_t *tab = nullptr,
                         const uint8_t *tabinf = nullptr, int kf = 0) {
    return run_host_job(ctx, n, ZKP_CHUNK, [=](Chunk &c) {
        const size_t np = c.cn * (size_t)k, p0 = c.c0 * (size_t)k;
        const size_t nq = c.cn * (size_t)(k - kf), q0 = c.c0 * (size_t)(k - kf);   // per-check G2 points
        const uint64_t *dg1 = nullptr, *dg2 = nullptr, *din = nullptr;
        const uint8_t *di1 = nullptr, *di2 = nullptr, *dti = nullptr;
        const uint8_t *dtab = nullptr;
        if (mode & 1) {
            dg1 = c.in(B_G1, g1, p0 * 12, np * 12);
            uint64_t *p2 = c.buf<uint64_t>(B_G2, nq * 24 + 2);
            if (nq) c.h2d(B_G2, p2, g2 + q0 * 24, nq * 24);
            dg2 = p2;
            if (kf) {
                const size_t tb = (size_t)kf * ZKP_LINE_STEPS * 3 * 2 * sizeof(Fp);
                uint8_t *t = c.buf<uint8_t>(B_TAB, tb + 16);
                c.h2d(B_TAB, t, (const uint8_t *)tab, tb);
                if (tabinf) {
                    c.h2d(B_TABINF, t + tb, tabinf, (size_t)kf);
                    dti = t + tb;
                }
                dtab = t;
            }
            di1 = c.in(B_G1INF, g1inf, p0, np);
            di2 = c.in(B_G2INF, nq ? g2inf : nullptr, q0, nq);
        } else {
            din = c.in(B_IN, in12, c.c0 * 72, c.cn * 72);
        }
        uint64_t *dout = c.buf<uint64_t>(B_OUT, c.cn * 72);
        uint8_t *dflag = flags ? c.buf<uint8_t>(B_FLAG, c.cn) : nullptr;
        CUT(launch_pairing(ctx, c.d, mode, dg1, di1, dg2, di2, c.cn, k, din, dout, dflag, c.d.d_err, c.st, dtab, dti, kf));
        c.out(B_OUT, out + c.c0 * 72, dout, c.cn * 72);
        if (flags) c.out(B_FLAG, flags + c.c0, dflag, c.cn);
    });
}
static int32_t checks_job(zkp_ctx *ctx, int mode, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                          size_t n, int32_t k, uint64_t *out, uint8_t *flags) {
    if (k < 1) return fail(ZKP_ERR_INVALID_ARG, "pairs_per_check < 1");
    if (k > ZKP_MAX_PAIRS_PER_CHECK) return fail(ZKP_ERR_TOO_MANY_PAIRS, "pairs_per_check > 8 (use zkp_multi_miller_product)");
    if (n && (!g1 || !g2 || !out)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return pairs_job(ctx, mode, g1, g1inf, g2, g2inf, nullptr, n, k, out, flags);
}
int32_t zkp_miller_loop_batch(zkp_ctx *ctx, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf, size_t n, uint64_t *out) {
    return checks_job(ctx, 1, g1, g1inf, g2, g2inf, n, 1, out, nullptr);
}
int32_t zkp_pairing_batch(zkp_ctx *ctx, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf, size_t n, uint64_t *out) {
    return checks_job(ctx, 3, g1, g1inf, g2, g2inf, n, 1, out, nullptr);
}
int32_t zkp_multi_miller_loop_batch(zkp_ctx *ctx, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                                    size_t n_checks, int32_t k, uint64_t *out) {
    return checks_job(ctx, 1, g1, g1inf, g2, g2inf, n_checks, k, out, nullptr);
}
int32_t zkp_multi_pairing_batch(zkp_ctx *ctx, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                                size_t n_checks, int32_t k, uint64_t *out, uint8_t *is_one) {
    return checks_job(ctx, 3, g1, g1inf, g2, g2inf, n_checks, k, out, is_one);
}
int32_t zkp_final_exp_batch(zkp_ctx *ctx, const uint64_t *in, size_t n, uint64_t *out) {
    if (n && (!in || !out)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return pairs_job(ctx, 2, nullptr, nullptr, nullptr, nullptr, in, n, 1, out, nullptr);
}
int32_t zkp_gen_points(zkp_ctx *ctx, uint64_t seed, uint64_t first, size_t n, uint64_t *g1, uint8_t *g1inf, uint64_t *g2, uint8_t *g2inf) {
    if (n && (!g1 || !g1inf || !g2 || !g2inf)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return run_host_job(ctx, n, ZKP_CHUNK, [=](Chunk &c) {
        uint64_t *d1 = c.buf<uint64_t>(B_G1, c.cn * 12), *d2 = c.buf<uint64_t>(B_G2, c.cn * 24);
        uint8_t *d1i = c.buf<uint8_t>(B_G1INF, c.cn), *d2i = c.buf<uint8_t>(B_G2INF, c.cn);
        k_gen_points<<<grid_for(c.cn), ZKP_TPB, 0, c.st>>>(seed, first + c.c0, c.cn, d1, d1i, d2, d2i);
        ctx->launches++;
        CUT(cudaGetLastError());
        c.out(B_G1, g1 + c.c0 * 12, d1, c.cn * 12);
        c.out(B_G2, g2 + c.c0 * 24, d2, c.cn * 24);
        c.out(B_G1INF, g1inf + c.c0, d1i, c.cn);
        c.out(B_G2INF, g2inf + c.c0, d2i, c.cn);
    });
}

// ---- prepared G2 points (SURVEY 8f-4)
int32_t zkp_g2_prepare_batch(zkp_ctx *ctx, const uint64_t *g2_xy, size_t n, uint64_t *out_tables) {
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (n == 0) return ZKP_OK;
    if (!g2_xy || !out_tables) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DevState &d = ctx->devs[0];   // a handful of verifying-key points: one device
    DeviceGuard guard;
    CU(cudaSetDevice(d.id));
    cudaStream_t st = d.stream[0];
    DevBuf *B = d.buf[0];
    const size_t tb = (size_t)ZKP_G2_PREPARED_U64 * 8;
    CU(cudaMemsetAsync(d.d_err, 0, sizeof(uint32_t), st));
    CU(B[B_G2].ensure(n * 192));
    CU(B[B_TAB].ensure(n * tb + 16));
    CU(cudaMemcpyAsync(B[B_G2].p, g2_xy, n * 192, cudaMemcpyHostToDevice, st));
    k_g2_prepare<<<grid_for(n), ZKP_TPB, 0, st>>>((const uint64_t *)B[B_G2].p, (Fp *)B[B_TAB].p, d.d_err, n);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out_tables, B[B_TAB].p, n * tb, cudaMemcpyDeviceToHost, st));
    uint32_t herr = 0;
    CU(cudaMemcpyAsync(&herr, d.d_err, sizeof herr, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (herr & 1) return fail(ZKP_ERR_NONCANONICAL, "input limb vector >= p (non-canonical field element)");
    return ZKP_OK;
}
int32_t zkp_g2_prepare_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g2_xy, size_t n, uint64_t *d_out_tables, uint32_t *d_err, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (n && (!d_g2_xy || !d_out_tables)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        if (n) {
            k_g2_prepare<<<grid_for(n), ZKP_TPB, 0, st>>>(d_g2_xy, (Fp *)d_out_tables, d_err, n);
            ctx->launches++;
            CU(cudaGetLastError());
        }
        return ZKP_OK;
    });
}
int32_t zkp_multi_pairing_prepared_batch(zkp_ctx *ctx, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                                         size_t n_checks, int32_t k, const uint64_t *tables, const uint8_t *tables_inf, int32_t kf,
                                         uint64_t *out, uint8_t *is_one) {
    if (k < 1 || kf < 0 || kf > k) return fail(ZKP_ERR_INVALID_ARG, "need 0 <= prepared pairs <= pairs_per_check");
    if (k > ZKP_MAX_PAIRS_PER_CHECK) return fail(ZKP_ERR_TOO_MANY_PAIRS, "pairs_per_check > 8");
    if (n_checks && (!g1 || !out || (kf < k && !g2) || (kf && !tables))) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return pairs_job(ctx, 3, g1, g1inf, g2, g2inf, nullptr, n_checks, k, out, is_one, tables, tables_inf, kf);
}
int32_t zkp_multi_pairing_prepared_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g1, const uint8_t *d_g1inf, const uint64_t *d_g2,
                                       const uint8_t *d_g2inf, size_t n_checks, int32_t k, const uint64_t *d_tables,
                                       const uint8_t *d_tables_inf, int32_t kf, uint64_t *d_out, uint8_t *d_is_one, uint32_t *d_err,
                                       void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (k < 1 || kf < 0 || kf > k || k > ZKP_MAX_PAIRS_PER_CHECK) return fail(ZKP_ERR_INVALID_ARG, "bad pairs_per_check / prepared count");
    if (!d_g1 || !d_out || (kf < k && !d_g2) || (kf && !d_tables)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_pairing(ctx, d, 3, d_g1, d_g1inf, d_g2, d_g2inf, n_checks, k, nullptr, d_out, d_is_one, d_err, st, d_tables, d_tables_inf, kf));
        return ZKP_OK;
    });
}

// bytes <-> limbs on device-resident buffers (dir 0: from_bytes, 1: to_bytes)
int32_t zkp_fp_bytes_dev(zkp_ctx *ctx, int32_t dev, int32_t dir, const void *d_in, void *d_out, uint8_t *d_ok, size_t n, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (n && (!d_in || !d_out)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_in | (uintptr_t)d_out) & 15) return fail(ZKP_ERR_INVALID_ARG, "buffers must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        if (n) {
            k_fp_bytes<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dir, (const uint4 *)d_in, (uint4 *)d_out, d_ok, n);
            ctx->launches++;
            CU(cudaGetLastError());
        }
        return ZKP_OK;
    });
}
static int32_t bytes_job(zkp_ctx *ctx, int dir, const void *in, void *out, uint8_t *ok, size_t n) {
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (n == 0) return ZKP_OK;
    if (!in || !out) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DevState &d = ctx->devs[0];   // HBM-bound byte shuffling: one device is already PCIe-limited
    DeviceGuard guard;
    CU(cudaSetDevice(d.id));
    cudaStream_t st = d.stream[0];
    DevBuf *B = d.buf[0];
    const size_t chunk = (size_t)ZKP_CHUNK * 8;
    for (size_t c0 = 0; c0 < n; c0 += chunk) {
        size_t cn = n - c0 < chunk ? n - c0 : chunk;
        CU(B[B_IN].ensure(cn * 48));
        CU(B[B_OUT].ensure(cn * 48));
        CU(B[B_FLAG].ensure(cn));
        CU(cudaMemcpyAsync(B[B_IN].p, (const uint8_t *)in + c0 * 48, cn * 48, cudaMemcpyHostToDevice, st));
        k_fp_bytes<<<(unsigned)((cn + 255) / 256), 256, 0, st>>>(dir, (const uint4 *)B[B_IN].p, (uint4 *)B[B_OUT].p,
                                                                  ok ? (uint8_t *)B[B_FLAG].p : nullptr, cn);
        ctx->launches++;
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync((uint8_t *)out + c0 * 48, B[B_OUT].p, cn * 48, cudaMemcpyDeviceToHost, st));
        if (ok && dir == 0) CU(cudaMemcpyAsync(ok + c0, B[B_FLAG].p, cn, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return ZKP_OK;
}
int32_t zkp_fp_from_bytes_batch(zkp_ctx *ctx, const uint8_t *bytes, size_t n, uint64_t *out_limbs, uint8_t *ok) {
    return bytes_job(ctx, 0, bytes, out_limbs, ok, n);
}
int32_t zkp_fp_to_bytes_batch(zkp_ctx *ctx, const uint64_t *limbs, size_t n, uint8_t *out_bytes) {
    return bytes_job(ctx, 1, limbs, out_bytes, nullptr, n);
}

static int32_t group_job(zkp_ctx *ctx, int gop, const uint64_t *pts, const uint8_t *inf, const uint64_t *scalars, size_t n,
                         uint64_t *out, uint8_t *flags, const uint8_t *inf2 = nullptr) {
    if (n && (!pts || !flags || (gop >= GOP_G1_MUL && (!scalars || !out)))) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    const size_t w = (gop & 1) ? 24 : 12;
    const bool is_mul = gop >= GOP_G1_MUL;   // has a second operand and an output point
    const bool is_add = gop >= GOP_G1_ADD;
    const size_t w2 = is_add ? w : 4;        // u64 per element of the second operand
    return run_host_job(ctx, n, ZKP_CHUNK, [=](Chunk &c) {
        const uint64_t *dp = c.in(B_IN, pts, c.c0 * w, c.cn * w);
        uint8_t *dflag = c.buf<uint8_t>(B_FLAG, c.cn);
        const uint8_t *dinf = c.in(B_G1INF, inf, c.c0, c.cn);
        const uint8_t *dinf2 = c.in(B_G2INF, is_add ? inf2 : nullptr, c.c0, c.cn);
        const uint64_t *dsc = nullptr;
        uint64_t *dout = nullptr;
        if (is_mul) {
            dsc = c.in(B_G2, scalars, c.c0 * w2, c.cn * w2);
            dout = c.buf<uint64_t>(B_OUT, c.cn * w);
        }
        k_group_op<<<grid_for(c.cn), ZKP_TPB, 0, c.st>>>(gop, dp, dinf, dsc, dout, dflag, c.d.d_err, c.cn, dinf2);
        ctx->launches++;
        CUT(cudaGetLastError());
        if (is_mul) c.out(B_OUT, out + c.c0 * w, dout, c.cn * w);
        c.out(B_FLAG, flags + c.c0, dflag, c.cn);
    });
}
int32_t zkp_g1_add_batch(zkp_ctx *ctx, const uint64_t *a_xy, const uint8_t *a_inf, const uint64_t *b_xy, const uint8_t *b_inf, size_t n,
                         uint64_t *out_xy, uint8_t *out_flag) {
    return group_job(ctx, GOP_G1_ADD, a_xy, a_inf, b_xy, n, out_xy, out_flag, b_inf);
}
int32_t zkp_g2_add_batch(zkp_ctx *ctx, const uint64_t *a_xy, const uint8_t *a_inf, const uint64_t *b_xy, const uint8_t *b_inf, size_t n,
                         uint64_t *out_xy, uint8_t *out_flag) {
    return group_job(ctx, GOP_G2_ADD, a_xy, a_inf, b_xy, n, out_xy, out_flag, b_inf);
}
int32_t zkp_g1_check_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf, size_t n, uint8_t *status) {
    return group_job(ctx, GOP_G1_CHECK, g1_xy, g1_inf, nullptr, n, nullptr, status);
}
int32_t zkp_g2_check_batch(zkp_ctx *ctx, const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n, uint8_t *status) {
    return group_job(ctx, GOP_G2_CHECK, g2_xy, g2_inf, nullptr, n, nullptr, status);
}
int32_t zkp_g1_mul_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf, const uint64_t *scalars, size_t n,
                         uint64_t *out_xy, uint8_t *out_inf) {
    return group_job(ctx, GOP_G1_MUL, g1_xy, g1_inf, scalars, n, out_xy, out_inf);
}
int32_t zkp_g2_mul_batch(zkp_ctx *ctx, const uint64_t *g2_xy, const uint8_t *g2_inf, const uint64_t *scalars, size_t n,
                         uint64_t *out_xy, uint8_t *out_inf) {
    return group_job(ctx, GOP_G2_MUL, g2_xy, g2_inf, scalars, n, out_xy, out_inf);
}

// One large product: per-device shared-accumulator Miller loops over a contiguous slice -> per-device Fp12
// partial -> gather the 576-byte partials on the first device -> multiply -> ONE final exponentiation.
int32_t zkp_multi_miller_product(zkp_ctx *ctx, const uint64_t *g1, const uint8_t *g1inf, const uint64_t *g2, const uint8_t *g2inf,
                                 size_t n, uint64_t *out_miller_product, uint64_t *out_gt) {
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (!g1 || !g2 || n == 0) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer or n == 0");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard guard;
    const size_t chunk = ZKP_CHUNK;
    const int miller_mode = out_miller_product ? 1 : 5;   // the un-exponentiated product is only well defined with SURVEY 9.1's lines
    // One product over all pairs of the slice: the pairs of a chunk are grouped four to a lane pair and run as
    // shared-accumulator Miller loops (one Fp12 squaring chain per FOUR pairs: 4,684 instead of 6,916 Fp products
    // per pair, SURVEY 8a), the chunk's outputs are folded to one Fp12 in d.partial[chunk].  Nothing returns to the
    // host per chunk.
    auto body = [=](Chunk &c) {
        DevState &d = c.d;
        if (c.c0 == c.lo) CUT(d.partial.ensure(((c.hi - c.lo + chunk - 1) / chunk + 1) * 576));   // the partials and their fold
        const size_t ci = (c.c0 - c.lo) / chunk, nc4 = c.cn / ZKP_PRODUCT_GROUP, rem = c.cn % ZKP_PRODUCT_GROUP, ne = nc4 + (rem ? 1 : 0);
        const uint64_t *dg1 = c.in(B_G1, g1, c.c0 * 12, c.cn * 12), *dg2 = c.in(B_G2, g2, c.c0 * 24, c.cn * 24);
        uint64_t *dout = c.buf<uint64_t>(B_OUT, ne * 72);
        uint64_t *dscr = c.buf<uint64_t>(B_IN, zkp_product_scratch_elems(ne) * 72);   // this buffer set's product scratch
        const uint8_t *di1 = c.in(B_G1INF, g1inf, c.c0, c.cn), *di2 = c.in(B_G2INF, g2inf, c.c0, c.cn);
        if (nc4) CUT(launch_pairing(ctx, d, miller_mode, dg1, di1, dg2, di2, nc4, ZKP_PRODUCT_GROUP, nullptr, dout, nullptr, d.d_err, c.st));
        if (rem) {
            const size_t o = nc4 * ZKP_PRODUCT_GROUP;
            CUT(launch_pairing(ctx, d, miller_mode, dg1 + 12 * o, di1 ? di1 + o : nullptr, dg2 + 24 * o, di2 ? di2 + o : nullptr, 1, (int)rem,
                               nullptr, dout + 72 * nc4, nullptr, d.d_err, c.st));
        }
        CUT(launch_product(ctx, dout, ne, dscr, (uint64_t *)d.partial.p + 72 * ci, d.d_err, c.st));
    };
    auto fold = [=](DevState &d, size_t lo, size_t hi) {   // this device's chunk partials into the slot after the last one
        const size_t nchunks = (hi - lo + chunk - 1) / chunk;
        CUT(d.buf[0][B_IN].ensure(zkp_product_scratch_elems(nchunks) * 576));
        CUT(launch_product(ctx, (const uint64_t *)d.partial.p, nchunks, (uint64_t *)d.buf[0][B_IN].p, (uint64_t *)d.partial.p + 72 * nchunks,
                           d.d_err, d.stream[0]));
        CUT(cudaStreamSynchronize(d.stream[0]));
    };
    int32_t rc = run_slices(ctx, n, chunk, body, fold);
    if (rc != ZKP_OK) return rc;
    // gather: one 576-byte partial per device -> first device (peer copy over NVLink when available)
    const size_t nd = fan_out(ctx, n);
    DevState &d0 = ctx->devs[0];
    CU(cudaSetDevice(d0.id));
    DevBuf &G = d0.buf[1][B_IN];
    CU(G.ensure((nd + 2) * 576));
    for (size_t di = 0; di < nd; di++) {
        DevState &d = ctx->devs[di];
        size_t lo, hi;
        slice_of(n, nd, di, lo, hi);
        size_t nchunks = (hi - lo + chunk - 1) / chunk;
        const uint64_t *src = (const uint64_t *)d.partial.p + 72 * nchunks;
        if (d.id == d0.id)
            CU(cudaMemcpyAsync((uint64_t *)G.p + 72 * di, src, 576, cudaMemcpyDeviceToDevice, d0.stream[0]));
        else
            CU(cudaMemcpyPeerAsync((uint64_t *)G.p + 72 * di, d0.id, src, d.id, 576, d0.stream[0]));
    }
    uint64_t *prod = (uint64_t *)G.p + 72 * nd, *gt = (uint64_t *)G.p + 72 * (nd + 1);
    CU(d0.scratch.ensure(zkp_product_scratch_elems(nd) * 576));
    CU(launch_product(ctx, (const uint64_t *)G.p, nd, (uint64_t *)d0.scratch.p, prod, d0.d_err, d0.stream[0]));
    if (out_gt) CU(launch_pairing(ctx, d0, 2, nullptr, nullptr, nullptr, nullptr, 1, 1, prod, gt, nullptr, d0.d_err, d0.stream[0]));
    if (out_miller_product) CU(cudaMemcpyAsync(out_miller_product, prod, 576, cudaMemcpyDeviceToHost, d0.stream[0]));
    if (out_gt) CU(cudaMemcpyAsync(out_gt, gt, 576, cudaMemcpyDeviceToHost, d0.stream[0]));
    CU(cudaStreamSynchronize(d0.stream[0]));
    return ZKP_OK;
}

// ---- multi-scalar multiplication over caller-given points
int32_t zkp_g1_msm(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf, const uint64_t *scalars, size_t n, uint64_t *out_xy,
                   uint8_t *out_inf, uint8_t *out_status) {
    return msm_job<OpsFp>(ctx, g1_xy, g1_inf, scalars, n, out_xy, out_inf, out_status);
}
int32_t zkp_g2_msm(zkp_ctx *ctx, const uint64_t *g2_xy, const uint8_t *g2_inf, const uint64_t *scalars, size_t n, uint64_t *out_xy,
                   uint8_t *out_inf, uint8_t *out_status) {
    return msm_job<OpsFp2>(ctx, g2_xy, g2_inf, scalars, n, out_xy, out_inf, out_status);
}
int32_t zkp_g1_msm_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g1_xy, const uint8_t *d_g1_inf, const uint64_t *d_scalars, size_t n,
                       uint64_t *d_out_xy, uint8_t *d_out_inf, uint8_t *d_status, uint32_t *d_err, void *d_scratch, void *stream) {
    return msm_dev<OpsFp>(ctx, dev, d_g1_xy, d_g1_inf, d_scalars, n, d_out_xy, d_out_inf, d_status, d_err, d_scratch, stream);
}
int32_t zkp_g2_msm_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g2_xy, const uint8_t *d_g2_inf, const uint64_t *d_scalars, size_t n,
                       uint64_t *d_out_xy, uint8_t *d_out_inf, uint8_t *d_status, uint32_t *d_err, void *d_scratch, void *stream) {
    return msm_dev<OpsFp2>(ctx, dev, d_g2_xy, d_g2_inf, d_scalars, n, d_out_xy, d_out_inf, d_status, d_err, d_scratch, stream);
}

// ---- Groth16 verification
static const char *g16_point_error(uint8_t st) { return st == ZKP_POINT_NOT_ON_CURVE ? "is not on the curve" : "is not torsion free"; }

int32_t zkp_groth16_vk_create(zkp_ctx *ctx, const uint64_t *alpha_g1, const uint64_t *beta_g2, const uint64_t *gamma_g2,
                              const uint64_t *delta_g2, const uint64_t *ic_g1, const uint8_t *ic_inf, int32_t n_public,
                              zkp_groth16_vk **out) {
    if (!out) return fail(ZKP_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (!alpha_g1 || !beta_g2 || !gamma_g2 || !delta_g2 || !ic_g1) return fail(ZKP_ERR_INVALID_ARG, "NULL verifying-key point");
    if (n_public < 0 || n_public > ZKP_GROTH16_MAX_PUBLIC)
        return fail(ZKP_ERR_INVALID_ARG, "n_public out of range (0 .. ZKP_GROTH16_MAX_PUBLIC)");
    const size_t nic = (size_t)n_public + 1;
    // every key point is validated on the GPU: alpha and IC_0 .. IC_l (G1), beta, gamma, delta (G2)
    std::vector<uint64_t> g1(12 * (nic + 1)), g2(72);
    std::vector<uint8_t> g1inf(nic + 1, 0), st1(nic + 1), st2(3);
    memcpy(g1.data(), alpha_g1, 96);
    memcpy(g1.data() + 12, ic_g1, 96 * nic);
    if (ic_inf) memcpy(g1inf.data() + 1, ic_inf, nic);
    memcpy(g2.data(), beta_g2, 192);
    memcpy(g2.data() + 24, gamma_g2, 192);
    memcpy(g2.data() + 48, delta_g2, 192);
    int32_t rc = zkp_g1_check_batch(ctx, g1.data(), g1inf.data(), nic + 1, st1.data());
    if (rc == ZKP_OK) rc = zkp_g2_check_batch(ctx, g2.data(), nullptr, 3, st2.data());
    if (rc != ZKP_OK) return rc;
    if (st1[0]) return fail(ZKP_ERR_INVALID_ARG, std::string("alpha_g1 ") + g16_point_error(st1[0]));
    static const char *g2names[3] = {"beta_g2", "gamma_g2", "delta_g2"};
    for (int i = 0; i < 3; i++)
        if (st2[i]) return fail(ZKP_ERR_INVALID_ARG, std::string(g2names[i]) + " " + g16_point_error(st2[i]));
    for (size_t j = 0; j < nic; j++)
        if (st1[j + 1]) return fail(ZKP_ERR_INVALID_ARG, "ic_g1[" + std::to_string(j) + "] " + g16_point_error(st1[j + 1]));

    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard guard;
    zkp_groth16_vk *vk = new zkp_groth16_vk();
    vk->ctx = ctx;
    vk->n_public = n_public;
    vk->devs.resize(ctx->devs.size());
    const size_t prep_b = align256(3 * (size_t)ZKP_G2_PREPARED_U64 * 8), tab_b = (size_t)n_public * ZKP_G16_TABLE_FP * sizeof(Fp);
    const size_t tmp_ic = align256(96 * nic), tmp_g2 = align256(192 * 3);
    const size_t tmp_b = tmp_ic + tmp_g2 + (size_t)n_public * ZKP_G16_WINDOWS * 2 * ZKP_G16_DIGITS * sizeof(Fp);
    cudaError_t e = cudaSuccess;
    for (size_t di = 0; di < ctx->devs.size() && e == cudaSuccess; di++) {
        DevState &d = ctx->devs[di];
        G16Dev &k = vk->devs[di];
        k.id = d.id;
        void *tmp = nullptr;
        e = cudaSetDevice(d.id);
        // resident layout: prepared tables | alpha | IC_0 | IC flags | window tables
        if (e == cudaSuccess) e = cudaMalloc(&k.mem, prep_b + 256 + 256 + align256(nic) + tab_b);
        if (e == cudaSuccess) e = cudaMalloc(&tmp, tmp_b);
        if (e == cudaSuccess) {
            uint8_t *m = (uint8_t *)k.mem, *t = (uint8_t *)tmp;
            k.prep = (const Fp *)m;
            k.key.alpha = (const uint64_t *)(m + prep_b);
            k.key.ic0 = (const uint64_t *)(m + prep_b + 256);
            k.key.ic_inf = m + prep_b + 512;
            k.key.tables = (const Fp *)(m + prep_b + 512 + align256(nic));
            k.key.n_public = n_public;
            cudaStream_t st = d.stream[0];
            e = cudaMemcpyAsync((void *)k.key.alpha, alpha_g1, 96, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync((void *)k.key.ic0, ic_g1, 96, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync((void *)k.key.ic_inf, g1inf.data() + 1, nic, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(t, ic_g1, 96 * nic, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(t + tmp_ic, g2.data(), 192 * 3, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) {
                k_g16_neg_prepare<<<grid_for(3), ZKP_TPB, 0, st>>>((const uint64_t *)(t + tmp_ic), (Fp *)k.prep, 3);
                ctx->launches++;
                e = cudaGetLastError();
            }
            if (e == cudaSuccess && n_public) {
                unsigned threads = (unsigned)n_public * ZKP_G16_WINDOWS;
                k_g16_window_tables<<<(threads + ZKP_TPB - 1) / ZKP_TPB, ZKP_TPB, 0, st>>>(
                    (const uint64_t *)t, k.key.ic_inf, n_public, (Fp *)k.key.tables, (Fp *)(t + tmp_ic + tmp_g2));
                ctx->launches++;
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        }
        if (tmp) cudaFree(tmp);
    }
    if (e != cudaSuccess) {
        std::string msg = std::string("verifying key setup failed: ") + cudaGetErrorString(e);
        zkp_groth16_vk_destroy(vk);
        return fail(ZKP_ERR_CUDA, msg);
    }
    *out = vk;
    return ZKP_OK;
}

void zkp_groth16_vk_destroy(zkp_groth16_vk *vk) {
    if (!vk) return;
    DeviceGuard guard;
    for (G16Dev &k : vk->devs) {
        if (!k.mem) continue;
        cudaSetDevice(k.id);
        cudaFree(k.mem);
    }
    delete vk;
}

size_t zkp_groth16_scratch_bytes(size_t n) { return g16_layout(n, nullptr, nullptr); }

int32_t zkp_groth16_verify_batch(zkp_ctx *ctx, const zkp_groth16_vk *vk, const uint64_t *proofs, const uint8_t *proof_inf,
                                 const uint64_t *public_inputs, size_t n, uint8_t *out_status) {
    if (!ctx || !vk) return fail(ZKP_ERR_INVALID_ARG, "ctx or vk is NULL");
    if (vk->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the verifying key belongs to another context");
    if (n && (!proofs || !out_status || (vk->n_public && !public_inputs))) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    const size_t np = (size_t)vk->n_public;
    return run_host_job(ctx, n, g16_chunk(vk->n_public), [=](Chunk &c) {
        const uint64_t *dp = c.in(B_G1, proofs, c.c0 * 48, c.cn * 48);
        uint8_t *dst = c.buf<uint8_t>(B_FLAG, c.cn);
        uint8_t *dscr = c.buf<uint8_t>(B_OUT, g16_layout(c.cn, nullptr, nullptr));
        const uint8_t *dpi = c.in(B_G1INF, proof_inf, c.c0 * 3, c.cn * 3);
        const uint64_t *dx = c.in(B_IN, np ? public_inputs : nullptr, c.c0 * np * 4, c.cn * np * 4);
        CUT(launch_groth16(ctx, c.d, vk->devs[c.dev], dp, dpi, dx, c.cn, dst, dscr, c.d.d_err, c.st));
        c.out(B_FLAG, out_status + c.c0, dst, c.cn);
    });
}

int32_t zkp_groth16_verify_dev(zkp_ctx *ctx, int32_t dev, const zkp_groth16_vk *vk, const uint64_t *d_proofs,
                               const uint8_t *d_proof_inf, const uint64_t *d_public_inputs, size_t n, uint8_t *d_status,
                               void *d_scratch, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (!vk) return fail(ZKP_ERR_INVALID_ARG, "vk is NULL");
    if (vk->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the verifying key belongs to another context");
    if (n && (!d_proofs || !d_status || !d_scratch || (vk->n_public && !d_public_inputs))) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if ((uintptr_t)d_scratch & 15) return fail(ZKP_ERR_INVALID_ARG, "d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_groth16(ctx, d, vk->devs[dev], d_proofs, d_proof_inf, d_public_inputs, n, d_status, d_scratch, nullptr, st));
        return ZKP_OK;
    });
}

// ---- KZG point-evaluation verification

// Lagrange tables of a prover setup on one device, and the consistency check of the points against [tau]G1: one MSM
// of two rows, sum_k L_k (must be G1) and sum_k omega^k L_k (= [tau]G1), then e(S1, G2) e(G1, -[tau]G2) == 1 on the
// setup's prepared tables.  *consistent receives the verdict.  tmp holds G1 at byte offset 96 (k_kzg_generators).
static cudaError_t kzg_lagrange_build(zkp_ctx *ctx, DevState &d, KzgDev &k, const uint64_t *g1_lagrange, const uint8_t *tmp,
                                      bool *consistent) {
    const size_t slice = 1024;   // bases per table launch: 32 768 threads, 384 MiB of chain scratch
    const size_t t_lag = 0, t_rows = align256((size_t)ZKP_BLOB_N * 96), t_pts = t_rows + 2 * ZKP_BLOB_BYTES, t_inf = t_pts + 512,
                 t_gt = t_inf + 256, t_ws = t_gt + 1024;
    const size_t tmp_b = t_ws + slice * ZKP_MSM_WINDOWS * 2 * ZKP_MSM_DIGITS * sizeof(Fp);
    cudaStream_t st = d.stream[0];
    void *scratch = nullptr;
    cudaError_t e = cudaMalloc(&k.lag_mem, (size_t)ZKP_BLOB_N * ZKP_MSM_TABLE_FP * sizeof(Fp));
    if (e == cudaSuccess) e = cudaMalloc(&scratch, tmp_b);
    if (e == cudaSuccess) {
        uint8_t *t = (uint8_t *)scratch;
        uint64_t *pts = (uint64_t *)(t + t_pts);   // S0 | S1 | G1
        uint8_t *inf = t + t_inf;                  // their flags | the two statuses | is_one
        e = cudaMemcpyAsync(t + t_lag, g1_lagrange, (size_t)ZKP_BLOB_N * 96, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(inf, 0, 8, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(pts + 24, tmp + 96, 96, cudaMemcpyDeviceToDevice, st);
        for (size_t f = 0; f < ZKP_BLOB_N && e == cudaSuccess; f += slice) {
            k_kzg_lagrange_tables<<<(unsigned)(slice * ZKP_MSM_WINDOWS / ZKP_TPB), ZKP_TPB, 0, st>>>(
                (const uint64_t *)(t + t_lag), (int)f, (int)slice, true, (Fp *)k.lag_mem, (Fp *)(t + t_ws));
            ctx->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) {
            k_kzg_check_rows<<<ZKP_BLOB_N / 128, 128, 0, st>>>(k.roots, t + t_rows);
            k_kzg_msm<<<2, ZKP_MSM_TPB, 0, st>>>((const Fp *)k.lag_mem, t + t_rows, nullptr, pts, inf, inf + 4);
            ctx->launches += 2;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess)
            e = launch_pairing(ctx, d, 3, pts + 12, inf + 1, nullptr, nullptr, 1, 2, nullptr, (uint64_t *)(t + t_gt), inf + 7, nullptr, st,
                               k.prep, nullptr, 2);
        uint64_t h[36];
        uint8_t hf[8];
        if (e == cudaSuccess) e = cudaMemcpyAsync(h, pts, sizeof h, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(hf, inf, sizeof hf, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) *consistent = !hf[0] && !memcmp(h, h + 24, 96) && hf[7] == 1;
    }
    if (scratch) cudaFree(scratch);
    return e;
}

// zkp_kzg_setup_create, and with g1_lagrange (4096 points, natural order) zkp_kzg_setup_create_prover
static int32_t kzg_setup_create(zkp_ctx *ctx, const uint64_t *tau_g2, const uint64_t *g1_lagrange, zkp_kzg_setup **out) {
    if (!out) return fail(ZKP_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (!tau_g2) return fail(ZKP_ERR_INVALID_ARG, "tau_g2 is NULL");
    uint8_t st2 = 0;
    int32_t rc = zkp_g2_check_batch(ctx, tau_g2, nullptr, 1, &st2);   // validated on the GPU
    if (rc != ZKP_OK) return rc;
    if (st2) return fail(ZKP_ERR_INVALID_ARG, std::string("tau_g2 ") + g16_point_error(st2));
    if (g1_lagrange) {   // every Lagrange point, validated on the GPU
        std::vector<uint8_t> st1(ZKP_BLOB_N);
        rc = zkp_g1_check_batch(ctx, g1_lagrange, nullptr, ZKP_BLOB_N, st1.data());
        if (rc == ZKP_ERR_NONCANONICAL) return fail(rc, "g1_lagrange has a limb >= p (non-canonical field element)");
        if (rc != ZKP_OK) return rc;
        for (int i = 0; i < ZKP_BLOB_N; i++)
            if (st1[i]) return fail(ZKP_ERR_INVALID_ARG, "g1_lagrange[" + std::to_string(i) + "] " + g16_point_error(st1[i]));
    }

    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard guard;
    zkp_kzg_setup *s = new zkp_kzg_setup();
    s->ctx = ctx;
    s->prover = g1_lagrange != nullptr;
    s->devs.resize(ctx->devs.size());
    bool consistent = true;
    const size_t prep_b = align256(2 * (size_t)ZKP_G2_PREPARED_U64 * 8), tab_b = align256((size_t)ZKP_G16_TABLE_FP * sizeof(Fp));
    const size_t roots_b = (size_t)ZKP_BLOB_N * sizeof(Fr);
    // temporary layout: IC_0 = 0 | IC_1 = G1 (the window-table kernel's key layout, one table) | their two flags | G2 |
    // tau_g2 | the window-table kernel's scratch
    const size_t t_inf = 256, t_g2 = 512, t_tau = 768, t_ws = 1024;
    const size_t tmp_b = t_ws + (size_t)ZKP_G16_WINDOWS * 2 * ZKP_G16_DIGITS * sizeof(Fp);
    cudaError_t e = cudaSuccess;
    for (size_t di = 0; di < ctx->devs.size() && e == cudaSuccess && consistent; di++) {
        DevState &d = ctx->devs[di];
        KzgDev &k = s->devs[di];
        k.id = d.id;
        void *tmp = nullptr;
        e = cudaSetDevice(d.id);
        // resident layout: prepared tables of G2, -[tau]G2 | window table of G1 | blob domain roots_brp
        if (e == cudaSuccess) e = cudaMalloc(&k.mem, prep_b + tab_b + roots_b);
        if (e == cudaSuccess) e = cudaMalloc(&tmp, tmp_b);
        if (e == cudaSuccess) {
            uint8_t *m = (uint8_t *)k.mem, *t = (uint8_t *)tmp;
            k.prep = (const Fp *)m;
            k.table = (const Fp *)(m + prep_b);
            k.roots = (const Fr *)(m + prep_b + tab_b);
            cudaStream_t st = d.stream[0];
            e = cudaMemsetAsync(t, 0, t_g2, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(t + t_tau, tau_g2, 192, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) {
                k_kzg_generators<<<1, 32, 0, st>>>((uint64_t *)t + 12, (uint64_t *)(t + t_g2));
                k_g2_prepare<<<grid_for(1), ZKP_TPB, 0, st>>>((const uint64_t *)(t + t_g2), (Fp *)k.prep, nullptr, 1);
                k_g16_neg_prepare<<<grid_for(1), ZKP_TPB, 0, st>>>((const uint64_t *)(t + t_tau),
                                                                   (Fp *)(m + (size_t)ZKP_G2_PREPARED_U64 * 8), 1);
                k_g16_window_tables<<<1, ZKP_TPB, 0, st>>>((const uint64_t *)t, t + t_inf, 1, (Fp *)k.table, (Fp *)(t + t_ws));
                k_blob_domain<<<ZKP_BLOB_N / 128, 128, 0, st>>>((Fr *)k.roots);
                ctx->launches += 5;
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e == cudaSuccess && g1_lagrange) e = kzg_lagrange_build(ctx, d, k, g1_lagrange, t, &consistent);
        }
        if (tmp) cudaFree(tmp);
    }
    if (e != cudaSuccess) {
        std::string msg = std::string("KZG setup failed: ") + cudaGetErrorString(e);
        zkp_kzg_setup_destroy(s);
        return fail(ZKP_ERR_CUDA, msg);
    }
    if (!consistent) {
        zkp_kzg_setup_destroy(s);
        return fail(ZKP_ERR_INVALID_ARG, "g1_lagrange is inconsistent with tau_g2");
    }
    *out = s;
    return ZKP_OK;
}

int32_t zkp_kzg_setup_create(zkp_ctx *ctx, const uint64_t *tau_g2, zkp_kzg_setup **out) {
    return kzg_setup_create(ctx, tau_g2, nullptr, out);
}

int32_t zkp_kzg_setup_create_prover(zkp_ctx *ctx, const uint64_t *tau_g2, const uint64_t *g1_lagrange, zkp_kzg_setup **out) {
    if (!g1_lagrange) {
        if (out) *out = nullptr;
        return fail(ZKP_ERR_INVALID_ARG, "g1_lagrange is NULL");
    }
    return kzg_setup_create(ctx, tau_g2, g1_lagrange, out);
}

void zkp_kzg_setup_destroy(zkp_kzg_setup *s) {
    if (!s) return;
    DeviceGuard guard;
    for (KzgDev &k : s->devs) {
        if (!k.mem && !k.lag_mem && !k.cell_mem) continue;
        cudaSetDevice(k.id);
        if (k.mem) cudaFree(k.mem);
        if (k.lag_mem) cudaFree(k.lag_mem);
        if (k.cell_mem) cudaFree(k.cell_mem);
    }
    delete s;
}

size_t zkp_kzg_scratch_bytes(size_t n) { return kzg_layout(n, nullptr, nullptr); }

int32_t zkp_kzg_verify_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *proofs, const uint8_t *proof_inf, const uint64_t *zy,
                             size_t n, uint8_t *out_status) {
    if (!ctx || !s) return fail(ZKP_ERR_INVALID_ARG, "ctx or setup is NULL");
    if (s->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup belongs to another context");
    if (n && (!proofs || !zy || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return run_host_job(ctx, n, ZKP_CHUNK, [=](Chunk &c) {
        const uint64_t *dp = c.in(B_G1, proofs, c.c0 * 24, c.cn * 24), *dzy = c.in(B_IN, zy, c.c0 * 8, c.cn * 8);
        uint8_t *dst = c.buf<uint8_t>(B_FLAG, c.cn);
        uint8_t *dscr = c.buf<uint8_t>(B_OUT, kzg_layout(c.cn, nullptr, nullptr));
        const uint8_t *dpi = c.in(B_G1INF, proof_inf, c.c0 * 2, c.cn * 2);
        CUT(launch_kzg(ctx, c.d, s->devs[c.dev], dp, dpi, dzy, c.cn, dst, dscr, c.d.d_err, c.st));
        c.out(B_FLAG, out_status + c.c0, dst, c.cn);
    });
}

int32_t zkp_kzg_verify_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_proofs, const uint8_t *d_proof_inf,
                           const uint64_t *d_zy, size_t n, uint8_t *d_status, void *d_scratch, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (!s) return fail(ZKP_ERR_INVALID_ARG, "setup is NULL");
    if (s->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup belongs to another context");
    if (n && (!d_proofs || !d_zy || !d_status || !d_scratch)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if ((uintptr_t)d_scratch & 15) return fail(ZKP_ERR_INVALID_ARG, "d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_kzg(ctx, d, s->devs[dev], d_proofs, d_proof_inf, d_zy, n, d_status, d_scratch, nullptr, st));
        return ZKP_OK;
    });
}

// ---- EIP-4844 blob verification

int32_t zkp_kzg_verify_blob_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *proofs,
                                  const uint8_t *proof_inf, size_t n, uint8_t *out_status, uint64_t *out_zy) {
    if (!ctx || !s) return fail(ZKP_ERR_INVALID_ARG, "ctx or setup is NULL");
    if (s->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup belongs to another context");
    if (n && (!blobs || !proofs || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return run_host_job(ctx, n, ZKP_BLOB_CHUNK, [=](Chunk &c) {
        const uint8_t *db = c.in(B_IN, blobs, c.c0 * ZKP_BLOB_BYTES, c.cn * ZKP_BLOB_BYTES);
        const uint64_t *dp = c.in(B_G1, proofs, c.c0 * 24, c.cn * 24);
        uint8_t *dst = c.buf<uint8_t>(B_FLAG, c.cn);
        uint8_t *dscr = c.buf<uint8_t>(B_OUT, zkp_kzg_blob_scratch_bytes(c.cn));
        const uint8_t *dpi = c.in(B_G1INF, proof_inf, c.c0 * 2, c.cn * 2);
        CUT(launch_kzg_blob(ctx, c.d, s->devs[c.dev], db, dp, dpi, c.cn, dst, nullptr, dscr, c.d.d_err, c.st));
        c.out(B_FLAG, out_status + c.c0, dst, c.cn);
        if (out_zy) c.out(B_OUT, out_zy + c.c0 * 8, (const uint64_t *)dscr, c.cn * 8);   // z | y, first in the scratch
    });
}

int32_t zkp_kzg_verify_blob_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, const uint64_t *d_proofs,
                                const uint8_t *d_proof_inf, size_t n, uint8_t *d_status, uint64_t *d_out_zy, void *d_scratch, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (!s) return fail(ZKP_ERR_INVALID_ARG, "setup is NULL");
    if (s->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup belongs to another context");
    if (n && (!d_blobs || !d_proofs || !d_status || !d_scratch)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_scratch & 15) || ((uintptr_t)d_blobs & 15)) return fail(ZKP_ERR_INVALID_ARG, "d_blobs and d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_kzg_blob(ctx, d, s->devs[dev], d_blobs, d_proofs, d_proof_inf, n, d_status, d_out_zy, d_scratch, nullptr, st));
        return ZKP_OK;
    });
}

// ---- EIP-4844 prover

static int32_t check_prover(zkp_ctx *ctx, const zkp_kzg_setup *s) {
    if (!ctx || !s) return fail(ZKP_ERR_INVALID_ARG, "ctx or setup is NULL");
    if (s->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup belongs to another context");
    if (!s->prover) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup has no Lagrange points (create it with zkp_kzg_setup_create_prover)");
    return ZKP_OK;
}

// The three prover calls over host buffers: commitments (z and c NULL), proofs at z (y to y_out) or blob proofs for
// the commitments c (flags cinf or NULL; z | y to zy_out when it is not NULL)
static int32_t prover_job(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *z, const uint64_t *c_pts,
                          const uint8_t *cinf, size_t n, uint64_t *out, uint8_t *out_inf, uint64_t *y_out, uint8_t *status, uint64_t *zy_out) {
    return run_host_job(ctx, n, ZKP_BLOB_CHUNK, [=](Chunk &c) {
        const KzgDev &kd = s->devs[c.dev];
        const uint8_t *db = c.in(B_IN, blobs, c.c0 * ZKP_BLOB_BYTES, c.cn * ZKP_BLOB_BYTES);
        uint64_t *dout = c.buf<uint64_t>(B_G2, c.cn * 12);
        uint8_t *dinf = c.buf<uint8_t>(B_G2INF, c.cn), *dst = c.buf<uint8_t>(B_FLAG, c.cn);
        if (!z && !c_pts) {
            CUT(launch_kzg_commit(ctx, kd, db, c.cn, dout, dinf, dst, c.st));
        } else {
            uint8_t *dscr = c.buf<uint8_t>(B_OUT, zkp_kzg_prover_scratch_bytes(c.cn));
            uint64_t *dzy = (uint64_t *)(dscr + prove_rows_bytes(c.cn));   // z | y, after the rows
            const uint64_t *dz = nullptr, *dc = nullptr;
            const uint8_t *dci = nullptr;
            uint64_t *dy = nullptr;
            if (z) {
                dz = c.in(B_G1, z, c.c0 * 4, c.cn * 4);
                dy = c.buf<uint64_t>(B_TAB, c.cn * 4);
            } else {
                dc = c.in(B_G1, c_pts, c.c0 * 12, c.cn * 12);
                dci = c.in(B_G1INF, cinf, c.c0, c.cn);
            }
            CUT(launch_kzg_prove(ctx, kd, db, dz, dc, dci, c.cn, dout, dinf, dy, dzy, dst, dscr, c.st));
            if (z) c.out(B_TAB, y_out + c.c0 * 4, dy, c.cn * 4);
            else if (zy_out) c.out(B_OUT, zy_out + c.c0 * 8, dzy, c.cn * 8);
        }
        c.out(B_G2, out + c.c0 * 12, dout, c.cn * 12);
        c.out(B_G2INF, out_inf + c.c0, dinf, c.cn);
        c.out(B_FLAG, status + c.c0, dst, c.cn);
    });
}

int32_t zkp_kzg_blob_to_commitment_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, size_t n, uint64_t *out_c,
                                         uint8_t *out_c_inf, uint8_t *out_status) {
    int32_t rc = check_prover(ctx, s);
    if (rc) return rc;
    if (n && (!blobs || !out_c || !out_c_inf || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return prover_job(ctx, s, blobs, nullptr, nullptr, nullptr, n, out_c, out_c_inf, nullptr, out_status, nullptr);
}

int32_t zkp_kzg_compute_proof_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *z, size_t n,
                                    uint64_t *out_proof, uint8_t *out_proof_inf, uint64_t *out_y, uint8_t *out_status) {
    int32_t rc = check_prover(ctx, s);
    if (rc) return rc;
    if (n && (!blobs || !z || !out_proof || !out_proof_inf || !out_y || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return prover_job(ctx, s, blobs, z, nullptr, nullptr, n, out_proof, out_proof_inf, out_y, out_status, nullptr);
}

int32_t zkp_kzg_compute_blob_proof_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *commitments,
                                         const uint8_t *commitment_inf, size_t n, uint64_t *out_proof, uint8_t *out_proof_inf,
                                         uint8_t *out_status, uint64_t *out_zy) {
    int32_t rc = check_prover(ctx, s);
    if (rc) return rc;
    if (n && (!blobs || !commitments || !out_proof || !out_proof_inf || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return prover_job(ctx, s, blobs, nullptr, commitments, commitment_inf, n, out_proof, out_proof_inf, nullptr, out_status, out_zy);
}

int32_t zkp_kzg_blob_to_commitment_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, size_t n,
                                       uint64_t *d_c, uint8_t *d_c_inf, uint8_t *d_status, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_prover(ctx, s);
    if (rc) return rc;
    if (n && (!d_blobs || !d_c || !d_c_inf || !d_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if ((uintptr_t)d_blobs & 15) return fail(ZKP_ERR_INVALID_ARG, "d_blobs must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_kzg_commit(ctx, s->devs[dev], d_blobs, n, d_c, d_c_inf, d_status, st));
        return ZKP_OK;
    });
}

int32_t zkp_kzg_compute_proof_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, const uint64_t *d_z, size_t n,
                                  uint64_t *d_proof, uint8_t *d_proof_inf, uint64_t *d_y, uint8_t *d_status, void *d_scratch, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_prover(ctx, s);
    if (rc) return rc;
    if (n && (!d_blobs || !d_z || !d_proof || !d_proof_inf || !d_y || !d_status || !d_scratch))
        return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_scratch & 15) || ((uintptr_t)d_blobs & 15)) return fail(ZKP_ERR_INVALID_ARG, "d_blobs and d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_kzg_prove(ctx, s->devs[dev], d_blobs, d_z, nullptr, nullptr, n, d_proof, d_proof_inf, d_y, nullptr, d_status, d_scratch,
                            st));
        return ZKP_OK;
    });
}

int32_t zkp_kzg_compute_blob_proof_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, const uint64_t *d_commitments,
                                       const uint8_t *d_commitment_inf, size_t n, uint64_t *d_proof, uint8_t *d_proof_inf, uint8_t *d_status,
                                       uint64_t *d_out_zy, void *d_scratch, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_prover(ctx, s);
    if (rc) return rc;
    if (n && (!d_blobs || !d_commitments || !d_proof || !d_proof_inf || !d_status || !d_scratch))
        return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_scratch & 15) || ((uintptr_t)d_blobs & 15)) return fail(ZKP_ERR_INVALID_ARG, "d_blobs and d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_kzg_prove(ctx, s->devs[dev], d_blobs, nullptr, d_commitments, d_commitment_inf, n, d_proof, d_proof_inf, nullptr, d_out_zy,
                            d_status, d_scratch, st));
        return ZKP_OK;
    });
}

// ---- EIP-7594 cells

// The cells parts of a setup on one device: the prepared tables of G2 and -[tau^64]G2, the twiddles pw and the window
// tables of the monomial points, then the checks of the points: g1_monomial[0] = G1, g2_monomial[0] = G2,
// e(M_{i+1}, G2) e(M_i, -[tau]G2) == 1 for i < 4095 on the setup's prepared tables, and e(-G1, g2_monomial[i])
// e(M_i, G2) == 1 for i <= 64 with g2_monomial[i] in the per-check slot.  why receives the first failed check.
static cudaError_t kzg_cells_build(zkp_ctx *ctx, DevState &d, KzgDev &k, const uint64_t *g2_mono, const uint64_t *g1_mono, std::string &why) {
    const int nc = ZKP_BLOB_N - 1, ng = ZKP_CELL_N + 1;   // chain checks, G2 checks
    const size_t prep1 = (size_t)ZKP_G2_PREPARED_U64 * 8, slice = 1024;
    const size_t c_pw = align256(2 * prep1), c_mono = c_pw + align256((size_t)ZKP_CELLS_EXT_N * sizeof(Fr));
    const size_t cell_b = c_mono + (size_t)ZKP_BLOB_N * ZKP_MSM_TABLE_FP * sizeof(Fp);
    // temporary layout: monomial points | G2 monomial points | G1 | G2 | chain pairs | G2-check pairs | Gt | is_one | table scratch
    const size_t t_g2 = align256((size_t)ZKP_BLOB_N * 96), t_gen = t_g2 + align256(ng * 192), t_chain = t_gen + 512,
                 t_pairs = t_chain + align256((size_t)nc * 192), t_gt = t_pairs + align256(ng * 192), t_one = t_gt + align256((size_t)nc * 576),
                 t_ws = t_one + align256(nc + ng);
    const size_t tmp_b = t_ws + slice * ZKP_MSM_WINDOWS * 2 * ZKP_MSM_DIGITS * sizeof(Fp);
    cudaStream_t st = d.stream[0];
    void *scratch = nullptr;
    cudaError_t e = cudaFuncSetAttribute(k_cells_extend, cudaFuncAttributeMaxDynamicSharedMemorySize, ZKP_BLOB_N * sizeof(Fr));
    if (e == cudaSuccess) {   // recovery's clusters; a failure here only disables recovery (its calls report it)
        k.recover_err = cudaFuncSetAttribute(k_cells_recover, cudaFuncAttributeMaxDynamicSharedMemorySize, ZKP_RECOVER_HALF * sizeof(Fr));
        if (k.recover_err == cudaSuccess) {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(2);
            cfg.blockDim = dim3(ZKP_CELLS_TPB);
            cfg.dynamicSmemBytes = ZKP_RECOVER_HALF * sizeof(Fr);
            k.recover_err = cudaOccupancyMaxActiveClusters(&k.recover_clusters, k_cells_recover, &cfg);
        }
        if (k.recover_err != cudaSuccess) {
            cudaGetLastError();
            k.recover_clusters = 0;
        }
    }
    if (e == cudaSuccess) e = cudaMalloc(&k.cell_mem, cell_b);
    if (e == cudaSuccess) e = cudaMalloc(&scratch, tmp_b);
    if (e == cudaSuccess) {
        uint8_t *m = (uint8_t *)k.cell_mem, *t = (uint8_t *)scratch;
        k.cell_prep = (const Fp *)m;
        k.pw = (const Fr *)(m + c_pw);
        k.mono = (const Fp *)(m + c_mono);
        e = cudaMemcpyAsync(t, g1_mono, (size_t)ZKP_BLOB_N * 96, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(t + t_g2, g2_mono, ng * 192, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(m, k.prep, prep1, cudaMemcpyDeviceToDevice, st);   // G2's table
        if (e == cudaSuccess) {
            k_g16_neg_prepare<<<grid_for(1), ZKP_TPB, 0, st>>>((const uint64_t *)(t + t_g2) + 24 * ZKP_CELL_N, (Fp *)(m + prep1), 1);
            k_cells_powers<<<ZKP_CELLS_EXT_N / 128, 128, 0, st>>>((Fr *)k.pw);
            k_kzg_generators<<<1, 32, 0, st>>>((uint64_t *)(t + t_gen), (uint64_t *)(t + t_gen) + 12);
            k_cells_setup_pairs<<<grid_for(nc), ZKP_TPB, 0, st>>>((const uint64_t *)t, (const uint64_t *)(t + t_gen), (uint64_t *)(t + t_chain),
                                                                 (uint64_t *)(t + t_pairs));
            ctx->launches += 4;
            e = cudaGetLastError();
        }
        for (size_t f = 0; f < ZKP_BLOB_N && e == cudaSuccess; f += slice) {
            k_kzg_lagrange_tables<<<(unsigned)(slice * ZKP_MSM_WINDOWS / ZKP_TPB), ZKP_TPB, 0, st>>>(
                (const uint64_t *)t, (int)f, (int)slice, false, (Fp *)k.mono, (Fp *)(t + t_ws));
            ctx->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess)
            e = launch_pairing(ctx, d, 3, (const uint64_t *)(t + t_chain), nullptr, nullptr, nullptr, nc, 2, nullptr, (uint64_t *)(t + t_gt),
                               t + t_one, nullptr, st, k.prep, nullptr, 2);
        if (e == cudaSuccess)
            e = launch_pairing(ctx, d, 3, (const uint64_t *)(t + t_pairs), nullptr, (const uint64_t *)(t + t_g2), nullptr, ng, 2, nullptr,
                               (uint64_t *)(t + t_gt), t + t_one + nc, nullptr, st, k.prep, nullptr, 1);
        uint64_t gen[36];
        std::vector<uint8_t> one(nc + ng);
        if (e == cudaSuccess) e = cudaMemcpyAsync(gen, t + t_gen, sizeof gen, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(one.data(), t + t_one, one.size(), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) {
            if (memcmp(g1_mono, gen, 96)) why = "g1_monomial[0] is not the G1 generator";
            else if (memcmp(g2_mono, gen + 12, 192)) why = "g2_monomial[0] is not the G2 generator";
            for (int i = 0; i < nc && why.empty(); i++)
                if (one[i] != 1)
                    why = "g1_monomial[" + std::to_string(i + 1) + "] is inconsistent with g1_monomial[" + std::to_string(i) + "] and g2_monomial[1]";
            for (int i = 0; i < ng && why.empty(); i++)
                if (one[nc + i] != 1) why = "g2_monomial[" + std::to_string(i) + "] is inconsistent with g1_monomial[" + std::to_string(i) + "]";
        }
    }
    if (scratch) cudaFree(scratch);
    return e;
}

int32_t zkp_kzg_setup_create_cells(zkp_ctx *ctx, const uint64_t *g2_monomial, const uint64_t *g1_monomial, const uint64_t *g1_lagrange,
                                   zkp_kzg_setup **out) {
    if (!out) return fail(ZKP_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (!ctx) return fail(ZKP_ERR_INVALID_ARG, "ctx is NULL");
    if (!g2_monomial || !g1_monomial) return fail(ZKP_ERR_INVALID_ARG, "g2_monomial or g1_monomial is NULL");
    std::vector<uint8_t> st2(ZKP_CELL_N + 1), st1(ZKP_BLOB_N);   // every point, validated on the GPU
    int32_t rc = zkp_g2_check_batch(ctx, g2_monomial, nullptr, st2.size(), st2.data());
    if (rc == ZKP_ERR_NONCANONICAL) return fail(rc, "g2_monomial has a limb >= p (non-canonical field element)");
    if (rc != ZKP_OK) return rc;
    for (size_t i = 0; i < st2.size(); i++)
        if (st2[i]) return fail(ZKP_ERR_INVALID_ARG, "g2_monomial[" + std::to_string(i) + "] " + g16_point_error(st2[i]));
    rc = zkp_g1_check_batch(ctx, g1_monomial, nullptr, st1.size(), st1.data());
    if (rc == ZKP_ERR_NONCANONICAL) return fail(rc, "g1_monomial has a limb >= p (non-canonical field element)");
    if (rc != ZKP_OK) return rc;
    for (size_t i = 0; i < st1.size(); i++)
        if (st1[i]) return fail(ZKP_ERR_INVALID_ARG, "g1_monomial[" + std::to_string(i) + "] " + g16_point_error(st1[i]));
    zkp_kzg_setup *s = nullptr;
    rc = kzg_setup_create(ctx, g2_monomial + 24, g1_lagrange, &s);   // tau from g2_monomial[1]
    if (rc != ZKP_OK) return rc;
    std::string why;
    cudaError_t e = cudaSuccess;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        DeviceGuard guard;
        for (size_t di = 0; di < ctx->devs.size() && e == cudaSuccess && why.empty(); di++) {
            e = cudaSetDevice(ctx->devs[di].id);
            if (e == cudaSuccess) e = kzg_cells_build(ctx, ctx->devs[di], s->devs[di], g2_monomial, g1_monomial, why);
        }
    }
    if (e != cudaSuccess) {
        std::string msg = std::string("KZG cells setup failed: ") + cudaGetErrorString(e);
        zkp_kzg_setup_destroy(s);
        return fail(ZKP_ERR_CUDA, msg);
    }
    if (!why.empty()) {
        zkp_kzg_setup_destroy(s);
        return fail(ZKP_ERR_INVALID_ARG, why);
    }
    s->cells = true;
    *out = s;
    return ZKP_OK;
}

static int32_t check_cells(zkp_ctx *ctx, const zkp_kzg_setup *s) {
    if (!ctx || !s) return fail(ZKP_ERR_INVALID_ARG, "ctx or setup is NULL");
    if (s->ctx != ctx) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup belongs to another context");
    if (!s->cells) return fail(ZKP_ERR_INVALID_ARG, "the KZG setup has no monomial points (create it with zkp_kzg_setup_create_cells)");
    return ZKP_OK;
}

// The cells of n blobs over host buffers, from the blobs or (blobs NULL) recovered from each blob's 128 indices, 128
// cells and count; with the proofs when proofs is not NULL
static int32_t cells_job(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *idx, const uint8_t *cells,
                         const uint64_t *num, size_t n, uint8_t *out_cells, uint64_t *proofs, uint8_t *proof_inf, uint8_t *status) {
    const size_t cb = (size_t)ZKP_CELLS_PER_EXT_BLOB * ZKP_CELL_BYTES;
    const size_t chunk = proofs ? ZKP_CELL_PROOF_CHUNK : blobs ? ZKP_CELLS_CHUNK : ZKP_CELLS_RECOVER_CHUNK;
    return run_host_job(ctx, n, chunk, [=](Chunk &c) {
        const size_t np = c.cn * ZKP_CELLS_PER_EXT_BLOB;
        const uint8_t *db = nullptr, *dcells = nullptr;
        const uint64_t *didx = nullptr, *dnum = nullptr;
        uint8_t *dout;
        if (blobs) {
            db = c.in(B_IN, blobs, c.c0 * ZKP_BLOB_BYTES, c.cn * ZKP_BLOB_BYTES);
            dout = c.buf<uint8_t>(B_G1, c.cn * cb);
        } else {
            dcells = c.in(B_IN, cells, c.c0 * cb, c.cn * cb);
            dout = c.buf<uint8_t>(B_G1, c.cn * cb);
            didx = c.in(B_TAB, idx, c.c0 * ZKP_CELLS_PER_EXT_BLOB, np);
            dnum = c.in(B_G1INF, num, c.c0, c.cn);
        }
        uint8_t *dst = c.buf<uint8_t>(B_FLAG, c.cn);
        uint64_t *dpf = nullptr;
        uint8_t *dpi = nullptr, *dscr = nullptr;
        if (proofs) {
            dpf = c.buf<uint64_t>(B_G2, np * 12);
            dpi = c.buf<uint8_t>(B_G2INF, np);
            dscr = c.buf<uint8_t>(B_OUT, zkp_kzg_cells_proofs_scratch_bytes(c.cn));
        }
        const KzgDev &kd = s->devs[c.dev];
        if (blobs) CUT(launch_cells(ctx, kd, db, c.cn, dout, dpf, dpi, dst, dscr, c.st));
        else CUT(launch_cells_recover(ctx, kd, didx, dcells, dnum, c.cn, dout, dpf, dpi, dst, dscr, c.st));
        c.out(B_G1, out_cells + c.c0 * cb, dout, c.cn * cb);
        if (proofs) {
            c.out(B_G2, proofs + c.c0 * ZKP_CELLS_PER_EXT_BLOB * 12, dpf, np * 12);
            c.out(B_G2INF, proof_inf + c.c0 * ZKP_CELLS_PER_EXT_BLOB, dpi, np);
        }
        c.out(B_FLAG, status + c.c0, dst, c.cn);
    });
}

int32_t zkp_kzg_compute_cells_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, size_t n, uint8_t *out_cells,
                                    uint8_t *out_status) {
    int32_t rc = check_cells(ctx, s);
    if (rc) return rc;
    if (n && (!blobs || !out_cells || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return cells_job(ctx, s, blobs, nullptr, nullptr, nullptr, n, out_cells, nullptr, nullptr, out_status);
}

int32_t zkp_kzg_compute_cells_and_proofs_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, size_t n, uint8_t *out_cells,
                                               uint64_t *out_proofs, uint8_t *out_proof_inf, uint8_t *out_status) {
    int32_t rc = check_cells(ctx, s);
    if (rc) return rc;
    if (n && (!blobs || !out_cells || !out_proofs || !out_proof_inf || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return cells_job(ctx, s, blobs, nullptr, nullptr, nullptr, n, out_cells, out_proofs, out_proof_inf, out_status);
}

int32_t zkp_kzg_verify_cell_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *commitments, const uint8_t *commitment_inf,
                                  const uint64_t *cell_indices, const uint8_t *cells, const uint64_t *proofs, const uint8_t *proof_inf, size_t n,
                                  uint8_t *out_status) {
    int32_t rc = check_cells(ctx, s);
    if (rc) return rc;
    if (n && (!commitments || !cell_indices || !cells || !proofs || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return run_host_job(ctx, n, ZKP_CELL_VERIFY_CHUNK, [=](Chunk &c) {
        const uint64_t *dc = c.in(B_G1, commitments, c.c0 * 12, c.cn * 12), *dpf = c.in(B_G2, proofs, c.c0 * 12, c.cn * 12);
        const uint64_t *didx = c.in(B_TAB, cell_indices, c.c0, c.cn);
        const uint8_t *dcells = c.in(B_IN, cells, c.c0 * ZKP_CELL_BYTES, c.cn * ZKP_CELL_BYTES);
        uint8_t *dst = c.buf<uint8_t>(B_FLAG, c.cn);
        uint8_t *dscr = c.buf<uint8_t>(B_OUT, zkp_kzg_verify_cell_scratch_bytes(c.cn));
        const uint8_t *dci = c.in(B_G1INF, commitment_inf, c.c0, c.cn), *dpi = c.in(B_G2INF, proof_inf, c.c0, c.cn);
        CUT(launch_cells_verify(ctx, c.d, s->devs[c.dev], dc, dci, didx, dcells, dpf, dpi, c.cn, dst, dscr, c.d.d_err, c.st));
        c.out(B_FLAG, out_status + c.c0, dst, c.cn);
    });
}

int32_t zkp_kzg_compute_cells_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, size_t n, uint8_t *d_cells,
                                  uint8_t *d_status, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_cells(ctx, s);
    if (rc) return rc;
    if (n && (!d_blobs || !d_cells || !d_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_blobs & 15) || ((uintptr_t)d_cells & 15)) return fail(ZKP_ERR_INVALID_ARG, "d_blobs and d_cells must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_cells(ctx, s->devs[dev], d_blobs, n, d_cells, nullptr, nullptr, d_status, nullptr, st));
        return ZKP_OK;
    });
}

int32_t zkp_kzg_compute_cells_and_proofs_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, size_t n,
                                             uint8_t *d_cells, uint64_t *d_proofs, uint8_t *d_proof_inf, uint8_t *d_status, void *d_scratch,
                                             void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_cells(ctx, s);
    if (rc) return rc;
    if (n && (!d_blobs || !d_cells || !d_proofs || !d_proof_inf || !d_status || !d_scratch)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_blobs & 15) || ((uintptr_t)d_cells & 15) || ((uintptr_t)d_scratch & 15))
        return fail(ZKP_ERR_INVALID_ARG, "d_blobs, d_cells and d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_cells(ctx, s->devs[dev], d_blobs, n, d_cells, d_proofs, d_proof_inf, d_status, d_scratch, st));
        return ZKP_OK;
    });
}

// recovery runs one cluster of two blocks with 128 KiB of shared memory each per blob: refuse (never substitute) a device
// on which no such cluster can be resident; dev < 0: every device of the context
static int32_t check_recover(zkp_ctx *ctx, const zkp_kzg_setup *s, int32_t dev) {
    int32_t rc = check_cells(ctx, s);
    if (rc) return rc;
    for (size_t di = 0; di < s->devs.size(); di++) {
        if (dev >= 0 && (size_t)dev != di) continue;
        const KzgDev &k = s->devs[di];
        if (k.recover_clusters < 1)
            return fail(ZKP_ERR_CUDA, "k_cells_recover cannot run on device " + std::to_string(ctx->devs[di].id) +
                                          ": no cluster of two 512-thread blocks with 128 KiB of shared memory each can be resident (" +
                                          (k.recover_err != cudaSuccess ? cudaGetErrorString(k.recover_err) : "0 active clusters") + ")");
    }
    return ZKP_OK;
}

int32_t zkp_kzg_recover_cells_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *cell_indices, const uint8_t *cells,
                                    const uint64_t *num_cells, size_t n, uint8_t *out_cells, uint8_t *out_status) {
    int32_t rc = check_recover(ctx, s, -1);
    if (rc) return rc;
    if (n && (!cell_indices || !cells || !num_cells || !out_cells || !out_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return cells_job(ctx, s, nullptr, cell_indices, cells, num_cells, n, out_cells, nullptr, nullptr, out_status);
}

int32_t zkp_kzg_recover_cells_and_proofs_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *cell_indices, const uint8_t *cells,
                                               const uint64_t *num_cells, size_t n, uint8_t *out_cells, uint64_t *out_proofs,
                                               uint8_t *out_proof_inf, uint8_t *out_status) {
    int32_t rc = check_recover(ctx, s, -1);
    if (rc) return rc;
    if (n && (!cell_indices || !cells || !num_cells || !out_cells || !out_proofs || !out_proof_inf || !out_status))
        return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    return cells_job(ctx, s, nullptr, cell_indices, cells, num_cells, n, out_cells, out_proofs, out_proof_inf, out_status);
}

int32_t zkp_kzg_recover_cells_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_cell_indices, const uint8_t *d_cells,
                                  const uint64_t *d_num_cells, size_t n, uint8_t *d_out_cells, uint8_t *d_status, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_recover(ctx, s, dev);
    if (rc) return rc;
    if (n && (!d_cell_indices || !d_cells || !d_num_cells || !d_out_cells || !d_status)) return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_cells & 15) || ((uintptr_t)d_out_cells & 15)) return fail(ZKP_ERR_INVALID_ARG, "d_cells and d_out_cells must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_cells_recover(ctx, s->devs[dev], d_cell_indices, d_cells, d_num_cells, n, d_out_cells, nullptr, nullptr, d_status, nullptr,
                                st));
        return ZKP_OK;
    });
}

int32_t zkp_kzg_recover_cells_and_proofs_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_cell_indices,
                                             const uint8_t *d_cells, const uint64_t *d_num_cells, size_t n, uint8_t *d_out_cells,
                                             uint64_t *d_proofs, uint8_t *d_proof_inf, uint8_t *d_status, void *d_scratch, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_recover(ctx, s, dev);
    if (rc) return rc;
    if (n && (!d_cell_indices || !d_cells || !d_num_cells || !d_out_cells || !d_proofs || !d_proof_inf || !d_status || !d_scratch))
        return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_cells & 15) || ((uintptr_t)d_out_cells & 15) || ((uintptr_t)d_scratch & 15))
        return fail(ZKP_ERR_INVALID_ARG, "d_cells, d_out_cells and d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_cells_recover(ctx, s->devs[dev], d_cell_indices, d_cells, d_num_cells, n, d_out_cells, d_proofs, d_proof_inf, d_status, d_scratch,
                                st));
        return ZKP_OK;
    });
}

int32_t zkp_kzg_verify_cell_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_commitments, const uint8_t *d_commitment_inf,
                                const uint64_t *d_cell_indices, const uint8_t *d_cells, const uint64_t *d_proofs, const uint8_t *d_proof_inf,
                                size_t n, uint8_t *d_status, void *d_scratch, void *stream) {
    int32_t rc = check_dev(ctx, dev);
    if (rc == ZKP_OK) rc = check_cells(ctx, s);
    if (rc) return rc;
    if (n && (!d_commitments || !d_cell_indices || !d_cells || !d_proofs || !d_status || !d_scratch))
        return fail(ZKP_ERR_INVALID_ARG, "NULL buffer");
    if (((uintptr_t)d_cells & 15) || ((uintptr_t)d_scratch & 15)) return fail(ZKP_ERR_INVALID_ARG, "d_cells and d_scratch must be 16-byte aligned");
    return on_device(ctx, dev, stream, [&](DevState &d, cudaStream_t st) {
        CU(launch_cells_verify(ctx, d, s->devs[dev], d_commitments, d_commitment_inf, d_cell_indices, d_cells, d_proofs, d_proof_inf, n, d_status,
                               d_scratch, nullptr, st));
        return ZKP_OK;
    });
}

// ------------------------------------------------------------------ measurement

int32_t zkp_imad_peak(zkp_ctx *ctx, int32_t dev, int32_t kind, double *macs_per_second) {
    int32_t rc = check_dev(ctx, dev);
    if (rc) return rc;
    if (!macs_per_second || kind < 0 || kind > 2) return fail(ZKP_ERR_INVALID_ARG, "bad kind / NULL out");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DevState &d = ctx->devs[dev];
    DeviceGuard guard;
    CU(cudaSetDevice(d.id));
    cudaStream_t st = d.stream[0];
    uint32_t *sink = d.d_err;
    // every issued multiply is counted (the multiplicand update is a shift + add on the ALU pipe); the launch
    // geometry is swept and the best sustained rate is the roofline denominator
    const int iters = 1 << 13;
    const double per_thread = (double)iters * (kind == 2 ? 12.0 : 8.0);
    static const int geom[][2] = {{8, 256}, {4, 256}, {16, 128}, {8, 128}, {4, 512}};   // blocks per SM, threads per block
    struct EventPair {   // destroyed on every exit path
        cudaEvent_t a = nullptr, b = nullptr;
        ~EventPair() {
            if (a) cudaEventDestroy(a);
            if (b) cudaEventDestroy(b);
        }
    } ev;
    CU(cudaEventCreate(&ev.a));
    CU(cudaEventCreate(&ev.b));
    double best_rate = 0;
    for (const auto &g : geom) {
        const int blocks = d.sms * g[0], threads = g[1];
        for (int rep = 0; rep < 3; rep++) {
            CU(cudaEventRecord(ev.a, st));
            if (kind == 0) k_imad_peak<0><<<blocks, threads, 0, st>>>(sink + 0, iters);
            else if (kind == 1) k_imad_peak<1><<<blocks, threads, 0, st>>>(sink + 0, iters);
            else k_imad_peak<2><<<blocks, threads, 0, st>>>(sink + 0, iters);
            ctx->launches++;
            CU(cudaEventRecord(ev.b, st));
            CU(cudaEventSynchronize(ev.b));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, ev.a, ev.b));
            double rate = per_thread * blocks * threads / (ms * 1e-3);
            if (rep > 0 && rate > best_rate) best_rate = rate;
        }
    }
    CU(cudaMemsetAsync(d.d_err, 0, sizeof(uint32_t), st));
    CU(cudaStreamSynchronize(st));
    *macs_per_second = best_rate;
    return ZKP_OK;
}

}  // extern "C"
