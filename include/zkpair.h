/*
 * zkpair.h -- C ABI of the B200-native batched BLS12-381 pairing engine (libzkpair.so).
 *
 * This is the drop-in boundary for the pairing hot path of 0xWOLAND/zkvm-pairings.  Citations are
 * into /root/reference/ (the Rust crate being replaced on this path).
 *
 * What it replaces
 *   - the per-operation accelerator boundary the reference has today, the SP1 zkVM precompile FFI
 *       bls12381_sys_bigint(result:&mut[u32;12], op:u32 /0=mul,1=add/, lhs:&[u32;12], rhs:&[u32;12])   src/fp.rs:376,443
 *       syscall_bls12381_fp_mulmod(lhs:*mut u32, rhs:*const u32)                                       src/fp.rs:126
 *     -> zkp_fp_mul_batch / zkp_tower_op_batch (same canonical 12xu32 = 6xu64 little-endian limbs,
 *        but batched so one call amortises the launch); zkp_sys_bigint / zkp_syscall_fp_mulmod keep the
 *        precompiles' one-operation shape for code that is not batched yet;
 *   - the tower methods on the path (Fp/Fp2/Fp6/Fp12 mul, square, invert, frobenius_map, conjugate,
 *     mul_by_1 / mul_by_01 / mul_by_014: src/fp2.rs:147-313, src/fp6.rs:102-309, src/fp12.rs:99-210)
 *     -> zkp_tower_op_batch with the ZKP_OP_* code of the method;
 *   - the module the reference declares but leaves EMPTY (src/lib.rs:12, src/pairings.rs = 0 bytes):
 *     pairing / miller_loop / multi_miller_loop / final_exponentiation and the batch entry points
 *     the north star adds -> zkp_miller_loop_batch, zkp_final_exp_batch, zkp_pairing_batch,
 *     zkp_multi_miller_loop_batch, zkp_multi_pairing_batch, zkp_multi_miller_product.
 *
 * Conventions
 *   - Every function returns int32_t: ZKP_OK (0) or a negative ZKP_ERR_* code; zkp_last_error()
 *     returns a thread-local message.  Nothing panics or aborts.  There is NO CPU fallback: with no
 *     CUDA device zkp_ctx_create fails with ZKP_ERR_NO_DEVICE.
 *   - The caller owns every buffer.  Element layout is array-of-structs of canonical (non-
 *     Montgomery, value in [0,p)) little-endian u64 limbs, exactly `Fp.0` (src/fp.rs:24):
 *       Fp = 6 u64; Fp2 = c0|c1 (12); Fp6 = c0|c1|c2 (36); Fp12 / Gt = c0|c1 (72 u64 = 576 bytes);
 *       G1 point = x|y (12 u64), G2 point = x.c0|x.c1|y.c0|y.c1 (24 u64); the `is_infinity` flag of
 *       G1Affine/G2Affine (src/g1.rs:7-11, src/g2.rs:8-12) travels in a separate uint8_t array
 *       (NULL = no point is at infinity).  A pair with either point at infinity contributes
 *       Fp12::one() (zkcrypto lineage behaviour).
 *   - Inputs with a limb vector >= p are rejected with ZKP_ERR_NONCANONICAL (the reference's neg is
 *     undefined there, src/fp.rs:383-405); outputs are then unspecified.
 *   - Host entry points (no suffix) copy host->device, run, copy device->host, and shard the batch
 *     in contiguous slices over the devices of the context (one host thread and two streams per device,
 *     2^18-element chunks double-buffered).  Pinned (page-locked or registered) caller buffers are used in
 *     place; pageable ones are staged through pinned memory so that copies and kernels still overlap.  *_dev entry points take DEVICE
 *     pointers valid on device `dev` (an index into the context's device list), enqueue on
 *     `stream` (a cudaStream_t; NULL = the legacy default stream, as everywhere in CUDA, so the launch is
 *     ordered after the caller's earlier default-stream work) and return without synchronising; their
 *     error/status words are device resident.  Every entry point restores the caller's current device.
 *   - Calls on one zkp_ctx are serialised by an internal mutex; distinct contexts are independent.
 *   - include/zkpair.hpp is a header-only C++17 mirror of the crate's value types (Fp .. Fp12, G1Affine,
 *     G2Affine, pairings::*) over these entry points.
 */
#ifndef ZKPAIR_H
#define ZKPAIR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZKP_OK 0
#define ZKP_ERR_INVALID_ARG (-1)
#define ZKP_ERR_CUDA (-2)
#define ZKP_ERR_NONCANONICAL (-3)
#define ZKP_ERR_NO_DEVICE (-4)
#define ZKP_ERR_TOO_MANY_PAIRS (-5)

#define ZKP_MAX_PAIRS_PER_CHECK 8

/* element-wise tower operations (zkp_tower_op_batch); reference method in the comment */
enum zkp_tower_op {
    ZKP_OP_FP_ADD = 0,        /* Fp::add            src/fp.rs:351-368 */
    ZKP_OP_FP_SUB = 1,        /* Fp::sub            src/fp.rs:407-411 */
    ZKP_OP_FP_NEG = 2,        /* Fp::neg            src/fp.rs:381-405 */
    ZKP_OP_FP_MUL = 3,        /* Fp::mul            src/fp.rs:413-434 */
    ZKP_OP_FP_SQR = 4,        /* Fp::square         src/fp.rs:452-455 */
    ZKP_OP_FP_INV = 5,        /* Fp::invert         src/fp.rs:306-319 (status bit1 set for zero) */
    ZKP_OP_FP_POW = 6,        /* Fp::pow_vartime    src/fp.rs:264-276; b = exponent, six RAW little-endian u64 */
    ZKP_OP_FP_SQRT = 7,       /* Fp::sqrt           src/fp.rs:280-300 (status bit1 set for a non-residue = Err(())) */
    ZKP_OP_FP2_ADD = 16, ZKP_OP_FP2_SUB = 17, ZKP_OP_FP2_NEG = 18,
    ZKP_OP_FP2_MUL = 19,      /* src/fp2.rs:192-209 */
    ZKP_OP_FP2_SQR = 20,      /* src/fp2.rs:171-189 */
    ZKP_OP_FP2_INV = 21,      /* src/fp2.rs:278-296 */
    ZKP_OP_FP2_MUL_NR = 22,   /* mul_by_nonresidue  src/fp2.rs:161-168 */
    ZKP_OP_FP2_CONJ = 23,     /* conjugate = frobenius_map  src/fp2.rs:147-157 */
    ZKP_OP_FP2_POW = 24,      /* Fp2::pow_vartime   src/fp2.rs:301-313; b = exponent, six raw u64 */
    ZKP_OP_FP6_ADD = 32, ZKP_OP_FP6_SUB = 33, ZKP_OP_FP6_NEG = 34,
    ZKP_OP_FP6_MUL = 35,      /* src/fp6.rs:188-267 */
    ZKP_OP_FP6_SQR = 36,      /* src/fp6.rs:274-288 */
    ZKP_OP_FP6_INV = 37,      /* src/fp6.rs:291-309 */
    ZKP_OP_FP6_MUL_NR = 38,   /* src/fp6.rs:128-139 */
    ZKP_OP_FP6_FROB = 39,     /* TRUE a^p; src/fp6.rs:142-176 has wrong constants (SURVEY 0.5) */
    ZKP_OP_FP6_MUL_BY_1 = 40, /* b = c1 (Fp2)            src/fp6.rs:102-108 */
    ZKP_OP_FP6_MUL_BY_01 = 41,/* b = c0|c1 (2 Fp2)       src/fp6.rs:110-125 */
    ZKP_OP_FP12_ADD = 48, ZKP_OP_FP12_SUB = 49, ZKP_OP_FP12_NEG = 50,
    ZKP_OP_FP12_MUL = 51,     /* src/fp12.rs:193-210 */
    ZKP_OP_FP12_SQR = 52,     /* src/fp12.rs:173-184 */
    ZKP_OP_FP12_INV = 53,     /* src/fp12.rs:186-190 */
    ZKP_OP_FP12_CONJ = 54,    /* src/fp12.rs:123-125 */
    ZKP_OP_FP12_FROB = 55,    /* TRUE a^p (src/fp12.rs:143-170 inherits the Fp6 defect) */
    ZKP_OP_FP12_MUL_BY_014 = 56, /* b = c0|c1|c4 (3 Fp2) src/fp12.rs:99-111 */
    ZKP_OP_FP12_CYC_SQR = 57, /* Granger-Scott cyclotomic squaring (SURVEY 9.2) */
    ZKP_OP_FP12_CYC_EXP = 58, /* f^x for the curve parameter x (negative): conj(f^|x|) */
    ZKP_OP_FP12_FROB2 = 59,   /* a^(p^2) */
    ZKP_OP_FP12_FROB3 = 60,   /* a^(p^3) */
    ZKP_OP_FP12_POW = 61      /* Fp12::pow_vartime  src/fp12.rs:127-139; b = exponent, six raw u64 */
};

typedef struct zkp_ctx zkp_ctx;

/* ---- context ------------------------------------------------------------------------------ */

/* Number of CUDA devices visible (0 when there is none / no driver). */
int32_t zkp_device_count(void);
/* devices == NULL or n_devices <= 0: use every visible device.  Fails with ZKP_ERR_NO_DEVICE when
 * no CUDA device is usable (there is no CPU path). */
int32_t zkp_ctx_create(const int *devices, int n_devices, zkp_ctx **out);
void zkp_ctx_destroy(zkp_ctx *ctx);
int32_t zkp_ctx_num_devices(const zkp_ctx *ctx);
/* Thread-local description of the last error returned to this thread. */
const char *zkp_last_error(void);
/* Library / build description string (arch, launch geometry). */
const char *zkp_version(void);

/* ---- tower operations (parity / test surface for the tower rows of SURVEY 8a) -------------- */

/* out[i] = op(a[i], b[i]).  b may be NULL for unary ops.  status (optional, n bytes): bit0 =
 * non-canonical input, bit1 = inverse of zero requested (the reference returns None; out = 0). */
int32_t zkp_tower_op_batch(zkp_ctx *ctx, int32_t op, const uint64_t *a, const uint64_t *b,
                           uint64_t *out, uint8_t *status, size_t n);
/* Named wrappers for the three ops SURVEY 8b lists. */
int32_t zkp_fp_mul_batch(zkp_ctx *ctx, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n);
int32_t zkp_fp12_mul_batch(zkp_ctx *ctx, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n);
int32_t zkp_fp12_mul_by_014_batch(zkp_ctx *ctx, const uint64_t *f, const uint64_t *c0_c1_c4,
                                  uint64_t *out, size_t n);

/* Scalar drop-ins with the argument meaning of the reference's zkVM precompile FFI (sp1_zkvm::syscalls, called at
 * src/fp.rs:126, :376, :443): ONE Fp operation on twelve little-endian u32 limbs (= the transmuted [u64; 6] of
 * src/fp.rs:124-128), canonical in and out.  zkp_sys_bigint: op 0 = lhs * rhs mod p (src/fp.rs:443), op 1 = lhs + rhs
 * mod p (src/fp.rs:376), written to `result` (which may alias an operand).  zkp_syscall_fp_mulmod: lhs <- lhs * rhs
 * mod p in place (src/fp.rs:126).  ctx = NULL uses a process-wide context on device 0, created on first use (the
 * precompiles carry no handle); unlike the precompiles they return a status (limbs >= p: ZKP_ERR_NONCANONICAL).
 * One launch per call: they exist so that the crate's `cfg(target_os = "zkvm")` bodies link unchanged; anything
 * hot belongs on the batch entry points. */
int32_t zkp_sys_bigint(zkp_ctx *ctx, uint32_t *result, uint32_t op, const uint32_t *lhs, const uint32_t *rhs);
int32_t zkp_syscall_fp_mulmod(zkp_ctx *ctx, uint32_t *lhs, const uint32_t *rhs);

/* ---- pairing path (host buffers) ---------------------------------------------------------- */

/* n independent Miller loops: out_fp12[i] = miller_loop(G1[i], G2[i])   (SURVEY 9.1 convention) */
int32_t zkp_miller_loop_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf,
                              const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n, uint64_t *out_fp12);
/* out_fp12[i] = in_fp12[i]^((p^12-1)/r) (SURVEY 9.2) */
int32_t zkp_final_exp_batch(zkp_ctx *ctx, const uint64_t *in_fp12, size_t n, uint64_t *out_fp12);
/* out_gt[i] = e(G1[i], G2[i]).  Points must be curve points (zkp_g1_check_batch / zkp_g2_check_batch validate them): the
 * fused path uses line steps that rely on the curve equation, so for off-curve inputs -- where no pairing is defined -- it need
 * not agree with zkp_final_exp_batch(zkp_miller_loop_batch(.)), which applies SURVEY 9.1's formulas to whatever it is given. */
int32_t zkp_pairing_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf,
                          const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n, uint64_t *out_gt);
/* n_checks checks of pairs_per_check (<= ZKP_MAX_PAIRS_PER_CHECK) pairs each, stored check-major;
 * every check runs ONE shared-accumulator Miller loop over its pairs. */
int32_t zkp_multi_miller_loop_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf,
                                    const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n_checks,
                                    int32_t pairs_per_check, uint64_t *out_fp12);
/* ... followed by one final exponentiation per check.  out_is_one (optional, n_checks bytes) is 1
 * where the product of pairings equals Gt one (e.g. a Groth16 verification equation holds). */
int32_t zkp_multi_pairing_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf,
                                const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n_checks,
                                int32_t pairs_per_check, uint64_t *out_gt, uint8_t *out_is_one);
/* prod_i e(G1[i], G2[i]) for one large product: per-device shared-accumulator Miller loops (four pairs per
 * loop) over a contiguous slice, streamed in double-buffered chunks, per-device Fp12 partial product, gather
 * of the 576-byte partials to the first device, multiply, ONE final exponentiation.  out_miller_product
 * (optional) receives the un-exponentiated product in SURVEY 9.1's line scaling (a field element: independent of the
 * grouping and of the number of devices); with out_miller_product == NULL the cheaper line steps are used. */
int32_t zkp_multi_miller_product(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf,
                                 const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n,
                                 uint64_t *out_miller_product, uint64_t *out_gt);

/* ---- device-resident entry points (asynchronous; pointers are device pointers on `dev`) ---- */

/* mode: 1 = Miller loop only, 2 = final exponentiation only (d_in_fp12 -> d_out), 3 = pairing, 5 = Miller loop whose
 * output is only meant for a later final exponentiation (or for products of such outputs): it equals the mode-1 value up
 * to a factor from a proper subfield, which the final exponentiation removes -- the cheaper homogeneous line steps the
 * fused pairing path uses (mode 3 == mode 2 after mode 1 == mode 2 after mode 5, bit for bit).
 * d_err (optional): device uint32_t that is OR-ed with 1 when an input is non-canonical. */
int32_t zkp_pairing_dev(zkp_ctx *ctx, int32_t dev, int32_t mode, const uint64_t *d_g1_xy,
                        const uint8_t *d_g1_inf, const uint64_t *d_g2_xy, const uint8_t *d_g2_inf,
                        size_t n_checks, int32_t pairs_per_check, const uint64_t *d_in_fp12,
                        uint64_t *d_out, uint8_t *d_is_one, uint32_t *d_err, void *stream);
int32_t zkp_tower_op_dev(zkp_ctx *ctx, int32_t dev, int32_t op, const uint64_t *d_a, const uint64_t *d_b,
                         uint64_t *d_out, uint8_t *d_status, uint32_t *d_err, size_t n, void *stream);
/* d_out (72 u64) = product of the n Fp12 elements at d_in (canonical limbs); d_scratch must hold
 * zkp_product_scratch_elems(n) * 72 u64. */
size_t zkp_product_scratch_elems(size_t n);
int32_t zkp_fp12_product_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_in, size_t n,
                             uint64_t *d_scratch, uint64_t *d_out, uint32_t *d_err, void *stream);
/* Synthetic valid inputs: G1[i] = a_i * G1gen, G2[i] = b_i * G2gen with 64-bit scalars
 * a_i = splitmix64(seed, 2*(first+i)), b_i = splitmix64(seed, 2*(first+i)+1) (zero mapped to 1). */
int32_t zkp_gen_points_dev(zkp_ctx *ctx, int32_t dev, uint64_t seed, uint64_t first, size_t n,
                           uint64_t *d_g1_xy, uint8_t *d_g1_inf, uint64_t *d_g2_xy, uint8_t *d_g2_inf,
                           void *stream);
/* Host-buffer version of the generator. */
int32_t zkp_gen_points(zkp_ctx *ctx, uint64_t seed, uint64_t first, size_t n, uint64_t *g1_xy,
                       uint8_t *g1_inf, uint64_t *g2_xy, uint8_t *g2_inf);

/* ---- prepared G2 points (SURVEY 8f; `G2Prepared` of the zkcrypto lineage, absent from the reference) --
 * The 68 line-coefficient triples the Miller loop derives from a G2 point (63 doubling + 5 addition
 * steps), computed once for points that are fixed across checks -- the verifying-key points of a
 * Groth16-style check -- so that those pairs skip the G2 arithmetic in every check.  A table is an
 * opaque blob of ZKP_G2_PREPARED_U64 u64 per point in the library's internal (Montgomery) limb format,
 * valid for this build of the library only; results are bit-identical to the unprepared calls. */
#define ZKP_G2_PREPARED_U64 (68 * 3 * 12)
int32_t zkp_g2_prepare_batch(zkp_ctx *ctx, const uint64_t *g2_xy, size_t n, uint64_t *out_tables);
int32_t zkp_g2_prepare_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g2_xy, size_t n, uint64_t *d_out_tables,
                           uint32_t *d_err, void *stream);
/* n_checks products of k pairs with a shared final exponentiation, like zkp_multi_pairing_batch, where
 * the LAST kf pairs of every check take their G2 point from `tables` (kf tables shared by all checks;
 * tables_inf = their is_infinity flags or NULL) and only the first k - kf pairs have per-check G2
 * points: g1_xy holds n_checks * k points, g2_xy holds n_checks * (k - kf). */
int32_t zkp_multi_pairing_prepared_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf,
                                         const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n_checks,
                                         int32_t pairs_per_check, const uint64_t *tables, const uint8_t *tables_inf,
                                         int32_t prepared_pairs, uint64_t *out_gt, uint8_t *out_is_one);
int32_t zkp_multi_pairing_prepared_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g1_xy, const uint8_t *d_g1_inf,
                                       const uint64_t *d_g2_xy, const uint8_t *d_g2_inf, size_t n_checks,
                                       int32_t pairs_per_check, const uint64_t *d_tables, const uint8_t *d_tables_inf,
                                       int32_t prepared_pairs, uint64_t *d_out_gt, uint8_t *d_is_one, uint32_t *d_err,
                                       void *stream);

/* ---- byte (de)serialisation (SURVEY 8f) ----------------------------------------------------------
 * Fp::from_bytes (src/fp.rs:165-191): n x 48 big-endian bytes -> n x 6 little-endian u64 limbs;
 * ok[i] = 1 when the value is canonical (< p, the reference's Ok), 0 for the reference's Err(())
 * (the limbs are still written).  Fp::to_bytes (src/fp.rs:195-207) is the inverse, no check.  An Fp2 /
 * Fp6 / Fp12 / point is a run of Fp, so the same calls serialise them coefficient by coefficient. */
int32_t zkp_fp_from_bytes_batch(zkp_ctx *ctx, const uint8_t *bytes, size_t n, uint64_t *out_limbs, uint8_t *ok);
int32_t zkp_fp_to_bytes_batch(zkp_ctx *ctx, const uint64_t *limbs, size_t n, uint8_t *out_bytes);
/* device-resident form: dir 0 = from_bytes, 1 = to_bytes; buffers 16-byte aligned; d_ok may be NULL */
int32_t zkp_fp_bytes_dev(zkp_ctx *ctx, int32_t dev, int32_t dir, const void *d_in, void *d_out, uint8_t *d_ok,
                         size_t n, void *stream);

/* ---- group-level batch operations (the callers either side of a pairing, SURVEY 8f) ------------ */

/* status byte per point */
#define ZKP_POINT_OK 0                 /* G1Affine::is_valid / G2Affine::is_valid == Ok(())            */
#define ZKP_POINT_NOT_ON_CURVE 1       /* Err("Point is not on curve")        src/g1.rs:54, src/g2.rs:61 */
#define ZKP_POINT_NOT_TORSION_FREE 2   /* Err("Point is not torsion free")    src/g1.rs:57, src/g2.rs:64 */

/* G1Affine::is_valid (src/g1.rs:49-62): identity -> ok; y^2 = x^3 + 4 (src/g1.rs:95-101); subgroup test
 * -[x^2]P == (beta x, y) (src/g1.rs:103-115).  g1_inf may be NULL. */
int32_t zkp_g1_check_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf, size_t n, uint8_t *status);
/* G2Affine::is_valid (src/g2.rs:57-69): y^2 = x^3 + 4(1+u) (src/g2.rs:109-120); psi(Q) == -[|x|]Q
 * (src/g2.rs:126-170). */
int32_t zkp_g2_check_batch(zkp_ctx *ctx, const uint64_t *g2_xy, const uint8_t *g2_inf, size_t n, uint8_t *status);
/* [k_i]P_i, k_i = 4 little-endian u64 (the limbs of an Fr, src/fr.rs): `&G1Affine * &Fr` (src/g1.rs:130-153)
 * and `&G2Affine * &Fr` (src/g2.rs:185-208) as the correct double-and-add over all 256 bits (the reference's
 * G1 loop drops bit 0 of the scalar, src/g1.rs:138-142 -- deliberately not reproduced).  Results are affine;
 * the identity is (0, 1) with out_inf = 1 (src/g1.rs:25-31). */
int32_t zkp_g1_mul_batch(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf, const uint64_t *scalars,
                         size_t n, uint64_t *out_xy, uint8_t *out_inf);
int32_t zkp_g2_mul_batch(zkp_ctx *ctx, const uint64_t *g2_xy, const uint8_t *g2_inf, const uint64_t *scalars,
                         size_t n, uint64_t *out_xy, uint8_t *out_inf);

/* `&G1Affine + &G1Affine` (src/g1.rs:155-187, double() :74-91) and `&G2Affine + &G2Affine` (src/g2.rs:210-242,
 * :81-105): the affine chord-and-tangent law, element-wise a[i] + b[i].  An identity operand passes the other one
 * through, equal points double.  out_flag[i]: bit0 = the sum is the identity (0, 1); bit1 = the reference divides
 * by zero and panics here (P + (-P) src/g1.rs:177, or doubling a point with y = 0) -- the identity is returned.
 * `a - b` is a + (-b) with -b = (x, p - y) (src/g1.rs:118-128): negate on the host or with ZKP_OP_FP_NEG. */
int32_t zkp_g1_add_batch(zkp_ctx *ctx, const uint64_t *a_xy, const uint8_t *a_inf, const uint64_t *b_xy, const uint8_t *b_inf,
                         size_t n, uint64_t *out_xy, uint8_t *out_flag);
int32_t zkp_g2_add_batch(zkp_ctx *ctx, const uint64_t *a_xy, const uint8_t *a_inf, const uint64_t *b_xy, const uint8_t *b_inf,
                         size_t n, uint64_t *out_xy, uint8_t *out_flag);

/* ---- multi-scalar multiplication over caller-given points (blst p1s_mult_pippenger / p2s_mult_pippenger,
 * arkworks VariableBaseMSM; absent from the reference) ------------------------------------------------
 * sum_i [k_i]P_i over n caller-given points, one result per call (Pippenger with signed-digit buckets).
 * Points and scalars follow zkp_g1_mul_batch / zkp_g2_mul_batch: canonical affine limbs, g*_inf optional (a flagged
 * point contributes the identity), k_i = 4 little-endian u64 of ANY 256-bit value, taken as an integer and not
 * reduced mod r.  The result is exactly the group element sum_i [k_i]P_i, in the prime-order subgroup or not: no
 * endomorphism split is used, and subgroup membership is NOT checked (the sum is exact without it).  For subgroup
 * points it equals the sum with every k_i reduced mod r.
 * Output: one point, canonical affine x|y and out_inf; the identity is (0, 1) with out_inf = 1.  n = 0 gives the
 * identity, out_status = ZKP_POINT_OK and ZKP_OK.
 * Validation: a limb >= p fails the call with ZKP_ERR_NONCANONICAL (the _dev forms OR 1 into d_err instead).  An
 * unflagged point off its curve gives out_status = ZKP_POINT_NOT_ON_CURVE, zero limbs and out_inf = 1; the call still
 * returns ZKP_OK.  Otherwise out_status = ZKP_POINT_OK.
 * Host forms: the points shard in contiguous slices over the context's devices; each device's Jacobian partial is
 * gathered on the first device, so the affine result is the same for any number of devices.
 * _dev forms: asynchronous on `stream` with d_scratch of zkp_g*_msm_scratch_bytes(n) bytes, 16-byte aligned; d_err
 * may be NULL.  The caller's current device is restored. */
int32_t zkp_g1_msm(zkp_ctx *ctx, const uint64_t *g1_xy, const uint8_t *g1_inf, const uint64_t *scalars, size_t n,
                   uint64_t *out_xy, uint8_t *out_inf, uint8_t *out_status);
int32_t zkp_g2_msm(zkp_ctx *ctx, const uint64_t *g2_xy, const uint8_t *g2_inf, const uint64_t *scalars, size_t n,
                   uint64_t *out_xy, uint8_t *out_inf, uint8_t *out_status);
size_t zkp_g1_msm_scratch_bytes(size_t n);
size_t zkp_g2_msm_scratch_bytes(size_t n);
int32_t zkp_g1_msm_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g1_xy, const uint8_t *d_g1_inf, const uint64_t *d_scalars,
                       size_t n, uint64_t *d_out_xy, uint8_t *d_out_inf, uint8_t *d_status, uint32_t *d_err,
                       void *d_scratch, void *stream);
int32_t zkp_g2_msm_dev(zkp_ctx *ctx, int32_t dev, const uint64_t *d_g2_xy, const uint8_t *d_g2_inf, const uint64_t *d_scalars,
                       size_t n, uint64_t *d_out_xy, uint8_t *d_out_inf, uint8_t *d_status, uint32_t *d_err,
                       void *d_scratch, void *stream);

/* ---- Groth16 verification (one verdict per proof) ----------------------------------------------
 * Verifying key: alpha in G1; beta, gamma, delta in G2; IC_0 .. IC_l in G1 (l = n_public).  Proof: A in G1,
 * B in G2, C in G1.  Public inputs: x_1 .. x_l, each an Fr as four little-endian u64 limbs.  A proof is
 * accepted iff A, B, C are canonical, on their curves and in the prime-order subgroups (G1Affine::is_valid /
 * G2Affine::is_valid), every x_j < r, and e(A, B) = e(alpha, beta) e(L, gamma) e(C, delta) with
 * L = IC_0 + sum_j x_j IC_j -- the Groth16 equation, evaluated as the prepared 4-pair check
 * e(A,B) e(alpha,-beta) e(L,-gamma) e(C,-delta) == 1.  A proof point at infinity is a valid group element.
 *
 * Malformed proofs are PER-PROOF rejections (a status byte), not call errors: the call returns ZKP_OK and the
 * other proofs are unaffected -- unlike the ZKP_ERR_NONCANONICAL convention of the other entry points. */
#define ZKP_G16_VALID 0       /* all checks pass and the equation holds */
#define ZKP_G16_INVALID 1     /* well formed, the equation fails */
#define ZKP_G16_BAD_POINT 2   /* A, B or C has a limb >= p, is off its curve or is not torsion free (precedes 3) */
#define ZKP_G16_BAD_INPUT 3   /* some x_j >= r */
#define ZKP_GROTH16_PROOF_U64 48   /* A.x|A.y | B.x.c0|B.x.c1|B.y.c0|B.y.c1 | C.x|C.y */
/* Public inputs per key.  The key keeps a fixed-base window table per IC_j on every device of its context: 32 x 255
 * affine points, 765 KiB per input, so 200 MB per device at the bound (and as much again while it is built). */
#define ZKP_GROTH16_MAX_PUBLIC 256

typedef struct zkp_groth16_vk zkp_groth16_vk;

/* Validates every key point on the GPU and builds the resident key on every device of ctx: the prepared tables of
 * -beta, -gamma, -delta and the window tables of IC_1 .. IC_l.  ic_g1 holds n_public + 1 points, ic_inf their
 * is_infinity flags or NULL (an identity IC_j is allowed and contributes nothing).  alpha, beta, gamma, delta have no
 * infinity flag: the identity is not a valid key point.  A limb >= p gives ZKP_ERR_NONCANONICAL; an off-curve or
 * non-subgroup point or n_public outside 0 .. ZKP_GROTH16_MAX_PUBLIC gives ZKP_ERR_INVALID_ARG, the message naming
 * the point.  The key belongs to ctx: other contexts reject it, and it must be destroyed before ctx. */
int32_t zkp_groth16_vk_create(zkp_ctx *ctx, const uint64_t *alpha_g1, const uint64_t *beta_g2, const uint64_t *gamma_g2,
                              const uint64_t *delta_g2, const uint64_t *ic_g1, const uint8_t *ic_inf, int32_t n_public,
                              zkp_groth16_vk **out);
void zkp_groth16_vk_destroy(zkp_groth16_vk *vk);
/* n proofs (n x ZKP_GROTH16_PROOF_U64 u64), proof_inf = n x 3 flags (A, B, C) or NULL, public_inputs = n x n_public
 * x 4 u64 (may be NULL when n_public = 0) -> out_status[i] = ZKP_G16_*.  Sharded over the context's devices in
 * contiguous slices, double-buffered chunks of at most 2^18 proofs and 64 MB of public inputs. */
int32_t zkp_groth16_verify_batch(zkp_ctx *ctx, const zkp_groth16_vk *vk, const uint64_t *proofs, const uint8_t *proof_inf,
                                 const uint64_t *public_inputs, size_t n, uint8_t *out_status);
/* Bytes of d_scratch zkp_groth16_verify_dev needs for n proofs (the assembled pairs, Gt outputs and is_one). */
size_t zkp_groth16_scratch_bytes(size_t n);
/* Device-resident form on device `dev` of the key's context; asynchronous, same buffer layouts; d_scratch
 * 16-byte aligned. */
int32_t zkp_groth16_verify_dev(zkp_ctx *ctx, int32_t dev, const zkp_groth16_vk *vk, const uint64_t *d_proofs,
                               const uint8_t *d_proof_inf, const uint64_t *d_public_inputs, size_t n, uint8_t *d_status,
                               void *d_scratch, void *stream);

/* ---- KZG point-evaluation verification (one verdict per proof) ----------------------------------
 * EIP-4844's verify_kzg_proof(C, z, y, pi) on the library's limb boundary.  Setup: [tau]G2.  Proof: commitment C in
 * G1, evaluation point z and claimed value y (each an Fr as four little-endian u64 limbs), opening proof pi in G1.
 * A proof is accepted iff C and pi are canonical, on the curve and torsion free (G1Affine::is_valid), z < r, y < r
 * and e(C - [y]G1, G2) = e(pi, [tau]G2 - [z]G2), evaluated as the prepared 2-pair check
 * e(C + [z]pi - [y]G1, G2) e(pi, -[tau]G2) == 1 (G1, G2 the standard generators).  C or pi at infinity is a valid
 * group element.  As for Groth16, malformed proofs are per-proof rejections and the call returns ZKP_OK. */
#define ZKP_KZG_VALID 0        /* all checks pass and the equation holds */
#define ZKP_KZG_INVALID 1      /* well formed, the equation fails */
#define ZKP_KZG_BAD_POINT 2    /* C or pi has a limb >= p, is off the curve or is not torsion free (precedes 3) */
#define ZKP_KZG_BAD_SCALAR 3   /* z >= r or y >= r */
#define ZKP_KZG_BAD_CELLS 4    /* cell recovery: a cell count outside [64, 128], indices not strictly ascending or one >= 128 (precedes 3) */
#define ZKP_KZG_PROOF_U64 24   /* C.x|C.y | pi.x|pi.y */

typedef struct zkp_kzg_setup zkp_kzg_setup;

/* Validates [tau]G2 on the GPU and builds the resident setup on every device of ctx: the prepared tables of G2 and
 * -[tau]G2, a fixed-base window table of G1 (32 x 255 affine points, 765 KiB) and the 4096-point evaluation domain of
 * zkp_kzg_verify_blob_batch (128 KiB).  There is no infinity flag: the
 * identity is not a valid setup.  A limb >= p gives ZKP_ERR_NONCANONICAL; an off-curve or non-subgroup point gives
 * ZKP_ERR_INVALID_ARG, the message naming tau_g2.  The setup belongs to ctx: other contexts reject it, and it must be
 * destroyed before ctx. */
int32_t zkp_kzg_setup_create(zkp_ctx *ctx, const uint64_t *tau_g2, zkp_kzg_setup **out);
void zkp_kzg_setup_destroy(zkp_kzg_setup *s);
/* n proofs (n x ZKP_KZG_PROOF_U64 u64), proof_inf = n x 2 flags (C, pi) or NULL, zy = n x 8 u64 (z | y) ->
 * out_status[i] = ZKP_KZG_*.  Sharded over the context's devices in contiguous slices, double-buffered chunks of at
 * most 2^18 proofs. */
int32_t zkp_kzg_verify_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *proofs, const uint8_t *proof_inf,
                             const uint64_t *zy, size_t n, uint8_t *out_status);
/* Bytes of d_scratch zkp_kzg_verify_dev needs for n proofs (the pairs [P, pi], their flags, Gt outputs and is_one). */
size_t zkp_kzg_scratch_bytes(size_t n);
/* Device-resident form on device `dev` of the setup's context; asynchronous, same buffer layouts; d_scratch
 * 16-byte aligned; stream NULL = the legacy default stream. */
int32_t zkp_kzg_verify_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_proofs, const uint8_t *d_proof_inf,
                           const uint64_t *d_zy, size_t n, uint8_t *d_status, void *d_scratch, void *stream);

/* ---- EIP-4844 blob verification (one verdict per blob) -------------------------------------------
 * verify_blob_kzg_proof(blob, C, pi) of the consensus specs (deneb polynomial-commitments.md) on the GPU: z is the
 * Fiat-Shamir challenge SHA-256(b"FSBLOBVERIFY_V1_" | 4096 as 16 big-endian bytes | blob | compressed C) mod r, y the
 * blob's polynomial (its 4096 big-endian elements are the values at the bit-reversed roots of unity of order 4096)
 * evaluated at z, and the verdict is that of zkp_kzg_verify_batch for (C, z, y, pi).  C and pi cross the boundary as
 * affine limbs with infinity flags, as for zkp_kzg_verify_batch; the compressed encoding of C that the transcript
 * hashes is derived on the device.  Verdicts are ZKP_KZG_*; z and y are derived here, so ZKP_KZG_BAD_SCALAR means
 * that some blob element is >= r (ZKP_KZG_BAD_POINT takes precedence).  The call returns ZKP_OK for malformed blobs
 * and proofs.  A blob is 128 KiB: the host path streams double-buffered chunks of at most 2^14 blobs (2 GiB) per
 * device, so a large batch takes up to 2 x 2 GiB of device buffers per device, and pageable blobs are staged through up
 * to 2 x 2 GiB of pinned memory per device (smaller batches take proportionally less). */
#define ZKP_BLOB_FIELD_ELEMENTS 4096
#define ZKP_BLOB_BYTES (32 * ZKP_BLOB_FIELD_ELEMENTS)
/* n blobs (n x ZKP_BLOB_BYTES), proofs / proof_inf exactly as zkp_kzg_verify_batch (C | pi) -> out_status[i] = ZKP_KZG_*.
 * out_zy (optional, n x 8 u64) receives the derived z | y; for a blob with an element >= r it holds r | 0, so
 * zkp_kzg_verify_batch(proofs, out_zy) reproduces out_status in every slot. */
int32_t zkp_kzg_verify_blob_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *proofs,
                                  const uint8_t *proof_inf, size_t n, uint8_t *out_status, uint64_t *out_zy);
/* Bytes of d_scratch zkp_kzg_verify_blob_dev needs for n blobs (z | y, then zkp_kzg_scratch_bytes(n)). */
size_t zkp_kzg_blob_scratch_bytes(size_t n);
/* Device-resident form on device `dev` of the setup's context; asynchronous, same buffer layouts; d_blobs and d_scratch
 * 16-byte aligned; d_out_zy optional; stream NULL = the legacy default stream. */
int32_t zkp_kzg_verify_blob_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, const uint64_t *d_proofs,
                                const uint8_t *d_proof_inf, size_t n, uint8_t *d_status, uint64_t *d_out_zy, void *d_scratch,
                                void *stream);

/* ---- EIP-4844 commitments and proofs (one status per blob) ---------------------------------------
 * blob_to_kzg_commitment, compute_kzg_proof and compute_blob_kzg_proof of the consensus specs (deneb
 * polynomial-commitments.md) on the GPU.  A commitment is C = sum_i p_i L_brp(i) over the blob's elements p_i and the
 * setup's Lagrange points in bit-reversed order; a proof is pi = sum_i q_i L_brp(i) over the quotient
 * q_i = (p_i - y) / (omega_i - z) of compute_kzg_proof_impl (for z = omega_m, q_m is compute_quotient_eval_within_domain
 * and y = p_m).  Points leave as canonical affine limbs x|y with an infinity flag; the identity is (0, 1) with the flag
 * set.  Statuses are ZKP_KZG_*: ZKP_KZG_VALID (0) when the point was computed, ZKP_KZG_BAD_SCALAR when a blob element
 * (or z) is >= r, ZKP_KZG_BAD_POINT when the commitment given to compute_blob_kzg_proof is non-canonical, off the curve
 * or not torsion free (precedes BAD_SCALAR).  A rejected slot holds zero limbs with its flag set (and y = 0); the call
 * returns ZKP_OK.  The host path streams double-buffered chunks of at most 2^14 blobs per device, like
 * zkp_kzg_verify_blob_batch; a proof chunk also holds its 4096 quotient scalars per blob (128 KiB), so a large proof
 * batch takes up to 2 x 4 GiB of device buffers per device (commitments 2 x 2 GiB), plus the resident setup. */

/* zkp_kzg_setup_create plus the 4096 G1 Lagrange points of the trusted setup, g1_lagrange = 4096 x 12 u64 (canonical
 * x|y, no infinity flags) in the natural order of the setup file, L_k = [l_k(tau)]G1 at omega^k; the library applies
 * the bit-reversal permutation itself.  Every point is validated on the GPU (a limb >= p gives ZKP_ERR_NONCANONICAL; an
 * off-curve or non-subgroup point ZKP_ERR_INVALID_ARG, the message naming its index), and the points are checked
 * against tau_g2 with one MSM and one pairing check: sum_k L_k = G1 and e(sum_k omega^k L_k, G2) = e(G1, [tau]G2).
 * A mismatch (a wrong order, a wrong tau, a truncated file) gives ZKP_ERR_INVALID_ARG "g1_lagrange is inconsistent
 * with tau_g2".  The setup verifies exactly as one from zkp_kzg_setup_create; it also holds, on every device of ctx,
 * signed-digit window tables of the Lagrange points: 4096 x 32 windows x 128 affine points, 1 610 612 736 bytes
 * (1.5 GiB) per device on top of the verifier's 1.0 MiB.  Creation takes about 400 MiB of temporary device memory. */
int32_t zkp_kzg_setup_create_prover(zkp_ctx *ctx, const uint64_t *tau_g2, const uint64_t *g1_lagrange, zkp_kzg_setup **out);
/* n blobs (n x ZKP_BLOB_BYTES) -> commitments out_c (n x 12 u64), out_c_inf (n), out_status (n).  The prover calls fail
 * with ZKP_ERR_INVALID_ARG on a setup made without Lagrange points. */
int32_t zkp_kzg_blob_to_commitment_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, size_t n, uint64_t *out_c,
                                         uint8_t *out_c_inf, uint8_t *out_status);
/* n blobs and evaluation points z (n x 4 u64, Fr limbs) -> proofs (n x 12 u64, flags), y = p(z) (n x 4 u64) and statuses. */
int32_t zkp_kzg_compute_proof_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *z, size_t n,
                                    uint64_t *out_proof, uint8_t *out_proof_inf, uint64_t *out_y, uint8_t *out_status);
/* n blobs and their commitments (n x 12 u64, commitment_inf n flags or NULL) -> proofs (n x 12 u64, flags) and statuses;
 * z is the transcript's challenge, as in zkp_kzg_verify_blob_batch.  out_zy (optional, n x 8 u64) receives z | y in the
 * convention of zkp_kzg_verify_blob_batch. */
int32_t zkp_kzg_compute_blob_proof_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, const uint64_t *commitments,
                                         const uint8_t *commitment_inf, size_t n, uint64_t *out_proof, uint8_t *out_proof_inf,
                                         uint8_t *out_status, uint64_t *out_zy);
/* Bytes of d_scratch the two proof _dev forms need for n blobs (the quotient rows, then z | y); commitments need none. */
size_t zkp_kzg_prover_scratch_bytes(size_t n);
/* Device-resident forms on device `dev` of the setup's context; asynchronous, same buffer layouts; d_blobs and
 * d_scratch 16-byte aligned; stream NULL = the legacy default stream. */
int32_t zkp_kzg_blob_to_commitment_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, size_t n,
                                       uint64_t *d_c, uint8_t *d_c_inf, uint8_t *d_status, void *stream);
int32_t zkp_kzg_compute_proof_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, const uint64_t *d_z, size_t n,
                                  uint64_t *d_proof, uint8_t *d_proof_inf, uint64_t *d_y, uint8_t *d_status, void *d_scratch, void *stream);
int32_t zkp_kzg_compute_blob_proof_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, const uint64_t *d_commitments,
                                       const uint8_t *d_commitment_inf, size_t n, uint64_t *d_proof, uint8_t *d_proof_inf, uint8_t *d_status,
                                       uint64_t *d_out_zy, void *d_scratch, void *stream);

/* ---- EIP-7594 cells and cell proofs (one status per blob or per cell) -----------------------------
 * compute_cells, compute_cells_and_kzg_proofs and the per-cell check of verify_cell_kzg_proof_batch of the consensus
 * specs (fulu polynomial-commitments-sampling.md) on the GPU.  The extended blob is the blob's polynomial evaluated over
 * the 8192nd roots of unity in bit-reversed order, cut into 128 cells of 64 big-endian elements (2048 bytes); cells
 * 0 .. 63 are the blob's own bytes.  Proof k is [q_k(tau)]G1 over the monomial setup, q_k = p div (X^64 - c_k) with
 * c_k = h_k^64 and h_k the first point of cell k.  A cell is accepted iff C and pi are canonical, on the curve and
 * torsion free, every element is < r, the index is < 128 and e(C + [c_k]pi - [I_k(tau)]G1, G2) e(pi, -[tau^64]G2) == 1,
 * I_k = the cell's interpolation polynomial.  Statuses are ZKP_KZG_*: ZKP_KZG_BAD_SCALAR for a blob or cell element
 * >= r or a cell index >= 128, ZKP_KZG_BAD_POINT for C or pi (precedes BAD_SCALAR).  The spec's boolean for a batch is
 * the AND of the cells' statuses being ZKP_KZG_VALID.  A rejected blob's slots hold zero cells and proofs of zero limbs
 * with the flag set; the calls return ZKP_OK for malformed blobs and cells.
 * Host paths stream double-buffered chunks per device: at most 2^11 blobs for cells (2 x 768 MiB of device buffers),
 * 2^7 blobs with proofs (128 quotient rows of 128 KiB per blob: 2 x 2.2 GiB) and 2^16 cells for verification
 * (2 x 180 MiB), plus the resident setup. */
#define ZKP_CELLS_PER_EXT_BLOB 128
#define ZKP_FIELD_ELEMENTS_PER_CELL 64
#define ZKP_CELL_BYTES (32 * ZKP_FIELD_ELEMENTS_PER_CELL)

/* The EIP-7594 trusted setup: g2_monomial = 65 G2 points [tau^i]G2 (65 x 24 u64), g1_monomial = 4096 G1 points
 * [tau^i]G1 (4096 x 12 u64) and, optionally, g1_lagrange as for zkp_kzg_setup_create_prover (NULL: the setup cannot run
 * the EIP-4844 prover calls).  Builds everything zkp_kzg_setup_create builds, with tau_g2 = g2_monomial[1], plus the
 * prepared table of -[tau^64]G2, the twiddles of the extended domain (256 KiB) and signed-digit window tables of the
 * monomial points (1.5 GiB per device, like the Lagrange tables).  Every point is validated on the GPU (a limb >= p
 * gives ZKP_ERR_NONCANONICAL; an off-curve or non-subgroup point ZKP_ERR_INVALID_ARG naming its index); then
 * g1_monomial[0] must be G1, g2_monomial[0] must be G2, e(M_{i+1}, G2) = e(M_i, g2_monomial[1]) for i < 4095 and
 * e(M_i, G2) = e(G1, g2_monomial[i]) for i <= 64 (ZKP_ERR_INVALID_ARG naming the first point that fails).  The cells
 * calls fail with ZKP_ERR_INVALID_ARG on setups made otherwise. */
int32_t zkp_kzg_setup_create_cells(zkp_ctx *ctx, const uint64_t *g2_monomial, const uint64_t *g1_monomial, const uint64_t *g1_lagrange,
                                   zkp_kzg_setup **out);
/* n blobs (n x ZKP_BLOB_BYTES) -> out_cells (n x 128 x ZKP_CELL_BYTES) and out_status (n). */
int32_t zkp_kzg_compute_cells_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, size_t n, uint8_t *out_cells,
                                    uint8_t *out_status);
/* n blobs -> out_cells, out_proofs (n x 128 x 12 u64), out_proof_inf (n x 128) and out_status (n). */
int32_t zkp_kzg_compute_cells_and_proofs_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint8_t *blobs, size_t n, uint8_t *out_cells,
                                               uint64_t *out_proofs, uint8_t *out_proof_inf, uint8_t *out_status);
/* n cells: commitments (n x 12 u64, commitment_inf n flags or NULL), cell_indices (n), cells (n x ZKP_CELL_BYTES),
 * proofs (n x 12 u64, proof_inf n flags or NULL) -> out_status[i] = ZKP_KZG_*. */
int32_t zkp_kzg_verify_cell_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *commitments, const uint8_t *commitment_inf,
                                  const uint64_t *cell_indices, const uint8_t *cells, const uint64_t *proofs, const uint8_t *proof_inf, size_t n,
                                  uint8_t *out_status);
/* Bytes of d_scratch zkp_kzg_compute_cells_and_proofs_dev needs for n blobs (coefficients, quotient rows and their
 * statuses: about 16 MiB per blob); zkp_kzg_compute_cells_dev needs none. */
size_t zkp_kzg_cells_proofs_scratch_bytes(size_t n);
/* Bytes of d_scratch zkp_kzg_verify_cell_dev needs for n cells (zkp_kzg_scratch_bytes(n), then [I_k(tau)]G1). */
size_t zkp_kzg_verify_cell_scratch_bytes(size_t n);
/* Device-resident forms on device `dev` of the setup's context; asynchronous, same buffer layouts; d_blobs, d_cells and
 * d_scratch 16-byte aligned; stream NULL = the legacy default stream. */
int32_t zkp_kzg_compute_cells_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, size_t n, uint8_t *d_cells,
                                  uint8_t *d_status, void *stream);
int32_t zkp_kzg_compute_cells_and_proofs_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint8_t *d_blobs, size_t n,
                                             uint8_t *d_cells, uint64_t *d_proofs, uint8_t *d_proof_inf, uint8_t *d_status, void *d_scratch,
                                             void *stream);
int32_t zkp_kzg_verify_cell_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_commitments, const uint8_t *d_commitment_inf,
                                const uint64_t *d_cell_indices, const uint8_t *d_cells, const uint64_t *d_proofs, const uint8_t *d_proof_inf,
                                size_t n, uint8_t *d_status, void *d_scratch, void *stream);

/* recover_cells_and_kzg_proofs: any 64 or more cells of each of n blobs -> all 128 cells (and proofs), exactly as the
 * spec's recover_polynomialcoeff (coset shift 7) followed by compute_cells_and_kzg_proofs, for consistent and
 * inconsistent cells alike.  Blob b's input is cell_indices[128 b ..] (n x 128 u64), cells[128 b ..] (n x 128 x
 * ZKP_CELL_BYTES) and num_cells[b]: its first num_cells[b] entries are the spec's cell_indices and cells, the entries
 * after them are ignored.  Outputs are those of zkp_kzg_compute_cells_and_proofs_batch.  Statuses per blob:
 * ZKP_KZG_BAD_CELLS for a count outside [64, 128], indices not strictly ascending (duplicates included) or an index
 * >= 128, else ZKP_KZG_BAD_SCALAR for an element >= r in a given cell; a rejected blob gets zero cells (and proofs of
 * zero limbs with the flag set) and the call returns ZKP_OK.  Each blob is one cluster of two thread blocks with 128 KiB
 * of shared memory each; a device on which no such cluster can be resident fails the call with ZKP_ERR_CUDA.  Host
 * paths stream double-buffered chunks per device of at most 2^11 blobs (512 MiB of cells in and out per buffer set),
 * 2^7 with proofs.  All four need a setup from zkp_kzg_setup_create_cells. */
int32_t zkp_kzg_recover_cells_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *cell_indices, const uint8_t *cells,
                                    const uint64_t *num_cells, size_t n, uint8_t *out_cells, uint8_t *out_status);
int32_t zkp_kzg_recover_cells_and_proofs_batch(zkp_ctx *ctx, const zkp_kzg_setup *s, const uint64_t *cell_indices, const uint8_t *cells,
                                               const uint64_t *num_cells, size_t n, uint8_t *out_cells, uint64_t *out_proofs,
                                               uint8_t *out_proof_inf, uint8_t *out_status);
/* Device-resident forms, conventions as zkp_kzg_compute_cells_dev; d_cells, d_out_cells and d_scratch 16-byte aligned;
 * the proof form takes zkp_kzg_cells_proofs_scratch_bytes(n) bytes of d_scratch. */
int32_t zkp_kzg_recover_cells_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_cell_indices, const uint8_t *d_cells,
                                  const uint64_t *d_num_cells, size_t n, uint8_t *d_out_cells, uint8_t *d_status, void *stream);
int32_t zkp_kzg_recover_cells_and_proofs_dev(zkp_ctx *ctx, int32_t dev, const zkp_kzg_setup *s, const uint64_t *d_cell_indices,
                                             const uint8_t *d_cells, const uint64_t *d_num_cells, size_t n, uint8_t *d_out_cells,
                                             uint64_t *d_proofs, uint8_t *d_proof_inf, uint8_t *d_status, void *d_scratch, void *stream);

/* ---- measurement helpers -------------------------------------------------------------------- */

/* Integer-multiply roofline probe: runs independent IMAD.WIDE.U32 (kind 0), IMAD lo (kind 1) or
 * carry-chained IMAD.WIDE.U32.X (kind 2) chains on every SM of device `dev` and reports the
 * sustained rate in multiply-accumulates per second (CUDA-event timed). */
int32_t zkp_imad_peak(zkp_ctx *ctx, int32_t dev, int32_t kind, double *macs_per_second);
/* Number of kernel launches issued by this context so far (for bench.py's gpu_launches). */
uint64_t zkp_launch_count(const zkp_ctx *ctx);
/* Name and average duration (ms, CUDA events on the launching stream) of the most recent timed
 * pairing-path kernel on device `dev`; timing is enabled with zkp_set_kernel_timing(ctx, 1). */
int32_t zkp_set_kernel_timing(zkp_ctx *ctx, int32_t enabled);
int32_t zkp_last_kernel_ms(zkp_ctx *ctx, int32_t dev, double *total_ms, uint64_t *launches);

#ifdef __cplusplus
}
#endif
#endif /* ZKPAIR_H */
