"""Host-side driver of the CUDA pairing engine (thin layer over the C ABI in include/zkpair.h).

Host buffers are numpy ``uint64`` arrays of canonical little-endian limbs in the reference's
``Fp.0`` layout (/root/reference/src/fp.rs:24):  Fp (n,6) - Fp2 (n,12) - Fp6 (n,36) - Fp12/Gt (n,72)
- G1 (n,12) = x|y - G2 (n,24) = x.c0|x.c1|y.c0|y.c1, infinity flags ``uint8`` (n,).
Device buffers are torch CUDA tensors with the same layout (any 8-byte dtype).

No CPU fallback: constructing an engine without libzkpair.so or without a CUDA device raises.
"""
from __future__ import annotations

import ctypes
import weakref
from typing import Optional, Sequence

import numpy as np

from . import _lib

TOWER_OPS = {
    "fp_add": 0, "fp_sub": 1, "fp_neg": 2, "fp_mul": 3, "fp_sqr": 4, "fp_inv": 5, "fp_pow": 6, "fp_sqrt": 7,
    "fp2_add": 16, "fp2_sub": 17, "fp2_neg": 18, "fp2_mul": 19, "fp2_sqr": 20, "fp2_inv": 21,
    "fp2_mul_nr": 22, "fp2_conj": 23, "fp2_pow": 24,
    "fp6_add": 32, "fp6_sub": 33, "fp6_neg": 34, "fp6_mul": 35, "fp6_sqr": 36, "fp6_inv": 37,
    "fp6_mul_nr": 38, "fp6_frob": 39, "fp6_mul_by_1": 40, "fp6_mul_by_01": 41,
    "fp12_add": 48, "fp12_sub": 49, "fp12_neg": 50, "fp12_mul": 51, "fp12_sqr": 52, "fp12_inv": 53,
    "fp12_conj": 54, "fp12_frob": 55, "fp12_mul_by_014": 56, "fp12_cyc_sqr": 57, "fp12_cyc_exp": 58,
    "fp12_frob2": 59, "fp12_frob3": 60, "fp12_pow": 61,
}
# operand b that is not of the same shape as a: sparse multipliers, and the RAW six-limb exponent of pow
_B_WIDTH = {"fp6_mul_by_1": 2, "fp6_mul_by_01": 4, "fp12_mul_by_014": 6, "fp_pow": 1, "fp2_pow": 1, "fp12_pow": 1}
_BINARY = {"add", "sub", "mul"}

MODE_MILLER, MODE_FINAL_EXP, MODE_PAIRING = 1, 2, 3
MODE_MILLER_FOR_FINAL_EXP = 5   # Miller loop whose output only feeds a final exponentiation (free line scaling, cheaper)

# per-proof verdicts of groth16_verify_batch / groth16_verify_dev (include/zkpair.h ZKP_G16_*)
G16_VALID, G16_INVALID, G16_BAD_POINT, G16_BAD_INPUT = 0, 1, 2, 3
GROTH16_PROOF_U64 = 48
GROTH16_MAX_PUBLIC = 256
# per-proof verdicts of kzg_verify_batch / kzg_verify_dev (include/zkpair.h ZKP_KZG_*)
KZG_VALID, KZG_INVALID, KZG_BAD_POINT, KZG_BAD_SCALAR = 0, 1, 2, 3
KZG_BAD_CELLS = 4         # cell recovery: a bad cell count or bad cell indices (include/zkpair.h ZKP_KZG_BAD_CELLS)
KZG_PROOF_U64 = 24
BLOB_N = 4096            # EIP-4844 FIELD_ELEMENTS_PER_BLOB (include/zkpair.h ZKP_BLOB_FIELD_ELEMENTS)
BLOB_BYTES = 32 * BLOB_N   # one EIP-4844 blob: 4096 big-endian field elements (include/zkpair.h ZKP_BLOB_BYTES)
CELLS_PER_EXT_BLOB = 128            # EIP-7594 (include/zkpair.h ZKP_CELLS_PER_EXT_BLOB)
FIELD_ELEMENTS_PER_CELL = 64        # include/zkpair.h ZKP_FIELD_ELEMENTS_PER_CELL
CELL_BYTES = 32 * FIELD_ELEMENTS_PER_CELL   # include/zkpair.h ZKP_CELL_BYTES


class ZkpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("zkpair error %d: %s" % (code, msg))
        self.code = code


class NonCanonicalError(ZkpError, ValueError):
    """An input limb vector is >= p (the reference rejects these in Fp::from_bytes, src/fp.rs:165-191)."""


def op_widths(name: str):
    """(#Fp of operand a, #Fp of operand b or 0, #Fp of the result) for a tower op name."""
    w = 1 if name.startswith("fp_") else 2 if name.startswith("fp2_") else 6 if name.startswith("fp6_") else 12
    if name in _B_WIDTH:
        return w, _B_WIDTH[name], w
    suffix = name.split("_", 1)[1]
    return w, (w if suffix in _BINARY else 0), w


def _np64(a, width):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.reshape(-1, width)


def _np8(a, n):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.uint8).reshape(-1)
    if a.shape[0] != n:
        raise ValueError("infinity flag array has %d entries, expected %d" % (a.shape[0], n))
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _dptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class _ContextObject:
    """Device memory that belongs to one engine's context (a C handle freed by ``_destroy``).  It holds a reference
    to its engine, so the engine's context outlives it; ``close()`` (or leaving a ``with`` block) frees the device
    memory, and the engine closes it first when the engine itself is closed."""
    _destroy = ""
    _what = ""

    def __init__(self, engine: "PairingEngine", handle: ctypes.c_void_p):
        self.engine, self._h = engine, handle
        engine._resident.add(self)

    @property
    def handle(self):
        if not self._h:
            raise ValueError("the %s is closed" % self._what)
        return self._h

    def close(self):
        if getattr(self, "_h", None):
            getattr(self.engine._lib, self._destroy)(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class Groth16VerifyingKey(_ContextObject):
    """A verifying key resident on every device of one engine (PairingEngine.groth16_prepare_vk)."""
    _destroy = "zkp_groth16_vk_destroy"
    _what = "verifying key"

    def __init__(self, engine: "PairingEngine", handle: ctypes.c_void_p, n_public: int):
        super().__init__(engine, handle)
        self.n_public = n_public


class KzgSetup(_ContextObject):
    """A KZG setup ([tau]G2) resident on every device of one engine (PairingEngine.kzg_setup)."""
    _destroy = "zkp_kzg_setup_destroy"
    _what = "KZG setup"


class PairingEngine:
    """One C-ABI context: a set of CUDA devices with their streams and scratch buffers."""

    def __init__(self, devices: Optional[Sequence[int]] = None):
        self._lib = _lib.load()
        self._resident = weakref.WeakSet()   # verifying keys and KZG setups of this context: freed before the context is
        self._ctx = ctypes.c_void_p()
        if devices is None:
            arr, n = None, 0
        else:
            arr = (ctypes.c_int * len(devices))(*devices)
            n = len(devices)
        rc = self._lib.zkp_ctx_create(arr, n, ctypes.byref(self._ctx))
        self._check(rc)

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc: int):
        if rc == _lib.ZKP_OK:
            return
        msg = (self._lib.zkp_last_error() or b"").decode()
        if rc == _lib.ZKP_ERR_NONCANONICAL:
            raise NonCanonicalError(rc, msg)
        raise ZkpError(rc, msg)

    def close(self):
        for obj in list(getattr(self, "_resident", ())):
            obj.close()
        if getattr(self, "_ctx", None):
            self._lib.zkp_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def num_devices(self) -> int:
        return self._lib.zkp_ctx_num_devices(self._ctx)

    @property
    def launch_count(self) -> int:
        return int(self._lib.zkp_launch_count(self._ctx))

    def version(self) -> str:
        return self._lib.zkp_version().decode()

    # ------------------------------------------------------------------ tower ops (host buffers)
    def tower_op(self, name: str, a, b=None, return_status: bool = False):
        """out[i] = op(a[i], b[i]) for the tower method ``name`` (see TOWER_OPS)."""
        na, nb, nr = op_widths(name)
        a = _np64(a, 6 * na)
        n = a.shape[0]
        if nb:
            if b is None:
                raise ValueError("%s needs a second operand" % name)
            b = _np64(b, 6 * nb)
            if b.shape[0] != n:
                raise ValueError("operand batch sizes differ")
        else:
            b = None
        out = np.empty((n, 6 * nr), dtype=np.uint64)
        status = np.zeros(n, dtype=np.uint8)
        self._check(self._lib.zkp_tower_op_batch(self._ctx, TOWER_OPS[name], _ptr(a), _ptr(b), _ptr(out), _ptr(status), n))
        return (out, status) if return_status else out

    def fp_mul_batch(self, a, b):
        a, b = _np64(a, 6), _np64(b, 6)
        out = np.empty_like(a)
        self._check(self._lib.zkp_fp_mul_batch(self._ctx, _ptr(a), _ptr(b), _ptr(out), a.shape[0]))
        return out

    def sys_bigint(self, op: int, lhs, rhs, use_default_ctx: bool = False):
        """The reference's zkVM precompile `bls12381_sys_bigint` (src/fp.rs:376,443): ONE Fp operation on twelve
        little-endian u32 limbs, op 0 = mul, 1 = add.  use_default_ctx passes ctx = NULL (the process-wide context)."""
        lhs = np.ascontiguousarray(lhs, dtype=np.uint32).reshape(12)
        rhs = np.ascontiguousarray(rhs, dtype=np.uint32).reshape(12)
        out = np.zeros(12, dtype=np.uint32)
        self._check(self._lib.zkp_sys_bigint(None if use_default_ctx else self._ctx, _ptr(out), op, _ptr(lhs), _ptr(rhs)))
        return out

    def syscall_fp_mulmod(self, lhs, rhs, use_default_ctx: bool = False):
        """`syscall_bls12381_fp_mulmod` (src/fp.rs:126): lhs <- lhs * rhs mod p IN PLACE (lhs must be a uint32[12] array)."""
        if not (isinstance(lhs, np.ndarray) and lhs.dtype == np.uint32 and lhs.size == 12 and lhs.flags["C_CONTIGUOUS"]):
            raise ValueError("lhs must be a contiguous uint32[12] array (updated in place)")
        rhs = np.ascontiguousarray(rhs, dtype=np.uint32).reshape(12)
        self._check(self._lib.zkp_syscall_fp_mulmod(None if use_default_ctx else self._ctx, _ptr(lhs), _ptr(rhs)))
        return lhs

    def fp12_mul_batch(self, a, b):
        a, b = _np64(a, 72), _np64(b, 72)
        out = np.empty_like(a)
        self._check(self._lib.zkp_fp12_mul_batch(self._ctx, _ptr(a), _ptr(b), _ptr(out), a.shape[0]))
        return out

    def fp12_mul_by_014_batch(self, f, c0_c1_c4):
        f, c = _np64(f, 72), _np64(c0_c1_c4, 36)
        out = np.empty_like(f)
        self._check(self._lib.zkp_fp12_mul_by_014_batch(self._ctx, _ptr(f), _ptr(c), _ptr(out), f.shape[0]))
        return out

    # ------------------------------------------------------------------ pairing path (host buffers)
    def _points(self, g1, g2, g1_inf, g2_inf):
        g1, g2 = _np64(g1, 12), _np64(g2, 24)
        if g1.shape[0] != g2.shape[0]:
            raise ValueError("G1 and G2 batches differ in length")
        n = g1.shape[0]
        return g1, g2, _np8(g1_inf, n), _np8(g2_inf, n), n

    def miller_loop_batch(self, g1, g2, g1_inf=None, g2_inf=None):
        g1, g2, i1, i2, n = self._points(g1, g2, g1_inf, g2_inf)
        out = np.empty((n, 72), dtype=np.uint64)
        self._check(self._lib.zkp_miller_loop_batch(self._ctx, _ptr(g1), _ptr(i1), _ptr(g2), _ptr(i2), n, _ptr(out)))
        return out

    def final_exponentiation_batch(self, f):
        f = _np64(f, 72)
        out = np.empty_like(f)
        self._check(self._lib.zkp_final_exp_batch(self._ctx, _ptr(f), f.shape[0], _ptr(out)))
        return out

    def pairing_batch(self, g1, g2, g1_inf=None, g2_inf=None, out=None):
        g1, g2, i1, i2, n = self._points(g1, g2, g1_inf, g2_inf)
        if out is None:
            out = np.empty((n, 72), dtype=np.uint64)
        assert out.shape == (n, 72) and out.dtype == np.uint64 and out.flags.c_contiguous
        self._check(self._lib.zkp_pairing_batch(self._ctx, _ptr(g1), _ptr(i1), _ptr(g2), _ptr(i2), n, _ptr(out)))
        return out

    def multi_miller_loop_batch(self, g1, g2, pairs_per_check: int, g1_inf=None, g2_inf=None):
        g1, g2, i1, i2, n = self._points(g1, g2, g1_inf, g2_inf)
        if pairs_per_check < 1 or n % pairs_per_check:
            raise ValueError("number of pairs is not a multiple of pairs_per_check")
        nc = n // pairs_per_check
        out = np.empty((nc, 72), dtype=np.uint64)
        self._check(self._lib.zkp_multi_miller_loop_batch(self._ctx, _ptr(g1), _ptr(i1), _ptr(g2), _ptr(i2), nc, pairs_per_check, _ptr(out)))
        return out

    def multi_pairing_batch(self, g1, g2, pairs_per_check: int, g1_inf=None, g2_inf=None):
        """-> (gt (n_checks,72), is_one (n_checks,) uint8)."""
        g1, g2, i1, i2, n = self._points(g1, g2, g1_inf, g2_inf)
        if pairs_per_check < 1 or n % pairs_per_check:
            raise ValueError("number of pairs is not a multiple of pairs_per_check")
        nc = n // pairs_per_check
        out = np.empty((nc, 72), dtype=np.uint64)
        is_one = np.zeros(nc, dtype=np.uint8)
        self._check(self._lib.zkp_multi_pairing_batch(self._ctx, _ptr(g1), _ptr(i1), _ptr(g2), _ptr(i2), nc, pairs_per_check,
                                                      _ptr(out), _ptr(is_one)))
        return out, is_one

    def multi_miller_product(self, g1, g2, g1_inf=None, g2_inf=None, want_miller_product: bool = True):
        """One product over ALL pairs (sharded over the devices) -> (miller_product (72,), gt (72,)).  With
        ``want_miller_product=False`` only Gt is computed (-> (None, gt)) and the cheaper line steps are used."""
        g1, g2, i1, i2, n = self._points(g1, g2, g1_inf, g2_inf)
        ml, gt = (np.empty(72, dtype=np.uint64) if want_miller_product else None), np.empty(72, dtype=np.uint64)
        self._check(self._lib.zkp_multi_miller_product(self._ctx, _ptr(g1), _ptr(i1), _ptr(g2), _ptr(i2), n, _ptr(ml), _ptr(gt)))
        return ml, gt

    def gen_points(self, seed: int, first: int, n: int):
        """Synthetic valid inputs a_i*G1gen, b_i*G2gen (scalars from SplitMix64) -> g1, g1_inf, g2, g2_inf."""
        g1, g2 = np.empty((n, 12), np.uint64), np.empty((n, 24), np.uint64)
        i1, i2 = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_gen_points(self._ctx, seed, first, n, _ptr(g1), _ptr(i1), _ptr(g2), _ptr(i2)))
        return g1, i1, g2, i2

    # ------------------------------------------------------------------ prepared G2 points (SURVEY 8f)
    G2_PREPARED_U64 = 68 * 3 * 12

    def g2_prepare_batch(self, g2):
        """Line tables ("G2Prepared") of fixed G2 points -> (n, 2448) uint64, opaque internal format."""
        pts, _, n = self._pts(g2, 24, None)
        out = np.empty((n, self.G2_PREPARED_U64), np.uint64)
        self._check(self._lib.zkp_g2_prepare_batch(self._ctx, _ptr(pts), n, _ptr(out)))
        return out

    def multi_pairing_prepared_batch(self, g1, g2, pairs_per_check: int, tables, g1_inf=None, g2_inf=None, tables_inf=None):
        """Like multi_pairing_batch, with the LAST len(tables) pairs of every check taking their G2 point from
        prepared tables shared by all checks; g2 holds only the per-check points."""
        tables = np.ascontiguousarray(tables, dtype=np.uint64).reshape(-1, self.G2_PREPARED_U64)
        kf, k = tables.shape[0], pairs_per_check
        g1, i1, n1 = self._pts(g1, 12, g1_inf)
        if k < 1 or kf > k or n1 % k:
            raise ValueError("bad pairs_per_check / number of G1 points")
        nc = n1 // k
        if kf < k:
            g2, i2, n2 = self._pts(g2, 24, g2_inf)
            if n2 != nc * (k - kf):
                raise ValueError("expected n_checks * (pairs_per_check - prepared) G2 points")
        else:
            g2, i2 = None, None
        ti = None if tables_inf is None else np.ascontiguousarray(tables_inf, dtype=np.uint8).reshape(kf)
        out, is_one = np.empty((nc, 72), np.uint64), np.zeros(nc, np.uint8)
        self._check(self._lib.zkp_multi_pairing_prepared_batch(self._ctx, _ptr(g1), _ptr(i1), _ptr(g2), _ptr(i2), nc, k, _ptr(tables),
                                                               _ptr(ti), kf, _ptr(out), _ptr(is_one)))
        return out, is_one

    def g2_prepare_dev(self, d_g2, n: int, d_tables, err=None, stream: int = 0, dev: int = 0):
        self._check(self._lib.zkp_g2_prepare_dev(self._ctx, dev, _dptr(d_g2), n, _dptr(d_tables), _dptr(err), ctypes.c_void_p(stream)))

    def multi_pairing_prepared_dev(self, out, g1, g2, n_checks: int, pairs_per_check: int, d_tables, prepared_pairs: int, g1_inf=None,
                                   g2_inf=None, tables_inf=None, is_one=None, err=None, stream: int = 0, dev: int = 0):
        self._check(self._lib.zkp_multi_pairing_prepared_dev(self._ctx, dev, _dptr(g1), _dptr(g1_inf), _dptr(g2), _dptr(g2_inf), n_checks,
                                                             pairs_per_check, _dptr(d_tables), _dptr(tables_inf), prepared_pairs,
                                                             _dptr(out), _dptr(is_one), _dptr(err), ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ Groth16 verification
    def groth16_prepare_vk(self, alpha, beta, gamma, delta, ic, ic_inf=None) -> Groth16VerifyingKey:
        """Verifying key (alpha (12,), beta/gamma/delta (24,), ic (n_public + 1, 12)) -> a key validated and resident on
        the GPU.  Raises NonCanonicalError for a limb >= p, ZkpError (INVALID_ARG) for an invalid point."""
        a = np.ascontiguousarray(alpha, dtype=np.uint64).reshape(12)
        b, g, d = (np.ascontiguousarray(v, dtype=np.uint64).reshape(24) for v in (beta, gamma, delta))
        ic = np.ascontiguousarray(ic, dtype=np.uint64).reshape(-1, 12)
        n_public = ic.shape[0] - 1
        ii = _np8(ic_inf, ic.shape[0])
        h = ctypes.c_void_p()
        self._check(self._lib.zkp_groth16_vk_create(self._ctx, _ptr(a), _ptr(b), _ptr(g), _ptr(d), _ptr(ic), _ptr(ii), n_public,
                                                    ctypes.byref(h)))
        return Groth16VerifyingKey(self, h, n_public)

    def groth16_verify_batch(self, vk: Groth16VerifyingKey, proofs, public_inputs, proof_inf=None):
        """proofs (n, 48) = A | B | C, public_inputs (n, n_public, 4) Fr limbs, proof_inf (n, 3) or None ->
        uint8 (n,) verdicts G16_*."""
        pr = np.ascontiguousarray(proofs, dtype=np.uint64).reshape(-1, GROTH16_PROOF_U64)
        n = pr.shape[0]
        x = np.ascontiguousarray(public_inputs, dtype=np.uint64).reshape(n, vk.n_public * 4)
        pi = None if proof_inf is None else _np8(proof_inf, 3 * n)
        st = np.zeros(n, np.uint8)
        self._check(self._lib.zkp_groth16_verify_batch(self._ctx, vk.handle, _ptr(pr), _ptr(pi), _ptr(x), n, _ptr(st)))
        return st

    def groth16_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_groth16_scratch_bytes(n))

    def groth16_verify_dev(self, vk: Groth16VerifyingKey, d_proofs, d_public_inputs, n: int, d_status, d_scratch, d_proof_inf=None,
                           stream: int = 0, dev: int = 0):
        """Asynchronous form on device-resident torch tensors; d_scratch holds groth16_scratch_bytes(n) bytes."""
        self._check(self._lib.zkp_groth16_verify_dev(self._ctx, dev, vk.handle, _dptr(d_proofs), _dptr(d_proof_inf), _dptr(d_public_inputs),
                                                     n, _dptr(d_status), _dptr(d_scratch), ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ KZG point-evaluation verification
    def kzg_setup(self, tau_g2, g1_lagrange=None) -> KzgSetup:
        """[tau]G2 (24,) -> a setup validated and resident on the GPU.  Raises NonCanonicalError for a limb >= p,
        ZkpError (INVALID_ARG) for an off-curve or non-subgroup point.  With g1_lagrange, the 4096 G1 Lagrange points of
        the trusted setup (4096, 12) in the setup file's natural order, the setup can also prove (kzg_blob_to_commitment_batch,
        kzg_compute_proof_batch, kzg_compute_blob_proof_batch); points inconsistent with tau_g2 raise ZkpError."""
        t = np.ascontiguousarray(tau_g2, dtype=np.uint64).reshape(24)
        h = ctypes.c_void_p()
        if g1_lagrange is None:
            self._check(self._lib.zkp_kzg_setup_create(self._ctx, _ptr(t), ctypes.byref(h)))
        else:
            lag = np.ascontiguousarray(g1_lagrange, dtype=np.uint64).reshape(BLOB_N * 12)
            self._check(self._lib.zkp_kzg_setup_create_prover(self._ctx, _ptr(t), _ptr(lag), ctypes.byref(h)))
        return KzgSetup(self, h)

    def kzg_verify_batch(self, setup: KzgSetup, proofs, zy, proof_inf=None):
        """proofs (n, 24) = C | pi, zy (n, 8) = z | y Fr limbs, proof_inf (n, 2) or None -> uint8 (n,) verdicts KZG_*."""
        pr = np.ascontiguousarray(proofs, dtype=np.uint64).reshape(-1, KZG_PROOF_U64)
        n = pr.shape[0]
        s = np.ascontiguousarray(zy, dtype=np.uint64).reshape(n, 8)
        pi = None if proof_inf is None else _np8(proof_inf, 2 * n)
        st = np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_verify_batch(self._ctx, setup.handle, _ptr(pr), _ptr(pi), _ptr(s), n, _ptr(st)))
        return st

    def kzg_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_kzg_scratch_bytes(n))

    def kzg_verify_dev(self, setup: KzgSetup, d_proofs, d_zy, n: int, d_status, d_scratch, d_proof_inf=None, stream: int = 0,
                       dev: int = 0):
        """Asynchronous form on device-resident torch tensors; d_scratch holds kzg_scratch_bytes(n) bytes."""
        self._check(self._lib.zkp_kzg_verify_dev(self._ctx, dev, setup.handle, _dptr(d_proofs), _dptr(d_proof_inf), _dptr(d_zy), n,
                                                 _dptr(d_status), _dptr(d_scratch), ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ EIP-4844 blob verification
    def kzg_verify_blob_batch(self, setup: KzgSetup, blobs, proofs, proof_inf=None, return_zy: bool = False):
        """blobs (n, BLOB_BYTES) uint8, proofs (n, 24) = C | pi, proof_inf (n, 2) or None -> uint8 (n,) verdicts KZG_*
        (verify_blob_kzg_proof); with return_zy also the derived z | y (n, 8) (r | 0 for a blob with an element >= r)."""
        b = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, BLOB_BYTES)
        n = b.shape[0]
        pr = np.ascontiguousarray(proofs, dtype=np.uint64).reshape(n, KZG_PROOF_U64)
        pi = None if proof_inf is None else _np8(proof_inf, 2 * n)
        st = np.zeros(n, np.uint8)
        zy = np.zeros((n, 8), np.uint64) if return_zy else None
        self._check(self._lib.zkp_kzg_verify_blob_batch(self._ctx, setup.handle, _ptr(b), _ptr(pr), _ptr(pi), n, _ptr(st), _ptr(zy)))
        return (st, zy) if return_zy else st

    def kzg_blob_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_kzg_blob_scratch_bytes(n))

    def kzg_verify_blob_dev(self, setup: KzgSetup, d_blobs, d_proofs, n: int, d_status, d_scratch, d_proof_inf=None, d_out_zy=None,
                            stream: int = 0, dev: int = 0):
        """Asynchronous form on device-resident torch tensors; d_scratch holds kzg_blob_scratch_bytes(n) bytes, d_blobs
        and d_scratch 16-byte aligned."""
        self._check(self._lib.zkp_kzg_verify_blob_dev(self._ctx, dev, setup.handle, _dptr(d_blobs), _dptr(d_proofs), _dptr(d_proof_inf), n,
                                                      _dptr(d_status), _dptr(d_out_zy), _dptr(d_scratch), ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ EIP-4844 commitments and proofs
    def kzg_blob_to_commitment_batch(self, setup: KzgSetup, blobs):
        """blobs (n, BLOB_BYTES) -> (C (n, 12), C_inf (n,), status (n,)) (blob_to_kzg_commitment; KZG_BAD_SCALAR for an
        element >= r, with a zeroed slot)."""
        b = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, BLOB_BYTES)
        n = b.shape[0]
        c, ci, st = np.zeros((n, 12), np.uint64), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_blob_to_commitment_batch(self._ctx, setup.handle, _ptr(b), n, _ptr(c), _ptr(ci), _ptr(st)))
        return c, ci, st

    def kzg_compute_proof_batch(self, setup: KzgSetup, blobs, z):
        """blobs (n, BLOB_BYTES), z (n, 4) Fr limbs -> (pi (n, 12), pi_inf (n,), y (n, 4), status (n,)) (compute_kzg_proof)."""
        b = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, BLOB_BYTES)
        n = b.shape[0]
        zz = np.ascontiguousarray(z, dtype=np.uint64).reshape(n, 4)
        pr, pi, y, st = np.zeros((n, 12), np.uint64), np.zeros(n, np.uint8), np.zeros((n, 4), np.uint64), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_compute_proof_batch(self._ctx, setup.handle, _ptr(b), _ptr(zz), n, _ptr(pr), _ptr(pi), _ptr(y), _ptr(st)))
        return pr, pi, y, st

    def kzg_compute_blob_proof_batch(self, setup: KzgSetup, blobs, commitments, commitment_inf=None, return_zy: bool = False):
        """blobs (n, BLOB_BYTES), commitments (n, 12), commitment_inf (n,) or None -> (pi (n, 12), pi_inf (n,), status (n,))
        (compute_blob_kzg_proof), with return_zy also z | y (n, 8) as kzg_verify_blob_batch returns them."""
        b = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, BLOB_BYTES)
        n = b.shape[0]
        c = np.ascontiguousarray(commitments, dtype=np.uint64).reshape(n, 12)
        ci = _np8(commitment_inf, n)
        pr, pi, st = np.zeros((n, 12), np.uint64), np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        zy = np.zeros((n, 8), np.uint64) if return_zy else None
        self._check(self._lib.zkp_kzg_compute_blob_proof_batch(self._ctx, setup.handle, _ptr(b), _ptr(c), _ptr(ci), n, _ptr(pr), _ptr(pi),
                                                               _ptr(st), _ptr(zy)))
        return (pr, pi, st, zy) if return_zy else (pr, pi, st)

    def kzg_prover_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_kzg_prover_scratch_bytes(n))

    def kzg_blob_to_commitment_dev(self, setup: KzgSetup, d_blobs, n: int, d_c, d_c_inf, d_status, stream: int = 0, dev: int = 0):
        """Asynchronous form on device-resident torch tensors; d_blobs 16-byte aligned."""
        self._check(self._lib.zkp_kzg_blob_to_commitment_dev(self._ctx, dev, setup.handle, _dptr(d_blobs), n, _dptr(d_c), _dptr(d_c_inf),
                                                             _dptr(d_status), ctypes.c_void_p(stream)))

    def kzg_compute_proof_dev(self, setup: KzgSetup, d_blobs, d_z, n: int, d_proof, d_proof_inf, d_y, d_status, d_scratch, stream: int = 0,
                              dev: int = 0):
        """Asynchronous form; d_scratch holds kzg_prover_scratch_bytes(n) bytes, d_blobs and d_scratch 16-byte aligned."""
        self._check(self._lib.zkp_kzg_compute_proof_dev(self._ctx, dev, setup.handle, _dptr(d_blobs), _dptr(d_z), n, _dptr(d_proof),
                                                        _dptr(d_proof_inf), _dptr(d_y), _dptr(d_status), _dptr(d_scratch),
                                                        ctypes.c_void_p(stream)))

    def kzg_compute_blob_proof_dev(self, setup: KzgSetup, d_blobs, d_commitments, n: int, d_proof, d_proof_inf, d_status, d_scratch,
                                   d_commitment_inf=None, d_out_zy=None, stream: int = 0, dev: int = 0):
        """Asynchronous form; d_scratch holds kzg_prover_scratch_bytes(n) bytes, d_blobs and d_scratch 16-byte aligned."""
        self._check(self._lib.zkp_kzg_compute_blob_proof_dev(self._ctx, dev, setup.handle, _dptr(d_blobs), _dptr(d_commitments),
                                                             _dptr(d_commitment_inf), n, _dptr(d_proof), _dptr(d_proof_inf), _dptr(d_status),
                                                             _dptr(d_out_zy), _dptr(d_scratch), ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ EIP-7594 cells and cell proofs
    def kzg_setup_cells(self, g2_monomial, g1_monomial, g1_lagrange=None) -> KzgSetup:
        """The EIP-7594 trusted setup, g2_monomial (65, 24) = [tau^i]G2 and g1_monomial (4096, 12) = [tau^i]G1, validated and
        resident on the GPU; with g1_lagrange (4096, 12) as for kzg_setup the setup can also run the EIP-4844 prover.  It
        verifies as kzg_setup(g2_monomial[1]) does.  Raises NonCanonicalError for a limb >= p, ZkpError (INVALID_ARG) for
        an invalid or inconsistent point, naming it."""
        g2 = np.ascontiguousarray(g2_monomial, dtype=np.uint64).reshape((FIELD_ELEMENTS_PER_CELL + 1) * 24)
        g1 = np.ascontiguousarray(g1_monomial, dtype=np.uint64).reshape(BLOB_N * 12)
        lag = None if g1_lagrange is None else np.ascontiguousarray(g1_lagrange, dtype=np.uint64).reshape(BLOB_N * 12)
        h = ctypes.c_void_p()
        self._check(self._lib.zkp_kzg_setup_create_cells(self._ctx, _ptr(g2), _ptr(g1), _ptr(lag), ctypes.byref(h)))
        return KzgSetup(self, h)

    def kzg_compute_cells_batch(self, setup: KzgSetup, blobs):
        """blobs (n, BLOB_BYTES) -> (cells (n, 128, CELL_BYTES), status (n,)) (compute_cells; KZG_BAD_SCALAR for an element
        >= r, with zero cells)."""
        b = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, BLOB_BYTES)
        n = b.shape[0]
        cells, st = np.zeros((n, CELLS_PER_EXT_BLOB, CELL_BYTES), np.uint8), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_compute_cells_batch(self._ctx, setup.handle, _ptr(b), n, _ptr(cells), _ptr(st)))
        return cells, st

    def kzg_compute_cells_and_proofs_batch(self, setup: KzgSetup, blobs):
        """blobs (n, BLOB_BYTES) -> (cells (n, 128, CELL_BYTES), proofs (n, 128, 12), proof_inf (n, 128), status (n,))
        (compute_cells_and_kzg_proofs)."""
        b = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, BLOB_BYTES)
        n = b.shape[0]
        cells = np.zeros((n, CELLS_PER_EXT_BLOB, CELL_BYTES), np.uint8)
        pr, pi, st = np.zeros((n, CELLS_PER_EXT_BLOB, 12), np.uint64), np.zeros((n, CELLS_PER_EXT_BLOB), np.uint8), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_compute_cells_and_proofs_batch(self._ctx, setup.handle, _ptr(b), n, _ptr(cells), _ptr(pr), _ptr(pi),
                                                                     _ptr(st)))
        return cells, pr, pi, st

    def kzg_verify_cell_batch(self, setup: KzgSetup, commitments, cell_indices, cells, proofs, commitment_inf=None, proof_inf=None):
        """Per cell: commitments (n, 12), cell_indices (n,), cells (n, CELL_BYTES), proofs (n, 12), flags (n,) or None ->
        status (n,) of KZG_* (verify_cell_kzg_proof_batch is the AND of status == KZG_VALID)."""
        c = np.ascontiguousarray(commitments, dtype=np.uint64).reshape(-1, 12)
        n = c.shape[0]
        idx = np.ascontiguousarray(cell_indices, dtype=np.uint64).reshape(n)
        cl = np.ascontiguousarray(cells, dtype=np.uint8).reshape(n, CELL_BYTES)
        pr = np.ascontiguousarray(proofs, dtype=np.uint64).reshape(n, 12)
        ci, pi = _np8(commitment_inf, n), _np8(proof_inf, n)
        st = np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_verify_cell_batch(self._ctx, setup.handle, _ptr(c), _ptr(ci), _ptr(idx), _ptr(cl), _ptr(pr), _ptr(pi), n,
                                                        _ptr(st)))
        return st

    @staticmethod
    def _recover_inputs(cell_indices, cells, num_cells):
        idx = np.ascontiguousarray(cell_indices, dtype=np.uint64).reshape(-1, CELLS_PER_EXT_BLOB)
        n = idx.shape[0]
        cl = np.ascontiguousarray(cells, dtype=np.uint8).reshape(n, CELLS_PER_EXT_BLOB, CELL_BYTES)
        num = np.ascontiguousarray(num_cells, dtype=np.uint64).reshape(n)
        return idx, cl, num, n

    def kzg_recover_cells_batch(self, setup: KzgSetup, cell_indices, cells, num_cells):
        """recover_cells_and_kzg_proofs without the proofs.  Per blob: cell_indices (n, 128), cells (n, 128, CELL_BYTES) and
        num_cells (n,), of which the first num_cells[b] entries are the given cells -> (cells (n, 128, CELL_BYTES), status
        (n,)); KZG_BAD_CELLS for a count outside [64, 128], indices not strictly ascending or one >= 128, KZG_BAD_SCALAR
        for an element >= r, both with zero cells."""
        idx, cl, num, n = self._recover_inputs(cell_indices, cells, num_cells)
        out, st = np.zeros((n, CELLS_PER_EXT_BLOB, CELL_BYTES), np.uint8), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_recover_cells_batch(self._ctx, setup.handle, _ptr(idx), _ptr(cl), _ptr(num), n, _ptr(out), _ptr(st)))
        return out, st

    def kzg_recover_cells_and_proofs_batch(self, setup: KzgSetup, cell_indices, cells, num_cells):
        """recover_cells_and_kzg_proofs: inputs as kzg_recover_cells_batch -> (cells (n, 128, CELL_BYTES), proofs (n, 128, 12),
        proof_inf (n, 128), status (n,)), as kzg_compute_cells_and_proofs_batch returns them."""
        idx, cl, num, n = self._recover_inputs(cell_indices, cells, num_cells)
        out = np.zeros((n, CELLS_PER_EXT_BLOB, CELL_BYTES), np.uint8)
        pr, pi, st = np.zeros((n, CELLS_PER_EXT_BLOB, 12), np.uint64), np.zeros((n, CELLS_PER_EXT_BLOB), np.uint8), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_kzg_recover_cells_and_proofs_batch(self._ctx, setup.handle, _ptr(idx), _ptr(cl), _ptr(num), n, _ptr(out),
                                                                     _ptr(pr), _ptr(pi), _ptr(st)))
        return out, pr, pi, st

    def kzg_recover_cells_dev(self, setup: KzgSetup, d_cell_indices, d_cells, d_num_cells, n: int, d_out_cells, d_status,
                              stream: int = 0, dev: int = 0):
        """Asynchronous form on device-resident torch tensors; d_cells and d_out_cells 16-byte aligned."""
        self._check(self._lib.zkp_kzg_recover_cells_dev(self._ctx, dev, setup.handle, _dptr(d_cell_indices), _dptr(d_cells), _dptr(d_num_cells),
                                                        n, _dptr(d_out_cells), _dptr(d_status), ctypes.c_void_p(stream)))

    def kzg_recover_cells_and_proofs_dev(self, setup: KzgSetup, d_cell_indices, d_cells, d_num_cells, n: int, d_out_cells, d_proofs,
                                         d_proof_inf, d_status, d_scratch, stream: int = 0, dev: int = 0):
        """Asynchronous form; d_scratch holds kzg_cells_proofs_scratch_bytes(n) bytes; d_cells, d_out_cells, d_scratch 16-byte
        aligned."""
        self._check(self._lib.zkp_kzg_recover_cells_and_proofs_dev(self._ctx, dev, setup.handle, _dptr(d_cell_indices), _dptr(d_cells),
                                                                   _dptr(d_num_cells), n, _dptr(d_out_cells), _dptr(d_proofs),
                                                                   _dptr(d_proof_inf), _dptr(d_status), _dptr(d_scratch),
                                                                   ctypes.c_void_p(stream)))

    def kzg_cells_proofs_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_kzg_cells_proofs_scratch_bytes(n))

    def kzg_verify_cell_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_kzg_verify_cell_scratch_bytes(n))

    def kzg_compute_cells_dev(self, setup: KzgSetup, d_blobs, n: int, d_cells, d_status, stream: int = 0, dev: int = 0):
        """Asynchronous form on device-resident torch tensors; d_blobs and d_cells 16-byte aligned."""
        self._check(self._lib.zkp_kzg_compute_cells_dev(self._ctx, dev, setup.handle, _dptr(d_blobs), n, _dptr(d_cells), _dptr(d_status),
                                                        ctypes.c_void_p(stream)))

    def kzg_compute_cells_and_proofs_dev(self, setup: KzgSetup, d_blobs, n: int, d_cells, d_proofs, d_proof_inf, d_status, d_scratch,
                                         stream: int = 0, dev: int = 0):
        """Asynchronous form; d_scratch holds kzg_cells_proofs_scratch_bytes(n) bytes; d_blobs, d_cells, d_scratch 16-byte aligned."""
        self._check(self._lib.zkp_kzg_compute_cells_and_proofs_dev(self._ctx, dev, setup.handle, _dptr(d_blobs), n, _dptr(d_cells),
                                                                   _dptr(d_proofs), _dptr(d_proof_inf), _dptr(d_status), _dptr(d_scratch),
                                                                   ctypes.c_void_p(stream)))

    def kzg_verify_cell_dev(self, setup: KzgSetup, d_commitments, d_cell_indices, d_cells, d_proofs, n: int, d_status, d_scratch,
                            d_commitment_inf=None, d_proof_inf=None, stream: int = 0, dev: int = 0):
        """Asynchronous form; d_scratch holds kzg_verify_cell_scratch_bytes(n) bytes; d_cells and d_scratch 16-byte aligned."""
        self._check(self._lib.zkp_kzg_verify_cell_dev(self._ctx, dev, setup.handle, _dptr(d_commitments), _dptr(d_commitment_inf),
                                                      _dptr(d_cell_indices), _dptr(d_cells), _dptr(d_proofs), _dptr(d_proof_inf), n,
                                                      _dptr(d_status), _dptr(d_scratch), ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ byte (de)serialisation (SURVEY 8f)
    def fp_from_bytes_batch(self, data):
        """Fp::from_bytes (src/fp.rs:165-191): (n,48) big-endian bytes -> (limbs (n,6) uint64, ok (n,) uint8)."""
        b = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1, 48)
        n = b.shape[0]
        out, ok = np.empty((n, 6), np.uint64), np.zeros(n, np.uint8)
        self._check(self._lib.zkp_fp_from_bytes_batch(self._ctx, _ptr(b), n, _ptr(out), _ptr(ok)))
        return out, ok

    def fp_to_bytes_batch(self, limbs):
        """Fp::to_bytes (src/fp.rs:195-207): (n,6) uint64 limbs -> (n,48) big-endian bytes."""
        a = np.ascontiguousarray(limbs, dtype=np.uint64).reshape(-1, 6)
        out = np.empty((a.shape[0], 48), np.uint8)
        self._check(self._lib.zkp_fp_to_bytes_batch(self._ctx, _ptr(a), a.shape[0], _ptr(out)))
        return out

    def fp_bytes_dev(self, direction: int, d_in, d_out, n: int, ok=None, stream: int = 0, dev: int = 0):
        self._check(self._lib.zkp_fp_bytes_dev(self._ctx, dev, direction, _dptr(d_in), _dptr(d_out), _dptr(ok), n, ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ group-level ops (SURVEY 8f)
    def _pts(self, pts, width, inf):
        pts = np.ascontiguousarray(pts, dtype=np.uint64).reshape(-1, width)
        n = pts.shape[0]
        if inf is not None:
            inf = np.ascontiguousarray(inf, dtype=np.uint8).reshape(-1)
            if inf.shape[0] != n:
                raise ValueError("infinity flags do not match the number of points")
        return pts, inf, n

    def g1_check_batch(self, g1, g1_inf=None):
        """G1Affine::is_valid per point (src/g1.rs:49-62) -> uint8 status: 0 ok, 1 not on curve, 2 not torsion free."""
        pts, inf, n = self._pts(g1, 12, g1_inf)
        st = np.zeros(n, np.uint8)
        self._check(self._lib.zkp_g1_check_batch(self._ctx, _ptr(pts), _ptr(inf), n, _ptr(st)))
        return st

    def g2_check_batch(self, g2, g2_inf=None):
        """G2Affine::is_valid per point (src/g2.rs:57-69) -> uint8 status."""
        pts, inf, n = self._pts(g2, 24, g2_inf)
        st = np.zeros(n, np.uint8)
        self._check(self._lib.zkp_g2_check_batch(self._ctx, _ptr(pts), _ptr(inf), n, _ptr(st)))
        return st

    def _mul(self, fn, pts, width, inf, scalars):
        pts, inf, n = self._pts(pts, width, inf)
        k = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
        if k.shape[0] != n:
            raise ValueError("one 4-limb scalar per point expected")
        out, oinf = np.empty((n, width), np.uint64), np.zeros(n, np.uint8)
        self._check(fn(self._ctx, _ptr(pts), _ptr(inf), _ptr(k), n, _ptr(out), _ptr(oinf)))
        return out, oinf

    def g1_mul_batch(self, g1, scalars, g1_inf=None):
        """[k_i]P_i (scalars: (n,4) little-endian u64 limbs of an Fr) -> (points (n,12), is_infinity (n,))."""
        return self._mul(self._lib.zkp_g1_mul_batch, g1, 12, g1_inf, scalars)

    def g2_mul_batch(self, g2, scalars, g2_inf=None):
        return self._mul(self._lib.zkp_g2_mul_batch, g2, 24, g2_inf, scalars)

    # ------------------------------------------------------------------ device-resident (torch tensors)
    def _add(self, fn, a, b, width, a_inf, b_inf):
        a, ai, n = self._pts(a, width, a_inf)
        b, bi, nb = self._pts(b, width, b_inf)
        if nb != n:
            raise ValueError("operands differ in length")
        out, flag = np.empty((n, width), np.uint64), np.zeros(n, np.uint8)
        self._check(fn(self._ctx, _ptr(a), _ptr(ai), _ptr(b), _ptr(bi), n, _ptr(out), _ptr(flag)))
        return out, flag

    def g1_add_batch(self, a, b, a_inf=None, b_inf=None):
        """a_i + b_i, `&G1Affine + &G1Affine` (src/g1.rs:155-187) -> (points (n,12), flag: bit0 identity, bit1 the
        reference panics here (P + (-P)): identity returned)."""
        return self._add(self._lib.zkp_g1_add_batch, a, b, 12, a_inf, b_inf)

    def g2_add_batch(self, a, b, a_inf=None, b_inf=None):
        """`&G2Affine + &G2Affine` (src/g2.rs:210-242)."""
        return self._add(self._lib.zkp_g2_add_batch, a, b, 24, a_inf, b_inf)

    def _msm(self, fn, pts, width, inf, scalars):
        pts, inf, n = self._pts(pts, width, inf)
        k = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
        if k.shape[0] != n:
            raise ValueError("one 4-limb scalar per point expected")
        out, oinf, st = np.zeros(width, np.uint64), np.zeros(1, np.uint8), np.zeros(1, np.uint8)
        self._check(fn(self._ctx, _ptr(pts), _ptr(inf), _ptr(k), n, _ptr(out), _ptr(oinf), _ptr(st)))
        return out, int(oinf[0]), int(st[0])

    def g1_msm(self, points, scalars, inf=None):
        """sum_i [k_i]P_i over caller-given G1 points (scalars: (n,4) little-endian u64, any 256-bit integer, not reduced
        mod r; no subgroup check) -> (point (12,) uint64, is_infinity, status: 0 ok, 1 a point off the curve (ZKP_POINT_*))."""
        return self._msm(self._lib.zkp_g1_msm, points, 12, inf, scalars)

    def g2_msm(self, points, scalars, inf=None):
        """sum_i [k_i]Q_i over caller-given G2 points -> (point (24,) uint64, is_infinity, status)."""
        return self._msm(self._lib.zkp_g2_msm, points, 24, inf, scalars)

    def g1_msm_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_g1_msm_scratch_bytes(n))

    def g2_msm_scratch_bytes(self, n: int) -> int:
        return int(self._lib.zkp_g2_msm_scratch_bytes(n))

    def g1_msm_dev(self, d_points, d_scalars, n: int, d_out, d_out_inf, d_status, d_scratch, d_inf=None, err=None, stream: int = 0,
                   dev: int = 0):
        """Asynchronous form on device-resident torch tensors; d_scratch holds g1_msm_scratch_bytes(n) bytes, 16-byte
        aligned; d_out takes 12 u64, d_out_inf and d_status one byte each."""
        self._check(self._lib.zkp_g1_msm_dev(self._ctx, dev, _dptr(d_points), _dptr(d_inf), _dptr(d_scalars), n, _dptr(d_out),
                                             _dptr(d_out_inf), _dptr(d_status), _dptr(err), _dptr(d_scratch), ctypes.c_void_p(stream)))

    def g2_msm_dev(self, d_points, d_scalars, n: int, d_out, d_out_inf, d_status, d_scratch, d_inf=None, err=None, stream: int = 0,
                   dev: int = 0):
        """The G2 form of g1_msm_dev (d_out takes 24 u64, d_scratch g2_msm_scratch_bytes(n) bytes)."""
        self._check(self._lib.zkp_g2_msm_dev(self._ctx, dev, _dptr(d_points), _dptr(d_inf), _dptr(d_scalars), n, _dptr(d_out),
                                             _dptr(d_out_inf), _dptr(d_status), _dptr(err), _dptr(d_scratch), ctypes.c_void_p(stream)))

    def pairing_dev(self, mode: int, out, g1=None, g2=None, g1_inf=None, g2_inf=None, in_fp12=None, n_checks=None,
                    pairs_per_check: int = 1, is_one=None, err=None, stream: int = 0, dev: int = 0):
        """Asynchronous launch on device-resident buffers (torch CUDA tensors).  ``stream`` is a raw
        cudaStream_t handle (``torch.cuda.current_stream().cuda_stream``); 0 = the legacy default stream,
        which is also torch's default stream, so the launch is ordered with the caller's torch work."""
        if n_checks is None:
            n_checks = out.numel() // 72
        self._check(self._lib.zkp_pairing_dev(self._ctx, dev, mode, _dptr(g1), _dptr(g1_inf), _dptr(g2), _dptr(g2_inf), n_checks,
                                              pairs_per_check, _dptr(in_fp12), _dptr(out), _dptr(is_one), _dptr(err),
                                              ctypes.c_void_p(stream)))

    def tower_op_dev(self, name: str, a, b, out, n: int, status=None, err=None, stream: int = 0, dev: int = 0):
        self._check(self._lib.zkp_tower_op_dev(self._ctx, dev, TOWER_OPS[name], _dptr(a), _dptr(b), _dptr(out), _dptr(status), _dptr(err),
                                               n, ctypes.c_void_p(stream)))

    def product_scratch_elems(self, n: int) -> int:
        return int(self._lib.zkp_product_scratch_elems(n))

    def fp12_product_dev(self, d_in, n: int, scratch, out, err=None, stream: int = 0, dev: int = 0):
        self._check(self._lib.zkp_fp12_product_dev(self._ctx, dev, _dptr(d_in), n, _dptr(scratch), _dptr(out), _dptr(err),
                                                   ctypes.c_void_p(stream)))

    def gen_points_dev(self, seed: int, first: int, n: int, g1, g1_inf, g2, g2_inf, stream: int = 0, dev: int = 0):
        self._check(self._lib.zkp_gen_points_dev(self._ctx, dev, seed, first, n, _dptr(g1), _dptr(g1_inf), _dptr(g2), _dptr(g2_inf),
                                                 ctypes.c_void_p(stream)))

    # ------------------------------------------------------------------ measurement
    def imad_peak(self, kind: int = 0, dev: int = 0) -> float:
        """Measured integer multiply-accumulates per second (kind 0: IMAD.WIDE.U32, 1: IMAD, 2: carry-chained wide MACs)."""
        v = ctypes.c_double(0)
        self._check(self._lib.zkp_imad_peak(self._ctx, dev, kind, ctypes.byref(v)))
        return v.value

    def set_kernel_timing(self, enabled: bool):
        self._check(self._lib.zkp_set_kernel_timing(self._ctx, 1 if enabled else 0))

    def last_kernel_ms(self, dev: int = 0):
        """(total ms, launches) of the pairing kernels timed with CUDA events since the last call."""
        ms, n = ctypes.c_double(0), ctypes.c_uint64(0)
        self._check(self._lib.zkp_last_kernel_ms(self._ctx, dev, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, int(n.value)


def device_count() -> int:
    return int(_lib.load().zkp_device_count())
