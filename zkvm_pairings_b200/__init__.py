"""zkvm_pairings_b200 -- B200-native batched BLS12-381 pairing engine.

Drop-in for the pairing hot path of 0xWOLAND/zkvm-pairings: hand-written sm_100a CUDA behind the
C ABI of include/zkpair.h (libzkpair.so), driven from Python through ctypes.  No CPU fallback.
"""
from .engine import (BLOB_BYTES, CELL_BYTES, CELLS_PER_EXT_BLOB, FIELD_ELEMENTS_PER_CELL, G16_BAD_INPUT, G16_BAD_POINT, G16_INVALID, G16_VALID, GROTH16_MAX_PUBLIC, KZG_BAD_CELLS, KZG_BAD_POINT, KZG_BAD_SCALAR,
                     KZG_INVALID, KZG_VALID, MODE_FINAL_EXP, MODE_MILLER, MODE_MILLER_FOR_FINAL_EXP, MODE_PAIRING, TOWER_OPS,
                     Groth16VerifyingKey, KzgSetup, NonCanonicalError, PairingEngine, ZkpError, device_count, op_widths)

__all__ = ["PairingEngine", "ZkpError", "NonCanonicalError", "TOWER_OPS", "MODE_MILLER", "MODE_FINAL_EXP",
           "MODE_PAIRING", "MODE_MILLER_FOR_FINAL_EXP", "device_count", "op_widths", "Groth16VerifyingKey",
           "G16_VALID", "G16_INVALID", "G16_BAD_POINT", "G16_BAD_INPUT", "GROTH16_MAX_PUBLIC", "KzgSetup",
           "KZG_VALID", "KZG_INVALID", "KZG_BAD_POINT", "KZG_BAD_SCALAR", "KZG_BAD_CELLS", "BLOB_BYTES",
           "CELLS_PER_EXT_BLOB", "FIELD_ELEMENTS_PER_CELL", "CELL_BYTES"]
