"""Host-side mirror of `ethereum_consensus::crypto::kzg`, backed by the CUDA library — no CPU fallback.

Same names, argument order and errors as the reference's ethereum-consensus/src/crypto/kzg.rs: the byte-size constants
(:5-9), `kzg_settings_from_json` (:39-45), `Error` with `CKzg` / `InvalidProof` (:47-53), `ProofAndEvaluation` (:55-59),
`blob_to_kzg_commitment` (:60-69), `compute_kzg_proof` (:71-86), `compute_blob_kzg_proof` (:88-99), `verify_kzg_proof`
(:101-122), `verify_blob_kzg_proof` (:124-137) and `verify_blob_kzg_proof_batch` (:139-174).  `verify_blob_kzg_proofs`,
`blob_to_kzg_commitments` and `compute_blob_kzg_proofs` are the per-blob throughput paths (one code per blob, no
counterpart in the reference).

Rust `Result<(), Error>` becomes: return None on Ok, raise on Err.
"""
from __future__ import annotations

import ctypes as C
import json
from dataclasses import dataclass
from typing import Sequence, Tuple

import numpy as np

from . import _lib

BYTES_PER_FIELD_ELEMENT = 32
BYTES_PER_COMMITMENT = 48
BYTES_PER_PROOF = 48
BYTES_PER_G1_POINT = 48
BYTES_PER_G2_POINT = 96
FIELD_ELEMENTS_PER_BLOB = 4096
BYTES_PER_BLOB = FIELD_ELEMENTS_PER_BLOB * BYTES_PER_FIELD_ELEMENT
MAX_BLOBS_PER_CALL = 16384   # B200_KZG_MAX_BLOBS

_lib.register_protos({
    "b200_kzg_settings_load": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "b200_kzg_settings_free": (None, [C.c_void_p]),
    "b200_verify_kzg_proof": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200_verify_blob_kzg_proof": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200_verify_blob_kzg_proof_batch": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200_verify_blob_kzg_proofs": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200_blob_to_kzg_commitment": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200_compute_kzg_proof": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200_compute_blob_kzg_proof": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200_blob_to_kzg_commitments": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "b200_compute_blob_kzg_proofs": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
})


class Error(Exception):
    """`kzg::Error` (crypto/kzg.rs:47-53)."""


class CKzgError(Error):
    """`Error::CKzg(..)`: malformed input (wrong length, field element >= r, point that does not decode or is not in G1,
    mismatched batch lengths, bad trusted setup)."""

    def __init__(self, what: str = "bad arguments"):
        super().__init__(f"c-kzg error: {what}")


class InvalidProof(Error):
    def __init__(self):
        super().__init__("proof verification failed")


class KzgSettings:
    """Device-resident settings (`c_kzg::KzgSettings`): [tau]G2 and the bit-reversed roots of unity for verification, and
    the prover's fixed-base table built from g1_lagrange."""

    def __init__(self, g1_lagrange: bytes, g2_monomial: bytes):
        g1, g2 = bytes(g1_lagrange), bytes(g2_monomial)
        if len(g1) % BYTES_PER_G1_POINT or len(g2) % BYTES_PER_G2_POINT:
            raise CKzgError("trusted setup point of the wrong length")
        self._h = None
        lib = _lib.init()
        h = C.c_void_p()
        rc = _lib.check(lib.b200_kzg_settings_load(g1, len(g1) // BYTES_PER_G1_POINT, g2, len(g2) // BYTES_PER_G2_POINT,
                                                   C.byref(h)), "b200_kzg_settings_load")
        if rc != 0:
            raise CKzgError("invalid trusted setup")
        self._h = h

    @classmethod
    def load_trusted_setup(cls, g1_points: Sequence[bytes], g2_points: Sequence[bytes]) -> "KzgSettings":
        return cls(b"".join(bytes(p) for p in g1_points), b"".join(bytes(p) for p in g2_points))

    @property
    def handle(self):
        return self._h

    def __del__(self):
        if getattr(self, "_h", None) is not None and _lib._lib is not None:
            _lib._lib.b200_kzg_settings_free(self._h)
            self._h = None


def _hex_points(items, n):
    out = []
    for s in items:
        b = bytes.fromhex(s[2:] if s.startswith("0x") else s)
        if len(b) != n:
            raise CKzgError("trusted setup point of the wrong length")
        out.append(b)
    return out


def kzg_settings_from_json(trusted_setup_json: str) -> KzgSettings:
    """crypto/kzg.rs:39-45: `{"g1_lagrange": [...], "g2_monomial": [...]}` with 0x-hex compressed points."""
    d = json.loads(trusted_setup_json)
    return KzgSettings.load_trusted_setup(_hex_points(d["g1_lagrange"], BYTES_PER_G1_POINT),
                                          _hex_points(d["g2_monomial"], BYTES_PER_G2_POINT))


def _bytes(x, n: int, what: str) -> bytes:
    b = bytes(x)
    if len(b) != n:
        raise CKzgError(f"{what} must be {n} bytes, got {len(b)}")
    return b


def _result(rc: int, where: str) -> None:
    _lib.check(rc, where)
    if rc == _lib.VERIFY_FAIL:
        raise InvalidProof()
    if rc != 0:
        raise CKzgError()


def verify_kzg_proof(commitment, evaluation_point, result_point, proof, kzg_settings: KzgSettings) -> None:
    c = _bytes(commitment, BYTES_PER_COMMITMENT, "commitment")
    z = _bytes(evaluation_point, BYTES_PER_FIELD_ELEMENT, "evaluation point")
    y = _bytes(result_point, BYTES_PER_FIELD_ELEMENT, "result point")
    p = _bytes(proof, BYTES_PER_PROOF, "proof")
    _result(_lib.init().b200_verify_kzg_proof(kzg_settings.handle, c, z, y, p), "b200_verify_kzg_proof")


def verify_blob_kzg_proof(blob, commitment, proof, kzg_settings: KzgSettings) -> None:
    b = _bytes(blob, BYTES_PER_BLOB, "blob")
    c = _bytes(commitment, BYTES_PER_COMMITMENT, "commitment")
    p = _bytes(proof, BYTES_PER_PROOF, "proof")
    _result(_lib.init().b200_verify_blob_kzg_proof(kzg_settings.handle, b, c, p), "b200_verify_blob_kzg_proof")


def _flat(xs, n: int, what: str):
    """A sequence of byte strings, or an already flat uint8 array / tensor (not copied), -> (buffer, count)."""
    if isinstance(xs, np.ndarray) or hasattr(xs, "data_ptr"):
        nbytes = xs.nbytes if isinstance(xs, np.ndarray) else xs.numel() * xs.element_size()
        if nbytes % n:
            raise CKzgError(f"{what}: {nbytes} bytes is not a multiple of {n}")
        if hasattr(xs, "is_contiguous") and not xs.is_contiguous():
            raise CKzgError(f"{what}: tensor must be contiguous")
        return xs, nbytes // n
    items = [_bytes(x, n, what) for x in xs]
    return b"".join(items), len(items)


def _batch_args(blobs, commitments, proofs):
    b, nb = _flat(blobs, BYTES_PER_BLOB, "blob")
    c, nc = _flat(commitments, BYTES_PER_COMMITMENT, "commitment")
    p, npf = _flat(proofs, BYTES_PER_PROOF, "proof")
    if not nb == nc == npf:
        raise CKzgError(f"batch lengths differ: {nb} blobs, {nc} commitments, {npf} proofs")
    if nb > MAX_BLOBS_PER_CALL:
        raise ValueError(f"at most {MAX_BLOBS_PER_CALL} blobs per call, got {nb}")
    return b, c, p, nb


def verify_blob_kzg_proof_batch(blobs, commitments, proofs, kzg_settings: KzgSettings) -> None:
    b, c, p, n = _batch_args(blobs, commitments, proofs)
    _result(_lib.init().b200_verify_blob_kzg_proof_batch(kzg_settings.handle, _lib.ptr(b), _lib.ptr(c), _lib.ptr(p), n),
            "b200_verify_blob_kzg_proof_batch")


def verify_blob_kzg_proofs(blobs, commitments, proofs, kzg_settings: KzgSettings) -> np.ndarray:
    """Per-blob codes (int32): 0 valid, 5 invalid proof, 17 malformed input — what `verify_blob_kzg_proof` decides for
    each blob.  `blobs` / `commitments` / `proofs` may be sequences of bytes or flat uint8 arrays (pinned tensors too)."""
    b, c, p, n = _batch_args(blobs, commitments, proofs)
    out = np.zeros(n, dtype=np.int32)
    if n:
        _lib.check(_lib.init().b200_verify_blob_kzg_proofs(kzg_settings.handle, _lib.ptr(b), _lib.ptr(c), _lib.ptr(p), n,
                                                           out.ctypes.data), "b200_verify_blob_kzg_proofs")
    return out


# ---------------------------------------------------------------------------------------------------- the prover
@dataclass(frozen=True)
class ProofAndEvaluation:
    """crypto/kzg.rs:55-59: the proof and y = p(z), compared by value."""
    proof: bytes
    evaluation: bytes


def blob_to_kzg_commitment(blob, kzg_settings: KzgSettings) -> bytes:
    b = _bytes(blob, BYTES_PER_BLOB, "blob")
    out = C.create_string_buffer(BYTES_PER_COMMITMENT)
    _result(_lib.init().b200_blob_to_kzg_commitment(kzg_settings.handle, b, out), "b200_blob_to_kzg_commitment")
    return out.raw


def compute_kzg_proof(blob, evaluation_point, kzg_settings: KzgSettings) -> ProofAndEvaluation:
    b = _bytes(blob, BYTES_PER_BLOB, "blob")
    z = _bytes(evaluation_point, BYTES_PER_FIELD_ELEMENT, "evaluation point")
    proof, y = C.create_string_buffer(BYTES_PER_PROOF), C.create_string_buffer(BYTES_PER_FIELD_ELEMENT)
    _result(_lib.init().b200_compute_kzg_proof(kzg_settings.handle, b, z, proof, y), "b200_compute_kzg_proof")
    return ProofAndEvaluation(proof.raw, y.raw)


def compute_blob_kzg_proof(blob, commitment, kzg_settings: KzgSettings) -> bytes:
    b = _bytes(blob, BYTES_PER_BLOB, "blob")
    c = _bytes(commitment, BYTES_PER_COMMITMENT, "commitment")
    out = C.create_string_buffer(BYTES_PER_PROOF)
    _result(_lib.init().b200_compute_blob_kzg_proof(kzg_settings.handle, b, c, out), "b200_compute_blob_kzg_proof")
    return out.raw


def _check_count(n: int) -> None:
    if n > MAX_BLOBS_PER_CALL:
        raise ValueError(f"at most {MAX_BLOBS_PER_CALL} blobs per call, got {n}")


def blob_to_kzg_commitments(blobs, kzg_settings: KzgSettings) -> Tuple[np.ndarray, np.ndarray]:
    """(commitments uint8 [n, 48], codes int32 [n]): per blob 0 and its commitment, or 17 (an element >= r) and zeros.
    `blobs` may be a sequence of bytes or a flat uint8 array (pinned tensors too)."""
    b, n = _flat(blobs, BYTES_PER_BLOB, "blob")
    _check_count(n)
    out, codes = np.zeros((n, BYTES_PER_COMMITMENT), np.uint8), np.zeros(n, np.int32)
    if n:
        _lib.check(_lib.init().b200_blob_to_kzg_commitments(kzg_settings.handle, _lib.ptr(b), n, out.ctypes.data,
                                                            codes.ctypes.data), "b200_blob_to_kzg_commitments")
    return out, codes


def compute_blob_kzg_proofs(blobs, commitments, kzg_settings: KzgSettings) -> Tuple[np.ndarray, np.ndarray]:
    """(proofs uint8 [n, 48], codes int32 [n]): per blob what `compute_blob_kzg_proof` returns (0 and the proof, or 17
    and zeros)."""
    b, nb = _flat(blobs, BYTES_PER_BLOB, "blob")
    c, nc = _flat(commitments, BYTES_PER_COMMITMENT, "commitment")
    if nb != nc:
        raise CKzgError(f"batch lengths differ: {nb} blobs, {nc} commitments")
    _check_count(nb)
    out, codes = np.zeros((nb, BYTES_PER_PROOF), np.uint8), np.zeros(nb, np.int32)
    if nb:
        _lib.check(_lib.init().b200_compute_blob_kzg_proofs(kzg_settings.handle, _lib.ptr(b), _lib.ptr(c), nb, out.ctypes.data,
                                                            codes.ctypes.data), "b200_compute_blob_kzg_proofs")
    return out, codes
